#!/usr/bin/env python
"""MAPPO + PFSP self-play on the batched environment (BASELINE.json config 5): the batched counterpart of the
reference's ``self_play_driver.py``.  One process per GPU under torchrun; worlds are sharded, gradients
all-reduced over NCCL per minibatch.

    python tools/train_selfplay.py --map agh-map --worlds 4096 --iterations 2 --timesteps 256
    python tools/train_selfplay.py --map squarinth,agh-map,labyrinth --worlds 4096   # one policy over three maps
    python tools/train_selfplay.py --map squarinth --procedural 2 --swap-every 4     # + 2 slots of fresh mazes
    python tools/train_selfplay.py --map squarinth,agh-map --episode-stats            # + episode returns / lengths
    python tools/train_selfplay.py --episode-stats --randomize "max_speed.thief=125:175,termination_radius=15:25"
    python tools/train_selfplay.py --map squarinth --scripted thief_0=evade --eval-scripted 2   # cops vs a scripted thief
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/train_selfplay.py ...

Prints one JSON line per self-play iteration (rank 0): environment agent-steps/s inside training, GAE / update /
all-reduce milliseconds per update, win rates; with --episode-stats also "episodes": what the training episodes of the
iteration added up to (all ranks), overall and per map slot (the evaluation's episodes are not counted); with
--eval-scripted also "eval_vs_scripted": the cops' win rate against an evading thief and the thief's against chasing
cops (the step kernel's controllers), overall and per map, on this rank's worlds.
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from as_cops_and_thieves_b200 import episodes, scripts, selfplay, world_params  # noqa: E402
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner  # noqa: E402
from as_cops_and_thieves_b200.maps import free_space_regions, generate_maze, load_named_map  # noqa: E402
from as_cops_and_thieves_b200.sharding import dist_env, shard_range  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map", default="agh-map",
                    help="built-in map, or a comma-separated list of them: one mixed-map environment whose worlds are "
                         "split evenly over the maps (every rank hosts the same split)")
    ap.add_argument("--worlds", type=int, default=4096, help="worlds per GPU")
    ap.add_argument("--iterations", type=int, default=2)
    ap.add_argument("--timesteps", type=int, default=256, help="lockstep steps per self-play iteration")
    ap.add_argument("--rollouts", type=int, default=64)
    ap.add_argument("--model", default="lstm", choices=["lstm", "mlp"])
    ap.add_argument("--max-step-count", type=int, default=2000)     # self_play_driver.py:34
    ap.add_argument("--archive", default="policy_archive")
    ap.add_argument("--free-spawn", type=int, default=1)
    ap.add_argument("--autocast", default="none", choices=["none", "bf16"])
    ap.add_argument("--schedule", default="scaled", choices=["scaled", "reference", "off"],
                    help="random_timesteps / learning_starts / freeze durations: the reference's values divided by the "
                         "number of worlds (same number of transitions), the reference's values as they are, or none")
    ap.add_argument("--time-limit-bootstrap", action="store_true",
                    help="bootstrap timed-out episodes from the critic's value of their final observation")
    ap.add_argument("--procedural", type=int, default=0,
                    help="add this many map slots holding generated mazes (maps.generate_maze) to --map")
    ap.add_argument("--swap-every", type=int, default=0,
                    help="with --procedural: every this many updates, replace one maze slot (round robin) by a fresh maze")
    ap.add_argument("--maze-seed", type=int, default=0, help="seed of the first maze; later mazes take the next seeds")
    ap.add_argument("--episode-stats", action="store_true",
                    help="report the returns, lengths and capture rate of the training episodes, overall and per map")
    ap.add_argument("--randomize", default="",
                    help="domain randomisation drawn at every re-spawn, e.g. 'max_speed.thief=125:175,termination_radius="
                         "15:25,max_step_count=300:500' (field[.cop|.thief]=lo:hi, or one number to pin it)")
    ap.add_argument("--scripted", default="",
                    help="agents played by the step kernel's controllers, e.g. 'thief_0=evade' (random, chase, evade): "
                         "the learner trains the remaining agents against them")
    ap.add_argument("--eval-scripted", type=int, default=0, metavar="K",
                    help="after each iteration, K episodes per world of the cops against an evading thief and of the "
                         "thief against chasing cops (a role the learner does not train is skipped)")
    a = ap.parse_args()
    randomize = world_params.parse_cli(a.randomize) if a.randomize else None
    scripted = scripts.parse_spec(a.scripted) if a.scripted or a.eval_scripted > 0 else None

    rank, local_rank, world_size = dist_env()
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world_size > 1:
        import os
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    names = [n.strip() for n in a.map.split(",") if n.strip()]
    maps = [load_named_map(n) for n in names]
    gid0, n_local = shard_range(a.worlds * world_size, rank, world_size)
    spawn = [free_space_regions(m) if a.free_spawn else None for m in maps]
    # every rank generates the same mazes from the same seeds, so the sharded worlds see the same layouts
    next_maze = a.maze_seed
    for _ in range(a.procedural):
        maps.append(generate_maze(next_maze))
        spawn.append(None)            # a maze brings its own spawn regions
        next_maze += 1
    swappable = a.procedural > 0
    swaps = {"updates": 0, "next": next_maze}
    if len(maps) == 1:
        env = BatchedCopsThievesEnv(maps[0], n_local, device=dev, seed=0, gid0=gid0, max_step_count=a.max_step_count,
                                    spawn_override=spawn[0], final_observations=a.time_limit_bootstrap,
                                    episode_statistics=a.episode_stats, randomize=randomize,
                                    scripted=scripted)
    else:
        env = BatchedCopsThievesEnv(maps, n_local, device=dev, seed=0, gid0=gid0, max_step_count=a.max_step_count,
                                    spawn_override=spawn, final_observations=a.time_limit_bootstrap,
                                    swappable_maps=swappable, episode_statistics=a.episode_stats, randomize=randomize,
                                    scripted=scripted)
    # the reference's schedule (10 000 random / 15 000 before learning / 15 000 frozen policy) counts steps of ONE
    # environment; with thousands of lockstep worlds the same number of TRANSITIONS is reached in a few steps, so the
    # driver scales the durations by the world count unless told otherwise
    scale = max(1, a.worlds * world_size) if a.schedule == "scaled" else 1
    cfg = MAPPOConfig(rollouts=a.rollouts, model=a.model, distributed=world_size > 1, world_size=world_size,
                      update_autocast=a.autocast, time_limit_bootstrap=a.time_limit_bootstrap, random_timesteps=-(-10000 // scale) if a.schedule != "off" else 0,
                      learning_starts=-(-15000 // scale) if a.schedule != "off" else 0,
                      policy_freeze_duration=-(-15000 // scale) if a.schedule != "off" else 0,
                      opponent_freeze_duration=-(-15000 // scale) if a.schedule != "off" else 0)
    learner = MAPPOLearner(env, cfg, seed=0)
    archive = Path(a.archive) if rank == 0 else Path(a.archive + f".rank{rank}")
    # training episodes of the current iteration: (slot, map name) -> totals, read (and cleared) from the environment
    # before a slot is swapped and after training; the evaluation's episodes are cleared unread
    ep_parts = {}

    def take_episodes():
        raw = env.worlds.episode_totals_raw(reset=True)
        for m in range(len(raw)):
            key = (m, env.map_names[m])
            ep_parts[key] = episodes.merge_totals(np.stack([ep_parts[key], raw[m]]) if key in ep_parts else raw[m:m + 1])

    def episode_report():
        keys = list(ep_parts)        # the same keys in the same order on every rank: every rank swaps the same slots
        tot = np.stack([ep_parts[k] for k in keys]) if keys else episodes.empty_totals(0)
        if world_size > 1:
            import torch.distributed as dist
            tot = episodes.allreduce_totals(tot, dist.group.WORLD)
        ep_parts.clear()
        out = episodes.summarize_maps(tot, env.possible_agents, [name for _, name in keys], by_map=True)
        for entry, (slot, _) in zip(out["maps"], keys):
            entry["slot"] = slot
        return out

    for it in range(a.iterations):
        agg = {"gae_ms": 0.0, "update_ms": 0.0, "allreduce_ms": 0.0, "updates": 0}

        def cb(_l, stats):
            for st in stats.values():
                agg["gae_ms"] += st.gae_ms; agg["update_ms"] += st.update_ms; agg["allreduce_ms"] += st.allreduce_ms
            agg["updates"] += 1
            swaps["updates"] += 1
            if swappable and a.swap_every > 0 and swaps["updates"] % a.swap_every == 0:
                seed = swaps["next"]
                slot = len(names) + (seed - a.maze_seed) % a.procedural
                if a.episode_stats:
                    take_episodes()
                learner.note_reset(env.set_map(slot, generate_maze(seed)))
                swaps["next"] = seed + 1
        env_s0, t0 = learner.env_seconds, time.perf_counter()
        step0 = learner.timestep
        learner.train(learner.timestep + a.timesteps, callback=cb)
        train_s = time.perf_counter() - t0
        if a.episode_stats:
            take_episodes()
        tc = selfplay.TrainingConfig
        res_c = selfplay.evaluate_agent(env, learner, tc.cop_role_prefix, tc.thief_role_prefix, archive / "thief", tc)
        res_t = selfplay.evaluate_agent(env, learner, tc.thief_role_prefix, tc.cop_role_prefix, archive / "cop", tc)
        ck = archive / f"joint_iter_{it}_full_agent.pt"
        archive.mkdir(parents=True, exist_ok=True)
        learner.save(str(ck))
        selfplay.add_policy_to_archive(str(ck), archive / "cop", it, "cop")
        selfplay.add_policy_to_archive(str(ck), archive / "thief", it, "thief")
        steps = learner.timestep - step0
        extra = {}
        if a.episode_stats:
            env.worlds.episode_totals_raw(reset=True)        # the evaluation's episodes
            extra["episodes"] = episode_report()
        if a.eval_scripted > 0:
            vs = {}
            mixed = len(env.map_names) > 1
            for key, role, controller in (("cop_vs_evade", tc.cop_role_prefix, "evade"),
                                          ("thief_vs_chase", tc.thief_role_prefix, "chase")):
                if not all(ag in learner.agents for ag in env.possible_agents if ag.startswith(role)):
                    vs[key] = None       # the role is scripted: the learner has no policy for it
                    continue
                r = selfplay.evaluate_vs_scripted(env, learner, role, controller, n_episodes=a.eval_scripted, by_map=mixed)
                vs[key] = r if not mixed else {"overall": r[0], "maps": r[1]}
            extra["eval_vs_scripted"] = vs
        if rank == 0:
            u = max(agg["updates"], 1)
            print(json.dumps({
                "iteration": it, "n_gpus": world_size, "map": a.map, "worlds_per_gpu": a.worlds, "model": a.model,
                "parameters": learner.n_parameters(), "rollouts": a.rollouts, "lockstep_steps": steps,
                "rollout_agent_steps_per_s": a.worlds * world_size * len(env.possible_agents) * steps / max(learner.env_seconds - env_s0, 1e-9),
                "train_agent_steps_per_s": a.worlds * world_size * len(env.possible_agents) * steps / train_s,
                "gae_ms_per_update": agg["gae_ms"] / u, "ppo_ms_per_update": agg["update_ms"] / u,
                "allreduce_ms_per_update": agg["allreduce_ms"] / u,
                "eval_vs_archive": {"cop_trained": res_c, "thief_trained": res_t}, **extra}), flush=True)
    env.close()
    if world_size > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
