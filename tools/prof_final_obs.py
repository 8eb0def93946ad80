#!/usr/bin/env python
"""Cost of final observations: the step with and without final outputs, and the learner's rollout with and without
time-limit bootstrapping.

    python tools/prof_final_obs.py [--worlds 16384] [--steps 200] [--rounds 3]

Step: agh-map x --worlds with BatchedCopsThievesEnv's outputs (record + obs_f32 + state_f32 + critic_f32), final
outputs off vs on, at max_step_count 400 and 50.  Each world's step counter starts at a random point of its episode, so
worlds end (time out) at a steady rate of about 1 / max_step_count per step plus the captures.  Cold L2: every variant
owns two environments whose outputs together exceed the 126 MB L2, and the timed steps alternate between them; --steps
steps are timed back to back with one CUDA-event pair.  Off and on alternate --rounds times; the median is reported with
every round.  The share of worlds that end per step is counted in a separate untimed run.

Rollout: MAPPOLearner (LSTM models, CUDA-graph rollout) on the same map and world count, bootstrap off vs on, one
rollout of 64 steps per timing, alternating --rounds times; agent-steps/s = 64 x worlds x 3 agents / rollout time.

Prints the card and its power limit first; one JSON line per result.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner  # noqa: E402
from as_cops_and_thieves_b200.maps import load_named_map  # noqa: E402


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or "unknown"
    except Exception:
        return "unknown"


def make_envs(m, N, msc, final, dev):
    envs = []
    for i in range(2):
        e = BatchedCopsThievesEnv(m, N, device=dev, seed=i, gid0=i * N, max_step_count=msc, final_observations=final)
        e.reset()
        g = torch.Generator().manual_seed(100 + i)
        e.worlds.set_state(step_count=torch.randint(0, msc, (N,), generator=g, dtype=torch.int32))
        envs.append(e)
    return envs


def step_times(m, N, msc, steps, rounds, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    acts = [torch.randint(0, 4, (N, 3), device=dev, generator=g, dtype=torch.uint8) for _ in range(16)]
    variants = {False: make_envs(m, N, msc, False, dev), True: make_envs(m, N, msc, True, dev)}
    for envs in variants.values():            # warm-up, and the untimed count of worlds that end per step
        ended = torch.zeros((), dtype=torch.int64, device=dev)
        for t in range(max(steps, 2 * msc)):
            e = envs[t % 2]
            e.step(acts[t % 16])
            ended += e.worlds.terminated.sum()
        frac = float(ended) / (max(steps, 2 * msc) * N)
    times = {False: [], True: []}
    for _ in range(rounds):
        for final, envs in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for t in range(steps):
                envs[t % 2].step(acts[t % 16])
            e1.record()
            e1.synchronize()
            times[final].append(e0.elapsed_time(e1) * 1e3 / steps)
    for envs in variants.values():
        for e in envs:
            e.close()
    return times, frac


def rollout_rates(m, N, rounds, dev):
    learners = {}
    for boot in (False, True):
        env = BatchedCopsThievesEnv(m, N, device=dev, seed=0, final_observations=boot)
        cfg = MAPPOConfig(rollouts=64, model="lstm", random_timesteps=0, learning_starts=0, time_limit_bootstrap=boot,
                          opponent_freeze_duration=0, policy_freeze_duration=0)
        lrn = MAPPOLearner(env, cfg, seed=0)
        lrn.collect()                          # eager warm-up
        lrn.collect()                          # capture + first replay
        learners[boot] = lrn
    rates = {False: [], True: []}
    for _ in range(rounds):
        for boot, lrn in learners.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            lrn.collect()                      # ends in a device synchronise
            rates[boot].append(64 * N * 3 / (time.perf_counter() - t0))
    return rates


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-rollout", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_final_obs.py measures the GPU step: no CUDA device is visible")
    dev = torch.device("cuda:0")
    print(f"# {torch.cuda.get_device_name(dev)}, power limit {power_limit()}")
    m = load_named_map("agh-map")
    for msc in (400, 50):
        times, frac = step_times(m, a.worlds, msc, a.steps, a.rounds, dev)
        off, on = statistics.median(times[False]), statistics.median(times[True])
        print(json.dumps({"what": "step, BatchedCopsThievesEnv outputs", "map": "agh-map", "worlds": a.worlds,
                          "max_step_count": msc, "ended_per_step": round(frac, 4), "us_final_off": round(off, 2),
                          "us_final_on": round(on, 2), "cost": f"{(on / off - 1) * 100:+.2f} %",
                          "rounds_off": [round(x, 2) for x in times[False]], "rounds_on": [round(x, 2) for x in times[True]]}))
    if not a.no_rollout:
        rates = rollout_rates(m, a.worlds, a.rounds, dev)
        off, on = statistics.median(rates[False]), statistics.median(rates[True])
        print(json.dumps({"what": "MAPPO rollout (lstm, CUDA graph, 64 steps)", "map": "agh-map", "worlds": a.worlds,
                          "agent_steps_per_s_bootstrap_off": round(off), "agent_steps_per_s_bootstrap_on": round(on),
                          "cost": f"{(off / on - 1) * 100:+.2f} % time",
                          "rounds_off": [round(x) for x in rates[False]], "rounds_on": [round(x) for x in rates[True]]}))


if __name__ == "__main__":
    main()
