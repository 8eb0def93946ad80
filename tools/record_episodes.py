#!/usr/bin/env python
"""Record episodes of a batched environment and draw them on the GPU.

    python tools/record_episodes.py --map squarinth --worlds 4 --steps 200 --rays --out episodes/
    python tools/record_episodes.py --map squarinth,agh-map --worlds 8 --checkpoint policy.pt --downsample 2

Steps an environment of --worlds worlds (split over the maps of a comma-separated --map) for --steps steps, with the
greedy actions of a MAPPOLearner checkpoint or, without one, uniform random actions, and records every world with
render.TrajectoryRecorder.  Writes into --out:

* ``trajectory.npz`` — positions, maps, rewards, flags (and the rays with --rays); render.redraw draws any step of it
  on a host without a GPU;
* ``frames.npy`` — (steps, worlds, W, H, 3) uint8, the recorded steps drawn in one launch at --downsample;
* ``world_<k>.gif`` — one animation per world, when PIL is importable.

Prints whether the last recorded step equals a live render of the environment.
"""
import argparse
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.maps import load_named_map  # noqa: E402
from as_cops_and_thieves_b200.render import TrajectoryRecorder  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map", default="squarinth", help="built-in map, or a comma-separated list of them")
    ap.add_argument("--worlds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--checkpoint", default=None, help="MAPPOLearner.save file: greedy actions (default: random)")
    ap.add_argument("--downsample", type=int, default=1)
    ap.add_argument("--rays", action="store_true", help="record the sensors and draw their rays")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="episodes")
    a = ap.parse_args()

    dev = torch.device("cuda:0")
    maps = [load_named_map(n.strip()) for n in a.map.split(",") if n.strip()]
    env = BatchedCopsThievesEnv(maps[0] if len(maps) == 1 else maps, a.worlds, device=dev, seed=a.seed)
    learner = None
    if a.checkpoint:
        from as_cops_and_thieves_b200.mappo import MAPPOLearner
        learner = MAPPOLearner(env)
        learner.load(a.checkpoint)
    obs, _ = env.reset()
    rec = TrajectoryRecorder(env, range(env.num_envs), a.steps, rays=a.rays)
    gen = torch.Generator(device=dev).manual_seed(a.seed)
    for _ in range(a.steps):
        if learner is not None:
            acts = learner.act(obs, greedy=True)
            obs, _, term, trunc, _ = env.step(acts)
            learner.note_done(term[env.possible_agents[0]] | trunc[env.possible_agents[0]])
        else:
            obs, *_ = env.step(torch.randint(0, 4, (env.num_envs, env.num_agents), device=dev, generator=gen,
                                             dtype=torch.uint8))
        rec.record()
    frames = rec.frames(downsample=a.downsample)
    live = env.render_frames(rays=a.rays, downsample=a.downsample)
    same = bool(torch.equal(frames[-1], live))

    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    rec.save(out / "trajectory.npz")
    frames = frames.cpu().numpy()
    np.save(out / "frames.npy", frames)
    gifs = 0
    try:
        from PIL import Image
    except ImportError:
        Image = None
    if Image is not None:
        for k in range(frames.shape[1]):
            imgs = [Image.fromarray(np.ascontiguousarray(frames[t, k].transpose(1, 0, 2))) for t in range(frames.shape[0])]
            imgs[0].save(out / f"world_{k}.gif", save_all=True, append_images=imgs[1:], duration=40, loop=0)
            gifs += 1
    print(f"recorded {a.steps} steps of {env.num_envs} worlds on {','.join(env.map_names)}: frames {frames.shape} "
          f"in {out}, {gifs} GIFs{'' if Image is not None else ' (PIL not importable)'}; "
          f"last step equals a live render: {same}")
    env.close()
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
