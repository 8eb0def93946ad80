#!/usr/bin/env python
"""Device renderer throughput on agh-map, against the bandwidth floor of the frame writes and the numpy renderer.

    python tools/prof_render.py [--reps 50]

For K in {1, 16, 256} frames, downsample d in {1, 2, 4}, rays off and on: one cat_render launch of K frames of
distinct worlds of a 16384-world environment, timed with CUDA events over --reps launches after warm-up.  Reports
frames/s, the frame-write rate in GB/s and the share of the write floor (frame bytes / 7.7 TB/s, the HGX B200 data
sheet's HBM3e bandwidth).  With rays the sensor report comes from one cat_env_observe of all 16384 worlds before the
timed launches (CatWorlds.sensor_rays); that observe is timed on its own, as is numpy's render_rgb per frame.  Prints
the card and its power limit first.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.maps import compile_map, load_named_map  # noqa: E402
from as_cops_and_thieves_b200.render import ray_directions, render_rgb  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or "unknown"
    except Exception:
        return "unknown"


def timed(fn, reps):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--worlds", type=int, default=16384)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    print(f"# {torch.cuda.get_device_name(dev)}, power limit {power_limit()}")
    N = a.worlds
    env = BatchedCopsThievesEnv(load_named_map("agh-map"), N, device=dev, seed=0)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(0)
    for _ in range(50):
        env.step(torch.randint(0, 4, (N, 3), device=dev, generator=g, dtype=torch.uint8))
    cw = env.worlds
    ren = cw.renderer()
    rays = cw.sensor_rays()
    t_obs = timed(cw.sensor_rays, a.reps)
    print(json.dumps({"what": "cat_env_observe (sensor_rays)", "worlds": N, "us": round(t_obs * 1e6, 1)}))
    for K in (1, 16, 256):
        ids = torch.randperm(N, device=dev, generator=g)[:K].contiguous()
        for d in (1, 2, 4):
            W, H = ren.frame_size(d)
            out = torch.empty((K, W, H, 3), dtype=torch.uint8, device=dev)
            for with_rays in (False, True):
                def go():
                    ren.render(cw.positions(), world=ids, map_of=cw.map_index, rays=rays if with_rays else None,
                               downsample=d, out=out)
                t = timed(go, a.reps)
                nbytes = out.numel()
                print(json.dumps({"K": K, "downsample": d, "rays": with_rays, "frame": [W, H], "us": round(t * 1e6, 2),
                                  "frames_per_s": round(K / t), "write_GB_s": round(nbytes / t / 1e9, 1),
                                  "share_of_write_floor": round(nbytes / HBM_BYTES_PER_S / t, 3)}))
    cmap = compile_map(load_named_map("agh-map"))
    pos = cw.get_state()["pos"][:4].cpu().numpy()
    dist, types = (x[:4].cpu().numpy() for x in rays)
    dirs = ray_directions(cw.R)
    for with_rays in (False, True):
        t0 = time.perf_counter()
        for w in range(4):
            render_rgb(cmap, pos[w], rays=(dist[w], types[w], dirs) if with_rays else None)
        t = (time.perf_counter() - t0) / 4
        print(json.dumps({"what": "numpy render_rgb per frame (one host core)", "rays": with_rays,
                          "ms": round(t * 1e3, 2)}))
    env.close()


if __name__ == "__main__":
    main()
