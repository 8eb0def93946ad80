"""Measure map swapping on the GPU: the device vs the host (cell, ray) list builder, cat_env_set_map latency, and the
step time of swappable vs plain environments (which run the mixed-map kernels and stage a blob of the default
capacity).  Writes a plain-text report (default profiles/map_swap_b200.txt) headed by the card and its power limit.

    python tools/prof_map_swap.py [--out FILE] [--rounds 3] [--steps 300]
"""
from __future__ import annotations

import argparse
import ctypes as C
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import parity_utils as pu  # noqa: E402
from as_cops_and_thieves_b200 import _lib  # noqa: E402
from as_cops_and_thieves_b200.maps import SHIPPED_MAPS, compile_map, generate_maze  # noqa: E402
from as_cops_and_thieves_b200.params import EnvParams  # noqa: E402
from as_cops_and_thieves_b200.worlds import CatWorlds, _map_desc  # noqa: E402


def card() -> str:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def list_build_times(cmap, reps=3):
    """(host s, device s, MB): one call of each builder with preallocated output buffers (the device call includes its
    own sizing passes and the upload of the map)."""
    L = _lib.load()
    p = EnvParams()
    md, keep = _map_desc(cmap)
    grid = (C.c_double * 5)()
    ns, no = C.c_int64(0), C.c_int64(0)
    args = (C.byref(md), p.n_rays, p.ray_length, p.wall_radius + p.ray_radius, 0.0, C.byref(grid))
    _lib.check(L.cat_ray_lists_host(*args, None, C.byref(ns), None, C.byref(no)), "size")
    hs, ho = np.zeros(ns.value, np.uint32), np.zeros(no.value, np.uint32)
    ds = torch.zeros(ns.value, dtype=torch.int32, device="cuda")
    do = torch.zeros(no.value, dtype=torch.int32, device="cuda")
    th, td = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        _lib.check(L.cat_ray_lists_host(*args, _lib.np_ptr(hs), C.byref(ns), _lib.np_ptr(ho), C.byref(no)), "host")
        th.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _lib.check(L.cat_ray_lists_device(*args, ds.data_ptr(), C.byref(ns), do.data_ptr(), C.byref(no), 0), "device")
        td.append(time.perf_counter() - t0)      # the call synchronises the device before it returns
    same = np.array_equal(hs, ds.cpu().numpy().view(np.uint32)) and np.array_equal(ho, do.cpu().numpy().view(np.uint32))
    return min(th), min(td), (ns.value + no.value) * 4 / 1e6, same


def us_per_step(w: CatWorlds, steps: int) -> float:
    g = torch.Generator().manual_seed(0)
    acts = [torch.randint(0, 4, (w.n_worlds, w.A), dtype=torch.uint8, generator=g).cuda() for _ in range(8)]
    w.reset()
    for i in range(20):
        w.step(acts[i % 8])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        w.step(acts[i % 8])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "map_swap_b200.txt"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_map_swap.py needs a CUDA device")
    lines = [f"# map swapping, measured on {card()} (name, power limit, max SM clock)", ""]

    lines.append("## (cell, ray) list build, automatic cells, 90 rays: host reference (16 threads max) vs device builder")
    maps = {n: pu.named_cmap(n) for n in SHIPPED_MAPS}
    maps.update({f"maze-{s}": compile_map(generate_maze(s)) for s in (0, 1)})
    for name, cm in maps.items():
        th, td, mb, same = list_build_times(cm)
        lines.append(f"{name:14s} {cm.n_edges:5d} edges  {mb:7.1f} MB  host {th * 1e3:8.1f} ms  device {td * 1e3:7.1f} ms"
                     f"  identical={same}")
    lines.append("")

    lines.append("## cat_env_set_map latency (squarinth x 4096, swappable; alternating two mazes; incl. the masked reset)")
    sw = CatWorlds(maps["squarinth"], 4096, swappable_maps=True)
    mz = [maps["maze-0"], maps["maze-1"]]
    sw.set_map(0, mz[1])
    ts = []
    for i in range(10):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sw.set_map(0, mz[i % 2])
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    lines.append(f"median {ts[len(ts) // 2] * 1e3:.2f} ms, min {ts[0] * 1e3:.2f} ms, max {ts[-1] * 1e3:.2f} ms "
                 f"(the maze lists are cached after the first two swaps)")
    sw.close()
    lines.append("")

    lines.append(f"## us per step, plain vs swappable, {args.steps} steps, CUDA events, alternated over {args.rounds} rounds")
    cases = {"agh-map x 16384": ([maps["agh-map"]], [16384]), "squarinth x 4096": ([maps["squarinth"]], [4096]),
             "3 maps x 4096": ([maps["squarinth"], maps["agh-map"], maps["labyrinth"]], [4096] * 3)}
    for name, (cms, counts) in cases.items():
        res = {"plain": [], "swappable": []}
        envs = {}
        for kind in res:
            arg = cms[0] if len(cms) == 1 else cms
            n = counts[0] if len(cms) == 1 else counts
            envs[kind] = CatWorlds(arg, n, swappable_maps=kind == "swappable")
        for _ in range(args.rounds):
            for kind in res:
                res[kind].append(us_per_step(envs[kind], args.steps))
        blob = {k: (e.info.map_blob_bytes, e.info.smem_bytes_per_cta, e.info.warps_per_cta, e.info.grid)
                for k, e in envs.items()}
        for kind, v in res.items():
            lines.append(f"{name:18s} {kind:9s} " + " ".join(f"{x:7.1f}" for x in v) +
                         f"   blob / smem per CTA / warps / grid = {blob[kind]}")
        for e in envs.values():
            e.close()
    lines.append("")
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
