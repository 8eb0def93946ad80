#!/usr/bin/env python
"""Mixed-map step vs the same worlds as one environment per map.

    python tools/prof_multimap.py [--steps K] [--warmup W] [--counts 3277,16384] [--json FILE]

For each per-map count c, all five shipped maps with c worlds each:

* mixed  — one environment holding the 5 c worlds (cat_env_create_multi): one launch per step;
* split  — five single-map environments of c worlds, stepped back to back on one stream: five launches per step.

Both step the record output only (the bench.py headline's outputs).  Cold L2 as in bench.py: each side rotates over
enough independent world sets that their state, record and action buffers exceed 1.5 x the 126 MB L2, so every
timed step reads and writes HBM.  Exactly K steps are timed between one pair of CUDA events after W warm-up steps per
set.  The (cell, ray) lists are shared by every environment of a map on the device, so both sides read the same lists.
Prints the card and its power limit, then one JSON line per workload.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from as_cops_and_thieves_b200.maps import compile_map, load_named_map  # noqa: E402
from as_cops_and_thieves_b200.worlds import CatWorlds  # noqa: E402

MAPS = ("squarinth", "agh-map", "labyrinth", "lbirinth", "grandbyrinth")
L2_BYTES = 126e6


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or "unknown"
    except Exception:
        return "unknown"


def footprint(w: CatWorlds) -> int:
    return w.state.numel() + w._out.numel() + w.n_worlds * w.A


def make_sets(make, first):
    n_sets = max(2, int(-(-1.5 * L2_BYTES // footprint(first))))
    return [first] + [make(j) for j in range(1, n_sets)]


def time_steps(step_fns, K, W):
    n = len(step_fns)
    for i in range(W * n):
        step_fns[i % n]()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step_fns[i % n]()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / K     # us per step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--counts", default="3277,16384", help="worlds per map, one workload each")
    ap.add_argument("--json", default=None, help="also write the results to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_multimap.py needs a CUDA device")
    dev = torch.device("cuda:0")
    card = torch.cuda.get_device_name(dev)
    plim = power_limit()
    print(f"# card: {card}, power limit: {plim}")
    print("# cold L2: each side rotates over world sets whose buffers exceed 1.5 x 126 MB")
    cmaps = [compile_map(load_named_map(n), name=n) for n in MAPS]
    kw = dict(device=dev, seed=0, want_f32=False, want_shared=False)
    results = []
    for c in [int(v) for v in a.counts.split(",")]:
        counts = [c] * len(MAPS)
        N = sum(counts)
        g = torch.Generator(device=dev).manual_seed(0)
        acts = torch.randint(0, 4, (N, 3), dtype=torch.uint8, device=dev, generator=g)
        # mixed: world sets with disjoint global ids, one launch per step
        first = CatWorlds(cmaps, counts, gid0=0, **kw)
        mixed = make_sets(lambda j: CatWorlds(cmaps, counts, gid0=j * N, **kw), first)
        for w in mixed:
            w.reset()
        t_mixed = time_steps([lambda w=w: w.step(acts) for w in mixed], a.steps, a.warmup)
        info = first.info
        ray_list_bytes = int(info.ray_list_bytes)
        grid, wpc = int(info.grid), int(info.warps_per_cta)
        for w in mixed:
            w.close()
        del mixed, first
        # split: one environment per map, the same worlds (gid0 + offset), stepped back to back
        offs = [sum(counts[:m]) for m in range(len(MAPS))]
        acts_m = [acts[o:o + c].contiguous() for o in offs]
        firsts = [CatWorlds(cm, c, gid0=o, **kw) for cm, o in zip(cmaps, offs)]
        n_sets = max(2, int(-(-1.5 * L2_BYTES // sum(footprint(w) for w in firsts))))
        split = [firsts] + [[CatWorlds(cm, c, gid0=j * N + o, **kw) for cm, o in zip(cmaps, offs)] for j in range(1, n_sets)]
        for s in split:
            for w in s:
                w.reset()

        def step_set(s):
            for w, am in zip(s, acts_m):
                w.step(am)
        t_split = time_steps([lambda s=s: step_set(s) for s in split], a.steps, a.warmup)
        split_grids = [int(w.info.grid) for w in firsts]
        for s in split:
            for w in s:
                w.close()
        del split, firsts
        r = {"maps": list(MAPS), "worlds_per_map": c, "worlds": N, "steps_timed": a.steps,
             "mixed_us_per_step": round(t_mixed, 2), "mixed_agent_steps_per_s": 3 * N / (t_mixed * 1e-6),
             "split_us_per_step": round(t_split, 2), "split_agent_steps_per_s": 3 * N / (t_split * 1e-6),
             "mixed_over_split": round(t_mixed / t_split, 4), "mixed_grid": grid, "warps_per_cta": wpc,
             "split_grids": split_grids, "ray_list_bytes_all_maps": ray_list_bytes, "card": card, "power_limit": plim}
        results.append(r)
        print(json.dumps(r), flush=True)
    if a.json:
        Path(a.json).parent.mkdir(parents=True, exist_ok=True)
        Path(a.json).write_text(json.dumps(results, indent=1) + "\n")


if __name__ == "__main__":
    main()
