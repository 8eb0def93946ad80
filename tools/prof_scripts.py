#!/usr/bin/env python
"""Cost of scripted agents: the step without scripts, with scripts attached and every mode 0, and with the thief
evading and both cops chasing.

    python tools/prof_scripts.py [--worlds 16384] [--steps 1000] [--rounds 3] [--out FILE]

agh-map x --worlds with BatchedCopsThievesEnv's outputs (record + obs_f32 + state_f32 + critic_f32) at max_step_count
400.  Each world's step counter starts at a random point of its episode, so worlds end at a steady rate.  Every variant
with scripts attached writes the controllers' decisions at every emitted observation; the "scripted" variant also
acts on them, so its episodes (and so its re-spawns) differ from the others': the worlds that end per step are reported
with the times.  Cold L2: every variant owns two environments whose outputs
together exceed the 126 MB L2, and the timed steps alternate between them; --steps steps are timed back to back with
one CUDA-event pair.  The variants alternate --rounds times; the median is reported with every round.

Prints the card and its power limit first; one JSON line per result.
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.maps import load_named_map  # noqa: E402

VARIANTS = ("none", "attached", "scripted")
SCRIPTED = {"none": None, "attached": {}, "scripted": {"cop_0": "chase", "cop_1": "chase", "thief_0": "evade"}}


def card() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or torch.cuda.get_device_name()
    except Exception:
        return torch.cuda.get_device_name()


def make_envs(m, N, msc, variant, dev):
    envs = []
    for i in range(2):
        e = BatchedCopsThievesEnv(m, N, device=dev, seed=i, gid0=i * N, max_step_count=msc, scripted=SCRIPTED[variant])
        e.reset()
        g = torch.Generator().manual_seed(100 + i)
        e.worlds.set_state(step_count=torch.randint(0, msc, (N,), generator=g, dtype=torch.int32))
        envs.append(e)
    return envs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--max-step-count", type=int, default=400)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_scripts.py needs a CUDA device")
    dev = torch.device("cuda:0")
    lines = [f"# {card()}"]
    print(lines[0], flush=True)
    m, N, msc = load_named_map("agh-map"), a.worlds, a.max_step_count
    g = torch.Generator(device=dev).manual_seed(0)
    acts = [torch.randint(0, 4, (N, 3), device=dev, generator=g, dtype=torch.uint8) for _ in range(16)]
    variants = {v: make_envs(m, N, msc, v, dev) for v in VARIANTS}
    ended = {}
    for v, envs in variants.items():          # warm-up, and the untimed count of worlds that end per step
        n = torch.zeros((), dtype=torch.int64, device=dev)
        for t in range(2 * msc):
            e = envs[t % 2]
            e.step(acts[t % 16])
            n += e.worlds.terminated.sum()
        ended[v] = float(n) / (2 * msc * N)
    times = {v: [] for v in VARIANTS}
    for _ in range(a.rounds):
        for v, envs in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for t in range(a.steps):
                envs[t % 2].step(acts[t % 16])
            e1.record()
            e1.synchronize()
            times[v].append(round(e0.elapsed_time(e1) * 1e3 / a.steps, 2))
    med = {v: statistics.median(t) for v, t in times.items()}
    res = {"what": "step, BatchedCopsThievesEnv outputs", "map": "agh-map", "worlds": N, "max_step_count": msc,
           "ended_per_step": {v: round(x, 4) for v, x in ended.items()}}
    for v in VARIANTS:
        res[f"us_{v}"] = med[v]
    res["cost_attached"] = f"{(med['attached'] / med['none'] - 1) * 100:+.2f} %"
    res["cost_scripted"] = f"{(med['scripted'] / med['none'] - 1) * 100:+.2f} %"
    for v in VARIANTS:
        res[f"rounds_{v}"] = times[v]
    lines.append(json.dumps(res))
    print(lines[-1], flush=True)
    for envs in variants.values():
        for e in envs:
            e.close()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
