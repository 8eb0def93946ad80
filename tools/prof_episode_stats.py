#!/usr/bin/env python
"""Cost of episode statistics: the step without them, with them (kept by the step kernel), and without them plus the
same tally done with torch ops after every step; and the host path without and with them.

    python tools/prof_episode_stats.py [--worlds 16384] [--steps 200] [--rounds 3] [--host-worlds 4096]

Step: agh-map x --worlds with BatchedCopsThievesEnv's outputs (record + obs_f32 + state_f32 + critic_f32), at
max_step_count 400 and 50.  Each world's step counter starts at a random point of its episode, so worlds end at a
steady rate of about 1 / max_step_count per step plus the captures.  The torch variant adds, after each step: acc +=
reward; length += 1; the return and length of the ended worlds (torch.where); zeroing both for them; and the episode
count and return sum (the per-world half of what the kernel does, plus two sums instead of per-map atomics).  Cold L2:
every variant owns two environments whose outputs together exceed the 126 MB L2, and the timed steps alternate between
them; --steps steps are timed back to back with one CUDA-event pair.  The variants alternate --rounds times; the median
is reported with every round.

Host path: CatWorlds.step_host("pipelined") on squarinth x --host-worlds (actions in pinned memory in, packed records
in pinned memory out, one device synchronise per call), statistics off vs on, timed by the host clock over --steps
calls per round.  With statistics attached the chunks run the full-output kernel instead of the record-only one.

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
sys.path.insert(0, str(ROOT / "tests"))
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv  # noqa: E402
from as_cops_and_thieves_b200.maps import load_named_map  # noqa: E402
from as_cops_and_thieves_b200.worlds import CatWorlds  # noqa: E402

VARIANTS = ("off", "on", "torch")


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or "unknown"
    except Exception:
        return "unknown"


class TorchTally:
    """What a tracker outside the kernel does after each step, with torch ops."""

    def __init__(self, env):
        N, A, dev = env.num_envs, env.num_agents, env.device
        w = env.worlds
        self.reward, self.done = w.reward, w.terminated.view(torch.bool)
        self.acc = torch.zeros((N, A), dtype=torch.float32, device=dev)
        self.length = torch.zeros(N, dtype=torch.int32, device=dev)
        self.ret = torch.zeros((N, A), dtype=torch.float32, device=dev)
        self.len_out = torch.zeros(N, dtype=torch.int32, device=dev)
        self.episodes = torch.zeros((), dtype=torch.int64, device=dev)
        self.ret_sum = torch.zeros(A, dtype=torch.float64, device=dev)

    def __call__(self):
        d = self.done
        self.acc.add_(self.reward)
        self.length.add_(1)
        torch.where(d.unsqueeze(1), self.acc, self.ret, out=self.ret)
        torch.where(d, self.length, self.len_out, out=self.len_out)
        self.episodes.add_(d.sum())
        self.ret_sum.add_((self.acc * d.unsqueeze(1)).sum(0))
        self.acc.masked_fill_(d.unsqueeze(1), 0.0)
        self.length.masked_fill_(d, 0)


def make_envs(m, N, msc, variant, dev):
    envs = []
    for i in range(2):
        e = BatchedCopsThievesEnv(m, N, device=dev, seed=i, gid0=i * N, max_step_count=msc,
                                  episode_statistics=variant == "on")
        e.reset()
        g = torch.Generator().manual_seed(100 + i)
        e.worlds.set_state(step_count=torch.randint(0, msc, (N,), generator=g, dtype=torch.int32))
        e.tally = TorchTally(e) if variant == "torch" else None
        envs.append(e)
    return envs


def step(e, acts):
    e.step(acts)
    if e.tally is not None:
        e.tally()


def step_times(m, N, msc, steps, rounds, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    acts = [torch.randint(0, 4, (N, 3), device=dev, generator=g, dtype=torch.uint8) for _ in range(16)]
    variants = {v: make_envs(m, N, msc, v, dev) for v in VARIANTS}
    for envs in variants.values():            # warm-up, and the untimed count of worlds that end per step
        ended = torch.zeros((), dtype=torch.int64, device=dev)
        for t in range(max(steps, 2 * msc)):
            e = envs[t % 2]
            step(e, acts[t % 16])
            ended += e.worlds.terminated.sum()
        frac = float(ended) / (max(steps, 2 * msc) * N)
    times = {v: [] for v in VARIANTS}
    for _ in range(rounds):
        for v, envs in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for t in range(steps):
                step(envs[t % 2], acts[t % 16])
            e1.record()
            e1.synchronize()
            times[v].append(e0.elapsed_time(e1) * 1e3 / steps)
    on = variants["on"][0].episode_statistics()
    for envs in variants.values():
        for e in envs:
            e.close()
    return times, frac, on


def host_times(N, steps, rounds, dev):
    import parity_utils as pu
    cmap = pu.named_cmap("squarinth", free_spawn=True)
    envs = {v: CatWorlds(cmap, N, device=dev, seed=1, want_episode_stats=v == "on") for v in ("off", "on")}
    g = torch.Generator().manual_seed(0)
    acts = [torch.randint(0, 4, (N, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(16)]
    for e in envs.values():
        e.reset()
        for t in range(20):
            e.step_host(acts[t % 16], mode="pipelined")
    times = {v: [] for v in envs}
    for _ in range(rounds):
        for v, e in envs.items():
            t0 = time.perf_counter()
            for t in range(steps):
                e.step_host(acts[t % 16], mode="pipelined")      # ends in a stream synchronise
            times[v].append((time.perf_counter() - t0) * 1e6 / steps)
    for e in envs.values():
        e.close()
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=16384)
    ap.add_argument("--host-worlds", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_episode_stats.py measures the GPU step: no CUDA device is visible")
    dev = torch.device("cuda:0")
    print(f"# {torch.cuda.get_device_name(dev)}, power limit, max SM clock: {power_limit()}")
    m = load_named_map("agh-map")
    for msc in (400, 50):
        times, frac, on = step_times(m, a.worlds, msc, a.steps, a.rounds, dev)
        med = {v: statistics.median(times[v]) for v in VARIANTS}
        print(json.dumps({"what": "step, BatchedCopsThievesEnv outputs", "map": "agh-map", "worlds": a.worlds,
                          "max_step_count": msc, "ended_per_step": round(frac, 4),
                          **{f"us_{v}": round(med[v], 2) for v in VARIANTS},
                          "cost_kernel": f"{(med['on'] / med['off'] - 1) * 100:+.2f} %",
                          "cost_torch_ops": f"{(med['torch'] / med['off'] - 1) * 100:+.2f} %",
                          **{f"rounds_{v}": [round(x, 2) for x in times[v]] for v in VARIANTS},
                          "episodes_counted": on["episodes"], "capture_rate": on["capture_rate"]}))
    ht = host_times(a.host_worlds, a.steps, a.rounds, dev)
    off, on = statistics.median(ht["off"]), statistics.median(ht["on"])
    print(json.dumps({"what": "step_host pipelined, packed records", "map": "squarinth", "worlds": a.host_worlds,
                      "us_off": round(off, 2), "us_on": round(on, 2), "cost": f"{(on / off - 1) * 100:+.2f} %",
                      "rounds_off": [round(x, 2) for x in ht["off"]], "rounds_on": [round(x, 2) for x in ht["on"]]}))


if __name__ == "__main__":
    main()
