"""Episode statistics the step kernel accumulates (``include/cat_b200.h`` ``CatEpisodeTotals``): decoding and summaries.

The kernel adds every episode that ends to its map slot's totals with atomics only: counts and sums by ``atomicAdd``,
minima and maxima as u32 keys under ``atomicMax`` (the maximum as an order-preserving key of the value, the minimum as
the key's complement, 0 = no episode).  Everything here runs on the host and needs no GPU: ``CatWorlds.episode_totals``
copies the buffer over once and hands it to these functions.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from ._lib import CAT_MAX_AGENTS, CatEpisodeTotals

#: numpy mirror of ``CatEpisodeTotals`` (one record per map slot); a zero-filled array is the empty state
TOTALS_DTYPE = np.dtype(CatEpisodeTotals)
_SUM_FIELDS = ("episodes", "captures", "timeouts", "length_sum", "return_sum", "return_sq_sum")
_KEY_FIELDS = ("length_min_key", "length_max_key", "return_min_key", "return_max_key")


def empty_totals(n_maps: int) -> np.ndarray:
    return np.zeros(n_maps, dtype=TOTALS_DTYPE)


def return_key(values) -> np.ndarray:
    """The kernel's u32 key of fp32 values: sign bit clear -> bits | 0x80000000, set -> ~bits (order-preserving, and
    neither the key nor its complement is 0 for a non-NaN value)."""
    b = np.asarray(values, dtype=np.float32).view(np.uint32)
    return np.where(b & np.uint32(0x80000000), ~b, b | np.uint32(0x80000000)).astype(np.uint32)


def key_value(keys) -> np.ndarray:
    """Inverse of ``return_key``: u32 keys -> float32 values."""
    k = np.asarray(keys, dtype=np.uint32)
    return np.where(k & np.uint32(0x80000000), k & np.uint32(0x7FFFFFFF), ~k).astype(np.uint32).view(np.float32)


def merge_totals(totals: np.ndarray) -> np.ndarray:
    """Several map slots (or ranks) folded into one record: counts and sums add, keys take their maximum."""
    t = np.atleast_1d(totals)
    out = empty_totals(1)
    for f in _SUM_FIELDS:
        out[f] = t[f].sum(axis=0)
    for f in _KEY_FIELDS:
        out[f] = t[f].max(axis=0) if len(t) else 0
    return out[0]


def summarize(rec: np.void, agents: Sequence[str]) -> Dict:
    """One ``CatEpisodeTotals`` record -> episodes, captures, timeouts, capture rate, length mean / min / max and per
    agent the return's mean / std (population) / min / max.  Without episodes the rates and moments are None."""
    n = int(rec["episodes"])
    out: Dict = {"episodes": n, "captures": int(rec["captures"]), "timeouts": int(rec["timeouts"])}
    if n == 0:
        out.update(capture_rate=None, length={"mean": None, "min": None, "max": None},
                   returns={a: {"mean": None, "std": None, "min": None, "max": None} for a in agents})
        return out
    out["capture_rate"] = out["captures"] / n
    out["length"] = {"mean": int(rec["length_sum"]) / n, "min": int(~np.uint32(rec["length_min_key"])),
                     "max": int(rec["length_max_key"])}
    rmin = key_value(~rec["return_min_key"].astype(np.uint32))
    rmax = key_value(rec["return_max_key"])
    returns = {}
    for i, a in enumerate(agents):
        mean = float(rec["return_sum"][i]) / n
        var = max(float(rec["return_sq_sum"][i]) / n - mean * mean, 0.0)
        returns[a] = {"mean": mean, "std": var ** 0.5, "min": float(rmin[i]), "max": float(rmax[i])}
    out["returns"] = returns
    return out


def summarize_maps(totals: np.ndarray, agents: Sequence[str], map_names: Optional[Sequence[str]] = None,
                   by_map: bool = False) -> Dict:
    """Every slot merged (``by_map=False``), or ``{"overall": ..., "maps": [per slot, with "slot" and "map"]}``."""
    overall = summarize(merge_totals(totals), agents)
    if not by_map:
        return overall
    maps: List[Dict] = []
    for m in range(len(totals)):
        name = map_names[m] if map_names is not None else str(m)
        maps.append({"slot": m, "map": name, **summarize(totals[m], agents)})
    return {"overall": overall, "maps": maps}


def allreduce_totals(totals: np.ndarray, group=None) -> np.ndarray:
    """Totals of every rank of ``group`` (``torch.distributed``): sums for counts and sums, maxima for keys.  The
    tensors go to the current CUDA device for an NCCL group and stay on the host otherwise."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = np.array(totals, dtype=TOTALS_DTYPE, copy=True)
    M = len(t)
    counts = torch.from_numpy(np.stack([t[f].astype(np.int64) for f in ("episodes", "captures", "timeouts", "length_sum")], 1)).to(dev)
    sums = torch.from_numpy(np.stack([t["return_sum"], t["return_sq_sum"]], 1).astype(np.float64)).to(dev)
    keys = torch.from_numpy(np.concatenate([t["length_min_key"].reshape(M, 1), t["length_max_key"].reshape(M, 1),
                                            t["return_min_key"], t["return_max_key"]], 1).astype(np.int64)).to(dev)
    dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(keys, op=dist.ReduceOp.MAX, group=group)
    counts, sums, keys = counts.cpu().numpy(), sums.cpu().numpy(), keys.cpu().numpy()
    for i, f in enumerate(("episodes", "captures", "timeouts", "length_sum")):
        t[f] = counts[:, i].astype(np.uint64)
    t["return_sum"], t["return_sq_sum"] = sums[:, 0], sums[:, 1]
    t["length_min_key"], t["length_max_key"] = keys[:, 0], keys[:, 1]
    t["return_min_key"] = keys[:, 2:2 + CAT_MAX_AGENTS]
    t["return_max_key"] = keys[:, 2 + CAT_MAX_AGENTS:]
    return t
