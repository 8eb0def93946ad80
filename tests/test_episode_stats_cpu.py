"""Episode statistics without a GPU: the numpy view of the totals against their C struct (whose layout test_abi.py checks
with every struct's), argument checks of cat_env_attach_episode_stats, the fp32 key encoding of the totals' minima and
maxima, the decoding and summary maths, and the all-reduce of the totals over a two-rank gloo group."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from as_cops_and_thieves_b200 import _lib, episodes

ROOT = Path(__file__).resolve().parents[1]
TOTALS_FIELDS = ("episodes", "captures", "timeouts", "length_sum", "length_min_key", "length_max_key", "return_sum",
                 "return_sq_sum", "return_min_key", "return_max_key")


def test_totals_dtype_matches_the_struct():
    T = _lib.CatEpisodeTotals
    assert C.sizeof(T) == 232 and C.alignment(T) == 8 and episodes.TOTALS_DTYPE.itemsize == 232
    assert all(episodes.TOTALS_DTYPE.fields[f][1] == getattr(T, f).offset for f in TOTALS_FIELDS)


def test_attach_checks_the_environment_first():
    assert "cat_env_attach_episode_stats" in _lib.EXPORTS
    L = _lib.load()
    io = _lib.CatEpisodeStatsIO()
    assert L.cat_env_attach_episode_stats(None, C.byref(io)) == -1
    assert b"null env" in L.cat_last_error()
    assert L.cat_env_attach_episode_stats(None, None) == -1


def test_return_key_round_trip_and_order():
    vals = np.array([0.0, -0.0, 1e-45, -1e-45, 1.17e-38, -1.17e-38, 3.4e38, -3.4e38, np.inf, -np.inf, -1.0, -0.3,
                     -29.75, 5.5, 1.0, 100.25], dtype=np.float32)
    keys = episodes.return_key(vals)
    assert keys.dtype == np.uint32
    assert np.all(keys != 0) and np.all(~keys != 0), "neither a key nor its complement may read as empty"
    back = episodes.key_value(keys)
    assert np.array_equal(back.view(np.uint32), vals.view(np.uint32)), "bit-exact round trip, signed zeros included"
    order = np.argsort(vals, kind="stable")
    srt = vals[order]
    ks = keys[order]
    for i in range(len(srt) - 1):
        if srt[i] < srt[i + 1]:
            assert ks[i] < ks[i + 1], (srt[i], srt[i + 1])
    assert episodes.return_key(np.float32(-0.0)) < episodes.return_key(np.float32(0.0))
    # the minimum is the complement under atomicMax
    assert episodes.key_value(~np.max(~keys)) == vals.min()
    assert episodes.key_value(np.max(keys)) == vals.max()


def _fold(tot, m, returns, length, captured):
    """What the kernel does for one episode ending in map slot m (sequentially)."""
    t = tot[m]
    t["episodes"] += 1
    t["captures" if captured else "timeouts"] += 1
    t["length_sum"] += length
    t["length_max_key"] = max(int(t["length_max_key"]), length)
    t["length_min_key"] = max(int(t["length_min_key"]), int(~np.uint32(length)))
    r = np.asarray(returns, np.float32)
    k = episodes.return_key(r)
    A = len(r)
    t["return_sum"][:A] += r.astype(np.float64)
    t["return_sq_sum"][:A] += r.astype(np.float64) ** 2
    t["return_max_key"][:A] = np.maximum(t["return_max_key"][:A], k)
    t["return_min_key"][:A] = np.maximum(t["return_min_key"][:A], ~k)


def _episodes_fixture():
    g = np.random.default_rng(3)
    eps = []
    for _ in range(57):
        m = int(g.integers(0, 3))
        r = g.normal(size=3).astype(np.float32) * 20
        eps.append((m if m != 2 else 0, r, int(g.integers(1, 400)), bool(g.integers(0, 2))))   # slot 2 stays empty
    tot = episodes.empty_totals(3)
    for m, r, n, c in eps:
        _fold(tot, m, r, n, c)
    return tot, eps


def _check_summary(s, eps, agents):
    assert s["episodes"] == len(eps)
    caps = sum(c for *_, c in eps)
    assert s["captures"] == caps and s["timeouts"] == len(eps) - caps
    assert s["capture_rate"] == pytest.approx(caps / len(eps))
    lens = np.array([n for _, _, n, _ in eps])
    assert s["length"]["min"] == lens.min() and s["length"]["max"] == lens.max()
    assert s["length"]["mean"] == pytest.approx(lens.mean())
    R = np.stack([r for _, r, _, _ in eps])
    for i, a in enumerate(agents):
        q = s["returns"][a]
        assert q["min"] == R[:, i].min() and q["max"] == R[:, i].max()
        assert q["mean"] == pytest.approx(R[:, i].astype(np.float64).mean(), rel=1e-12, abs=1e-12)
        assert q["std"] == pytest.approx(R[:, i].astype(np.float64).std(), rel=1e-9)


def test_summaries_of_hand_built_totals():
    agents = ["cop_0", "cop_1", "thief_0"]
    tot, eps = _episodes_fixture()
    _check_summary(episodes.summarize_maps(tot, agents), eps, agents)
    out = episodes.summarize_maps(tot, agents, ["squarinth", "agh-map", "labyrinth"], by_map=True)
    _check_summary(out["overall"], eps, agents)
    for m in range(2):
        assert out["maps"][m]["slot"] == m and out["maps"][m]["map"] == ["squarinth", "agh-map"][m]
        _check_summary(out["maps"][m], [e for e in eps if e[0] == m], agents)
    empty = out["maps"][2]
    assert empty["episodes"] == 0 and empty["capture_rate"] is None and empty["length"]["min"] is None
    assert empty["returns"]["thief_0"] == {"mean": None, "std": None, "min": None, "max": None}
    # merged slots: counts and sums add, keys take the maximum
    merged = episodes.merge_totals(tot)
    assert merged["episodes"] == tot["episodes"].sum()
    assert np.array_equal(merged["return_max_key"], tot["return_max_key"].max(axis=0))
    assert episodes.summarize(episodes.empty_totals(1)[0], agents)["episodes"] == 0


def _allreduce_worker(rank: int, world_size: int, port: int, tmp: str):
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        from as_cops_and_thieves_b200 import episodes as E
        tot, eps = _episodes_fixture()
        mine = [e for i, e in enumerate(eps) if i % world_size == rank]
        part = E.empty_totals(3)
        for m, r, n, c in mine:
            _fold(part, m, r, n, c)
        red = E.allreduce_totals(part, dist.group.WORLD)
        for f in ("episodes", "captures", "timeouts", "length_sum", "length_min_key", "length_max_key", "return_min_key",
                  "return_max_key"):
            assert np.array_equal(red[f], tot[f]), f
        assert np.allclose(red["return_sum"], tot["return_sum"], rtol=1e-12, atol=1e-9)
        assert np.allclose(red["return_sq_sum"], tot["return_sq_sum"], rtol=1e-12, atol=1e-9)
        Path(tmp, f"ok{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


def test_two_rank_allreduce_of_totals(tmp_path):
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_allreduce_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
