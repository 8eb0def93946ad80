"""The GAE reference (tests/gae_reference.py) against the fp64 C oracle and a plain Python loop, and the argument checks
of cat_gae / cat_adv_normalize that return before any CUDA call.  Runs without a device."""
import ctypes as C

import numpy as np
import pytest

import gae_reference as gr
from as_cops_and_thieves_b200 import _lib
from oracle import cat_oracle as co

CAT_ERR_INVALID = -1


def _case(T, M, pattern, seed):
    rng = np.random.default_rng(seed)
    r = rng.standard_normal((T, M)).astype(np.float32)
    v = rng.standard_normal((T, M)).astype(np.float32)
    lv = rng.standard_normal(M).astype(np.float32)
    d = gr.done_mask(pattern, T, M, rng)
    return r, d, v, lv


def _python_loop(r, d, v, lv, gamma, lam):
    T, M = r.shape
    adv = np.zeros((T, M))
    for m in range(M):
        a = 0.0
        for t in reversed(range(T)):
            nv = float(lv[m]) if t == T - 1 else float(v[t + 1, m])
            a = float(r[t, m]) - float(v[t, m]) + gamma * (0.0 if d[t, m] else 1.0) * (nv + lam * a)
            adv[t, m] = a
    return adv


@pytest.mark.parametrize("pattern", gr.DONE_PATTERNS)
@pytest.mark.parametrize("T,M", [(1, 3), (8, 5), (33, 4), (97, 2)])
def test_reference_matches_oracle_and_python_loop(T, M, pattern):
    r, d, v, lv = _case(T, M, pattern, seed=T * 100 + M)
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.99, 0.0), (0.0, 0.95)):
        adv, ret = gr.gae_fp64(r, d, v, lv, gamma, lam)
        assert adv.dtype == np.float64 and ret.dtype == np.float64
        # the oracle runs the same fp64 operations in the same order (built with -ffp-contract=off)
        oret, oadv = co.gae(r, d, v, lv, gamma, lam, normalize=False)
        np.testing.assert_array_equal(adv.astype(np.float32), oadv)
        np.testing.assert_array_equal(ret.astype(np.float32), oret)
        np.testing.assert_array_equal(adv, _python_loop(r, d, v, lv, gamma, lam))
        np.testing.assert_array_equal(ret, adv + v.astype(np.float64))
        S = gr.gae_abs_bound(r, d, v, lv, gamma, lam)
        assert np.all(S >= np.abs(adv))
        if gamma == 0.0 or pattern == "all":
            np.testing.assert_array_equal(adv, r.astype(np.float64) - v)


def test_reference_runs_on_torch_tensors():
    torch = pytest.importorskip("torch")
    r, d, v, lv = _case(40, 6, "random8", seed=1)
    adv, ret = gr.gae_fp64(r, d, v, lv, 0.99, 0.95)
    tadv, tret = gr.gae_fp64(torch.from_numpy(r), torch.from_numpy(d), torch.from_numpy(v), torch.from_numpy(lv), 0.99, 0.95)
    assert tadv.dtype == torch.float64
    np.testing.assert_array_equal(tadv.numpy(), adv)
    np.testing.assert_array_equal(tret.numpy(), ret)
    S = gr.gae_abs_bound(r, d, v, lv, 0.99, 0.95)
    np.testing.assert_array_equal(gr.gae_abs_bound(torch.from_numpy(r), torch.from_numpy(d), torch.from_numpy(v),
                                                   torch.from_numpy(lv), 0.99, 0.95).numpy(), S)


def test_done_masks_sit_on_the_seams():
    rng = np.random.default_rng(0)
    T = 96                                   # a multiple of 32: every seam is where its name says
    t = np.arange(T)
    assert np.array_equal(np.flatnonzero(gr.done_mask("t%8==7", T, 1, rng)[:, 0]), t[t % 8 == 7])
    assert np.array_equal(np.flatnonzero(gr.done_mask("t%32==0", T, 1, rng)[:, 0]), t[t % 32 == 0])
    m = gr.done_mask("t%32==31", 97, 1, rng)[:, 0]   # chunks end at t = 96, 64, 32, 0 when T = 97
    assert set(np.flatnonzero(m)) == {31, 63, 95, 96, 64, 32, 0}
    assert gr.done_mask("all", 5, 2, rng).all() and not gr.done_mask("none", 5, 2, rng).any()


def test_normalize_exact_follows_the_formula():
    rng = np.random.default_rng(2)
    a = rng.standard_normal(1000).astype(np.float32)
    a64 = a.astype(np.float64)
    s, q, n = float(a64.sum()), float((a64 * a64).sum()), a.size
    got = gr.normalize_exact(a, s, q, n)
    want = (a64 - a64.mean()) / (a64.std(ddof=1) + 1e-8)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
    fm, inv = gr.normalize_params(s, q, n)
    assert fm.dtype == np.float32 and inv.dtype == np.float32
    assert np.array_equal(got, (a - fm) * inv) and got.dtype == np.float32
    # count == 1 and sumsq below count·mean²: the variance is 0, so 1/(0 + 1e-8)
    assert gr.normalize_params(3.0, 9.0, 1)[1] == np.float32(1e8)
    assert gr.normalize_params(10.0, 1.0, 10)[1] == np.float32(1e8)
    # the fused multiply-add: sumsq - count·mean² rounded once
    assert gr._fma(1.0 + 2.0 ** -30, 1.0 + 2.0 ** -30, -1.0) == 2.0 ** -29 + 2.0 ** -60


def test_gae_entry_points_reject_bad_sizes_before_any_cuda_call():
    """Non-null placeholder pointers: the checks come before the launch, so nothing is dereferenced."""
    L = _lib.load()
    p = C.c_void_p(4096)
    for T, M in ((0, 16), (16, 0), (-1, 16), (16, -5), (0, 0)):
        assert L.cat_gae(p, p, p, p, p, p, p, T, M, 0.99, 0.95, None) == CAT_ERR_INVALID
        assert b"T and M" in L.cat_last_error()
    assert L.cat_adv_normalize(p, 0, p, 16, None) == CAT_ERR_INVALID
    assert L.cat_adv_normalize(p, -4, p, 16, None) == CAT_ERR_INVALID
    assert L.cat_adv_normalize(p, 16, p, 0, None) == CAT_ERR_INVALID
    assert b"n and count" in L.cat_last_error()
    for misaligned in (4100, 4097, 4104):
        assert L.cat_adv_normalize(C.c_void_p(misaligned), 16, p, 16, None) == CAT_ERR_INVALID
        assert b"16-byte aligned" in L.cat_last_error()
    assert L.cat_adv_normalize(None, 16, p, 16, None) == CAT_ERR_INVALID
    assert L.cat_adv_normalize(p, 16, None, 16, None) == CAT_ERR_INVALID
