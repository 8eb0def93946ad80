"""Float64 reference of the GAE scan and the exact replay of the advantage normalisation.

``cat_gae`` computes skrl's ``compute_gae`` in float32 as a parallel scan; ``cat_adv_normalize`` then normalises in place.
This module is what the tests hold the two kernels against:

* ``gae_fp64`` — the plain sequential recurrence in float64 (numpy arrays, or torch tensors on any device);
* ``gae_abs_bound`` — the same recurrence over absolute values, which scales the float32 error allowed at each element;
* ``normalize_exact`` — the normalisation the kernel performs, replayed bit for bit from its statistics buffer.

The kernel receives γ and λ as float32: pass ``f32(gamma)``, ``f32(lam)`` to compare with it.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

EPS32 = 2.0 ** -24

# A kernel advantage a32 passes when |a32 - a64| <= GAE_BOUND_C * EPS32 * S_t (S_t from gae_abs_bound).
# Observed maximum of |a32 - a64| / (EPS32 * S_t) over tests/test_gae_gpu.py on a B200 (1000 W power limit): 2.88,
# for the TMA-fed and the register kernel alike (T = 1024, M = 49152, γ = 0.99, λ = 0.95).  12 is about 4x that.
GAE_BOUND_C = 12.0


def f32(x: float) -> float:
    """x rounded to float32, as the C ABI's float parameters receive it."""
    return float(np.float32(x))


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _f64(x):
    return x.double() if _is_torch(x) else np.asarray(x, dtype=np.float64)


def _not_done(d):
    return (d == 0).double() if _is_torch(d) else (np.asarray(d) == 0).astype(np.float64)


def _zeros_like(x):
    return x.new_zeros(x.shape) if _is_torch(x) else np.zeros_like(x)


def gae_fp64(r, d, v, lv, gamma: float, lam: float):
    """skrl's recurrence ``a_t = r_t - V_t + γ(1 - done_t)(V_{t+1} + λ a_{t+1})`` in float64, V_T = ``lv``.

    ``r``, ``d``, ``v`` are (T, M) and ``lv`` is (M,).  Returns ``(adv, ret)`` in float64, unnormalised, with
    ``ret = adv + V``.  The operations run in the order of ``oracle/cat_oracle.c:orc_gae``."""
    r, v, lv, nd = _f64(r), _f64(v), _f64(lv), _not_done(d)
    T = r.shape[0]
    adv = _zeros_like(r)
    a = _zeros_like(lv)
    for t in range(T - 1, -1, -1):
        nv = lv if t == T - 1 else v[t + 1]
        a = r[t] - v[t] + gamma * nd[t] * (nv + lam * a)
        adv[t] = a
    return adv, adv + v


def gae_abs_bound(r, d, v, lv, gamma: float, lam: float):
    """S_t = |r_t| + |V_t| + γ·nd_t·(|V_{t+1}| + λ·S_{t+1}), S_T = 0, in float64.

    Every term the recurrence adds into a_t is bounded by S_t, so a float32 evaluation of the scan, in any order, is
    off by a modest multiple of 2^-24·S_t.  A carry lost or doubled at a chunk seam is off by |a| itself."""
    r, v, lv, nd = _f64(r), _f64(v), _f64(lv), _not_done(d)
    T = r.shape[0]
    S = _zeros_like(r)
    s = _zeros_like(lv)
    for t in range(T - 1, -1, -1):
        nv = lv if t == T - 1 else v[t + 1]
        s = abs(r[t]) + abs(v[t]) + gamma * nd[t] * (abs(nv) + lam * s)
        S[t] = s
    return S


# Done flags placed on the scan's seams: segments of 8 steps start at t ≡ 0 and end at t ≡ 7 (mod 8); chunks and TMA
# tiles of 32 steps at t ≡ 0 and 31 (mod 32).  The scan walks T backwards from T - 1, so those residues are taken
# from the end of the rollout too.
DONE_PATTERNS = ("none", "all", "t%8==7", "t%8==0", "t%32==31", "t%32==0", "last", "first", "random8")


def done_mask(pattern: str, T: int, M: int, rng: np.random.Generator) -> np.ndarray:
    """(T, M) bool done flags of one pattern of DONE_PATTERNS, for every column alike (``random8``: 8 % at random)."""
    t = np.arange(T)[:, None]
    u = (T - 1 - t)      # steps before the end: the kernels' chunks are aligned to T
    m = {"none": np.zeros_like(t, bool), "all": np.ones_like(t, bool),
         "t%8==7": (t % 8 == 7) | (u % 8 == 0), "t%8==0": (t % 8 == 0) | (u % 8 == 7),
         "t%32==31": (t % 32 == 31) | (u % 32 == 0), "t%32==0": (t % 32 == 0) | (u % 32 == 31),
         "last": t == T - 1, "first": t == 0}.get(pattern)
    if pattern == "random8":
        return rng.random((T, M)) < 0.08
    return np.broadcast_to(m, (T, M)).copy()


def _fma(a: float, b: float, c: float) -> float:
    """a·b + c rounded once to float64 (the exact rational result, correctly rounded)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def normalize_params(stats_sum: float, stats_sumsq: float, count: int):
    """(float32 mean, float32 1/(std + 1e-8)) exactly as ``cat_adv_normalize_kernel`` forms them.

    The float64 part is IEEE: the build's ``-prec-div=false -prec-sqrt=false`` only touch float32.  nvcc contracts
    ``sumsq - count·mean·mean`` into one fused multiply-add, ``fma(-(count·mean), mean, sumsq)``, so that is replayed
    with a single rounding."""
    count = int(count)
    mean = float(stats_sum) / float(count)
    if count > 1:
        var = _fma(-(float(count) * mean), mean, float(stats_sumsq)) / float(count - 1)
    else:
        var = 0.0
    if var < 0.0:
        var = 0.0
    return np.float32(mean), np.float32(1.0 / (np.sqrt(var) + 1e-8))


def normalize_exact(adv32, stats_sum: float, stats_sumsq: float, count: int) -> np.ndarray:
    """The kernel's in-place ``(adv - fm) * inv`` in float32, bit for bit, for a float32 array of advantages."""
    fm, inv = normalize_params(stats_sum, stats_sumsq, count)
    a = np.asarray(adv32, dtype=np.float32)
    return (a - fm) * inv
