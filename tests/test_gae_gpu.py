"""cat_gae (both kernels) and cat_adv_normalize against the float64 reference of tests/gae_reference.py.

Each scan case runs on the TMA-fed kernel (the default when M % 16 == 0) and on the register-pipelined kernel
(CAT_GAE_TMA=0).  The unnormalised advantages must lie within GAE_BOUND_C·2^-24·S_t of the fp64 recurrence, where S_t
is the recurrence over absolute values; returns must be fp32(adv + V) bit for bit; the statistics buffer must hold the
sums of the kernel's own advantages; and the normalised output must be exactly what the statistics determine."""
import time

import numpy as np
import pytest
import torch

import gae_reference as gr
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.gae import compute_gae

pytestmark = pytest.mark.gpu

EPS = gr.EPS32
C_BOUND = gr.GAE_BOUND_C
GAMMA_LAMBDA = [(0.99, 0.95), (1.0, 1.0), (0.99, 0.0)]
T_SEAMS = (1, 7, 8, 9, 31, 32, 33, 63, 64, 65, 95, 96, 97, 1000)
M_SEAMS = (1, 15, 16, 17, 31, 32, 33, 48, 63, 64, 65, 112, 4096)


@pytest.fixture(params=["tma", "reg"])
def kernel(request, monkeypatch):
    """tma: the TMA-fed kernel wherever M % 16 == 0 and the pointers are 16-byte aligned; reg: the register kernel."""
    monkeypatch.setenv("CAT_GAE_TMA", "1" if request.param == "tma" else "0")
    return request.param


def _stream():
    return torch.cuda.current_stream().cuda_stream


def raw_gae(r, d, v, lv, gamma, lam, stats, ret=None, adv=None):
    """cat_gae without the normalisation: (T, M) float32 r, v, uint8 d, (M,) lv, all contiguous on the device."""
    L = _lib.load()
    T, M = r.shape
    ret = torch.empty_like(r) if ret is None else ret
    adv = torch.empty_like(r) if adv is None else adv
    _lib.check(L.cat_gae(r.data_ptr(), d.data_ptr(), v.data_ptr(), lv.data_ptr(), ret.data_ptr(), adv.data_ptr(),
                         stats.data_ptr(), T, M, gamma, lam, _stream()), "cat_gae")
    return ret, adv


def raw_normalize(adv, stats, count):
    L = _lib.load()
    _lib.check(L.cat_adv_normalize(adv.data_ptr(), adv.numel(), stats.data_ptr(), count, _stream()), "cat_adv_normalize")


def latest_sums(stats):
    """{sum, sumsq} of the latest call: slot (calls & 1) of the statistics buffer."""
    slot = int(stats.view(torch.int64)[4].item()) & 1
    s = stats.cpu()
    return float(s[2 * slot]), float(s[2 * slot + 1])


def mixed_dones(T, M, rng, offset=0):
    """Done pattern (column + offset) % 9 of gr.DONE_PATTERNS on each column."""
    masks = np.stack([gr.done_mask(p, T, M, rng) for p in gr.DONE_PATTERNS])
    pid = (np.arange(M) + offset) % len(gr.DONE_PATTERNS)
    return masks[pid, :, np.arange(M)].T.copy()


def make_case(T, M, rng, dones, dev):
    r = torch.from_numpy(rng.standard_normal((T, M)).astype(np.float32)).to(dev)
    v = torch.from_numpy(rng.standard_normal((T, M)).astype(np.float32)).to(dev)
    lv = torch.from_numpy(rng.standard_normal(M).astype(np.float32)).to(dev)
    return r, torch.from_numpy(dones.astype(np.uint8)).to(dev), v, lv


def check_scan(r, d, v, lv, gamma, lam, ret, adv, stats=None):
    """The kernel's (ret, adv) against the fp64 reference (computed where the inputs are); returns the largest
    |adv - adv64| / (2^-24·S_t)."""
    g, l = gr.f32(gamma), gr.f32(lam)
    a64, _ = gr.gae_fp64(r, d, v, lv, g, l)
    S = gr.gae_abs_bound(r, d, v, lv, g, l)
    err = (adv.double() - a64).abs()
    bad = err > C_BOUND * EPS * S
    if bad.any():
        t, m = (int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"T={r.shape[0]} M={r.shape[1]} γ={gamma} λ={lam}: {int(bad.sum())} advantages outside "
                             f"{C_BOUND}·2^-24·S_t, first at t={t} m={m}: kernel {float(adv[t, m])!r}, fp64 "
                             f"{float(a64[t, m])!r}, S_t {float(S[t, m])!r}")
    assert torch.equal(ret, adv + v), "returns must be fp32(adv + V) bit for bit"
    if stats is not None:
        s, q = latest_sums(stats)
        a = adv.double()
        # per thread, 8 steps are summed in fp32 before the fp64 reduction: |error| <= 8·2^-24·Σ|a|
        assert abs(s - float(a.sum())) <= 8 * EPS * float(a.abs().sum()), (s, float(a.sum()))
        assert abs(q - float((a * a).sum())) <= 8 * EPS * float((a * a).sum()), (q, float((a * a).sum()))
    return float((err / (EPS * S).clamp_min(1e-300)).max())


def check_normalized(adv, a64, S):
    """Normalised kernel output against the fp64 two-pass (a64 - mean) / (std + 1e-8).  Stated tolerance: the scan's
    error C·2^-24·S_t scaled by 1/std; its mean over the array, which moves the mean and the std, by (1 + |want|);
    and 16·2^-24·(1 + |want|) for the roundings of the mean, 1/std and the two fp32 operations."""
    std = float(a64.std())
    want = (a64 - a64.mean()) / (std + 1e-8)
    k = C_BOUND * EPS * float(S.mean()) / std
    tol = C_BOUND * EPS * S / std + (k + 16 * EPS) * (1.0 + want.abs())
    err = (adv.double() - want).abs()
    assert bool((err <= tol).all()), f"normalised advantages off by up to {float((err / tol).max()):.2f}x the tolerance"


@pytest.mark.parametrize("gamma,lam", GAMMA_LAMBDA, ids=["0.99-0.95", "1-1", "0.99-0"])
def test_scan_seams(cuda_device, kernel, gamma, lam):
    """Done flags on every segment / chunk / tile seam, ragged T and ragged column counts.  With γ = λ = 1 a carry
    lost or doubled at a seam does not decay, and the bound is relative to each element's own conditioning."""
    rng = np.random.default_rng(17)
    worst = 0.0
    stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
    shapes = [(T, 16 * len(gr.DONE_PATTERNS)) for T in T_SEAMS] + [(T, M) for M in M_SEAMS for T in (33, 97)]
    for i, (T, M) in enumerate(shapes):
        r, d, v, lv = make_case(T, M, rng, mixed_dones(T, M, rng, offset=i), cuda_device)
        ret, adv = raw_gae(r, d, v, lv, gamma, lam, stats)
        worst = max(worst, check_scan(r, d, v, lv, gamma, lam, ret, adv, stats))
    print(f"[{kernel} γ={gamma} λ={lam}] max |adv - adv64| / (2^-24 S) = {worst:.3f}")


def test_gamma_zero_is_exact(cuda_device, kernel):
    """γ = 0: every advantage is fp32(r - V) and every return fp32(adv + V), bit for bit."""
    rng = np.random.default_rng(5)
    stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
    for i, (T, M) in enumerate(((1, 16), (33, 17), (97, 64), (1000, 144), (256, 4096))):
        r, d, v, lv = make_case(T, M, rng, mixed_dones(T, M, rng, offset=i), cuda_device)
        for lam in (0.95, 1.0):
            ret, adv = raw_gae(r, d, v, lv, 0.0, lam, stats)
            assert torch.equal(adv, r - v), (T, M, lam)
            assert torch.equal(ret, adv + v), (T, M, lam)


def test_kernels_agree_bit_for_bit(cuda_device, monkeypatch):
    """Both kernels scan the same 32-step chunks as 4 segments of 8 with the same arithmetic, so their unnormalised
    advantages and returns are identical."""
    rng = np.random.default_rng(23)
    stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
    for i, (T, M) in enumerate(((1, 16), (33, 144), (97, 64), (1000, 144), (256, 49152), (1024, 4096))):
        r, d, v, lv = make_case(T, M, rng, mixed_dones(T, M, rng, offset=i), cuda_device)
        for gamma, lam in GAMMA_LAMBDA:
            out = {}
            for k in ("1", "0"):
                monkeypatch.setenv("CAT_GAE_TMA", k)
                out[k] = raw_gae(r, d, v, lv, gamma, lam, stats)
            assert torch.equal(out["1"][1], out["0"][1]), (T, M, gamma, lam)
            assert torch.equal(out["1"][0], out["0"][0]), (T, M, gamma, lam)


N_UNROLL = 148 * 16 * 256 * 4 * 3   # 7 274 496: above this the normalise kernel's 4-way unrolled loop runs


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 1023, N_UNROLL - 4, N_UNROLL, N_UNROLL + 4, 12582912, 2 ** 25 + 3])
def test_normalize_from_given_statistics_is_exact(cuda_device, n):
    """cat_adv_normalize reads {sum, sumsq} from slot (calls & 1) and is then fully determined: compare bit for bit with
    the replay, for count == n, count != n (the distributed path), a clamped variance and count == 1."""
    gen = torch.Generator(device=cuda_device).manual_seed(n)
    base = torch.randn(n, generator=gen, device=cuda_device) * 3.0 + 0.7
    a_np = base.cpu().numpy()
    a64 = a_np.astype(np.float64)
    s, q = float(a64.sum()), float((a64 * a64).sum())
    cases = [(s, q, n), (4.0 * s - 1.5, 4.0 * q + 2.0, 4 * n + 3), (s, 0.5 * q if n > 1 else 0.0, n),
             (s, q, 1), (-2.5 * n, 0.25 * q, n)]
    # the clamp: sumsq below count·mean²
    cases.append((2.0 * n, 3.0 * n, n))
    for calls, (cs, cq, count) in enumerate(cases):
        stats = torch.full((6,), 1e30, dtype=torch.float64)          # the other slot holds garbage
        slot = calls & 1
        stats[2 * slot], stats[2 * slot + 1] = cs, cq
        stats.view(torch.int64)[4], stats.view(torch.int64)[5] = calls, 0
        stats = stats.to(cuda_device)
        adv = base.clone()
        raw_normalize(adv, stats, count)
        want = gr.normalize_exact(a_np, cs, cq, count)
        got = adv.cpu().numpy()
        if not np.array_equal(got, want):
            i = int(np.flatnonzero(got != want)[0])
            raise AssertionError(f"n={n} count={count} sums=({cs!r}, {cq!r}): {int((got != want).sum())} values differ, "
                                 f"first at {i}: {got[i]!r} != {want[i]!r}")


@pytest.mark.parametrize("T,M", [(256, 49152), (1024, 49152), (64, 16384)])
def test_bench_and_learner_shapes(cuda_device, kernel, T, M):
    """Multi-wave launches at the sizes bench.py times and the learner runs, with bool dones; the reference runs on the
    device in float64."""
    gen = torch.Generator(device=cuda_device).manual_seed(T * 7 + M)
    r = torch.randn((T, M), generator=gen, device=cuda_device)
    v = torch.randn((T, M), generator=gen, device=cuda_device)
    lv = torch.randn((M,), generator=gen, device=cuda_device)
    d = torch.rand((T, M), generator=gen, device=cuda_device) < 0.08
    stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
    ret, adv = raw_gae(r, d.view(torch.uint8), v, lv, 0.99, 0.95, stats)
    worst = check_scan(r, d, v, lv, 0.99, 0.95, ret, adv, stats)
    s, q = latest_sums(stats)
    raw = adv.cpu().numpy()
    raw_normalize(adv, stats, T * M)
    assert np.array_equal(adv.cpu().numpy(), gr.normalize_exact(raw, s, q, T * M))
    a64, _ = gr.gae_fp64(r, d, v, lv, gr.f32(0.99), gr.f32(0.95))
    check_normalized(adv, a64, gr.gae_abs_bound(r, d, v, lv, gr.f32(0.99), gr.f32(0.95)))
    print(f"[{kernel} T={T} M={M}] max |adv - adv64| / (2^-24 S) = {worst:.3f}")


def _chunked_sums(a, rows=64):
    s = q = sa = 0.0
    for i in range(0, a.shape[0], rows):
        x = a[i:i + rows].double()
        s += float(x.sum()); q += float((x * x).sum()); sa += float(x.abs().sum())
    return s, q, sa


def test_gae_64bit_indexing(cuda_device, monkeypatch):
    """T·M = 1040·2^21 > 2^31: both kernels take their 64-bit-index instantiations, and rows t >= 1024 lie above
    element 2^31.  Every row of 384 columns is checked against the fp64 reference, then the normalisation."""
    T, M = 1040, 2 ** 21
    need = 48e9
    free, _ = torch.cuda.mem_get_info(cuda_device)
    if free < need:
        pytest.skip(f"needs about {need / 1e9:.0f} GB of free device memory (inputs and outputs take 37 GB), "
                    f"{free / 1e9:.1f} GB free")
    t0 = time.perf_counter()
    torch.cuda.reset_peak_memory_stats(cuda_device)
    gen = torch.Generator(device=cuda_device).manual_seed(2024)
    r = torch.empty((T, M), device=cuda_device)
    v = torch.empty((T, M), device=cuda_device)
    d = torch.empty((T, M), dtype=torch.uint8, device=cuda_device)
    for i in range(0, T, 64):
        r[i:i + 64].normal_(generator=gen)
        v[i:i + 64].normal_(generator=gen)
        d[i:i + 64] = torch.rand(r[i:i + 64].shape, generator=gen, device=cuda_device) < 0.08
    lv = torch.randn((M,), generator=gen, device=cuda_device)
    rng = np.random.default_rng(7)
    cols = np.concatenate([np.arange(64), np.arange(M - 64, M), np.sort(rng.choice(np.arange(64, M - 64), 256, replace=False))])
    ci = torch.from_numpy(cols).to(cuda_device)
    rc, dc, vc, lvc = (x.index_select(-1, ci).cpu().numpy() for x in (r, d, v, lv))
    g, l = gr.f32(0.99), gr.f32(0.95)
    a64, _ = gr.gae_fp64(rc, dc, vc, lvc, g, l)
    S = gr.gae_abs_bound(rc, dc, vc, lvc, g, l)
    ret, adv = torch.empty_like(r), torch.empty_like(r)
    seen = {}
    for k in ("tma", "reg"):
        monkeypatch.setenv("CAT_GAE_TMA", "1" if k == "tma" else "0")
        stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
        raw_gae(r, d, v, lv, 0.99, 0.95, stats, ret, adv)
        ac = adv.index_select(1, ci).cpu().numpy()
        retc = ret.index_select(1, ci).cpu().numpy()
        err = np.abs(ac.astype(np.float64) - a64)
        assert (err <= C_BOUND * EPS * S).all(), f"{k}: {int((err > C_BOUND * EPS * S).sum())} advantages outside the bound"
        assert np.array_equal(retc, ac + vc)
        for i in range(0, T, 64):
            assert torch.equal(ret[i:i + 64], adv[i:i + 64] + v[i:i + 64]), (k, i)
        s, q = latest_sums(stats)
        s64, q64, sa64 = _chunked_sums(adv)
        assert abs(s - s64) <= 8 * EPS * sa64 and abs(q - q64) <= 8 * EPS * q64, (k, s, s64, q, q64)
        n = T * M
        raw_normalize(adv, stats, n)
        nc = adv.index_select(1, ci).cpu().numpy()
        assert np.array_equal(nc, gr.normalize_exact(ac, s, q, n)), k
        mean = s64 / n
        std = np.sqrt((q64 - n * mean * mean) / (n - 1))
        want = (ac.astype(np.float64) - mean) / (std + 1e-8)
        assert (np.abs(nc - want) <= 16 * EPS * (1.0 + np.abs(want))).all(), k
        seen[k] = (ac, retc, float((err / (EPS * S)).max()))
    assert np.array_equal(seen["tma"][0], seen["reg"][0]) and np.array_equal(seen["tma"][1], seen["reg"][1])
    peak = torch.cuda.max_memory_allocated(cuda_device)
    print(f"[64-bit] {time.perf_counter() - t0:.1f} s, peak {peak / 1e9:.1f} GB allocated, max |adv - adv64| / (2^-24 S): "
          f"tma {seen['tma'][2]:.3f}, reg {seen['reg'][2]:.3f}")
    del r, v, d, lv, ret, adv, ci, stats
    torch.cuda.empty_cache()


def test_compute_gae_input_forms(cuda_device, monkeypatch):
    """(T, N, A) shapes, float64 and transposed inputs, uint8 / bool / float dones, and a view whose base is one float
    past a 16-byte boundary (M % 16 == 0, so only the alignment sends it to the register kernel)."""
    gen = torch.Generator().manual_seed(4)
    T, N, A = 97, 48, 3
    r = torch.randn((T, N, A), generator=gen)
    v = torch.randn((T, N, A), generator=gen)
    d = torch.rand((T, N, A), generator=gen) < 0.1
    lv = torch.randn((N, A), generator=gen)
    dev = cuda_device
    ret0, adv0 = compute_gae(r.to(dev), d.to(dev), v.to(dev), lv.to(dev), normalize=False)
    assert ret0.shape == (T, N, A) and adv0.shape == (T, N, A)
    M = N * A
    check_scan(r.reshape(T, M).to(dev), d.reshape(T, M).to(dev), v.reshape(T, M).to(dev), lv.reshape(M).to(dev),
               0.99, 0.95, ret0.reshape(T, M), adv0.reshape(T, M))
    for name, args in (
            ("float64", (r.double(), d, v.double(), lv.double())),
            ("transposed", (r.permute(1, 2, 0).contiguous().permute(2, 0, 1), d, v.permute(2, 1, 0).contiguous().permute(2, 1, 0),
                            lv.t().contiguous().t())),
            ("uint8 dones", (r, d.to(torch.uint8), v, lv)),
            ("float dones", (r, d.float(), v, lv))):
        x = [a.to(dev) for a in args]
        if name == "transposed":
            assert not x[0].is_contiguous() and not x[2].is_contiguous() and not x[3].is_contiguous()
        ret, adv = compute_gae(*x, normalize=False)
        assert torch.equal(ret, ret0) and torch.equal(adv, adv0), name
    # the normalised result of the same call: (adv - mean) / (std + 1e-8) of the unnormalised advantages
    ret, adv = compute_gae(r.to(dev), d.to(dev), v.to(dev), lv.to(dev))
    a = adv0.double()
    torch.testing.assert_close(adv.double(), (a - a.mean()) / (a.std() + 1e-8), rtol=1e-5, atol=1e-5)
    # misaligned views, M = 256
    T, M = 100, 256
    r = torch.randn((T, M), generator=gen).to(dev)
    v = torch.randn((T, M), generator=gen).to(dev)
    d = (torch.rand((T, M), generator=gen) < 0.1).to(torch.uint8).to(dev)
    lv = torch.randn((M,), generator=gen).to(dev)
    rb, vb = torch.empty(T * M + 1, device=dev), torch.empty(T * M + 1, device=dev)
    db = torch.empty(T * M + 1, dtype=torch.uint8, device=dev)
    ro, vo, do = rb[1:].view(T, M), vb[1:].view(T, M), db[1:].view(T, M)
    ro.copy_(r); vo.copy_(v); do.copy_(d)
    assert ro.data_ptr() % 16 == 4 and do.data_ptr() % 16 == 1
    monkeypatch.setenv("CAT_GAE_TMA", "0")
    ret_reg, adv_reg = compute_gae(r, d, v, lv, normalize=False)
    monkeypatch.setenv("CAT_GAE_TMA", "1")
    ret_tma, adv_tma = compute_gae(r, d, v, lv, normalize=False)
    check_scan(r, d, v, lv, 0.99, 0.95, ret_reg, adv_reg)
    # the two kernels are bit-identical (test_kernels_agree_bit_for_bit), so the aligned call of either kernel is the answer
    assert torch.equal(ret_tma, ret_reg) and torch.equal(adv_tma, adv_reg)
    for x in ((ro, d, v, lv), (r, do, v, lv), (r, d, vo, lv), (ro, do, vo, lv)):
        ret, adv = compute_gae(*x, normalize=False)
        assert torch.equal(ret, ret_reg) and torch.equal(adv, adv_reg)


def test_compute_gae_on_two_streams_at_once(cuda_device):
    """Each (device, stream) has its own statistics buffer, so two concurrent calls normalise with their own sums."""
    gen = torch.Generator(device=cuda_device).manual_seed(9)
    dev = cuda_device
    inputs = []
    for (T, M), shift in (((256, 49152), 0.0), ((128, 30001), 2.0)):
        inputs.append((torch.randn((T, M), generator=gen, device=dev) + shift, torch.rand((T, M), generator=gen, device=dev) < 0.08,
                       torch.randn((T, M), generator=gen, device=dev), torch.randn((M,), generator=gen, device=dev)))
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
    torch.cuda.synchronize()
    outs = [None, None]
    for rep in range(2):
        for i in (0, 1):
            with torch.cuda.stream(streams[i]):
                outs[i] = compute_gae(*inputs[i])
    torch.cuda.synchronize()
    for (r, d, v, lv), (ret, adv) in zip(inputs, outs):
        a64, ret64 = gr.gae_fp64(r, d, v, lv, gr.f32(0.99), gr.f32(0.95))
        S = gr.gae_abs_bound(r, d, v, lv, gr.f32(0.99), gr.f32(0.95))
        assert bool(((ret.double() - ret64).abs() <= (C_BOUND + 2) * EPS * S).all())    # |ret| <= |adv| + |V| <= 2·S
        check_normalized(adv, a64, S)
