"""Batched device-resident r2c / c2r (phastft_{r2c,c2r}_*_dev_batch, api.r2c_fft_batch / c2r_fft_batch).

Tolerances as in test_gpu_r2c.py: vs numpy (f64 truth) rel-Linf <= 4 eps log2 N, vs the oracle that plus the oracle's own
error.  At one-CTA sizes the r2c untangle runs inside the transform kernel (MODE_R2C_OUT) unless PHASTFT_R2C_FUSE=0; both
forms do the same operations and must agree bit for bit.  Every batched c2r builds the inverse transform's input while
loading the spectrum, so it differs from the single call's separate sweep by one rounding at most (test_gpu_r2c.py's
fused-vs-sweep tolerance).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PAD = 1234.5


def _pf():
    import phastft_b200 as pf
    return pf


def tol(dt, n):
    return 4.0 * np.finfo(dt).eps * max(np.log2(n), 1.0)


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _tdt(dt):
    import torch
    return torch.float64 if dt == np.float64 else torch.float32


def _planner(dt, n):
    pf = _pf()
    return (pf.PlannerR2c64 if dt == np.float64 else pf.PlannerR2c32)(n)


def _real_batch(dt, n, batch, stride, seed):
    """`batch` members of n reals at `stride`, padding PAD; returns (device tensor, host (batch, n) view)"""
    import torch
    x = np.full(max((batch - 1) * stride + n, 1), PAD, dt)
    v = np.lib.stride_tricks.as_strided(x, (batch, n), (stride * x.itemsize, x.itemsize))
    v[:] = np.random.default_rng(seed).uniform(-1, 1, (batch, n)).astype(dt)
    return torch.from_numpy(x).cuda(), v.copy()


def _members(t, batch, length, stride):
    a = t.cpu().numpy()
    return np.stack([a[b * stride:b * stride + length] for b in range(batch)])


def _padding_intact(t, batch, length, stride):
    a = t.cpu().numpy()
    mask = np.ones(a.size, bool)
    for b in range(batch):
        mask[b * stride:b * stride + length] = False
    return bool(np.all(a[mask] == PAD))


def _run_r2c(dt, n, batch, in_stride, out_stride, x):
    import torch
    pf = _pf()
    half = n // 2
    ore = torch.full(((batch - 1) * out_stride + half + 1,), PAD, dtype=_tdt(dt), device="cuda")
    oim = ore.clone()
    pf.r2c_fft_batch(x, ore, oim, _planner(dt, n), batch, in_stride, out_stride)
    torch.cuda.synchronize()
    return ore, oim


SIZES = [2, 3, 4, 6, 8, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22]


def _batch_for(log_n):
    return 3 if log_n >= 20 else 5 if log_n >= 16 else 37


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("log_n", SIZES)
@pytest.mark.parametrize("padded", [False, True])
def test_r2c_batch_members_vs_truth_and_oracle(dt, log_n, padded):
    from oracle import oracle as O
    n = 1 << log_n; half = n // 2
    batch = _batch_for(log_n)
    in_stride = n + 6 if padded else n
    out_stride = half + 4 if padded else half + 1
    x, xh = _real_batch(dt, n, batch, in_stride, 100 + log_n)
    x0 = x.clone()
    ore, oim = _run_r2c(dt, n, batch, in_stride, out_stride, x)
    G = _members(ore, batch, half + 1, out_stride).astype(np.float64) + 1j * _members(oim, batch, half + 1, out_stride)
    truth = np.fft.rfft(xh.astype(np.float64), axis=1)
    for b in range(batch):
        assert rel(G[b], truth[b]) <= tol(dt, n), (b, rel(G[b], truth[b]))
    for b in (0, batch - 1):
        o_re = np.zeros(half + 1, dt); o_im = np.zeros(half + 1, dt)
        O.r2c_fft(np.ascontiguousarray(xh[b]), o_re, o_im)
        Oc = o_re.astype(np.float64) + 1j * o_im
        assert rel(G[b], Oc) <= tol(dt, n) + rel(Oc, truth[b])
    assert np.all(G[:, 0].imag == 0) and np.all(G[:, half].imag == 0)
    assert _padding_intact(ore, batch, half + 1, out_stride) and _padding_intact(oim, batch, half + 1, out_stride)
    import torch
    assert torch.equal(x, x0)


# one-CTA half-lengths: f64 up to 2^13, f32 up to 2^14 points
ONE_CTA = [(np.float64, ln) for ln in range(2, 15)] + [(np.float32, ln) for ln in range(2, 16)]


@pytest.mark.parametrize("dt,log_n", ONE_CTA)
def test_r2c_fused_matches_unfused_bitwise(dt, log_n, monkeypatch):
    import torch
    n = 1 << log_n; half = n // 2
    # a small batch (lone-transform kernel) and one of >= 2^21 half-length points (batch kernel); neither a multiple of the
    # members per CTA, so the last CTA is partial
    pf = _pf()
    for batch in (5, (1 << 21) // half + 3):
        x, _ = _real_batch(dt, n, batch, n, 7 + log_n)
        outs, launches = [], []
        for fuse in ("1", "0"):
            monkeypatch.setenv("PHASTFT_R2C_FUSE", fuse)
            before = pf.launch_count()
            outs.append(_run_r2c(dt, n, batch, n, half + 1, x))
            launches.append(pf.launch_count() - before)
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), (n, batch)
        assert launches[0] <= launches[1]
        if batch > 5 and half >= 4:
            # the batch kernel of every half-length >= 4 has a shared-memory stage, so its MODE_R2C_OUT build runs: one launch,
            # against the half-length transform plus the untangle sweep
            assert launches == [1, 2], launches


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("log_n", [2, 5, 11, 13, 16, 20])
def test_batch_of_one_is_the_single_call(dt, log_n):
    import torch
    pf = _pf()
    n = 1 << log_n; half = n // 2
    pl = _planner(dt, n)
    r2c_p = pf.r2c_fft_f64_with_planner if dt == np.float64 else pf.r2c_fft_f32_with_planner
    c2r_p = pf.c2r_fft_f64_with_planner if dt == np.float64 else pf.c2r_fft_f32_with_planner
    x, _ = _real_batch(dt, n, 1, n, 3 + log_n)
    a_re = torch.empty(half + 1, dtype=_tdt(dt), device="cuda"); a_im = torch.empty_like(a_re)
    b_re = torch.empty_like(a_re); b_im = torch.empty_like(a_re)
    r2c_p(x, a_re, a_im, pl)
    pf.r2c_fft_batch(x, b_re, b_im, pl, 1)
    assert torch.equal(a_re, b_re) and torch.equal(a_im, b_im)
    ya = torch.empty(n, dtype=_tdt(dt), device="cuda"); yb = torch.empty_like(ya)
    c2r_p(a_re, a_im, ya, pl)
    pf.c2r_fft_batch(a_re, a_im, yb, pl, 1)
    assert torch.equal(ya, yb)


def _spectra(dt, n, batch, stride, seed):
    import torch
    half = n // 2
    rng = np.random.default_rng(seed)
    re = np.full((batch - 1) * stride + half + 1, PAD, dt); im = re.copy()
    for b in range(batch):
        re[b * stride:b * stride + half + 1] = rng.uniform(-1, 1, half + 1)
        im[b * stride:b * stride + half + 1] = rng.uniform(-1, 1, half + 1)
        im[b * stride] = 0; im[b * stride + half] = 0       # Hermitian-valid: DC and Nyquist real
    return torch.from_numpy(re).cuda(), torch.from_numpy(im).cuda()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("log_n", SIZES)
@pytest.mark.parametrize("padded", [False, True])
def test_c2r_batch_vs_truth_single_call_and_roundtrip(dt, log_n, padded):
    import torch
    pf = _pf()
    n = 1 << log_n; half = n // 2
    batch = _batch_for(log_n)
    in_stride = half + 4 if padded else half + 1
    out_stride = n + 6 if padded else n
    pl = _planner(dt, n)
    s_re, s_im = _spectra(dt, n, batch, in_stride, 500 + log_n)
    k_re, k_im = s_re.clone(), s_im.clone()
    y = torch.full(((batch - 1) * out_stride + n,), PAD, dtype=_tdt(dt), device="cuda")
    pf.c2r_fft_batch(s_re, s_im, y, pl, batch, in_stride, out_stride)
    torch.cuda.synchronize()
    assert torch.equal(s_re, k_re) and torch.equal(s_im, k_im)           # the spectrum is never written
    assert _padding_intact(y, batch, n, out_stride)
    Y = _members(y, batch, n, out_stride)
    S = _members(s_re, batch, half + 1, in_stride).astype(np.float64) + 1j * _members(s_im, batch, half + 1, in_stride)
    truth = np.fft.irfft(S, n, axis=1)
    scale = max(float(np.max(np.abs(truth))), 1.0)
    assert np.max(np.abs(Y - truth)) <= tol(dt, n) * scale * 4
    c2r_p = pf.c2r_fft_f64_with_planner if dt == np.float64 else pf.c2r_fft_f32_with_planner
    for b in (0, batch - 1):
        one = torch.empty(n, dtype=_tdt(dt), device="cuda")
        c2r_p(s_re[b * in_stride:b * in_stride + half + 1].contiguous(), s_im[b * in_stride:b * in_stride + half + 1].contiguous(), one, pl)
        ref = one.cpu().numpy()
        assert np.max(np.abs(Y[b] - ref)) <= tol(dt, n) * max(float(np.max(np.abs(ref))), 1.0)
    # round trip c2r_batch(r2c_batch(x)) ~ x
    x, xh = _real_batch(dt, n, batch, out_stride, 900 + log_n)
    ore, oim = _run_r2c(dt, n, batch, out_stride, in_stride, x)
    z = torch.full_like(y, PAD)
    pf.c2r_fft_batch(ore, oim, z, pl, batch, in_stride, out_stride)
    torch.cuda.synchronize()
    assert np.max(np.abs(_members(z, batch, n, out_stride) - xh)) <= tol(dt, n) * 4


@pytest.mark.parametrize("dt,log_n,batch,padded", [(np.float64, 16, 64, False), (np.float32, 16, 64, False),
                                                   (np.float64, 22, 3, True)])
def test_c2r_batch_multipass_batch_kernel(dt, log_n, batch, padded):
    """batch * N/2 >= 2^21 (the first pass runs the batch kernel's MODE_C2R_IN build), and a 3-pass inner plan"""
    import torch
    pf = _pf()
    n = 1 << log_n; half = n // 2
    in_stride = half + 4 if padded else half + 1
    out_stride = n + 6 if padded else n
    s_re, s_im = _spectra(dt, n, batch, in_stride, 41)
    y = torch.full(((batch - 1) * out_stride + n,), PAD, dtype=_tdt(dt), device="cuda")
    pf.c2r_fft_batch(s_re, s_im, y, _planner(dt, n), batch, in_stride, out_stride)
    torch.cuda.synchronize()
    S = _members(s_re, batch, half + 1, in_stride).astype(np.float64) + 1j * _members(s_im, batch, half + 1, in_stride)
    truth = np.fft.irfft(S, n, axis=1)
    assert np.max(np.abs(_members(y, batch, n, out_stride) - truth)) <= tol(dt, n) * max(float(np.max(np.abs(truth))), 1.0) * 4
    assert _padding_intact(y, batch, n, out_stride)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_batches_above_grid_y_limit(dt, monkeypatch):
    import torch
    pf = _pf()
    n, batch = 16, 70000
    x, xh = _real_batch(dt, n, batch, n, 11)
    for fuse in ("1", "0"):
        monkeypatch.setenv("PHASTFT_R2C_FUSE", fuse)
        ore, oim = _run_r2c(dt, n, batch, n, n // 2 + 1, x)
        G = ore.cpu().numpy().reshape(batch, -1).astype(np.float64) + 1j * oim.cpu().numpy().reshape(batch, -1)
        assert rel(G, np.fft.rfft(xh.astype(np.float64), axis=1)) <= tol(dt, n)
    y = torch.empty(batch * n, dtype=_tdt(dt), device="cuda")
    pf.c2r_fft_batch(ore, oim, y, _planner(dt, n), batch)
    torch.cuda.synchronize()
    assert np.max(np.abs(y.cpu().numpy().reshape(batch, n) - xh)) <= tol(dt, n) * 4


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_argument_errors_raise_before_any_launch(dt):
    import torch
    pf = _pf()
    n, half, batch = 64, 32, 4
    pl = _planner(dt, n)
    T = _tdt(dt)
    x = torch.zeros(batch * n + 2, dtype=T, device="cuda")
    re = torch.zeros(batch * (half + 1), dtype=T, device="cuda"); im = torch.zeros_like(re)
    y = torch.zeros(batch * n + 2, dtype=T, device="cuda")
    bad = [
        lambda: pf.r2c_fft_batch(x[: 3 * n], re, im, pl, batch),                      # short input
        lambda: pf.r2c_fft_batch(x, re[: 3 * (half + 1)], im, pl, batch),             # short output
        lambda: pf.r2c_fft_batch(x, re, im, pl, batch, in_stride=n - 2),              # stride < N
        lambda: pf.r2c_fft_batch(x, re, im, pl, 2, out_stride=half),                  # stride < N/2 + 1
        lambda: pf.r2c_fft_batch(x, re, im, pl, 2, in_stride=n + 1),                  # odd real stride
        lambda: pf.r2c_fft_batch(x[1:], re, im, pl, 2),                               # misaligned real base
        lambda: pf.c2r_fft_batch(re[: 3 * (half + 1)], im, y, pl, batch),             # short spectrum
        lambda: pf.c2r_fft_batch(re, im, y[: 3 * n], pl, batch),                      # short output
        lambda: pf.c2r_fft_batch(re, im, y, pl, 2, in_stride=half),                   # stride < N/2 + 1
        lambda: pf.c2r_fft_batch(re, im, y, pl, 2, out_stride=n - 2),                 # stride < N
        lambda: pf.c2r_fft_batch(re, im, y, pl, 2, out_stride=n + 1),                 # odd real stride
        lambda: pf.c2r_fft_batch(re, im, y[1:], pl, 2),                               # misaligned real base
        lambda: pf.r2c_fft_batch(x, re, im, pl, 0),                                   # empty batch
    ]
    before = pf.launch_count()
    for i, call in enumerate(bad):
        with pytest.raises(pf.PhastFTPanic) as e:
            call()
        assert e.value.code == 13, i
    assert pf.launch_count() == before


@pytest.mark.parametrize("dt,log_n,batch", [(np.float64, 10, 64), (np.float64, 18, 8), (np.float32, 18, 8)])
def test_graph_capture_after_reserve(dt, log_n, batch):
    import torch
    pf = _pf()
    n = 1 << log_n; half = n // 2
    T = _tdt(dt)
    x, _ = _real_batch(dt, n, batch, n, 5)
    ore = torch.empty(batch * (half + 1), dtype=T, device="cuda"); oim = torch.empty_like(ore)
    y = torch.empty(batch * n, dtype=T, device="cuda")
    eager_pl = _planner(dt, n)
    pf.r2c_fft_batch(x, ore, oim, eager_pl, batch)
    pf.c2r_fft_batch(ore, oim, y, eager_pl, batch)
    torch.cuda.synchronize()
    e_re, e_im, e_y = ore.clone(), oim.clone(), y.clone()
    if log_n >= 14:
        # a fresh multi-pass plan has a one-transform workspace: capturing a batch without reserve fails cleanly
        fresh = _planner(dt, n)
        s = torch.cuda.Stream()
        with pytest.raises(Exception):
            with torch.cuda.graph(torch.cuda.CUDAGraph(), stream=s):
                pf.r2c_fft_batch(x, ore, oim, fresh, batch)
        torch.cuda.synchronize()
    pl = _planner(dt, n)
    pl.reserve(batch)
    ore.zero_(); oim.zero_(); y.zero_()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.graph(g, stream=s):
        pf.r2c_fft_batch(x, ore, oim, pl, batch)
        pf.c2r_fft_batch(ore, oim, y, pl, batch)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(ore, e_re) and torch.equal(oim, e_im) and torch.equal(y, e_y)
