"""Pin the CPU oracle (oracle/phastft_oracle.cpp) against every known-answer test the
reference holds for the path (SURVEY.md section 8c), plus the committed golden vectors.

Each test cites the reference test it restates.  numpy.fft (pocketfft, f64) and the
extended-precision golden DFTs stand in for RustFFT, the reference's own test oracle
(utilities/src/lib.rs:1).
"""
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as O

GOLD = Path(__file__).resolve().parent / "golden"
F = {np.float64: "f64", np.float32: "f32"}


def rel_linf(a_re, a_im, b_re, b_im):
    a = np.asarray(a_re, np.float64) + 1j * np.asarray(a_im, np.float64)
    b = np.asarray(b_re, np.float64) + 1j * np.asarray(b_im, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), np.finfo(np.float64).tiny))


# --- lib.rs:171-178 doctest, codelets.rs:529-531 -------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("n", [1, 2, 4, 8, 16, 32, 64, 1024, 4096])
def test_impulse_gives_all_ones(dt, n):
    re = np.zeros(n, dt); im = np.zeros(n, dt); re[0] = 1
    O.fft_dit(re, im, O.FORWARD)
    assert np.array_equal(re, np.ones(n, dt))
    assert np.array_equal(im, np.zeros(n, dt))


# --- lib.rs:298-338 fft_correctness_{32,64}: ramp re=im=1..=n vs independent FFT, abs 0.01 ---
@pytest.mark.parametrize("dt,ks", [(np.float32, range(4, 9)), (np.float64, range(4, 17))])
def test_ramp_vs_independent_fft(dt, ks):
    for k in ks:
        n = 1 << k
        re = np.arange(1, n + 1, dtype=dt); im = re.copy()
        O.fft_dit(re, im, O.FORWARD)
        ref = np.fft.fft(np.arange(1, n + 1, dtype=np.float64) * (1 + 1j))
        assert np.max(np.abs(re - ref.real)) < 0.01
        assert np.max(np.abs(im - ref.imag)) < 0.01


# --- lib.rs:380-425 forward then reverse restores a unit-norm random signal ---------------
@pytest.mark.parametrize("dt,eps", [(np.float64, 1e-10), (np.float32, 1e-7)])
def test_roundtrip_random(dt, eps):
    for k in range(4, 12):
        n = 1 << k
        re0, im0 = O.gen_random_signal(n, dt, seed=k)
        re, im = re0.copy(), im0.copy()
        O.fft_dit(re, im, O.FORWARD)
        O.fft_dit(re, im, O.REVERSE)
        assert np.max(np.abs(re - re0)) < eps
        assert np.max(np.abs(im - im0)) < eps


# --- BASELINE.json configs[0]: single 2^10 f64 forward+inverse, round trip abs 1e-10 ---------
def test_config0_2pow10_f64_roundtrip():
    re0, im0 = O.gen_random_signal(1 << 10, np.float64, seed=1234)
    re, im = re0.copy(), im0.copy()
    O.fft_dit(re, im, O.FORWARD)
    ref = np.fft.fft(re0 + 1j * im0)
    assert rel_linf(re, im, ref.real, ref.imag) < 4 * 2.0 ** -52 * 10
    O.fft_dit(re, im, O.REVERSE)
    assert np.max(np.abs(re - re0)) < 1e-10 and np.max(np.abs(im - im0)) < 1e-10


# --- lib.rs:238-296 planner misuse -------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_non_power_of_two_planner_panics(dt):
    with pytest.raises(O.OraclePanic) as e:
        O.PlannerDit(5, dt)
    assert e.value.code == 2
    with pytest.raises(O.OraclePanic):
        O.PlannerDit(0, dt)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_wrong_num_points_in_planner_panics(dt):
    planner = O.PlannerDit(16, dt)
    re = np.zeros(1 << 16, dt); im = np.zeros(1 << 16, dt)
    with pytest.raises(O.OraclePanic) as e:
        O.fft_dit(re, im, O.FORWARD, planner)
    assert e.value.code == 3


def test_length_mismatch_panics():
    with pytest.raises(O.OraclePanic) as e:
        O.fft_dit(np.zeros(16), np.zeros(8), O.FORWARD)
    assert e.value.code == 1


# --- planner reuse == convenience wrapper, bit for bit (r2c.rs:979-1131 style equivalences) ---
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_planner_matches_convenience_bit_exact(dt):
    n = 4096
    re0, im0 = O.gen_random_signal(n, dt)
    a, b = re0.copy(), im0.copy(); O.fft_dit(a, b, O.FORWARD)
    pl = O.PlannerDit(n, dt)
    c, d = re0.copy(), im0.copy(); O.fft_dit(c, d, O.FORWARD, pl)
    assert np.array_equal(a, c) and np.array_equal(b, d)
    e, f = re0.copy(), im0.copy(); O.fft_dit(e, f, O.FORWARD, pl, parallel=True)
    assert np.array_equal(a, e) and np.array_equal(b, f)


# --- planner.rs:74-93 table contents --------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_planner_tables(dt):
    pl = O.PlannerDit(1 << 10, dt)
    tabs = pl.stage_twiddles()
    assert len(tabs) == 10 - 6
    for i, (re, im) in enumerate(tabs):
        dist = 64 << i
        assert re.size == dist
        k = np.arange(dist, dtype=dt)
        pi = dt(np.pi)
        ang = (dt(-2.0) * pi / dt(2 * dist)) * k
        assert ang.dtype == np.dtype(dt)
        tol = 1e-15 if dt == np.float64 else 2e-7
        assert np.max(np.abs(re - np.cos(ang.astype(np.float64)))) < tol
        assert np.max(np.abs(im - np.sin(ang.astype(np.float64)))) < tol


# --- bravo.rs:373-407 bit reversal of iota, exact, n = 2..=23 (trimmed to 2..=20 for CPU time) -
def _bit_reverse_reference(n):
    """bravo.rs:355-371: recursive even/odd permutation."""
    idx = np.arange(1 << n)
    rev = np.zeros_like(idx)
    for b in range(n):
        rev |= ((idx >> b) & 1) << (n - 1 - b)
    return rev


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("tiled", [False, True])
def test_bit_reversal_exact(dt, tiled):
    for n in range(2, 21):
        x = np.arange(1 << n, dtype=dt)
        O.bit_reverse(x, tiled=tiled)
        assert np.array_equal(x, _bit_reverse_reference(n).astype(dt)), n


# --- codelets.rs:522-698 codelet == chunk_2 -> ... -> chunk_16/32 chain -------------------------
def _staged(re, im, stages):
    for s in range(stages):
        O.stage(re, im, s)


@pytest.mark.parametrize("dt,tol", [(np.float64, 1e-13), (np.float32, 1e-5)])
def test_codelet_matches_staged(dt, tol):
    st = O.codelet_stages(dt)
    size = 1 << st
    cases = []
    imp_re = np.zeros(size, dt); imp_re[0] = 1
    cases.append((imp_re, np.zeros(size, dt)))
    cases.append((np.arange(1, size + 1, dtype=dt), np.arange(size, 0, -1).astype(dt)))
    i = np.arange(8 * size, dtype=dt)
    cases.append((dt(0.1) * i, dt(-0.05) * i))
    for re0, im0 in cases:
        a, b = re0.copy(), im0.copy(); O.codelet(a, b)
        c, d = re0.copy(), im0.copy(); _staged(c, d, st)
        scale = max(np.max(np.abs(c)), np.max(np.abs(d)), 1)
        assert np.max(np.abs(a - c)) <= tol * scale
        assert np.max(np.abs(b - d)) <= tol * scale


# --- committed golden vectors (extended-precision DFT) -------------------------------------------
@pytest.mark.parametrize("dt,c", [(np.float64, 4.0), (np.float32, 4.0)])
def test_golden_c2c(dt, c):
    g = np.load(GOLD / "c2c_golden.npz")
    eps = np.finfo(dt).eps
    for n in (1, 2, 4, 8, 16, 32, 64, 128, 256, 1024, 4096):
        re = g[f"rand_{n}_in_re"].astype(dt); im = g[f"rand_{n}_in_im"].astype(dt)
        O.fft_dit(re, im, O.FORWARD)
        err = rel_linf(re, im, g[f"rand_{n}_out_re"], g[f"rand_{n}_out_im"])
        assert err <= c * eps * max(np.log2(n), 1), (n, err)
    for n in (16, 64, 256, 1024):
        re = np.arange(1, n + 1, dtype=dt); im = re.copy()
        O.fft_dit(re, im, O.FORWARD)
        err = rel_linf(re, im, g[f"ramp_{n}_out_re"], g[f"ramp_{n}_out_im"])
        assert err <= c * eps * np.log2(n), (n, err)


# ======================================= r2c / c2r ==============================================

# --- r2c.rs:915-956 r2c equals the first N/2+1 bins of the c2c -----------------------------------
@pytest.mark.parametrize("dt,hi,tol", [(np.float64, 14, 1e-4), (np.float32, 10, None)])
def test_r2c_vs_c2c(dt, hi, tol):
    for n_log in range(2, hi + 1):
        n = 1 << n_log; half = n // 2
        x = np.arange(1, n + 1, dtype=dt)
        ore = np.zeros(half + 1, dt); oim = np.zeros(half + 1, dt)
        O.r2c_fft(x, ore, oim)
        rre = x.copy(); rim = np.zeros(n, dt)
        O.fft_dit(rre, rim, O.FORWARD)
        if tol is not None:
            assert np.max(np.abs(ore - rre[: half + 1])) < tol
            assert np.max(np.abs(oim - rim[: half + 1])) < tol
        else:  # r2c.rs:904-911 relative 1e-2 with denominator max(|expected|, EPSILON)
            for got, exp in ((ore, rre[: half + 1]), (oim, rim[: half + 1])):
                # the reference's per-bin relative test is vacuous-prone at exact-zero bins; use the
                # bound it implies on the spectrum scale as well
                assert np.max(np.abs(got - exp)) <= 1e-2 * np.max(np.abs(rre))


# --- r2c.rs:959-976, 1168-1229 round trips --------------------------------------------------------
@pytest.mark.parametrize("dt,hi,tol", [(np.float64, 14, 1e-6), (np.float32, 12, None)])
def test_r2c_c2r_roundtrip(dt, hi, tol):
    for n_log in range(2, hi + 1):
        n = 1 << n_log; half = n // 2
        for x in (np.arange(1, n + 1, dtype=dt), np.random.default_rng(n).uniform(-1, 1, n).astype(dt)):
            ore = np.zeros(half + 1, dt); oim = np.zeros(half + 1, dt)
            O.r2c_fft(x, ore, oim)
            y = np.zeros(n, dt)
            O.c2r_fft(ore, oim, y)
            if tol is not None:
                assert np.max(np.abs(y - x)) < tol * max(1.0, np.max(np.abs(x))) if x[0] == 1 else np.max(np.abs(y - x)) < tol
            else:
                assert np.max(np.abs(y - x)) <= 1e-2 * np.max(np.abs(x))


# --- r2c.rs:1236-1386 known answers ---------------------------------------------------------------
@pytest.mark.parametrize("dt,tol", [(np.float64, 1e-10), (np.float32, 1e-4)])
def test_r2c_dc_only(dt, tol):
    n = 16; half = 8
    ore = np.zeros(half + 1, dt); oim = np.zeros(half + 1, dt)
    O.r2c_fft(np.ones(n, dt), ore, oim)
    assert abs(ore[0] - n) < tol and abs(oim[0]) < tol
    assert np.max(np.abs(ore[1:])) < tol and np.max(np.abs(oim[1:])) < tol


@pytest.mark.parametrize("dt,tol", [(np.float64, 1e-10), (np.float32, 1e-4)])
def test_r2c_nyquist_only(dt, tol):
    n = 16; half = 8
    x = np.where(np.arange(n) % 2 == 0, 1, -1).astype(dt)
    ore = np.zeros(half + 1, dt); oim = np.zeros(half + 1, dt)
    O.r2c_fft(x, ore, oim)
    exp = np.zeros(half + 1); exp[half] = n
    assert np.max(np.abs(ore - exp)) < tol and np.max(np.abs(oim)) < tol


def test_r2c_single_tone_f64():
    n = 32; half = 16
    x = np.cos(2 * np.pi * np.arange(n) / n)
    ore = np.zeros(half + 1); oim = np.zeros(half + 1)
    O.r2c_fft(x, ore, oim)
    exp = np.zeros(half + 1); exp[1] = n / 2
    assert np.max(np.abs(ore - exp)) < 1e-9 and np.max(np.abs(oim)) < 1e-9


@pytest.mark.parametrize("dt,tol", [(np.float64, 1e-12), (np.float32, 1e-6)])
def test_r2c_all_zeros_overwrites_output(dt, tol):
    n = 16; half = 8
    ore = np.ones(half + 1, dt); oim = np.ones(half + 1, dt)
    O.r2c_fft(np.zeros(n, dt), ore, oim)
    assert np.max(np.abs(ore)) < tol and np.max(np.abs(oim)) < tol


@pytest.mark.parametrize("dt,tol", [(np.float64, 1e-10), (np.float32, 1e-3)])
def test_r2c_dc_and_nyquist_are_real(dt, tol):
    n = 64; half = 32
    ore = np.zeros(half + 1, dt); oim = np.zeros(half + 1, dt)
    O.r2c_fft(np.arange(1, n + 1, dtype=dt), ore, oim)
    assert abs(oim[0]) < tol and abs(oim[half]) < tol


# --- r2c.rs:979-1131 API-variant equivalences are bit exact; :1134-1165 scratch reuse ------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_r2c_c2r_variants_bit_exact(dt):
    n = 1024; half = n // 2
    x = np.arange(1, n + 1, dtype=dt)
    a_re = np.zeros(half + 1, dt); a_im = np.zeros(half + 1, dt); O.r2c_fft(x, a_re, a_im)
    pl = O.PlannerR2c(n, dt)
    b_re = np.zeros(half + 1, dt); b_im = np.zeros(half + 1, dt); O.r2c_fft(x, b_re, b_im, pl)
    assert np.array_equal(a_re, b_re) and np.array_equal(a_im, b_im)
    y1 = np.zeros(n, dt); O.c2r_fft(a_re, a_im, y1)
    y2 = np.zeros(n, dt); O.c2r_fft(a_re, a_im, y2, pl)
    s_re = np.full(half, 7, dt); s_im = np.full(half, -3, dt)
    y3 = np.zeros(n, dt); O.c2r_fft(a_re, a_im, y3, pl, s_re, s_im)
    assert np.array_equal(y1, y2) and np.array_equal(y1, y3)
    for _ in range(4):  # scratch reuse
        y4 = np.zeros(n, dt); O.c2r_fft(a_re, a_im, y4, pl, s_re, s_im)
        assert np.array_equal(y1, y4)


# --- r2c.rs:1392-1540 panics with the exact messages ----------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_r2c_c2r_panic_messages(dt):
    def z(n):
        return np.zeros(n, dt)
    for bad in (0, 1, 2, 3, 6, 12):
        with pytest.raises(O.OraclePanic, match="n must be a power of 2 >= 4"):
            O.r2c_fft(z(bad), z(bad // 2 + 1), z(bad // 2 + 1))
        with pytest.raises(O.OraclePanic, match="n must be a power of 2 >= 4"):
            O.c2r_fft(z(bad // 2 + 1), z(bad // 2 + 1), z(bad))
        with pytest.raises(O.OraclePanic, match="n must be a power of 2 >= 4"):
            O.PlannerR2c(bad, dt)
    n = 16
    pl = O.PlannerR2c(n, dt)
    with pytest.raises(O.OraclePanic, match="input length must match planner size"):
        O.r2c_fft(z(8), z(9), z(9), pl)
    with pytest.raises(O.OraclePanic, match="output_re must have length N/2 \\+ 1"):
        O.r2c_fft(z(n), z(8), z(9), pl)
    with pytest.raises(O.OraclePanic, match="output_im must have length N/2 \\+ 1"):
        O.r2c_fft(z(n), z(9), z(8), pl)
    with pytest.raises(O.OraclePanic, match="output length must match planner size"):
        O.c2r_fft(z(9), z(9), z(8), pl)
    with pytest.raises(O.OraclePanic, match="input_re must have length N/2 \\+ 1"):
        O.c2r_fft(z(8), z(9), z(n), pl)
    with pytest.raises(O.OraclePanic, match="input_im must have length N/2 \\+ 1"):
        O.c2r_fft(z(9), z(8), z(n), pl)
    with pytest.raises(O.OraclePanic, match="scratch_re must have length N/2"):
        O.c2r_fft(z(9), z(9), z(n), pl, z(7), z(8))
    with pytest.raises(O.OraclePanic, match="scratch_im must have length N/2"):
        O.c2r_fft(z(9), z(9), z(n), pl, z(8), z(7))


# --- planner.rs:120-162 r2c twiddles: 0.5 * W_N^k by recurrence --------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_r2c_twiddles(dt):
    n = 4096
    w_re, w_im = O.PlannerR2c(n, dt).twiddles()
    k = np.arange(n // 2)
    tol = 1e-13 if dt == np.float64 else 1e-7
    assert np.max(np.abs(w_re - 0.5 * np.cos(2 * np.pi * k / n))) < tol
    assert np.max(np.abs(w_im + 0.5 * np.sin(2 * np.pi * k / n))) < tol
    assert w_re[0] == dt(0.5) and w_im[0] == dt(0.0)


def test_golden_r2c():
    g = np.load(GOLD / "r2c_golden.npz")
    for dt in (np.float64, np.float32):
        eps = np.finfo(dt).eps
        for n in (4, 8, 16, 64, 256, 2048):
            x = g[f"real_{n}_in"].astype(dt)
            ore = np.zeros(n // 2 + 1, dt); oim = np.zeros(n // 2 + 1, dt)
            O.r2c_fft(x, ore, oim)
            err = rel_linf(ore, oim, g[f"real_{n}_out_re"], g[f"real_{n}_out_im"])
            # the reference's recurrence twiddles lose ~log2(N) extra bits (planner.rs:128-138)
            assert err <= 16 * eps * np.log2(n), (dt, n, err)


def test_literal_twiddles_match_reference_source():
    """The 312 decimal twiddle literals of the reference's kernels/dit.rs and codelets.rs (stored as data in
    golden/reference_literal_twiddles.npz by oracle/check_literals.py) equal the oracle's regenerated tables bit for bit."""
    from oracle import check_literals
    tabs = check_literals.load_golden(GOLD / "reference_literal_twiddles.npz")
    assert len(tabs) == 38 and {t[3] for t in tabs} == {"f32", "f64"}
    n_checked, failures = check_literals.compare(tabs)
    assert n_checked == 312
    assert not failures, [f[:3] for f in failures]
