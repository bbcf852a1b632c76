"""CPU-only checks of the batched r2c / c2r entry points: argument errors come back as status codes, never a crash, and
without a GPU the library refuses to plan (no CPU fallback)."""
import ctypes

import pytest

INVALID_ARG, NO_DEVICE = 13, 102


@pytest.fixture(scope="module")
def pf():
    import __graft_entry__ as g
    g.build()
    import phastft_b200
    return phastft_b200


@pytest.mark.parametrize("sfx", ["f64", "f32"])
def test_null_plan_is_an_invalid_argument(pf, sfx):
    from phastft_b200._lib import fn
    buf = ctypes.create_string_buffer(1024)
    p = ctypes.cast(buf, ctypes.c_void_p)
    before = pf.launch_count()
    assert fn("phastft_r2c_{s}_dev_batch", sfx)(None, p, p, p, 4, 16, 9, None) == INVALID_ARG
    assert fn("phastft_c2r_{s}_dev_batch", sfx)(None, p, p, p, 4, 9, 16, None) == INVALID_ARG
    assert fn("phastft_plan_r2c_{s}_reserve", sfx)(None, 4) == INVALID_ARG
    assert pf.launch_count() == before


@pytest.mark.parametrize("sfx", ["f64", "f32"])
def test_no_device_means_no_plan(pf, sfx):
    if pf.device_count() > 0:
        pytest.skip("a GPU is present")
    from phastft_b200._lib import fn
    h = ctypes.c_void_p()
    assert fn("phastft_plan_r2c_{s}_create", sfx)(64, 0, ctypes.byref(h)) == NO_DEVICE
    assert not h.value
    P = pf.PlannerR2c64 if sfx == "f64" else pf.PlannerR2c32
    with pytest.raises(pf.PhastFTPanic) as e:
        P(64)
    assert e.value.code == NO_DEVICE
    assert pf.launch_count() == 0


def test_public_names(pf):
    for name in ("r2c_fft_batch", "c2r_fft_batch"):
        assert name in pf.api.__all__ and callable(getattr(pf, name))
    assert callable(pf.PlannerR2c64.reserve) and callable(pf.PlannerR2c32.reserve)
