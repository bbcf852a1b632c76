"""ctypes binding of libphastft_cuda.so (the C ABI declared in include/phastft_cuda.h).

There is deliberately no fallback: if the shared library is missing this module raises at
import time, and if no CUDA device is present every call returns PHASTFT_ERR_NO_DEVICE.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
# PHASTFT_LIB: load another build of the same library (tools/experiments/build_variant.py); still no fallback.
LIB_PATH = Path(os.environ["PHASTFT_LIB"]) if os.environ.get("PHASTFT_LIB") else _PKG / "libphastft_cuda.so"

OK = 0
ERR_NO_DEVICE = 102

MESSAGES = {
    1: "assertion `left == right` failed: reals.len() == imags.len()",
    2: "assertion failed: length must be a non-zero power of two",
    3: "assertion `left == right` failed: log_n == planner.log_n",
    4: "n must be a power of 2 >= 4",
    5: "input length must match planner size",
    6: "output_re must have length N/2 + 1",
    7: "output_im must have length N/2 + 1",
    8: "output length must match planner size",
    9: "input_re must have length N/2 + 1",
    10: "input_im must have length N/2 + 1",
    11: "scratch_re must have length N/2",
    12: "scratch_im must have length N/2",
    13: "invalid argument",
    100: "CUDA error",
    101: "NCCL error",
    102: "no CUDA device available (phastft_cuda has no CPU fallback)",
}


class PhastFTPanic(AssertionError):
    """Raised where the reference would `panic!`; str() starts with the reference's message."""

    def __init__(self, code: int, detail: str = ""):
        self.code = code
        msg = MESSAGES.get(code, f"phastft status {code}")
        if detail and detail != msg:
            msg = f"{msg} [{detail}]"
        super().__init__(msg)


def _load():
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). phastft_b200 has no CPU fallback.")
    return C.CDLL(str(LIB_PATH))


lib = _load()

_sz, _vp, _i32, _ci = C.c_size_t, C.c_void_p, C.c_int32, C.c_int

lib.phastft_last_error.restype = C.c_char_p
lib.phastft_version.restype = C.c_char_p
lib.phastft_launch_count.restype = C.c_uint64
lib.phastft_device_count.argtypes = [C.POINTER(_ci)]
lib.phastft_device_count.restype = _i32


class Options(C.Structure):
    _fields_ = [("multithreaded_bit_reversal", C.c_int32), ("smallest_parallel_chunk_size", C.c_size_t)]


lib.phastft_options_default.argtypes = [C.POINTER(Options)]
lib.phastft_options_guess.argtypes = [_sz, C.POINTER(Options)]

# every symbol include/phastft_cuda.h declares, with its signature
SIGNATURES = {
    "phastft_plan_dit_{s}_create": ([_sz, _ci, _ci, C.POINTER(_vp)], _i32),
    "phastft_plan_dit_{s}_destroy": ([_vp], None),
    "phastft_plan_dit_{s}_size": ([_vp], _sz),
    "phastft_plan_dit_{s}_describe": ([_vp], C.c_char_p),
    "phastft_plan_dit_{s}_reserve": ([_vp, _sz], _i32),
    "phastft_plan_dit_{s}_tables_bytes": ([_vp], _sz),
    "phastft_plan_dit_{s}_tables_export": ([_vp, _vp, _vp], _i32),
    "phastft_plan_dit_{s}_tables_import": ([_vp, _vp, _vp], _i32),
    "phastft_plan_dit_{s}_tables_broadcast": ([_vp, _vp, _ci, _vp], _i32),
    "phastft_fft_dit_{s}_host": ([_vp, _vp, _sz, _vp, _sz, _ci, C.POINTER(Options)], _i32),
    "phastft_fft_dit_{s}_oneshot": ([_vp, _sz, _vp, _sz, _ci, _ci], _i32),
    "phastft_fft_dit_{s}_dev": ([_vp, _vp, _vp, _ci, _sz, _sz, _vp], _i32),
    "phastft_fft_dit_{s}_dev_profile": ([_vp, _vp, _vp, _ci, _sz, _sz, _vp, C.POINTER(C.c_float), C.POINTER(_ci)], _i32),
    "phastft_fft_dit_{s}_batch_sharded_host": ([C.POINTER(_vp), _ci, _vp, _vp, _sz, _sz, _ci], _i32),
    "phastft_fft_interleaved_{s}_host": ([_vp, _vp, _sz, _ci], _i32),
    "phastft_fft_interleaved_{s}_dev": ([_vp, _vp, _ci, _sz, _sz, _vp], _i32),
    "phastft_plan_r2c_{s}_create": ([_sz, _ci, C.POINTER(_vp)], _i32),
    "phastft_plan_r2c_{s}_destroy": ([_vp], None),
    "phastft_plan_r2c_{s}_size": ([_vp], _sz),
    "phastft_r2c_{s}_host": ([_vp, _vp, _sz, _vp, _sz, _vp, _sz], _i32),
    "phastft_r2c_{s}_oneshot": ([_vp, _sz, _vp, _sz, _vp, _sz, _ci], _i32),
    "phastft_r2c_{s}_dev": ([_vp, _vp, _vp, _vp, _vp], _i32),
    "phastft_c2r_{s}_host": ([_vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz], _i32),
    "phastft_c2r_{s}_oneshot": ([_vp, _sz, _vp, _sz, _vp, _sz, _ci], _i32),
    "phastft_c2r_{s}_dev": ([_vp, _vp, _vp, _vp, _vp, _vp, _vp], _i32),
    "phastft_r2c_{s}_dev_batch": ([_vp, _vp, _vp, _vp, _sz, _sz, _sz, _vp], _i32),
    "phastft_c2r_{s}_dev_batch": ([_vp, _vp, _vp, _vp, _sz, _sz, _sz, _vp], _i32),
    "phastft_plan_r2c_{s}_reserve": ([_vp, _sz], _i32),
}
def check(code: int):
    if code != OK:
        raise PhastFTPanic(code, (lib.phastft_last_error() or b"").decode())


lib.phastft_host_register.argtypes = [_vp, _sz]
lib.phastft_host_register.restype = _i32
lib.phastft_host_unregister.argtypes = [_vp]
lib.phastft_host_unregister.restype = _i32
lib.phastft_oneshot_cache_clear.argtypes = []
lib.phastft_oneshot_cache_clear.restype = None

lib.phastft_plan_factorization.argtypes = [_sz, _ci, C.POINTER(_ci), C.POINTER(_ci)]
lib.phastft_plan_factorization.restype = _i32


def plan_factorization(n: int, precision_bits: int = 64):
    """Host-only: log2 of the pass sizes the planner uses for an n-point transform."""
    f = (_ci * 3)()
    k = _ci(0)
    check(lib.phastft_plan_factorization(int(n), int(precision_bits), f, C.byref(k)))
    return [f[i] for i in range(k.value)]


GLOBAL_SYMBOLS = ["phastft_host_register", "phastft_host_unregister", "phastft_oneshot_cache_clear", "phastft_plan_factorization", "phastft_last_error", "phastft_version", "phastft_launch_count", "phastft_device_count",
                  "phastft_options_default", "phastft_options_guess"]

for _name, (_args, _res) in SIGNATURES.items():
    for _s in ("f64", "f32"):
        _f = getattr(lib, _name.format(s=_s))
        _f.argtypes = _args
        _f.restype = _res


def fn(name: str, sfx: str):
    return getattr(lib, name.format(s=sfx))




def launch_count() -> int:
    return int(lib.phastft_launch_count())


def device_count() -> int:
    n = _ci(0)
    lib.phastft_device_count(C.byref(n))
    return n.value
