"""Host-side mirror of PhastFT's public API over libphastft_cuda.so.

Same names, argument meaning and error behaviour as the reference crate
(/root/reference/src/lib.rs:33-226, planner.rs, options.rs, algorithms/r2c.rs:521-895), so the
parity tests read like the reference's own tests:

    fft_64_dit(reals, imags, Direction.Forward)          # lib.rs:180
    planner = PlannerDit64(n); fft_64_dit_with_planner(reals, imags, Direction.Reverse, planner)
    r2c_fft_f64(x, out_re, out_im); c2r_fft_f64(out_re, out_im, y)

Arrays: numpy arrays (host slices -> `*_host` entry points: H2D, kernels, D2H, synchronous,
in place) or torch CUDA tensors (device-resident -> `*_dev` entry points on torch's current
stream, asynchronous, nothing copied).  Where the reference panics these raise `PhastFTPanic`
(an AssertionError) whose message starts with the reference's panic text.

The Rust crate that keeps the exact Rust signatures over the same C ABI is rust/src/lib.rs.
"""
from __future__ import annotations

import ctypes as C
import enum
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import PhastFTPanic, check, fn

__all__ = [
    "Direction", "PlannerMode", "Options", "PhastFTPanic",
    "PlannerDit64", "PlannerDit32", "PlannerR2c64", "PlannerR2c32",
    "fft_64_dit", "fft_64_dit_with_planner", "fft_64_dit_with_planner_and_opts",
    "fft_32_dit", "fft_32_dit_with_planner", "fft_32_dit_with_planner_and_opts",
    "fft_64_interleaved", "fft_64_interleaved_with_planner", "fft_64_interleaved_with_planner_and_opts",
    "fft_32_interleaved", "fft_32_interleaved_with_planner", "fft_32_interleaved_with_planner_and_opts",
    "r2c_fft_f64", "r2c_fft_f64_with_planner", "c2r_fft_f64", "c2r_fft_f64_with_planner",
    "c2r_fft_f64_with_planner_and_scratch",
    "r2c_fft_f32", "r2c_fft_f32_with_planner", "c2r_fft_f32", "c2r_fft_f32_with_planner",
    "c2r_fft_f32_with_planner_and_scratch",
    "fft_dit_batch", "fft_dit_batch_sharded", "r2c_fft_batch", "c2r_fft_batch", "host_register", "host_unregister",
]


class Direction(enum.IntEnum):
    """planner.rs:10-16"""
    Forward = 1
    Reverse = -1


class PlannerMode(enum.IntEnum):
    """planner.rs:25-32 (accepted; the reference ignores it, planner.rs:65)"""
    Heuristic = 0
    Tune = 1


@dataclass
class Options:
    """options.rs:10-43.  Hints only on the GPU (kept for source compatibility)."""
    multithreaded_bit_reversal: bool = False
    smallest_parallel_chunk_size: int = 16384

    @staticmethod
    def guess_options(input_size: int) -> "Options":
        o = _lib.Options()
        _lib.lib.phastft_options_guess(int(input_size), C.byref(o))
        return Options(bool(o.multithreaded_bit_reversal), int(o.smallest_parallel_chunk_size))


# ----------------------------------------------------------------------------------------------
# array plumbing
# ----------------------------------------------------------------------------------------------
def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


def _np_ptr(a: np.ndarray, dtype, writable: bool):
    if not isinstance(a, np.ndarray):
        raise TypeError("expected a numpy array or a torch CUDA tensor")
    if a.dtype != dtype:
        raise TypeError(f"expected dtype {np.dtype(dtype)}, got {a.dtype}")
    if a.ndim != 1 or not a.flags.c_contiguous:
        raise ValueError("slices must be 1-D and contiguous")
    if writable and not a.flags.writeable:
        raise ValueError("output slice is read-only")
    return a.ctypes.data_as(C.c_void_p), a.size


def _torch_ptr(t, dtype):
    import torch
    want = torch.float64 if np.dtype(dtype) == np.float64 else torch.float32
    if not t.is_cuda:
        raise TypeError("torch tensors must live on a CUDA device (use numpy arrays for host slices)")
    if t.dtype != want or t.dim() != 1 or not t.is_contiguous():
        raise TypeError("expected a contiguous 1-D tensor of the planner's precision")
    return C.c_void_p(t.data_ptr()), t.numel()


def _torch_stream(t):
    import torch
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


# ----------------------------------------------------------------------------------------------
# planners
# ----------------------------------------------------------------------------------------------
class _PlannerDit:
    _sfx = ""
    _dtype = None

    def __init__(self, num_points: int, device: int = 0, mode: PlannerMode = PlannerMode.Heuristic):
        """PlannerDit{64,32}::new / with_mode (planner.rs:55-100): panics unless num_points is a
        non-zero power of two."""
        self._h = C.c_void_p()
        self.device = int(device)
        check(fn("phastft_plan_dit_{s}_create", self._sfx)(int(num_points), self.device, int(mode), C.byref(self._h)))
        self.num_points = int(num_points)

    @classmethod
    def new(cls, num_points: int, device: int = 0):
        return cls(num_points, device)

    @classmethod
    def with_mode(cls, num_points: int, mode: PlannerMode, device: int = 0):
        return cls(num_points, device, mode)

    def describe(self) -> str:
        return fn("phastft_plan_dit_{s}_describe", self._sfx)(self._h).decode()

    # planner-table blob, for the one init-time broadcast of a multi-GPU job
    def reserve(self, batch: int) -> None:
        """Size the device workspace for calls of up to `batch` transforms now (otherwise the first larger call grows
        it, synchronising the device -- an error inside a CUDA-graph capture)."""
        check(fn("phastft_plan_dit_{s}_reserve", self._sfx)(self._h, int(batch)))

    def tables_bytes(self) -> int:
        return int(fn("phastft_plan_dit_{s}_tables_bytes", self._sfx)(self._h))

    def tables_export(self, dst_tensor) -> None:
        check(fn("phastft_plan_dit_{s}_tables_export", self._sfx)(self._h, C.c_void_p(dst_tensor.data_ptr()),
                                                                  _torch_stream(dst_tensor)))

    def tables_import(self, src_tensor) -> None:
        check(fn("phastft_plan_dit_{s}_tables_import", self._sfx)(self._h, C.c_void_p(src_tensor.data_ptr()),
                                                                  _torch_stream(src_tensor)))

    def broadcast_tables(self, src: int = 0, group=None) -> None:
        """One collective at init: rank `src`'s twiddle tables to every rank (torch.distributed,
        NCCL on GPUs).  After this no call communicates."""
        import torch
        import torch.distributed as dist
        buf = torch.empty(self.tables_bytes(), dtype=torch.uint8, device=f"cuda:{self.device}")
        self.tables_export(buf)
        dist.broadcast(buf, src=src, group=group)
        self.tables_import(buf)
        torch.cuda.current_stream(buf.device).synchronize()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._h = None
            try:
                fn("phastft_plan_dit_{s}_destroy", self._sfx)(h)
            except (AttributeError, TypeError):      # interpreter shutdown: the module globals are already gone
                pass


class PlannerDit64(_PlannerDit):
    _sfx, _dtype = "f64", np.float64


class PlannerDit32(_PlannerDit):
    _sfx, _dtype = "f32", np.float32


class _PlannerR2c:
    _sfx = ""
    _dtype = None

    def __init__(self, n: int, device: int = 0):
        """PlannerR2c{64,32}::new (planner.rs:194-206): panics with "n must be a power of 2 >= 4"."""
        self._h = C.c_void_p()
        self.device = int(device)
        check(fn("phastft_plan_r2c_{s}_create", self._sfx)(int(n), self.device, C.byref(self._h)))
        self.n = int(n)

    @classmethod
    def new(cls, n: int, device: int = 0):
        return cls(n, device)

    def reserve(self, batch: int) -> None:
        """Size the workspace of the half-length transform for r2c_fft_batch / c2r_fft_batch calls of up to `batch`
        members now (otherwise the first larger call grows it, synchronising the device -- an error inside a CUDA-graph
        capture)."""
        check(fn("phastft_plan_r2c_{s}_reserve", self._sfx)(self._h, int(batch)))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._h = None
            try:
                fn("phastft_plan_r2c_{s}_destroy", self._sfx)(h)
            except (AttributeError, TypeError):      # interpreter shutdown: the module globals are already gone
                pass


class PlannerR2c64(_PlannerR2c):
    _sfx, _dtype = "f64", np.float64


class PlannerR2c32(_PlannerR2c):
    _sfx, _dtype = "f32", np.float32


# The convenience functions plan per call like the reference (lib.rs:180-183); building a plan and allocating its workspace
# per call costs far more than the transform, and destroying a plan while its kernels are still queued relies on cudaFree's
# implicit synchronisation -- so the most recent one-shot planner per (class, size, device) is kept, like the C library
# does for host slices (phastft_*_oneshot).
_ONESHOT_PLANNERS: dict = {}


def _oneshot_planner(cls, n: int, device: int):
    key = (cls.__name__, device)
    hit = _ONESHOT_PLANNERS.get(key)
    if hit is not None and hit[0] == n:
        return hit[1]
    planner = cls(n, device)           # raises the reference's panic for an invalid size before anything is cached
    if hit is not None and _is_torch_available():
        import torch
        torch.cuda.synchronize(device)     # the replaced planner may still have work queued
    _ONESHOT_PLANNERS[key] = (n, planner)
    return planner


def _is_torch_available() -> bool:
    try:
        import torch  # noqa: F401
        return True
    except Exception:  # noqa: BLE001
        return False


def oneshot_cache_clear() -> None:
    """Drop the planners kept for the convenience functions (here and inside the C library)."""
    _ONESHOT_PLANNERS.clear()
    _lib.lib.phastft_oneshot_cache_clear()


# ----------------------------------------------------------------------------------------------
# c2c
# ----------------------------------------------------------------------------------------------
def _fft_dit_with_planner(sfx, dtype, reals, imags, direction, planner, opts=None):
    if planner._sfx != sfx:
        raise TypeError("planner precision does not match the function")
    if _is_torch(reals):
        pr, nr = _torch_ptr(reals, dtype)
        pi, ni = _torch_ptr(imags, dtype)
        # the asserts of algorithms/dit.rs:284-289, in the reference's order
        if nr != ni:
            raise PhastFTPanic(1)
        if nr == 0 or nr & (nr - 1):
            raise PhastFTPanic(2)
        if nr != planner.num_points:
            raise PhastFTPanic(3)
        check(fn("phastft_fft_dit_{s}_dev", sfx)(planner._h, pr, pi, int(direction), 1, nr, _torch_stream(reals)))
    else:
        pr, nr = _np_ptr(reals, dtype, True)
        pi, ni = _np_ptr(imags, dtype, True)
        o = None
        if opts is not None:
            o = _lib.Options(int(opts.multithreaded_bit_reversal), int(opts.smallest_parallel_chunk_size))
        check(fn("phastft_fft_dit_{s}_host", sfx)(planner._h, pr, nr, pi, ni, int(direction),
                                                  C.byref(o) if o is not None else None))


def _fft_dit(sfx, dtype, planner_cls, reals, imags, direction, device=0):
    # lib.rs:180-183: a planner per call
    if not _is_torch(reals):
        # host slices: the library's one-shot entry (it keeps the latest plan for the next same-size call)
        pr, nr = _np_ptr(reals, dtype, True)
        pi, ni = _np_ptr(imags, dtype, True)
        check(fn("phastft_fft_dit_{s}_oneshot", sfx)(pr, nr, pi, ni, int(direction), int(device)))
        return
    planner = _oneshot_planner(planner_cls, reals.numel(), reals.device.index or 0)
    _fft_dit_with_planner(sfx, dtype, reals, imags, direction, planner)


def fft_64_dit(reals, imags, direction: Direction, device: int = 0) -> None:
    """lib.rs:180"""
    _fft_dit("f64", np.float64, PlannerDit64, reals, imags, direction, device)


def fft_64_dit_with_planner(reals, imags, direction: Direction, planner: PlannerDit64) -> None:
    """lib.rs:143"""
    _fft_dit_with_planner("f64", np.float64, reals, imags, direction, planner)


def fft_64_dit_with_planner_and_opts(reals, imags, direction: Direction, planner: PlannerDit64, opts: Options) -> None:
    """algorithms/dit.rs:263"""
    _fft_dit_with_planner("f64", np.float64, reals, imags, direction, planner, opts)


def fft_32_dit(reals, imags, direction: Direction, device: int = 0) -> None:
    """lib.rs:223"""
    _fft_dit("f32", np.float32, PlannerDit32, reals, imags, direction, device)


def fft_32_dit_with_planner(reals, imags, direction: Direction, planner: PlannerDit32) -> None:
    """lib.rs:186"""
    _fft_dit_with_planner("f32", np.float32, reals, imags, direction, planner)


def fft_32_dit_with_planner_and_opts(reals, imags, direction: Direction, planner: PlannerDit32, opts: Options) -> None:
    """algorithms/dit.rs:338"""
    _fft_dit_with_planner("f32", np.float32, reals, imags, direction, planner, opts)


def fft_dit_batch(reals, imags, direction: Direction, planner, batch: int, batch_stride: int | None = None) -> None:
    """Batched device-resident transform: `batch` signals of planner.num_points, transform b at
    offset b*batch_stride of the planar torch CUDA tensors.  (The reference has no batch API; a
    batch is a caller loop sharing one planner, examples/benchmark.rs:24-36.)"""
    n = planner.num_points
    stride = n if batch_stride is None else int(batch_stride)
    pr, nr = _torch_ptr(reals, planner._dtype)
    pi, ni = _torch_ptr(imags, planner._dtype)
    if nr != ni:
        raise PhastFTPanic(1)
    if batch < 1 or nr < (batch - 1) * stride + n:
        raise PhastFTPanic(13, "tensors shorter than batch * batch_stride")
    check(fn("phastft_fft_dit_{s}_dev", planner._sfx)(planner._h, pr, pi, int(direction), int(batch), stride,
                                                      _torch_stream(reals)))


def fft_dit_batch_sharded(reals: np.ndarray, imags: np.ndarray, direction: Direction, planners, batch: int,
                          batch_stride: int | None = None) -> None:
    """Host planar batch sharded over several devices from ONE process (one planner per device)."""
    sfx, dtype = planners[0]._sfx, planners[0]._dtype
    n = planners[0].num_points
    stride = n if batch_stride is None else int(batch_stride)
    pr, nr = _np_ptr(reals, dtype, True)
    pi, ni = _np_ptr(imags, dtype, True)
    if nr != ni:
        raise PhastFTPanic(1)
    if nr < (batch - 1) * stride + n:
        raise PhastFTPanic(13, "arrays shorter than batch * batch_stride")
    arr = (C.c_void_p * len(planners))(*[p._h for p in planners])
    check(fn("phastft_fft_dit_{s}_batch_sharded_host", sfx)(arr, len(planners), pr, pi, int(batch), stride, int(direction)))


def _real_batch_args(x_real, planes, planner, batch, real_stride, spec_stride):
    n, half = planner.n, planner.n // 2
    real_stride = n if real_stride is None else int(real_stride)
    spec_stride = half + 1 if spec_stride is None else int(spec_stride)
    px, nx = _torch_ptr(x_real, planner._dtype)
    (pa, na), (pb, nb) = (_torch_ptr(t, planner._dtype) for t in planes)
    if batch < 1 or real_stride < n or spec_stride < half + 1:
        raise PhastFTPanic(13, "batch >= 1, real-side stride >= N and spectrum stride >= N/2 + 1 required")
    if nx < (batch - 1) * real_stride + n:
        raise PhastFTPanic(13, "real tensor shorter than (batch - 1) * stride + N")
    if min(na, nb) < (batch - 1) * spec_stride + half + 1:
        raise PhastFTPanic(13, "spectrum tensors shorter than (batch - 1) * stride + N/2 + 1")
    return px, pa, pb, real_stride, spec_stride


def r2c_fft_batch(x, out_re, out_im, planner, batch: int, in_stride: int | None = None, out_stride: int | None = None) -> None:
    """Batched device-resident r2c: member b reads x[b*in_stride:][:N] and writes bins out_re/out_im[b*out_stride:][:N/2+1]
    (1-D contiguous torch CUDA tensors, strides in elements, defaults N and N/2+1).  in_stride must be even and x's start
    aligned to two elements (the reals are read as complex pairs).  Asynchronous on torch's current stream."""
    px, pr, pi, in_stride, out_stride = _real_batch_args(x, (out_re, out_im), planner, batch, in_stride, out_stride)
    check(fn("phastft_r2c_{s}_dev_batch", planner._sfx)(planner._h, px, pr, pi, int(batch), in_stride, out_stride, _torch_stream(x)))


def c2r_fft_batch(in_re, in_im, out, planner, batch: int, in_stride: int | None = None, out_stride: int | None = None) -> None:
    """Batched device-resident c2r, the inverse of r2c_fft_batch: member b reads bins in_re/in_im[b*in_stride:][:N/2+1]
    (not modified) and writes out[b*out_stride:][:N], normalised so that c2r(r2c(x)) == x.  out_stride must be even and
    out's start aligned to two elements.  No scratch."""
    po, pr, pi, out_stride, in_stride = _real_batch_args(out, (in_re, in_im), planner, batch, out_stride, in_stride)
    check(fn("phastft_c2r_{s}_dev_batch", planner._sfx)(planner._h, pr, pi, po, int(batch), in_stride, out_stride, _torch_stream(out)))


def host_register(array: np.ndarray) -> None:
    """Page-lock a numpy array in place (cudaHostRegister) so the host-slice calls copy at full PCIe speed
    (~52 GB/s instead of ~13 GB/s from pageable memory); undo with host_unregister before freeing it."""
    check(_lib.lib.phastft_host_register(array.ctypes.data_as(C.c_void_p), array.nbytes))


def host_unregister(array: np.ndarray) -> None:
    check(_lib.lib.phastft_host_unregister(array.ctypes.data_as(C.c_void_p)))


# ----------------------------------------------------------------------------------------------
# interleaved Complex<T> API (lib.rs:41-140, feature `complex-nums`)
# ----------------------------------------------------------------------------------------------
def _interleaved(sfx, dtype, cdtype, signal, direction, planner):
    if _is_torch(signal):
        import torch
        if not signal.is_cuda or signal.dtype != (torch.complex128 if sfx == "f64" else torch.complex64):
            raise TypeError("expected a CUDA complex tensor of the planner's precision")
        n = signal.numel()
        if n == 0 or n & (n - 1):
            raise PhastFTPanic(2)
        if n != planner.num_points:
            raise PhastFTPanic(3)
        check(fn("phastft_fft_interleaved_{s}_dev", sfx)(planner._h, C.c_void_p(signal.data_ptr()), int(direction), 1, n,
                                                          _torch_stream(signal)))
    else:
        if signal.dtype != cdtype or signal.ndim != 1 or not signal.flags.c_contiguous:
            raise TypeError(f"expected a contiguous 1-D {np.dtype(cdtype)} array")
        check(fn("phastft_fft_interleaved_{s}_host", sfx)(planner._h, signal.ctypes.data_as(C.c_void_p), signal.size,
                                                           int(direction)))


def fft_64_interleaved_with_planner_and_opts(signal, direction, planner: PlannerDit64, opts: Options | None = None):
    _interleaved("f64", np.float64, np.complex128, signal, direction, planner)


def fft_64_interleaved_with_planner(signal, direction, planner: PlannerDit64):
    _interleaved("f64", np.float64, np.complex128, signal, direction, planner)


def fft_64_interleaved(signal, direction, device: int = 0):
    n = signal.numel() if _is_torch(signal) else signal.size
    _interleaved("f64", np.float64, np.complex128, signal, direction, _oneshot_planner(PlannerDit64, n, device))


def fft_32_interleaved_with_planner_and_opts(signal, direction, planner: PlannerDit32, opts: Options | None = None):
    _interleaved("f32", np.float32, np.complex64, signal, direction, planner)


def fft_32_interleaved_with_planner(signal, direction, planner: PlannerDit32):
    _interleaved("f32", np.float32, np.complex64, signal, direction, planner)


def fft_32_interleaved(signal, direction, device: int = 0):
    n = signal.numel() if _is_torch(signal) else signal.size
    _interleaved("f32", np.float32, np.complex64, signal, direction, _oneshot_planner(PlannerDit32, n, device))


# ----------------------------------------------------------------------------------------------
# r2c / c2r
# ----------------------------------------------------------------------------------------------
def _r2c_with_planner(sfx, dtype, x, out_re, out_im, planner):
    if _is_torch(x):
        px, nx = _torch_ptr(x, dtype)
        pr, nr = _torch_ptr(out_re, dtype)
        pi, ni = _torch_ptr(out_im, dtype)
        half = planner.n // 2
        if nx != planner.n:
            raise PhastFTPanic(5)
        if nr != half + 1:
            raise PhastFTPanic(6)
        if ni != half + 1:
            raise PhastFTPanic(7)
        check(fn("phastft_r2c_{s}_dev", sfx)(planner._h, px, pr, pi, _torch_stream(x)))
    else:
        px, nx = _np_ptr(x, dtype, False)
        pr, nr = _np_ptr(out_re, dtype, True)
        pi, ni = _np_ptr(out_im, dtype, True)
        check(fn("phastft_r2c_{s}_host", sfx)(planner._h, px, nx, pr, nr, pi, ni))


def _c2r_with_planner(sfx, dtype, in_re, in_im, out, planner, scratch_re=None, scratch_im=None):
    if _is_torch(out):
        pr, nr = _torch_ptr(in_re, dtype)
        pi, ni = _torch_ptr(in_im, dtype)
        po, no = _torch_ptr(out, dtype)
        half = planner.n // 2
        if no != planner.n:
            raise PhastFTPanic(8)
        if nr != half + 1:
            raise PhastFTPanic(9)
        if ni != half + 1:
            raise PhastFTPanic(10)
        psr = psi = None
        if scratch_re is not None or scratch_im is not None:
            psr, nsr = _torch_ptr(scratch_re, dtype)
            psi, nsi = _torch_ptr(scratch_im, dtype)
            if nsr != half:
                raise PhastFTPanic(11)
            if nsi != half:
                raise PhastFTPanic(12)
        check(fn("phastft_c2r_{s}_dev", sfx)(planner._h, pr, pi, po, psr, psi, _torch_stream(out)))
    else:
        pr, nr = _np_ptr(in_re, dtype, False)
        pi, ni = _np_ptr(in_im, dtype, False)
        po, no = _np_ptr(out, dtype, True)
        if scratch_re is None and scratch_im is None:
            psr, nsr, psi, nsi = None, 0, None, 0
        else:
            psr, nsr = _np_ptr(scratch_re, dtype, True)
            psi, nsi = _np_ptr(scratch_im, dtype, True)
        check(fn("phastft_c2r_{s}_host", sfx)(planner._h, pr, nr, pi, ni, po, no, psr, nsr, psi, nsi))


def _len(a):
    return a.numel() if _is_torch(a) else a.size


def _dev_of(a, device):
    return (a.device.index or 0) if _is_torch(a) else device


def r2c_fft_f64(input_re, output_re, output_im, device: int = 0) -> None:
    """r2c.rs:521: PlannerR2c64::new(input_re.len()) then the planner path."""
    if not _is_torch(input_re):
        px, nx = _np_ptr(input_re, np.float64, False)
        pr, nr = _np_ptr(output_re, np.float64, True)
        pi, ni = _np_ptr(output_im, np.float64, True)
        check(fn("phastft_r2c_{s}_oneshot", "f64")(px, nx, pr, nr, pi, ni, int(device)))
        return
    _r2c_with_planner("f64", np.float64, input_re, output_re, output_im, _oneshot_planner(PlannerR2c64, _len(input_re), _dev_of(input_re, device)))


def r2c_fft_f64_with_planner(input_re, output_re, output_im, planner: PlannerR2c64) -> None:
    """r2c.rs:535"""
    _r2c_with_planner("f64", np.float64, input_re, output_re, output_im, planner)


def c2r_fft_f64(input_re, input_im, output, device: int = 0) -> None:
    """r2c.rs:695: PlannerR2c64::new(output.len())"""
    if not _is_torch(output):
        pr, nr = _np_ptr(input_re, np.float64, False)
        pi, ni = _np_ptr(input_im, np.float64, False)
        po, no = _np_ptr(output, np.float64, True)
        check(fn("phastft_c2r_{s}_oneshot", "f64")(pr, nr, pi, ni, po, no, int(device)))
        return
    _c2r_with_planner("f64", np.float64, input_re, input_im, output, _oneshot_planner(PlannerR2c64, _len(output), _dev_of(output, device)))


def c2r_fft_f64_with_planner(input_re, input_im, output, planner: PlannerR2c64) -> None:
    """r2c.rs:708"""
    _c2r_with_planner("f64", np.float64, input_re, input_im, output, planner)


def c2r_fft_f64_with_planner_and_scratch(input_re, input_im, output, planner: PlannerR2c64, scratch_re, scratch_im) -> None:
    """r2c.rs:740"""
    _c2r_with_planner("f64", np.float64, input_re, input_im, output, planner, scratch_re, scratch_im)


def r2c_fft_f32(input_re, output_re, output_im, device: int = 0) -> None:
    """r2c.rs:598"""
    if not _is_torch(input_re):
        px, nx = _np_ptr(input_re, np.float32, False)
        pr, nr = _np_ptr(output_re, np.float32, True)
        pi, ni = _np_ptr(output_im, np.float32, True)
        check(fn("phastft_r2c_{s}_oneshot", "f32")(px, nx, pr, nr, pi, ni, int(device)))
        return
    _r2c_with_planner("f32", np.float32, input_re, output_re, output_im, _oneshot_planner(PlannerR2c32, _len(input_re), _dev_of(input_re, device)))


def r2c_fft_f32_with_planner(input_re, output_re, output_im, planner: PlannerR2c32) -> None:
    """r2c.rs:607"""
    _r2c_with_planner("f32", np.float32, input_re, output_re, output_im, planner)


def c2r_fft_f32(input_re, input_im, output, device: int = 0) -> None:
    """r2c.rs:804"""
    if not _is_torch(output):
        pr, nr = _np_ptr(input_re, np.float32, False)
        pi, ni = _np_ptr(input_im, np.float32, False)
        po, no = _np_ptr(output, np.float32, True)
        check(fn("phastft_c2r_{s}_oneshot", "f32")(pr, nr, pi, ni, po, no, int(device)))
        return
    _c2r_with_planner("f32", np.float32, input_re, input_im, output, _oneshot_planner(PlannerR2c32, _len(output), _dev_of(output, device)))


def c2r_fft_f32_with_planner(input_re, input_im, output, planner: PlannerR2c32) -> None:
    """r2c.rs:813"""
    _c2r_with_planner("f32", np.float32, input_re, input_im, output, planner)


def c2r_fft_f32_with_planner_and_scratch(input_re, input_im, output, planner: PlannerR2c32, scratch_re, scratch_im) -> None:
    """r2c.rs:835"""
    _c2r_with_planner("f32", np.float32, input_re, input_im, output, planner, scratch_re, scratch_im)
