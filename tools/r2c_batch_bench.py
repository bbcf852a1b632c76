#!/usr/bin/env python
"""Batched r2c / c2r on the device: batches of 2^24 real points, N = 2^4 .. 2^22, f64 and f32.

For each size: device time per batch (CUDA events over a window of >= 0.2 s after warm-up, rotating buffer sets so the
working set exceeds the 126 MB L2), Gpoint/s, and whole-transform bytes (N + 2 (N/2 + 1) values of T per member, both
directions) over time as a fraction of bench.py's copy peak.  r2c runs alternately with the untangle fused into the one-CTA
kernel (default) and with PHASTFT_R2C_FUSE=0 (half-length c2c + untangle sweep).  torch.fft.rfft / irfft on the same batch
is the cuFFT yardstick, and at a few sizes a Python loop of single-signal calls over the same members.

    python tools/r2c_batch_bench.py [--out FILE]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
import phastft_b200 as pf  # noqa: E402
from phastft_b200 import _lib  # noqa: E402

POINTS = 1 << 24
WINDOW_S = 0.2
dev = torch.device("cuda", 0)


def timed(step, nbuf):
    """ms per call of step(i), i rotating over nbuf buffer sets: warm-up, then repeat until the window is >= WINDOW_S"""
    for i in range(2 * nbuf):
        step(i)
    torch.cuda.synchronize()
    reps = nbuf
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            step(i)
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= WINDOW_S * 1e3:
            return ms / reps
        reps = max(reps * 2, int(reps * WINDOW_S * 1.2e3 / max(ms, 1e-3)))


def run_size(sfx, log_n, out):
    dt = torch.float64 if sfx == "f64" else torch.float32
    es = 8 if sfx == "f64" else 4
    n = 1 << log_n; half = n // 2; batch = POINTS // n
    P = pf.PlannerR2c64 if sfx == "f64" else pf.PlannerR2c32
    pl = P(n)
    pl.reserve(batch)
    set_bytes = (batch * n + 2 * batch * (half + 1)) * es
    nbuf = max(2, -(-3 * 126 * 2 ** 20 // set_bytes))
    bufs = []
    for _ in range(nbuf):
        x = torch.rand(batch * n, dtype=dt, device=dev) * 2 - 1
        bufs.append((x, torch.empty(batch * (half + 1), dtype=dt, device=dev), torch.empty(batch * (half + 1), dtype=dt, device=dev),
                     torch.empty(batch * n, dtype=dt, device=dev)))
    r2c = _lib.fn("phastft_r2c_{s}_dev_batch", sfx)
    c2r = _lib.fn("phastft_c2r_{s}_dev_batch", sfx)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def r2c_step(i):
        x, re, im, _ = bufs[i % nbuf]
        _lib.check(r2c(pl._h, C.c_void_p(x.data_ptr()), C.c_void_p(re.data_ptr()), C.c_void_p(im.data_ptr()), batch, n, half + 1, stream))

    def c2r_step(i):
        _, re, im, y = bufs[i % nbuf]
        _lib.check(c2r(pl._h, C.c_void_p(re.data_ptr()), C.c_void_p(im.data_ptr()), C.c_void_p(y.data_ptr()), batch, half + 1, n, stream))

    def rfft_step(i):
        x = bufs[i % nbuf][0]
        torch.fft.rfft(x.view(batch, n), dim=1)

    spec = [torch.fft.rfft(b[0].view(batch, n), dim=1) for b in bufs]

    def irfft_step(i):
        torch.fft.irfft(spec[i % nbuf], n=n, dim=1)

    t = {}
    for rnd in range(2):                 # fused and unfused r2c alternated, twice
        for fuse in ("1", "0"):
            os.environ["PHASTFT_R2C_FUSE"] = fuse
            t.setdefault("r2c" + fuse, []).append(timed(r2c_step, nbuf))
        os.environ.pop("PHASTFT_R2C_FUSE", None)
    t["c2r"] = [timed(c2r_step, nbuf)]
    t["rfft"] = [timed(rfft_step, nbuf)]
    t["irfft"] = [timed(irfft_step, nbuf)]
    peak, _ = bench.peaks()
    gbytes = batch * (n + 2 * (half + 1)) * es / 1e9
    row = {k: min(v) for k, v in t.items()}

    def fmt(ms):
        return f"{ms * 1e3:9.1f} us {POINTS / ms / 1e6:7.2f} Gpt/s {gbytes / (ms / 1e3) / peak:5.2f}"
    line = (f"{sfx} N=2^{log_n:<2d} batch={batch:<8d} r2c fused {fmt(row['r2c1'])} | unfused {fmt(row['r2c0'])} "
            f"| fused/unfused {row['r2c1'] / row['r2c0']:5.2f} | c2r {fmt(row['c2r'])} | torch rfft {row['rfft'] * 1e3:9.1f} us "
            f"irfft {row['irfft'] * 1e3:9.1f} us")
    if log_n in (10, 14, 18):
        x, re, im, y = bufs[0]
        r1 = _lib.fn("phastft_r2c_{s}_dev", sfx)
        c1 = _lib.fn("phastft_c2r_{s}_dev", sfx)
        ptr = (x.data_ptr(), re.data_ptr(), im.data_ptr(), y.data_ptr())

        def loop_r2c(_):
            for b in range(batch):
                _lib.check(r1(pl._h, C.c_void_p(ptr[0] + b * n * es), C.c_void_p(ptr[1] + b * (half + 1) * es),
                              C.c_void_p(ptr[2] + b * (half + 1) * es), stream))

        def loop_c2r(_):
            for b in range(batch):
                _lib.check(c1(pl._h, C.c_void_p(ptr[1] + b * (half + 1) * es), C.c_void_p(ptr[2] + b * (half + 1) * es),
                              C.c_void_p(ptr[3] + b * n * es), None, None, stream))
        line += f" | loop of {batch} single calls: r2c {timed(loop_r2c, 1) * 1e3:9.1f} us c2r {timed(loop_c2r, 1) * 1e3:9.1f} us"
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()
    del bufs, spec, pl
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="4-22")
    args = ap.parse_args()
    lo, hi = (int(v) for v in args.sizes.split("-"))
    out = open(args.out, "w") if args.out else open(os.devnull, "w")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    peak, src = bench.peaks()
    head = (f"# tools/r2c_batch_bench.py: batches of 2^24 real points, CUDA events, window >= {WINDOW_S} s, rotating buffers > L2\n"
            f"# {q.stdout.strip()}\n# copy peak {peak:.0f} GB/s ({src}); fraction = whole-transform bytes / time / peak\n")
    print(head, end="")
    out.write(head)
    for sfx in ("f64", "f32"):
        for log_n in range(lo, hi + 1):
            run_size(sfx, log_n, out)


if __name__ == "__main__":
    main()
