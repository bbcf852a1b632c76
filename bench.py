#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the B200 FFT hot path.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPUs
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Metric (BASELINE.json): Gpoint/s (complex) for a 2^20-point f64 forward FFT, planar re/im.
A "step" is one in-place forward FFT of one 2^20-point signal through
phastft_fft_dit_f64_dev (device-resident, planner built outside the timed region).  Steps
rotate over NBUF distinct signals whose total size exceeds the 126 MB L2, so every step
reads its input from HBM.  With N GPUs every rank transforms its own stream of signals
(the batch of independent transforms is sharded over the ranks, no data-path collective;
the only collective is the init-time broadcast of the planner tables): weak scaling, and
`value` is the whole-job aggregate = N * 2^20 * K / max-over-ranks time.

The same JSON line carries, as `batched`, BASELINE.json's configs[3] (4096 x 2^16 f32 forward, batch
sharded over the N ranks: strong scaling, with a cross-rank bit-exactness check of the shards), so the driver's
1/2/4/8-GPU runs record the curve the north star names.  `--workload batch_f32` measures only that;
`--workload c2c_f64_2p26` and `r2c_f64_2p24` measure configs[2] and configs[4] on one GPU.

Only this file's cpu_baseline / --impl reference legs touch oracle/ (the CPU restatement of the
reference): there it is the thing timed as the CPU baseline, never part of our arm.
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "Gpoint/s (complex) for 2^20 f64 forward FFT"
L2_BYTES = 126 * 1024 * 1024


# ------------------------------------------------------------------------------------------------
def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU baseline = the oracle (C++ restatement of the reference; the Rust reference cannot be built
# in this image: no cargo/rustc, dependencies not vendored -- see DESIGN.md)
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(workload: str, steps: int, warmup: int, budget_s: float):
    """Time the reference algorithm on the host cores with the reference's big-N protocol
    (examples/benchmark.rs:42-63: planner reused, fresh random unit-norm signal per iteration,
    wall clock around exactly one in-place FFT, median).  Returns (value, unit, info dict)."""
    from oracle import oracle as O
    # all host threads the process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm ignores that)
    try:
        threads = len(os.sched_getaffinity(0))
    except AttributeError:
        threads = os.cpu_count() or 1
    O.set_threads(threads)
    if workload == "batch_f32":
        n, dt = 1 << 16, np.float32
    elif workload == "c2c_f64_2p26":
        n, dt = 1 << 26, np.float64
    elif workload == "r2c_f64_2p24":
        n, dt = 1 << 24, np.float64
    else:
        n, dt = 1 << 20, np.float64
    rng = np.random.default_rng(1234)
    results = {}
    t_start = time.perf_counter()
    if workload == "r2c_f64_2p24":
        pl = O.PlannerR2c(n, dt)
        x = rng.uniform(-1, 1, n)
        ore = np.zeros(n // 2 + 1); oim = np.zeros(n // 2 + 1)
        for par in (True, False):
            ts = []
            for it in range(warmup + steps):
                t0 = time.perf_counter()
                O.r2c_fft(x, ore, oim, pl, parallel=par)
                dtm = time.perf_counter() - t0
                if it >= warmup:
                    ts.append(dtm)
                if time.perf_counter() - t_start > budget_s and len(ts) >= 3:
                    break
            results[par] = ts
    else:
        planner = O.PlannerDit(n, dt)
        # the reference's fork-join threading (rayon::join) does not scale to every core count -- the
        # upper stages are single-threaded and spinning idle workers cost on a shared host -- so give it
        # its best shot: time it with several thread counts and with one thread, keep the fastest median
        counts = sorted({c for c in (8, 16, 32, threads) if c <= threads}, reverse=True)
        modes = [(True, c) for c in counts] + [(False, 1)]
        for par, cnt in modes:
            O.set_threads(cnt)
            ts = []
            t_mode = time.perf_counter()
            for it in range(warmup + steps):
                re, im = O.gen_random_signal(n, dt, seed=1234 + it)
                t0 = time.perf_counter()
                O.fft_dit(re, im, O.FORWARD, planner, parallel=par)
                dtm = time.perf_counter() - t0
                if it >= warmup:
                    ts.append(dtm)
                if time.perf_counter() - t_mode > budget_s / len(modes) and len(ts) >= 3:
                    break
            results[(par, cnt)] = ts
        O.set_threads(threads)
        med = {k: statistics.median(ts) for k, ts in results.items() if ts}
        best = min(med, key=med.get)
        t = med[best]
        value = n / t / 1e9
        info = {
            "value": value, "unit": "Gpoint/s", "cores": best[1], "kind": "port",
            "sample": f"{len(results[best])} x one 2^{n.bit_length() - 1}-point {np.dtype(dt).name} forward c2c FFT, planner reused, "
                      f"fresh unit-norm signal per iteration, median; PhastFT-restatement (C++), "
                      f"{'fork-join on ' + str(best[1]) + ' threads' if best[0] else 'single thread'} (fastest of "
                      f"{[('fork-join x' + str(c)) if p_ else 'single' for p_, c in modes]})",
            "ms_per_transform": t * 1e3,
            "ms_by_mode": {(("fork_join_x" + str(c)) if p_ else "single"): round(m * 1e3, 3) for (p_, c), m in med.items()},
            "host_threads": threads,
        }
        return value, "Gpoint/s", info
    med = {par: statistics.median(ts) for par, ts in results.items() if ts}
    best_par = min(med, key=med.get)
    t = med[best_par]
    value = n / t / 1e9
    info = {
        "value": value, "unit": "Gpoint/s", "cores": threads if best_par else 1, "kind": "port",
        "sample": f"{len(results[best_par])} x one 2^{n.bit_length() - 1}-point {np.dtype(dt).name} "
                  f"{'r2c' if workload == 'r2c_f64_2p24' else 'forward c2c'} FFT, planner reused, median; "
                  f"PhastFT-restatement (C++), {'fork-join on ' + str(threads) + ' threads' if best_par else 'single thread (faster than fork-join here)'}",
        "ms_per_transform": t * 1e3,
        "ms_single_thread": med.get(False, float("nan")) * 1e3,
        "ms_all_threads": med.get(True, float("nan")) * 1e3,
        "host_threads": threads,
    }
    return value, "Gpoint/s", info


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    t0 = time.perf_counter()
    value, unit, info = cpu_reference_run(args.workload, args.steps, args.warmup, budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC if args.workload == "c2c_f64_2p20" else f"Gpoint/s ({args.workload})",
        "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": info["ms_per_transform"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if args.workload == "batch_f32" else "f64", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus),
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)
    return 0


def planner_passes(planner) -> int:
    d = planner.describe().split(" || ")[0]
    return 1 if "[fused launch" in d else d.count(" | ") + 1


def workload_config(workload: str, gpus: int):
    if workload == "batch_f32":
        return {"workload": "batch of 4096 x 2^16-point f32 forward FFTs, planar re/im, sharded over ranks (BASELINE.json configs[3])",
                "l2": "input 2 GiB per pass > L2", "parallelism": f"batch sharded x{gpus}, no data-path collective"}
    if workload == "c2c_f64_2p26":
        return {"workload": "single 2^26-point f64 forward FFT, planar re/im (BASELINE.json configs[2])", "l2": "input 1 GiB > L2"}
    if workload == "r2c_f64_2p24":
        return {"workload": "r2c_fft_f64 2^24 real input + c2r round trip (BASELINE.json configs[4])", "l2": "input 128 MiB > L2"}
    return {"workload": "single 2^20-point f64 forward FFT, planar re/im, 1 stream per GPU (BASELINE.json configs[1])",
            "l2": "steps rotate over 16 distinct 16 MiB signals (256 MiB > 126 MB L2): every step reads HBM",
            "parallelism": f"independent transforms sharded x{gpus} (one stream of signals per rank), planner tables broadcast once at init"}


# ------------------------------------------------------------------------------------------------
def traffic_table():
    """Measured DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum from the committed ncu captures)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        f = ROOT / "profiles" / name
        if f.exists():
            try:
                return json.loads(f.read_text()), name
            except Exception:
                pass
    return {}, None


def roofline_block(wl, alg_bytes, ms_per_step, pass_ms_alone, hbm_peak, peak_src, plan_desc, units_note):
    """SURVEY.md 8(d): achieved = algorithmic bytes of the WHOLE transform (each planar array read once and written once)
    / its time; frac = achieved / measured peak.  A k-pass plan moves k x those bytes, so the per-pass view is kept beside it:
    each pass's share of the step time (from per-pass CUDA events) and the same bytes over that time."""
    ach = alg_bytes / (ms_per_step * 1e-3) / 1e9
    table, tname = traffic_table()
    tr = table.get(wl) if isinstance(table, dict) else None
    per_pass = None
    if pass_ms_alone:
        tot = sum(pass_ms_alone) or 1.0
        per_pass = []
        for j, x in enumerate(pass_ms_alone):
            ms = ms_per_step * x / tot          # launch latency seen by events around a lone launch is overlapped in the timed region
            a = alg_bytes / (ms * 1e-3) / 1e9
            e = {"pass": j + 1, "ms": ms, "ms_timed_alone": x, "achieved": a, "frac": a / hbm_peak}
            if isinstance(tr, dict) and isinstance(tr.get("per_pass"), list) and j < len(tr["per_pass"]):
                e["traffic"] = tr["per_pass"][j]
            per_pass.append(e)
    total_traffic = None
    if isinstance(tr, dict):
        total_traffic = tr.get("total")
    elif isinstance(tr, (int, float)):
        total_traffic = tr
    note = None
    if per_pass and any(e["frac"] > 1.0 for e in per_pass):
        note = ("a per-pass fraction above 1 means that pass streams its bytes faster than the copy kernel behind the measured peak did "
                "(the peak is a measured copy bandwidth, not the HBM3e pin rate); the whole-transform `frac` is the roofline figure")
    return {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "note": note,
            "traffic": total_traffic, "traffic_source": (f"profiles/{tname}" if tname and tr is not None else None),
            "peak_source": peak_src, "algorithmic_bytes": alg_bytes, "units": units_note,
            "per_pass": per_pass, "per_pass_frac": [e["frac"] for e in per_pass] if per_pass else None,
            "passes": len(pass_ms_alone) if pass_ms_alone else None, "kernel": plan_desc,
            "definition": "frac = algorithmic bytes of the whole transform (SURVEY.md 8d: 2 arrays x N x sizeof x (read + write)) / step time / measured "
                          "copy peak; per_pass[j].frac = the same bytes / that pass's share of the step time (a k-pass plan is bounded by 1/k overall)"}


class Ctx:
    pass


def setup(args):
    import torch
    import __graft_entry__ as ge
    with contextlib.redirect_stdout(sys.stderr):      # stdout carries exactly one JSON line
        ge.build()
    import phastft_b200 as pf
    from phastft_b200 import _lib
    from phastft_b200.sharding import max_over_ranks, shard_range
    c = Ctx()
    c.torch, c.pf, c.lib, c.shard_range = torch, pf, _lib, shard_range
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.rank = int(os.environ.get("RANK", "0"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if c.world != args.gpus and c.world > 1:
        args.gpus = c.world
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    c.dist = None
    if c.world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=c.rank, world_size=c.world, device_id=c.dev)
        c.dist = dist

    def barrier():
        if c.dist is not None:
            c.dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        return max_over_ranks(x, device=c.dev) if c.dist is not None else x
    c.barrier, c.maxr = barrier, maxr
    c.hbm_peak, c.peak_src = peaks()
    c.stream = torch.cuda.current_stream(c.dev)
    c.cur_stream = lambda: C.c_void_p(torch.cuda.current_stream(c.dev).cuda_stream)   # inside a graph capture: the capture stream
    c.gen = torch.Generator(device=c.dev)
    c.gen.manual_seed(1234 + c.rank)
    return c


def timed(c, step, K, graph=None, group=1, graph_rem=None):
    """EXACTLY K steps between barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks."""
    torch = c.torch
    c.barrier()
    launches0 = c.pf.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(c.stream)
    if graph is not None:
        for _ in range(K // group):
            graph.replay()
        if K % group:
            if graph_rem is not None:
                graph_rem.replay()
            else:
                for i in range(K % group):
                    step(i)
    else:
        for i in range(K):
            step(i)
    ev1.record(c.stream)
    torch.cuda.synchronize()
    launched = c.pf.launch_count() - launches0
    ms_total = c.maxr(ev0.elapsed_time(ev1))
    c.barrier()
    return ms_total / K, launched


DUMP_MAX_ELEMS = 1 << 21                  # per dumped array: at most 16 MiB of f64 / 8 MiB of f32
DUMP_MAX_BYTES = 64 * 1024 * 1024


def dump_sample(t, seed=1234):
    """A 1-D device tensor as a host array: whole up to DUMP_MAX_ELEMS elements, else a fixed seeded sample of its
    elements in index order (the same indices in every run of the same workload)."""
    import torch
    if t.numel() <= DUMP_MAX_ELEMS:
        return t.cpu().numpy()
    idx = np.sort(np.random.default_rng(seed).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
    return t[torch.from_numpy(idx).to(t.device)].cpu().numpy()


def write_dump(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, total
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(d / f"{name}.npy", a)
    print(f"[bench] dumped {sorted(arrays)} ({total / 2**20:.1f} MiB) to {d}", file=sys.stderr, flush=True)


def per_pass_times(c, sfx, planner, get, batch, n, reps):
    fprof = c.lib.fn("phastft_fft_dit_{s}_dev_profile", sfx)
    pass_ms = (C.c_float * 3)()
    npass = C.c_int(0)
    acc = None
    for i in range(reps):
        a, b = get(i)
        c.lib.check(fprof(planner._h, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), 1, batch, n, c.cur_stream(), pass_ms, C.byref(npass)))
        cur = [pass_ms[j] for j in range(npass.value)]
        acc = cur if acc is None else [x + y for x, y in zip(acc, cur)]
    return [x / reps for x in acc]


# ---- C4: 4096 x 2^16 f32, sharded over the ranks (strong scaling), the reference's caller loop examples/benchmark.rs:24-36 ----
def measure_batch(c, K, W, with_e2e=True, dump=None):
    """`dump`: a dict that receives, as batch_f32_re / batch_f32_im [transforms, 2^16], a fixed seeded sample of the
    transforms the last timed step computes from the seeded inputs."""
    torch, pf, _lib = c.torch, c.pf, c.lib
    n, total = 1 << 16, 4096
    lo, hi = c.shard_range(total, c.rank, c.world)
    nb = hi - lo
    planner = pf.PlannerDit32(n, c.local)
    if c.dist is not None:
        planner.broadcast_tables(src=0)          # the one collective: every rank computes with rank 0's tables
    planner.reserve(nb)
    # the 4096 x 2^16 values come from ONE seeded stream, so shard contents do not depend on the number of ranks (SURVEY.md 8d)
    g = torch.Generator(device=c.dev)
    g.manual_seed(1234)
    # (generating the whole 2 x 1 GiB batch on every rank and slicing keeps the contents rank-count independent)
    full_re = torch.rand(total * n, dtype=torch.float32, device=c.dev, generator=g) * 2 - 1
    full_im = torch.rand(total * n, dtype=torch.float32, device=c.dev, generator=g) * 2 - 1
    re = full_re[lo * n:hi * n].clone(); im = full_im[lo * n:hi * n].clone()
    # every step transforms the shard in place, so after a few steps it holds inf / NaN; the dumped step starts again from a copy
    seeded = (re.clone(), im.clone()) if dump is not None else None
    f = _lib.fn("phastft_fft_dit_{s}_dev", "f32")

    def step(i):
        _lib.check(f(planner._h, C.c_void_p(re.data_ptr()), C.c_void_p(im.data_ptr()), 1, nb, n, c.cur_stream()))

    # ---- shard parity: two transforms from each end of every rank's shard, recomputed on rank 0 from the seeded inputs with
    # the same batched entry point (same kernels: a deterministic library must reproduce them bit for bit) ----
    step(0)
    torch.cuda.synchronize()
    picks = sorted({0, 1, nb - 2, nb - 1} & set(range(nb)))
    mine = torch.stack([torch.stack([re[k * n:(k + 1) * n], im[k * n:(k + 1) * n]]) for k in picks])       # [<=4, 2, n]
    if c.dist is not None:
        gathered = [torch.empty_like(mine) for _ in range(c.world)]
        c.dist.all_gather(gathered, mine)
    else:
        gathered = [mine]
    parity = None
    if c.rank == 0:
        idx = []
        for r in range(c.world):
            rlo, rhi = c.shard_range(total, r, c.world)
            idx += [rlo + k for k in sorted({0, 1, rhi - rlo - 2, rhi - rlo - 1} & set(range(rhi - rlo)))]
        slots = max(128, len(idx))                                     # >= 32 MiB per array: the call takes the same kernels as the shards (TMA pair)
        chk_re = torch.zeros(slots * n, dtype=torch.float32, device=c.dev); chk_im = torch.zeros_like(chk_re)
        for j, k in enumerate(idx):
            chk_re[j * n:(j + 1) * n] = full_re[k * n:(k + 1) * n]; chk_im[j * n:(j + 1) * n] = full_im[k * n:(k + 1) * n]
        _lib.check(f(planner._h, C.c_void_p(chk_re.data_ptr()), C.c_void_p(chk_im.data_ptr()), 1, slots, n, c.cur_stream()))
        torch.cuda.synchronize()
        got = torch.cat([g_.to(c.dev) for g_ in gathered])               # [len(idx), 2, n]
        ok = all(bool(torch.equal(chk_re[j * n:(j + 1) * n], got[j][0])) and bool(torch.equal(chk_im[j * n:(j + 1) * n], got[j][1])) for j in range(len(idx)))
        parity = {"checked_transforms": len(idx), "bit_exact": ok,
                  "what": "two transforms from each end of every rank's shard, gathered to rank 0 and recomputed there from the seeded inputs"}
        del chk_re, chk_im
    del full_re, full_im
    for i in range(W):
        step(i)
    torch.cuda.synchronize()
    ms_per_step, launched = timed(c, step, K)
    if seeded is not None:
        re.copy_(seeded[0]); im.copy_(seeded[1])
        del seeded
        step(K - 1)
        torch.cuda.synchronize()
        picks = np.sort(np.random.default_rng(1234).choice(nb, min(nb, DUMP_MAX_ELEMS // n), replace=False))
        rows = torch.from_numpy(picks).to(c.dev)
        dump["batch_f32_re"] = re.view(nb, n)[rows].cpu().numpy()
        dump["batch_f32_im"] = im.view(nb, n)[rows].cpu().numpy()
    value = total * n / (ms_per_step * 1e-3) / 1e9
    alone = per_pass_times(c, "f32", planner, lambda b: (re, im), nb, n, 5)
    alg = 2 * n * 4 * 2 * nb                   # this rank's shard; the fraction is per GPU (every rank streams its own HBM)
    roof = roofline_block("batch_f32", alg, ms_per_step, alone, c.hbm_peak, c.peak_src, planner.describe(),
                          f"per GPU: {nb} transforms x 16 N bytes")
    out = {"metric": "Gpoint/s (complex), batch of 4096 x 2^16-point f32 forward FFTs sharded over the ranks", "value": value, "unit": "Gpoint/s",
           "ms_per_step": ms_per_step, "steps": K, "warmup": W, "scaling": "strong", "transforms_per_rank": nb, "gpu_launches": int(launched),
           "roofline": roof, "shard_parity": parity, "plan": planner.describe()}
    if with_e2e:
        h_re = torch.empty(nb * n, dtype=torch.float32).pin_memory(); h_im = torch.empty_like(h_re).pin_memory()
        h_re.uniform_(-1, 1); h_im.uniform_(-1, 1)
        a_re, a_im = h_re.numpy(), h_im.numpy()
        fh = _lib.fn("phastft_fft_dit_{s}_batch_sharded_host", "f32")
        arr = (C.c_void_p * 1)(planner._h)

        def host_step():
            _lib.check(fh(arr, 1, a_re.ctypes.data_as(C.c_void_p), a_im.ctypes.data_as(C.c_void_p), nb, n, 1))
        host_step()
        c.barrier()
        ke = 3
        t0 = time.perf_counter()
        for _ in range(ke):
            host_step()
        t_e = c.maxr(time.perf_counter() - t0)
        c.barrier()
        out["e2e"] = {"value": total * n / (t_e / ke) / 1e9, "unit": "Gpoint/s", "h2d_bytes_per_step": 2 * nb * n * 4, "d2h_bytes_per_step": 2 * nb * n * 4,
                      "ms_per_step": t_e / ke * 1e3, "steps": ke,
                      "api": "phastft_fft_dit_f32_batch_sharded_host (one call per step: the rank's whole shard, 3-slot H2D/FFT/D2H pipeline), pinned host memory"}
    return out, planner


def run_ours(args):
    c = setup(args)
    torch, pf, _lib = c.torch, c.pf, c.lib
    world, rank, local, dev = c.world, c.rank, c.local, c.dev
    K, W = args.steps, max(args.warmup, 3)
    wl = args.workload
    sampler = ClockSampler(local)
    sampler.start()
    extra = {}
    roofline = e2e = None
    dump = {} if args.dump_outputs else None

    if wl == "batch_f32":
        out, planner = measure_batch(c, K, W, with_e2e=True, dump=dump)
        clocks = sampler.stop()
        if rank == 0 and dump is not None:
            write_dump(args.dump_outputs, dump)
        cpu = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            _, _, cpu = cpu_reference_run(wl, steps=30, warmup=2, budget_s=25.0)
        if rank == 0:
            line = {"metric": f"Gpoint/s ({wl})", "value": out["value"], "unit": "Gpoint/s", "n_gpus": world, "steps": K, "warmup": W,
                    "ms_per_step": out["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                    "data": "synthetic", "config": workload_config(wl, world), "clocks": clocks, "e2e": out.get("e2e"),
                    "gpu_launches": out["gpu_launches"], "roofline": out["roofline"], "shard_parity": out["shard_parity"], "cpu_baseline": cpu,
                    "plan": out["plan"]}
            print(json.dumps(line), flush=True)
        if c.dist is not None:
            c.dist.destroy_process_group()
        return 0

    if wl in ("c2c_f64_2p20", "c2c_f64_2p26"):
        n = 1 << (20 if wl == "c2c_f64_2p20" else 26)
        planner = pf.PlannerDit64(n, local)
        if c.dist is not None:
            planner.broadcast_tables(src=0)          # the one collective of the whole job
        nbuf = 16 if n == (1 << 20) else 2
        bufs_re = [(torch.rand(n, dtype=torch.float64, device=dev, generator=c.gen) * 2 - 1) for _ in range(nbuf)]
        bufs_im = [(torch.rand(n, dtype=torch.float64, device=dev, generator=c.gen) * 2 - 1) for _ in range(nbuf)]
        f = _lib.fn("phastft_fft_dit_{s}_dev", "f64")

        def step(i):
            b = i % nbuf
            _lib.check(f(planner._h, C.c_void_p(bufs_re[b].data_ptr()), C.c_void_p(bufs_im[b].data_ptr()), 1, 1, n, c.cur_stream()))

        def reset():
            for b in range(nbuf):
                bufs_re[b].uniform_(-1, 1, generator=c.gen); bufs_im[b].uniform_(-1, 1, generator=c.gen)
        points_per_step = n
        alg_bytes = 2 * n * 8 * 2                     # each planar array read once + written once (SURVEY.md 8d)
        dtype = "f64"
        units_note = "one transform: 32 N bytes"
    elif wl == "r2c_f64_2p24":
        n = 1 << 24
        planner = pf.PlannerR2c64(n, local)
        x = torch.rand(n, dtype=torch.float64, device=dev, generator=c.gen) * 2 - 1
        y = torch.empty_like(x)
        sre = torch.empty(n // 2 + 1, dtype=torch.float64, device=dev); sim = torch.empty_like(sre)
        scr_re = torch.empty(n // 2, dtype=torch.float64, device=dev); scr_im = torch.empty_like(scr_re)

        def step(i):
            pf.r2c_fft_f64_with_planner(x, sre, sim, planner)
            pf.c2r_fft_f64_with_planner_and_scratch(sre, sim, y, planner, scr_re, scr_im)

        def reset():
            pass
        points_per_step = n
        # SURVEY.md 8(d): r2c reads 8 N and writes 2 x 8 (N/2 + 1); c2r the reverse
        alg_bytes = 2 * (8 * n + 16 * (n // 2 + 1))
        dtype = "f64"
        units_note = "one r2c + one c2r of 2^24 reals: 2 x (8 N + 16 (N/2 + 1)) bytes"
    else:
        raise SystemExit(f"unknown workload {wl}")

    # ---- warm-up, then EXACTLY K timed steps between barrier+synchronize -------------------------
    for i in range(W):
        step(i)
    torch.cuda.synchronize()
    # The 2^20 step is ~19 us of GPU work issued by one C-ABI call (2 kernel launches): capture the rotation over the NBUF
    # signals into a CUDA graph (and the K mod NBUF leftover steps into a second one) so the host launch path is never the bottleneck.
    graph, group, graph_rem = None, 1, None
    if wl == "c2c_f64_2p20" and not args.no_graph:
        group = nbuf
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(group):
                step(i)
        if K % group:
            graph_rem = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph_rem):
                for i in range(K % group):
                    step(i)
        torch.cuda.synchronize()
    # extra untimed load (~0.3 s) so the clocks are at their loaded level when timing starts
    t_pre = time.perf_counter()
    while time.perf_counter() - t_pre < 0.3:
        if graph is not None:
            graph.replay()
        else:
            step(0)
        torch.cuda.synchronize()
    reset()
    seeded = None
    if dump is not None and wl != "r2c_f64_2p24":
        # the c2c steps transform their buffers in place, so after ~100 passes over a buffer it holds inf / NaN: keep the last
        # step's seeded input and run that step once more from it after the timed loop
        last = (K - 1) % nbuf
        seeded = (bufs_re[last].clone(), bufs_im[last].clone())
    ms_per_step, launches = timed(c, step, K, graph, group, graph_rem)
    if graph is not None:
        launches += K * planner_passes(planner)          # graph replays launch kernels without entering the library
    if dump is not None:
        if seeded is not None:
            bufs_re[last].copy_(seeded[0]); bufs_im[last].copy_(seeded[1])
            del seeded
            step(K - 1)
            torch.cuda.synchronize()
            dump["c2c_re"], dump["c2c_im"] = dump_sample(bufs_re[last]), dump_sample(bufs_im[last])
        else:
            torch.cuda.synchronize()
            dump["r2c_re"], dump["r2c_im"], dump["c2r_out"] = dump_sample(sre), dump_sample(sim), dump_sample(y)
    value = world * points_per_step / (ms_per_step * 1e-3) / 1e9

    # ---- roofline: whole-transform fraction from the timed region; per-pass split from CUDA events, live, on the launching stream ----
    alone = None
    if wl != "r2c_f64_2p24":
        reset()
        alone = per_pass_times(c, "f64", planner, lambda b: (bufs_re[b % nbuf], bufs_im[b % nbuf]), 1, n, 40 if wl == "c2c_f64_2p20" else 10)
    roofline = roofline_block(wl, alg_bytes, ms_per_step, alone, c.hbm_peak, c.peak_src,
                              planner.describe() if hasattr(planner, "describe") else "r2c: half-length c2c passes + untangle; c2r: preprocess + passes", units_note)

    # ---- e2e: the reference-facing host-slice call, pinned host buffers, H2D + D2H inside the timed region ----
    if wl in ("c2c_f64_2p20", "c2c_f64_2p26"):
        h_re = torch.empty(n, dtype=torch.float64).pin_memory(); h_im = torch.empty_like(h_re).pin_memory()
        h_re.uniform_(-1, 1); h_im.uniform_(-1, 1)
        a_re, a_im = h_re.numpy(), h_im.numpy()
        pristine = (a_re.copy(), a_im.copy())

        def host_step():
            pf.fft_64_dit_with_planner(a_re, a_im, pf.Direction.Forward, planner)
        bytes_one_way = 2 * n * 8
        ke = max(5, min(K, 30))
        for _ in range(3):
            host_step()
        a_re[:] = pristine[0]; a_im[:] = pristine[1]
        c.barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            host_step()                      # synchronous: returns after the D2H copy has landed
        t_e = c.maxr(time.perf_counter() - t0)
        c.barrier()
        e2e = {"value": world * n / (t_e / ke) / 1e9, "unit": "Gpoint/s", "h2d_bytes_per_step": bytes_one_way,
               "d2h_bytes_per_step": bytes_one_way, "ms_per_step": t_e / ke * 1e3, "steps": ke,
               "api": "phastft_fft_dit_f64_host (= fft_64_dit_with_planner on host slices; one synchronous call per step), pinned host memory"}
        if wl == "c2c_f64_2p20":
            # the same job -- a stream of independent 2^20 transforms in host memory -- handed to the library as ONE
            # batched call, so H2D of signal j+1, the FFT of j and D2H of j-1 overlap (both PCIe directions busy)
            nsig = 32
            s_re = torch.empty(nsig * n, dtype=torch.float64).pin_memory(); s_im = torch.empty_like(s_re).pin_memory()
            s_re.uniform_(-1, 1); s_im.uniform_(-1, 1)
            b_re, b_im = s_re.numpy(), s_im.numpy()
            fhb = _lib.fn("phastft_fft_dit_{s}_batch_sharded_host", "f64")
            arr1 = (C.c_void_p * 1)(planner._h)

            def stream_step():
                _lib.check(fhb(arr1, 1, b_re.ctypes.data_as(C.c_void_p), b_im.ctypes.data_as(C.c_void_p), nsig, n, 1))
            stream_step()
            s_re.uniform_(-1, 1); s_im.uniform_(-1, 1)
            c.barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                stream_step()
            t_s = c.maxr(time.perf_counter() - t0)
            c.barrier()
            e2e["pipelined"] = {"value": world * 3 * nsig * n / t_s / 1e9, "unit": "Gpoint/s", "transforms_per_call": nsig,
                                "ms_per_transform": t_s / (3 * nsig) * 1e3,
                                "api": "phastft_fft_dit_f64_batch_sharded_host: 32 host-resident 2^20 signals per call, 3-slot H2D/FFT/D2H pipeline"}
            del s_re, s_im

    # ---- the batched configuration of the north star beside the headline: 4096 x 2^16 f32 sharded over the N ranks ----
    batched = None
    if wl == "c2c_f64_2p20" and not args.no_batched:
        del bufs_re, bufs_im
        torch.cuda.empty_cache()
        batched, _ = measure_batch(c, min(K, 20), 3, with_e2e=True, dump=dump)      # --steps also bounds this leg
    clocks = sampler.stop()
    if rank == 0 and dump is not None:
        write_dump(args.dump_outputs, dump)

    # ---- CPU baseline beside it (rank 0, N = 1 only; bounded sample) ------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, _, cpu = cpu_reference_run(wl, steps=30, warmup=2, budget_s=25.0)

    if rank == 0:
        line = {
            "metric": METRIC if wl == "c2c_f64_2p20" else f"Gpoint/s ({wl})", "value": value, "unit": "Gpoint/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": workload_config(wl, world), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "plan": planner.describe() if hasattr(planner, "describe") else None,
            "batched": batched,
        }
        print(json.dumps(line), flush=True)
    if c.dist is not None:
        c.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default="c2c_f64_2p20", choices=["c2c_f64_2p20", "c2c_f64_2p26", "batch_f32", "r2c_f64_2p24"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every step through the C ABI instead of replaying a captured CUDA graph")
    ap.add_argument("--no-batched", action="store_true", help="skip the 4096 x 2^16 f32 sharded measurement that the default workload adds as `batched`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computes from its seeded inputs as DIR/<name>.npy "
                         "(f32 / f64, at most 64 MiB in all; arrays longer than 2^21 as a fixed seeded sample): c2c_re / c2c_im, "
                         "batch_f32_re / batch_f32_im (a seeded sample of [transforms, 2^16]), r2c_re / r2c_im / c2r_out.  The inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    # defaults sized so the timed region lasts ~0.2-0.5 s (clock sampling needs that) and a run takes < 2 min
    dflt = {"c2c_f64_2p20": (20000, 200), "c2c_f64_2p26": (100, 5), "batch_f32": (100, 5), "r2c_f64_2p24": (200, 10)}[args.workload]
    if args.impl == "reference":
        dflt = {"c2c_f64_2p20": (100, 5), "c2c_f64_2p26": (5, 1), "batch_f32": (500, 20), "r2c_f64_2p24": (10, 1)}[args.workload]
    if args.steps is None:
        args.steps = dflt[0]
    if args.warmup is None:
        args.warmup = dflt[1]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
