"""bench.py's host-side logic (no GPU): the roofline arithmetic of SURVEY.md 8(d) and the traffic table lookup."""
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def test_roofline_block_is_the_whole_transform_fraction():
    import bench
    n = 1 << 20
    alg = 2 * n * 8 * 2                              # 32 N bytes: each planar f64 array read once and written once
    r = bench.roofline_block("c2c_f64_2p20", alg, ms_per_step=0.020, pass_ms_alone=[0.012, 0.013], hbm_peak=6569.6,
                             peak_src="test", plan_desc="x", units_note="one transform")
    assert abs(r["achieved"] - alg / 20e-6 / 1e9) < 1e-6
    assert abs(r["frac"] - r["achieved"] / 6569.6) < 1e-12
    assert len(r["per_pass"]) == 2 and abs(sum(e["ms"] for e in r["per_pass"]) - 0.020) < 1e-12
    # a k-pass plan: every pass's fraction is above the whole-transform fraction, and 1/sum(1/f_j) gives it back
    fr = r["per_pass_frac"]
    assert all(f > r["frac"] for f in fr)
    assert abs(1.0 / sum(1.0 / f for f in fr) - r["frac"]) < 1e-9


def test_traffic_table_is_json_with_sources():
    import bench
    table, name = bench.traffic_table()
    assert name is not None and isinstance(table, dict)
    for key in ("c2c_f64_2p20", "c2c_f64_2p26", "batch_f32"):
        assert key in table, key
    json.dumps(table)


def test_dump_sample_is_fixed_and_bounded(tmp_path):
    """--dump-outputs: short arrays whole, long ones as the same seeded sample of elements in every run, at most 64 MiB in all."""
    import numpy as np
    import pytest
    import torch
    import bench
    short = torch.arange(1000, dtype=torch.float64)
    assert np.array_equal(bench.dump_sample(short), short.numpy())
    long = torch.arange(1 << 23, dtype=torch.float64)
    a, b = bench.dump_sample(long), bench.dump_sample(long.clone())
    assert a.size == bench.DUMP_MAX_ELEMS and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and a[-1] < long.numel()           # distinct elements, in index order
    bench.write_dump(tmp_path / "d", {"x": a, "y": a.astype(np.float32)})
    assert np.array_equal(np.load(tmp_path / "d" / "x.npy"), a) and np.load(tmp_path / "d" / "y.npy").dtype == np.float32
    with pytest.raises(AssertionError):
        bench.write_dump(tmp_path / "e", {f"x{i}": a for i in range(5)})   # 5 x 16 MiB


def test_criterion_writer_matches_the_overlay_scripts_reader(tmp_path):
    """tools/sweep.py --criterion writes what benches/plot_criterion_overlay.py reads: <group>/<series>/<n>/new/sample.json with
    per-sample iters and total times (ns) and benchmark.json with throughput ElementsAndBytes (benches/common/mod.rs:91-105)."""
    import ast
    import statistics
    src = (ROOT / "tools" / "sweep.py").read_text()
    tree = ast.parse(src)
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "write_id")
    ns = {"json": json, "statistics": statistics, "Path": Path}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "sweep_write_id", "exec"), ns)
    n = 1 << 10
    ns["write_id"](tmp_path, "c2c_forward_f64", "PhastFT-B200 device", n, n, 2 * n * 8, [1000.0, 1100.0, 900.0], [50, 50, 50])
    d = tmp_path / "c2c_forward_f64" / "PhastFT-B200 device" / str(n) / "new"
    sample = json.loads((d / "sample.json").read_text())
    per_iter = [t / i for t, i in zip(sample["times"], sample["iters"])]
    assert sorted(per_iter) == [900.0, 1000.0, 1100.0]
    eb = json.loads((d / "benchmark.json").read_text())["throughput"]["ElementsAndBytes"]
    assert eb == {"elements": n, "bytes": 2 * n * 8}
    assert json.loads((d / "estimates.json").read_text())["median"]["point_estimate"] == 1000.0
