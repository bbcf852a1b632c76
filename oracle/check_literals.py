#!/usr/bin/env python
"""Verify that the oracle's regenerated literal twiddles equal the decimal literals the
reference spells out in src/kernels/dit.rs and src/kernels/codelets.rs.

The numbers are parsed from a checkout of the reference and stored, as data, in
tests/golden/reference_literal_twiddles.npz (nothing else of the reference is kept);
tests/test_oracle.py compares the oracle against that file, so the check needs no reference
checkout.  Result is recorded in DESIGN.md.

Usage: python oracle/check_literals.py REFERENCE_ROOT                  # compare against the sources
       python oracle/check_literals.py REFERENCE_ROOT --write-golden   # (re)write the stored tables
"""
from __future__ import annotations

import re
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import oracle as O  # noqa: E402

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden" / "reference_literal_twiddles.npz"
SOURCES = ("src/kernels/dit.rs", "src/kernels/codelets.rs")

_FN = re.compile(r"fn\s+(fft_dit_chunk_(\d+)_simd_(f32|f64)|fft_dit_codelet_(\d+)_simd_(f32|f64))\s*<")
_ARR = re.compile(r"let\s+(\w+)\s*=\s*(f32|f64)x(\d+)::simd_from\(\s*simd,\s*\[(.*?)\]\s*,?\s*\)", re.S)


def _parse_value(tok: str, ty: str) -> float:
    tok = tok.strip()
    neg = tok.startswith("-")
    if neg:
        tok = tok[1:].strip()
    if "FRAC_1_SQRT_2" in tok:
        v = np.float32(np.sqrt(np.float64(0.5))) if ty == "f32" else np.sqrt(np.float64(0.5))
    else:
        tok = tok.replace("_f32", "").replace("_f64", "").replace("_", "")
        v = np.float32(tok) if ty == "f32" else np.float64(tok)
    return -v if neg else v


def _strip_comments(s: str) -> str:
    return re.sub(r"//[^\n]*", "", s)


def collect(path: Path):
    """Yield (function, array-name, dtype, values) for every simd_from literal array."""
    text = path.read_text()
    fns = [(m.start(), m.group(1)) for m in _FN.finditer(text)]
    fns.append((len(text), None))
    for (start, name), (end, _) in zip(fns, fns[1:]):
        body = text[start:end]
        for m in _ARR.finditer(body):
            var, ty, _lanes, inner = m.groups()
            toks = [t for t in _strip_comments(inner).split(",") if t.strip()]
            if not toks or any(ch.isalpha() and "FRAC" not in t and "f32" not in t and "f64" not in t
                               for t in toks for ch in t.replace("std", "").replace("consts", "")):
                # not a numeric literal table (e.g. simd_from(simd, *tw_re))
                try:
                    vals = [_parse_value(t, ty) for t in toks]
                except ValueError:
                    continue
            else:
                vals = [_parse_value(t, ty) for t in toks]
            yield name, var, ty, vals


def tables(reference_root: str):
    """Every literal table of the reference as (source, function, array, dtype, chunk, part, first index, values):
    the table holds W_chunk^k for k = first index, first index + 1, ..., real part (part "re") or imaginary part ("im")."""
    root = Path(reference_root)
    out = []
    for rel in SOURCES:
        for fn, var, ty, vals in collect(root / rel):
            part = "im" if "_im" in var or var.endswith("im") else "re"
            m = re.search(r"_(\d+)_(\d+)$", var)
            lo = int(m.group(1)) if m else 0
            # which W_chunk table is it?  chunk kernels: from the function name; codelets: from the var/lanes
            mchunk = re.match(r"fft_dit_chunk_(\d+)_simd", fn)
            if mchunk:
                chunk = int(mchunk.group(1))
            else:
                # codelets: tw_re/tw_im with 4 lanes (f64 stage 2) = W_8; tw_lo/tw_hi f64 = W_16 lo/hi;
                # f32: tw_re/tw_im 8 lanes = W_16, tw_lo/tw_hi = W_32
                if ty == "f64":
                    chunk = 8 if var in ("tw_re", "tw_im") else 16
                else:
                    chunk = 16 if var in ("tw_re", "tw_im") else 32
                if "_hi_" in var:
                    lo = chunk // 4
            out.append((rel, fn, var, ty, chunk, part, lo, np.array(vals, dtype=np.float32 if ty == "f32" else np.float64)))
    return out


def write_golden(reference_root: str, path: Path = GOLDEN) -> None:
    tabs = tables(reference_root)
    index = np.array([[rel, fn, var, ty, str(chunk), part, str(lo)] for rel, fn, var, ty, chunk, part, lo, _ in tabs])
    np.savez_compressed(path, index=index, **{f"values_{i:03d}": t[-1] for i, t in enumerate(tabs)})
    print(f"wrote {sum(t[-1].size for t in tabs)} literal twiddles of {len(tabs)} tables to {path}")


def load_golden(path: Path = GOLDEN):
    g = np.load(path)
    return [(rel, fn, var, ty, int(chunk), part, int(lo), g[f"values_{i:03d}"])
            for i, (rel, fn, var, ty, chunk, part, lo) in enumerate(g["index"])]


def compare(tabs):
    """(number of literals checked, tables that differ from the oracle's regenerated twiddles)."""
    n_checked = 0
    failures = []
    for rel, fn, var, ty, chunk, part, lo, got in tabs:
        ere, eim = O.literal_twiddles(chunk, np.float32 if ty == "f32" else np.float64)
        exp = (eim if part == "im" else ere)[lo:lo + got.size]
        n_checked += got.size
        if got.dtype != exp.dtype or not np.array_equal(got, exp):
            failures.append((rel, fn, var, got, exp))
    return n_checked, failures


def check(reference_root: str) -> int:
    n_checked, failures = compare(tables(reference_root))
    for f in failures:
        print("MISMATCH", *f, sep="\n  ")
    print(f"checked {n_checked} literal twiddles against {reference_root}: "
          f"{'ALL EQUAL' if not failures else str(len(failures)) + ' arrays differ'}")
    return 1 if failures else 0


if __name__ == "__main__":
    if len(sys.argv) < 2:
        sys.exit(__doc__)
    if "--write-golden" in sys.argv[2:]:
        write_golden(sys.argv[1])
    sys.exit(check(sys.argv[1]))
