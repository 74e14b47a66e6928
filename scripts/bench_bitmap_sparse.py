#!/usr/bin/env python
"""The sparse bitmap-index layout (value-sorted position lists) on one B200: build time per column, index bytes against
the D * N/8 bytes per-value bitsets would need, and bitmap-scan times of point, range and NE terms, each under the
automatic choice and under both forced forms (scatter, compare), so the crossover between the forms is measured here.
Every scan's result bitmap is compared with mbc_scan's on the same terms in the same run.  Prints one JSON line and
writes it to --out.

Workload (generated on the device, 100 M rows by default, so every column is larger than the 126 MB L2):
  K: all distinct ints (kind 3, domain = rows)   M: 10 M-distinct ints (kind 0)
  S: char(16) (kind 2)                           H: 4-value ints (kind 0): keeps the dense layout

    python scripts/bench_bitmap_sparse.py [--rows 100000000] [--reps 5] [--out profiles/r3/bench_bitmap_sparse.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import mbcol

N = mbcol._native
SEED = 20260101
LAYOUT = {N.BITMAP_NONE: "none", N.BITMAP_DENSE: "dense", N.BITMAP_SPARSE: "sparse"}


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # the numbers are still device times; say what is missing
        return {"name": "unknown", "power_limit": f"not read ({e.__class__.__name__})"}


def forms_taken(fn):
    """Run fn() once with MBC_BM_SPARSE_TRACE set and return the form the library reports for each sparse term."""
    os.environ["MBC_BM_SPARSE_TRACE"] = "1"
    with tempfile.TemporaryFile() as tf:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(tf.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["MBC_BM_SPARSE_TRACE"]
        tf.seek(0)
        lines = tf.read().decode().splitlines()
    return [ln.split(", ")[-1] for ln in lines if "sparse bitmap term" in ln]


def timed(ctx, t, terms, reps, form=None):
    if form:
        os.environ["MBC_BM_SPARSE_FORM"] = form
    try:
        times, count = [], None
        for _ in range(reps + 2):                           # two warm-up calls of the same shape
            r = t.bitmap_scan(terms, want=N.WANT_AGG, aggs=[(0, 0)])
            times.append(ctx.last_kernel_ms)
            count = r.count
            r.close()
        return statistics.median(times[2:]), count
    finally:
        os.environ.pop("MBC_BM_SPARSE_FORM", None)


def parity(t, terms):
    a = t.bitmap_scan(terms, want=N.WANT_BITMAP | N.WANT_HOST)
    b = t.scan(terms, want=N.WANT_BITMAP | N.WANT_HOST)
    ok = a.count == b.count and np.array_equal(a.bitmap(), b.bitmap())
    a.close(); b.close()
    return ok


def measure(ctx, t, name, terms, rows, reps):
    auto_ms, count = timed(ctx, t, terms, reps)
    scatter_ms, _ = timed(ctx, t, terms, reps, "scatter")
    compare_ms, _ = timed(ctx, t, terms, reps, "compare")
    return {"query": name, "count": count, "selectivity": count / rows, "ms": auto_ms, "forced_scatter_ms": scatter_ms,
            "forced_compare_ms": compare_ms, "forms": forms_taken(lambda: t.bitmap_scan(terms, want=N.WANT_AGG, aggs=[(0, 0)]).close()),
            "parity_with_mbc_scan": parity(t, terms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3", "bench_bitmap_sparse.json"))
    a = ap.parse_args()
    rows = a.rows
    ctx = mbcol.Context(0)
    t = ctx.create_table([(1, 4), (1, 4), (0, 16), (1, 4)], rows)
    t.generate(0, 3, SEED, rows)
    t.generate(1, 0, SEED, 10_000_000)
    t.generate(2, 2, SEED)
    t.generate(3, 0, SEED, 4)
    words_pad = (rows + 8191) // 8192 * 8192 // 32
    build = {}
    for col, name in ((0, "K"), (1, "M"), (2, "S"), (3, "H")):
        t.bitmap_build(col)
        ms = ctx.last_kernel_ms
        layout, nbytes = t.bitmap_layout(col)
        nvals = int(t.bitmap_values(col).shape[0])
        build[name] = {"ms": ms, "rows_per_s": rows / (ms * 1e-3), "layout": LAYOUT[layout], "values": nvals,
                       "index_bytes": nbytes, "dense_bytes_needed": nvals * words_pad * 4}
    assert [build[n]["layout"] for n in "KMSH"] == ["sparse", "sparse", "sparse", "dense"], build
    svals = t.bitmap_values(2)
    mvals = t.bitmap_values(1)
    T = mbcol.Term
    scans = [measure(ctx, t, "K = 4242", [T(N.OP_EQ, ("col", 0), ("int", 4242), 0)], rows, a.reps),
             measure(ctx, t, "S = <a present value>", [T(N.OP_EQ, ("col", 2), ("str", bytes(svals[len(svals) // 3]).rstrip(b"\0")), 0)],
                     rows, a.reps)]
    for pct in (1, 3, 10, 50):
        k = rows * pct // 100
        scans.append(measure(ctx, t, f"K < {k} ({pct} %)", [T(N.OP_LT, ("col", 0), ("int", k), 0)], rows, a.reps))
    scans.append(measure(ctx, t, "K != 4242", [T(N.OP_NE, ("col", 0), ("int", 4242), 0)], rows, a.reps))
    for pct in (1, 10, 50):
        lit = bytes(svals[len(svals) * pct // 100]).rstrip(b"\0")
        scans.append(measure(ctx, t, f"S < <the {pct} % quantile>", [T(N.OP_LT, ("col", 2), ("str", lit), 0)], rows, a.reps))
    m, k = int(mvals[len(mvals) // 2]), rows // 100
    scans.append(measure(ctx, t, f"{{(M,=,{m})|(K,<,{k})}}^{{(H,=,2)}}",
                         [T(N.OP_EQ, ("col", 1), ("int", m), 0), T(N.OP_LT, ("col", 0), ("int", k), 0), T(N.OP_EQ, ("col", 3), ("int", 2), 1)],
                         rows, a.reps))
    out = {"bench": "sparse bitmap layout", "rows": rows, "card": card(), "build": build, "scans": scans,
           "timing": "ms = median over --reps calls (after two warm-up calls) of mbc_last_kernel_ms: CUDA events around the "
                     "call's kernels; a scan's time covers the terms' flat bitmaps, the CNF combine and the select / count pass",
           "parity_all": all(s["parity_with_mbc_scan"] for s in scans)}
    t.close()
    ctx.close()
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
