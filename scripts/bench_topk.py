#!/usr/bin/env python
"""mbc_topk on one B200: ORDER BY key LIMIT k over the C2 table at 10 % and 100 % selectivity, for the keys I1, R, S,
(S, I1) and a 16-valued int key (ties), ascending and descending, with k in {1, 100, 10^4, 10^6, 10 % of Q, Q}.  Beside
every top-k it times, in the same run and on the same table, mbc_sort of the whole table by the same keys and direction,
and the filter alone (mbc_scan, positions only, same terms).  Every time is the median of --reps calls after two warm-up
calls, as device time from CUDA events around the call's kernels (mbc_last_kernel_ms; a top-k's includes its filter, an
mbc_sort's does not include its no-predicate scan); host wall time of the same calls is reported beside it.  `path` names
the branch the call took under MBC_TOPK_SORT_FRACTION as csrc/mbc_topk.cu defines it (k above that share of Q: filtered
sort, else radix select).  The card's name and power limit are read in the same run.  Prints one JSON line and writes it
to --out.

The table (generated on the device, 100 M rows by default; every column is larger than the 126 MB L2):
  I1, I2: ints in [0, 2^20)   R: real in [0, 1000)   S: char(16)   K16: ints of 16 values

    python scripts/bench_topk.py [--rows 100000000] [--reps 20] [--out profiles/r3/bench_topk.json]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mbcol

N = mbcol._native
SEED = 20260101
DESCS = [(1, 4), (1, 4), (2, 4), (0, 16), (1, 4)]
KEYS = {"I1": [0], "R": [2], "S": [3], "S,I1": [3, 0], "K16": [4]}


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # the numbers are still device times; say what is missing
        return {"name": "unknown", "power_limit": f"not read ({e.__class__.__name__})"}


def sort_fraction():
    src = open(os.path.join(ROOT, "minibase-columnar-database_b200", "csrc", "mbc_topk.cu")).read()
    return float(re.search(r"#define MBC_TOPK_SORT_FRACTION\s+([0-9.eE+-]+)", src).group(1))


def terms_for(selectivity):
    """C2's {(I1 < t1)} ^ {(R < t2)} with per-predicate selectivity sqrt(s); none at 100 %."""
    if selectivity >= 1.0:
        return []
    r = selectivity ** 0.5
    return [mbcol.Term(N.OP_LT, ("col", 0), ("int", int(-(-r * (1 << 20) // 1))), 0),
            mbcol.Term(N.OP_LT, ("col", 2), ("real", r * 1000.0), 1)]


def timed(ctx, fn, reps):
    dev, wall, out = [], [], None
    for i in range(reps + 2):                               # two warm-up calls of the same shape
        t0 = time.perf_counter()
        r = fn()
        out = r.count
        w = (time.perf_counter() - t0) * 1e3               # every call below returns after its kernels finished
        d = ctx.last_kernel_ms
        r.close()
        if i >= 2:
            dev.append(d)
            wall.append(w)
    return statistics.median(dev), statistics.median(wall), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3", "bench_topk.json"))
    a = ap.parse_args()
    frac = sort_fraction()
    ctx = mbcol.Context(0)
    t = ctx.create_table(DESCS, a.rows)
    t.generate(0, 0, SEED, 1 << 20)
    t.generate(1, 0, SEED, 1 << 20)
    t.generate(2, 1, SEED)
    t.generate(3, 2, SEED)
    t.generate(4, 0, SEED, 16)
    rows = []
    scan = {}
    for sel in (0.10, 1.0):
        scan[sel] = timed(ctx, lambda: t.scan(terms_for(sel), want=N.WANT_POSITIONS), a.reps)
    for name, keys in KEYS.items():
        for desc in (False, True):
            sort_ms = timed(ctx, lambda: t.sort(keys, descending=desc, want=N.WANT_POSITIONS), a.reps)[0]
            for sel in (0.10, 1.0):
                terms = terms_for(sel)
                scan_ms, _, q = scan[sel]
                for k in sorted({1, 100, 10**4, 10**6, q // 10, q}):
                    ms, wall, cnt = timed(ctx, lambda: t.top_k(terms, keys, k, descending=desc, want=N.WANT_POSITIONS), a.reps)
                    assert cnt == min(k, q), (cnt, k, q)
                    rows.append({"key": name, "descending": desc, "selectivity": sel, "qualifying_rows": q, "k": k,
                                 "path": "sort" if k > frac * q else "select", "topk_ms": round(ms, 3),
                                 "topk_wall_ms": round(wall, 3), "sort_table_ms": round(sort_ms, 3),
                                 "scan_ms": round(scan_ms, 3)})
                    print(json.dumps(rows[-1]), file=sys.stderr)
    out = {"bench": "topk", "card": card(), "rows": a.rows, "reps": a.reps, "sort_fraction": frac,
           "want": "MBC_WANT_POSITIONS (device-resident)", "timing": "median device ms (CUDA events), 2 warm-ups",
           "results": rows}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
    t.close()
    ctx.close()


if __name__ == "__main__":
    main()
