#!/usr/bin/env python
"""mbc_group_aggregate on one B200: GROUP BY over the C2 table at 10 % and 100 % selectivity, with COUNT, SUM(I2),
SUM(R), MIN(I1), MAX(I1), for int keys of 16, 1 000 and 2^20 distinct values, all-unique int keys and a char(16) key.
Beside every grouping it times, in the same run and on the same table, the parts the grouping is built from: the
filter alone (mbc_scan, positions only), the grouping without aggregates (scan + sort + group boundaries), and mbc_sort
of the whole table by the same key.  The aggregate fold is the difference of the first two grouping times.  Every time is
the median of --reps calls after two warm-up calls, as device time from CUDA events around the call's kernels
(mbc_last_kernel_ms); host wall time of the same calls is reported beside it.  The card's name and power limit are read in
the same run.  Prints one JSON line and writes it to --out.

The table (generated on the device, 100 M rows by default; every column is larger than the 126 MB L2):
  I1, I2: ints in [0, 2^20)   R: real in [0, 1000)   S: char(16)   K16, K1000: ints of 16 / 1 000 values   KU: a permutation

    python scripts/bench_group.py [--rows 100000000] [--reps 20] [--out profiles/r3/bench_group.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mbcol

N = mbcol._native
SEED = 20260101
DESCS = [(1, 4), (1, 4), (2, 4), (0, 16), (1, 4), (1, 4), (1, 4)]
KEYS = {"int16": 4, "int1000": 5, "int2^20": 0, "unique": 6, "char16": 3}
AGGS = [(N.AGG_COUNT, 0), (N.AGG_SUM, 1), (N.AGG_SUM, 2), (N.AGG_MIN, 0), (N.AGG_MAX, 0)]


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # the numbers are still device times; say what is missing
        return {"name": "unknown", "power_limit": f"not read ({e.__class__.__name__})"}


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3", "bench_group.json"))
    a = ap.parse_args()
    ctx = mbcol.Context(0)
    t = ctx.create_table(DESCS, a.rows)
    t.generate(0, 0, SEED, 1 << 20)
    t.generate(1, 0, SEED, 1 << 20)
    t.generate(2, 1, SEED)
    t.generate(3, 2, SEED)
    t.generate(4, 0, SEED, 16)
    t.generate(5, 0, SEED, 1000)
    t.generate(6, 3, SEED, a.rows)
    rows = []
    sort_ms = {}
    for name, col in KEYS.items():
        sort_ms[name] = timed(ctx, lambda: t.sort([col], want=N.WANT_POSITIONS), a.reps)[0]
        for sel in (0.10, 1.0):
            terms = terms_for(sel)
            scan_ms, _, qual = timed(ctx, lambda: t.scan(terms, want=N.WANT_POSITIONS), a.reps)
            keys_ms, _, _ = timed(ctx, lambda: t.group_aggregate(terms, [col], want=N.WANT_POSITIONS | N.WANT_COLUMNS), a.reps)
            ms, wall, groups = timed(ctx, lambda: t.group_aggregate(terms, [col], AGGS, want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG),
                                     a.reps)
            rows.append({"key": name, "selectivity": sel, "qualifying_rows": qual, "groups": groups,
                         "group_ms": round(ms, 3), "group_wall_ms": round(wall, 3), "rows_per_s": round(a.rows / ms * 1e3),
                         "scan_ms": round(scan_ms, 3), "group_without_aggs_ms": round(keys_ms, 3),
                         "fold_ms": round(ms - keys_ms, 3), "sort_table_ms": round(sort_ms[name], 3)})
            print(json.dumps(rows[-1]), file=sys.stderr)
    out = {"bench": "group_aggregate", "card": card(), "rows": a.rows, "reps": a.reps,
           "aggregates": "COUNT, SUM(I2), SUM(R), MIN(I1), MAX(I1)", "timing": "median device ms (CUDA events), 2 warm-ups",
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
