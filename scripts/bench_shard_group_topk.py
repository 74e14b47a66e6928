#!/usr/bin/env python
"""Sharded GROUP BY and top-k (mbc_shard_group / mbc_shard_topk) in one process, one context per GPU of the box, each rank
holding a position-range slice of the C2 table (--rows per rank, generated on the device; every column is larger than the
126 MB L2).  Per query and step, as in a real sharded query:
  1. every rank runs the single-GPU operator on its slice (mbc_group_aggregate / mbc_topk, device-resident), the ranks
     in parallel threads (the library releases the GIL in every call);
  2. the ranks gather their results into the root's window in rank order (peer stores), and the root collects;
  3. the root merges (mbc_shard_group / mbc_shard_topk) and releases the step.
Reported per query (median of --reps steps after one warm-up step): the slowest rank's local operator time (device time,
mbc_last_kernel_ms), the gather time (host wall from the first gather to the end of the collect), the root's merge time
(device time of the merge's kernels), the total step wall time, and the same query by the single-GPU operator on rank 0's
slice alone (device time).  The card's name and power limit are read in the same run.

With one GPU on the box the ranks of world 2 and 4 all run on that GPU: those numbers are overhead figures (what the
gather and the merge add), not scaling.

Queries: GROUP BY K16 (16 values), K1000 (1000 values) and I1 (2^20 values) with C2's COUNT, SUM(I2), SUM(R), MIN(I1),
MAX(I1); top-k ascending on I1 and on S with k in {100, 10^4, 10^6}, projecting (I1, S); each at 10 % and 100 %.

    python scripts/bench_shard_group_topk.py [--rows 100000000] [--reps 5] [--out profiles/r3/bench_shard_group_topk.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mbcol

N = mbcol._native
SEED = 20260101
DESCS = [(1, 4), (1, 4), (2, 4), (0, 16), (1, 4), (1, 4)]        # I1, I2, R, S, K16, K1000
GROUP_KEYS = {"K16": 4, "K1000": 5, "I1": 0}
TOPK_KEYS = {"I1": 0, "S": 3}
C2_AGGS = [(0, 0), (1, 1), (1, 2), (2, 0), (3, 0)]
TOPK_PROJ = [0, 3]                                                  # the top-k window: I1, S


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                          # the numbers are still device times; say what is missing
        return {"name": "unknown", "power_limit": f"not read ({e.__class__.__name__})"}


def terms_for(selectivity):
    """C2's {(I1 < t1)} ^ {(R < t2)} with per-predicate selectivity sqrt(s); none at 100 %."""
    if selectivity >= 1.0:
        return []
    r = selectivity ** 0.5
    return [mbcol.Term(N.OP_LT, ("col", 0), ("int", int(-(-r * (1 << 20) // 1))), 0),
            mbcol.Term(N.OP_LT, ("col", 2), ("real", r * 1000.0), 1)]


def run_world(world, ndev, rows, reps):
    ctxs = [mbcol.Context(r % ndev) for r in range(world)]
    tables = []
    for r, c in enumerate(ctxs):
        t = c.create_table(DESCS, rows, position_base=r * rows)
        for col, (kind, dom) in enumerate([(0, 1 << 20), (0, 1 << 20), (1, 0), (2, 0), (0, 16), (0, 1000)]):
            t.generate(col, kind, SEED, dom)
        tables.append(t)
    pool = ThreadPoolExecutor(world)
    types = [N.ATTR_INTEGER if k == 0 else DESCS[c][0] for k, c in C2_AGGS]

    def local(op):                                                  # every rank's operator, in parallel -> results, ms
        def one(r):
            res = op(tables[r])
            res.count
            return res, ctxs[r].last_kernel_ms
        out = list(pool.map(one, range(world)))
        return [o[0] for o in out], max(o[1] for o in out)

    def step(shards, op, merge):
        t0 = time.perf_counter()
        results, local_ms = local(op)
        t1 = time.perf_counter()
        for r, res in enumerate(results):                           # rank order, each push finished before the next
            shards[r].gather(res)
            shards[r].fence()
            ctxs[r].sync()
        total, _ = shards[0].collect()
        t2 = time.perf_counter()
        m = merge(shards[0], total)
        merge_ms = ctxs[0].last_kernel_ms
        count = m.count
        shards[0].release()
        ctxs[0].sync()
        t3 = time.perf_counter()
        for res in results + [m]:
            res.close()
        return {"local_ms": local_ms, "gather_ms": (t2 - t1) * 1e3, "merge_ms": merge_ms, "merge_wall_ms": (t3 - t2) * 1e3,
                "step_ms": (t3 - t0) * 1e3, "gathered_rows": total, "result_rows": count}

    def single(op):
        ms = []
        for i in range(reps + 1):
            res = op(tables[0])
            res.count
            if i:
                ms.append(ctxs[0].last_kernel_ms)
            res.close()
        return statistics.median(ms)

    def measure(shards, op, merge, query):
        steps = [step(shards, op, merge) for _ in range(reps + 1)][1:]
        row = dict(query)
        for key in ("local_ms", "gather_ms", "merge_ms", "merge_wall_ms", "step_ms"):
            row[key] = round(statistics.median(s[key] for s in steps), 3)
        row["gathered_rows"], row["result_rows"] = steps[-1]["gathered_rows"], steps[-1]["result_rows"]
        row["single_gpu_ms"] = round(single(op), 3)
        print(json.dumps(row), file=sys.stderr)
        return row

    def shard_set(make_window):
        shards = [mbcol.Shard(c, r, world) for r, c in enumerate(ctxs)]
        make_window(shards[0])
        for s in shards[1:]:
            s.attach(shards[0])
        return shards

    out = []
    # one window shape for the three group keys: an int key column + 5 aggregate columns
    shards = shard_set(lambda s: s.create_group_window(world * (1 << 20) + 4096, [(1, 4)], len(C2_AGGS)))
    for name, key in GROUP_KEYS.items():
        for sel in (0.10, 1.0):
            terms = terms_for(sel)
            out.append(measure(shards, lambda t: t.group_aggregate(terms, [key], C2_AGGS, want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG),
                               lambda s, total: s.group_aggregate([(1, 4)], [k for k, _ in C2_AGGS], types,
                                                                   want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG),
                               {"query": "group", "key": name, "selectivity": sel}))
    for s in shards[1:] + shards[:1]:
        s.close()
    pdescs = [DESCS[c] for c in TOPK_PROJ]
    shards = shard_set(lambda s: s.create_window(world * 10**6 + 4096, pdescs))
    for name, key in TOPK_KEYS.items():
        for sel in (0.10, 1.0):
            terms = terms_for(sel)
            for k in (100, 10**4, 10**6):
                out.append(measure(shards, lambda t: t.top_k(terms, [key], k, proj=TOPK_PROJ, want=N.WANT_POSITIONS | N.WANT_COLUMNS),
                                   lambda s, total: s.top_k(pdescs, [TOPK_PROJ.index(key)], k, proj_fields=[0, 1],
                                                            want=N.WANT_POSITIONS | N.WANT_COLUMNS),
                                   {"query": "topk", "key": name, "selectivity": sel, "k": k}))
    for s in shards[1:] + shards[:1]:
        s.close()
    pool.shutdown()
    for t in tables:
        t.close()
    for c in ctxs:
        c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows per rank")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3", "bench_shard_group_topk.json"))
    a = ap.parse_args()
    import torch
    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise SystemExit("no GPU: this benchmark measures device times only")
    worlds = [ndev] if ndev > 1 else [2, 4]
    runs = []
    for w in worlds:
        runs.append({"world": w, "gpus_used": min(w, ndev),
                     "form": "scaling: one rank per GPU" if ndev > 1 else "overhead: every rank on the one GPU, not scaling",
                     "results": run_world(w, ndev, a.rows, a.reps)})
    out = {"bench": "shard_group_topk", "card": card(), "gpus": ndev, "rows_per_rank": a.rows, "reps": a.reps,
           "timing": "median over reps steps after one warm-up; local / merge / single_gpu: device ms (CUDA events); "
                     "gather / step: host wall ms", "runs": runs}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
