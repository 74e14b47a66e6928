#!/usr/bin/env python
"""bench.py -- filtered-scan rows/s (BASELINE.json metric) on N B200s of one node.

Workloads (SURVEY.md 8d; `--workload auto` picks C2 on one GPU and C5 on several, the configs BASELINE.json quotes):

  c2  100 M-row table (I1,I2 int; R real; S char(16) = 2.8 GB in HBM).  One step = the hot path at each of the three
      selectivities: `{(I1,<,t1)}^{(R,<,t2)}` at 1 % / 10 % / 50 %, project [I1,I2,R,S], COUNT/SUM(I2)/SUM(R)/MIN(I1)/MAX(I1).
  c5  8-column table (I1..I5 int, R1,R2 real, S char(16) = 44 B/row), 500 M rows (22 GB) PER GPU, sharded by TID range
      (4 G rows on 8 GPUs).  One step = `{(I1,<,t1)}^{(R1,<,t2)}` at 1 %, project [I1,I2,R1], the same five aggregates, and
      the gather of every rank's positions + projected values + aggregates on rank 0.

On N > 1 GPUs every rank scans its own position range with no data-path collective; the result rows travel ONCE, as
peer-memory stores over NVLink from a kernel of libmbcol.so into rank 0's window (mbc_shard_* in include/mbcol.h, driven
through ctypes); torch.distributed (NCCL) only carries the 64-byte IPC handle, the barriers and the max-over-ranks time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload auto|c2|c5] [--rows R] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` (one GPU) writes what the last timed step returned as .npy files, so that two builds can be compared
output for output on the same seeded table.

`--impl reference` times the reference's CPU algorithm (oracle/: the literal C++ restatement; the Java original cannot
run here -- no JDK in the image, probed at start) on the box's host cores.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 20260101
SELECTIVITIES = (0.01, 0.10, 0.50)
DESCS = [(1, 4), (1, 4), (2, 4), (0, 16)]                # C2: I1 int, I2 int, R real, S char(16)
AGGS = [(0, 0), (1, 1), (1, 2), (2, 0), (3, 0)]          # COUNT, SUM(I2), SUM(R), MIN(I1), MAX(I1)
ROW_BYTES_IN = 28                                        # every referenced column read once
ROW_BYTES_OUT = 36                                       # 8 B position + 28 B projected values

C5_DESCS = [(1, 4)] * 5 + [(2, 4)] * 2 + [(0, 16)]       # I1..I5, R1, R2, S
C5_AGGS = [(0, 0), (1, 1), (1, 5), (2, 0), (3, 0)]       # COUNT, SUM(I2), SUM(R1), MIN(I1), MAX(I1)

DUMP_BYTES = 64_000_000                                  # --dump-outputs: size limit of all files of one dump


def pred_terms(term_cls, sel: float, int_col: int, real_col: int):
    """{(int_col,<,t1)}^{(real_col,<,t2)} with per-predicate selectivity sqrt(sel) (SURVEY.md 8d)."""
    r = float(np.sqrt(sel))
    t1 = int(np.ceil(r * (1 << 20)))
    t2 = float(np.float32(r * 1000.0))
    return [term_cls(1, ("col", int_col), ("int", t1), 0), term_cls(1, ("col", real_col), ("real", t2), 1)]    # op 1 = aopLT


def c2_terms(term_cls, sel: float):
    return pred_terms(term_cls, sel, 0, 2)


def algorithmic_bytes(nrows: int, sel: float) -> float:
    """SURVEY.md 8(d), config C2: N * (28 + 36 * s)."""
    return nrows * (ROW_BYTES_IN + ROW_BYTES_OUT * sel)


class Workload:
    """What one step scans: the table's shape, the queries of a step, which query's rows are gathered on rank 0."""

    def __init__(self, name):
        self.name = name
        if name == "c2":
            self.descs, self.aggs, self.proj = DESCS, AGGS, [0, 1, 2, 3]
            self.gens = [(0, 1 << 20), (0, 1 << 20), (1, 0), (2, 0)]          # mbc_table_generate (kind, domain) per column
            self.sels = SELECTIVITIES
            self.int_col, self.real_col = 0, 2
            self.default_rows = 100_000_000
            self.gather_query = 0                                            # the 1 % query's rows go to rank 0
            self.row_bytes_in = ROW_BYTES_IN
            self.text = ("C2: synthetic 4-column table (I1,I2 int in [0,2^20); R real in [0,1000); S char(16)), "
                         "{(I1,<,t1)}^{(R,<,t2)} at 1%/10%/50% selectivity, project [I1,I2,R,S], COUNT/SUM(I2)/SUM(R)/MIN(I1)/MAX(I1)")
        else:
            self.descs, self.aggs, self.proj = C5_DESCS, C5_AGGS, [0, 1, 5]
            self.gens = [(0, 1 << 20)] * 5 + [(1, 0), (1, 0), (2, 0)]
            self.sels = (0.01,)
            self.int_col, self.real_col = 0, 5
            self.default_rows = 500_000_000
            self.gather_query = 0
            self.row_bytes_in = 12
            self.text = ("C5: synthetic 8-column table (I1..I5 int, R1,R2 real, S char(16) = 44 B/row) sharded by TID range, "
                         "{(I1,<,t1)}^{(R1,<,t2)} at 1% selectivity, project [I1,I2,R1], COUNT/SUM(I2)/SUM(R1)/MIN(I1)/MAX(I1), "
                         "gather of positions + projected values + aggregates on rank 0")
        self.row_bytes_out = 8 + sum(4 if t != 0 else w for t, w in (self.descs[c] for c in self.proj))
        self.used_cols = sorted(set(self.proj) | {self.int_col, self.real_col} | {c for k, c in self.aggs if k != 0})

    def terms(self, term_cls, sel):
        return pred_terms(term_cls, sel, self.int_col, self.real_col)

    def bytes(self, nrows, sel):
        """SURVEY.md 8(d): every referenced column once + 8 B position + projected values per qualifying row."""
        return nrows * (self.row_bytes_in + self.row_bytes_out * sel)

    def host_columns(self, orc, nrows, base=0, only_used=False):
        cols = []
        for c, ((t, w), (kind, dom)) in enumerate(zip(self.descs, self.gens)):
            if only_used and c not in self.used_cols:
                cols.append(None)
            elif kind == 0:
                cols.append(orc.synth_int(SEED, c, nrows, dom, base))
            elif kind == 1:
                cols.append(orc.synth_real(SEED, c, nrows, base))
            else:
                cols.append(orc.synth_str(SEED, c, nrows, w, base))
        return cols


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash() -> str:
    """sha256 over the kernel sources: an ncu traffic capture is only quoted for the code it was taken from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "minibase-columnar-database_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.startswith("mbc_scan") or name == "mbc_internal.cuh":          # what the measured scan runs
            with open(os.path.join(d, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def measured_traffic(workload, rows_per_gpu):
    """DRAM bytes per scan from the committed ncu --set full capture (profiles/r2/traffic.json, written by
    scripts/ncu_traffic.py).  Quoted only when the capture was taken from the kernel sources now in the tree (source hash)
    and for this workload and table size; otherwise null -- the bench never prints a stale constant."""
    path = os.path.join(ROOT, "profiles", "r2", "traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
    except Exception:
        return None, "no capture"
    if t.get("workload") != workload or t.get("rows") != rows_per_gpu:
        return None, "capture is for another workload / size"
    if t.get("kernel_source_hash") != kernel_source_hash():
        return None, f"capture {t.get('kernel_source_hash')} predates the kernel sources {kernel_source_hash()}"
    return t, "profiles/r2/traffic.json"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def java_probe() -> dict:
    """BASELINE.md 3.1: is there a JDK (and the reference's sources) to time the Java scan itself?"""
    java, javac = shutil.which("java"), shutil.which("javac")
    src = os.path.isdir("/root/reference/minijava/src")
    return {"java": bool(java), "javac": bool(javac), "reference_sources": src,
            "usable": bool(java and javac and src)}


def cpu_scan_rate(wl: Workload, nrows_sample: int, nthreads: int, repeats: int = 1):
    """Time the oracle (CPU restatement of TupleScan -> PredEval -> Projection) on a sample of the workload."""
    from oracle import oracle as orc
    orc.build()
    cols = wl.host_columns(orc, nrows_sample)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for s in wl.sels:
            orc.scan(wl.descs, cols, wl.terms(orc.Term, s), proj=wl.proj, aggs=wl.aggs, nthreads=nthreads)
        times.append(time.perf_counter() - t0)
    return len(wl.sels) * nrows_sample / min(times), times


def workload_config(wl: Workload, args, rows_per_gpu, world):
    cfg = {"workload": wl.text, "rows_per_gpu": rows_per_gpu, "scans_per_step": len(wl.sels), "selectivities": list(wl.sels),
           "l2": f"inputs ({rows_per_gpu * wl.row_bytes_in / 1e9:.1f} GB of referenced columns per GPU) are larger than the 126 MB L2; no flush needed"}
    if world > 1:
        cfg["sharding"] = ("TID range per rank, no data-path collective; per step every rank pushes the gathered query's positions + "
                           "projected values + count + aggregates into rank 0's IPC-mapped window over NVLink (mbc_shard_* ABI of libmbcol.so "
                           "through ctypes: counts published by a kernel, rows moved by the copy engines at the exclusive-scan offset; no "
                           "NCCL kernel on the data path); the "
                           "push of step i runs beside the scans of step i+1; the last one is drained inside the timed region")
    else:
        cfg["sharding"] = "single GPU"
        cfg["pipelining"] = ("the scans of step i+1 are queued before the host reads the counts of step i (results are double "
                             "buffered); every step's counts are read and its results freed inside the timed region")
    return cfg


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    wl = Workload(resolve_workload(args, world))
    threads = orc.max_threads()
    sample = args.cpu_rows if args.cpu_rows > 0 else (wl.default_rows if wl.name == "c2" else 100_000_000)
    cols = wl.host_columns(orc, sample)

    def step():
        for s in wl.sels:
            orc.scan(wl.descs, cols, wl.terms(orc.Term, s), proj=wl.proj, aggs=wl.aggs, nthreads=threads)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = len(wl.sels) * sample * args.steps / dt
    probe = java_probe()
    sample_desc = (f"{sample} rows of the {wl.name.upper()} table per scan ({len(wl.sels)} scans/step), oracle/mbc_oracle.cpp orc_scan with "
                   f"{threads} std::threads; the Java reference itself cannot run (JDK probe: {probe})")
    print(json.dumps({
        "impl": "reference", "metric": "filtered_scan_rows_per_s", "value": value, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/float32/u8x16 compare, int64/float64 aggregate",
        "data": "synthetic", "config": workload_config(wl, args, sample, 1),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample_desc, "java_probe": probe},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def resolve_workload(args, world):
    if args.workload != "auto":
        return args.workload
    return "c2" if max(world, args.gpus) == 1 else "c5"


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist
    import mbcol
    N = mbcol._native

    wl = Workload(resolve_workload(args, world))
    rows = args.rows if args.rows > 0 else wl.default_rows
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    real_stdout = None
    if world > 1:
        # stdout carries ONE JSON line: NCCL's version banner and INFO lines (NCCL_DEBUG is left as the caller set it: the
        # driver's rank check reads them) are sent to stderr -- by NCCL_DEBUG_FILE where NCCL honours it, and by pointing
        # file descriptor 1 at stderr until the JSON line is printed for whatever still writes to stdout
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    ctx = mbcol.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    table = ctx.create_table(wl.descs, rows, position_base=rank * rows)
    for c, (kind, dom) in enumerate(wl.gens):
        table.generate(c, kind, SEED, dom)
    terms = {s: wl.terms(mbcol.Term, s) for s in wl.sels}
    want_dev = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG
    kernel_ms = {s: [] for s in wl.sels}
    phase_ms = {s: [] for s in wl.sels}
    counts = {}
    proj_descs = [wl.descs[c] for c in wl.proj]
    gsel = wl.sels[wl.gather_query]

    # ---- the shard group: rank 0 owns the window, the peers map it through a CUDA IPC handle -------------------------
    shard = None
    if world > 1:
        shard = mbcol.Shard(ctx, rank, world)
        cap = int(rows * world * gsel * 1.25) + 65536               # 25 % above the expected result of the gathered query
        hbuf = torch.zeros(N.IPC_HANDLE_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            hbuf.copy_(torch.frombuffer(bytearray(shard.create_window(cap, proj_descs)), dtype=torch.uint8))
        dist.broadcast(hbuf, 0)                                     # control plane only: 64 bytes
        if rank != 0:
            shard.open_window(bytes(hbuf.cpu().numpy().tobytes()), cap, proj_descs)
        dist.barrier()

    # rows over the copy engines (default; measured at N=8: 1.26 ms per step against 1.60 ms with SM stores -- 7 ranks' stores
    # into one GPU reached ~500 GB/s of its NVLink ingress, the DMA engines ~760 GB/s) or as peer-memory stores from a kernel
    copy_engines = os.environ.get("MBC_BENCH_GATHER", "dma") == "dma"
    pending = []                                                    # results of the previous step: its push may still be running
    collected = {"total": None, "counts": None}

    def exchange_previous(record=False):
        """The previous step's exchange, issued while THIS step's scans (already queued) run: every rank publishes its count
        and pushes its rows into rank 0's window, rank 0 waits for all of them (on the shard's side stream, so the host never
        waits for the scans just queued), notes the totals and releases the window slot; then the results are freed.  The host
        reads the previous step's counts here -- they are complete, nothing in the loop waits for the scans in flight."""
        if not pending:
            return
        results = list(pending)
        pending.clear()
        shard.gather(results[wl.gather_query], beside_next_scan=True, copy_engines=copy_engines)
        for s, res in zip(wl.sels, results):
            counts[s] = res.count
            if record:
                kernel_ms[s].append(res.kernel_ms)
        if rank == 0:
            collected["total"], collected["counts"] = shard.collect()
            shard.release()
        shard.fence()                                               # the frees below are stream-ordered behind the push
        for res in results:
            res.close()

    def read_previous(record=False, keep=False):
        """N=1: the host reads the counts of the PREVIOUS step (and frees its results) after this step's scans are queued, so
        the GPU is not idle while the host waits and launches; every step's results are read inside the timed region.
        keep: the results are returned to the caller instead of freed."""
        results = list(pending)
        pending.clear()
        for s, res in zip(wl.sels, results):                        # the host reads every count (this is the wait)
            counts[s] = res.count
            if record:
                kernel_ms[s].append(res.kernel_ms)
        if keep:
            return results
        for res in results:
            res.close()

    def step(record=False):
        results = []
        for s in wl.sels:                                           # device-resident results complete asynchronously:
            results.append(table.scan(terms[s], proj=wl.proj, want=want_dev, aggs=wl.aggs))   # the scans queue back to back
        if world > 1:
            exchange_previous(record)                               # step i-1's rows travel while step i's scans run
        else:
            read_previous(record)
        pending.extend(results)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    if world > 1:
        exchange_previous()
    else:
        read_previous()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step(record=True)
    if world > 1:
        exchange_previous(record=True)                              # the last step's exchange is inside the timed region
    else:
        last = read_previous(record=True, keep=bool(args.dump_outputs))   # ... and so is the read of the last step's results
    e1.record(stream)
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wl, last, dev)
        for res in last:
            res.close()
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches - launches0
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    nscan = len(wl.sels)
    value = float(nscan) * rows * world * args.steps / (ms_total * 1e-3)

    push_ms = None
    if world > 1:                                                   # device time of every rank's last push (rank order)
        pm = torch.tensor([shard.push_ms], dtype=torch.float64, device=dev)
        allp = [torch.zeros_like(pm) for _ in range(world)]
        dist.all_gather(allp, pm)
        push_ms = [round(float(x.item()), 4) for x in allp]
    # ---- per-kernel device times: a separate, untimed pass with the three extra events per scan switched on ---------------
    os.environ["MBC_PHASE_EVENTS"] = "1"
    for _ in range(min(args.steps, 5)):
        rs = [table.scan(terms[s], proj=wl.proj, want=want_dev, aggs=wl.aggs) for s in wl.sels]
        for s, r_ in zip(wl.sels, rs):
            _ = r_.count
            phase_ms[s].append(r_.phase_ms)
            r_.close()
    os.environ.pop("MBC_PHASE_EVENTS", None)
    # ---- scan-only time of the same shard (no gather): what the multi-GPU step is compared with ----------------------
    scan_only_ms = None
    if world > 1:
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            rs = [table.scan(terms[s], proj=wl.proj, want=want_dev, aggs=wl.aggs) for s in wl.sels]
            for r_ in rs:
                _ = r_.count
                r_.close()
        e1.record(stream)
        torch.cuda.synchronize()
        t_ = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        scan_only_ms = float(t_.item()) / args.steps

    # ---- parity of the multi-GPU path, after the timed region: one more step, checked on rank 0 --------------------
    parity = None
    if world > 1:
        parity = check_sharded_step(wl, table, terms, shard, rank, world, rows, proj_descs, mbcol, dist, dev, torch)

    # ---- end to end: host-resident columns -> mbc_scan_host -> host-resident results -------------------------------
    if args.no_e2e:
        if rank == 0:
            sys.stdout.flush()
            os.dup2(real_stdout, 1) if real_stdout is not None else None
            print(json.dumps({"tuning_run": True, "n_gpus": world, "ms_per_step": ms_total / args.steps, "value": value,
                              "scan_only_ms_per_step": scan_only_ms, "parity_checked": bool(parity and parity.get("ok")),
                              "push_ms_per_rank": push_ms,
                              "per_selectivity_kernel_ms": {str(s): statistics.mean(kernel_ms[s]) for s in wl.sels},
                              "env": {k: v for k, v in os.environ.items() if k.startswith("MBC_")}}))
        if shard is not None:
            barrier()
            shard.close()
        table.close()
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return
    host_cols = []
    dummy = np.zeros(64, dtype=np.uint8)
    for c, (t, w) in enumerate(wl.descs):
        if c not in wl.used_cols:
            host_cols.append(dummy)                                 # never read: the query does not touch the column
            continue
        dt = np.int32 if t == 1 else np.float32 if t == 2 else np.uint8
        shape = (rows,) if t != 0 else (rows, w)
        pinned = torch.empty(int(np.prod(shape)) * np.dtype(dt).itemsize, dtype=torch.uint8, pin_memory=True).numpy()
        arr = pinned.view(dt).reshape(shape)
        arr[...] = table.read_column(c)
        host_cols.append(arr)
    want_host = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG | N.WANT_HOST
    h2d = d2h = 0

    def e2e_step(count_bytes=False):
        nonlocal d2h, h2d
        moved0 = ctx.h2d_bytes
        for s in wl.sels:
            res = scan_host_rows(ctx, mbcol, wl, host_cols, rows, terms[s], want_host, rank * rows)
            if count_bytes:
                d2h += res.count * wl.row_bytes_out + 8 * (len(wl.aggs) + 1)
            res.close()
        if count_bytes:
            h2d = ctx.h2d_bytes - moved0           # counted by the library: selective scans upload the predicate columns only

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    for _ in range(2 if wl.name == "c2" else 1):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(e2e_steps):
        e2e_step(count_bytes=(i == 0))
    e1.record(stream)
    barrier()
    e2e_wall_ms = 1e3 * (time.perf_counter() - t0)
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    e2e_t = torch.tensor([max(e2e_ms, e2e_wall_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = float(nscan) * rows * world * e2e_steps / (float(e2e_t.item()) * 1e-3)
    if world > 1:                                                   # whole-job bytes: every rank moved its own
        hb = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
        dist.all_reduce(hb)
        h2d, d2h = int(hb[0].item()), int(hb[1].item())
    # the same with pageable (unpinned) host columns, one step: what a caller that does not allocate through mbc_host_alloc gets
    e2e_pageable = None
    if world == 1 and not args.no_pageable:
        pageable = [np.array(a, copy=True) if a is not dummy else dummy for a in host_cols]
        t0 = time.perf_counter()
        for s in wl.sels:
            scan_host_rows(ctx, mbcol, wl, pageable, rows, terms[s], want_host, 0).close()
        e2e_pageable = float(nscan) * rows / (time.perf_counter() - t0)
        del pageable
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        step_ms = ms_total / args.steps
        per_sel = {}
        tot_bytes = tot_ms = 0.0
        for s in wl.sels:
            m = statistics.mean(kernel_ms[s])
            b = wl.bytes(rows, s)
            per_sel[str(s)] = {"kernel_ms": m, "rows_per_s": rows / (m * 1e-3), "achieved_gbs": b / (m * 1e-3) / 1e9,
                               "frac_of_measured_peak": b / (m * 1e-3) / 1e9 / peak,
                               "frac_of_8000": b / (m * 1e-3) / 1e9 / 8000.0, "count": counts[s]}
            tot_bytes += b
            tot_ms += m
        achieved_step = tot_bytes / (step_ms * 1e-3) / 1e9           # on the step time the driver can check
        achieved_dev = tot_bytes / (tot_ms * 1e-3) / 1e9             # on the sum of the scans' device times (no gaps)
        # per kernel (CUDA events between the launches of every scan)
        kernels = {}
        names = ("pass 1 (fused_scan_kernel when one launch does the scan, else filter_kernel)", "tile_offsets_kernel", "write pass (write_kernel + write_staged_kernel)", "agg_finish_kernel")
        for s in wl.sels:
            ph = np.asarray(phase_ms[s], dtype=np.float64).mean(0)
            for i, name in enumerate(names):
                k = kernels.setdefault(name, {"ms_per_step": 0.0, "per_selectivity_ms": {}})
                k["ms_per_step"] += float(ph[i])
                k["per_selectivity_ms"][str(s)] = float(ph[i])
        for name, k in kernels.items():
            k["share_of_step"] = k["ms_per_step"] / tot_ms
        dominant = max(kernels, key=lambda n: kernels[n]["ms_per_step"])
        traffic, traffic_note = measured_traffic(wl.name, rows)
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle as orc
            sample = args.cpu_sample_rows
            v1, _ = cpu_scan_rate(wl, sample // 4, 1)
            vn, _ = cpu_scan_rate(wl, sample, orc.max_threads())
            cpu = {"value": vn, "unit": "rows/s", "cores": orc.max_threads(), "kind": "port",
                   "single_thread_rows_per_s": v1, "java_probe": java_probe(),
                   "sample": f"{sample} rows of the {wl.name.upper()} table per scan x {nscan} selectivities (all threads) and "
                             f"{sample // 4} rows (1 thread); oracle/mbc_oracle.cpp orc_scan"}
        roofline = {"bound": "hbm", "kernel": "mbc_scan: filter_kernel + tile_offsets_kernel + write_kernel + write_staged_kernel + agg_finish_kernel (or the opt-in fused_scan_kernel)",
                    "achieved": achieved_step, "peak": peak, "unit": "GB/s", "frac": achieved_step / peak,
                    "frac_of_nominal_8000": achieved_step / 8000.0, "peak_source": peak_src,
                    "basis": "algorithmic bytes of the step (SURVEY 8d) / ms_per_step",
                    "achieved_on_device_time": achieved_dev, "frac_on_device_time": achieved_dev / peak,
                    "traffic": (traffic or {}).get("per_scan_mean"), "traffic_source": traffic_note,
                    "traffic_per_selectivity": (traffic or {}).get("per_selectivity"),
                    "algorithmic_bytes_per_launch": tot_bytes / nscan,
                    "per_selectivity": per_sel, "dominant_kernel": dominant, "kernels": kernels}
        for k_, v_ in roofline.items():
            if k_.startswith("frac") and isinstance(v_, float):
                assert v_ <= 2.5, (k_, v_)                          # late materialisation may exceed 1 on the 8d bytes; far above means no work
        out = {
            "metric": "filtered_scan_rows_per_s", "value": value, "unit": "rows/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32/float32/u8x16 compare, int64/float64 aggregate", "data": "synthetic",
            "config": workload_config(wl, args, rows, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "pageable_host_buffers_rows_per_s": e2e_pageable,
                    "api": "mbc_scan_host (host columns pinned through mbc_host_alloc / cudaHostAlloc -> chunked H2D + scan -> D2H results; "
                           "selective scans read the survivors' projected values in place); pageable_host_buffers_rows_per_s = the same call on "
                           "ordinary malloc'd columns (one step)"},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if world > 1:
            out["multi_gpu"] = {"scan_only_ms_per_step": scan_only_ms, "step_ms": step_ms,
                                "efficiency_vs_scan_only": scan_only_ms / step_ms if scan_only_ms else None,
                                "gathered_rows": collected["total"], "rank_counts": collected["counts"],
                                "push_kernel_ms_per_rank": push_ms,
                                "gathered_bytes_per_step": (collected["total"] or 0) * wl.row_bytes_out,
                                "gather": "mbc_shard_gather into rank 0's IPC-mapped window, " + ("copy engines (cudaMemcpyAsync peer copies at the offset a one-warp kernel resolves)" if copy_engines else "peer-memory stores from shard_push_kernel") + "; no NCCL on the data path"}
            out["parity_checked"] = bool(parity and parity.get("ok"))
            out["parity"] = parity
        sys.stdout.flush()
        if real_stdout is not None:
            os.dup2(real_stdout, 1)
        print(json.dumps(out))
        sys.stdout.flush()
    if shard is not None:
        barrier()
        shard.close()
    table.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


class _CudaArray:
    """__cuda_array_interface__ view of library-owned device memory (tests and scripts wrap it with torch.as_tensor)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def dump_outputs(out_dir, wl, results, dev):
    """Write what a caller of the timed path received from its last step to out_dir, per query (file prefix sel<s>_): the
    positions, every projected column (col<c>) and the aggregates.  Positions, integers and aggregates are stored as
    float64, reals and string bytes as float32.  An aggregate without a value (MIN / MAX of no rows) is NaN.  A query with
    more rows than its share of DUMP_BYTES is represented by a sample: sorted row indices drawn with a fixed seed, the same
    on every run that returns as many rows, so that dumps of two builds compare element for element."""
    import torch
    from mbcol import _native as N

    def rows_of(ptr, stride, n, idx):
        """Rows idx of a device array of n rows of `stride` bytes, as a host uint8 array of shape (len(idx), stride)."""
        if n == 0:
            return np.zeros((0, stride), dtype=np.uint8)
        rows = torch.as_tensor(_CudaArray(ptr, n * stride), device=dev).view(n, stride)
        return rows[torch.from_numpy(idx).to(dev)].cpu().numpy()

    os.makedirs(out_dir, exist_ok=True)
    row_bytes = 8 + sum(4 * w if t == N.ATTR_STRING else 8 if t == N.ATTR_INTEGER else 4 for t, w in (wl.descs[c] for c in wl.proj))
    cap = (DUMP_BYTES - (1 << 16)) // (len(wl.sels) * row_bytes)      # 64 KB left for the .npy headers and the aggregates
    for s, res in zip(wl.sels, results):
        n = res.count
        idx = np.arange(n) if n <= cap else np.sort(np.random.default_rng(SEED).choice(n, cap, replace=False))
        out = {"positions": rows_of(res.device_pointers()["positions"], 8, n, idx).view(np.int64)[:, 0].astype(np.float64)}
        for i, c in enumerate(wl.proj):
            t, w = wl.descs[c]
            raw = rows_of(*res.column_device(i), n, idx)
            out[f"col{c}"] = (raw[:, :w].astype(np.float32) if t == N.ATTR_STRING else
                              raw.view(np.int32)[:, 0].astype(np.float64) if t == N.ATTR_INTEGER else raw.view(np.float32)[:, 0])
        aggs = []
        for a, (kind, col) in enumerate(wl.aggs):
            gi, gf, valid = res.agg(a)
            integral = kind == N.AGG_COUNT or wl.descs[col][0] == N.ATTR_INTEGER
            aggs.append((float(gi) if integral else gf) if valid else np.nan)
        out["aggs"] = np.asarray(aggs, dtype=np.float64)
        for name, arr in out.items():
            np.save(os.path.join(out_dir, f"sel{s}_{name}.npy"), arr)


def scan_host_rows(ctx, mbcol, wl, host_cols, rows, terms, want, position_base):
    """Context.scan_host with the row count given explicitly (untouched columns are passed as a dummy buffer)."""
    import ctypes as C
    N = mbcol._native
    from mbcol.engine import Result, pack_terms
    ncols = len(wl.descs)
    descs = (N.mbc_coldesc * ncols)(*[N.mbc_coldesc(int(t), int(w)) for t, w in wl.descs])
    ptrs = (C.c_void_p * ncols)(*[C.c_void_p(a.ctypes.data) for a in host_cols])
    tarr, nt, keep = pack_terms(terms)
    parr = (C.c_int32 * max(len(wl.proj), 1))(*wl.proj)
    aarr = (N.mbc_aggspec * max(len(wl.aggs), 1))(*[N.mbc_aggspec(int(k), int(c)) for k, c in wl.aggs])
    h = C.c_void_p()
    N.check(N.lib().mbc_scan_host(ctx._h, ncols, descs, ptrs, rows, position_base, tarr, nt, parr, len(wl.proj), want, aarr,
                                  len(wl.aggs), C.byref(h)))
    del keep
    return Result(ctx, h, [wl.descs[c] for c in wl.proj], want, len(wl.aggs))


def check_sharded_step(wl, table, terms, shard, rank, world, rows, proj_descs, mbcol, dist, dev, torch):
    """One un-timed step of the multi-GPU path, verified on rank 0: the gathered rows against the oracle on a regenerated
    1 M-row window of EVERY rank's position range, strictly ascending positions, total == sum of the ranks' counts, and the
    folded COUNT/SUM/MIN/MAX against the gathered columns themselves."""
    N = mbcol._native
    s = wl.sels[wl.gather_query]
    res = table.scan(terms[s], proj=wl.proj, want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG, aggs=wl.aggs)
    shard.gather(res, beside_next_scan=False)
    mine = torch.tensor([res.count], dtype=torch.int64, device=dev)
    allc = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allc, mine)                                     # an independent path for the per-rank counts (NCCL)
    out = None
    if rank == 0:
        from oracle import oracle as orc
        orc.build()
        total, cnts = shard.collect()
        ok = cnts == [int(c.item()) for c in allc] and total == sum(cnts)
        pos = shard.positions(0, total)
        ok = ok and bool(np.all(np.diff(pos) > 0)) and (total == 0 or (pos[0] >= 0 and pos[-1] < rows * world))
        cols = [shard.column(i, 0, total) for i in range(len(wl.proj))]
        window = min(1_000_000, rows)
        checked = 0
        for r in range(world):                                      # the oracle on a window of every rank's slice
            lo = r * rows + (rows - window) // 3
            host = wl.host_columns(orc, window, lo)
            exp = orc.scan(wl.descs, host, wl.terms(orc.Term, s), proj=wl.proj, nthreads=orc.max_threads())
            a, b = np.searchsorted(pos, lo), np.searchsorted(pos, lo + window)
            ok = ok and np.array_equal(pos[a:b] - lo, exp["positions"])
            for i, c in enumerate(wl.proj):
                want = host[c][exp["positions"]]
                got = cols[i][a:b]
                ok = ok and (np.array_equal(got.view(np.uint32), want.view(np.uint32)) if wl.descs[c][0] != 0 else np.array_equal(got, want))
            checked += int(b - a)
        aggs_ok = True
        folded = []
        for a_i, (kind, col) in enumerate(wl.aggs):
            ctype = N.ATTR_INTEGER if kind == 0 else wl.descs[col][0]
            gi, gf, gv = shard.agg(a_i, kind, ctype)
            folded.append(gi if ctype == N.ATTR_INTEGER else gf)
            if kind == 0:
                aggs_ok = aggs_ok and gi == total
                continue
            if col not in wl.proj:
                continue
            v = cols[wl.proj.index(col)]
            if ctype == N.ATTR_INTEGER:
                ref = int(v.astype(np.int64).sum()) if kind == 1 else int(v.min()) if kind == 2 else int(v.max())
                aggs_ok = aggs_ok and (total == 0 or gi == ref)
            else:
                ref = float(v.astype(np.float64).sum()) if kind == 1 else float(v.min()) if kind == 2 else float(v.max())
                aggs_ok = aggs_ok and (total == 0 or abs(gf - ref) <= 1e-6 * max(abs(ref), 1e-30))
        shard.release()
        out = {"ok": bool(ok and aggs_ok), "rows_gathered": int(total), "rank_counts": cnts, "window_rows_per_rank": window,
               "rows_checked_against_oracle": checked, "aggregates_checked_against_gathered_columns": bool(aggs_ok),
               "folded_aggregates": folded, "positions_strictly_ascending": bool(np.all(np.diff(pos) > 0))}
    shard.fence()
    res.close()
    dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c5"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (0 = the workload's: 100 M for c2, 500 M for c5)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-rows", type=int, default=0, help="--impl reference: rows per scan (0 = the full C2 table / 100 M rows of C5)")
    ap.add_argument("--cpu-sample-rows", type=int, default=8_000_000, help="rows of the cpu_baseline sample of the GPU arm")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="tuning runs only: skip the end-to-end leg (the line then carries e2e: null)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as .npy files under DIR (one GPU)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or max(world, args.gpus) > 1):
        ap.error("--dump-outputs writes the outputs of the GPU path on one GPU (--impl ours --gpus 1)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under it
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port", "29577",
                                   os.path.abspath(__file__)] + sys.argv[1:])
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
