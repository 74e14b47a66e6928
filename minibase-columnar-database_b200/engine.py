"""Thin object layer over the C ABI: Context / Table / Result.

Nothing is computed here; every method is one libmbcol.so call plus numpy views of the
buffers it returns.  The Java-surface mirror (columnar.py, iterator.py, index.py, input.py)
is written against this layer.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _native as N


@dataclass
class Term:
    """One CondExpr term, 0-based columns.  lhs/rhs = ("col", idx) | ("int", v) | ("real", v) | ("str", bytes)."""
    op: int
    lhs: tuple
    rhs: tuple
    conj: int = 0


def _fill_operand(o: N.mbc_operand, spec: tuple, keep: list) -> None:
    kind, val = spec
    o.kind, o.type, o.col, o.lit_i, o.lit_f, o.lit_slen, o.lit_s = 0, 0, 0, 0, 0.0, 0, None
    if kind == "col":
        o.kind, o.type, o.col = N.OPERAND_OUTER, N.ATTR_SYMBOL, int(val)
    elif kind == "icol":
        o.kind, o.type, o.col = N.OPERAND_INNER, N.ATTR_SYMBOL, int(val)
    elif kind == "int":
        o.kind, o.type = N.OPERAND_LITERAL, N.ATTR_INTEGER
        o.lit_i = int(np.int32(np.int64(val) & 0xFFFFFFFF if not (-2**31 <= int(val) < 2**31) else val))
    elif kind == "real":
        o.kind, o.type, o.lit_f = N.OPERAND_LITERAL, N.ATTR_REAL, float(np.float32(val))
    elif kind == "str":
        b = val.encode("utf-8") if isinstance(val, str) else bytes(val)
        buf = (C.c_uint8 * max(len(b), 1)).from_buffer_copy(b + (b"\0" if not b else b""))
        keep.append(buf)
        o.kind, o.type, o.lit_slen = N.OPERAND_LITERAL, N.ATTR_STRING, len(b)
        o.lit_s = C.cast(buf, C.POINTER(C.c_uint8))
    else:
        raise ValueError(f"unknown operand kind {kind!r}")


def pack_terms(terms: Sequence[Term]):
    """Term list -> (ctypes array, keepalive list).  Terms are sorted by conjunct id (stable)."""
    terms = sorted(terms, key=lambda t: t.conj)
    arr = (N.mbc_term * max(len(terms), 1))()
    keep: list = []
    for i, t in enumerate(terms):
        arr[i].op, arr[i].conj_id = int(t.op), int(t.conj)
        _fill_operand(arr[i].lhs, t.lhs, keep)
        _fill_operand(arr[i].rhs, t.rhs, keep)
    return arr, len(terms), keep


def _np_from_ptr(ptr: int, nbytes: int, dtype) -> np.ndarray:
    if not ptr or nbytes == 0:
        return np.empty(0, dtype=dtype)
    buf = (C.c_uint8 * nbytes).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype)


class Context:
    """One GPU.  Replaces global.SystemDefs' buffer pool + DB singletons for this path."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        N.check(N.lib().mbc_init(device, C.byref(self._h)))
        self.device = device

    def close(self) -> None:
        if self._h:
            N.lib().mbc_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int) -> None:
        N.check(N.lib().mbc_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self) -> None:
        N.check(N.lib().mbc_sync(self._h))

    @property
    def kernel_launches(self) -> int:
        return int(N.lib().mbc_kernel_launches(self._h))

    @property
    def h2d_bytes(self) -> int:
        return int(N.lib().mbc_h2d_bytes(self._h))

    @property
    def last_kernel_ms(self) -> float:
        return float(N.lib().mbc_last_kernel_ms(self._h))

    def create_table(self, coldescs: Sequence[tuple], nrows: int, position_base: int = 0) -> "Table":
        return Table(self, coldescs, nrows, position_base)

    def ingest_dbfile(self, db_bytes, cf_name: str) -> "Table":
        """K1: decode a reference-format DB file image into a resident table."""
        data = np.frombuffer(db_bytes, dtype=np.uint8)
        h = C.c_void_p()
        N.check(N.lib().mbc_table_ingest_dbfile(self._h, data.ctypes.data_as(C.c_void_p), data.size,
                                                cf_name.encode(), C.byref(h)))
        return Table._adopt(self, h)

    def scan_host(self, coldescs: Sequence[tuple], host_cols: Sequence[np.ndarray], terms: Sequence[Term],
                  proj: Sequence[int] = (), want: int = 0, aggs: Sequence[tuple] = (), position_base: int = 0) -> "Result":
        """End-to-end scan over host-resident columns (H2D streaming + scan + D2H)."""
        ncols = len(coldescs)
        descs = (N.mbc_coldesc * ncols)(*[N.mbc_coldesc(int(t), int(w)) for t, w in coldescs])
        nrows = _rows_of(host_cols[0], coldescs[0])
        if len(host_cols) != ncols:
            raise ValueError(f"{len(host_cols)} host columns for {ncols} column descriptors")
        for c, ((t, w), a) in enumerate(zip(coldescs, host_cols)):     # the library reads nrows * width bytes from every pointer
            dt = np.int32 if t == N.ATTR_INTEGER else np.float32 if t == N.ATTR_REAL else np.uint8
            if not isinstance(a, np.ndarray) or a.dtype != dt or not a.flags["C_CONTIGUOUS"]:
                raise ValueError(f"host column {c}: a C-contiguous {np.dtype(dt).name} array is required "
                                 f"(got {getattr(a, 'dtype', type(a))}); buffers are not copied, so pinned memory stays pinned")
            if a.size != nrows * (w if t == N.ATTR_STRING else 1):
                raise ValueError(f"host column {c}: {a.size} elements for {nrows} rows of width {w}")
        ptrs = (C.c_void_p * ncols)(*[C.c_void_p(a.ctypes.data) for a in host_cols])
        tarr, nt, keep = pack_terms(terms)
        parr = (C.c_int32 * max(len(proj), 1))(*proj)
        aarr = (N.mbc_aggspec * max(len(aggs), 1))(*[N.mbc_aggspec(int(k), int(c)) for k, c in aggs])
        h = C.c_void_p()
        N.check(N.lib().mbc_scan_host(self._h, ncols, descs, ptrs, nrows, position_base, tarr, nt, parr, len(proj),
                                      want, aarr, len(aggs), C.byref(h)))
        del keep
        return Result(self, h, [coldescs[c] for c in proj], want, len(aggs))


def _rows_of(arr: np.ndarray, desc: tuple) -> int:
    t, w = desc
    return arr.size // w if t == N.ATTR_STRING else arr.size


class Table:
    """A device-resident Columnarfile: one contiguous array per column + deleted bitmap + bitmap indexes."""

    def __init__(self, ctx: Context, coldescs: Sequence[tuple], nrows: int, position_base: int = 0):
        self.ctx = ctx
        n = len(coldescs)
        descs = (N.mbc_coldesc * n)(*[N.mbc_coldesc(int(t), int(w)) for t, w in coldescs])
        self._h = C.c_void_p()
        N.check(N.lib().mbc_table_create(ctx._h, n, descs, nrows, position_base, C.byref(self._h)))
        self.coldescs = [(int(t), int(w)) for t, w in coldescs]
        self.nrows = nrows
        self.position_base = position_base

    @classmethod
    def _adopt(cls, ctx: Context, handle: C.c_void_p) -> "Table":
        self = cls.__new__(cls)
        self.ctx, self._h = ctx, handle
        self.nrows = int(N.lib().mbc_table_nrows(handle))
        self.position_base = 0
        self.coldescs = []
        for c in range(int(N.lib().mbc_table_ncols(handle))):
            d = N.mbc_coldesc()
            N.check(N.lib().mbc_table_coldesc(handle, c, C.byref(d)))
            self.coldescs.append((int(d.type), int(d.width)))
        return self

    def close(self) -> None:
        if self._h:
            N.lib().mbc_table_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_column(self, col: int, values: np.ndarray) -> None:
        t, w = self.coldescs[col]
        if t == N.ATTR_INTEGER:
            a = np.ascontiguousarray(values, dtype=np.int32)
        elif t == N.ATTR_REAL:
            a = np.ascontiguousarray(values, dtype=np.float32)
        else:
            a = np.ascontiguousarray(values, dtype=np.uint8).reshape(-1)
            if a.size != self.nrows * w:
                raise ValueError(f"string column {col}: expected {self.nrows}x{w} bytes, got {a.size}")
        N.check(N.lib().mbc_table_load_column(self._h, col, a.ctypes.data_as(C.c_void_p), self.nrows))

    def read_column(self, col: int) -> np.ndarray:
        t, w = self.coldescs[col]
        if t == N.ATTR_STRING:
            out = np.empty((self.nrows, w), dtype=np.uint8)
        else:
            out = np.empty(self.nrows, dtype=np.int32 if t == N.ATTR_INTEGER else np.float32)
        N.check(N.lib().mbc_table_read_column(self._h, col, out.ctypes.data_as(C.c_void_p), self.nrows))
        return out

    def generate(self, col: int, kind: int, seed: int, domain: int = 0) -> None:
        N.check(N.lib().mbc_table_generate(self._h, col, kind, C.c_uint64(seed), domain))

    def set_deleted(self, words64: np.ndarray) -> None:
        a = np.ascontiguousarray(words64, dtype=np.uint64)
        N.check(N.lib().mbc_table_set_deleted(self._h, a.ctypes.data_as(C.c_void_p), a.size))

    def column_device(self, col: int) -> tuple[int, int]:
        p, s = C.c_void_p(), C.c_int32()
        N.check(N.lib().mbc_table_column_device(self._h, col, C.byref(p), C.byref(s)))
        return int(p.value or 0), int(s.value)

    # ---- scans -----------------------------------------------------------------------------
    def _run(self, fn, terms, proj, want, aggs) -> "Result":
        tarr, nt, keep = pack_terms(terms)
        parr = (C.c_int32 * max(len(proj), 1))(*proj)
        aarr = (N.mbc_aggspec * max(len(aggs), 1))(*[N.mbc_aggspec(int(k), int(c)) for k, c in aggs])
        h = C.c_void_p()
        N.check(fn(self._h, tarr, nt, parr, len(proj), want, aarr, len(aggs), C.byref(h)))
        del keep
        return Result(self.ctx, h, [self.coldescs[c] for c in proj], want, len(aggs))

    def scan(self, terms: Sequence[Term], proj: Sequence[int] = (), want: int = 0, aggs: Sequence[tuple] = ()) -> "Result":
        """K2: fused filter -> ordered positions -> projection -> aggregates."""
        return self._run(N.lib().mbc_scan, terms, proj, want, aggs)

    def bitmap_scan(self, terms: Sequence[Term], proj: Sequence[int] = (), want: int = 0, aggs: Sequence[tuple] = ()) -> "Result":
        """K4+K5: CNF over bitmap indexes."""
        return self._run(N.lib().mbc_bitmap_scan, terms, proj, want, aggs)

    def sort(self, key_cols: Sequence[int], descending: bool = False, proj: Sequence[int] = (), want: int = 0) -> "Result":
        """ColumnarSort: positions (and projected fields) of the live rows ordered by the key columns, ties by position."""
        karr = (C.c_int32 * max(len(key_cols), 1))(*key_cols)
        parr = (C.c_int32 * max(len(proj), 1))(*proj)
        h = C.c_void_p()
        N.check(N.lib().mbc_sort(self._h, karr, len(key_cols), 1 if descending else 0, parr, len(proj), want, C.byref(h)))
        return Result(self.ctx, h, [self.coldescs[c] for c in proj], want, 0)

    def group_aggregate(self, terms: Sequence[Term], key_cols: Sequence[int], aggs: Sequence[tuple] = (),
                        want: int = N.WANT_COLUMNS | N.WANT_POSITIONS | N.WANT_AGG | N.WANT_HOST) -> "Result":
        """GROUP BY key_cols over the rows that satisfy the CNF: one row per group in ascending key order.  The result's
        columns are the key columns (values of each group's lowest-position row), its positions those rows' positions,
        and group_agg(i) aggregate i of every group; count = number of groups."""
        tarr, nt, keep = pack_terms(terms)
        karr = (C.c_int32 * max(len(key_cols), 1))(*key_cols)
        aarr = (N.mbc_aggspec * max(len(aggs), 1))(*[N.mbc_aggspec(int(k), int(c)) for k, c in aggs])
        h = C.c_void_p()
        N.check(N.lib().mbc_group_aggregate(self._h, tarr, nt, karr, len(key_cols), aarr, len(aggs), want, C.byref(h)))
        del keep
        return Result(self.ctx, h, [self.coldescs[c] for c in key_cols], want, len(aggs))

    def top_k(self, terms: Sequence[Term], key_cols: Sequence[int], k: int, descending: bool = False, proj: Sequence[int] = (),
              want: int = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST) -> "Result":
        """ORDER BY key_cols LIMIT k over the rows that satisfy the CNF: the first min(k, Q) rows of sort()'s order over
        the Q qualifying rows (ties by ascending position in both directions), with their positions and projected fields."""
        tarr, nt, keep = pack_terms(terms)
        karr = (C.c_int32 * max(len(key_cols), 1))(*key_cols)
        parr = (C.c_int32 * max(len(proj), 1))(*proj)
        h = C.c_void_p()
        N.check(N.lib().mbc_topk(self._h, tarr, nt, karr, len(key_cols), 1 if descending else 0, k, parr, len(proj), want,
                                 C.byref(h)))
        del keep
        return Result(self.ctx, h, [self.coldescs[c] for c in proj], want, 0)

    # ---- bitmap indexes --------------------------------------------------------------------
    def bitmap_build(self, col: int) -> None:
        N.check(N.lib().mbc_bitmap_build(self._h, col))

    def bitmap_exists(self, col: int) -> bool:
        return bool(N.lib().mbc_bitmap_exists(self._h, col))

    def bitmap_layout(self, col: int) -> tuple[int, int]:
        """(BITMAP_NONE / BITMAP_DENSE / BITMAP_SPARSE, HBM bytes) of the column's bitmap index."""
        nbytes = C.c_int64()
        layout = N.lib().mbc_bitmap_layout(self._h, col, C.byref(nbytes))
        if layout < 0:
            N.check(layout)
        return int(layout), int(nbytes.value)

    def bitmap_values(self, col: int):
        p, n = C.c_void_p(), C.c_int64()
        N.check(N.lib().mbc_bitmap_values(self._h, col, C.byref(p), C.byref(n)))
        t, w = self.coldescs[col]
        if t == N.ATTR_STRING:
            return _np_from_ptr(p.value, n.value * w, np.uint8).reshape(-1, w).copy()
        return _np_from_ptr(p.value, n.value * 4, np.int32).copy()

    def bitmap_get(self, col: int, value) -> np.ndarray:
        """The value's bitmap as BitSet.toLongArray()-ordered uint64 words."""
        t, w = self.coldescs[col]
        if t == N.ATTR_STRING:
            b = value.encode("utf-8") if isinstance(value, str) else bytes(value)
            v = np.zeros(w, dtype=np.uint8)
            v[:min(len(b), w)] = np.frombuffer(b[:w], dtype=np.uint8)
            if len(b) > w:                   # can never have been indexed
                return np.zeros((self.nrows + 63) // 64, dtype=np.uint64)
        else:
            v = np.array([value], dtype=np.int32)
        out = np.zeros((self.nrows + 63) // 64, dtype=np.uint64)
        N.check(N.lib().mbc_bitmap_get(self._h, col, v.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), out.size))
        return out


def bitmap_join(outer: Table, inner: Table, join_terms: Sequence[Term], proj: Sequence[tuple], want: int,
                aggs: Sequence[tuple] = (), outer_sel: Optional["Result"] = None,
                inner_sel: Optional["Result"] = None) -> "Result":
    """K6: BitMapQuery.executeJoin.  proj = [(rel, col)] with rel 1 = outer, 2 = inner."""
    tarr, nt, keep = pack_terms(join_terms)
    parr = (N.mbc_projspec * max(len(proj), 1))(*[N.mbc_projspec(int(r), int(c)) for r, c in proj])
    aarr = (N.mbc_aggspec * max(len(aggs), 1))(*[N.mbc_aggspec(int(k), int(c)) for k, c in aggs])
    h = C.c_void_p()
    N.check(N.lib().mbc_bitmap_join(outer._h, inner._h, outer_sel._h if outer_sel else None,
                                    inner_sel._h if inner_sel else None, tarr, nt, parr, len(proj), want, aarr,
                                    len(aggs), C.byref(h)))
    del keep
    descs = [(outer if r == N.OPERAND_OUTER else inner).coldescs[c] for r, c in proj]
    return Result(outer.ctx, h, descs, want, len(aggs))


class Result:
    """Owner of one mbc_result; numpy views stay valid until close()."""

    def __init__(self, ctx: Context, handle: C.c_void_p, proj_descs, want: int, nagg: int):
        self.ctx, self._h, self.proj_descs, self.want, self.nagg = ctx, handle, list(proj_descs), want, nagg

    def close(self) -> None:
        if self._h:
            N.lib().mbc_result_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def count(self) -> int:
        return int(N.lib().mbc_result_count(self._h))

    @property
    def kernel_ms(self) -> float:
        """Device time of this result's kernels (waits for a deferred result)."""
        return float(N.lib().mbc_result_kernel_ms(self._h))

    @property
    def phase_ms(self) -> tuple:
        """(pass 1, tile offsets, write pass, aggregate finish) device times of a resident scan, ms."""
        ms = (C.c_float * 4)()
        N.check(N.lib().mbc_result_phase_ms(self._h, ms))
        return tuple(float(x) for x in ms)

    def positions(self) -> np.ndarray:
        return _np_from_ptr(N.lib().mbc_result_positions(self._h), self.count * 8, np.int64)

    def positions2(self) -> np.ndarray:
        return _np_from_ptr(N.lib().mbc_result_positions2(self._h), self.count * 8, np.int64)

    def column(self, i: int) -> np.ndarray:
        w = C.c_int32()
        p = N.lib().mbc_result_column(self._h, i, C.byref(w))
        t, width = self.proj_descs[i]
        if t == N.ATTR_STRING:
            return _np_from_ptr(p, self.count * width, np.uint8).reshape(-1, width)
        return _np_from_ptr(p, self.count * 4, np.int32 if t == N.ATTR_INTEGER else np.float32)

    def tuples(self) -> np.ndarray:
        tl = C.c_int32()
        p = N.lib().mbc_result_tuples(self._h, C.byref(tl))
        if tl.value == 0:
            return np.empty((0, 0), dtype=np.uint8)
        return _np_from_ptr(p, self.count * tl.value, np.uint8).reshape(-1, tl.value)

    def agg(self, i: int):
        """(int64 value, float64 value, valid)."""
        a, f, v = C.c_int64(), C.c_double(), C.c_int32()
        N.check(N.lib().mbc_result_agg(self._h, i, C.byref(a), C.byref(f), C.byref(v)))
        return int(a.value), float(f.value), bool(v.value)

    def group_agg(self, i: int) -> tuple:
        """Aggregate i of a grouped result, one entry per group: (int64 array, float64 array), copies."""
        a, f = C.c_void_p(), C.c_void_p()
        N.check(N.lib().mbc_result_group_agg(self._h, i, C.byref(a), C.byref(f)))
        n = self.count
        return _np_from_ptr(a.value, n * 8, np.int64).copy(), _np_from_ptr(f.value, n * 8, np.float64).copy()

    def bitmap(self) -> np.ndarray:
        n = C.c_int64()
        p = N.lib().mbc_result_bitmap(self._h, C.byref(n))
        return _np_from_ptr(p, n.value * 8, np.uint64)

    def device_pointers(self) -> dict:
        a, b, c, d = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        N.check(N.lib().mbc_result_device(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"positions": a.value or 0, "positions2": b.value or 0, "bitmap": c.value or 0, "aggs": d.value or 0}

    def column_device(self, i: int) -> tuple[int, int]:
        p, s = C.c_void_p(), C.c_int32()
        N.check(N.lib().mbc_result_column_device(self._h, i, C.byref(p), C.byref(s)))
        return int(p.value or 0), int(s.value)


def device_stride(desc: tuple) -> int:
    """Device row stride of a column (csrc/mbc_internal.cuh str_stride): 4 for int / real; char(W) rounded up to 4 below 16
    bytes, to 16 above."""
    t, w = desc
    if t != N.ATTR_STRING:
        return 4
    return (w + 3) // 4 * 4 if w < 16 else (w + 15) // 16 * 16


class Shard:
    """One rank of a table sharded by position (TID) range over the GPUs of a node (SURVEY.md 8e), through the mbc_shard_*
    ABI: every rank scans its slice, then `gather` pushes its positions / projected columns / count / aggregates into the
    root rank's window over NVLink peer memory (a kernel of libmbcol.so; no NCCL).  The root `collect`s.

    Same process (one host driving several GPUs):    root = Shard(ctx0, 0, n); root.create_window(...);
                                                     peer = Shard(ctx1, 1, n); peer.attach(root)
    One process per GPU: the root's `create_window` returns 64 handle bytes that the host ships to the peers by any
    channel (torch.distributed broadcast in bench.py; a socket or a file in a JVM), and the peers `open_window(handle)`.

    Besides scans, the ranks may gather the results of `Table.top_k` / `Table.sort` (into a window shaped like their
    projection) and of `Table.group_aggregate` (into a `create_group_window`); the root then merges them with `top_k` /
    `group_aggregate` after `collect`."""

    def __init__(self, ctx: Context, rank: int, world: int):
        self.ctx, self.rank, self.world = ctx, rank, world
        self._h = C.c_void_p()
        N.check(N.lib().mbc_shard_create(ctx._h, rank, world, C.byref(self._h)))
        self.proj_descs: list = []
        self.capacity = 0

    def close(self) -> None:
        if self._h:
            N.lib().mbc_shard_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _strides(self, proj_descs, nagg: int = 0):
        st = [device_stride(d) for d in proj_descs] + [8] * nagg
        return (C.c_int32 * max(len(st), 1))(*st), len(st)

    def create_window(self, capacity_rows: int, proj_descs: Sequence[tuple]) -> bytes:
        arr, n = self._strides(proj_descs)
        handle = (C.c_uint8 * N.IPC_HANDLE_BYTES)()
        N.check(N.lib().mbc_shard_window_create(self._h, capacity_rows, n, arr, handle))
        self.proj_descs, self.capacity = list(proj_descs), capacity_rows
        return bytes(handle)

    def create_group_window(self, capacity_groups: int, key_descs: Sequence[tuple], nagg: int) -> bytes:
        """A window for the results of Table.group_aggregate: the key columns, then one 8-byte column per aggregate."""
        arr, n = self._strides(key_descs, nagg)
        handle = (C.c_uint8 * N.IPC_HANDLE_BYTES)()
        N.check(N.lib().mbc_shard_window_create(self._h, capacity_groups, n, arr, handle))
        self.proj_descs, self.capacity = list(key_descs), capacity_groups
        return bytes(handle)

    def open_window(self, handle: bytes, capacity_rows: int, proj_descs: Sequence[tuple]) -> None:
        arr, n = self._strides(proj_descs)
        h = (C.c_uint8 * N.IPC_HANDLE_BYTES)(*handle)
        N.check(N.lib().mbc_shard_window_open(self._h, h, capacity_rows, n, arr))
        self.proj_descs, self.capacity = list(proj_descs), capacity_rows

    def attach(self, root: "Shard") -> None:
        N.check(N.lib().mbc_shard_window_attach(self._h, root._h))
        self.proj_descs, self.capacity = list(root.proj_descs), root.capacity

    def gather(self, result: "Result", beside_next_scan: bool = False, copy_engines: bool = False) -> None:
        N.check(N.lib().mbc_shard_gather(self._h, result._h, (1 if beside_next_scan else 0) | (2 if copy_engines else 0)))

    def fence(self) -> None:
        N.check(N.lib().mbc_shard_fence(self._h))

    @property
    def push_ms(self) -> float:
        """Device time of this rank's last push (waits for it)."""
        return float(N.lib().mbc_shard_push_ms(self._h))

    def collect(self) -> tuple:
        """Root: wait for every rank's rows of the last gathered step -> (total rows, [rows per rank])."""
        total = C.c_int64()
        counts = (C.c_int64 * self.world)()
        N.check(N.lib().mbc_shard_collect(self._h, C.byref(total), counts))
        return int(total.value), [int(x) for x in counts]

    def agg(self, i: int, kind: int, col_type: int):
        """Aggregate i folded over the ranks -> (int64 value, float64 value, valid)."""
        a, f, v = C.c_int64(), C.c_double(), C.c_int32()
        N.check(N.lib().mbc_shard_agg(self._h, i, kind, col_type, C.byref(a), C.byref(f), C.byref(v)))
        return int(a.value), float(f.value), bool(v.value)

    def positions(self, first: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.int64)
        N.check(N.lib().mbc_shard_read(self._h, -1, first, n, out.ctypes.data_as(C.c_void_p)))
        return out

    def column(self, i: int, first: int, n: int) -> np.ndarray:
        t, w = self.proj_descs[i]
        st = device_stride((t, w))
        raw = np.empty(n * st, dtype=np.uint8)
        N.check(N.lib().mbc_shard_read(self._h, i, first, n, raw.ctypes.data_as(C.c_void_p)))
        if t == N.ATTR_STRING:
            return raw.reshape(n, st)[:, :w]
        return raw.view(np.int32 if t == N.ATTR_INTEGER else np.float32)

    def release(self) -> None:
        N.check(N.lib().mbc_shard_release(self._h))

    def top_k(self, descs: Sequence[tuple], key_fields: Sequence[int], k: int, descending: bool = False,
              proj_fields: Sequence[int] = (), want: int = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST) -> "Result":
        """Root, after collect: ORDER BY the window fields key_fields LIMIT k over the rows the ranks gathered from
        Table.top_k (or Table.sort).  descs: (type, width) of every window column.  Same contract as Table.top_k over the
        whole sharded table; positions are global."""
        darr = (N.mbc_coldesc * max(len(descs), 1))(*[N.mbc_coldesc(int(t), int(w)) for t, w in descs])
        karr = (C.c_int32 * max(len(key_fields), 1))(*key_fields)
        parr = (C.c_int32 * max(len(proj_fields), 1))(*proj_fields)
        h = C.c_void_p()
        N.check(N.lib().mbc_shard_topk(self._h, darr, karr, len(key_fields), 1 if descending else 0, k, parr, len(proj_fields),
                                       want, C.byref(h)))
        return Result(self.ctx, h, [descs[f] for f in proj_fields], want, 0)

    def group_aggregate(self, key_descs: Sequence[tuple], agg_kinds: Sequence[int], agg_types: Sequence[int],
                        want: int = N.WANT_COLUMNS | N.WANT_POSITIONS | N.WANT_AGG | N.WANT_HOST) -> "Result":
        """Root, after collect: GROUP BY over the grouped results the ranks gathered (Table.group_aggregate with the same
        keys and aggregates).  agg_kinds / agg_types: AGG_* kind and aggregated column type of each aggregate.  Same
        contract as Table.group_aggregate over the whole sharded table."""
        darr = (N.mbc_coldesc * max(len(key_descs), 1))(*[N.mbc_coldesc(int(t), int(w)) for t, w in key_descs])
        karr = (C.c_int32 * max(len(agg_kinds), 1))(*agg_kinds)
        tarr = (C.c_int32 * max(len(agg_types), 1))(*agg_types)
        if len(agg_kinds) != len(agg_types):
            raise ValueError(f"{len(agg_kinds)} aggregate kinds for {len(agg_types)} types")
        h = C.c_void_p()
        N.check(N.lib().mbc_shard_group(self._h, darr, len(key_descs), karr, tarr, len(agg_kinds), want, C.byref(h)))
        return Result(self.ctx, h, list(key_descs), want, len(agg_kinds))
