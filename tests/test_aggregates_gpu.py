"""COUNT / SUM / MIN / MAX, exactly, on every path of libmbcol.so that folds them.

Scan (every write-pass engine, the persistent write_kernel forced on and off), bitmap scan (dense and sparse layouts),
mbc_scan_host (streamed and late-materialised), join (direct, hash, composite keys, the unique-key slot
path at every slot width, theta) and the shard fold.  References are numpy over the qualifying rows:
  - integers in Python / int64 arithmetic, exact;
  - reals of the DYADIC design: multiples of 2^-6 with |x| < 2^17 are exact floats, and every partial sum of up to
    2^27 of them is exact in double in any order, so the GPU's SUM must equal numpy's float64 sum bit for bit whatever
    the engine and its association (joins: while sum |x| * weight < 2^47);
  - the non-dyadic C2 reals against math.fsum with the bound |err| <= n * 2^-53 * sum |x|.
Zero results are compared numerically: the sign of a MIN / MAX that is a zero is not part of the contract.
A real aggregate's as_i64 is Java's (long) of its double.  Needs a B200."""
import math

import numpy as np
import pytest

import mbcol
from mbcol import _native as N
from util import C2_DESCS, c2_columns, c2_device_table, c2_terms, load_table

pytestmark = pytest.mark.gpu

COUNT, SUM, MIN, MAX = 0, 1, 2, 3
I32_MIN, I32_MAX = -2**31, 2**31 - 1
FLT_MAX = float(np.finfo(np.float32).max)
TINY = float(np.float32(2.0**-149))                    # smallest subnormal float
AGGS_ONLY = N.WANT_AGG | N.WANT_HOST
ENGINES = ["twopass", "staged2", "gather", "fused", "persistent"]
GROUP = 8 * 4096                                       # rows of one group of 8 scan tiles
CHUNK = 4 << 20                                        # rows of one mbc_scan_host chunk


@pytest.fixture(params=ENGINES)
def engine(request, monkeypatch):
    """twopass: the default split (write_kernel one CTA per tile + write_staged_kernel above 28 %); staged2: the shallowest
    ring, every group above 12.5 % staged; gather: staged off; fused: the single-residency kernel; persistent: the
    persistent write_kernel that very large tables take, forced at every size (the others force it off)."""
    e = request.param
    monkeypatch.setenv("MBC_SCAN_PATH", "fused" if e == "fused" else "twopass")
    monkeypatch.setenv("MBC_WRITE_STAGED", "0" if e == "gather" else "1")
    monkeypatch.setenv("MBC_WRITE_PERSISTENT_TILES", "1" if e == "persistent" else str(1 << 30))
    if e == "staged2":
        monkeypatch.setenv("MBC_STAGED_STAGES", "2")
        monkeypatch.setenv("MBC_STAGED_MIN_PCT", "0")
    return e


# ---- references ---------------------------------------------------------------------------------------------------------
def java_long(x: float) -> int:
    if math.isnan(x):
        return 0
    if x >= 2.0**63:
        return 2**63 - 1
    if x < -2.0**63:
        return -2**63
    return int(x)


def expect(kind, v):
    """(as_i64, as_f64, valid) of one aggregate over the qualifying values v (int32 or float32)."""
    n = int(v.size)
    if kind == COUNT:
        return n, float(n), True
    if kind != SUM and n == 0:
        return 0, 0.0, False
    if v.dtype == np.int32:
        x = int(v.astype(np.int64).sum()) if kind == SUM else int(v.min() if kind == MIN else v.max())
        return x, float(x), True
    with np.errstate(invalid="ignore"):
        x = float(v.astype(np.float64).sum()) if kind == SUM else float(v.min() if kind == MIN else v.max())
    return java_long(x), x, True


def check_agg(got, exp, what=""):
    gi, gf, gv = got
    ei, ef, ev = exp
    assert gv == ev, (what, got, exp)
    if not ev:
        return
    assert gi == ei, (what, got, exp)
    assert (math.isnan(gf) and math.isnan(ef)) or gf == ef, (what, got, exp)


def expect_all(cols, mask, aggs):
    return [expect(kind, cols[c][mask] if kind != COUNT else mask[mask]) for kind, c in aggs]


def check_scan(res, cols, mask, aggs, what="", exp=None):
    assert res.count == int(mask.sum()), what
    for a, e in enumerate(exp or expect_all(cols, mask, aggs)):
        check_agg(res.agg(a), e, (what, a, aggs[a]))


def dyadic(rng, n, limit=2**23):
    """Multiples of 2^-6 with |x| < limit / 64 (at most 2^17)."""
    return (rng.integers(-limit + 1, limit, n) / 64).astype(np.float32)


def full_range_ints(rng, n):
    v = rng.integers(I32_MIN, I32_MAX + 1, n, dtype=np.int64).astype(np.int32)
    edges = np.array([I32_MIN, I32_MAX, -1, 0], dtype=np.int32)
    v[rng.integers(0, n, min(n, 64))] = edges[rng.integers(0, 4, min(n, 64))]
    v[: min(n, 4)] = edges[: min(n, 4)]
    return v


def selection(rng, n, pattern):
    """Qualifying mask: empty, sparse (<= 4096 of a group's 32 768 rows), mid, dense (> 1/3), or per-group mixed."""
    p = {"empty": 0.0, "sparse": 0.01, "mid": 0.2, "dense": 0.7, "all": 1.0}
    if pattern in p:
        return rng.random(n) < p[pattern]
    cls = np.array([0.0, 0.01, 0.2, 0.7, 1.0])[(np.arange(n) // GROUP) % 5]
    return rng.random(n) < cls


def sel_terms(col=0):
    return [mbcol.Term(N.OP_EQ, ("col", col), ("int", 1), 0)]


# ---- scan: every engine -------------------------------------------------------------------------------------------------
EXACT_AGGS = [(COUNT, 0), (SUM, 1), (MIN, 1), (MAX, 1), (SUM, 2), (MIN, 2), (MAX, 2)]


@pytest.mark.parametrize("nrows", [1, 4095, 4097, 32_767, 32_769, 2_000_003, 6_000_000])
def test_exact_sums_under_every_engine(ctx, engine, nrows):
    """Full-range ints (INT32_MIN, INT32_MAX, -1, 0 included) and dyadic reals: SUM, MIN, MAX and COUNT exact over empty,
    sparse, mid, dense, mixed and full selections; 6 M rows take more waves than the fused kernel has ring slots.  Once
    with the values projected and positions asked for, once aggregates only and deferred."""
    rng = np.random.default_rng(nrows)
    descs = [(1, 4), (1, 4), (2, 4)]
    cols = [np.zeros(nrows, np.int32), full_range_ints(rng, nrows), dyadic(rng, nrows)]
    t = load_table(ctx, descs, cols)
    patterns = ["mixed", "sparse", "all"] if nrows > 4_000_000 else ["empty", "sparse", "mid", "dense", "mixed", "all"]
    for pattern in patterns:
        mask = selection(rng, nrows, pattern)
        cols[0] = mask.astype(np.int32)
        t.load_column(0, cols[0])
        terms = [] if pattern == "all" else sel_terms()
        exp = expect_all(cols, mask, EXACT_AGGS)
        res = t.scan(terms, proj=[1, 2], want=N.WANT_POSITIONS | N.WANT_COLUMNS | AGGS_ONLY, aggs=EXACT_AGGS)
        np.testing.assert_array_equal(res.positions(), np.nonzero(mask)[0])
        check_scan(res, cols, mask, EXACT_AGGS, pattern, exp)
        res.close()
        res = t.scan(terms, want=N.WANT_AGG, aggs=EXACT_AGGS)           # device-resident: completes asynchronously
        check_scan(res, cols, mask, EXACT_AGGS, (pattern, "deferred"), exp)
        res.close()
    t.close()


def test_integer_sum_past_2_53(ctx, engine):
    """8 Mi ints near INT32_MAX sum to about 2^54 (and a twin near INT32_MIN to about -2^54): as_i64 exact, as_f64 its
    double."""
    n = 8 << 20
    rng = np.random.default_rng(53)
    descs = [(1, 4), (1, 4), (1, 4)]
    cols = [np.zeros(n, np.int32), (I32_MAX - rng.integers(0, 1000, n)).astype(np.int32),
            (I32_MIN + rng.integers(0, 1000, n)).astype(np.int32)]
    t = load_table(ctx, descs, cols)
    aggs = [(COUNT, 0), (SUM, 1), (SUM, 2), (MIN, 1), (MAX, 2)]
    for pattern in ("all", "dense"):
        mask = selection(rng, n, pattern)
        cols[0] = mask.astype(np.int32)
        t.load_column(0, cols[0])
        res = t.scan([] if pattern == "all" else sel_terms(), want=AGGS_ONLY, aggs=aggs)
        check_scan(res, cols, mask, aggs, pattern)
        assert res.agg(1)[0] > 2**53 and res.agg(2)[0] < -2**53
        for a in (1, 2):
            assert res.agg(a)[1] == float(res.agg(a)[0])
        res.close()
    t.close()


def _neighbours(p, n):
    """A non-qualifying row q and a deleted row d next to p."""
    q = p + 1 if p + 1 < n else p - 1
    d = p - 1 if p >= 1 and p - 1 != q else (p + 2 if p + 2 < n else p - 2)
    return q, d


PLANT_AGGS = [(COUNT, 0), (MAX, 1), (MIN, 2), (MAX, 3), (MIN, 4), (SUM, 1), (SUM, 3)]


def _plant(cols, p, q, d):
    """Unique int MAX / MIN and real MAX / MIN on row p; more extreme values on q (made non-qualifying) and d."""
    saved = [c[[p, q, d]].copy() for c in cols]
    cols[0][p], cols[0][q], cols[0][d] = 1, 0, 1
    for c, (vp, vq, vd) in zip(range(1, 5), ((10**6, I32_MAX, I32_MAX - 1), (-10**6, I32_MIN, I32_MIN + 1),
                                             (5000.5, FLT_MAX, 1e30), (-5000.25, -FLT_MAX, -1e30))):
        cols[c][p], cols[c][q], cols[c][d] = vp, vq, vd
    return saved


def _unplant(cols, p, q, d, saved):
    for c, s in zip(cols, saved):
        c[[p, q, d]] = s


def _plant_columns(rng, n, pattern):
    mask = selection(rng, n, pattern)
    return [mask.astype(np.int32), rng.integers(-1000, 1000, n).astype(np.int32), rng.integers(-1000, 1000, n).astype(np.int32),
            dyadic(rng, n, 64_000), dyadic(rng, n, 64_000)]


def test_extremum_placement(ctx, engine):
    """A unique MIN / MAX on a qualifying row at each tile and group edge and the last row of a ragged tail, in sparse,
    mid and dense tiles; a more extreme value on the non-qualifying neighbour and on a deleted neighbour must not win.
    One case again with a position base past 2^32."""
    n = 100_003
    descs = [(1, 4), (1, 4), (1, 4), (2, 4), (2, 4)]
    rng = np.random.default_rng(7)
    cases = [(p, pat, 0) for pat in ("sparse", "mid", "dense") for p in (0, 2047, 2048, 4095, 4096, 32_767, 32_768, n - 1)]
    cases.append((4096, "mid", (1 << 32) + 7))
    for p, pattern, base in cases:
        cols = _plant_columns(rng, n, pattern)
        q, d = _neighbours(p, n)
        _plant(cols, p, q, d)
        dele = np.unique(np.concatenate([rng.integers(0, n, n // 50), [d]]))
        dele = dele[dele != p]
        t = load_table(ctx, descs, cols, base)
        t.set_deleted(mbcol_bits(dele, n))
        mask = (cols[0] == 1)
        mask[dele] = False
        res = t.scan(sel_terms(), proj=[3, 1], want=N.WANT_COLUMNS | AGGS_ONLY, aggs=PLANT_AGGS)
        check_scan(res, cols, mask, PLANT_AGGS, (p, pattern, base))
        assert [res.agg(a)[1] for a in (1, 2, 3, 4)] == [10**6, -10**6, 5000.5, -5000.25], (p, pattern)
        res.close(); t.close()


def mbcol_bits(positions, n):
    words = np.zeros((n + 63) // 64, dtype=np.uint64)
    positions = np.asarray(positions, dtype=np.int64)
    np.bitwise_or.at(words, positions >> 6, np.uint64(1) << (positions & 63).astype(np.uint64))
    return words


def test_extremum_at_scan_host_chunk_edges(ctx):
    """mbc_scan_host folds partials across 4 Mi-row chunks: the extremum on either side of each chunk edge and on the
    last row, in sparse, mid and dense tiles."""
    n = 9_000_011
    descs = [(1, 4), (1, 4), (1, 4), (2, 4), (2, 4)]
    rng = np.random.default_rng(11)
    for pattern in ("sparse", "mid", "dense"):
        cols = _plant_columns(rng, n, pattern)
        for p in (CHUNK - 1, CHUNK, 2 * CHUNK - 1, 2 * CHUNK, n - 1):
            q, d = _neighbours(p, n)
            saved = _plant(cols, p, q, d)
            cols[0][d] = 0                                                  # no deleted rows here: d does not qualify
            mask = cols[0] == 1
            res = ctx.scan_host(descs, cols, sel_terms(), want=AGGS_ONLY, aggs=PLANT_AGGS)
            check_scan(res, cols, mask, PLANT_AGGS, (p, pattern))
            assert [res.agg(a)[1] for a in (1, 2, 3, 4)] == [10**6, -10**6, 5000.5, -5000.25], (p, pattern)
            res.close()
            _unplant(cols, p, q, d, saved)


def test_real_edge_values(ctx, engine):
    """±inf, ±FLT_MAX, ±smallest subnormal and interleaved ±0.0: MIN / MAX exact, SUM with +inf is +inf, SUM with both
    infinities NaN (as_i64 0), SUM of subnormals and zeros exact."""
    n = 300_007
    rng = np.random.default_rng(17)
    cls = rng.choice(6, n, p=[0.80, 0.05, 0.0005, 0.0005, 0.0005, 0.1485]).astype(np.int32)
    cls[[0, 4095, n - 1]] = [3, 4, 2]
    r = np.where(np.arange(n) % 2 == 0, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
    sub = np.float32(TINY) * rng.integers(1, 4, n).astype(np.float32) * np.where(rng.random(n) < 0.5, -1, 1).astype(np.float32)
    r[cls == 1] = sub[cls == 1]
    r[cls == 2] = np.where(rng.random(int((cls == 2).sum())) < 0.5, -FLT_MAX, FLT_MAX).astype(np.float32)
    r[cls == 3] = np.inf
    r[cls == 4] = -np.inf
    r[cls == 5] = dyadic(rng, int((cls == 5).sum()))
    descs = [(1, 4), (2, 4)]
    cols = [cls, r]
    t = load_table(ctx, descs, cols)
    aggs = [(COUNT, 0), (SUM, 1), (MIN, 1), (MAX, 1)]
    for classes, sum_exact in (((0,), True), ((0, 1), True), ((0, 1, 2, 5), False), ((0, 1, 3, 5), True),
                               ((0, 3, 4), True), ((4, 5), True), ((1,), True)):
        mask = np.isin(cls, classes)
        terms = [mbcol.Term(N.OP_EQ, ("col", 0), ("int", k), 0) for k in classes]
        for proj in ([], [1]):
            res = t.scan(terms, proj=proj, want=(N.WANT_COLUMNS if proj else 0) | AGGS_ONLY, aggs=aggs)
            for a, (kind, c) in enumerate(aggs):
                if kind == SUM and not sum_exact:
                    continue
                check_agg(res.agg(a), expect(kind, r[mask] if kind != COUNT else mask[mask]), (classes, proj, kind))
            res.close()
    # the checks above bite: these are the values they compared against
    assert expect(SUM, r[np.isin(cls, (0, 3, 4))])[0] == 0 and math.isnan(expect(SUM, r[np.isin(cls, (0, 3, 4))])[1])
    assert expect(MAX, r[np.isin(cls, (0, 1, 2, 5))])[:2] == (2**63 - 1, FLT_MAX)
    t.close()


def test_eight_aggregates_sharing_a_column(ctx, engine):
    """Eight aggregates over two source columns: every source projected (folded from the gathered values), none projected
    (one gather per source column), and the two mixed.  A ninth is refused."""
    n = 1_000_003
    rng = np.random.default_rng(8)
    mask = selection(rng, n, "mixed")
    descs = [(1, 4), (1, 4), (2, 4), (1, 4)]
    cols = [mask.astype(np.int32), full_range_ints(rng, n), dyadic(rng, n), full_range_ints(rng, n)]
    t = load_table(ctx, descs, cols)
    eight = [(SUM, 1), (MIN, 1), (MAX, 1), (SUM, 2), (MIN, 2), (MAX, 2), (COUNT, 0), (MAX, 1)]
    mixed = [(SUM, 1), (MIN, 1), (MAX, 3), (SUM, 2), (MIN, 2), (MAX, 2), (COUNT, 0), (SUM, 3)]
    for proj, aggs in (([1, 2], eight), ([], eight), ([0], eight), ([1], mixed), ([3, 2], mixed)):
        res = t.scan(sel_terms(), proj=proj, want=(N.WANT_COLUMNS if proj else 0) | AGGS_ONLY, aggs=aggs)
        check_scan(res, cols, mask, aggs, proj)
        res.close()
    with pytest.raises(mbcol.MbcError) as e:
        t.scan(sel_terms(), want=AGGS_ONLY, aggs=eight + [(MIN, 2)])
    assert e.value.status == N.ERR_UNSUPPORTED
    t.close()


@pytest.mark.parametrize("sel", [0.01, 0.5, 1.0])
def test_c2_real_sum_within_the_summation_bound(ctx, oracle, engine, sel):
    """C2's non-dyadic R: SUM within n * 2^-53 * sum |x| of math.fsum (not 1e-6 relative); the integer aggregates exact."""
    nrows = 2_000_003
    t = c2_device_table(ctx, nrows)
    cols = c2_columns(oracle, nrows)
    terms = c2_terms(oracle, sel) if sel < 1 else []
    mask = np.ones(nrows, bool) if sel >= 1 else (cols[0] < terms[0].rhs[1]) & (cols[2] < np.float32(terms[1].rhs[1]))
    aggs = [(COUNT, 0), (SUM, 1), (MIN, 0), (MAX, 0), (SUM, 2), (MIN, 2), (MAX, 2)]
    res = t.scan(terms, proj=[2], want=N.WANT_COLUMNS | AGGS_ONLY, aggs=aggs)
    for a in (0, 1, 2, 3, 5, 6):
        kind, c = aggs[a]
        check_agg(res.agg(a), expect(kind, cols[c][mask] if kind != COUNT else mask[mask]), a)
    x = cols[2][mask].astype(np.float64)
    exact = math.fsum(x)
    bound = x.size * 2.0**-53 * float(np.abs(x).sum())
    assert abs(res.agg(4)[1] - exact) <= bound, (res.agg(4)[1], exact, bound)
    res.close(); t.close()


# ---- bitmap scan --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sparse", [False, True])
def test_bitmap_scan_aggregates(ctx, monkeypatch, sparse):
    """CNF over bitmap indexes (dense layout, and the value-sorted sparse layout forced), rows deleted after the build:
    MIN / MAX / SUM / COUNT exact.  The scan behind every bitmap scan is the selection-only path (no terms, the CNF's
    bitmap as the selection: select_bitmap_kernel)."""
    n = 500_003
    rng = np.random.default_rng(21)
    descs = [(1, 4), (1, 4), (1, 4), (2, 4)]
    cols = [rng.integers(0, 100, n).astype(np.int32), rng.integers(0, 16, n).astype(np.int32), full_range_ints(rng, n),
            dyadic(rng, n)]
    t = load_table(ctx, descs, cols)
    if sparse:
        monkeypatch.setenv("MBC_BM_SPARSE", "1")
    for c in (0, 1):
        t.bitmap_build(c)
        assert t.bitmap_layout(c)[0] == (N.BITMAP_SPARSE if sparse else N.BITMAP_DENSE)
    monkeypatch.delenv("MBC_BM_SPARSE", raising=False)
    dele = np.unique(rng.integers(0, n, n // 20))
    t.set_deleted(mbcol_bits(dele, n))
    live = np.ones(n, bool)
    live[dele] = False
    aggs = [(COUNT, 0), (SUM, 2), (MIN, 2), (MAX, 2), (SUM, 3), (MIN, 3), (MAX, 3)]
    A, B = cols[0], cols[1]
    cases = [([mbcol.Term(N.OP_LT, ("col", 0), ("int", 30), 0), mbcol.Term(N.OP_EQ, ("col", 1), ("int", 3), 0),
               mbcol.Term(N.OP_NE, ("col", 1), ("int", 7), 1)], ((A < 30) | (B == 3)) & (B != 7)),
             ([mbcol.Term(N.OP_EQ, ("col", 0), ("int", 5), 0), mbcol.Term(N.OP_EQ, ("col", 1), ("int", 1), 1)], (A == 5) & (B == 1)),
             ([mbcol.Term(N.OP_GE, ("col", 0), ("int", 20), 0)], A >= 20)]
    for terms, m in cases:
        mask = m & live
        for proj in ([], [2, 3]):
            res = t.bitmap_scan(terms, proj=proj, want=(N.WANT_COLUMNS if proj else 0) | AGGS_ONLY, aggs=aggs)
            check_scan(res, cols, mask, aggs, (len(terms), proj))
            res.close()
    t.close()


# ---- mbc_scan_host ------------------------------------------------------------------------------------------------------
def _pinned_copy(arr):
    import torch
    buf = torch.empty(arr.nbytes, dtype=torch.uint8, pin_memory=True).numpy()
    out = buf.view(arr.dtype).reshape(arr.shape)
    out[...] = arr
    return out


def test_scan_host_sums_equal_the_resident_scan(ctx):
    """9 M+ rows from pageable and from pinned columns (a selective predicate on pinned columns reads the survivors in
    place): dyadic SUM bit-equal to the resident scan and to numpy, every other aggregate exact."""
    n = 9_000_011
    rng = np.random.default_rng(31)
    descs = [(1, 4), (1, 4), (2, 4)]
    cols = [np.zeros(n, np.int32), full_range_ints(rng, n), dyadic(rng, n)]
    t = load_table(ctx, descs, cols)
    for pattern in ("sparse", "mixed", "dense"):
        mask = selection(rng, n, pattern)
        cols[0] = mask.astype(np.int32)
        t.load_column(0, cols[0])
        exp = expect_all(cols, mask, EXACT_AGGS)
        resident = t.scan(sel_terms(), want=AGGS_ONLY, aggs=EXACT_AGGS)
        check_scan(resident, cols, mask, EXACT_AGGS, pattern, exp)
        for pinned in (False, True):
            hc = [_pinned_copy(c) for c in cols] if pinned else cols
            before = ctx.h2d_bytes
            res = ctx.scan_host(descs, hc, sel_terms(), proj=[2], want=N.WANT_COLUMNS | AGGS_ONLY, aggs=EXACT_AGGS)
            moved = ctx.h2d_bytes - before
            if pinned and pattern == "sparse":
                assert moved < 0.5 * 12 * n                                   # late materialisation took place
            elif not pinned:
                assert moved >= 12 * n
            check_scan(res, cols, mask, EXACT_AGGS, (pattern, pinned), exp)
            for a in range(len(EXACT_AGGS)):
                assert res.agg(a) == resident.agg(a), (pattern, pinned, a)
            res.close()
        resident.close()
    t.close()


# ---- join ---------------------------------------------------------------------------------------------------------------
def _key_ids(outer_keys, inner_keys):
    """Dense ids of the join keys (lists of columns; string columns as (n, w) uint8) over both sides."""
    def rec(keys):
        n = len(keys[0])
        dt = [(f"f{i}", (f"V{k.shape[1]}" if k.ndim == 2 else k.dtype)) for i, k in enumerate(keys)]
        out = np.empty(n, dtype=dt)
        for i, k in enumerate(keys):
            out[f"f{i}"] = np.ascontiguousarray(k).view(f"V{k.shape[1]}").reshape(-1) if k.ndim == 2 else k
        return out
    ro, ri = rec(outer_keys), rec(inner_keys)
    _, inv = np.unique(np.concatenate([ro, ri]), return_inverse=True)
    inv = inv.reshape(-1)
    return inv[:len(ro)], inv[len(ro):], int(inv.max()) + 1 if inv.size else 0


def join_reference(ko, ki, omask, imask, ocols, icols, proj, aggs):
    """Aggregates of the equi-join from group counts: COUNT = sum n_o(k) n_i(k); an inner value weighs n_o(its key), an
    outer value n_i(its key); MIN / MAX over the rows that have a partner."""
    K = max(int(ko.max(initial=-1)), int(ki.max(initial=-1))) + 1
    no = np.bincount(ko[omask], minlength=K).astype(np.int64)
    ni = np.bincount(ki[imask], minlength=K).astype(np.int64)
    out = []
    for kind, pi in aggs:
        if kind == COUNT:
            c = int(np.dot(no, ni))
            out.append((c, float(c), True))
            continue
        rel, col = proj[pi]
        keys, m, vals, weight = (ko, omask, ocols[col], ni) if rel == 1 else (ki, imask, icols[col], no)
        k, v = keys[m], vals[m]
        w = weight[k]
        if kind == SUM:
            if v.dtype == np.int32:
                s = np.zeros(K, dtype=np.int64)
                np.add.at(s, k, v.astype(np.int64))
                nz = np.nonzero(weight)[0]
                x = sum(int(a) * int(b) for a, b in zip(s[nz], weight[nz]))
                out.append((x, float(x), True))
            else:
                assert float(np.dot(np.abs(v.astype(np.float64)), w)) < 2.0**47
                x = float(np.dot(v.astype(np.float64), w.astype(np.float64)))
                out.append((java_long(x), x, True))
        else:
            out.append(expect(kind, v[w > 0]))
    return out


def _check_join(res, exp, what=""):
    for a, e in enumerate(exp):
        check_agg(res.agg(a), e, (what, a))


def _sel_bitmap(t, terms):
    return t.scan(terms, want=N.WANT_BITMAP | N.WANT_HOST)


JOIN_PROJ = [(1, 1), (1, 2), (2, 1), (2, 2)]            # outer int, outer real, inner int, inner real
JOIN_AGGS = [(COUNT, 0), (SUM, 2), (SUM, 3), (SUM, 0), (SUM, 1), (MIN, 0), (MAX, 2), (MIN, 3)]


def _join_tables(rng, nO, nI, okey, ikey):
    Od, Id = [(1, 4), (1, 4), (2, 4)], [(1, 4), (1, 4), (2, 4)]
    Oc = [okey, full_range_ints(rng, nO), dyadic(rng, nO, 2**16)]
    Ic = [ikey, full_range_ints(rng, nI), dyadic(rng, nI, 2**16)]
    return Od, Oc, Id, Ic


@pytest.mark.parametrize("mode", ["direct_few", "direct_many", "hash"])
def test_join_aggregates(ctx, monkeypatch, mode):
    """Int equi-join, aggregates only and with the pair list: direct addressing with <= 4096 and with more key groups, and
    the hash map on sparse keys; then side filters and deleted rows on both sides."""
    rng = np.random.default_rng({"direct_few": 1, "direct_many": 2, "hash": 3}[mode])
    if mode == "direct_few":
        nO, nI = 30_000, 200_000
        okey, ikey = rng.integers(0, 3000, nO), rng.integers(-100, 3100, nI)
    elif mode == "direct_many":
        nO, nI = 100_000, 300_000
        okey, ikey = rng.integers(0, 200_000, nO), rng.integers(0, 210_000, nI)
    else:
        domain = rng.integers(I32_MIN, I32_MAX, 5000)
        nO, nI = 20_000, 100_000
        okey = domain[rng.integers(0, 5000, nO)]
        ikey = np.concatenate([domain[rng.integers(0, 5000, nI - 500)], rng.integers(-9, 9, 500)])
    Od, Oc, Id, Ic = _join_tables(rng, nO, nI, okey.astype(np.int32), ikey.astype(np.int32))
    O, I = load_table(ctx, Od, Oc), load_table(ctx, Id, Ic)
    jt = [mbcol.Term(N.OP_EQ, ("col", 0), ("icol", 0), 0)]
    ko, ki, _ = _key_ids([Oc[0]], [Ic[0]])
    allo, alli = np.ones(nO, bool), np.ones(nI, bool)
    exp = join_reference(ko, ki, allo, alli, Oc, Ic, JOIN_PROJ, JOIN_AGGS)
    assert exp[0][0] > 0
    for want in (N.WANT_AGG, N.WANT_POSITIONS | N.WANT_AGG | N.WANT_HOST):
        res = mbcol.bitmap_join(O, I, jt, JOIN_PROJ, want, aggs=JOIN_AGGS)
        _check_join(res, exp, (mode, want))
        res.close()
    # side filters, then deleted rows on both sides
    so = _sel_bitmap(O, [mbcol.Term(N.OP_LT, ("col", 1), ("int", 1 << 30), 0)])
    si = _sel_bitmap(I, [mbcol.Term(N.OP_GE, ("col", 2), ("real", -100.0), 0)])
    omask, imask = Oc[1] < (1 << 30), Ic[2] >= np.float32(-100.0)
    exp = join_reference(ko, ki, omask, imask, Oc, Ic, JOIN_PROJ, JOIN_AGGS)
    res = mbcol.bitmap_join(O, I, jt, JOIN_PROJ, N.WANT_AGG, aggs=JOIN_AGGS, outer_sel=so, inner_sel=si)
    _check_join(res, exp, (mode, "filters"))
    res.close(); so.close(); si.close()
    dO, dI = np.unique(rng.integers(0, nO, nO // 10)), np.unique(rng.integers(0, nI, nI // 10))
    O.set_deleted(mbcol_bits(dO, nO))
    I.set_deleted(mbcol_bits(dI, nI))
    omask[dO] = False
    imask[dI] = False
    so = _sel_bitmap(O, [mbcol.Term(N.OP_LT, ("col", 1), ("int", 1 << 30), 0)])
    si = _sel_bitmap(I, [mbcol.Term(N.OP_GE, ("col", 2), ("real", -100.0), 0)])
    exp = join_reference(ko, ki, omask, imask, Oc, Ic, JOIN_PROJ, JOIN_AGGS)
    for force in ("1", "0"):
        monkeypatch.setenv("MBC_JOIN_UNIQUE", force)
        res = mbcol.bitmap_join(O, I, jt, JOIN_PROJ, N.WANT_AGG, aggs=JOIN_AGGS, outer_sel=so, inner_sel=si)
        _check_join(res, exp, (mode, "deleted", force))
        res.close()
    so.close(); si.close(); O.close(); I.close()


def test_join_aggregates_on_a_composite_key(ctx):
    """char(8) + int composite key: the hash map over two key columns."""
    rng = np.random.default_rng(4)
    from oracle import oracle as orc
    words = [f"w{i:03d}" for i in range(60)] + ["", "abcdefgh"]
    nO, nI = 20_000, 80_000
    Od, Id = [(0, 8), (1, 4), (1, 4), (2, 4)], [(0, 8), (1, 4), (1, 4), (2, 4)]
    Oc = [orc.pack_strings([words[i] for i in rng.integers(0, len(words), nO)], 8), rng.integers(0, 20, nO).astype(np.int32),
          full_range_ints(rng, nO), dyadic(rng, nO, 2**16)]
    Ic = [orc.pack_strings([words[i] for i in rng.integers(0, len(words), nI)], 8), rng.integers(0, 21, nI).astype(np.int32),
          full_range_ints(rng, nI), dyadic(rng, nI, 2**16)]
    O, I = load_table(ctx, Od, Oc), load_table(ctx, Id, Ic)
    jt = [mbcol.Term(N.OP_EQ, ("col", 0), ("icol", 0), 0), mbcol.Term(N.OP_EQ, ("col", 1), ("icol", 1), 1)]
    proj = [(1, 2), (1, 3), (2, 2), (2, 3)]
    ko, ki, _ = _key_ids([Oc[0].reshape(nO, 8), Oc[1]], [Ic[0].reshape(nI, 8), Ic[1]])
    exp = join_reference(ko, ki, np.ones(nO, bool), np.ones(nI, bool), {2: Oc[2], 3: Oc[3]}, {2: Ic[2], 3: Ic[3]}, proj, JOIN_AGGS)
    assert exp[0][0] > 0
    res = mbcol.bitmap_join(O, I, jt, proj, N.WANT_AGG, aggs=JOIN_AGGS)
    _check_join(res, exp, "composite")
    res.close(); O.close(); I.close()


@pytest.mark.parametrize("dense", [True, False])
def test_join_unique_key_slot_widths(ctx, monkeypatch, dense):
    """PK-FK join, aggregates only: the slot path with 0, 1, 2 and 3 distinct outer-side columns (slot widths 0 / 1 / 2 / 4
    words), on a key range the outer keys fill (dense) and one with gaps, forced on and off."""
    rng = np.random.default_rng(5 + dense)
    nO, nI = 50_000, 400_000
    okey = (rng.permutation(nO) - 7) if dense else (rng.choice(3 * nO, nO, replace=False) + 11)
    Od, Id = [(1, 4), (1, 4), (2, 4), (1, 4)], [(1, 4), (1, 4), (2, 4)]
    Oc = [okey.astype(np.int32), full_range_ints(rng, nO), dyadic(rng, nO, 2**16), full_range_ints(rng, nO)]
    Ic = [rng.integers(int(okey.min()) - 20, int(okey.max()) + 20, nI).astype(np.int32), full_range_ints(rng, nI),
          dyadic(rng, nI, 2**16)]
    O, I = load_table(ctx, Od, Oc), load_table(ctx, Id, Ic)
    jt = [mbcol.Term(N.OP_EQ, ("col", 0), ("icol", 0), 0)]
    proj = [(2, 1), (2, 2), (1, 1), (1, 2), (1, 3)]
    inner_aggs = [(COUNT, 0), (SUM, 0), (MAX, 1), (MIN, 0)]
    outer_aggs = [[], [(SUM, 2), (MIN, 2)], [(SUM, 2), (SUM, 3), (MAX, 3), (MIN, 2)],
                  [(SUM, 2), (MIN, 2), (SUM, 3), (MAX, 3)]]
    ko, ki, _ = _key_ids([Oc[0]], [Ic[0]])
    cols = {1: Oc[1], 2: Oc[2], 3: Oc[3]}
    for nouter, extra in enumerate(outer_aggs):
        aggs = inner_aggs + extra
        if nouter == 3:
            aggs = [(COUNT, 0), (SUM, 0), (MAX, 1), (SUM, 2), (MIN, 2), (SUM, 3), (MAX, 3), (SUM, 4)]
        ex = join_reference(ko, ki, np.ones(nO, bool), np.ones(nI, bool), cols, {1: Ic[1], 2: Ic[2]}, proj, aggs)
        for force in ("1", "0"):
            monkeypatch.setenv("MBC_JOIN_UNIQUE", force)
            res = mbcol.bitmap_join(O, I, jt, proj, N.WANT_AGG, aggs=aggs)
            _check_join(res, ex, (nouter, dense, force))
            res.close()
    O.close(); I.close()


def test_join_count_past_2_32(ctx):
    """One key on 70 000 outer x 70 000 inner rows: COUNT = 4.9e9 > 2^32 and an inner int SUM weighted by 70 000 past
    2^53 (aggregates only; integer aggregates)."""
    rng = np.random.default_rng(6)
    nO, nI = 70_000, 70_010
    okey = np.full(nO, 7, np.int32)
    ikey = np.full(nI, 7, np.int32)
    ikey[-10:] = 8
    Od, Id = [(1, 4), (1, 4)], [(1, 4), (1, 4)]
    Oc = [okey, full_range_ints(rng, nO)]
    Ic = [ikey, rng.integers(1 << 29, 3 << 29, nI).astype(np.int32)]
    O, I = load_table(ctx, Od, Oc), load_table(ctx, Id, Ic)
    jt = [mbcol.Term(N.OP_EQ, ("col", 0), ("icol", 0), 0)]
    proj = [(1, 1), (2, 1)]
    aggs = [(COUNT, 0), (SUM, 1), (SUM, 0), (MIN, 1), (MAX, 0), (MIN, 0)]
    ko, ki, _ = _key_ids([Oc[0]], [Ic[0]])
    exp = join_reference(ko, ki, np.ones(nO, bool), np.ones(nI, bool), {1: Oc[1]}, {1: Ic[1]}, proj, aggs)
    assert exp[0][0] == 70_000 * 70_000 > 2**32 and exp[1][0] > 2**53
    res = mbcol.bitmap_join(O, I, jt, proj, N.WANT_AGG, aggs=aggs)
    _check_join(res, exp, "count > 2^32")
    res.close(); O.close(); I.close()


def test_theta_join_aggregates(ctx):
    """outer.a < inner.b on a few thousand rows a side: pair weights from numpy broadcasting."""
    rng = np.random.default_rng(12)
    nO, nI = 3000, 4000
    Od, Id = [(1, 4), (1, 4), (2, 4)], [(1, 4), (1, 4), (2, 4)]
    Oc = [rng.integers(0, 5000, nO).astype(np.int32), full_range_ints(rng, nO), dyadic(rng, nO, 2**16)]
    Ic = [rng.integers(0, 5000, nI).astype(np.int32), full_range_ints(rng, nI), dyadic(rng, nI, 2**16)]
    O, I = load_table(ctx, Od, Oc), load_table(ctx, Id, Ic)
    jt = [mbcol.Term(N.OP_LT, ("col", 0), ("icol", 0), 0)]
    pairs = Oc[0][:, None] < Ic[0][None, :]
    wo, wi = pairs.sum(1).astype(np.int64), pairs.sum(0).astype(np.int64)
    aggs = JOIN_AGGS
    exp = []
    for kind, pi in aggs:
        if kind == COUNT:
            exp.append((int(pairs.sum()), float(pairs.sum()), True))
            continue
        rel, col = JOIN_PROJ[pi]
        v, w = (Oc[col], wo) if rel == 1 else (Ic[col], wi)
        if kind == SUM and v.dtype == np.int32:
            x = sum(int(a) * int(b) for a, b in zip(v, w))
            exp.append((x, float(x), True))
        elif kind == SUM:
            x = float(np.dot(v.astype(np.float64), w.astype(np.float64)))
            exp.append((java_long(x), x, True))
        else:
            exp.append(expect(kind, v[w > 0]))
    res = mbcol.bitmap_join(O, I, jt, JOIN_PROJ, N.WANT_AGG, aggs=aggs)
    _check_join(res, exp, "theta")
    res.close(); O.close(); I.close()


# ---- shard fold ---------------------------------------------------------------------------------------------------------
SHARD_AGGS = [(COUNT, 0), (SUM, 1), (MIN, 1), (MAX, 2), (SUM, 3), (MIN, 3), (MAX, 4)]
SHARD_DESCS = [(1, 4), (1, 4), (1, 4), (2, 4), (2, 4)]


def _shard_agg_type(kind, col):
    return N.ATTR_INTEGER if kind == COUNT else SHARD_DESCS[col][0]


def test_shard_fold_world_1(ctx):
    """mbc_shard_agg of one rank equals the scan's aggregates; a step with no survivors leaves MIN / MAX invalid."""
    n = 1_000_003
    rng = np.random.default_rng(41)
    mask = selection(rng, n, "mixed")
    cols = [mask.astype(np.int32), full_range_ints(rng, n), full_range_ints(rng, n), dyadic(rng, n), dyadic(rng, n)]
    t = load_table(ctx, SHARD_DESCS, cols)
    sh = mbcol.Shard(ctx, 0, 1)
    sh.create_window(n, [SHARD_DESCS[1]])
    for terms, m in ((sel_terms(), mask), ([mbcol.Term(N.OP_EQ, ("col", 0), ("int", 99), 0)], np.zeros(n, bool))):
        res = t.scan(terms, proj=[1], want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG, aggs=SHARD_AGGS)
        sh.gather(res)
        sh.fence()
        tot, _ = sh.collect()
        assert tot == int(m.sum())
        for a, (kind, c) in enumerate(SHARD_AGGS):
            got = sh.agg(a, kind, _shard_agg_type(kind, c))
            assert got == res.agg(a), (a, got, res.agg(a))
            check_agg(got, expect(kind, cols[c][m] if kind != COUNT else m[m]), a)
        sh.release()
        res.close()
    sh.close(); t.close()


@pytest.mark.parametrize("world,live", [(2, 1), (3, 1)])
def test_shard_fold_skips_empty_ranks(oracle, world, live):
    """World 2 and 3 (on distinct GPUs when the box has them): only rank `live` has survivors, with MIN > 0 and MAX < 0,
    so an empty rank that folded its identity or a stale value would show."""
    import torch
    ndev = torch.cuda.device_count()
    per = 200_000 + 4096 + 5
    n = per * world
    rng = np.random.default_rng(43)
    cols = [np.zeros(n, np.int32), rng.integers(1, 1000, n).astype(np.int32), rng.integers(-1000, -1, n).astype(np.int32),
            (rng.integers(1, 4096, n) / 64).astype(np.float32), (rng.integers(-4096, -1, n) / 64).astype(np.float32)]
    mask = np.zeros(n, bool)
    mask[live * per:(live + 1) * per] = rng.random(per) < 0.3
    cols[0] = mask.astype(np.int32)
    ctxs = [mbcol.Context(r % ndev) for r in range(world)]
    tables = [load_table(c, SHARD_DESCS, [x[r * per:(r + 1) * per] for x in cols], r * per) for r, c in enumerate(ctxs)]
    shards = [mbcol.Shard(c, r, world) for r, c in enumerate(ctxs)]
    shards[0].create_window(n, [SHARD_DESCS[1]])
    for s in shards[1:]:
        s.attach(shards[0])
    results = [t.scan(sel_terms(), proj=[1], want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_AGG, aggs=SHARD_AGGS) for t in tables]
    for r in range(world):
        shards[r].gather(results[r])
        shards[r].fence()
        ctxs[r].sync()
    tot, counts = shards[0].collect()
    assert tot == int(mask.sum()) and counts == [res.count for res in results]
    for a, (kind, c) in enumerate(SHARD_AGGS):
        check_agg(shards[0].agg(a, kind, _shard_agg_type(kind, c)), expect(kind, cols[c][mask] if kind != COUNT else mask[mask]), a)
    shards[0].release()
    for res in results:
        res.close()
    for s in shards[1:] + shards[:1]:
        s.close()
    for t in tables:
        t.close()
    for c in ctxs:
        c.close()
