"""mbc_shard_topk / mbc_shard_group: per-rank mbc_topk / mbc_sort / mbc_group_aggregate results gathered into the root's
window and merged there, against the same operator on one table holding every row (and, for GROUP BY, tests/group_oracle.py).

One process drives every rank, as in test_shard_gpu.py: one Context per rank, on distinct GPUs when the box has them, else
all on cuda:0.  Each rank holds a position-range slice of about 250 K rows.  Counts, positions, key values, projected
values, Tuple bytes, COUNT, integer aggregates and real MIN / MAX must be bit-exact; a real SUM within 1e-6 relative (its
partials are added in another association than the single-table fold).  Needs a B200."""
import numpy as np
import pytest

import mbcol
from mbcol import _native as N
from group_oracle import group_aggregate as oracle_group
from util import C2_AGGS, load_table

pytestmark = pytest.mark.gpu

COUNT, SUM, MIN, MAX = N.AGG_COUNT, N.AGG_SUM, N.AGG_MIN, N.AGG_MAX
POS, COLS, TUP, AGG, HOST = N.WANT_POSITIONS, N.WANT_COLUMNS, N.WANT_TUPLES, N.WANT_AGG, N.WANT_HOST
NRANK = 250_000 + 4096 * 3 + 7

# I1, I2, R, S as C2 (so C2_AGGS applies), then K16 (16 values), Z (reals with -0.0 and +0.0), B (ints near 2^31: sums
# pass 2^31 within a group), F (0 everywhere but on rank 1: the filter leaves that rank nothing)
DESCS = [(1, 4), (1, 4), (2, 4), (0, 16), (1, 4), (2, 4), (1, 4), (1, 4)]
I1, I2, R, S, K16, Z, B, F = range(8)
AGGS = C2_AGGS + [(SUM, B), (MIN, R), (MAX, R)]


def _ndev():
    import torch
    return torch.cuda.device_count()


def _columns(world):
    rng = np.random.default_rng(world)
    n = NRANK * world
    words = [rng.integers(97, 123, rng.integers(1, 17)).astype(np.uint8).tobytes() for _ in range(3000)]
    s = np.zeros((n, 16), np.uint8)
    for i, w in enumerate(words):
        s[i::len(words), :len(w)] = np.frombuffer(w, np.uint8)
    s = s[rng.permutation(n)]
    z = rng.choice(np.array([0.0, 1.5, -2.25, 3.0], np.float32), n)
    z[(z == 0) & (np.arange(n) < n // 2)] = np.float32(-0.0)            # -0.0 in the lower ranks, +0.0 in the upper ones
    f = np.zeros(n, np.int32)
    if world > 1:
        f[NRANK:2 * NRANK] = 1
    return [rng.integers(0, 1 << 20, n).astype(np.int32), rng.integers(0, 1 << 20, n).astype(np.int32),
            (rng.random(n, np.float32) * 1000).astype(np.float32), s, rng.integers(0, 16, n).astype(np.int32), z,
            rng.integers(2**31 - 2**20, 2**31 - 1, n).astype(np.int32), f]


def _words(mask):
    return np.packbits(np.append(mask, np.zeros((-mask.size) % 64, bool)), bitorder="little").view(np.uint64)


class Setup:
    """world ranks with their slice of the table, and a reference table holding every row on rank 0's context."""

    def __init__(self, world, deleted=True):
        self.world = world
        self.cols = _columns(world)
        n = NRANK * world
        self.deleted = np.zeros(n, bool)
        if deleted:                                                    # 10 % of rank 0's rows
            self.deleted[np.random.default_rng(7).choice(NRANK, NRANK // 10, replace=False)] = True
        ndev = _ndev()
        self.ctxs = [mbcol.Context(r % ndev) for r in range(world)]
        self.tables = []
        for r, c in enumerate(self.ctxs):
            lo = r * NRANK
            t = load_table(c, DESCS, [col[lo:lo + NRANK] for col in self.cols], position_base=lo)
            t.set_deleted(_words(self.deleted[lo:lo + NRANK]))
            self.tables.append(t)
        self.ref = load_table(self.ctxs[0], DESCS, self.cols)
        self.ref.set_deleted(_words(self.deleted))

    def shards(self):
        return [mbcol.Shard(c, r, self.world) for r, c in enumerate(self.ctxs)]

    def close(self):
        for t in self.tables + [self.ref]:
            t.close()
        for c in self.ctxs:
            c.close()


@pytest.fixture(params=[1, 2, 3], ids=lambda w: f"world{w}")
def setup(request):
    s = Setup(request.param)
    yield s
    s.close()


def _attach(shards):
    for s in shards[1:]:
        s.attach(shards[0])


def _close(shards, results=()):
    for res in results:
        res.close()
    for s in shards[1:] + shards[:1]:
        s.close()


def _gather(shards, ctxs, results, step):
    for r, res in enumerate(results):                                 # rank order; each push has finished before the next
        shards[r].gather(res, beside_next_scan=bool(step & 1), copy_engines=step % 3 == 2)
        shards[r].fence()
        ctxs[r].sync()
    return shards[0].collect()


def _terms(kind):
    if kind == "all":
        return []
    if kind == "none":
        return [mbcol.Term(N.OP_LT, ("col", I1), ("int", 0), 0)]
    return [mbcol.Term(N.OP_LT, ("col", I1), ("int", 600_000), 0), mbcol.Term(N.OP_EQ, ("col", F), ("int", 0), 1)]


def _same(a, b):
    if a.dtype == np.float32:
        a, b = a.view(np.uint32), b.view(np.uint32)
    np.testing.assert_array_equal(a, b)


# ---- GROUP BY ---------------------------------------------------------------------------------------------------------
def _agg_types(aggs):
    return [N.ATTR_INTEGER if k == COUNT else DESCS[c][0] for k, c in aggs]


def _sharded_group(su, key_cols, aggs, terms, step=0, shards=None, cap=None):
    own = shards is None
    if own:
        shards = su.shards()
        shards[0].create_group_window(cap or NRANK * su.world, [DESCS[c] for c in key_cols], len(aggs))
        _attach(shards)
    results = [t.group_aggregate(terms, key_cols, aggs, want=POS | COLS | AGG) for t in su.tables]
    total, counts = _gather(shards, su.ctxs, results, step)
    assert counts == [r.count for r in results] and total == sum(counts)
    res = shards[0].group_aggregate([DESCS[c] for c in key_cols], [k for k, _ in aggs], _agg_types(aggs))
    shards[0].release()
    for r in results:
        r.close()
    if own:
        _close(shards)
    return res


def _check_groups(got, exp, key_cols, aggs):
    assert got.count == exp.count
    np.testing.assert_array_equal(got.positions(), exp.positions())
    for k in range(len(key_cols)):
        _same(got.column(k), exp.column(k))
    for a, (kind, col) in enumerate(aggs):
        gi, gf = got.group_agg(a)
        ei, ef = exp.group_agg(a)
        if kind == SUM and DESCS[col][0] == N.ATTR_REAL:
            assert np.all(np.abs(gf - ef) <= 1e-6 * np.maximum(np.abs(ef), 1e-30)), a
        else:
            np.testing.assert_array_equal(gi, ei)
            np.testing.assert_array_equal(gf.view(np.uint64), ef.view(np.uint64))


@pytest.mark.parametrize("key_cols", [[K16], [I1], [S], [S, I1], [Z]], ids=["k16", "i1", "s", "s_i1", "z"])
def test_group_by_matches_one_table(setup, key_cols):
    su = setup
    shards = su.shards()
    shards[0].create_group_window(NRANK * su.world, [DESCS[c] for c in key_cols], len(AGGS))
    _attach(shards)
    for step, kind in enumerate(["some", "all", "none", "some", "all"]):   # five steps through one window: both slots reused
        terms = _terms(kind)
        got = _sharded_group(su, key_cols, AGGS, terms, step, shards)
        exp = su.ref.group_aggregate(terms, key_cols, AGGS)
        if kind == "none":
            assert got.count == 0
        _check_groups(got, exp, key_cols, AGGS)
        if key_cols == [Z] and kind == "all":                          # -0.0 and +0.0 (in different ranks) are one group
            zero = got.column(0) == 0
            assert zero.sum() == 1 and got.group_agg(0)[0][zero][0] == np.sum(~su.deleted & (su.cols[Z] == 0))
        got.close()
        exp.close()
    _close(shards)


def test_group_by_matches_the_oracle(oracle):
    su = Setup(3)
    try:
        terms = _terms("some")
        for key_cols in ([K16], [S, I1]):
            got = _sharded_group(su, key_cols, AGGS, terms)
            exp = oracle_group(DESCS, su.cols, terms, key_cols, AGGS, deleted_words=_words(su.deleted))
            assert got.count == exp["count"]
            np.testing.assert_array_equal(got.positions(), exp["positions"])
            for k, kv in enumerate(exp["keys"]):
                _same(got.column(k), kv)
            for a, (kind, col) in enumerate(AGGS):
                gi, gf = got.group_agg(a)
                ei, ef = exp["aggs"][a]
                if kind == SUM and DESCS[col][0] == N.ATTR_REAL:
                    assert np.all(np.abs(gf - ef) <= 1e-6 * np.maximum(np.abs(ef), 1e-30)), a
                else:
                    np.testing.assert_array_equal(gi, ei)
                    np.testing.assert_array_equal(gf, ef)
            if key_cols == [K16]:
                assert got.count == 16 and np.all(got.group_agg(5)[0] > 2**31)    # SUM(B) past 2^31 in every group
            got.close()
    finally:
        su.close()


def test_group_by_is_deterministic():
    su = Setup(3)
    try:
        a = _sharded_group(su, [K16], AGGS, [], step=0)
        b = _sharded_group(su, [K16], AGGS, [], step=2)                  # the other gather form
        for i in range(len(AGGS)):
            np.testing.assert_array_equal(a.group_agg(i)[1].view(np.uint64), b.group_agg(i)[1].view(np.uint64))
        np.testing.assert_array_equal(a.positions(), b.positions())
    finally:
        su.close()


def test_group_window_overflow_is_reported():
    su = Setup(2, deleted=False)
    try:
        shards = su.shards()
        shards[0].create_group_window(1000, [DESCS[I1]], 1)
        _attach(shards)
        results = [t.group_aggregate([], [I1], [(COUNT, 0)], want=POS | COLS | AGG) for t in su.tables]
        for r, res in enumerate(results):
            shards[r].gather(res)
            shards[r].fence()
        with pytest.raises(mbcol.MbcError) as e:
            shards[0].collect()
        assert e.value.status == N.ERR_UNSUPPORTED and "did not fit" in e.value.message
        with pytest.raises(mbcol.MbcError) as e:                         # nothing to merge from a step that did not fit
            shards[0].group_aggregate([DESCS[I1]], [COUNT], [N.ATTR_INTEGER])
        assert e.value.status == N.ERR_ARG
        _close(shards, results)
    finally:
        su.close()


# ---- top-k and ORDER BY -----------------------------------------------------------------------------------------------
def _window_fields(key_cols, proj):
    wcols = list(dict.fromkeys(list(key_cols) + list(proj)))
    return wcols, [wcols.index(c) for c in key_cols], [wcols.index(c) for c in proj]


@pytest.mark.parametrize("key_cols", [[K16], [S], [S, I1], [Z]], ids=["k16", "s", "s_i1", "z"])
def test_top_k_matches_one_table(setup, key_cols):
    su = setup
    proj = [I2, R]                                                     # the keys are not projected by the merge
    wcols, kf, pf = _window_fields(key_cols, proj)
    wdescs = [DESCS[c] for c in wcols]
    shards = su.shards()
    shards[0].create_window(NRANK * su.world, wdescs)
    _attach(shards)
    terms = _terms("some")
    live = ~su.deleted & (su.cols[I1] < 600_000) & (su.cols[F] == 0)
    q_rank = [int(live[r * NRANK:(r + 1) * NRANK].sum()) for r in range(su.world)]
    q = sum(q_rank)
    mid = (max(q_rank) + q) // 2 if su.world > 1 else q - 7
    step = 0
    for desc in (False, True):
        for k in (0, 1, 100, mid, q + 5):
            results = [t.top_k(terms, key_cols, k, desc, proj=wcols, want=POS | COLS) for t in su.tables]
            total, _ = _gather(shards, su.ctxs, results, step)
            assert total == sum(min(k, x) for x in q_rank)
            got = shards[0].top_k(wdescs, kf, k, desc, pf, want=POS | COLS | TUP | HOST)
            shards[0].release()
            exp = su.ref.top_k(terms, key_cols, k, desc, proj=proj, want=POS | COLS | TUP | HOST)
            assert got.count == exp.count == min(k, q)
            np.testing.assert_array_equal(got.positions(), exp.positions())
            for i in range(len(proj)):
                _same(got.column(i), exp.column(i))
            np.testing.assert_array_equal(got.tuples(), exp.tuples())
            if key_cols == [K16] and 1 < got.count:                    # ties across ranks: ascending global position
                kv = su.cols[K16][got.positions()]
                same = kv[1:] == kv[:-1]
                assert np.all(np.diff(got.positions())[same] > 0)
            for r in results + [got, exp]:
                r.close()
            step += 1
    _close(shards)


@pytest.mark.parametrize("desc", [False, True], ids=["asc", "desc"])
def test_sharded_order_by_equals_sort(setup, desc):
    su = setup
    key_cols, proj = [S, I1], [R, I2, S]
    wcols, kf, pf = _window_fields(key_cols, proj)
    wdescs = [DESCS[c] for c in wcols]
    shards = su.shards()
    shards[0].create_window(NRANK * su.world, wdescs)
    _attach(shards)
    results = [t.sort(key_cols, desc, proj=wcols, want=POS | COLS) for t in su.tables]
    total, _ = _gather(shards, su.ctxs, results, 1)
    got = shards[0].top_k(wdescs, kf, total, desc, pf, want=POS | COLS | TUP | HOST)
    exp = su.ref.sort(key_cols, desc, proj=proj, want=POS | COLS | TUP | HOST)
    assert got.count == exp.count == int((~su.deleted).sum())
    np.testing.assert_array_equal(got.positions(), exp.positions())
    np.testing.assert_array_equal(got.tuples(), exp.tuples())
    shards[0].release()
    _close(shards, results + [got, exp])


# ---- refusals ---------------------------------------------------------------------------------------------------------
def _refused(ctx, status, fn, *args, **kw):
    before = ctx.kernel_launches
    with pytest.raises(mbcol.MbcError) as e:
        fn(*args, **kw)
    assert e.value.status == status, e.value.message
    assert ctx.kernel_launches == before                               # refused on the host, nothing launched


def test_refusals():
    su = Setup(2, deleted=False)
    ctx = su.ctxs[0]
    t = su.tables[0]
    try:
        # a join result: two position lists, nothing a window holds
        small = load_table(ctx, [(1, 4)], [np.arange(1000, dtype=np.int32)])
        join = mbcol.bitmap_join(small, small, [mbcol.Term(N.OP_EQ, ("col", 0), ("icol", 0), 0)], [(1, 0)], POS | COLS)
        assert join.count == 1000
        sh = mbcol.Shard(ctx, 0, 1)
        sh.create_window(4096, [(1, 4)])
        _refused(ctx, N.ERR_ARG, sh.gather, join)
        # a grouped result in a window without its aggregate columns, and a sorted result without positions
        grp = t.group_aggregate([], [K16], [(COUNT, 0)], want=POS | COLS | AGG)
        _refused(ctx, N.ERR_ARG, sh.gather, grp)
        _refused(ctx, N.ERR_ARG, sh.gather, t.top_k([], [I1], 10, proj=[I1], want=COLS))
        # 9 key columns + 8 aggregates do not fit the window's 16 columns
        wide = t.group_aggregate([], [K16] * 9, [(COUNT, 0)] * 8, want=POS | COLS | AGG)
        _refused(ctx, N.ERR_UNSUPPORTED, sh.gather, wide)
        sh.close()

        shards = su.shards()
        shards[0].create_group_window(NRANK * 2, [DESCS[K16]], 2)
        _attach(shards)
        kd, kinds, types = [DESCS[K16]], [COUNT, SUM], [N.ATTR_INTEGER, N.ATTR_INTEGER]
        _refused(ctx, N.ERR_ARG, shards[0].group_aggregate, kd, kinds, types)             # nothing gathered yet
        results = [tb.group_aggregate([], [K16], [(COUNT, 0), (SUM, I2)], want=POS | COLS | AGG) for tb in su.tables]
        for r, res in enumerate(results):
            shards[r].gather(res)
            shards[r].fence()
        _refused(ctx, N.ERR_ARG, shards[0].group_aggregate, kd, kinds, types)             # gathered, not collected
        shards[0].collect()
        _refused(su.ctxs[1], N.ERR_ARG, shards[1].group_aggregate, kd, kinds, types)      # not the window's owner
        _refused(su.ctxs[1], N.ERR_ARG, shards[1].top_k, kd * 3, [0], 5)
        _refused(ctx, N.ERR_ARG, shards[0].group_aggregate, [DESCS[S]], kinds, types)     # stride 16, window 4
        _refused(ctx, N.ERR_ARG, shards[0].group_aggregate, kd, [COUNT], types[:1])       # window has 2 aggregates
        _refused(ctx, N.ERR_UNSUPPORTED, shards[0].group_aggregate, kd * 9, kinds * 4, types * 4)   # 9 + 8 > 16
        _refused(ctx, N.ERR_UNSUPPORTED, shards[0].group_aggregate, kd, kinds, types, want=POS | TUP)
        _refused(ctx, N.ERR_UNSUPPORTED, shards[0].group_aggregate, kd, kinds, types, want=POS | N.WANT_BITMAP)
        got = shards[0].group_aggregate(kd, kinds, types)
        exp = su.ref.group_aggregate([], [K16], [(COUNT, 0), (SUM, I2)])
        _check_groups(got, exp, [K16], [(COUNT, 0), (SUM, I2)])
        shards[0].release()
        _refused(ctx, N.ERR_ARG, shards[0].group_aggregate, kd, kinds, types)             # released
        _close(shards, results + [got, exp])

        shards = su.shards()
        shards[0].create_window(4096, [DESCS[I1]])
        _attach(shards)
        results = [tb.top_k([], [I1], 100, proj=[I1], want=POS | COLS) for tb in su.tables]
        _gather(shards, su.ctxs, results, 0)
        d = [DESCS[I1]]
        _refused(ctx, N.ERR_ARG, shards[0].top_k, d, [0], -1)
        _refused(ctx, N.ERR_ARG, shards[0].top_k, d, [1], 5)
        _refused(ctx, N.ERR_ARG, shards[0].top_k, d, [0], 5, proj_fields=[1])
        _refused(ctx, N.ERR_ARG, shards[0].top_k, [DESCS[S]], [0], 5)
        _refused(ctx, N.ERR_UNSUPPORTED, shards[0].top_k, d, [0], 5, want=POS | AGG)
        _refused(ctx, N.ERR_UNSUPPORTED, shards[0].top_k, d, [0], 5, want=POS | N.WANT_BITMAP)
        empty = shards[0].top_k(d, [0], 0, proj_fields=[0])
        assert empty.count == 0 and empty.positions().size == 0
        top = shards[0].top_k(d, [0], 100, proj_fields=[0], want=POS | COLS | HOST)
        exp = su.ref.top_k([], [I1], 100, proj=[I1])
        np.testing.assert_array_equal(top.positions(), exp.positions())
        shards[0].release()
        _close(shards, results + [empty, top, exp, grp, wide, join])
        small.close()
    finally:
        su.close()
