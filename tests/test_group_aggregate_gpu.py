"""mbc_group_aggregate (Table.group_aggregate) on a B200 against numpy over the qualifying rows and the oracle: key types
and their edges, sizes on and beside the 4096-element fold chunk and the 8192-row padding, filters, deleted rows, one
giant group and all-singleton groups, cross-checks with mbc_scan's scalar aggregates, determinism, argument errors and the
ColumnarFileScan mirror.  Integers are exact, dyadic reals bit-equal, other real SUMs within n*2^-53*sum|x|."""
import numpy as np
import pytest

from mbcol import _native as N
from group_oracle import group_aggregate
from util import C2_AGGS, C2_DESCS, SEED, c2_columns, c2_device_table, c2_terms, load_table

pytestmark = pytest.mark.gpu

ALL = N.WANT_COLUMNS | N.WANT_POSITIONS | N.WANT_AGG | N.WANT_HOST
COUNT, SUM, MIN, MAX = N.AGG_COUNT, N.AGG_SUM, N.AGG_MIN, N.AGG_MAX
I32_MIN, I32_MAX = -2**31, 2**31 - 1


def _expect(descs, cols, key_cols, aggs, qual):
    """numpy: groups of the qualifying positions `qual` (ascending) in key order -> (positions, keys, [(i64, f64, kind)])."""
    ranks = []
    for c in key_cols:
        v = cols[c][qual]
        if descs[c][0] == 0:
            v = np.ascontiguousarray(v).view(f"S{v.shape[1]}").ravel()
        elif descs[c][0] == 2:
            v = v + np.float32(0.0)                                      # -0.0 and +0.0 are one key
        ranks.append(np.unique(v, return_inverse=True)[1].ravel())
    order = np.lexsort(ranks[::-1]) if qual.size else np.empty(0, np.int64)
    heads = np.ones(qual.size, bool)
    if qual.size:
        heads[1:] = np.any(np.stack([r[order][1:] != r[order][:-1] for r in ranks]), axis=0)
    st = np.nonzero(heads)[0]
    first = qual[order][st]
    out = []
    for kind, col in aggs:
        if kind == COUNT:
            cnt = np.diff(np.append(st, qual.size)).astype(np.int64)
            out.append((cnt, cnt.astype(np.float64), None))
            continue
        x = cols[col][qual][order]
        if st.size == 0:
            out.append((np.empty(0, np.int64), np.empty(0), None))
            continue
        if descs[col][0] == 1:
            x = x.astype(np.int64)
            r = (np.add if kind == SUM else np.minimum if kind == MIN else np.maximum).reduceat(x, st)
            out.append((r, r.astype(np.float64), None))
        elif kind == SUM:
            exact = np.add.reduceat(x.astype(np.longdouble), st)
            bound = np.diff(np.append(st, x.size)) * 2.0**-53 * np.add.reduceat(np.abs(x.astype(np.float64)), st)
            out.append((None, exact.astype(np.float64), bound))
        else:
            r = (np.minimum if kind == MIN else np.maximum).reduceat(x.astype(np.float64), st)
            out.append((None, r, None))
    return first, [cols[c][first] for c in key_cols], out


def _check(res, exp, dyadic=False):
    first, keys, aggs = exp
    assert res.count == first.size
    np.testing.assert_array_equal(res.positions(), first)
    for k, kv in enumerate(keys):
        got = res.column(k)
        if got.dtype == np.float32:                          # the key of the group's lowest-position row, sign of zero included
            np.testing.assert_array_equal(got.view(np.uint32), kv.view(np.uint32))
        else:
            np.testing.assert_array_equal(got, kv)
    for a, (ei, ef, bound) in enumerate(aggs):
        gi, gf = res.group_agg(a)
        if ei is not None:
            np.testing.assert_array_equal(gi, ei)
            np.testing.assert_array_equal(gf, ef)
        elif bound is None or dyadic:
            assert np.all((gf == ef) | (np.isnan(gf) & np.isnan(ef))), a
        else:
            assert np.all(np.abs(gf - ef) <= np.maximum(bound, 1e-300)), a


def _run(ctx, descs, cols, key_cols, aggs, terms=(), qual=None, dyadic=False):
    t = load_table(ctx, descs, cols)
    res = t.group_aggregate(list(terms), key_cols, aggs)
    n = len(cols[0])
    _check(res, _expect(descs, cols, key_cols, aggs, np.arange(n) if qual is None else qual), dyadic)
    return t, res


def _int_table(rng, n, domain):
    keys = rng.integers(0, domain, n).astype(np.int32) if domain else np.zeros(n, np.int32)
    vals = rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32)
    reals = (rng.integers(-4096, 4096, n) / 8.0).astype(np.float32)         # dyadic: every sum order is exact
    return [(1, 4), (1, 4), (2, 4)], [keys, vals, reals]


AGGS8 = [(COUNT, 0), (SUM, 1), (SUM, 2), (MIN, 1), (MAX, 1), (MIN, 2), (MAX, 2), (SUM, 0)]


@pytest.mark.parametrize("n,domain", [(0, 1), (1, 1), (4095, 2), (4096, 1), (4097, 2), (8191, 1000), (8192, 1), (8193, 2),
                                      (12_289, 1000), (1_000_003, 1 << 20), (3 * 4096 + 1, 3), (16_777_217, 1000)])
def test_int_keys(ctx, n, domain):
    descs, cols = _int_table(np.random.default_rng(n), n, domain)
    _run(ctx, descs, cols, [0], AGGS8, dyadic=True)


def test_all_unique_full_range_keys(ctx):
    n = 4_000_037
    rng = np.random.default_rng(5)
    k = np.arange(n, dtype=np.int64) * ((2**32 - 1) // (n - 1)) + I32_MIN
    k[-1] = I32_MAX
    descs, cols = _int_table(rng, n, 1)
    cols[0] = rng.permutation(k).astype(np.int32)
    _, res = _run(ctx, descs, cols, [0], AGGS8, dyadic=True)
    assert res.count == n and res.column(0)[0] == I32_MIN and res.column(0)[-1] == I32_MAX


def _strings(rng, n, width, words):
    out = np.zeros((n, width), np.uint8)
    idx = rng.integers(0, len(words), n)
    for i, w in enumerate(words):
        out[idx == i, :len(w)] = np.frombuffer(w, np.uint8)
    return out


def test_char_keys(ctx):
    rng = np.random.default_rng(11)
    n = 300_001
    prefix = bytes(range(65, 65 + 60))
    descs = [(0, 16), (0, 5), (0, 64), (1, 4), (2, 4)]
    cols = [_strings(rng, n, 16, [b"", b"a", b"ab", b"abc", b"b", b"\xc3\xa9t\xc3\xa9", b"zzzzzzzzzzzzzzzz"]),
            _strings(rng, n, 5, [b"x", b"xy", b"xyz", b"xyzw", b"xyzwv", b"y"]),
            _strings(rng, n, 64, [prefix, prefix + b"a", prefix + b"ab", prefix + b"b", prefix[:59] + b"\xff", prefix + b"\x01\x02\x03\x04"]),
            rng.integers(-1000, 1000, n).astype(np.int32), rng.standard_normal(n).astype(np.float32)]
    aggs = [(COUNT, 0), (SUM, 3), (SUM, 4), (MIN, 3), (MAX, 4)]
    for keys in ([0], [1], [2], [2, 1, 0]):
        _run(ctx, descs, cols, keys, aggs)


def test_real_key_edges(ctx):
    rng = np.random.default_rng(12)
    n = 200_003
    edges = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.1754942e-38, 3.4028235e38, -3.4028235e38, 1.5, -1.5],
                     dtype=np.float32)
    key = edges[rng.integers(0, edges.size, n)]
    key[0], key[1], key[2] = -0.0, 0.0, -0.0                               # the zero group's lowest-position row is -0.0
    vals = rng.integers(-10**6, 10**6, n).astype(np.int32)
    descs, cols = [(2, 4), (1, 4), (2, 4)], [key, vals, (vals / 4.0).astype(np.float32)]
    _, res = _run(ctx, descs, cols, [0], [(COUNT, 0), (SUM, 1), (SUM, 2), (MIN, 2), (MAX, 1)], dyadic=True)
    assert res.count == 10                                                 # 11 edges, the two zeros one key
    z = int(np.nonzero(res.column(0) == 0.0)[0][0])
    assert res.positions()[z] == 0 and np.signbit(res.column(0)[z])
    _run(ctx, [(1, 4)] + descs, [rng.integers(0, 3, n).astype(np.int32)] + cols, [0, 1], [(COUNT, 0), (SUM, 2)])


def test_three_mixed_keys(ctx):
    rng = np.random.default_rng(13)
    n = 2_000_000
    descs = [(1, 4), (0, 5), (2, 4), (1, 4), (2, 4)]
    cols = [rng.integers(-3, 4, n).astype(np.int32), _strings(rng, n, 5, [b"", b"a", b"ab", b"abcde", b"b"]),
            np.array([0.0, -0.0, 2.5, -np.inf], np.float32)[rng.integers(0, 4, n)],
            rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32), rng.random(n).astype(np.float32)]
    _run(ctx, descs, cols, [0, 1, 2], [(COUNT, 0), (SUM, 3), (SUM, 4), (MIN, 3), (MAX, 3), (MIN, 4), (MAX, 4)])


def test_int_sum_past_2_53_within_a_group(ctx):
    n = 2 * (1 << 22) + 2 * 4096 + 7
    key = (np.arange(n) % 2).astype(np.int32)
    vals = np.where(key == 0, I32_MAX, I32_MIN).astype(np.int32)
    _, res = _run(ctx, [(1, 4), (1, 4)], [key, vals], [0], [(SUM, 1), (COUNT, 0)])
    s = res.group_agg(0)[0]
    assert s[0] > 2**53 and s[1] < -2**53


def test_aggregate_limits_and_argument_errors(ctx):
    descs, cols = _int_table(np.random.default_rng(3), 10_000, 10)
    t = load_table(ctx, descs, cols)
    _run(ctx, descs, cols, [0], AGGS8, dyadic=True)
    bad = [dict(key_cols=[0], aggs=AGGS8 + [(COUNT, 0)], status=N.ERR_UNSUPPORTED),
           dict(key_cols=[3], aggs=[], status=N.ERR_ARG), dict(key_cols=[-1], aggs=[], status=N.ERR_ARG),
           dict(key_cols=[], aggs=[], status=N.ERR_ARG), dict(key_cols=[0], aggs=[(SUM, 7)], status=N.ERR_ARG),
           dict(key_cols=[0], aggs=[(9, 1)], status=N.ERR_ARG),
           dict(key_cols=[0], aggs=[], want=ALL | N.WANT_TUPLES, status=N.ERR_UNSUPPORTED),
           dict(key_cols=[0], aggs=[], want=ALL | N.WANT_BITMAP, status=N.ERR_UNSUPPORTED)]
    for b in bad:
        with pytest.raises(N.MbcError) as e:
            t.group_aggregate([], b["key_cols"], b["aggs"], want=b.get("want", ALL))
        assert e.value.status == b["status"], b
    g = t.group_aggregate([], [0], [(COUNT, 0)])
    s = t.scan([], want=N.WANT_AGG, aggs=[(COUNT, 0)])
    with pytest.raises(N.MbcError) as e:
        g.agg(0)
    assert e.value.status == N.ERR_ARG
    with pytest.raises(N.MbcError) as e:
        s.group_agg(0)
    assert e.value.status == N.ERR_ARG
    with pytest.raises(N.MbcError):
        g.group_agg(1)
    assert int(g.group_agg(0)[0].sum()) == s.agg(0)[0] == 10_000


@pytest.mark.parametrize("sel", [None, 0.01, 0.10, 0.50, 0.0])
def test_c2_filters_and_cross_checks(ctx, oracle, sel):
    n = 2_000_003
    cols = c2_columns(oracle, n)
    t = c2_device_table(ctx, n)
    terms = [] if sel is None else c2_terms(oracle, sel) if sel else [oracle.Term(oracle.OP_LT, ("col", 0), ("int", -1), 0)]
    key = [1]
    res = t.group_aggregate(terms, key, C2_AGGS)
    exp = group_aggregate(C2_DESCS, cols, terms, key, C2_AGGS)
    assert res.count == exp["count"]
    np.testing.assert_array_equal(res.positions(), exp["positions"])
    np.testing.assert_array_equal(res.column(0), exp["keys"][0])
    for a, (kind, col) in enumerate(C2_AGGS):
        gi, gf = res.group_agg(a)
        ei, ef = exp["aggs"][a]
        if col == 2 and kind == SUM:
            np.testing.assert_allclose(gf, ef, rtol=1e-6)
        else:
            np.testing.assert_array_equal(gi, ei)
    s = t.scan(terms, want=N.WANT_AGG, aggs=C2_AGGS)
    assert int(res.group_agg(0)[0].sum()) == s.agg(0)[0]                  # sum of COUNT = scan COUNT
    assert int(res.group_agg(1)[0].sum()) == s.agg(1)[0]                  # int SUM folds to the scalar SUM
    if res.count:
        assert int(res.group_agg(3)[0].min()) == s.agg(3)[0] and int(res.group_agg(4)[0].max()) == s.agg(4)[0]
    else:
        assert not s.agg(3)[2]


def test_deleted_rows_position_base_past_2_32(ctx, oracle):
    n, base = 300_007, (1 << 32) + 4096 * 3
    rng = np.random.default_rng(21)
    descs, cols = _int_table(rng, n, 1000)
    t = load_table(ctx, descs, cols, base)
    deleted = np.unique(np.concatenate([rng.choice(n, 20_000, replace=False), [0, 4095, 4096, 8191, n - 1]]))
    t.set_deleted(oracle.bits_from_positions(deleted, n))
    live = np.setdiff1d(np.arange(n), deleted)
    terms = [oracle.Term(oracle.OP_GT, ("col", 1), ("int", -2**30), 0)]
    qual = live[cols[1][live] > -2**30]
    res = t.group_aggregate(terms, [0], AGGS8)
    first, keys, aggs = _expect(descs, cols, [0], AGGS8, qual)
    _check(res, (first + base, keys, aggs), dyadic=True)


def test_skew_one_giant_group(ctx):
    n = (1 << 26) + 5
    rng = np.random.default_rng(31)
    key = np.zeros(n, np.int32)
    single = np.array([0, 4096, 1 << 25, n - 2, n - 1])
    key[single] = [-5, 7, 3, 9, -1]
    vals = rng.integers(-1000, 1000, n).astype(np.int32)
    reals = (vals / 8.0).astype(np.float32)
    aggs = [(COUNT, 0), (SUM, 1), (SUM, 2), (MIN, 1), (MAX, 2)]
    t = load_table(ctx, [(1, 4), (1, 4), (2, 4)], [key, vals, reals])
    res = t.group_aggregate([], [0], aggs)
    assert res.column(0).tolist() == [-5, -1, 0, 3, 7, 9]
    big = np.ones(n, bool)
    big[single] = False
    g = 2
    assert res.positions()[g] == 1
    assert res.group_agg(0)[0][g] == n - 5
    assert res.group_agg(1)[0][g] == int(vals[big].astype(np.int64).sum())
    assert res.group_agg(2)[1][g] == float(vals[big].astype(np.int64).sum()) / 8.0
    assert res.group_agg(3)[0][g] == int(vals[big].min()) and res.group_agg(4)[1][g] == float(reals[big].max())
    for gi, p in zip([0, 1, 3, 4, 5], [0, n - 1, 1 << 25, 4096, n - 2]):
        assert res.positions()[gi] == p and res.group_agg(1)[0][gi] == vals[p]


def test_deterministic_real_sums(ctx, oracle):
    """16 groups of ~250 K rows: every group straddles many 4096-element chunks, so the chunk partials and their fold
    decide the association of the real SUM."""
    n = 4_000_000
    descs = [(1, 4), (2, 4)]
    cols = [np.random.default_rng(41).integers(0, 16, n).astype(np.int32), oracle.synth_real(SEED, 2, n)]
    t = load_table(ctx, descs, cols)
    runs = []
    for _ in range(10):
        r = t.group_aggregate([], [0], [(SUM, 1), (COUNT, 0)], want=N.WANT_AGG | N.WANT_HOST)
        runs.append(r.group_agg(0)[1].view(np.uint64).copy())
        r.close()
    assert runs[0].size == 16 and all(np.array_equal(runs[0], x) for x in runs[1:])
    _check(t.group_aggregate([], [0], [(SUM, 1), (MIN, 1), (MAX, 1)]), _expect(descs, cols, [0], [(SUM, 1), (MIN, 1), (MAX, 1)], np.arange(n)))


def test_columnarfilescan_group_aggregate_mirror(tmp_path, oracle, minidata):
    from mbcol.global_ import AttrOperator, AttrType, SystemDefs
    from mbcol.iterator import ColumnarFileScan, CondExpr, FldSpec, RelSpec
    names, descs, cols = minidata
    w = oracle.DBWriter()
    oracle.write_columnar_file(w, "cf", names, descs, cols)
    path = str(tmp_path / "db")
    with open(path, "wb") as f:
        f.write(w.tobytes())
    SystemDefs.shutdown()
    SystemDefs(path, 0, 100, None)
    try:
        from mbcol.columnar import Columnarfile
        cf = Columnarfile("cf")
        types, sizes = cf.getAttributeTypes(), cf.getStringSizes()
        expr = CondExpr()
        expr.op = AttrOperator(AttrOperator.aopGE)
        expr.type1, expr.type2 = AttrType(AttrType.attrSymbol), AttrType(AttrType.attrInteger)
        expr.operand1.symbol = FldSpec(RelSpec(RelSpec.outer), 3)
        expr.operand2.integer = 2
        specs = [(COUNT, 0), (SUM, 3), (MIN, 3), (MAX, 2)]
        for keys, filt, terms in (([2], [expr, None], [oracle.Term(oracle.OP_GE, ("col", 2), ("int", 2), 0)]),
                                  ([0, 3], None, [])):
            fs = ColumnarFileScan("cf", types, sizes, 4, filt)
            got = fs.group_aggregate(keys, specs)
            fs.close()
            exp = group_aggregate(descs, cols, terms, keys, specs)
            assert len(got) == exp["count"] > 1
            for g, row in enumerate(got):
                kv = [bytes(exp["keys"][k][g]).split(b"\0", 1)[0].decode() if descs[c][0] == 0 else int(exp["keys"][k][g])
                      for k, c in enumerate(keys)]
                assert list(row[:len(keys)]) == kv
                assert list(row[len(keys):]) == [int(exp["aggs"][a][0][g]) for a in range(len(specs))]
    finally:
        SystemDefs.shutdown()
