"""mbc_topk (Table.top_k) on a B200: ORDER BY ... LIMIT k over a filtered table.

The expected positions are the first min(k, Q) entries of oracle.sort's order restricted to oracle.scan's qualifying
positions; projected columns are compared bit for bit with the table's rows at those positions (so -0.0 and +0.0 are told
apart) and Tuple bytes with the oracle scan's.  Small k goes through the radix select (csrc/mbc_topk.cu), k above
MBC_TOPK_SORT_FRACTION of Q through the filtered sort; both must give mbc_sort's order, ties by ascending position in
both directions."""
import itertools
import os
import re

import numpy as np
import pytest

import mbcol
from mbcol import _native as N
from util import load_table

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS = N.WANT_POSITIONS | N.WANT_HOST
PC = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST
ALL = PC | N.WANT_TUPLES
I32_MIN, I32_MAX = -2**31, 2**31 - 1
INT, REAL = (N.ATTR_INTEGER, 4), (N.ATTR_REAL, 4)
F32 = np.finfo(np.float32)


def _sort_fraction():
    src = open(os.path.join(ROOT, "minibase-columnar-database_b200", "csrc", "mbc_topk.cu")).read()
    return float(re.search(r"#define MBC_TOPK_SORT_FRACTION\s+([0-9.eE+-]+)", src).group(1))


def _str(width):
    return (N.ATTR_STRING, width)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype.itemsize == 4 else a


def _full_range(rng, n):
    return rng.integers(I32_MIN, I32_MAX + 1, n, dtype=np.int64).astype(np.int32)


def _words(rng, count, width):
    alphabet = list("abcxyzAZ09-_~")
    out = []
    for i in range(count):
        s = "".join(rng.choice(alphabet, int(rng.integers(0, width + 1))))
        out.append(s[:width - 2] + "é" if i % 10 == 0 else s)
    return out


def _strings(oracle, rng, words, width, n):
    return oracle.pack_strings(words, width)[rng.integers(0, len(words), n)]


def _expected(oracle, descs, cols, terms, keys, desc, deleted=()):
    """mbc_sort's order over the qualifying rows (all of them: callers slice the first k)."""
    order = oracle.sort(descs, cols, keys, descending=desc, deleted_positions=deleted)
    if terms:
        qual = oracle.scan(descs, cols, terms, want_tuples=False)["positions"]
        order = order[np.isin(order, qual)]
    return order


def _check(res, exp, cols, proj, base=0):
    assert res.count == exp.size
    np.testing.assert_array_equal(res.positions(), exp + base)
    for i, c in enumerate(proj):
        np.testing.assert_array_equal(_bits(res.column(i)), _bits(cols[c][exp]), err_msg=f"projected column {c}")


def _ks(q):
    return sorted({k for k in (0, 1, 7, 100, 4096, q - 1, q, q + 1, 2**62) if k >= 0})


# ---- a. sizes, selectivities, k, key types ------------------------------------------------------------------------

DESCS = [INT, REAL, _str(16), _str(5), INT]                     # column 4 draws the selectivity
KEY_SETS = [[0], [1], [2], [3], [2, 0], [1, 3, 0]]


def _table_cols(oracle, rng, n):
    ints = rng.integers(-50, 50, n).astype(np.int32)
    ints[::3] = _full_range(rng, ints[::3].size)
    reals = (rng.standard_normal(n) * 10).astype(np.float32)
    reals[rng.random(n) < 0.2] = np.float32(-0.0)
    reals[rng.random(n) < 0.2] = np.float32(0.0)
    return [ints, reals, _strings(oracle, rng, _words(rng, 200, 16), 16, n), _strings(oracle, rng, _words(rng, 40, 5), 5, n),
            rng.integers(0, 100, n).astype(np.int32)]


@pytest.mark.parametrize("n", [1, 4095, 4096, 8193, 1_000_003])
@pytest.mark.parametrize("sel", [0, 1, 50, 100])
def test_sizes_selectivities_and_k(ctx, oracle, n, sel):
    """Every k of {0, 1, 7, 100, 4096, Q-1, Q, Q+1, 2^62}, both directions, every key type alone and in 2- and 3-key
    tuples, against the oracle; at 100 % (no terms) and k >= Q the result equals mbc_sort's bit for bit."""
    rng = np.random.default_rng(n * 101 + sel)
    cols = _table_cols(oracle, rng, n)
    t = load_table(ctx, DESCS, cols)
    terms = [] if sel == 100 else [oracle.Term(oracle.OP_LT, ("col", 4), ("int", sel), 0)]
    proj = [2, 0, 1, 3]
    for keys, desc in itertools.product(KEY_SETS, (False, True)):
        order = _expected(oracle, DESCS, cols, terms, keys, desc)
        q = order.size
        for k in _ks(q):
            res = t.top_k(terms, keys, k, descending=desc, proj=proj, want=PC)
            _check(res, order[:k], cols, proj)
            res.close()
        if not terms:
            full = t.sort(keys, descending=desc, proj=proj, want=ALL)
            top = t.top_k([], keys, q, descending=desc, proj=proj, want=ALL)
            np.testing.assert_array_equal(top.positions(), full.positions())
            np.testing.assert_array_equal(top.tuples(), full.tuples())
            for i in range(len(proj)):
                np.testing.assert_array_equal(_bits(top.column(i)), _bits(full.column(i)))
            top.close()
            full.close()
    t.close()


# ---- b. ties at the cut -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("desc", [False, True])
def test_ties_at_the_cut(ctx, oracle, desc):
    """A 4-valued key whose runs the cut ends inside: the boundary key's lowest positions win; an all-equal key (the
    select reaches the row-id word); buckets holding exactly the rows still needed."""
    n = 300_017
    rng = np.random.default_rng(3)
    four = np.array([-7, 0, 5, 1 << 20], np.int32)[rng.choice(4, n, p=[0.05, 0.1, 0.35, 0.5])]
    exact = np.repeat(np.arange(6, dtype=np.int32), [10, 20, 256, 4096, 1, n - 4383])
    rng.shuffle(exact)
    descs = [INT, INT, INT, INT]
    cols = [four, np.full(n, 42, np.int32), 5 - exact if desc else exact, np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    for key, ks in (([0], [1, 1000, 20_000, 60_000]),
                    ([1], [1, 99, 4096, 60_000]),
                    ([2], [10, 30, 286, 4382, 4383, 4384])):      # buckets of exactly the rows still needed
        order = _expected(oracle, descs, cols, [], key, desc)
        for k in ks:
            res = t.top_k([], key, k, descending=desc, proj=[key[0], 3], want=PC)
            _check(res, order[:k], cols, [key[0], 3])
            if key == [1]:
                np.testing.assert_array_equal(res.positions(), np.arange(k))
            if key == [0]:                            # the boundary key's rows are the lowest positions holding it
                v = cols[0][order[k - 1]]
                got = res.positions()[res.column(0) == v]
                assert np.array_equal(got, np.nonzero(cols[0] == v)[0][:got.size])
            res.close()
    t.close()


# ---- c. digit edges -----------------------------------------------------------------------------------------------

DIGIT_KEYS = {
    "full range": lambda x, rng: np.concatenate([[I32_MIN, I32_MAX, -1, 0] * 3, _full_range(rng, x.size - 12)]).astype(np.int32),
    "byte 0": lambda x, rng: (0x12345600 + x).astype(np.int32),
    "byte 1": lambda x, rng: (5 + 256 * x).astype(np.int32),
    "byte 2": lambda x, rng: (9 + (x << 16)).astype(np.int32),
    "byte 3": lambda x, rng: ((x << 24) + I32_MIN).astype(np.int32),
}


@pytest.mark.parametrize("name", list(DIGIT_KEYS))
@pytest.mark.parametrize("desc", [False, True])
def test_int_digit_edges(ctx, oracle, name, desc):
    n = 100_003
    rng = np.random.default_rng(11)
    descs = [INT, INT]
    cols = [DIGIT_KEYS[name](rng.integers(0, 256, n), rng), np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    order = _expected(oracle, descs, cols, [], [0], desc)
    for k in (1, 13, 100, 390, 1000, 9999):
        res = t.top_k([], [0], k, descending=desc, proj=[0, 1], want=PC)
        _check(res, order[:k], cols, [0, 1])
        res.close()
    t.close()


PREFIX = ("common-prefix-" * 5)[:60]


def _string_vocab():
    tails = ["".join(p) for k in range(1, 5) for p in itertools.product("a~b", repeat=k)]
    tails += ["é", "aé", "é~", "€", "中", "ÿÿ", "Ā", "ߦ"]
    w64 = [PREFIX + s for s in tails] + [PREFIX[:k] for k in (1, 30, 59, 60)] + ["a" * k for k in range(1, 65)]
    w64 += ["", "é", "ü", "€", "中文", "日本語", "￿", "Z", "z", "~"]
    w5 = ["", "a", "ab", "abcd", "abcde", "abcdd", "b", "é", "éé", "a€", "a€b", "中", "中a", "zzzz", "zzzzz", "￿"]
    return w64, w5


@pytest.mark.parametrize("keys", [[0], [1], [1, 0]], ids=["char64", "char5", "char5-char64"])
@pytest.mark.parametrize("desc", [False, True])
def test_string_digit_edges(ctx, oracle, keys, desc):
    """char(64) keys sharing a 60-byte prefix, keys that differ only in length, UTF-8 bytes >= 0x80, char(5) in an
    8-byte stride."""
    n = 120_001
    rng = np.random.default_rng(13)
    w64, w5 = _string_vocab()
    w64p = [w for w in w64 if w.startswith(PREFIX)]
    c64 = _strings(oracle, rng, w64, 64, n)
    c64[: n // 2] = _strings(oracle, rng, w64p, 64, n // 2)          # half the rows share the 60-byte prefix
    descs = [_str(64), _str(5), INT]
    cols = [c64, _strings(oracle, rng, w5, 5, n), np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    order = _expected(oracle, descs, cols, [], keys, desc)
    for k in (1, 50, 2000, 30_000):
        res = t.top_k([], keys, k, descending=desc, proj=[2, 0, 1], want=PC)
        _check(res, order[:k], cols, [2, 0, 1])
        res.close()
    t.close()


EDGE_REALS = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.17e-38, -1.17e-38, F32.tiny, -F32.tiny, F32.max, -F32.max,
                       1.0, -1.0, 0.1, -0.1], dtype=np.float32)


@pytest.mark.parametrize("desc", [False, True])
def test_real_digit_edges(ctx, oracle, desc):
    """Interleaved +-0.0 are one key (ties by position, each row keeping its own sign), +-inf, subnormals, +-FLT_MAX."""
    n = 50_021
    rng = np.random.default_rng(17)
    pick = rng.random(n)
    zeros = np.where(rng.random(n) < 0.5, np.float32(0.0), np.float32(-0.0))
    reals = np.where(pick < 0.4, zeros, np.where(pick < 0.7, EDGE_REALS[rng.integers(0, EDGE_REALS.size, n)],
                                                 rng.standard_normal(n) * 1e3)).astype(np.float32)
    descs = [REAL, INT]
    cols = [reals, np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    order = _expected(oracle, descs, cols, [], [0], desc)
    nz = int((order.size - (reals == 0).sum()) // 2)                    # a cut inside the run of zeros
    for k in (1, 17, 500, nz + 1000):
        res = t.top_k([], [0], k, descending=desc, proj=[0, 1], want=PC)
        _check(res, order[:k], cols, [0, 1])
        res.close()
    t.close()


# ---- d. deleted rows and a position base past 2^32 ----------------------------------------------------------------

@pytest.mark.parametrize("desc", [False, True])
def test_deleted_rows_and_position_base(ctx, oracle, desc):
    """The rows with the first keys are deleted (they would otherwise be the top k); positions start past 2^32."""
    n, base = 200_003, 3 * 2**31 + 7
    rng = np.random.default_rng(29)
    descs = [INT, _str(16), INT]
    cols = [rng.integers(-50, 50, n).astype(np.int32), _strings(oracle, rng, _words(rng, 300, 16), 16, n), _full_range(rng, n)]
    t = load_table(ctx, descs, cols, base)
    first = _expected(oracle, descs, cols, [], [2], desc)
    dele = np.unique(np.concatenate([first[:500:2], [0, n - 1], rng.choice(n, n // 10, replace=False)]))
    t.set_deleted(oracle.bits_from_positions(dele, n))
    terms = [oracle.Term(oracle.OP_GT, ("col", 0), ("int", -40), 0)]
    for keys in ([2], [0, 1]):
        order = _expected(oracle, descs, cols, terms, keys, desc, deleted=dele)
        for k in (1, 300, 5000):
            res = t.top_k(terms, keys, k, descending=desc, proj=[2, 1, 0], want=PC)
            _check(res, order[:k], cols, [2, 1, 0], base)
            res.close()
    t.close()


# ---- e. what is asked for -----------------------------------------------------------------------------------------

def test_each_part_of_the_result_alone(ctx, oracle):
    """Positions, columns and Tuple bytes asked for alone equal the parts of the full result; the Tuple bytes are the
    oracle scan's; a device-resident result (no MBC_WANT_HOST) read through mbc_result_device / column_device agrees."""
    import torch
    from bench import _CudaArray
    n = 100_003
    rng = np.random.default_rng(37)
    descs = [INT, _str(16), REAL]
    cols = [rng.integers(-30, 30, n).astype(np.int32), _strings(oracle, rng, _words(rng, 500, 16), 16, n),
            (rng.standard_normal(n) * 5).astype(np.float32)]
    t = load_table(ctx, descs, cols)
    keys, proj, terms = [1, 0], [2, 0, 1], [oracle.Term(oracle.OP_GE, ("col", 0), ("int", -10), 0)]
    scan = oracle.scan(descs, cols, [], proj=proj, want_positions=False, nthreads=oracle.max_threads())
    order = _expected(oracle, descs, cols, terms, keys, False)
    for k in (1000, order.size):                                      # the select and the filtered sort
        exp = order[:k]
        full = t.top_k(terms, keys, k, proj=proj, want=ALL)
        _check(full, exp, cols, proj)
        np.testing.assert_array_equal(full.tuples(), scan["tuples"][exp])
        r = t.top_k(terms, keys, k, proj=proj, want=POS)
        np.testing.assert_array_equal(r.positions(), exp)
        r.close()
        r = t.top_k(terms, keys, k, proj=proj, want=N.WANT_COLUMNS | N.WANT_HOST)
        assert r.count == k
        for i in range(len(proj)):
            np.testing.assert_array_equal(_bits(r.column(i)), _bits(full.column(i)))
        r.close()
        r = t.top_k(terms, keys, k, proj=proj, want=N.WANT_TUPLES | N.WANT_HOST)
        np.testing.assert_array_equal(r.tuples(), full.tuples())
        r.close()
        r = t.top_k(terms, keys, k, proj=[], want=ALL)
        assert r.tuples().size == 0
        np.testing.assert_array_equal(r.positions(), exp)
        r.close()
        r = t.top_k(terms, keys, k, proj=proj, want=N.WANT_POSITIONS | N.WANT_COLUMNS)
        assert r.count == k
        pos = torch.as_tensor(_CudaArray(r.device_pointers()["positions"], k * 8), device="cuda:0").view(torch.int64).cpu().numpy()
        np.testing.assert_array_equal(pos, exp)
        p, s = r.column_device(0)
        assert s == 4
        got = torch.as_tensor(_CudaArray(p, k * s), device="cuda:0").view(torch.int32).cpu().numpy()
        np.testing.assert_array_equal(got, cols[2][exp].view(np.int32))
        p, s = r.column_device(2)
        got = torch.as_tensor(_CudaArray(p, k * s), device="cuda:0").cpu().numpy().reshape(-1, s)
        np.testing.assert_array_equal(got[:, :16], cols[1][exp])
        r.close()
        full.close()
    t.close()


# ---- f. both sides of the select / sort threshold -----------------------------------------------------------------

@pytest.mark.parametrize("desc", [False, True])
def test_both_sides_of_the_sort_threshold(ctx, oracle, desc):
    """k at and just above MBC_TOPK_SORT_FRACTION * Q (select, then filtered sort) and well on either side; the two paths
    launch different kernels (the select's histogram passes), and both give mbc_sort's order."""
    frac = _sort_fraction()
    assert 0.0 < frac < 1.0
    n = 400_009
    rng = np.random.default_rng(53)
    descs = [INT, _str(16), INT]
    cols = [rng.integers(-1000, 1000, n).astype(np.int32), _strings(oracle, rng, _words(rng, 1000, 16), 16, n),
            rng.integers(0, 10, n).astype(np.int32)]
    t = load_table(ctx, descs, cols)
    terms = [oracle.Term(oracle.OP_LT, ("col", 2), ("int", 7), 0)]
    order = _expected(oracle, descs, cols, terms, [0, 1], desc)
    q = order.size
    edge = int(np.floor(frac * q))
    launches = {}
    for k in (max(edge // 10, 1), edge, edge + 1, min(2 * edge + 1, q)):
        before = ctx.kernel_launches
        res = t.top_k(terms, [0, 1], k, descending=desc, proj=[0, 1], want=PC)
        launches[k] = ctx.kernel_launches - before
        _check(res, order[:k], cols, [0, 1])
        res.close()
    assert launches[edge] != launches[edge + 1], launches
    t.close()


# ---- g. scale -----------------------------------------------------------------------------------------------------

def test_scale_full_range_int_keys(ctx):
    """10^8 + 7 full-range int keys, k = 1 000 and 10^6, both directions, against numpy's argpartition: the returned
    keys are the k extreme ones in order, and among rows equal to the boundary key the lowest positions were taken."""
    n = 10**8 + 7
    keys = np.random.default_rng(61).integers(I32_MIN, I32_MAX + 1, n, dtype=np.int64).astype(np.int32)
    t = ctx.create_table([INT], n)
    t.load_column(0, keys)
    for desc, k in itertools.product((False, True), (1000, 10**6)):
        res = t.top_k([], [0], k, descending=desc, proj=[0], want=PC)
        assert res.count == k
        pos, got = res.positions(), res.column(0)
        np.testing.assert_array_equal(keys[pos], got)
        s = -keys.astype(np.int64) if desc else keys.astype(np.int64)
        part = np.sort(s[np.argpartition(s, k - 1)[:k]])
        np.testing.assert_array_equal(-got.astype(np.int64) if desc else got, part)
        tie = got[1:] == got[:-1]
        assert (pos[1:][tie] > pos[:-1][tie]).all()
        boundary = got[-1]
        taken = np.sort(pos[got == boundary])
        np.testing.assert_array_equal(taken, np.nonzero(keys == boundary)[0][:taken.size])
        res.close()
    t.close()


# ---- h. determinism -----------------------------------------------------------------------------------------------

def test_repeats_are_bit_identical(ctx, oracle):
    """Ten top-k calls on a 4 M-row tie-heavy key return the same positions and bytes (the candidate compaction's order
    varies from run to run; the result must not)."""
    n = 4_000_037
    rng = np.random.default_rng(43)
    descs = [INT, _str(16)]
    cols = [rng.integers(0, 8, n).astype(np.int32), _strings(oracle, rng, _words(rng, 50, 16), 16, n)]
    t = load_table(ctx, descs, cols)
    first = t.top_k([], [0, 1], 100_000, proj=[1, 0], want=ALL)
    pos, tup = first.positions().copy(), first.tuples().copy()
    first.close()
    np.testing.assert_array_equal(pos, _expected(oracle, descs, cols, [], [0, 1], False)[:100_000])
    for _ in range(9):
        r = t.top_k([], [0, 1], 100_000, proj=[1, 0], want=ALL)
        assert np.array_equal(r.positions(), pos) and np.array_equal(r.tuples(), tup)
        r.close()
    t.close()


# ---- i. errors ----------------------------------------------------------------------------------------------------

def test_argument_errors(ctx, oracle):
    """k < 0, a bad key or projected column and 17 keys fail as mbc_sort does; MBC_WANT_AGG / MBC_WANT_BITMAP are
    unsupported; malformed terms fail as mbc_scan does."""
    t = load_table(ctx, [INT, _str(8)], [np.arange(10, dtype=np.int32), oracle.pack_strings(["a"] * 10, 8)])
    bad = [dict(keys=[0], k=-1, status=N.ERR_ARG), dict(keys=[2], status=N.ERR_ARG), dict(keys=[-1], status=N.ERR_ARG),
           dict(keys=[], status=N.ERR_ARG), dict(keys=[0], proj=[5], status=N.ERR_ARG), dict(keys=[0] * 17, status=N.ERR_UNSUPPORTED),
           dict(keys=[0], want=PC | N.WANT_AGG, status=N.ERR_UNSUPPORTED),
           dict(keys=[0], want=PC | N.WANT_BITMAP, status=N.ERR_UNSUPPORTED)]
    for b in bad:
        with pytest.raises(mbcol.MbcError) as e:
            t.top_k([], b["keys"], b.get("k", 3), proj=b.get("proj", [0]), want=b.get("want", PC))
        assert e.value.status == b["status"], b
        assert e.value.message
        if b.get("k", 3) >= 0 and "want" not in b:
            with pytest.raises(mbcol.MbcError) as s:
                t.sort(b["keys"], proj=b.get("proj", [0]), want=PC)
            assert s.value.status == b["status"], b
    terms = [[mbcol.Term(N.OP_EQ, ("col", 7), ("int", 1), 0)], [mbcol.Term(N.OP_EQ, ("col", 0), ("str", "x"), 0)],
             [mbcol.Term(N.OP_EQ, ("col", 1), ("int", 1), 0)], [mbcol.Term(11, ("col", 0), ("int", 1), 0)],
             [mbcol.Term(N.OP_EQ, ("col", 0), ("int", i), i) for i in range(17)]]
    for tm in terms:
        with pytest.raises(mbcol.MbcError) as s:
            t.scan(tm, want=POS)
        with pytest.raises(mbcol.MbcError) as e:
            t.top_k(tm, [0], 3, want=POS)
        assert e.value.status == s.value.status
    r = t.top_k([], [0], 0, proj=[0, 1], want=ALL)
    assert r.count == 0 and r.positions().size == 0 and r.tuples().size == 0
    r.close()
    t.close()


# ---- j. the ColumnarFileScan mirror -------------------------------------------------------------------------------

def test_columnarfilescan_top_k_mirror(tmp_path, oracle, minidata):
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
        proj = [FldSpec(RelSpec(RelSpec.outer), c + 1) for c in range(len(descs))]
        int_col = next(c for c, d in enumerate(descs) if d[0] == N.ATTR_INTEGER)
        str_col = next(c for c, d in enumerate(descs) if d[0] == N.ATTR_STRING)
        filters = [([expr, None], [oracle.Term(oracle.OP_GE, ("col", 2), ("int", 2), 0)]), (None, [])]
        for keys, desc, (filt, terms) in itertools.product([[int_col], [str_col], [str_col, int_col]], (False, True), filters):
            fs = ColumnarFileScan("cf", types, sizes, len(descs), len(descs), proj, filt)
            got = fs.top_k(keys, 25, desc)
            fs.close()
            exp = _expected(oracle, descs, cols, terms, keys, desc)[:25]
            assert len(got) == exp.size == 25
            for (p, row), e in zip(got, exp):
                assert p == int(e)
                want = [bytes(cols[c][e]).split(b"\0", 1)[0].decode() if d[0] == N.ATTR_STRING else
                        (int(cols[c][e]) if d[0] == N.ATTR_INTEGER else float(cols[c][e])) for c, d in enumerate(descs)]
                assert list(row) == want
    finally:
        SystemDefs.shutdown()
