"""The sparse bitmap-index layout (value-sorted position lists): chosen automatically where per-value bitsets cannot be
built (more than 2^19 distinct values, or D * N/8 bytes beyond the device), and forced with MBC_BM_SPARSE=1.  Every
call returns what the dense layout returns.  Needs a B200."""
import numpy as np
import pytest

import mbcol
from mbcol import _native as N
from mbcol.columnar import Columnarfile
from mbcol.global_ import SystemDefs
import test_bitmap_gpu as dense_suite
from util import load_table

pytestmark = pytest.mark.gpu

ALL = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_TUPLES | N.WANT_AGG | N.WANT_BITMAP | N.WANT_HOST
OPS = {"=": N.OP_EQ, "<": N.OP_LT, ">": N.OP_GT, "!=": N.OP_NE, "<=": N.OP_LE, ">=": N.OP_GE}


@pytest.fixture(autouse=True)
def _automatic_layout(monkeypatch):
    """Each test sets the layout switches it needs: automatic selection unless it forces one (also when the whole
    suite runs under MBC_BM_SPARSE=1)."""
    for v in ("MBC_BM_SPARSE", "MBC_BM_SPARSE_FORM", "MBC_BM_SPARSE_TRACE"):
        monkeypatch.delenv(v, raising=False)


def _mask_of(op, col, lit):
    """numpy `col op lit`; strings compare as zero-padded byte rows (lit padded to the width, not longer)."""
    if col.ndim == 2:
        w = col.shape[1]
        lb = np.zeros(w, np.uint8)
        lb[:len(lit)] = np.frombuffer(lit, np.uint8)
        diff = col != lb
        first = np.where(diff.any(axis=1), diff.argmax(axis=1), w)
        row_b = col[np.arange(col.shape[0]), np.minimum(first, w - 1)].astype(int)
        cmp = np.where(first == w, 0, np.sign(row_b - lb[np.minimum(first, w - 1)].astype(int)))
    else:
        cmp = np.sign(col.astype(np.int64) - lit)
    return {"=": cmp == 0, "<": cmp < 0, ">": cmp > 0, "!=": cmp != 0, "<=": cmp <= 0, ">=": cmp >= 0}[op]


def _check_scan(oracle, t, terms, mask, cols, proj):
    """bitmap scan == numpy mask == mbc_scan on the same terms: positions, projected columns, COUNT/SUM, result bitmap."""
    exp = np.nonzero(mask)[0]
    res = t.bitmap_scan(terms, proj=proj, want=ALL, aggs=[(0, 0), (1, 2)])
    np.testing.assert_array_equal(res.positions(), exp)
    np.testing.assert_array_equal(res.bitmap(), oracle.mask_to_words(mask))
    for i, c in enumerate(proj):
        np.testing.assert_array_equal(res.column(i), cols[c][exp])
    assert res.agg(0)[0] == exp.size and res.agg(1)[0] == int(cols[2][exp].astype(np.int64).sum())
    scan = t.scan(terms, want=N.WANT_POSITIONS | N.WANT_HOST)
    np.testing.assert_array_equal(scan.positions(), exp)
    res.close(); scan.close()
    return exp.size


def _distinct_strings(rng, n, width):
    lens = rng.integers(10, width + 1, n)
    rows = rng.integers(ord("A"), ord("Z") + 1, (n, width)).astype(np.uint8)
    rows[np.arange(width)[None, :] >= lens[:, None]] = 0
    assert np.unique(rows, axis=0).shape[0] == n
    return rows


def test_all_distinct_columns_build_sparse(ctx, oracle):
    """600 000 distinct ints and char(16) strings: more than 2^19 values, which the dense layout refuses."""
    n = 600_000
    rng = np.random.default_rng(600)
    K = (rng.permutation(n) - 250_000).astype(np.int32)
    S = _distinct_strings(rng, n, 16)
    V = rng.integers(-1000, 1000, n).astype(np.int32)
    cols = [K, S, V]
    t = load_table(ctx, [(1, 4), (0, 16), (1, 4)], cols)
    dead = np.unique(rng.integers(0, n, n // 100))
    t.set_deleted(oracle.bits_from_positions(dead, n))
    live = np.ones(n, bool)
    live[dead] = False
    for c in (0, 1):
        t.bitmap_build(c)
        layout, nbytes = t.bitmap_layout(c)
        assert layout == N.BITMAP_SPARSE and 4 * live.sum() <= nbytes < 4 * n + n // 8 + 8192
    assert t.bitmap_layout(2) == (N.BITMAP_NONE, 0)

    # values: the live ones, ascending (byte order for the strings)
    np.testing.assert_array_equal(t.bitmap_values(0), np.unique(K[live]))
    np.testing.assert_array_equal(t.bitmap_values(1), np.unique(S[live], axis=0))
    # bitmaps: each value has exactly its one live row
    for c, col in ((0, K), (1, S)):
        vals = t.bitmap_values(c)
        rows = np.nonzero(live)[0]
        order = np.argsort(col[live]) if c == 0 else np.lexsort(col[live].T[::-1])
        row_of = rows[order]                                   # row of the k-th smallest live value
        pick = np.unique(np.concatenate([[0, vals.shape[0] - 1], rng.integers(0, vals.shape[0], 2000)]))
        for k in pick:
            v = int(vals[k]) if c == 0 else bytes(vals[k])
            np.testing.assert_array_equal(oracle.positions_from_bits(t.bitmap_get(c, v), n), [row_of[k]])
        absent = int(K[dead[0]]) if c == 0 else bytes(S[dead[0]])
        assert not t.bitmap_get(c, absent).any()

    # scans: EQ present / absent, ranges at 0.1 %, 2 %, 40 %, NE
    sk, ss = np.sort(K[live]), np.unique(S[live], axis=0)
    for c, col, srt in ((0, K, sk), (1, S, ss)):
        lit_of = (lambda k: int(srt[k])) if c == 0 else (lambda k: bytes(srt[k]).rstrip(b"\0"))
        kind = "int" if c == 0 else "str"
        cases = [("=", lit_of(1234)), ("=", int(K[dead[0]]) if c == 0 else bytes(S[dead[0]]).rstrip(b"\0")), ("!=", lit_of(77))]
        for frac in (0.001, 0.02, 0.4):
            k = int(frac * srt.shape[0])
            cases += [("<", lit_of(k)), ("<=", lit_of(k)), (">", lit_of(srt.shape[0] - k)), (">=", lit_of(srt.shape[0] - k))]
        for op, lit in cases:
            terms = [mbcol.Term(OPS[op], ("col", c), (kind, lit), 0)]
            mask = _mask_of(op, col, lit) & live
            _check_scan(oracle, t, terms, mask, cols, [0, 2, 1])
    t.close()


def test_bitsets_beyond_the_device_build_sparse(ctx, oracle):
    """About 400 000 values over 16 M rows: 800 GB of per-value bitsets.  Point and range scans, alone and in a CNF with a
    dense column."""
    n = 16_000_000
    rng = np.random.default_rng(16)
    K = rng.integers(0, 400_000, n).astype(np.int32)
    H = rng.integers(0, 4, n).astype(np.int32)
    cols = [K, H, rng.integers(-50, 50, n).astype(np.int32)]
    t = load_table(ctx, [(1, 4), (1, 4), (1, 4)], cols)
    t.bitmap_build(0)
    t.bitmap_build(1)
    layout, nbytes = t.bitmap_layout(0)
    assert layout == N.BITMAP_SPARSE and nbytes == 4 * n + n // 8 + (-n % 8192) // 8
    assert t.bitmap_layout(1) == (N.BITMAP_DENSE, 4 * ((n + 8191) // 8192 * 8192) // 8)
    np.testing.assert_array_equal(t.bitmap_values(0), np.unique(K))
    np.testing.assert_array_equal(oracle.positions_from_bits(t.bitmap_get(0, 31337), n), np.nonzero(K == 31337)[0])
    for op, lit in (("=", 31337), ("=", 400_001), ("<", 4000), (">=", 200_000), ("!=", 5)):
        _check_scan(oracle, t, [mbcol.Term(OPS[op], ("col", 0), ("int", lit), 0)], _mask_of(op, K, lit), cols, [0, 1])
    terms = [mbcol.Term(N.OP_EQ, ("col", 0), ("int", 17), 0), mbcol.Term(N.OP_LT, ("col", 0), ("int", 1000), 0),
             mbcol.Term(N.OP_EQ, ("col", 1), ("int", 2), 1)]
    _check_scan(oracle, t, terms, ((K == 17) | (K < 1000)) & (H == 2), cols, [0, 1, 2])
    t.close()


def _build(t, cols_, sparse, monkeypatch):
    if sparse:
        monkeypatch.setenv("MBC_BM_SPARSE", "1")
    for c in cols_:
        t.bitmap_build(c)
        assert t.bitmap_layout(c)[0] == (N.BITMAP_SPARSE if sparse else N.BITMAP_DENSE)
    monkeypatch.delenv("MBC_BM_SPARSE", raising=False)


@pytest.mark.parametrize("nrows,nvalues", [(1, 1), (8191, 3), (100_003, 1000), (300_000, 3000)])
def test_forced_sparse_equals_dense_int(ctx, oracle, monkeypatch, nrows, nvalues):
    """The shapes of test_bitmap_gpu.py: deleted rows at build, more deleted after it, every query under both forms."""
    rng = np.random.default_rng(nrows + nvalues)
    descs = [(1, 4), (1, 4), (1, 4), (2, 4)]
    domain = rng.choice(np.arange(-5000, 5000), size=nvalues, replace=False).astype(np.int32)
    cols = [domain[rng.integers(0, nvalues, nrows)], rng.integers(0, 16, nrows).astype(np.int32),
            rng.integers(0, 4, nrows).astype(np.int32), rng.random(nrows).astype(np.float32)]
    dele = oracle.bits_from_positions(np.unique(rng.integers(0, nrows, nrows // 20)), nrows) if nrows > 1000 else None
    dense, sparse, mixed = (load_table(ctx, descs, cols) for _ in range(3))
    for x in (dense, sparse, mixed):
        if dele is not None:
            x.set_deleted(dele)
    _build(dense, range(3), False, monkeypatch)
    _build(sparse, range(3), True, monkeypatch)
    _build(mixed, [0], True, monkeypatch)                      # K sparse, G and H dense in one CNF
    _build(mixed, [1, 2], False, monkeypatch)
    indexes = {}
    for c in range(3):
        indexes[c] = oracle.bitmap_build(descs[c], cols[c], dele)
        vals = dense.bitmap_values(c)
        np.testing.assert_array_equal(sparse.bitmap_values(c), vals)
        assert vals.tolist() == sorted(indexes[c])
        for v in vals.tolist()[:200] + [12345]:
            got = sparse.bitmap_get(c, v)
            np.testing.assert_array_equal(got, dense.bitmap_get(c, v))
            np.testing.assert_array_equal(got, indexes[c].get(v, np.zeros_like(got)))
    names = ["K", "G", "H", "X"]
    srt = np.sort(domain)
    k0, k1, klo, khi = int(domain[0]), int(srt[nvalues // 2]), int(srt[nvalues // 100]), int(srt[-1 - nvalues // 100])
    queries = [f"{{(K,=,{k0})|(G,=,5)}}^{{(H,=,2)}}", f"{{(K,<,{k1})}}^{{(G,!=,3)|(H,>=,2)}}", f"{{(K,>=,{k1})|(K,=,999999)}}",
               f"{{(G,<=,7)}}^{{(G,>,2)}}^{{(H,!=,0)}}", "{(K,=,999999)}", f"{{(K,<=,{klo})}}", f"{{(K,>,{khi})}}",
               f"{{(K,!=,{k0})}}", f"{{(K,<,{int(srt[0])})}}", f"{{(K,>=,{int(srt[0])})}}"]
    after = dele
    for round_ in range(2):
        if round_ == 1 and nrows > 1000:                       # rows deleted after the build: dropped by the combine
            after = dele | oracle.bits_from_positions(np.unique(rng.integers(0, nrows, nrows // 10)), nrows)
            for x in (dense, sparse, mixed):
                x.set_deleted(after)
        for q in queries:
            conj = oracle.parse_cnf(q, names, descs)
            bits = oracle.bitmap_cnf(indexes, names, conj, nrows, deleted_words=after, emulate_duplicate_cache=False)
            terms = oracle.cnf_to_terms(conj, descs)
            ref = dense.bitmap_scan(terms, proj=[0, 3, 1], want=ALL, aggs=[(0, 0), (1, 1)])
            np.testing.assert_array_equal(ref.bitmap(), bits, err_msg=q)
            for form in ("scatter", "compare", None):
                if form:
                    monkeypatch.setenv("MBC_BM_SPARSE_FORM", form)
                for x in (sparse, mixed):
                    res = x.bitmap_scan(terms, proj=[0, 3, 1], want=ALL, aggs=[(0, 0), (1, 1)])
                    np.testing.assert_array_equal(res.bitmap(), bits, err_msg=f"{q} {form}")
                    np.testing.assert_array_equal(res.tuples(), ref.tuples())
                    assert [res.agg(a) for a in range(2)] == [ref.agg(a) for a in range(2)]
                    res.close()
                monkeypatch.delenv("MBC_BM_SPARSE_FORM", raising=False)
            ref.close()
    for x in (dense, sparse, mixed):
        x.close()


def test_forced_sparse_equals_dense_strings(ctx, oracle, monkeypatch):
    """test_bitmap_gpu's string index with over-long and prefix literals, under both forms."""
    nrows = 50_001
    rng = np.random.default_rng(3)
    words = ["Alabama", "Alaska", "Arizona", "Arkansas", "California", "Colorado", "a", "ab", "abc", "abcdefghijklmnop"]
    descs = [(0, 16), (0, 7)]
    cols = [oracle.pack_strings([words[i] for i in rng.integers(0, len(words), nrows)], 16),
            oracle.pack_strings([words[i][:7] for i in rng.integers(0, len(words), nrows)], 7)]
    dense, sparse = load_table(ctx, descs, cols), load_table(ctx, descs, cols)
    _build(dense, [0, 1], False, monkeypatch)
    _build(sparse, [0, 1], True, monkeypatch)
    names = ["S", "T"]
    indexes = {c: oracle.bitmap_build(descs[c], cols[c]) for c in range(2)}
    for c in range(2):
        np.testing.assert_array_equal(sparse.bitmap_values(c), dense.bitmap_values(c))
        for v in indexes[c]:
            np.testing.assert_array_equal(sparse.bitmap_get(c, v), indexes[c][v])
    for q in ["{(S,=,Colorado)}", "{(S,<=,Arkansas)|(T,=,ab)}", "{(S,>,abc)}^{(T,!=,Alaska)}", "{(S,<,A)}", "{(T,=,Alabama1)}",
              "{(T,<=,Alabama1)}", "{(T,>,Alabama1)}", "{(T,>=,Alabama)}", "{(S,>=,abcdefghijklmnop)}", "{(S,!=,a)}", "{(T,<,abcdefgh)}"]:
        conj = oracle.parse_cnf(q, names, descs)
        bits = oracle.bitmap_cnf(indexes, names, conj, nrows, emulate_duplicate_cache=False)
        terms = oracle.cnf_to_terms(conj, descs)
        ref = dense.bitmap_scan(terms, proj=[1, 0], want=ALL)
        np.testing.assert_array_equal(ref.bitmap(), bits, err_msg=q)
        for form in ("scatter", "compare", None):
            if form:
                monkeypatch.setenv("MBC_BM_SPARSE_FORM", form)
            res = sparse.bitmap_scan(terms, proj=[1, 0], want=ALL)
            np.testing.assert_array_equal(res.bitmap(), bits, err_msg=f"{q} {form}")
            np.testing.assert_array_equal(res.tuples(), ref.tuples())
            res.close()
            monkeypatch.delenv("MBC_BM_SPARSE_FORM", raising=False)
        ref.close()
    dense.close(); sparse.close()


def test_golden_sizes_and_indexes_query_under_sparse(ctx, oracle, minidata, golden, monkeypatch):
    """G13/G14 (per-value BitSet.toByteArray() sizes) and G10-G12 (indexes_query rows) with every index sparse."""
    monkeypatch.setenv("MBC_BM_SPARSE", "1")
    dense_suite.test_minidata_bitmaps_match_golden_sizes(ctx, oracle, minidata, golden)
    dense_suite.test_minidata_indexes_query_golden(ctx, oracle, minidata, golden)


def _persisted_image(tmp_path, oracle, minidata, tag):
    names, descs, cols = minidata
    w = oracle.DBWriter()
    oracle.write_columnar_file(w, "cf", names, descs, cols)
    n = 20_011
    sdescs = [(1, 4), (0, 16), (0, 5)]
    scols = [oracle.synth_int(7, 0, n, 50), oracle.synth_str(7, 2, n, 16),
             oracle.pack_strings([["x", "yy", "zzz", "abcde"][i % 4] for i in range(n)], 5)]
    oracle.write_columnar_file(w, "syn", ["I", "S", "T"], sdescs, scols, deleted_positions=[0, 5, 77, 12345, n - 1])
    path = str(tmp_path / f"db_{tag}")
    with open(path, "wb") as f:
        f.write(w.tobytes())
    SystemDefs.shutdown()
    sd = SystemDefs(path, 0, 100, None)
    try:
        cf, syn = Columnarfile("cf"), Columnarfile("syn")
        for c in range(4):
            assert cf.createBitMapIndex(c)
        assert syn.createBitMapIndex(0) and syn.createBitMapIndex(2)
        layouts = [cf.table.bitmap_layout(c)[0] for c in range(4)]
        return bytes(sd.db_bytes), layouts
    finally:
        SystemDefs.shutdown()


def test_persisted_image_is_the_same_under_sparse(tmp_path, oracle, minidata, monkeypatch):
    """Columnarfile.createBitMapIndex writes the same DB image bytes whichever layout built the index."""
    dense_img, dense_layouts = _persisted_image(tmp_path, oracle, minidata, "dense")
    monkeypatch.setenv("MBC_BM_SPARSE", "1")
    sparse_img, sparse_layouts = _persisted_image(tmp_path, oracle, minidata, "sparse")
    assert dense_layouts == [N.BITMAP_DENSE] * 4 and sparse_layouts == [N.BITMAP_SPARSE] * 4
    assert sparse_img == dense_img


def test_scattered_sparse_scan_repeats_bit_identically(ctx, oracle, monkeypatch):
    """50 repeats of a scan whose sparse terms take the scatter form (atomics from many warps) give the same bits."""
    n = 1_000_003
    rng = np.random.default_rng(50)
    K = rng.integers(0, 200_000, n).astype(np.int32)
    G = rng.integers(0, 16, n).astype(np.int32)
    t = load_table(ctx, [(1, 4), (1, 4)], [K, G])
    monkeypatch.setenv("MBC_BM_SPARSE", "1")
    t.bitmap_build(0)
    t.bitmap_build(1)
    monkeypatch.setenv("MBC_BM_SPARSE_FORM", "scatter")
    terms = [mbcol.Term(N.OP_LT, ("col", 0), ("int", 30_000), 0), mbcol.Term(N.OP_EQ, ("col", 1), ("int", 3), 0),
             mbcol.Term(N.OP_NE, ("col", 1), ("int", 7), 1)]
    exp = oracle.mask_to_words(((K < 30_000) | (G == 3)) & (G != 7))
    for _ in range(50):
        r = t.bitmap_scan(terms, want=N.WANT_BITMAP | N.WANT_HOST)
        np.testing.assert_array_equal(r.bitmap(), exp)
        r.close()
    t.close()
