"""mbc_sort at scale and at the edges of its radix sort, through Table.sort only.

The sort (csrc/mbc_sort.cu) reorders row ids with a stable LSD radix sort, one 8-bit pass per byte of every 32-bit key
word, skipping the bytes that are the same in all keys (radix_sort_pairs, csrc/mbc_join.cu).  A pass's scatter kernel
takes 8192 pairs per block, 1024 consecutive ones per warp.  exclusive_scan_u32 scans the pass's 256 x blocks digit
counts in chunks of 4096 entries and carries the chunk sums 1024 chunks at a time.  The sizes below sit on and beside
those boundaries.  The same code orders the bitmap join's pairs and builds the sparse bitmap layout.

Expected orders come from oracle.sort (ties by ascending position); the full-size test uses an O(n) property check.
Projected columns are compared bit for bit, so -0.0 and +0.0 are told apart."""
import itertools

import numpy as np
import pytest

from mbcol import _native as N
from util import load_table

pytestmark = pytest.mark.gpu

POS = N.WANT_POSITIONS | N.WANT_HOST
PC = N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST
ALL = PC | N.WANT_TUPLES
CHUNK = 8192                                   # pairs per rsort_scatter_kernel block
I32_MIN, I32_MAX = -2**31, 2**31 - 1
INT, REAL = (N.ATTR_INTEGER, 4), (N.ATTR_REAL, 4)
F32 = np.finfo(np.float32)


def _str(width):
    return (N.ATTR_STRING, width)


def _bits(a):
    """int / real columns as their uint32 bit patterns (assert_array_equal takes -0.0 == +0.0); strings as bytes."""
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype.itemsize == 4 else a


def _full_range(rng, n):
    return rng.integers(I32_MIN, I32_MAX + 1, n, dtype=np.int64).astype(np.int32)


def _words(rng, count, width):
    """`count` random ASCII strings of 0..width bytes, a few ending in a 2-byte UTF-8 letter (bytes >= 0x80)."""
    alphabet = list("abcxyzAZ09-_~")
    out = []
    for i in range(count):
        s = "".join(rng.choice(alphabet, int(rng.integers(0, width + 1))))
        out.append(s[:width - 2] + "é" if i % 10 == 0 else s)
    return out


def _strings(oracle, rng, words, width, n):
    return oracle.pack_strings(words, width)[rng.integers(0, len(words), n)]


def _check(res, exp, cols, proj, base=0):
    assert res.count == exp.size
    np.testing.assert_array_equal(res.positions(), exp + base)
    for i, c in enumerate(proj):
        np.testing.assert_array_equal(_bits(res.column(i)), _bits(cols[c][exp]), err_msg=f"projected column {c}")


def _sort_and_check(oracle, t, descs, cols, keys, desc, proj, deleted=(), base=0):
    exp = oracle.sort(descs, cols, keys, descending=desc, deleted_positions=deleted)
    res = t.sort(keys, descending=desc, proj=proj, want=PC)
    _check(res, exp, cols, proj, base)
    res.close()
    return exp


# ---- a. block and scan-chunk boundaries ---------------------------------------------------------------------------

def _ints_with_ties(rng, n):
    """Full-range int32 keys, each value about 8 times (so ties straddle blocks); INT32_MIN, INT32_MAX, -1 and 0 twice
    each at least."""
    pool = _full_range(rng, max(n // 8, 4))
    v = pool[rng.integers(0, pool.size, n)]
    v[rng.choice(n, 8, replace=False)] = [I32_MIN, I32_MAX, -1, 0] * 2
    return v


@pytest.mark.parametrize("n", [CHUNK - 1, CHUNK, CHUNK + 1, 5 * CHUNK + 1000, 5 * CHUNK + 1024, 16 * CHUNK, 16 * CHUNK + 1,
                               3_000_017])
@pytest.mark.parametrize("desc", [False, True])
def test_block_and_scan_chunk_boundaries(ctx, oracle, n, desc):
    """One block short of full, full, and one row into a second block; a last block that ends inside a warp's 1024-row
    slice, and one that ends on a warp boundary; 16 blocks, whose 4096-entry histogram is exactly one scan chunk, and
    16 blocks + 1 row, whose histogram takes two; 367 blocks."""
    rng = np.random.default_rng(n)
    descs = [INT, INT]
    cols = [_ints_with_ties(rng, n), _full_range(rng, n)]
    t = load_table(ctx, descs, cols)
    _sort_and_check(oracle, t, descs, cols, [0], desc, proj=[1, 0])
    t.close()


# ---- b. digit skipping --------------------------------------------------------------------------------------------

# int keys by which bytes of their sign-biased form (the radix digits) vary; x is uniform in [0, 256)
DIGIT_KEYS = {
    "constant": lambda x, rng: np.full(x.size, -7, np.int32),
    "byte 0": lambda x, rng: (0x12345600 + x).astype(np.int32),
    "byte 1": lambda x, rng: (5 + 256 * x).astype(np.int32),
    "byte 2": lambda x, rng: (9 + (x << 16)).astype(np.int32),
    "byte 3": lambda x, rng: ((x << 24) + I32_MIN).astype(np.int32),          # INT32_MIN (x = 0) and 0 (x = 128) among them
    "all bytes": lambda x, rng: _full_range(rng, x.size),
}


@pytest.mark.parametrize("desc", [False, True])
def test_digit_skipping(ctx, oracle, desc):
    """A byte that is the same in every key needs no pass: the order is right whichever passes run, a constant key
    keeps position order, and four varying bytes cost three more passes than one (pinned by kernel-launch deltas on
    tables of one size, so the launches of one pass are not hard-coded)."""
    n = 100_003
    rng = np.random.default_rng(11)
    x = rng.integers(0, 256, n)
    descs = [INT, INT]
    launches = {}
    for name, make in DIGIT_KEYS.items():
        cols = [make(x, rng), np.arange(n, dtype=np.int32)]
        t = load_table(ctx, descs, cols)
        before = ctx.kernel_launches
        res = t.sort([0], descending=desc, proj=[0, 1], want=PC)
        launches[name] = ctx.kernel_launches - before
        exp = oracle.sort(descs, cols, [0], descending=desc)
        if name == "constant":
            np.testing.assert_array_equal(exp, np.arange(n))
        _check(res, exp, cols, [0, 1])
        res.close()
        t.close()
    l0, l1, l4 = launches["constant"], launches["byte 1"], launches["all bytes"]
    assert all(launches[f"byte {b}"] == l1 for b in range(4)), launches
    assert l4 - l1 == 3 * (l1 - l0) > 0, launches


# ---- c. string keys -----------------------------------------------------------------------------------------------

PREFIX = ("common-prefix-" * 5)[:60]


def _string_vocab():
    tails = ["".join(p) for k in range(1, 5) for p in itertools.product("a~b", repeat=k)]     # the last 1-4 bytes differ
    tails += ["é", "aé", "é~", "€", "中", "ÿÿ", "Ā", "ߦ"]                                         # 2- and 3-byte UTF-8
    w64 = [PREFIX + s for s in tails]
    w64 += [PREFIX[:k] for k in (1, 30, 59, 60)]                                                # proper prefixes of those
    w64 += ["a" * k for k in range(1, 65)]                                                      # differ only in length
    w64 += ["", "é", "ü", "€", "中文", "日本語", "\uffff", "Z", "z", "~"]
    w5 = ["", "a", "ab", "abcd", "abcde", "abcdd", "b", "é", "éé", "a€", "a€b", "中", "中a", "zzzz", "zzzzz", "\uffff"]
    return w64, w5


@pytest.mark.parametrize("keys", [[0], [1], [1, 0]], ids=["char64", "char5", "char5-char64"])
@pytest.mark.parametrize("desc", [False, True])
def test_string_keys(ctx, oracle, keys, desc):
    """char(64): 16 key words, of which only the last varies among the prefixed keys; keys that differ only in length
    (zero padding against a byte); UTF-8 bytes >= 0x80.  char(5): a 2-word key in an 8-byte stride whose padding
    must not count."""
    n = 120_001
    rng = np.random.default_rng(13)
    w64, w5 = _string_vocab()
    descs = [_str(64), _str(5), INT]
    cols = [_strings(oracle, rng, w64, 64, n), _strings(oracle, rng, w5, 5, n), np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    _sort_and_check(oracle, t, descs, cols, keys, desc, proj=[2, 0, 1])
    t.close()


# ---- d. real keys -------------------------------------------------------------------------------------------------

EDGE_REALS = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.17e-38, -1.17e-38, F32.tiny, -F32.tiny, F32.max, -F32.max,
                       1.0, -1.0, 0.1, -0.1], dtype=np.float32)


def _edge_reals(rng, n):
    """40 % zeros of either sign interleaved, 30 % EDGE_REALS (infinities, subnormals, FLT_MAX), 30 % ordinary values."""
    pick = rng.random(n)
    zeros = np.where(rng.random(n) < 0.5, np.float32(0.0), np.float32(-0.0))
    v = np.where(pick < 0.4, zeros, np.where(pick < 0.7, EDGE_REALS[rng.integers(0, EDGE_REALS.size, n)],
                                             rng.standard_normal(n) * 1e3)).astype(np.float32)
    v[:10] = [0.0, -0.0, 1.5, -0.0, 0.0, -1.0, np.inf, -np.inf, 1e-45, -1e-45]
    return v


@pytest.mark.parametrize("keys", [[1], [0, 1]], ids=["real", "int-then-real"])
@pytest.mark.parametrize("desc", [False, True])
def test_real_keys_at_their_edges(ctx, oracle, keys, desc):
    """Reals compare as floats (TupleUtils), so -0.0 and +0.0 are one key and tie by position; infinities, subnormals
    and +-FLT_MAX sort numerically.  No NaN: real columns exclude it."""
    n = 50_021
    rng = np.random.default_rng(17)
    descs = [INT, REAL, INT]
    cols = [rng.integers(0, 3, n).astype(np.int32), _edge_reals(rng, n), np.arange(n, dtype=np.int32)]
    t = load_table(ctx, descs, cols)
    exp = _sort_and_check(oracle, t, descs, cols, keys, desc, proj=[1, 2, 0])
    if keys == [1]:                                  # the zeros of both signs form one run, in position order
        z = exp[cols[1][exp] == 0]
        assert z.size > n // 4 and np.all(np.diff(z) > 0)
    t.close()


# ---- e. three keys at scale ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("desc", [False, True])
def test_three_keys_at_scale(ctx, oracle, desc):
    """int (20 values), char(16) (~1000 values), real (5 % zeros, so all three keys tie): positions, the three
    projected columns and the Tuple bytes, which must be those of the oracle's scan row at each position."""
    n = 2_000_003
    rng = np.random.default_rng(23)
    descs = [INT, _str(16), REAL]
    reals = (rng.standard_normal(n) * 100).astype(np.float32)
    reals[rng.random(n) < 0.05] = np.float32(0.0)
    cols = [rng.integers(-10, 10, n).astype(np.int32), _strings(oracle, rng, _words(rng, 1000, 16), 16, n), reals]
    t = load_table(ctx, descs, cols)
    exp = oracle.sort(descs, cols, [0, 1, 2], descending=desc)
    res = t.sort([0, 1, 2], descending=desc, proj=[0, 1, 2], want=ALL)
    _check(res, exp, cols, [0, 1, 2])
    scan = oracle.scan(descs, cols, [], proj=[0, 1, 2], want_positions=False, nthreads=oracle.max_threads())
    np.testing.assert_array_equal(res.tuples(), scan["tuples"][exp])
    res.close()
    t.close()


# ---- f. deleted rows and a position base past 2^32 ----------------------------------------------------------------

@pytest.mark.parametrize("desc", [False, True])
def test_deleted_rows_and_position_base(ctx, oracle, desc):
    """Positions start at 3 * 2^31 + 7, past 2^32, while row ids stay small.  Deleted: the first and the last row, a
    run across the 8192-row block boundary, and 10 % at random; the deleted bitmap is indexed by row."""
    n, base = 200_003, 3 * 2**31 + 7
    rng = np.random.default_rng(29)
    descs = [INT, _str(16), INT]
    cols = [rng.integers(-50, 50, n).astype(np.int32), _strings(oracle, rng, _words(rng, 300, 16), 16, n), _full_range(rng, n)]
    t = load_table(ctx, descs, cols, base)
    dele = np.unique(np.concatenate([[0, n - 1], np.arange(CHUNK - 300, CHUNK + 300), rng.choice(n, n // 10, replace=False)]))
    t.set_deleted(oracle.bits_from_positions(dele, n))
    exp = _sort_and_check(oracle, t, descs, cols, [0, 1], desc, proj=[2, 1, 0], deleted=dele, base=base)
    assert exp.size == n - dele.size
    t.close()


# ---- g. what is asked for -----------------------------------------------------------------------------------------

def test_each_part_of_the_result_alone(ctx, oracle):
    """Positions only, columns only, Tuple bytes only, and positions with no projected field: each equals that part of
    the full result of the same sort."""
    n = 100_003
    rng = np.random.default_rng(37)
    descs = [INT, _str(16), REAL]
    cols = [rng.integers(-30, 30, n).astype(np.int32), _strings(oracle, rng, _words(rng, 500, 16), 16, n),
            _edge_reals(rng, n)]
    t = load_table(ctx, descs, cols)
    keys, proj = [1, 0], [2, 0, 1]
    full = t.sort(keys, proj=proj, want=ALL)
    exp = oracle.sort(descs, cols, keys)
    _check(full, exp, cols, proj)
    pos, tup = full.positions().copy(), full.tuples().copy()
    fcols = [full.column(i).copy() for i in range(len(proj))]
    full.close()

    r = t.sort(keys, proj=proj, want=POS)
    assert r.count == n
    np.testing.assert_array_equal(r.positions(), pos)
    r.close()
    r = t.sort(keys, proj=proj, want=N.WANT_COLUMNS | N.WANT_HOST)
    assert r.count == n
    for i in range(len(proj)):
        np.testing.assert_array_equal(_bits(r.column(i)), _bits(fcols[i]))
    r.close()
    r = t.sort(keys, proj=proj, want=N.WANT_TUPLES | N.WANT_HOST)
    assert r.count == n
    np.testing.assert_array_equal(r.tuples(), tup)
    r.close()
    r = t.sort(keys, proj=[], want=ALL)
    assert r.count == n and r.tuples().size == 0
    np.testing.assert_array_equal(r.positions(), pos)
    r.close()
    t.close()


# ---- h. full size -------------------------------------------------------------------------------------------------

def _check_sorted_permutation(keys, pos, descending):
    """O(n): pos is a permutation of range(n), keys[pos] is monotone, and equal neighbours keep position order."""
    n = keys.size
    assert pos.size == n and pos.min() >= 0 and pos.max() < n
    seen = np.zeros(n, dtype=bool)
    seen[pos] = True
    assert seen.all()
    k = keys[pos]
    assert (k[1:] <= k[:-1] if descending else k[1:] >= k[:-1]).all()
    tie = k[1:] == k[:-1]
    assert tie.any() and (pos[1:][tie] > pos[:-1][tie]).all()


def test_full_size_int_key(ctx):
    """2^27 + 3 rows of full-range int32 keys (about 2 M equal neighbours): 16 385 scatter blocks, so the digit
    histogram's 1025 scan chunks take the chunk-sum carry past its first 1024.  Keys are drawn on the host because the
    device generator's int domain stops at 2^31 and never yields negatives."""
    n = 2**27 + 3
    keys = np.random.default_rng(41).integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
    t = ctx.create_table([INT], n)
    t.load_column(0, keys)
    for desc in (False, True):
        res = t.sort([0], descending=desc, want=POS)
        assert res.count == n
        _check_sorted_permutation(keys, res.positions(), desc)
        res.close()
    t.close()


# ---- i. determinism -----------------------------------------------------------------------------------------------

def test_repeats_are_bit_identical(ctx, oracle):
    """Ten sorts of one 4 M-row, two-key table return the same positions (the scatter's placement must not depend on
    the timing of its atomics)."""
    n = 4_000_037
    rng = np.random.default_rng(43)
    descs = [INT, _str(16)]
    cols = [rng.integers(-1000, 1000, n).astype(np.int32), _strings(oracle, rng, _words(rng, 1000, 16), 16, n)]
    t = load_table(ctx, descs, cols)
    res = t.sort([0, 1], want=POS)
    first = res.positions().copy()
    res.close()
    np.testing.assert_array_equal(first, oracle.sort(descs, cols, [0, 1]))
    for _ in range(9):
        res = t.sort([0, 1], want=POS)
        assert np.array_equal(res.positions(), first)
        res.close()
    t.close()
