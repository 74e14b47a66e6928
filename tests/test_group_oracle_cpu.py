"""The grouped-aggregation oracle (tests/group_oracle.py) pinned against a plain-Python dict fold (CPU): random small tables with -0.0 / +0.0 real keys,
char keys that differ only in length, deleted rows, with and without a filter."""
import numpy as np
import pytest
from group_oracle import group_aggregate


def _dict_fold(descs, cols, live_positions, key_cols, aggs):
    """{key tuple: [first position, per aggregate (i, f)]} folded row by row in position order, groups in key order."""
    groups = {}
    for p in live_positions:
        key = []
        for c in key_cols:
            t, w = descs[c]
            if t == 0:
                key.append(bytes(cols[c][p]).rstrip(b"\0"))
            elif t == 2:
                key.append(float(cols[c][p]) + 0.0)            # -0.0 and +0.0 are one key
            else:
                key.append(int(cols[c][p]))
        key = tuple(key)
        if key not in groups:
            groups[key] = [p, [None] * len(aggs), 0]
        g = groups[key]
        g[2] += 1
        for a, (kind, col) in enumerate(aggs):
            if kind == 0:
                g[1][a] = g[2]
                continue
            v = int(cols[col][p]) if descs[col][0] == 1 else float(cols[col][p])
            cur = g[1][a]
            g[1][a] = v if cur is None else cur + v if kind == 1 else min(cur, v) if kind == 2 else max(cur, v)
    return [(k, groups[k]) for k in sorted(groups)]


def _table(rng, n):
    descs = [(1, 4), (2, 4), (0, 5), (1, 4), (2, 4)]
    zeros = np.array([0.0, -0.0, 1.5, -2.25, np.inf, -np.inf], dtype=np.float32)
    words = [b"", b"a", b"ab", b"abc", b"abcd", b"abcde", b"b"]
    strs = np.zeros((n, 5), dtype=np.uint8)
    for i, k in enumerate(rng.integers(0, len(words), n)):
        strs[i, :len(words[k])] = np.frombuffer(words[k], dtype=np.uint8) if words[k] else []
    cols = [rng.integers(-3, 4, n).astype(np.int32), zeros[rng.integers(0, zeros.size, n)], strs,
            rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32), rng.standard_normal(n).astype(np.float32) * 1e3]
    return descs, cols


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("key_cols", [[0], [1], [2], [2, 0], [1, 2, 0]])
def test_group_aggregate_oracle_matches_a_dict_fold(oracle, seed, key_cols):
    rng = np.random.default_rng(seed)
    n = 700
    descs, cols = _table(rng, n)
    deleted = np.sort(rng.choice(n, 40, replace=False))
    words = oracle.bits_from_positions(deleted, n)
    aggs = [(0, 0), (1, 3), (1, 4), (2, 3), (3, 3), (2, 4), (3, 4)]
    for terms, qual in (([], np.ones(n, bool)),
                        ([oracle.Term(oracle.OP_LT, ("col", 3), ("int", 2**30), 0)], cols[3] < 2**30)):
        live = [p for p in range(n) if qual[p] and p not in set(deleted.tolist())]
        exp = _dict_fold(descs, cols, live, key_cols, aggs)
        got = group_aggregate(descs, cols, terms, key_cols, aggs, deleted_words=words)
        assert got["count"] == len(exp)
        assert got["positions"].tolist() == [g[0] for _, g in exp]
        for g, (key, (first, vals, _)) in enumerate(exp):
            for k, c in enumerate(key_cols):
                kv = got["keys"][k][g]
                if descs[c][0] == 0:
                    assert bytes(kv).rstrip(b"\0") == key[k]
                else:
                    assert kv == key[k]
            for a, (kind, col) in enumerate(aggs):
                gi, gf = got["aggs"][a][0][g], got["aggs"][a][1][g]
                if kind == 0 or descs[col][0] == 1:
                    assert gi == vals[a] and gf == float(vals[a])
                else:
                    assert gf == vals[a] or (np.isnan(gf) and np.isnan(vals[a]))


def test_group_aggregate_oracle_empty_and_all_filtered(oracle):
    descs, cols = _table(np.random.default_rng(9), 50)
    got = group_aggregate(descs, cols, [oracle.Term(oracle.OP_LT, ("col", 0), ("int", -100), 0)], [0], [(0, 0), (1, 3)])
    assert got["count"] == 0 and got["positions"].size == 0 and got["aggs"][1][0].size == 0
    got = group_aggregate([(1, 4)], [np.empty(0, np.int32)], [], [0], [(0, 0)])
    assert got["count"] == 0
