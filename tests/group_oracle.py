"""GROUP BY restated on the CPU for the grouped-aggregation tests (test infrastructure, like oracle/).

The reference has no aggregates; a grouped aggregate is defined like the scan's (SURVEY.md F5, oracle/mbc_oracle.cpp):
the qualifying positions come from the row-at-a-time filter (`oracle.scan`), groups are keyed like `oracle.sort`
ascending (reals compare numerically, so -0.0 and +0.0 are one key), and per group COUNT, exact int SUM, the double SUM
of the float32 values in ascending position order, and exact MIN / MAX."""
import numpy as np

from oracle import oracle as orc

_I64_MAX, _I64_MIN = 2**63 - 1, -2**63


def _real_as_i64(d: np.ndarray) -> np.ndarray:
    """Java's (long) of a double: toward zero, saturated to INT64_MIN / INT64_MAX (±inf too), NaN -> 0."""
    out = np.zeros(d.shape, dtype=np.int64)
    fin = np.isfinite(d) & (d < 9223372036854775808.0) & (d >= -9223372036854775808.0)
    out[fin] = np.trunc(d[fin]).astype(np.int64)
    out[~np.isnan(d) & (d >= 9223372036854775808.0)] = _I64_MAX
    out[~np.isnan(d) & (d < -9223372036854775808.0)] = _I64_MIN
    return out


def _sequential_sums(x: np.ndarray, starts: np.ndarray) -> np.ndarray:
    """Per group, the double sum of its values added one at a time in order, from 0.0 (vectorised over the groups)."""
    sizes = np.diff(starts)
    acc = np.zeros(sizes.size, dtype=np.float64)
    for k in range(int(sizes.max()) if sizes.size else 0):
        live = sizes > k
        acc[live] = acc[live] + x[starts[:-1][live] + k]
    return acc


def group_aggregate(coldescs, columns, terms, key_cols, aggs=(), deleted_words=None) -> dict:
    """{"count", "positions" (lowest qualifying position per group), "keys" (per key column: that row's values),
    "aggs" (per aggregate: (int64 array, float64 array), the pair mbc_result_agg gives for the group's rows)}."""
    pos = orc.scan(coldescs, columns, terms, deleted_words=deleted_words, want_tuples=False)["positions"]
    n, nrows = pos.size, orc.nrows_of(coldescs, columns)
    ranks = []
    for c in key_cols:
        t, w = coldescs[c]
        col = np.asarray(columns[c])
        if t == orc.ATTR_STRING:
            vals = np.ascontiguousarray(col.reshape(nrows, -1)[pos, :w]).view(f"S{w}").reshape(n)   # bytes, NUL padded
        elif t == orc.ATTR_REAL:
            vals = col.reshape(-1)[pos].astype(np.float32) + np.float32(0.0)                        # -0.0 + 0.0 = +0.0
        else:
            vals = col.reshape(-1)[pos]
        ranks.append(np.unique(vals, return_inverse=True)[1].reshape(n))
    order = np.lexsort(tuple(reversed(ranks))) if n else np.empty(0, dtype=np.int64)                # stable: ties by position
    heads = np.ones(n, dtype=bool)
    if n:
        srt = np.stack([r[order] for r in ranks])
        heads[1:] = np.any(srt[:, 1:] != srt[:, :-1], axis=0)
    starts = np.append(np.nonzero(heads)[0], n).astype(np.int64)
    rows = pos[order]
    first = rows[starts[:-1]].astype(np.int64)
    keys = []
    for c in key_cols:
        t, w = coldescs[c]
        col = np.asarray(columns[c])
        keys.append(col.reshape(nrows, -1)[first, :w] if t == orc.ATTR_STRING else col.reshape(-1)[first])
    out = []
    G = starts.size - 1
    for kind, c in aggs:
        if kind == orc.AGG_COUNT:
            i = np.diff(starts)
            out.append((i, i.astype(np.float64)))
            continue
        if G == 0:
            out.append((np.empty(0, np.int64), np.empty(0, np.float64)))
            continue
        x = np.asarray(columns[c]).reshape(-1)[rows]
        if coldescs[c][0] == orc.ATTR_INTEGER:
            ufunc = np.add if kind == orc.AGG_SUM else np.minimum if kind == orc.AGG_MIN else np.maximum
            i = ufunc.reduceat(x.astype(np.int64), starts[:-1])
            out.append((i, i.astype(np.float64)))
        else:
            x = x.astype(np.float32).astype(np.float64)
            if kind == orc.AGG_SUM:
                f = _sequential_sums(x, starts)
            else:
                f = (np.minimum if kind == orc.AGG_MIN else np.maximum).reduceat(x, starts[:-1])
            out.append((_real_as_i64(f), f))
    return {"count": G, "positions": first, "keys": keys, "aggs": out}
