"""bench.py --dump-outputs: the files hold what the timed scans returned -- checked against the oracle on the same seeded
table, through the row sample where a query returns more rows than the dump's size limit allows -- and two runs with the
same arguments write identical files.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

from util import C2_AGGS, C2_DESCS, c2_columns, c2_terms

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 1_000_000                      # the 50 % query returns more rows than fit the dump: it is sampled


def _bench_dump(out_dir):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--rows", str(ROWS),
                        "--no-cpu-baseline", "--no-pageable", "--e2e-steps", "1", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert len([ln for ln in p.stdout.splitlines() if ln.strip()]) == 1
    return {f: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_hold_the_last_steps_results(oracle, tmp_path):
    a = _bench_dump(tmp_path / "a")
    b = _bench_dump(tmp_path / "b")
    assert a.keys() == b.keys()
    for f in a:
        np.testing.assert_array_equal(a[f], b[f])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in a) <= 64_000_000
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())

    cols = c2_columns(oracle, ROWS)
    for sel in (0.01, 0.1, 0.5):
        exp = oracle.scan(C2_DESCS, cols, c2_terms(oracle, sel), aggs=C2_AGGS, want_tuples=False,
                          nthreads=oracle.max_threads())
        pos = a[f"sel{sel}_positions.npy"].astype(np.int64)
        if sel == 0.5:
            assert 100_000 < len(pos) < exp["count"]
            assert np.all(np.diff(pos) > 0) and np.all(np.isin(pos, exp["positions"]))
        else:
            np.testing.assert_array_equal(pos, exp["positions"])
        np.testing.assert_array_equal(a[f"sel{sel}_col0.npy"], cols[0][pos].astype(np.float64))
        np.testing.assert_array_equal(a[f"sel{sel}_col1.npy"], cols[1][pos].astype(np.float64))
        np.testing.assert_array_equal(a[f"sel{sel}_col2.npy"].view(np.uint32), cols[2][pos].view(np.uint32))
        np.testing.assert_array_equal(a[f"sel{sel}_col3.npy"], cols[3][pos].astype(np.float32))
        aggs = a[f"sel{sel}_aggs.npy"]
        assert aggs.dtype == np.float64 and len(aggs) == len(C2_AGGS)
        for got, (ei, ef, ev) in zip(aggs, exp["aggs"]):
            assert ev
            if float(ei) == ef:
                assert got == ei
            else:
                assert abs(got - ef) <= 1e-6 * abs(ef)
