"""CPU: bench.py --dump-outputs writes float64 .npy files, at most 64 MB, the same ones on every run (a fixed sample of a long
solution), so that two builds of the project can be compared output for output."""
import os

import numpy as np
import pytest

import bench


class _Solved:
    """stands in for a Solver after its last timed solve: only get_solution is read"""

    def __init__(self, n):
        self.n0 = n

    def get_solution(self):
        return np.cos(np.arange(self.n0) * 0.37)


def _dump(d, n, hist, corr, rel):
    bench.dump_outputs(str(d), _Solved(n), hist, corr, rel)
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_sync_solve_dumps_history_and_whole_solution(tmp_path):
    hist = np.asarray([1.0, 0.1, 3e-10])
    out = _dump(tmp_path, 1000, hist, None, hist[-1])
    assert sorted(out) == ["relres_history", "solution"]
    assert np.array_equal(out["relres_history"], hist)
    assert np.array_equal(out["solution"], _Solved(1000).get_solution())


@pytest.mark.parametrize("n", [bench.DUMP_SAMPLE + 1, 256 ** 3])
def test_long_solution_is_a_fixed_sample_under_64_mb(tmp_path, n):
    corr = np.asarray([40, 40, 41], dtype=np.int32)
    a = _dump(tmp_path / "a", n, None, corr, 4e-10)
    b = _dump(tmp_path / "b", n, None, corr, 4e-10)
    assert sorted(a) == ["corrections_per_level", "final_relres", "solution_sample", "solution_sample_rows"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)
    rows = a["solution_sample_rows"].astype(np.int64)
    assert len(rows) == bench.DUMP_SAMPLE and np.all(np.diff(rows) > 0) and rows[-1] < n
    assert np.array_equal(a["solution_sample"], _Solved(n).get_solution()[rows])
    assert list(a["corrections_per_level"]) == [40, 40, 41] and a["final_relres"][0] == 4e-10
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64 * 2 ** 20
