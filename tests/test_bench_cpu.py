"""CPU: bench.py's output dump -- one .npy per array, dtypes kept, a fixed seeded sample of games past the size limit --
and its argument checks."""
import sys

import numpy as np
import pytest

import bench


def _arrays(n=1000, A=24):
    rs = np.random.RandomState(5)
    return {"root_visits": rs.randint(0, 800, (n, A)).astype(np.float32), "root_priors": rs.rand(n, A)}


def test_dump_outputs_writes_every_array_whole_below_the_limit(tmp_path):
    arrays = _arrays()
    bench.dump_outputs(str(tmp_path / "d"), arrays)
    for name, a in arrays.items():
        got = np.load(str(tmp_path / "d" / (name + ".npy")))
        assert got.dtype == a.dtype and np.array_equal(got, a)


def test_dump_outputs_samples_the_same_games_past_the_limit(tmp_path):
    arrays = _arrays()
    limit = 64 * 1024
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=limit)
    a = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in arrays}
    b = {k: np.load(str(tmp_path / "b" / (k + ".npy"))) for k in arrays}
    assert 0 < sum(v.nbytes for v in a.values()) <= limit
    assert all(np.array_equal(a[k], b[k]) for k in arrays)
    # every array keeps the same games, in game order
    rows = [int(np.flatnonzero((arrays["root_priors"] == r).all(1))[0]) for r in a["root_priors"]]
    assert rows == sorted(rows) and np.array_equal(a["root_visits"], arrays["root_visits"][rows])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse_args()
