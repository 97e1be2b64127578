"""CPU: bench.py --dump-outputs writes the four solution vectors and the stats of one solve_two_mixed call as
float64 .npy files, whole below 64 MB and as the same seeded sample of every vector above."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def _solve_output(n, m):
    rng = np.random.default_rng(3)
    vecs = [torch.tensor(rng.standard_normal(k)) for k in (n, m, n, m)]
    stats = [dict(niter=12, solved=True, inconsistent=False, status=2, rnorm=1e-9, arnorm=2e-9, anorm=3.0,
                  acond=4.0, xnorm=5.0), dict(niter=9, solved=True, inconsistent=False, status=2, rnorm=6e-9,
                                              arnorm=0.0, anorm=7.0, acond=8.0, xnorm=9.0)]
    return (*vecs, stats)


def test_dump_outputs_whole(tmp_path):
    out = _solve_output(100, 40)
    bench.dump_outputs(str(tmp_path), out)
    assert sorted(os.listdir(tmp_path)) == ["p1.npy", "p2.npy", "q1.npy", "q2.npy", "stats.npy"]
    for name, x in zip(bench.OUTPUT_NAMES, out[:4]):
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, x.numpy())
    st = np.load(tmp_path / "stats.npy")
    assert st.dtype == np.float64 and st.shape == (2, len(bench.STAT_FIELDS))
    assert st[0, 0] == 12 and st[1, 0] == 9 and st[1, bench.STAT_FIELDS.index("xnorm")] == 9.0


def test_dump_outputs_sampled_past_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 16 << 10)
    out = _solve_output(3000, 1000)
    bench.dump_outputs(str(tmp_path / "a"), out)
    bench.dump_outputs(str(tmp_path / "b"), out)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= 16 << 10
    for name, x in zip(bench.OUTPUT_NAMES, out[:4]):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert 0 < len(a) < len(x) and np.array_equal(a, b)
        assert np.isin(a, x.numpy()).all()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bad_arguments_rejected(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
