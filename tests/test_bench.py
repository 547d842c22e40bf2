"""CPU: ``bench.py --dump-outputs`` stays within its stated size and is the same on every run."""
import os

import numpy as np
import pytest

import bench


@pytest.mark.parametrize("workload,shapes", [
    ("lstm", [(8192, 1024), (8192, 1024)]),   # two outputs of exactly half the budget each
    ("elemwise", [(1 << 25,)]),               # one output far over the budget: sampled
    ("mlp", [(), (4096, 4096), (4096,), (4096, 4096), (4096,)]),
])
def test_dump_outputs_stay_within_the_budget(tmp_path, workload, shapes):
    names = bench.workload_spec(workload)["outputs"]
    rng = np.random.default_rng(0)
    outs = [rng.standard_normal(s, dtype=np.float32) for s in shapes]
    for run in ("a", "b"):
        bench.dump_outputs(outs, names, str(tmp_path / run))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(n + ".npy" for n in names)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BUDGET
    for f, o in zip([n + ".npy" for n in names], outs):
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
        assert a.shape == o.shape or (a.ndim == 1 and a.size < o.size)  # whole, or a sample
