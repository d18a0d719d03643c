"""bench.py --dump-outputs: the helper on CPU tensors, and on a GPU the wiring through the timed
path (the dumped arrays are what the C ABI returns for the same grid)."""
import json
import sys

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_whole_grid_and_fixed_sample(tmp_path, monkeypatch):
    shape = (2, 3, 5)
    s = torch.arange(30, dtype=torch.float64)
    ds = -s
    bench.dump_outputs(str(tmp_path / "all"), {"s": s, "ds": ds}, shape)
    got = np.load(tmp_path / "all" / "s.npy")
    assert got.dtype == np.float64 and np.array_equal(got, s.numpy().reshape(shape))
    assert np.array_equal(np.load(tmp_path / "all" / "ds.npy"), -got)
    # above the size limit: the same seeded sample of every array, identical from run to run
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 8 * 7)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"s": s, "ds": ds}, shape)
    sa, dsa = np.load(tmp_path / "a" / "s.npy"), np.load(tmp_path / "a" / "ds.npy")
    assert sa.shape == (7,) and (np.diff(sa) > 0).all() and np.array_equal(dsa, -sa)   # s = flat index
    assert np.array_equal(sa, np.load(tmp_path / "b" / "s.npy"))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path, monkeypatch, capsys):
    import unconfined_b200 as ub
    out = tmp_path / "dump"
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "1", "--nr", "4", "--nt", "1",
                                      "--nz", "8", "--no-cpu", "--dump-outputs", str(out)])
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 2 and "4r x 8z x 1t" in line["config"]["workload"]
    d, t, r, z = bench.c5a_grid(0, nr=4, nz=8, nt=1)
    p, tD, sv, rD, zD, lay = bench.derive(d, t, r, z, ub)
    s, ds = ub.eval_grid(ub.Params(p), tD, sv, rD, zD, lay)
    assert np.isfinite(s).all() and np.isfinite(ds).all()
    assert np.array_equal(np.load(out / "s.npy"), s) and np.array_equal(np.load(out / "ds.npy"), ds)
