"""bench.py --dump-outputs: the sampled rows are the rows of the result, every file is float64 and within the size
budget, and on the GPU the dump of the timed step equals what Interpolator.interpolate returns for the same mesh."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from helpers import ROOT

import bench


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d) if f.endswith(".npy")}


def _check_rows(out, indptr, indices, data, neumann):
    rows = out["rows"].astype(np.int64)
    assert np.all(np.diff(rows) > 0)
    assert np.array_equal(out["row_nnz"], np.diff(indptr)[rows])
    take = np.concatenate([np.arange(indptr[p], indptr[p + 1]) for p in rows])
    assert np.array_equal(out["indices"], indices[take])
    assert np.array_equal(out["data"], data[take], equal_nan=True)
    assert np.array_equal(out["neumann"], neumann[rows])


def test_dump_samples_rows_of_the_fetched_csr(tmp_path, monkeypatch):
    rng = np.random.default_rng(3)
    n_rows, n_cols = 100_000, 400_000
    cnt = rng.integers(0, 30, n_rows)
    cnt[::5] = 0                                     # Dirichlet rows are empty
    indptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    indices = rng.integers(0, n_cols, int(indptr[-1])).astype(np.int32)
    data = rng.standard_normal(int(indptr[-1]))
    data[7] = np.nan
    neumann = rng.standard_normal(n_rows)

    class Ctx:
        def interpolate_fetch(self, *dst):
            for d, s in zip(dst, (indptr, indices, data, neumann)):
                if d is not None:
                    d[:] = s
    I = types.SimpleNamespace(_ctx=Ctx(), grid=types.SimpleNamespace(n_points=n_rows, n_elems=n_cols))

    bench.dump_outputs(I, str(tmp_path / "a"))
    out = _load(tmp_path / "a")
    assert sorted(out) == ["data", "indices", "neumann", "row_nnz", "rows", "totals"]
    assert all(a.dtype == np.float64 for a in out.values())
    assert len(out["rows"]) == bench.DUMP_ROWS
    _check_rows(out, indptr, indices, data, neumann)
    assert out["totals"][:4].tolist() == [n_rows, n_cols, indptr[-1], 1]
    assert out["totals"][4] == np.nansum(data) and out["totals"][7] == np.sum(neumann)

    bench.dump_outputs(I, str(tmp_path / "b"))       # same inputs, same files
    again = _load(tmp_path / "b")
    assert all(np.array_equal(out[k], again[k], equal_nan=True) for k in out)

    monkeypatch.setattr(bench, "DUMP_CHUNK", 1000)  # the sums, taken a chunk at a time, are the same to rounding
    bench.dump_outputs(I, str(tmp_path / "chunked"))
    chunked = _load(tmp_path / "chunked")["totals"]
    want = [np.nansum(data), np.nansum(np.abs(data)), np.nansum(data * (indices + 1.0))]
    assert chunked[3] == 1 and np.allclose(chunked[4:7], want, rtol=1e-12, atol=1e-9)

    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    bench.dump_outputs(I, str(tmp_path / "c"))
    small = _load(tmp_path / "c")
    assert sum(os.path.getsize(tmp_path / "c" / f) for f in os.listdir(tmp_path / "c")) <= 1 << 20
    assert 0 < len(small["rows"]) < bench.DUMP_ROWS
    _check_rows(small, indptr, indices, data, neumann)


@pytest.mark.parametrize("args,word", [(["--steps", "0"], "--steps"), (["--impl", "reference", "--dump-outputs", "d"], "--dump-outputs")])
def test_bad_arguments_are_rejected(args, word):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and word in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["gls", "ls"])
def test_dump_is_what_interpolate_returns(tmp_path, method):
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tet7", "--method", method, "--steps", "2",
                        "--warmup", "1", "--also", "", "--no-configs", "--no-cpu", "--dump-outputs", str(d)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    import ninpol_b200
    mesh = bench.make_mesh("tet", 7)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    W, nv = I.interpolate(bench.VARIABLE, method)
    out = _load(d)
    assert len(out["rows"]) == W.shape[0]           # 512 nodes: every row is in the sample
    _check_rows(out, W.indptr, W.indices, W.data, np.asarray(nv))
    assert out["totals"][:3].tolist() == [W.shape[0], W.shape[1], W.nnz]
