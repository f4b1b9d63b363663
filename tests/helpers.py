import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GRID_ARRAYS = ("esup", "esup_ptr", "psup", "psup_ptr", "esuel", "infael", "inpofa", "fsup", "fsup_ptr", "esuf", "esuf_ptr",
               "boundary_faces", "boundary_points", "centroids", "faces_centers", "normal_faces", "faces_areas")
GRID_SCALARS = ("n_elems", "n_points", "n_faces", "MX_ELEMENTS_PER_POINT", "MX_POINTS_PER_POINT", "MX_ELEMENTS_PER_FACE",
                "MX_FACES_PER_POINT")
GOLDEN_CASES = ("tet_n4", "hex_n4", "hex_n3_perturbed", "mixed_n6")
GLS_TOL = 1e-12   # BASELINE.json north_star: <= 1e-12 relative weight error in FP64


def digest(a):
    """sha256 of an array's shape and values in a canonical form (integers as int64, floats as float64 with -0.0 as +0.0
    and one NaN): two arrays have equal digests exactly when they have the same shape and np.array_equal(a, b,
    equal_nan=True) holds."""
    import hashlib
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = a.astype(np.float64) + 0.0
        a = np.where(np.isnan(a), np.nan, a)
    else:
        a = a.astype(np.int64)
    h = hashlib.sha256(str(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def load_golden(name):
    sys.path.insert(0, GOLDEN)
    import make_golden
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    return make_golden.arrays_to_mesh(d), d


def row_normwise_error(W, indptr, data_ref):
    """max |w - w_ref| / max_row |w_ref| (SURVEY.md 8d parity metric); structures must be equal."""
    if len(data_ref) == 0:
        return 0.0
    rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
    scale = np.zeros(len(indptr) - 1)
    np.maximum.at(scale, rows, np.abs(np.nan_to_num(data_ref)))
    scale[scale == 0] = 1.0
    return float(np.nanmax(np.abs(W.data - data_ref) / scale[rows]))


def check_against_golden(I, d, gls_tol=GLS_TOL, exact_gls=False):
    """I: anything with .grid and .interpolate (oracle, reference or the CUDA Interpolator)."""
    g = I.grid
    for s, v in zip(GRID_SCALARS, d["grid_scalars"]):
        assert getattr(g, s) == int(v), s
    for a in GRID_ARRAYS:
        got, want = np.asarray(getattr(g, a)), d["grid_" + a]
        assert got.shape == want.shape and got.dtype == want.dtype, a
        assert np.array_equal(got, want), a
    for method in ("idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        assert np.array_equal(W.indptr, d[method + "_indptr"]), method
        assert np.array_equal(W.indices, d[method + "_indices"]), method
        if method == "gls" and not exact_gls:
            assert np.array_equal(np.isnan(W.data), np.isnan(d["gls_data"]))
            assert row_normwise_error(W, W.indptr, d["gls_data"]) <= gls_tol
            scale = max(1.0, float(np.max(np.abs(d["gls_neumann"]))))
            assert np.max(np.abs(np.asarray(nv) - d["gls_neumann"])) <= gls_tol * scale
        else:
            assert np.array_equal(W.data, d[method + "_data"], equal_nan=True), method
            assert np.array_equal(np.asarray(nv), d[method + "_neumann"]), method


def load_reference_outputs(kind, n, kw):
    """(mesh, digests, GLS row sample) of the reference's outputs on meshgen.make_case(kind, n, **kw), as stored by
    tests/golden/make_golden.py --digests."""
    import json
    sys.path.insert(0, GOLDEN)
    import make_golden
    from ninpol_b200 import meshgen
    key = make_golden.case_key(kind, n, kw)
    with open(make_golden.DIGESTS) as f:
        d = json.load(f)["at_size"][key]
    mesh = meshgen.make_case(kind, n, **kw)
    assert make_golden.mesh_digest(mesh) == d["mesh"], "the mesh generator no longer makes the stored mesh"
    return mesh, d, dict(np.load(make_golden.gls_sample_path(key)))


def check_against_reference_outputs(I, d, sample):
    """Every Grid array, the IDW / LS CSR and neumann vectors and the GLS structure bit for bit against the stored
    digests.  Returns the GLS result and, for the stored sample of rows, (row pointer, CUDA values)."""
    g = I.grid
    for s in GRID_SCALARS:
        assert getattr(g, s) == d["grid_scalars"][s], s
    for a in GRID_ARRAYS:
        assert digest(getattr(g, a)) == d["grid"][a], a
    for method in ("idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        want = d[method]
        assert digest(W.indptr) == want["indptr"] and digest(W.indices) == want["indices"], method
        assert digest(np.isnan(W.data)) == want["nan"], method
        if method != "gls":
            assert digest(W.data) == want["data"] and digest(nv) == want["neumann"], method
    nodes = sample["nodes"]
    ptr = np.concatenate([[0], np.cumsum(sample["row_nnz"])])
    assert np.array_equal(np.diff(W.indptr)[nodes], sample["row_nnz"])
    take = np.concatenate([np.arange(W.indptr[p], W.indptr[p + 1]) for p in nodes])
    assert np.array_equal(W.indices[take], sample["indices"])
    return W, np.asarray(nv), ptr, W.data[take]
