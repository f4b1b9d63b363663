"""Interpolator.nodal_adjoint: W.T @ values on the GPU from the resident weights (K5, csrc/k5_apply.cu).

Bar: bit-identical to scipy's `W.T @ values` (csc_matvec(s) on the free CSC view: for every element the products of its
entries in ascending node order, each product and addition rounded on its own), NaN positions included, for all three
methods and every supported shape and dtype of `values`."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from helpers import ROOT
from test_gpu_nodal_values import SUBSET, _pair, same_bits, value_sets
from test_gpu_parity import CASES, CASES_2D

pytestmark = pytest.mark.gpu


def check_interpolator(I, O=None, methods=("idw", "ls", "gls"), seed=0):
    """For each method: a first nodal_adjoint on fresh inputs (weights computed by the adjoint itself, nothing
    downloaded), then interpolate(), then every value set with the weights resident; all bit-equal to W.T @ values (and,
    for IDW / LS, to the oracle's Wo.T @ values)."""
    sets = value_sets(I.grid.n_points, seed)
    first = sets["special"]
    for method in methods:
        z0 = I.nodal_adjoint("u", method, first)
        assert I.last_timings["adjoint_weights_reused"] is False
        assert I.last_timings["adjoint_map_ms"] > 0.0
        W, _ = I.interpolate("u", method)
        assert same_bits(z0, W.T @ first), method
        Wo = O.interpolate("u", method)[0] if (O is not None and method != "gls") else None
        if Wo is not None:
            assert same_bits(z0, Wo.T @ first), method
        for name, vals in sets.items():
            z = I.nodal_adjoint("u", method, vals)
            assert I.last_timings["adjoint_weights_reused"] is True, (method, name)
            assert same_bits(z, W.T @ vals), (method, name)
            if Wo is not None:
                assert same_bits(z, Wo.T @ vals), (method, name)


@pytest.mark.parametrize("kind,n,kw", CASES + CASES_2D)
def test_bit_equal_to_scipy_transposed_product(kind, n, kw):
    I, O, _ = _pair(kind, n, kw)
    check_interpolator(I, O)


@pytest.mark.parametrize("opts", [{"stream_chunks": 0}, {"pinned_outputs": False, "pin_inputs": False}],
                         ids=["two_pass", "pageable"])
@pytest.mark.parametrize("kind,n,kw", SUBSET)
def test_bit_equal_in_other_configurations(kind, n, kw, opts):
    I, O, _ = _pair(kind, n, kw, **opts)
    check_interpolator(I, O)


def test_exact_zero_weights_fill_the_rows_and_get_no_slot():
    """LS on an unperturbed hex box has exact-zero weights: the plan is voided, the two-pass count leaves the rows
    unwritten and npb_apply_transpose writes them, then maps only the entries that survived the elimination."""
    I, O, _ = _pair("hex", 10, {})
    y = value_sets(I.grid.n_points, 4)["special"]
    z = I.nodal_adjoint("u", "ls", y)
    assert I._ctx.timing("k3_fill") >= 0.0        # only the adjoint fills on this path
    W, _ = I.interpolate("u", "ls")
    assert W.nnz < int(I._ctx.scalar("len_esup"))
    Wo = O.interpolate("u", "ls")[0]
    assert same_bits(z, W.T @ y) and same_bits(z, Wo.T @ y)
    I2, _, _ = _pair("hex", 10, {})
    check_interpolator(I2, O, methods=("ls",))


def test_map_and_weights_are_reused_and_rebuilt_when_inputs_change():
    import ninpol_b200
    from ninpol_b200 import meshgen
    rng = np.random.default_rng(3)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case("tet", 8))
    n_elems, n_points = I.grid.n_elems, I.grid.n_points
    y = rng.standard_normal(n_points)
    x = rng.standard_normal(n_elems)

    def launches(fn):
        n0 = I._ctx.launch_count()
        out = fn()
        return I._ctx.launch_count() - n0, out

    # the first adjoint after nodal_values: the weights are reused, the map is built, then the product
    I.nodal_values("u", "gls", x)
    n, z = launches(lambda: I.nodal_adjoint("u", "gls", y))
    assert n == 2 and I.last_timings["adjoint_weights_reused"] is True and I.last_timings["adjoint_map_ms"] > 0.0
    # weights and map reused: one launch
    y2 = rng.standard_normal((n_points, 3))
    n, z2 = launches(lambda: I.nodal_adjoint("u", "gls", y2))
    assert n == 1 and I.last_timings["adjoint_weights_reused"] is True and I.last_timings["adjoint_map_ms"] == 0.0
    for key in ("adjoint_h2d_ms", "adjoint_apply_ms", "adjoint_d2h_ms"):
        assert I.last_timings[key] >= 0.0
    # nodal_values after nodal_adjoint recomputes nothing
    n, _ = launches(lambda: I.nodal_values("u", "gls", x))
    assert n == 1 and I.last_timings["nodal_weights_reused"] is True
    W_old, _ = I.interpolate("u", "gls")
    assert same_bits(z, W_old.T @ y) and same_bits(z2, W_old.T @ y2)

    def fresh(method):
        z = I.nodal_adjoint("u", method, y)
        reused = I.last_timings["adjoint_weights_reused"]
        W, _ = I.interpolate("u", method)
        assert same_bits(z, W.T @ y), method
        return reused, W

    fresh("gls")
    # new permeability through the cells_data setter
    cd = np.array(I.cells_data)
    k = I.variable_to_index["cells"]["permeability"]
    cd[k, :9 * n_elems] = meshgen.random_spd_permeability(n_elems, seed=77).ravel()
    I.cells_data = cd
    reused, W_new = fresh("gls")
    assert not reused and not np.array_equal(W_new.data, W_old.data)
    # invalidate_inputs, the dense plug-in path, another method
    I.invalidate_inputs()
    assert not fresh("gls")[0]
    mx = I.grid.MX_ELEMENTS_PER_POINT
    I.gls.prepare(I.grid, I._rows["cells"], I._rows["points"], None, I.variable_to_index, "u", np.array([], dtype=np.int64),
                  np.zeros((n_points, mx)), np.zeros(n_points))
    assert not fresh("gls")[0]
    assert not fresh("idw")[0]
    assert not fresh("gls")[0]
    # load_mesh of another mesh (another element count and node stride: hex, spe = 8)
    I.load_mesh(mesh_obj=meshgen.make_case("hex", 7))
    n_points = I.grid.n_points
    y = rng.standard_normal(n_points)
    assert not fresh("ls")[0]


def test_apply_transpose_refuses_when_no_weights_are_resident():
    import ninpol_b200
    from ninpol_b200 import _capi, meshgen
    mesh = meshgen.make_case("tet", 5)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    y = np.ones(I.grid.n_points)
    out = np.full(I.grid.n_elems, 7.0)
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply_transpose("idw", y, out)       # before any interpolate
    assert np.all(out == 7.0)
    W, _ = I.interpolate("u", "idw")
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply_transpose("ls", y, out)        # weights of another method
    assert np.all(out == 7.0)
    I._ctx.apply_transpose("idw", y, out)
    assert same_bits(out, W.T @ y)
    out[:] = 7.0
    I._ctx.set_point_flags(np.asarray(mesh.point_data["neumann_flag_u"]))
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply_transpose("idw", y, out)       # the flags changed: the CSR on the device is stale
    assert np.all(out == 7.0)


def _raised(fn):
    try:
        fn()
    except Exception as e:       # noqa: BLE001 - the exception itself is compared
        return type(e), str(e)
    return None


def test_errors_match_interpolate():
    import ninpol_b200
    from ninpol_b200 import meshgen
    I = ninpol_b200.Interpolator()
    assert _raised(lambda: I.nodal_adjoint("u", "idw", np.ones(3))) == _raised(lambda: I.interpolate("u", "idw"))
    assert _raised(lambda: I.nodal_adjoint("u", "idw", np.ones(3)))[0] is ValueError
    mesh = meshgen.make_case("tet", 4)
    I.load_mesh(mesh_obj=mesh)
    n_elems, n_points = I.grid.n_elems, I.grid.n_points
    y = np.ones(n_points)
    for args in (("u", "lpew3"), ("nope", "idw")):
        got = _raised(lambda: I.nodal_adjoint(*args, y))
        assert got is not None and got == _raised(lambda: I.interpolate(*args)), args
    with pytest.raises(TypeError):
        I.nodal_adjoint("u", "idw")                 # values are required
    with pytest.raises(ValueError):
        I.nodal_adjoint("u", "idw", np.ones(n_elems))
    with pytest.raises(ValueError):
        I.nodal_adjoint("u", "idw", np.ones(n_points + 1))
    with pytest.raises(ValueError):
        I.nodal_adjoint("u", "idw", np.ones((n_points, 2, 2)))
    with pytest.raises(ValueError):
        I.nodal_adjoint("u", "idw", np.float64(1.0))
    with pytest.raises(TypeError):
        I.nodal_adjoint("u", "idw", np.ones(n_points, dtype=np.complex128))
    empty = I.nodal_adjoint("u", "idw", np.ones((n_points, 0)))
    assert empty.shape == (n_elems, 0) and empty.dtype == np.float64
    # more than one GPU: refused before anything is staged or launched
    comm = I.comm
    I.comm = types.SimpleNamespace(world=2, rank=0, local_rank=0)
    n0 = I._ctx.launch_count()
    with pytest.raises(NotImplementedError, match="single-GPU"):
        I.nodal_adjoint("u", "idw", y)
    assert I._ctx.launch_count() == n0
    I.comm = comm
    # missing per-variable inputs: KeyError, as interpolate
    del mesh.point_data["neumann_flag_u"]
    del mesh.cell_data["permeability"]
    I2 = ninpol_b200.Interpolator()
    I2.load_mesh(mesh_obj=mesh)
    for method in ("idw", "gls"):
        got = _raised(lambda: I2.nodal_adjoint("u", method, y))
        assert got is not None and got[0] is KeyError and got == _raised(lambda: I2.interpolate("u", method)), method


@pytest.mark.parametrize("method", ["gls", "idw"])
def test_at_size_kuhn_tets(method):
    """Kuhn tets n = 69 (about 2M cells, 343,000 nodes): the full result bit-equal to W.T @ y."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case("tet", 69))
    rng = np.random.default_rng(9)
    y1 = rng.standard_normal(I.grid.n_points)
    z1 = I.nodal_adjoint("u", method, y1)
    y3 = rng.standard_normal((I.grid.n_points, 3))
    z3 = I.nodal_adjoint("u", method, y3)
    W, _ = I.interpolate("u", method)
    assert same_bits(z1, W.T @ y1) and same_bits(z3, W.T @ y3)


GUARD_SCRIPT = """
import numpy as np, ninpol_b200
from ninpol_b200 import meshgen
damaged = 0
for kind, n, method in (("tet", 9, "gls"), ("mixed", 8, "idw"), ("hex", 10, "ls")):
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case(kind, n))
    rng = np.random.default_rng(0)
    for k in (1, 3, 7):
        y = rng.standard_normal(I.grid.n_points) if k == 1 else rng.standard_normal((I.grid.n_points, k))
        z = I.nodal_adjoint("u", method, y)
        W, _ = I.interpolate("u", method)
        assert np.array_equal(z, W.T @ y, equal_nan=True), (kind, method, k)
        I.invalidate_inputs()           # the next call computes the weights again (hex / ls: fill inside the call)
    nb, nd = I._ctx.check_guards()
    assert nb > 0
    damaged += nd
print("adjoint guards damaged", damaged)
"""


def test_no_write_past_buffers_with_guards():
    env = dict(os.environ, NPB_DEBUG_GUARDS="1")
    r = subprocess.run([sys.executable, "-c", GUARD_SCRIPT], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "adjoint guards damaged 0" in r.stdout
