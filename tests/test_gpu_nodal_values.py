"""Interpolator.nodal_values: W @ values on the GPU from the resident weights (K5, csrc/k5_apply.cu).

Bar: bit-identical to scipy's `W @ values` (the same sums in the same order, each product and addition rounded on its
own), NaN positions included, for all three methods and every supported shape and dtype of `values`."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from helpers import GOLDEN, ROOT
from test_gpu_parity import CASES, CASES_2D

pytestmark = pytest.mark.gpu


def same_bits(a, b):
    """Equal shape and dtype, NaN at the same positions and every other element equal bit for bit (so -0.0 != +0.0)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64)))


def value_sets(n_elems, seed=0):
    rng = np.random.default_rng(seed)
    special = rng.standard_normal(n_elems) * 10.0 ** rng.integers(-9, 10, n_elems)
    pos = rng.choice(n_elems, size=min(n_elems, 8), replace=False)
    special[pos] = np.resize([np.nan, np.inf, -np.inf, -0.0], len(pos))
    return {
        "special": special,
        "k3": rng.standard_normal((n_elems, 3)),
        "k7": rng.standard_normal((n_elems, 7)) * 1e5,
        "float32": rng.standard_normal((n_elems, 2)).astype(np.float32),
        "fortran": np.asfortranarray(rng.standard_normal((n_elems, 4))),
        "strided": rng.standard_normal((2 * n_elems, 6))[::2, ::2],
    }


def own_values(I, variable="u"):
    return np.asarray(I._rows["cells"][I.variable_to_index["cells"][variable]])[:I.grid.n_elems]


def check_interpolator(I, O=None, methods=("idw", "ls", "gls"), seed=0):
    """For each method: a first nodal_values (weights computed without any download), then interpolate(), then every
    value set with the weights resident; all bit-equal to W @ values (and, for IDW / LS, to the oracle's W @ values)."""
    sets = value_sets(I.grid.n_elems, seed)
    for method in methods:
        y0 = I.nodal_values("u", method)
        assert I.last_timings["nodal_weights_reused"] is False
        W, _ = I.interpolate("u", method)
        u = own_values(I)
        assert same_bits(y0, W @ u), method
        Wo = O.interpolate("u", method)[0] if (O is not None and method != "gls") else None
        if Wo is not None:
            assert same_bits(y0, Wo @ u), method
        for name, vals in sets.items():
            y = I.nodal_values("u", method, vals)
            assert I.last_timings["nodal_weights_reused"] is True, (method, name)
            want = W @ vals
            assert same_bits(y, want), (method, name)
            if Wo is not None:
                assert same_bits(y, Wo @ vals), (method, name)


def _pair(kind, n, kw, **opts):
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case(kind, n, **kw)
    I = ninpol_b200.Interpolator(**opts)
    I.load_mesh(mesh_obj=mesh)
    return I, oracle.OracleInterpolator().load_mesh(mesh), mesh


@pytest.mark.parametrize("kind,n,kw", CASES + CASES_2D)
def test_bit_equal_to_scipy_product(kind, n, kw):
    I, O, _ = _pair(kind, n, kw)
    check_interpolator(I, O)


SUBSET = [("tet", 9, {"scramble": True}), ("mixed", 8, {"a": 2, "b": 4}), ("hex", 6, {"perturb": 0.2}), ("quad2d", 6, {})]


@pytest.mark.parametrize("opts", [{"stream_chunks": 0}, {"pinned_outputs": False, "pin_inputs": False}],
                         ids=["two_pass", "pageable"])
@pytest.mark.parametrize("kind,n,kw", SUBSET)
def test_bit_equal_in_other_configurations(kind, n, kw, opts):
    I, O, _ = _pair(kind, n, kw, **opts)
    check_interpolator(I, O)


def test_exact_zero_weights_fill_the_rows_inside_apply():
    """LS on an unperturbed hex box has exact-zero weights: the plan is voided, the two-pass count leaves the rows
    unwritten and npb_apply writes them before the product."""
    I, O, _ = _pair("hex", 10, {})
    y = I.nodal_values("u", "ls")
    assert I._ctx.timing("k3_fill") >= 0.0        # only npb_apply fills on this path
    W, _ = I.interpolate("u", "ls")
    assert W.nnz < int(I._ctx.scalar("len_esup"))
    Wo = O.interpolate("u", "ls")[0]
    assert same_bits(y, W @ own_values(I)) and same_bits(y, Wo @ own_values(I))
    I2, _, _ = _pair("hex", 10, {})
    check_interpolator(I2, O, methods=("ls",))


def test_resident_weights_are_reused_and_recomputed_when_inputs_change():
    import ninpol_b200
    from ninpol_b200 import meshgen
    rng = np.random.default_rng(3)
    mesh = meshgen.make_case("tet", 8)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    n_elems = I.grid.n_elems

    def fresh(method, vals=None):
        y = I.nodal_values("u", method, vals)
        reused = I.last_timings["nodal_weights_reused"]
        W, _ = I.interpolate("u", method)
        assert same_bits(y, W @ (own_values(I) if vals is None else vals)), method
        return reused, W

    reused, W_old = fresh("gls")
    assert not reused
    # a second call with new values: only the upload, one kernel and the download
    u2 = rng.standard_normal(n_elems)
    n0 = I._ctx.launch_count()
    y2 = I.nodal_values("u", "gls", u2)
    assert I._ctx.launch_count() - n0 == 1 and I.last_timings["nodal_weights_reused"] is True
    assert same_bits(y2, W_old @ u2)
    for key in ("nodal_h2d_ms", "nodal_apply_ms", "nodal_d2h_ms"):
        assert I.last_timings[key] >= 0.0

    # new permeability through the cells_data setter
    cd = np.array(I.cells_data)
    k = I.variable_to_index["cells"]["permeability"]
    cd[k, :9 * n_elems] = meshgen.random_spd_permeability(n_elems, seed=77).ravel()
    I.cells_data = cd
    reused, W_new = fresh("gls", u2)
    assert not reused and not np.array_equal(W_new.data, W_old.data)

    # invalidate_inputs, the dense plug-in path, another method
    I.invalidate_inputs()
    assert not fresh("gls", u2)[0]
    n, mx = I.grid.n_points, I.grid.MX_ELEMENTS_PER_POINT
    I.gls.prepare(I.grid, I._rows["cells"], I._rows["points"], None, I.variable_to_index, "u", np.array([], dtype=np.int64),
                  np.zeros((n, mx)), np.zeros(n))
    assert not fresh("gls", u2)[0]
    assert not fresh("idw", u2)[0]
    assert not fresh("gls", u2)[0]

    # load_mesh of another mesh
    I.load_mesh(mesh_obj=meshgen.make_case("hex", 7))
    assert not fresh("ls")[0]

    # interpolate after nodal_values: identical to a fresh Interpolator's
    I.nodal_values("u", "idw")
    I2 = ninpol_b200.Interpolator()
    I2.load_mesh(mesh_obj=meshgen.make_case("hex", 7))
    for method in ("idw", "ls", "gls"):
        I.nodal_values("u", method, rng.standard_normal((I.grid.n_elems, 3)))
        W, nv = I.interpolate("u", method)
        W2, nv2 = I2.interpolate("u", method)
        assert np.array_equal(W.indptr, W2.indptr) and np.array_equal(W.indices, W2.indices)
        assert same_bits(W.data, W2.data) and same_bits(nv, nv2)


def test_apply_refuses_when_no_weights_are_resident():
    import ninpol_b200
    from ninpol_b200 import _capi, meshgen
    mesh = meshgen.make_case("tet", 5)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    x = np.ones(I.grid.n_elems)
    out = np.full(I.grid.n_points, 7.0)
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply("idw", x, out)                 # before any interpolate
    I.interpolate("u", "idw")
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply("ls", x, out)                  # weights of another method
    I._ctx.apply("idw", x, out)
    assert np.allclose(out[np.asarray(I.grid.boundary_points) == 0], 1.0)
    out[:] = 7.0
    I._ctx.set_point_flags(np.asarray(mesh.point_data["neumann_flag_u"]))
    with pytest.raises(_capi.NinpolB200Error, match="no weights"):
        I._ctx.apply("idw", x, out)                 # the flags changed: the CSR on the device is stale
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
    assert _raised(lambda: I.nodal_values("u", "idw")) == _raised(lambda: I.interpolate("u", "idw"))
    assert _raised(lambda: I.nodal_values("u", "idw"))[0] is ValueError
    mesh = meshgen.make_case("tet", 4)
    n_cells = len(mesh.cells[0].data)
    mesh.cell_data["vel"] = [np.random.default_rng(1).standard_normal((n_cells, 3))]
    mesh.point_data["neumann_flag_vel"] = mesh.point_data["neumann_flag_u"]
    mesh.point_data["neumann_vel"] = mesh.point_data["neumann_u"]
    I.load_mesh(mesh_obj=mesh)
    for args in (("u", "lpew3"), ("nope", "idw")):
        got = _raised(lambda: I.nodal_values(*args))
        assert got is not None and got == _raised(lambda: I.interpolate(*args)), args
    n_elems, n_points = I.grid.n_elems, I.grid.n_points
    with pytest.raises(ValueError):
        I.nodal_values("u", "idw", np.ones(n_elems + 1))
    with pytest.raises(ValueError):
        I.nodal_values("u", "idw", np.ones((n_elems, 2, 2)))
    with pytest.raises(ValueError):
        I.nodal_values("u", "idw", np.float64(1.0))
    with pytest.raises(TypeError):
        I.nodal_values("u", "idw", np.ones(n_elems, dtype=np.complex128))
    empty = I.nodal_values("u", "idw", np.ones((n_elems, 0)))
    assert empty.shape == (n_points, 0) and empty.dtype == np.float64
    # a vector variable: accepted here (interpolate refuses it); same weights as "u" since its flags are the same
    vel = np.asarray(mesh.cell_data["vel"][0])
    for method in ("idw", "ls", "gls"):
        y = I.nodal_values("vel", method)
        assert y.shape == (n_points, 3)
        W, _ = I.interpolate("u", method)
        assert same_bits(y, W @ vel), method
    # missing per-variable inputs: KeyError, as interpolate
    del mesh.point_data["neumann_flag_u"]
    del mesh.cell_data["permeability"]
    I2 = ninpol_b200.Interpolator()
    I2.load_mesh(mesh_obj=mesh)
    for method in ("idw", "gls"):
        got = _raised(lambda: I2.nodal_values("u", method))
        assert got is not None and got[0] is KeyError and got == _raised(lambda: I2.interpolate("u", method)), method
    got = _raised(lambda: I2.nodal_values("vel", "gls"))
    assert got is not None and got[0] is KeyError


def test_reproduces_published_accuracy():
    """accuracy.yaml hexa rows (QUAD, FAN, ALH; n = 4, 8, 16) with the product taken on the GPU."""
    import json
    sys.path.insert(0, GOLDEN)
    import make_golden
    import ninpol_b200
    table = json.load(open(os.path.join(GOLDEN, "accuracy_hexa.json")))["table"]
    for case in ("QUAD", "FAN", "ALH"):
        for n_i, n in enumerate((4, 8, 16)):
            mesh, sol = make_golden.analytic_mesh(case, n)
            I = ninpol_b200.Interpolator()
            I.load_mesh(mesh_obj=mesh)
            for method in ("gls", "idw", "ls"):
                W = types.SimpleNamespace(dot=lambda u, m=method: I.nodal_values(case, m))
                err = make_golden.interior_l2(W, mesh, sol, case, I.grid.boundary_points)
                pub = table[case][method]["published"][n_i]
                assert abs(err - pub) <= 1e-11 * max(1.0, abs(pub)), (case, method, n, err, pub)


@pytest.mark.parametrize("method", ["gls", "idw"])
def test_at_size_kuhn_tets(method):
    """Kuhn tets n = 69 (about 2M cells, 343,000 nodes): the full result bit-equal to W @ u."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case("tet", 69))
    rng = np.random.default_rng(9)
    u = own_values(I)
    y0 = I.nodal_values("u", method)
    x3 = rng.standard_normal((I.grid.n_elems, 3))
    y3 = I.nodal_values("u", method, x3)
    W, _ = I.interpolate("u", method)
    assert same_bits(y0, W @ u) and same_bits(y3, W @ x3)


GUARD_SCRIPT = """
import numpy as np, ninpol_b200
from ninpol_b200 import meshgen
damaged = 0
for kind, n, method in (("tet", 9, "gls"), ("mixed", 8, "idw"), ("hex", 10, "ls")):
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case(kind, n))
    rng = np.random.default_rng(0)
    for k in (1, 3, 7):
        x = rng.standard_normal(I.grid.n_elems) if k == 1 else rng.standard_normal((I.grid.n_elems, k))
        y = I.nodal_values("u", method, x)
        W, _ = I.interpolate("u", method)
        assert np.array_equal(y, W @ x, equal_nan=True), (kind, method, k)
        I.invalidate_inputs()           # the next call computes the weights again (hex / ls: fill inside apply)
    nb, nd = I._ctx.check_guards()
    assert nb > 0
    damaged += nd
print("nodal guards damaged", damaged)
"""


def test_no_write_past_buffers_with_guards():
    env = dict(os.environ, NPB_DEBUG_GUARDS="1")
    r = subprocess.run([sys.executable, "-c", GUARD_SCRIPT], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "nodal guards damaged 0" in r.stdout


def test_two_gpu_nodal_values_match_full_product():
    from ninpol_b200 import _capi
    if _capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tools", "check_multi_gpu_nodal.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MISMATCH" not in r.stdout and " OK" in r.stdout
