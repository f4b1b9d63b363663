"""Parity of the CUDA path (through the C ABI, via ninpol_b200.Interpolator) against the oracle.

Bar (BASELINE.json north_star, SURVEY.md 8d): bit-exact for every connectivity / geometry array, the
CSR structure of all three methods and the IDW / LS values (NaN positions included); GLS weights and
neumann within 1e-12, measured row-normwise (|w - w_ref| / max_row |w_ref|).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GRID_ARRAYS = ("inpoel", "element_types", "esup", "esup_ptr", "psup", "psup_ptr", "esuel", "infael", "inpofa", "fsup",
               "fsup_ptr", "esuf", "esuf_ptr", "boundary_faces", "boundary_points", "point_coords", "centroids",
               "faces_centers", "normal_faces", "faces_areas")
GRID_SCALARS = ("n_elems", "n_points", "n_faces", "MX_ELEMENTS_PER_POINT", "MX_POINTS_PER_POINT",
                "MX_ELEMENTS_PER_FACE", "MX_FACES_PER_POINT")
GLS_TOL = 1e-12

CASES = [("tet", 9, {"scramble": True}), ("mixed", 10, {"a": 2, "b": 5, "scramble": True}), ("tet", 7, {}), ("hex", 8, {}), ("mixed", 8, {"a": 2, "b": 4}), ("tet", 14, {}), ("hex", 20, {}),
         ("hex", 6, {"perturb": 0.2}), ("mixed", 12, {"a": 3, "b": 6}), ("tet", 3, {}), ("hex", 1, {}), ("tet", 1, {})]


CASES_2D = [("quad2d", 6, {}), ("tri2d", 6, {"perturb": 0.2}), ("quad2d", 9, {"perturb": 0.2}), ("tri2d", 12, {})]


def _pair(kind, n, kw):
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case(kind, n, **kw)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    return I, O


def gls_errors(W, Wo):
    rows = np.repeat(np.arange(W.shape[0]), np.diff(W.indptr))
    scale = np.zeros(W.shape[0])
    np.maximum.at(scale, rows, np.abs(Wo.data))
    scale[scale == 0] = 1.0
    return float(np.max(np.abs(W.data - Wo.data) / scale[rows])) if W.nnz else 0.0


@pytest.mark.parametrize("kind,n,kw", CASES)
def test_connectivity_and_geometry_bit_exact(kind, n, kw):
    I, O = _pair(kind, n, kw)
    for s in GRID_SCALARS:
        assert getattr(I.grid, s) == getattr(O.grid, s), s
    for name in GRID_ARRAYS:
        a, b = np.asarray(getattr(I.grid, name)), np.asarray(getattr(O.grid, name))
        assert a.dtype == b.dtype and a.shape == b.shape, name
        assert np.array_equal(a, b), name


@pytest.mark.parametrize("kind,n,kw", CASES)
@pytest.mark.parametrize("method", ["idw", "ls"])
def test_idw_ls_bit_exact(kind, n, kw, method):
    I, O = _pair(kind, n, kw)
    W, nv = I.interpolate("u", method)
    Wo, nvo = O.interpolate("u", method)
    assert W.shape == Wo.shape and W.indptr.dtype == np.int32 and W.indices.dtype == np.int32
    assert np.array_equal(W.indptr, Wo.indptr)
    assert np.array_equal(W.indices, Wo.indices)
    assert np.array_equal(W.data, Wo.data, equal_nan=True)
    assert np.array_equal(nv, nvo)


@pytest.mark.parametrize("kind,n,kw", CASES)
def test_gls_within_tolerance(kind, n, kw):
    I, O = _pair(kind, n, kw)
    W, nv = I.interpolate("u", "gls")
    Wo, nvo = O.interpolate("u", "gls")
    assert np.array_equal(W.indptr, Wo.indptr)
    assert np.array_equal(W.indices, Wo.indices)
    assert np.array_equal(np.isnan(W.data), np.isnan(Wo.data))
    assert gls_errors(W, Wo) <= GLS_TOL
    scale = max(1.0, float(np.max(np.abs(nvo))))
    assert np.max(np.abs(nv - nvo)) <= GLS_TOL * scale


def test_gls_small_spacing_tolerance():
    """cond(M) grows like 1/h: the 50M-tet mesh has h = 0.005 (SURVEY.md 7.4)."""
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case("tet", 8)
    mesh.points = mesh.points * 0.04
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    W, nv = I.interpolate("u", "gls")
    Wo, nvo = O.interpolate("u", "gls")
    assert np.array_equal(W.indices, Wo.indices)
    assert gls_errors(W, Wo) <= GLS_TOL


def test_row_sums_and_linear_exactness():
    """Size-independent properties (SURVEY.md 4): processed rows sum to 1; LS and GLS with
    homogeneous K reproduce a linear field at interior nodes."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case("tet", 16)
    K = np.array([[1.0, 0.5, 0.0], [0.5, 1.0, 0.5], [0.0, 0.5, 1.0]]).reshape(1, 9)
    mesh.cell_data["permeability"] = [np.repeat(K, len(b), axis=0) for b in mesh.cells]
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    u = np.concatenate([c for c in mesh.cell_data["u"]])
    interior = np.asarray(I.grid.boundary_points) == 0
    exact = mesh.points.sum(axis=1)
    for method in ("ls", "gls"):
        W, _ = I.interpolate("u", method)
        rs = np.asarray(W.sum(axis=1)).ravel()
        assert np.allclose(rs[interior], 1.0, atol=1e-12)
        err = np.abs(W.dot(u) - exact)[interior].max()
        assert err < 1e-12, (method, err)


def test_errors_match_reference_conventions():
    import ninpol_b200
    from ninpol_b200 import meshgen
    I = ninpol_b200.Interpolator()
    with pytest.raises(ValueError):
        I.load_mesh()
    with pytest.raises(ValueError, match="Grid not initialized"):
        I.interpolate("u", "idw")
    mesh = meshgen.make_case("tet", 3)
    I.load_mesh(mesh_obj=mesh)
    with pytest.raises(ValueError, match="not supported"):
        I.interpolate("u", "lpew3")
    with pytest.raises(ValueError, match="not found in cells data"):
        I.interpolate("nope", "idw")
    with pytest.raises(ValueError, match="more than one dimension"):
        I.interpolate("permeability", "idw")
    with pytest.raises(ValueError):
        I.interpolate("u", "idw", target_points=np.arange(5, dtype=np.int64))
    del mesh.point_data["neumann_flag_u"]
    I2 = ninpol_b200.Interpolator()
    I2.load_mesh(mesh_obj=mesh)
    with pytest.raises(KeyError):
        I2.interpolate("u", "ls")
    assert list(I.supported_methods) == ["gls", "idw", "ls"]
    W, nv = I.interpolate("u", "idw", target_points=np.arange(I.grid.n_points, dtype=np.int64))
    assert W.shape == (I.grid.n_points, I.grid.n_elems)


@pytest.mark.parametrize("kind,n,kw", [("tet", 9, {}), ("hex", 10, {}), ("mixed", 8, {"a": 2, "b": 4})])
def test_fallback_kernels_agree(kind, n, kw, monkeypatch):
    """The general-purpose fallbacks (thread-per-node IDW/LS + two-pass emit; dense Householder GLS) must
    give the same answers as the fast paths: bit-exact for IDW/LS, <= 1e-12 for GLS."""
    monkeypatch.setenv("NPB_FORCE_SIMPLE_IDW_LS", "1")
    monkeypatch.setenv("NPB_FORCE_GLS_DENSE", "1")
    I, O = _pair(kind, n, kw)
    for method in ("idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        Wo, nvo = O.interpolate("u", method)
        assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices)
        if method == "gls":
            assert gls_errors(W, Wo) <= GLS_TOL
        else:
            assert np.array_equal(W.data, Wo.data, equal_nan=True)
            assert np.array_equal(nv, nvo)


@pytest.mark.parametrize("kind,n,kw", [("tet", 9, {"scramble": True}), ("hex", 8, {}), ("mixed", 10, {"a": 2, "b": 5})])
def test_gls_general_fronts_only(kind, n, kw, monkeypatch):
    """NPB_GLS_NO_LEAF=1 sends every front through the general warp-per-front loop (no lane-per-leaf
    phase): same tolerance against the oracle, and both paths agree with each other to rounding."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    I, O = _pair(kind, n, kw)
    W1, nv1 = I.interpolate("u", "gls")
    monkeypatch.setenv("NPB_GLS_NO_LEAF", "1")
    J = ninpol_b200.Interpolator()
    J.load_mesh(mesh_obj=meshgen.make_case(kind, n, **kw))
    W2, nv2 = J.interpolate("u", "gls")
    Wo, nvo = O.interpolate("u", "gls")
    assert np.array_equal(W2.indptr, Wo.indptr) and np.array_equal(W2.indices, Wo.indices)
    assert gls_errors(W2, Wo) <= GLS_TOL and gls_errors(W1, Wo) <= GLS_TOL
    assert gls_errors(W1, W2) <= GLS_TOL
    assert np.allclose(nv1, nv2, rtol=0, atol=1e-12)


@pytest.mark.parametrize("kind,n,kw", [("tet", 12, {}), ("hex", 8, {}), ("mixed", 10, {"a": 2, "b": 5}), ("tet", 2, {})])
@pytest.mark.parametrize("team", ["0,4", "1,16", "3,64"])
def test_gls_team_launch_is_bit_identical(kind, n, kw, team, monkeypatch):
    """NPB_GLS_TEAM forces the team launch (the warps of an SM in one CTA, loosely in step; taken by itself only for
    classes of uniform stars) for every class: the per-node arithmetic is the same, so the result equals the one-warp
    launch bit for bit - also with fewer nodes than warps in a team."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    monkeypatch.setenv("NPB_GLS_TEAM", "off")
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case(kind, n, **kw))
    W1, nv1 = I.interpolate("u", "gls")
    monkeypatch.setenv("NPB_GLS_TEAM", team)
    J = ninpol_b200.Interpolator()
    J.load_mesh(mesh_obj=meshgen.make_case(kind, n, **kw))
    W2, nv2 = J.interpolate("u", "gls")
    assert np.array_equal(W1.indptr, W2.indptr) and np.array_equal(W1.indices, W2.indices)
    assert np.array_equal(W1.data, W2.data, equal_nan=True) and np.array_equal(nv1, nv2, equal_nan=True)
    O = _pair(kind, n, kw)[1]
    Wo, nvo = O.interpolate("u", "gls")
    assert gls_errors(W2, Wo) <= GLS_TOL


@pytest.mark.parametrize("kind,n,kw,chunks", [("tet", 9, {"scramble": True}, 4), ("mixed", 10, {"a": 2, "b": 5}, 7),
                                              ("hex", 8, {}, 3), ("tet", 12, {}, 64), ("tet", 1, {}, 8)])
def test_streamed_pipeline_is_bit_identical(kind, n, kw, chunks):
    """The default path — npb_interpolate_run: optimistic row plan, node chunks, uploads / kernels / downloads on
    separate streams, pooled page-locked outputs — returns exactly what the plain count + fetch path returns, with
    the cell fields streamed in and with them resident, and with pageable inputs / outputs as well."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case(kind, n, **kw)
    I = ninpol_b200.Interpolator(pinned_outputs=False, pin_inputs=False, stream_chunks=0)   # plain two-pass path
    I.load_mesh(mesh_obj=mesh)
    J = ninpol_b200.Interpolator(stream_chunks=chunks)
    J.load_mesh(mesh_obj=mesh)
    P = ninpol_b200.Interpolator(pinned_outputs=False, pin_inputs=False, stream_chunks=chunks)   # pipeline, pageable host memory
    P.load_mesh(mesh_obj=mesh)
    J.min_chunk_nodes = P.min_chunk_nodes = 1        # really cut these small meshes into `chunks` pieces
    for method in ("gls", "idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        assert "streamed_ms" not in I.last_timings
        for K in (J, P):
            for resident in (False, True):
                if not resident:
                    K.invalidate_inputs()
                W2, nv2 = K.interpolate("u", method)
                assert W2.shape == W.shape and W2.indptr.dtype == np.int32 and W2.indices.dtype == np.int32
                assert np.array_equal(W.indptr, W2.indptr) and np.array_equal(W.indices, W2.indices)
                assert np.array_equal(W.data, W2.data, equal_nan=True)
                assert np.array_equal(nv, nv2, equal_nan=True)


def test_results_are_never_overwritten_while_referenced():
    """Drop-in semantics of the pooled page-locked outputs: a result the caller still holds survives later
    interpolate() calls untouched; a dropped one gives its buffers back (no growth in a steady loop)."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=meshgen.make_case("tet", 8))
    W1, n1 = I.interpolate("u", "gls")
    keep = (W1.indptr.copy(), W1.indices.copy(), W1.data.copy(), n1.copy())
    W2, n2 = I.interpolate("u", "idw")
    W3, n3 = I.interpolate("u", "ls")
    for a, b in zip((W1.indptr, W1.indices, W1.data, n1), keep):
        assert np.array_equal(a, b)
    assert not np.array_equal(W2.data, W3.data)
    del W2, n2, W3, n3
    for _ in range(4):
        W, nv = I.interpolate("u", "idw")
        del W, nv
    assert max(len(v) for v in I._pool._blocks.values()) <= 3
    assert np.array_equal(W1.data, keep[2])


def test_exact_zero_weights_void_the_plan_and_fall_back():
    """LS on an unperturbed hex box with Neumann hull nodes produces exact-zero weights (dropped by scipy's
    eliminate_zeros, interpolator.pyx:624): the planned single-pass result is discarded and the two-pass path
    answers — bit-identical to the oracle either way."""
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case("hex", 10)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    W, nv = I.interpolate("u", "ls")
    Wo, nvo = O.interpolate("u", "ls")
    assert W.nnz < int(I._ctx.scalar("len_esup"))
    assert "streamed_ms" not in I.last_timings or I.last_timings.get("k3_fill_ms", 0) >= 0
    assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices)
    assert np.array_equal(W.data, Wo.data, equal_nan=True)


def test_flag_truncation_matches_astype_int():
    """points_data[neumann_flag].astype(int) (idw.pyx:27, ls.pyx:28, gls.pyx:49): fractions truncate toward
    zero, NaN / inf cast to a non-zero integer.  The device does the cast from the float64 row."""
    import warnings
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case("tet", 6)
    rng = np.random.default_rng(5)
    vals = np.array([0.0, 0.5, -0.5, 0.999, 1.0, -1.0, 2.7, -3.2, np.nan, np.inf, -np.inf, 1e-300, -0.0])
    mesh.point_data["neumann_flag_u"] = vals[rng.integers(0, len(vals), len(mesh.points))]
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")        # numpy warns about the NaN -> int cast the reference performs
        O = oracle.OracleInterpolator().load_mesh(mesh)
        for method in ("idw", "ls"):
            W, nv = I.interpolate("u", method)
            Wo, nvo = O.interpolate("u", method)
            assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices)
            assert np.array_equal(W.data, Wo.data, equal_nan=True)


@pytest.mark.parametrize("kind,n,kw", CASES_2D)
def test_2d_meshes_bit_exact(kind, n, kw):
    """dim == 2: faces are edges (interpolator.pyx:296-298), 2-D normal branch (grid.pyx:787-806), LS
    z-degenerate fix-up (ls.pyx:79-80,105-106).  GLS is not compared in 2-D: its system has all-zero
    z-columns there and the reference returns whatever DGELS leaves for a singular matrix."""
    I, O = _pair(kind, n, kw)
    assert I.grid.dim == 2
    for s_ in GRID_SCALARS:
        assert getattr(I.grid, s_) == getattr(O.grid, s_), s_
    for name in GRID_ARRAYS:
        assert np.array_equal(np.asarray(getattr(I.grid, name)), np.asarray(getattr(O.grid, name))), name
    for method in ("idw", "ls"):
        W, nv = I.interpolate("u", method)
        Wo, nvo = O.interpolate("u", method)
        assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices)
        assert np.array_equal(W.data, Wo.data, equal_nan=True)
        assert np.array_equal(nv, nvo)


@pytest.mark.parametrize("kind,n,kw", [("tet", 6, {}), ("hex", 7, {}), ("mixed", 8, {"a": 2, "b": 4}), ("tri2d", 9, {}), ("tet", 24, {})])
def test_edge_structures_bit_exact(kind, n, kw):
    """build_edges=True: inedel / inpoed / n_edges (grid.pyx:527-580), hash-identity semantics included."""
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case(kind, n, **kw)
    I = ninpol_b200.Interpolator(build_edges=True)
    I.load_mesh(mesh_obj=mesh)
    O = oracle.OracleInterpolator().load_mesh(mesh, build_edges=True)
    assert I.grid.n_edges == O.grid.n_edges
    assert np.array_equal(np.asarray(I.grid.inedel), O.grid.inedel)
    assert np.array_equal(np.asarray(I.grid.inpoed), O.grid.inpoed)
    d = I.grid.get_data()
    assert d["esup"].shape == (I.grid.n_points, I.grid.MX_ELEMENTS_PER_POINT) and d["n_edges"] == O.grid.n_edges
    assert np.array_equal(d["psup"][d["psup"] >= 0], O.grid.psup)
    # without build_edges the reference leaves (0, 0) arrays (grid.pyx:132-133)
    J = ninpol_b200.Interpolator()
    J.load_mesh(mesh_obj=mesh)
    assert J.grid.inedel.shape == (0, 0) and J.grid.n_edges == 0


@pytest.mark.parametrize("kind,n,kw", [("tet", 8, {}), ("mixed", 8, {"a": 2, "b": 4}), ("hex", 6, {})])
def test_plugin_abi_prepare_fills_dense_weights(kind, n, kw):
    """The reference's plug-in contract (idw.pxd:19-24, ls.pxd:20-25, gls.pxd:22-27): the callables in
    `supported_methods` fill the caller's zeroed weights[n_points, MX_ELEMENTS_PER_POINT] and neumann_ws[n_points]
    (interpolator.pyx:645-664); column k of row p belongs to esup[esup_ptr[p] + k]."""
    I, O = _pair(kind, n, kw)
    g = I.grid
    assert list(I.supported_methods) == ["gls", "idw", "ls"]
    for method, prepare in I.supported_methods.items():
        weights = np.zeros((g.n_points, g.MX_ELEMENTS_PER_POINT))
        neumann_ws = np.zeros(g.n_points)
        prepare(g, I.cells_data, I.points_data, I.faces_data, I.variable_to_index, "u", np.array([], dtype=np.int64),
                weights, neumann_ws)
        wo, no = O.weights_dense("u", method)
        assert weights.shape == wo.shape
        if method == "gls":
            scale = np.maximum(np.abs(wo).max(axis=1), 1e-300)[:, None]
            assert np.max(np.abs(weights - wo) / scale) <= GLS_TOL
            assert np.max(np.abs(neumann_ws - no)) <= GLS_TOL * max(1.0, np.abs(no).max())
        else:
            assert np.array_equal(weights, wo, equal_nan=True), method
            assert np.array_equal(neumann_ws, no), method
    with pytest.raises(ValueError):
        I.supported_methods["idw"](g, I.cells_data, I.points_data, I.faces_data, I.variable_to_index, "u",
                                   np.array([], dtype=np.int64), np.zeros((3, 3)), np.zeros(g.n_points))


@pytest.mark.parametrize("kind,n,kw", CASES_2D)
def test_2d_gls_within_tolerance(kind, n, kw):
    """GLS on 2-D meshes (interpolator.pyx:296-330, gls.pyx:252-356).  With a full anisotropic K the z-columns are
    coupled through (K N)_z and the system has full rank, so the reference's DGELS result is well defined and
    compared here; an isotropic K leaves the constant-g_z mode undetermined (the reference then returns the
    leftovers of a rank-deficient DGELS) — that input has no defined answer and is not compared."""
    import oracle
    from at_size_checks import gls_verdict
    I, O = _pair(kind, n, kw)
    W, nv = I.interpolate("u", "gls")
    Wo, nvo = O.interpolate("u", "gls")
    assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices)
    g = O.grid
    flags = np.asarray(O.points["neumann_flag_u"]).astype(np.int64)

    def exact_row(p):
        M, _w, _n = oracle.gls_system_of(g, p, flags, O.cells["permeability"], O.cells["diff_mag"], O.points["neumann_u"])
        return oracle.gls_exact_row(M, int(g.esup_ptr[p + 1] - g.esup_ptr[p]), bool(flags[p]) and bool(g.boundary_points[p]))[0]

    # 2-D stars are nearly consistent systems (weights of +-75 at a Neumann corner): the same verdict as at BASELINE
    # sizes - within 1e-12 of the reference, or arbitrated against the exact solution (tests/at_size_checks.py)
    gls_verdict(Wo.indptr, W.data, Wo.data, exact_row, nearly_consistent=True)
    assert np.max(np.abs(nv - nvo)) <= 5e-12 * max(1.0, np.abs(nvo).max())


def test_out_of_range_node_ids_are_rejected_before_any_scatter():
    """A 1-based (or otherwise mis-indexed) mesh must fail with a Python exception, not fault the device."""
    import ninpol_b200
    from ninpol_b200 import meshgen
    from ninpol_b200._capi import NinpolB200Error
    mesh = meshgen.make_case("tet", 4)
    mesh.cells[0].data = mesh.cells[0].data + 1          # 1-based: the last node id is out of range
    I = ninpol_b200.Interpolator()
    with pytest.raises(NinpolB200Error, match="node id outside"):
        I.load_mesh(mesh_obj=mesh)
    mesh = meshgen.make_case("mixed", 6, a=1, b=3)
    mesh.cells[1].data = mesh.cells[1].data.copy()
    mesh.cells[1].data[7, 2] = -5
    with pytest.raises(NinpolB200Error, match="node id outside"):
        I.load_mesh(mesh_obj=mesh)
    good = meshgen.make_case("tet", 4)                   # the context is still usable
    I.load_mesh(mesh_obj=good)
    W, _ = I.interpolate("u", "idw")
    assert W.nnz > 0


def test_tile_kernels_bit_exact():
    """The IDW / LS tile kernels (k2_idw_ls_tile.cu) give bit-for-bit the oracle's values, over whole meshes and over
    the node chunks of the pipeline (tiles then start at arbitrary nodes), on 64-node and wide 128-node LS tiles."""
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    for kind, n, kw in (("tet", 14, {}), ("hex", 20, {}), ("hex", 20, {"perturb": 0.2}), ("mixed", 12, {"a": 3, "b": 6}),
                        ("tet", 9, {"scramble": True}), ("tri2d", 12, {}), ("quad2d", 9, {"perturb": 0.2})):
        mesh = meshgen.make_case(kind, n, **kw)
        O = oracle.OracleInterpolator().load_mesh(mesh)
        for chunks in (1, 7):
            I = ninpol_b200.Interpolator(stream_chunks=chunks)
            I.min_chunk_nodes = 1
            I.load_mesh(mesh_obj=mesh)
            for method in ("idw", "ls"):
                W, nv = I.interpolate("u", method)
                Wo, nvo = O.interpolate("u", method)
                assert np.array_equal(W.indptr, Wo.indptr) and np.array_equal(W.indices, Wo.indices), (kind, method, chunks)
                assert np.array_equal(W.data, Wo.data, equal_nan=True), (kind, method, chunks)
                assert np.array_equal(nv, nvo)


@pytest.mark.parametrize("kind,n,kw", [("tet", 9, {"scramble": True}), ("mixed", 10, {"a": 2, "b": 5}), ("quad2d", 9, {"perturb": 0.2})])
def test_both_esuel_kernels_bit_exact(kind, n, kw, monkeypatch):
    """esuel comes from the node-star kernel (k_esuel_star) by default and from the per-face candidate search
    (k_esuel, also the fallback for stars of more than 64 elements) with NPB_K1_ESUEL_PLAIN=1: both equal the oracle."""
    import ninpol_b200
    import oracle
    from ninpol_b200 import meshgen
    mesh = meshgen.make_case(kind, n, **kw)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    for plain in ("0", "1"):
        monkeypatch.setenv("NPB_K1_ESUEL_PLAIN", plain)
        I = ninpol_b200.Interpolator()
        I.load_mesh(mesh_obj=mesh)
        for name in ("esuel", "infael", "inpofa", "esuf", "esuf_ptr", "boundary_faces", "boundary_points", "fsup"):
            assert np.array_equal(np.asarray(getattr(I.grid, name)), getattr(O.grid, name)), (name, plain)
