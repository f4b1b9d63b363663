"""Parity at BASELINE.json's sizes (SURVEY.md 8d "Parity checks").

* C2 (Kuhn tets n = 69, 1.97 M cells; hex 128^3, 2.10 M cells; heterogeneous anisotropic K, 50 % Neumann hull
  nodes): comparison of the CUDA path with the outputs of the compiled reference (unmodified sources), stored under
  tests/golden/ as digests and a seeded sample of GLS rows — every Grid array bit for bit, IDW / LS and the GLS
  structure bit for bit, sampled GLS rows row-normwise <= 1e-12 with the element-wise error measured beside it.  Reference protocol: tests/performance_test.py:192-214; code compared:
  ninpol/_methods/gls.pyx:161-219,252-474, idw.pyx:57-84, ls.pyx:56-135, grid.pyx:233-525,661-809.
* C4 (Kuhn tets n = 203, 50.2 M cells) and C5 (mixed n = 170, 19.2 M cells): the reference needs ~40 GB and tens
  of minutes there, so (a) the connectivity is proven complete by vectorised numpy restatements of the
  reference's definitions over ALL entries (esup / fsup: counts, strictly ascending rows, membership; face
  numbering: first-encounter order; boundary tags: an independent geometric hull criterion) plus sampled
  esuel / geometry checks against the C oracle, and (b) the weights of >= 12,000 seeded sample nodes are
  recomputed by the C oracle's per-node routines (orc_idw_nodes / orc_ls_nodes / orc_gls_nodes, the very
  dgels the reference binds) from the exported arrays and compared: bit-exact IDW / LS, GLS <= 1e-12.
The measured errors are written to gpurun_out/parity_at_size.json (copied to profiles/ per round).
"""
import json
import os
import time

import numpy as np
import pytest

from at_size_checks import gls_verdict
from helpers import GRID_ARRAYS, ROOT

pytestmark = pytest.mark.gpu

N_SAMPLE = 12000
_RESULTS = {}


def _record(key, **kw):
    _RESULTS.setdefault(key, {}).update(kw)
    out = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_at_size.json"), "w") as f:
            json.dump(_RESULTS, f, indent=1, sort_keys=True)
    except OSError:
        pass


# ----------------------------------------------------------------------------------------------------
# C2: full comparison with the stored outputs of the compiled reference
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n", [("tet", 69), ("hex", 128)])
def test_c2_full_comparison_with_compiled_reference(kind, n):
    import oracle
    import ninpol_b200
    from helpers import check_against_reference_outputs, load_reference_outputs
    mesh, d, sample = load_reference_outputs(kind, n, {})
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    W, nv, ptr, got = check_against_reference_outputs(I, d, sample)
    key = f"C2_{kind}{n}"
    _record(key, n_cells=int(I.grid.n_elems), n_nodes=int(I.grid.n_points), against="stored outputs of the compiled reference",
            grid_arrays_bit_exact=list(GRID_ARRAYS), idw_ls_bit_exact=True, gls_structure_bit_exact=True)
    g = I.grid
    nodes = sample["nodes"]
    flags = np.asarray(mesh.point_data["neumann_flag_u"]).astype(np.int64)
    perm = np.concatenate([np.asarray(v) for v in mesh.cell_data["permeability"]])
    dm = I.compute_diffusion_magnitude(perm)
    bp = np.asarray(g.boundary_points)
    esup_ptr = np.asarray(g.esup_ptr)

    def exact_row(i):
        p = int(nodes[i])
        M, _w, _n = oracle.gls_system_of(g, p, flags, perm, dm, mesh.point_data["neumann_u"])
        return oracle.gls_exact_row(M, int(esup_ptr[p + 1] - esup_ptr[p]), bool(flags[p]) and bool(bp[p]))[0]

    try:
        v = gls_verdict(ptr, got, sample["data"], exact_row)
    except AssertionError as e:
        _record(key, gls=e.args[0] if e.args and isinstance(e.args[0], dict) else str(e)[:600])
        raise
    nvr = sample["neumann"]
    nerr = float(np.max(np.abs(nv[nodes] - nvr))) / max(1.0, float(np.max(np.abs(nvr))))
    _record(key, gls=v, gls_sampled_nodes=int(len(nodes)), gls_neumann_abs=nerr, gls_nnz=int(W.nnz))
    assert nerr <= 5e-12, nerr


# ----------------------------------------------------------------------------------------------------
# C4 / C5: complete connectivity proofs + sampled-node oracle parity
# ----------------------------------------------------------------------------------------------------
def _at_size(kind, n, kw, key):
    import oracle
    import ninpol_b200
    from ninpol_b200 import meshgen
    from at_size_checks import check_connectivity_and_geometry
    rng = np.random.default_rng(20261018)
    mesh = meshgen.make_case(kind, n, **kw)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    g = I.grid
    ne, npts, nf = g.n_elems, g.n_points, g.n_faces
    check_connectivity_and_geometry(g, mesh, rng, oracle)
    bpoints = np.asarray(g.boundary_points)
    _record(key, n_cells=int(ne), n_nodes=int(npts), n_faces=int(nf),
            connectivity="esup, fsup, face numbering, esuf, boundary tags: every entry; esuel / infael pairing: 4M sampled faces; "
                         "inpofa: 2M sampled faces; centroids / face centres / normals / areas: 500k sampled items, bit-exact")
    # ---- the weights of sampled nodes, recomputed by the C oracle ----
    flags = np.asarray(mesh.point_data["neumann_flag_u"]).astype(np.int64)
    processed = ~((bpoints != 0) & (flags == 0))
    neu = np.nonzero(processed & (bpoints != 0))[0]
    inter = np.nonzero(bpoints == 0)[0]
    n_neu = min(len(neu), N_SAMPLE // 4)
    nodes = np.sort(np.concatenate([rng.choice(neu, size=n_neu, replace=False),
                                    rng.choice(inter, size=N_SAMPLE - n_neu, replace=False),
                                    rng.choice(np.nonzero(~processed)[0], size=200, replace=False)]))
    perm = np.concatenate([np.asarray(v) for v in mesh.cell_data["permeability"]])
    dm = I.compute_diffusion_magnitude(perm)
    assert np.array_equal(dm, oracle.diffusion_magnitude(perm))
    for method in ("idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        assert W.indptr.dtype == np.int32 and W.indices.dtype == np.int32 and W.shape == (npts, ne)
        # structure of EVERY row: the esup row of a processed node, nothing for a Dirichlet node
        cnt = np.diff(W.indptr)
        assert np.array_equal(cnt[~processed], np.zeros(int((~processed).sum()), dtype=cnt.dtype))
        t0 = time.time()
        wd, nws = oracle.sample_rows(g, method, nodes, flags, perm, dm, mesh.point_data["neumann_u"])
        t_or = time.time() - t0
        rows = oracle.sample_csr_rows(g, nodes, wd, nws)
        ptr = np.concatenate([[0], np.cumsum([len(r[0]) for r in rows])])
        ref_idx = np.concatenate([r[0] for r in rows])
        ref_dat = np.concatenate([r[1] for r in rows])
        take = np.concatenate([np.arange(W.indptr[p], W.indptr[p + 1]) for p in nodes]) if len(nodes) else np.zeros(0, dtype=np.int64)
        got_ptr = np.concatenate([[0], np.cumsum(cnt[nodes])])
        assert np.array_equal(got_ptr, ptr), method + ": sampled row lengths"
        assert np.array_equal(W.indices[take], ref_idx), method + ": sampled column indices"
        got = W.data[take]
        if method == "gls":
            assert np.array_equal(np.isnan(got), np.isnan(ref_dat))
            esup_ptr = np.asarray(g.esup_ptr)

            def exact_row(i):
                p = int(nodes[i])
                M, _w, _n = oracle.gls_system_of(g, p, flags, perm, dm, mesh.point_data["neumann_u"])
                return oracle.gls_exact_row(M, int(esup_ptr[p + 1] - esup_ptr[p]), bool(flags[p]) and bool(bpoints[p]))[0]

            try:
                v = gls_verdict(ptr, got, ref_dat, exact_row)
            except AssertionError as e:
                _record(key, gls=e.args[0] if e.args and isinstance(e.args[0], dict) else str(e)[:600])
                raise
            nerr = float(np.max(np.abs(nv[nodes] - nws))) / max(1.0, float(np.max(np.abs(nws))))
            _record(key, gls=v, gls_sampled_nodes=int(len(nodes)), gls_sampled_neumann_nodes=int(n_neu), gls_neumann_abs=nerr,
                    oracle_gls_s=round(t_or, 2))
            assert nerr <= 5e-12, nerr
        else:
            assert np.array_equal(got, ref_dat, equal_nan=True), method
            assert np.array_equal(nv[nodes], nws), method
            _record(key, **{method + "_sampled_nodes_bit_exact": int(len(nodes))})
    return I, mesh


def test_c4_kuhn_tets_50m_cells_sampled_oracle_parity():
    _at_size("tet", 203, {}, "C4_tet203")


def test_c5_mixed_19m_cells_sampled_oracle_parity():
    _at_size("mixed", 170, {"a": 40, "b": 80}, "C5_mixed170")
