"""Generates the golden fixtures of tests/golden/ from the COMPILED REFERENCE (oracle/_ref, built by
oracle/build_ref.py from /root/reference).  Run in the build container only (the reference does not
exist on the GPU box); the .npz / .json outputs are committed.

    python tests/golden/make_golden.py

Fixtures
  <name>.npz            synthetic mesh (points, one cell array per type, cell/point data) and every
                        output of the reference on it: Grid arrays, and for idw / ls / gls the CSR
                        (indptr, indices, data) and the neumann vector.
  reference_digests.json, reference_gls_<mesh>.npz
                        outputs of the reference on the meshes of the tests that compare with it, as digests
                        and a sample of GLS rows (--digests; see make_digests).
  accuracy_hexa.json    the reference's own published known-answer numbers: relative L2 errors at interior
                        nodes on unit-cube n^3 hexahedral meshes, copied from
                        /root/reference/tests/results/yaml/accuracy.yaml (hexa rows; ALH :2-41, FAN :148-187,
                        LIN :294-333, QUAD :440-479) for n = 4, 8, 16 — and re-measured here with the
                        compiled reference to confirm they are reproducible without the unshipped meshes.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from ninpol_b200 import meshgen  # noqa: E402

GRID_ARRAYS = ("esup", "esup_ptr", "psup", "psup_ptr", "esuel", "infael", "inpofa", "fsup", "fsup_ptr", "esuf", "esuf_ptr",
               "boundary_faces", "boundary_points", "centroids", "faces_centers", "normal_faces", "faces_areas")
GRID_SCALARS = ("n_elems", "n_points", "n_faces", "MX_ELEMENTS_PER_POINT", "MX_POINTS_PER_POINT", "MX_ELEMENTS_PER_FACE",
                "MX_FACES_PER_POINT")
CASES = {"tet_n4": ("tet", 4, {}), "hex_n4": ("hex", 4, {}), "hex_n3_perturbed": ("hex", 3, {"perturb": 0.2}),
         "mixed_n6": ("mixed", 6, {"a": 1, "b": 3})}


def mesh_to_arrays(mesh):
    out = {"points": mesh.points, "cell_types": np.array([c.type for c in mesh.cells])}
    for i, c in enumerate(mesh.cells):
        out[f"cells_{i}"] = c.data
        for name, per_block in mesh.cell_data.items():
            out[f"celldata_{name}_{i}"] = np.asarray(per_block[i])
    for name, v in mesh.point_data.items():
        out[f"pointdata_{name}"] = np.asarray(v)
    return out


def arrays_to_mesh(d):
    types = [str(t) for t in d["cell_types"]]
    cells = [meshgen.CellBlock(t, d[f"cells_{i}"]) for i, t in enumerate(types)]
    cell_names = sorted({k[len("celldata_"):].rsplit("_", 1)[0] for k in d.files if k.startswith("celldata_")})
    cell_data = {n: [d[f"celldata_{n}_{i}"] for i in range(len(types))] for n in cell_names}
    point_data = {k[len("pointdata_"):]: d[k] for k in d.files if k.startswith("pointdata_")}
    return meshgen.SimpleMesh(d["points"], cells, point_data, cell_data)


# analytic cases of the reference's tests/utils/analytical.py:249-325
def K_const(n, Ku):
    K = np.zeros((n, 3, 3))
    K[:] = np.asarray(Ku)
    return K


def alh_K(n, c):
    x, y, z = c[:, 0], c[:, 1], c[:, 2]
    K = np.zeros((n, 3, 3))
    K[:, 0, 0] = y ** 2 + z ** 2 + 1; K[:, 0, 1] = -x * y; K[:, 0, 2] = -x * z
    K[:, 1, 0] = -y * x; K[:, 1, 1] = x ** 2 + z ** 2 + 1; K[:, 1, 2] = -y * z
    K[:, 2, 0] = -z * x; K[:, 2, 1] = -z * y; K[:, 2, 2] = x ** 2 + y ** 2 + 1
    return K


_KU = [[1.0, 0.5, 0.0], [0.5, 1.0, 0.5], [0.0, 0.5, 1.0]]
ANALYTIC = {
    "LIN": (lambda x, y, z: x + y + z, lambda n, c: K_const(n, _KU)),
    "QUAD": (lambda x, y, z: x ** 2 + y ** 2 + z ** 2, lambda n, c: K_const(n, _KU)),
    "FAN": (lambda x, y, z: np.sin(2 * np.pi * x) * np.sin(2 * np.pi * y) * np.sin(2 * np.pi * z),
            lambda n, c: K_const(n, [[2464.36, 0.0, 1148.68], [0.0, 536.64, 0.0], [1148.68, 0.0, 536.64]])),
    "ALH": (lambda x, y, z: (x ** 3) * (y ** 2) * z + x * np.sin(2 * np.pi * x * z) * np.sin(2 * np.pi * x * y) * np.sin(2 * np.pi * z),
            alh_K),
}


def analytic_mesh(case, n):
    """unit-cube n^3 hex mesh carrying the analytic case `case`; all boundary nodes Dirichlet (the
    interior-node error does not depend on the reference test's random Dirichlet/Neumann split)."""
    sol, Kf = ANALYTIC[case]
    mesh = meshgen.hex_box(n)
    cen = mesh.points[mesh.cells[0].data].mean(axis=1)
    K = Kf(len(cen), cen).reshape(-1, 9)
    npts = len(mesh.points)
    mesh.cell_data = {"permeability": [K], case: [sol(cen[:, 0], cen[:, 1], cen[:, 2])]}
    mesh.point_data = {"neumann_flag_" + case: np.zeros(npts), "neumann_" + case: np.zeros(npts)}
    return mesh, sol


def interior_l2(W, mesh, sol, case, boundary_points):
    u = mesh.cell_data[case][0]
    vals = W.dot(u)
    P = mesh.points
    exact = sol(P[:, 0], P[:, 1], P[:, 2])
    inner = np.asarray(boundary_points) == 0
    ref = exact[inner]
    return float(np.sqrt(np.sum((vals[inner] - ref) ** 2) / np.sum(ref ** 2)))


def main():
    ninpol = oracle.load_reference()
    if ninpol is None:
        sys.exit("compiled reference not available: run `python oracle/build_ref.py` first")
    for name, (kind, n, kw) in CASES.items():
        mesh = meshgen.make_case(kind, n, **kw)
        I = ninpol.Interpolator()
        I.load_mesh(mesh_obj=oracle.to_reference_mesh(mesh))
        out = mesh_to_arrays(mesh)
        for a in GRID_ARRAYS:
            out["grid_" + a] = np.asarray(getattr(I.grid, a))
        out["grid_scalars"] = np.array([getattr(I.grid, s) for s in GRID_SCALARS], dtype=np.int64)
        for method in ("idw", "ls", "gls"):
            W, nv = I.interpolate("u", method)
            out[f"{method}_indptr"], out[f"{method}_indices"], out[f"{method}_data"] = W.indptr, W.indices, W.data
            out[f"{method}_neumann"] = np.asarray(nv)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, "elems", I.grid.n_elems, "points", I.grid.n_points, os.path.getsize(os.path.join(HERE, name + ".npz")), "bytes")
    # known-answer accuracy numbers: published vs re-measured with the compiled reference
    import yaml
    pub = yaml.safe_load(open("/root/reference/tests/results/yaml/accuracy.yaml"))
    table = {}
    for case in ("LIN", "QUAD", "FAN", "ALH"):
        table[case] = {}
        for method in ("gls", "idw", "ls"):
            published = [float(x) for x in pub[case]["hexa"]["methods"][method]["error"][:3]]
            measured = []
            for n in (4, 8, 16):
                mesh, sol = analytic_mesh(case, n)
                I = ninpol.Interpolator()
                I.load_mesh(mesh_obj=oracle.to_reference_mesh(mesh))
                W, _ = I.interpolate(case, method)
                measured.append(interior_l2(W, mesh, sol, case, I.grid.boundary_points))
            table[case][method] = {"n": [4, 8, 16], "published": published, "reference_here": measured}
            print(case, method, ["%.6e" % x for x in published], ["%.6e" % x for x in measured])
    json.dump({"source": "reference tests/results/yaml/accuracy.yaml hexa rows (ALH :2-41, FAN :148-187, LIN :294-333, QUAD :440-479)",
               "metric": "relative L2 error of W @ u_cells at interior nodes (tests/utils/analytical.py:106-110, 233-243)",
               "table": table}, open(os.path.join(HERE, "accuracy_hexa.json"), "w"), indent=1)


# ------------------------------------------------------------------------------------------------------------
# Digests: the outputs of the reference on the meshes of the tests that compare with it on fresh meshes
# (tests/test_oracle.py) and at size (tests/test_gpu_golden.py, tests/test_gpu_at_size.py), stored so that those
# comparisons need nothing outside the repository.  Every array is stored as a digest (tests/helpers.py), which
# settles a bit-exact comparison; GLS weights, compared within a tolerance, are stored as a seeded row sample.
#
#     python tests/golden/make_golden.py --digests [--source reference|oracle]
#
# --source oracle takes the outputs from the C oracle instead of the compiled reference; the source used is recorded.
# On SMALL_CASES and EDGE_CASES the oracle's outputs were equal to the compiled reference's bit for bit (every Grid
# array, every CSR of IDW / LS / GLS, the neumann vectors, the edge tables: test_oracle.py compared them directly), so
# both sources write the same digests there.  AT_SIZE_CASES run the same C code and the same scipy DGELS on larger
# meshes of the same generator.
# ------------------------------------------------------------------------------------------------------------
SMALL_CASES = [("tet", 6, {}), ("hex", 7, {}), ("mixed", 8, {"a": 2, "b": 4}), ("hex", 5, {"perturb": 0.2}),
               ("tet", 1, {}), ("hex", 1, {}), ("quad2d", 6, {}), ("tri2d", 6, {"perturb": 0.2}),
               ("tet", 6, {"scramble": True}), ("mixed", 8, {"a": 2, "b": 4, "scramble": True})]
EDGE_CASES = [("tet", 5, {}), ("mixed", 8, {"a": 2, "b": 4}), ("tri2d", 7, {})]
AT_SIZE_CASES = [("tet", 40, {}), ("tet", 69, {}), ("hex", 128, {})]
GLS_SAMPLE = (100, 280, 20)        # Neumann boundary / interior / Dirichlet nodes of the stored GLS rows
DIGESTS = os.path.join(HERE, "reference_digests.json")


def case_key(kind, n, kw):
    return "-".join([kind, str(n)] + [f"{k}={kw[k]}" for k in sorted(kw)])


def gls_sample_path(key):
    return os.path.join(HERE, f"reference_gls_{key}.npz")


def mesh_digest(mesh):
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import digest
    parts = [digest(mesh.points)] + [c.type + digest(c.data) for c in mesh.cells]
    parts += [k + digest(np.concatenate([np.ravel(v) for v in mesh.cell_data[k]])) for k in sorted(mesh.cell_data)]
    parts += [k + digest(mesh.point_data[k]) for k in sorted(mesh.point_data)]
    return digest(np.frombuffer(" ".join(parts).encode(), dtype=np.uint8))


def gls_sample_nodes(boundary_points, flags, rng):
    bp = np.asarray(boundary_points) != 0
    processed = ~(bp & (flags == 0))
    groups = (np.nonzero(processed & bp)[0], np.nonzero(~bp)[0], np.nonzero(~processed)[0])
    return np.sort(np.concatenate([rng.choice(g, size=min(len(g), k), replace=False) for g, k in zip(groups, GLS_SAMPLE)]))


def outputs_digests(I, grid_arrays=GRID_ARRAYS):
    from helpers import digest
    g = I.grid
    out = {"grid_scalars": {s: int(getattr(g, s)) for s in GRID_SCALARS},
           "grid": {a: digest(getattr(g, a)) for a in grid_arrays}}
    results = {}
    for method in ("idw", "ls", "gls"):
        W, nv = I.interpolate("u", method)
        results[method] = (W, np.asarray(nv))
        out[method] = {"indptr": digest(W.indptr), "indices": digest(W.indices), "nan": digest(np.isnan(W.data))}
        if method != "gls":
            out[method].update(data=digest(W.data), neumann=digest(nv))
    return out, results


def make_digests(source):
    sys.path.insert(0, os.path.dirname(HERE))
    if source == "reference" and oracle.load_reference() is None:
        sys.exit("compiled reference not available: run `python oracle/build_ref.py` first, or pass --source oracle")

    def interpolator(mesh, build_edges=False):
        if source == "reference":
            ninpol = oracle.load_reference()
            I = ninpol.Interpolator(build_edges=True) if build_edges else ninpol.Interpolator()
            I.load_mesh(mesh_obj=oracle.to_reference_mesh(mesh))
            return I
        return oracle.OracleInterpolator().load_mesh(mesh, build_edges=build_edges)

    from helpers import digest
    doc = {"source": "compiled reference (oracle/_ref)" if source == "reference" else
           "C oracle (oracle/), equal to the compiled reference bit for bit on these meshes",
           "small": {}, "edges": {}, "at_size": {}}
    for kind, n, kw in SMALL_CASES:
        mesh = meshgen.make_case(kind, n, **kw)
        d, res = outputs_digests(interpolator(mesh))
        W, nv = res["gls"]
        d["gls"].update(data=digest(W.data), neumann=digest(nv))     # the oracle's GLS is the reference's bit for bit
        doc["small"][case_key(kind, n, kw)] = dict(mesh=mesh_digest(mesh), **d)
    for kind, n, kw in EDGE_CASES:
        mesh = meshgen.make_case(kind, n, **kw)
        g = interpolator(mesh, build_edges=True).grid
        doc["edges"][case_key(kind, n, kw)] = {"mesh": mesh_digest(mesh), "n_edges": int(g.n_edges),
                                               "inedel": digest(g.inedel), "inpoed": digest(g.inpoed)}
    for kind, n, kw in AT_SIZE_CASES:
        key = case_key(kind, n, kw)
        mesh = meshgen.make_case(kind, n, **kw)
        I = interpolator(mesh)
        d, res = outputs_digests(I)
        doc["at_size"][key] = dict(mesh=mesh_digest(mesh), **d)
        W, nv = res["gls"]
        flags = np.asarray(mesh.point_data["neumann_flag_u"]).astype(np.int64)
        nodes = gls_sample_nodes(I.grid.boundary_points, flags, np.random.default_rng(20261020))
        take = np.concatenate([np.arange(W.indptr[p], W.indptr[p + 1]) for p in nodes])
        np.savez_compressed(gls_sample_path(key), nodes=nodes.astype(np.int64), row_nnz=np.diff(W.indptr)[nodes].astype(np.int64),
                            indices=W.indices[take].astype(np.int64), data=W.data[take], neumann=nv[nodes])
        print(key, "nodes", I.grid.n_points, "gls sample", len(nodes), os.path.getsize(gls_sample_path(key)), "bytes", flush=True)
    with open(DIGESTS, "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    if "--digests" in sys.argv:
        make_digests(sys.argv[sys.argv.index("--source") + 1] if "--source" in sys.argv else "reference")
    else:
        main()
