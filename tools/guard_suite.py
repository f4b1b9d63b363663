"""Small-mesh pass over every kernel family with guard words behind every device block (NPB_DEBUG_GUARDS=1).

usage: python tools/guard_suite.py [quick]

compute-sanitizer is closed on the pool, so out-of-bounds WRITES are looked for this way: the library puts 64 known
bytes behind every block it allocates and `npb_check_guards` reads them back after each case.  Each case is one
load_mesh + idw / ls / gls through the default pipeline, the plain two-pass path and the plug-in (dense) entry point,
plus the lazily built exports (psup, edges).  Alternative kernels are selected the way the tests select them
(environment switches read at call time).  Prints one line per case; exits non-zero when a guard was overwritten.
tests/test_gpu_guards.py runs it in a subprocess (the guard switch is read once per process).
"""
import os
import sys

os.environ["NPB_DEBUG_GUARDS"] = "1"   # before the library's first use

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import ninpol_b200
from ninpol_b200 import meshgen

QUICK = len(sys.argv) > 1 and sys.argv[1] == "quick"


def run(kind, n, label, env=None, ctor=None, methods=("idw", "ls", "gls"), exports=False, **kw):
    saved = {}
    for k, v in (env or {}).items():
        saved[k] = os.environ.get(k)
        os.environ[k] = v
    try:
        mesh = meshgen.make_case(kind, n, **kw)
        ctor = dict(ctor or {})
        min_chunk = ctor.pop("min_chunk_nodes", None)
        I = ninpol_b200.Interpolator(build_edges=exports, **ctor)
        if min_chunk is not None:
            I.min_chunk_nodes = min_chunk
        I.load_mesh(mesh_obj=mesh)
        out = []
        for m in methods:
            W, nv = I.interpolate("u", m)
            out.append((m, int(W.nnz), float(np.nansum(W.data))))
        if exports:
            g = I.grid
            out.append(("psup", int(np.asarray(g.psup).size), 0.0))
            out.append(("inpoed", int(np.asarray(g.inpoed).shape[0]), 0.0))
            out.append(("esuf", int(np.asarray(g.esuf).size), 0.0))
        blocks, damaged = I._ctx.check_guards()
        print(label, kind, n, out, "guards", blocks, "damaged", damaged, flush=True)
        if blocks == 0:
            raise SystemExit("guards are off: NPB_DEBUG_GUARDS was not seen by the library")
        if damaged:
            raise SystemExit(f"{label} {kind} {n}: {damaged} guard(s) overwritten: {ninpol_b200._capi.load_library().npb_last_error().decode()}")
        del I
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def plugin(kind, n):
    mesh = meshgen.make_case(kind, n)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    g = I.grid
    for m in ("idw", "ls", "gls"):
        weights = np.zeros((g.n_points, g.MX_ELEMENTS_PER_POINT))
        neumann = np.zeros(g.n_points)
        I.supported_methods[m](g, I.cells_data, I.points_data, I.faces_data, I.variable_to_index, "u",
                               np.arange(g.n_points), weights, neumann)
        blocks, damaged = I._ctx.check_guards()
        print("plugin", kind, n, m, float(np.nansum(weights)), "guards", blocks, "damaged", damaged, flush=True)
        if damaged:
            raise SystemExit(f"plugin {m}: {damaged} guard(s) overwritten")


n3 = 4 if QUICK else 6
run("tet", n3, "default", exports=True)
run("hex", n3, "default", exports=True)
run("mixed", n3 + 2, "default")
run("quad2d", 6, "default-2d")
run("tri2d", 6, "default-2d")
run("tet", n3, "scrambled", scramble=True)
run("tet", n3, "two-pass", ctor=dict(stream_chunks=0, pinned_outputs=False, pin_inputs=False))
run("hex", n3, "chunks-of-few-nodes", ctor=dict(stream_chunks=4, min_chunk_nodes=16))
run("tet", n3, "plain-esuel", env={"NPB_K1_ESUEL_PLAIN": "1"}, methods=("idw",))
run("tet", n3, "simple-idw-ls", env={"NPB_FORCE_SIMPLE_IDW_LS": "1"}, methods=("idw", "ls"))
run("tet", n3, "gls-dense", env={"NPB_FORCE_GLS_DENSE": "1"}, methods=("gls",))
run("tet", n3, "gls-no-leaf", env={"NPB_GLS_NO_LEAF": "1"}, methods=("gls",))
run("tet", n3 + 4, "gls-team", env={"NPB_GLS_TEAM": "1,16"}, methods=("gls",))
run("mixed", n3 + 2, "gls-team", env={"NPB_GLS_TEAM": "0,4"}, methods=("gls",))
run("hex", n3, "no-neumann", neumann_rate=0.0)
plugin("tet", n3)
print("guard suite done", flush=True)
