"""Multi-GPU check of Interpolator.nodal_values, to be launched with torchrun (one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29547 tools/check_multi_gpu_nodal.py
Every rank computes the weights of its node range with the two-pass count (only row counts and neumann entries travel),
multiplies its rows by the values of the elements they refer to, and the row blocks of the result are all-gathered.  For
every gather mode and method, every rank's result must be bit-equal to W_full @ u, where W_full is the full CSR that
interpolate() returns with gather="all"."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ninpol_b200
from ninpol_b200 import dist, meshgen


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64)))


comm = dist.init_from_env()
ok = True
I = ninpol_b200.Interpolator(comm=comm)      # one NCCL communicator per unique id: reuse the object
I.min_chunk_nodes = 16

CASES = [("tet", 10, {}), ("mixed", 10, {"a": 2, "b": 5}), ("hex", 12, {}), ("tet", 8, {"scramble": True})]
for kind, n, kw in CASES:
    mesh = meshgen.make_case(kind, n, **kw)
    I.load_mesh(mesh_obj=mesh)
    rng = np.random.default_rng(11)          # the same values on every rank
    u1 = rng.standard_normal(I.grid.n_elems)
    u3 = rng.standard_normal((I.grid.n_elems, 3))
    I.set_gather("all")
    W_full = {}
    for method in ("idw", "ls", "gls"):
        W, _ = I.interpolate("u", method)
        W_full[method] = W.copy()
    own = np.asarray(I._rows["cells"][I.variable_to_index["cells"]["u"]])[:I.grid.n_elems]
    for gather, chunks in (("all", 8), ("all", 0), ("root", 8), ("host", 3)):
        I.set_gather(gather)
        I.stream_chunks = chunks
        for method in ("idw", "ls", "gls"):
            y0 = I.nodal_values("u", method)
            fresh = not I.last_timings["nodal_weights_reused"]
            y1 = I.nodal_values("u", method, u1)
            y3 = I.nodal_values("u", method, u3)
            reused = I.last_timings["nodal_weights_reused"]
            Wf = W_full[method]
            good = fresh and reused and same_bits(y0, Wf @ own) and same_bits(y1, Wf @ u1) and same_bits(y3, Wf @ u3)
            print(f"rank {comm.rank}/{comm.world} {kind}{n}{'s' if kw.get('scramble') else ''} gather={gather} "
                  f"chunks={chunks} {method}: {'OK' if good else 'MISMATCH'} bounds {[int(b) for b in I.partition_bounds]}",
                  flush=True)
            ok = ok and good
        # interpolate after nodal_values still returns what it returned before
        if gather == "all":
            W, _ = I.interpolate("u", "idw")
            good = np.array_equal(W.indptr, W_full["idw"].indptr) and same_bits(W.data, W_full["idw"].data)
            print(f"rank {comm.rank}/{comm.world} {kind}{n} interpolate after nodal_values: {'OK' if good else 'MISMATCH'}",
                  flush=True)
            ok = ok and good
sys.exit(0 if ok else 1)
