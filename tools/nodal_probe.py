"""Interpolator.nodal_values at size: wall time, apply-kernel time and its share of the measured copy bandwidth.

    python tools/nodal_probe.py [--out profiles/nodal_probe.json] [--workloads c4_gls,c3_idw] [--reps 7]

Workloads: C4 (Kuhn tets n = 203, 50,192,562 cells / 8,489,664 nodes) with GLS, and C3 (hex box 200^3, no Neumann nodes)
with IDW.  For k = 1 and 3 value columns, with the weights resident: the median wall time of nodal_values() on fresh
values (upload + kernel + download), the median device time of the apply kernel (npb_timing "apply") and the bytes the
kernel has to move, 12 nnz + 4 (rows + 1) + 8k (elements read) + 8k rows, over that time as a fraction of the device copy
rate (npb_measure_copy_bw).  The working set (> 2 GB at C4) is far larger than the 126 MB L2, so every call reads HBM.
For comparison: interpolate() + scipy's W @ u on the host, and the first nodal_values() call, which computes the
weights.  The full results are checked bit for bit against W @ u.  The card's name, power limit and SM clock are read
with nvidia-smi in the same run.

    python tools/nodal_probe.py --adjoint [--out profiles/nodal_adjoint_probe.json] [--workloads ...] [--reps 7]

The same for Interpolator.nodal_adjoint (W.T @ y) on the same workloads: the first call (weights and map computed by the
adjoint itself) and the map build inside it, the median wall time on fresh values with weights and map resident split
into H2D / kernel (npb_timing "adjoint") / D2H, the kernel's bytes, 8 spe n_elems (map) + 8 nnz (data) + 8k nnz (y
gathers) + 8k n_elems (out), as a fraction of the copy rate (and the same with y counted once, 8k n_points), scipy's
W.T @ y on the host, and bit-equality of the full results."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ninpol_b200
from ninpol_b200 import meshgen

WORKLOADS = {
    "c4_gls": ("tet", 203, 0.5, "gls", "C4: Kuhn tets n=203 (50,192,562 cells / 8,489,664 nodes), 50% Neumann hull nodes"),
    "c3_idw": ("hex", 200, 0.0, "idw", "C3: hex box 200^3 (8,000,000 cells / 8,120,601 nodes), no Neumann nodes"),
}


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64)))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def wall(fn, I):
    I._ctx.synchronize()
    t0 = time.perf_counter()
    out = fn()
    I._ctx.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def probe(name, reps, copy_gbs):
    kind, n, rate, method, desc = WORKLOADS[name]
    t0 = time.perf_counter()
    mesh = meshgen.make_case(kind, n, neumann_rate=rate)
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    g = I.grid
    print(f"[{name}] mesh ready in {time.perf_counter() - t0:.1f} s: {g.n_elems} cells, {g.n_points} nodes", flush=True)
    res = {"workload": desc, "method": method, "n_elems": int(g.n_elems), "n_points": int(g.n_points)}
    u = np.asarray(I._rows["cells"][I.variable_to_index["cells"]["u"]])[:g.n_elems]

    # the first call computes the weights (no CSR download); timed after one untimed warm-up
    first = []
    for rep in range(1 + min(reps, 3)):
        I.invalidate_inputs()
        ms, y_first = wall(lambda: I.nodal_values("u", method), I)
        assert not I.last_timings["nodal_weights_reused"]
        if rep:
            first.append(ms)
    res["first_call_with_weights_ms_median"] = float(np.median(first))

    # what a caller does today: interpolate (CSR to the host) + scipy on one core
    t_int, t_dot = [], []
    for rep in range(1 + min(reps, 3)):
        I.invalidate_inputs()
        ms_i, (W, _) = wall(lambda: I.interpolate("u", method), I)
        t1 = time.perf_counter()
        ref = W @ u
        ms_d = (time.perf_counter() - t1) * 1e3
        if rep:
            t_int.append(ms_i)
            t_dot.append(ms_d)
    res["interpolate_ms_median"] = float(np.median(t_int))
    res["host_scipy_dot_k1_ms_median"] = float(np.median(t_dot))
    res["bit_equal_first_call"] = same_bits(y_first, ref)
    nnz = int(W.nnz)
    elems_read = int(np.count_nonzero(np.bincount(W.indices, minlength=g.n_elems)))
    res.update({"nnz": nnz, "elements_read": elems_read})

    rng = np.random.default_rng(5)
    for k in (1, 3):
        xs = [rng.standard_normal(g.n_elems) if k == 1 else rng.standard_normal((g.n_elems, k)) for _ in range(2)]
        walls, kern, h2d, d2h = [], [], [], []
        for rep in range(reps + 2):
            x = xs[rep % 2]
            x = x + rep            # fresh values every call (not timed)
            ms, y = wall(lambda: I.nodal_values("u", method, x), I)
            assert I.last_timings["nodal_weights_reused"]
            if rep >= 2:
                walls.append(ms)
                kern.append(I.last_timings["nodal_apply_ms"])
                h2d.append(I.last_timings["nodal_h2d_ms"])
                d2h.append(I.last_timings["nodal_d2h_ms"])
        t1 = time.perf_counter()
        want = W @ x
        ms_host = (time.perf_counter() - t1) * 1e3
        bytes_needed = 12 * nnz + 4 * (g.n_points + 1) + 8 * k * elems_read + 8 * k * g.n_points
        kms = float(np.median(kern))
        res[f"k{k}"] = {
            "nodal_values_wall_ms_median": float(np.median(walls)),
            "apply_kernel_ms_median": kms,
            "apply_kernel_ms_min": float(np.min(kern)),
            "h2d_ms_median": float(np.median(h2d)),
            "d2h_ms_median": float(np.median(d2h)),
            "bytes_model": int(bytes_needed),
            "apply_gbs": bytes_needed / (kms * 1e-3) / 1e9,
            "fraction_of_copy_bw": bytes_needed / (kms * 1e-3) / (copy_gbs * 1e9),
            "host_scipy_dot_ms": ms_host,
            "bit_equal": same_bits(y, want),
        }
        print(f"[{name}] k={k}: {json.dumps(res[f'k{k}'])}", flush=True)
    del W
    return res


def probe_adjoint(name, reps, copy_gbs):
    kind, n, rate, method, desc = WORKLOADS[name]
    t0 = time.perf_counter()
    mesh = meshgen.make_case(kind, n, neumann_rate=rate)
    spe = 4 if max(len(c.data[0]) for c in mesh.cells) <= 4 else 8
    I = ninpol_b200.Interpolator()
    I.load_mesh(mesh_obj=mesh)
    g = I.grid
    print(f"[{name}] mesh ready in {time.perf_counter() - t0:.1f} s: {g.n_elems} cells, {g.n_points} nodes", flush=True)
    res = {"workload": desc, "method": method, "n_elems": int(g.n_elems), "n_points": int(g.n_points), "spe": spe}
    rng = np.random.default_rng(5)

    # the first call computes the weights (no CSR download) and builds the map; timed after one untimed warm-up
    y_first = rng.standard_normal(g.n_points)
    first, maps = [], []
    for rep in range(1 + min(reps, 3)):
        I.invalidate_inputs()
        ms, z_first = wall(lambda: I.nodal_adjoint("u", method, y_first), I)
        assert not I.last_timings["adjoint_weights_reused"]
        if rep:
            first.append(ms)
            maps.append(I.last_timings["adjoint_map_ms"])
    res["first_call_with_weights_ms_median"] = float(np.median(first))
    res["map_build_ms_median"] = float(np.median(maps))

    W, _ = I.interpolate("u", method)
    res["bit_equal_first_call"] = same_bits(z_first, W.T @ y_first)
    nnz = int(W.nnz)
    res["nnz"] = nnz
    for k in (1, 3):
        ys = [rng.standard_normal(g.n_points) if k == 1 else rng.standard_normal((g.n_points, k)) for _ in range(2)]
        walls, kern, h2d, d2h = [], [], [], []
        for rep in range(reps + 2):        # the first call after interpolate() rebuilds the map: warm-up
            y = ys[rep % 2] + rep          # fresh values every call (not timed)
            ms, z = wall(lambda: I.nodal_adjoint("u", method, y), I)
            assert I.last_timings["adjoint_weights_reused"]
            if rep >= 2:
                assert I.last_timings["adjoint_map_ms"] == 0.0
                walls.append(ms)
                kern.append(I.last_timings["adjoint_apply_ms"])
                h2d.append(I.last_timings["adjoint_h2d_ms"])
                d2h.append(I.last_timings["adjoint_d2h_ms"])
        t1 = time.perf_counter()
        want = W.T @ y
        ms_host = (time.perf_counter() - t1) * 1e3
        bytes_needed = 8 * spe * g.n_elems + 8 * nnz + 8 * k * nnz + 8 * k * g.n_elems
        # each array once (the y gathers of one node repeat over its elements and mostly hit L2)
        bytes_once = 8 * spe * g.n_elems + 8 * nnz + 8 * k * g.n_points + 8 * k * g.n_elems
        kms = float(np.median(kern))
        res[f"k{k}"] = {
            "nodal_adjoint_wall_ms_median": float(np.median(walls)),
            "adjoint_kernel_ms_median": kms,
            "adjoint_kernel_ms_min": float(np.min(kern)),
            "h2d_ms_median": float(np.median(h2d)),
            "d2h_ms_median": float(np.median(d2h)),
            "bytes_model": int(bytes_needed),
            "adjoint_gbs": bytes_needed / (kms * 1e-3) / 1e9,
            "fraction_of_copy_bw": bytes_needed / (kms * 1e-3) / (copy_gbs * 1e9),
            "bytes_each_array_once": int(bytes_once),
            "fraction_of_copy_bw_each_array_once": bytes_once / (kms * 1e-3) / (copy_gbs * 1e9),
            "host_scipy_transposed_dot_ms": ms_host,
            "bit_equal": same_bits(z, want),
        }
        print(f"[{name}] k={k}: {json.dumps(res[f'k{k}'])}", flush=True)
    del W
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--adjoint", action="store_true", help="probe nodal_adjoint (W.T @ y) instead of nodal_values")
    ap.add_argument("--out", default=None)
    ap.add_argument("--workloads", default="c4_gls,c3_idw")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if args.out is None:
        args.out = os.path.join("profiles", "nodal_adjoint_probe.json" if args.adjoint else "nodal_probe.json")
    from ninpol_b200 import _capi
    ctx = _capi.Context(0)
    copy_gbs = ctx.measure_copy_bw(1 << 31)
    ctx.close()
    out = {"card": card(), "card_query": "nvidia-smi --query-gpu=name,power.limit,clocks.max.sm", "copy_gbs": copy_gbs,
           "reps": args.reps, "results": {}}
    print(f"card {out['card']}; device copy {copy_gbs:.0f} GB/s", flush=True)
    ok = True
    for name in args.workloads.split(","):
        r = (probe_adjoint if args.adjoint else probe)(name, args.reps, copy_gbs)
        out["results"][name] = r
        ok = ok and r["bit_equal_first_call"] and r["k1"]["bit_equal"] and r["k3"]["bit_equal"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("nodal adjoint probe" if args.adjoint else "nodal probe", "bit-equal" if ok else "MISMATCH", "->", args.out, flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
