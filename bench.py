#!/usr/bin/env python
"""bench.py — node weights/sec of the ninpol hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the unmodified reference, host cores

A step is one pass of `interpolate` (K2 weights + K3 CSR emit + K4 NCCL gather of the row blocks when N > 1)
over every node of one synthetic mesh.  Default workload = BASELINE config C4: Kuhn tetrahedra n = 203
(50.2 M cells, 8.49 M nodes), perturbed 0.25 h, heterogeneous anisotropic K, 50 % Neumann hull nodes, GLS.
For N > 1 (launched by torchrun, one rank per GPU) the SAME mesh is split by nodes over the ranks (strong
scaling); value = n_nodes / max-over-ranks device time per step.

One JSON line on stdout (rank 0):
  value         device-timed (CUDA events on the library stream, max over ranks), inputs resident in HBM, result left
                on the device; at N > 1 the step ends with every rank holding the full CSR (gather = all over NCCL);
                `device_compute_only` is the same step with the blocks left on their owners (gather = host);
  e2e           `Interpolator.interpolate` with host buffers: H2D of the per-variable inputs and D2H of the CSR inside
                the timed region, default constructor arguments (N > 1: gather='host', and gather='all' beside it);
  roofline      the dominant kernel against the measured HBM peak (+ an FP64 view for GLS);
  configs       every other BASELINE config (C1, C2 both meshes, C3, C5) on the same GPUs, short runs;
  cpu_baseline  the compiled reference (oracle/_ref) on the box's host cores on C2 (Kuhn n = 69), mean of 3.
The reference arm times the unmodified reference on C2 (Kuhn tets n = 69, 1.97 M cells: the largest BASELINE config
its Python ingest and 16-thread GLS finish in minutes); `configs.C2_tet69` of this arm is the same mesh.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (kind, n, description)
    "tet203": ("tet", 203, "C4: Kuhn tets n=203 (50,192,562 cells / 8,489,664 nodes), perturb 0.25h, heterogeneous anisotropic K, 50% Neumann hull nodes"),
    "tet69": ("tet", 69, "C2: Kuhn tets n=69 (1,971,054 cells / 343,000 nodes), perturb 0.25h, heterogeneous anisotropic K, 50% Neumann hull nodes"),
    "tet40": ("tet", 40, "Kuhn tets n=40 (384,000 cells / 68,921 nodes)"),
    "tet7": ("tet", 7, "C1: Kuhn tets n=7 (2,058 cells / 512 nodes)"),
    "hex200": ("hex", 200, "C3: structured hex box 200^3 (8,000,000 cells / 8,120,601 nodes)"),
    "hex128": ("hex", 128, "C2: structured hex box 128^3 (2,097,152 cells / 2,146,689 nodes)"),
    "mixed170": ("mixed", 170, "C5: conforming mixed hex/wedge/pyramid/tet box n=170, a=40, b=80 (19.2M cells), 50% Neumann hull nodes"),
    "mixed60": ("mixed", 60, "mixed hex/wedge/pyramid/tet box n=60 (a=15, b=30)"),
}
REF_WORKLOAD = "tet69"     # what the reference arm and cpu_baseline time (config C2)
REF_REPEATS = 3            # tests/config.yaml:3-4 n_repeats, tests/performance_test.py:192-214
VARIABLE = "u"
# (key, workload, methods, neumann_rate): the BASELINE configs beside the headline one
CONFIG_RUNS = [
    ("C1_tet7", "tet7", ("idw",), 0.5),
    ("C2_tet69", "tet69", ("gls", "ls"), 0.5),
    ("C2_hex128", "hex128", ("gls", "ls"), 0.5),
    ("C3_hex200", "hex200", ("idw", "ls"), 0.0),
    ("C3_hex200_neumann50", "hex200", ("ls",), 0.5),
    ("C5_mixed170", "mixed170", ("gls",), 0.5),
]


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def make_mesh(kind, n, neumann_rate=0.5):
    from ninpol_b200 import meshgen
    kw = {"a": (n * 40) // 170, "b": (n * 80) // 170} if kind == "mixed" else {}
    return meshgen.make_case(kind, n, variable=VARIABLE, neumann_rate=neumann_rate, **kw)


# ------------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# algorithmic bytes / flops (SURVEY.md 8d; stated again in DESIGN.md)
# ------------------------------------------------------------------------------------------------
def algorithmic_model(I, method, lo=0, hi=None):
    """bytes / flops / processed nodes of the node range [lo, hi) (a rank's share)."""
    g = I.grid
    esup_ptr, fsup_ptr = np.asarray(g.esup_ptr), np.asarray(g.fsup_ptr)
    hi = len(esup_ptr) - 1 if hi is None else hi
    E = np.diff(esup_ptr[lo:hi + 1]).astype(np.float64)
    F = np.diff(fsup_ptr[lo:hi + 1]).astype(np.float64)
    flags = np.asarray(I._flags_host)[lo:hi]
    bpts = np.asarray(g.boundary_points)[lo:hi] != 0
    processed = ~(bpts & (flags == 0))
    per = 120.0 * E + 60.0 * F + 42.0 if method == "gls" else 40.0 * E + 42.0
    nbytes = float(np.where(processed, per, 18.0).sum())
    flops = 0.0
    if method == "gls":
        # B (boundary faces at the node) only enters m for Neumann nodes; interior nodes have B = 0
        B = np.zeros_like(E)
        nb = np.nonzero(bpts)[0]                      # only boundary nodes have boundary faces
        if len(nb):
            fs, bf = np.asarray(g.fsup), np.asarray(g.boundary_faces)
            starts = fsup_ptr[lo + nb]
            lens = fsup_ptr[lo + nb + 1] - starts
            owner = np.repeat(np.arange(len(nb)), lens)
            idx = np.repeat(starts - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
            B[nb] = np.bincount(owner, weights=(bf[fs[idx]] != 0).astype(np.float64), minlength=len(nb))
        m = E + 3.0 * F + np.where(flags != 0, B, 0.0)
        n = 3.0 * E + 1.0
        per_f = 2.0 * m * n * n - (2.0 / 3.0) * n ** 3 + 4.0 * m * n
        live = processed & ~(B >= F)
        flops = float(np.where(live, per_f, 0.0).sum())
    return nbytes, flops, int(processed.sum())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (driver-measured copy bandwidth, burst)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def profiled(kind, method):
    """Per-node DRAM traffic and counters of the dominant kernel from the committed ncu capture of this mesh family."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(p)).get(f"{kind}:{method}:per_node", {})
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference (oracle/_ref) on the host cores
# ------------------------------------------------------------------------------------------------
def reference_interpolator(kind, n):
    import oracle
    ninpol = oracle.load_reference()
    mesh = make_mesh(kind, n)
    if ninpol is not None:
        I = ninpol.Interpolator()
        t0 = time.time()
        I.load_mesh(mesh_obj=oracle.to_reference_mesh(mesh))
        return I, "reference", time.time() - t0, len(mesh.points), mesh.n_cells
    O = oracle.OracleInterpolator()
    t0 = time.time()
    O.load_mesh(mesh)
    return O, "port", time.time() - t0, len(mesh.points), mesh.n_cells


def time_reference(workload, method, steps, warmup):
    kind, n, desc = WORKLOADS[workload]
    I, how, t_load, n_points, n_cells = reference_interpolator(kind, n)
    for _ in range(warmup):
        I.interpolate(VARIABLE, method)
    ts = []
    for _ in range(steps):
        t0 = time.time()
        I.interpolate(VARIABLE, method)
        ts.append(time.time() - t0)
    t = float(np.mean(ts))
    ncpu = os.cpu_count() or 1
    threads = min(16, ncpu) if how == "reference" else 1
    return {"value": n_points / t, "unit": "nodes/s", "cores": threads, "kind": how,
            "sample": f"{desc}: {n_cells} cells / {n_points} nodes, time.time() around interpolate('{VARIABLE}','{method}'), mean of {steps} "
                      f"after {warmup} warm-up (tests/performance_test.py:192-214 protocol); the reference caps itself at 16 OpenMP threads "
                      f"(gls.pyx:87; min(16, ceil(n/400)) for IDW / LS), host has {ncpu} logical cores; OPENBLAS_NUM_THREADS=1 "
                      f"(gls.pyx:61-70); load_mesh {t_load:.2f}s (Python ingest) not counted",
            "seconds_per_step": t, "load_mesh_s": t_load, "workload": workload, "n_nodes": n_points, "n_cells": n_cells}


def run_reference(args, rank):
    if rank != 0:
        return
    workload = args.ref_workload
    base = time_reference(workload, args.method, args.steps, args.warmup)
    line = {"impl": "reference", "metric": f"node weights/sec ({args.method.upper()})", "value": base["value"], "unit": "nodes/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload][2], "method": args.method,
                       "sample_workload": WORKLOADS[workload][2],
                       "note": "the reference's CPU path timed on a bounded sample of the workload: BASELINE config C2 (same generator, "
                               "n = 69); this repository's arm reports the same mesh under configs.C2_tet69"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------
# this repository's arm
# ------------------------------------------------------------------------------------------------
class Plumbing:
    """barrier + max-over-ranks; torch.distributed (gloo) only when world > 1."""

    def __init__(self, rank, world):
        self.rank, self.world, self.dist = rank, world, None
        if world > 1:
            import torch
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("gloo", rank=rank, world_size=world)
            self.dist, self.torch = dist, torch

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def _red(self, v, op):
        if not self.dist:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, v):
        return self._red(v, self.dist.ReduceOp.MAX if self.dist else None)

    def sum(self, v):
        return self._red(v, self.dist.ReduceOp.SUM if self.dist else None)

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def device_step(I, method, chunks=1):
    """One pass with the result left on the device: plan + kernels (+ NCCL gather when gather = all; with chunks > 1
    the broadcast of chunk k runs on its own stream under the kernels of chunk k+1)."""
    nnz, fell_back = I._ctx.interpolate_run(method, chunks)
    if fell_back:   # an exact-zero weight: the general two-pass path (counts exchanged, scan, emit, gather)
        I._ctx.interpolate_count(method)
        I._ctx.interpolate_fetch(None, None, None, None)


def timed_device_steps(I, plumb, method, steps, warmup, sampler=None, chunks=1):
    ctx = I._ctx
    for _ in range(warmup):
        device_step(I, method, chunks)
    main_ms, step_ms = [], []
    plumb.barrier()
    ctx.synchronize()
    if sampler:
        sampler.start()
    l0 = ctx.launch_count()
    ctx.timer_start()
    for _ in range(steps):
        device_step(I, method, chunks)
        main_ms.append(ctx.timing_or("k2_main", ctx.timing_or("k2")))
        step_ms.append(ctx.timing_or("streamed"))
    ms = ctx.timer_stop()
    ctx.synchronize()
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    plumb.barrier()
    return {"ms_per_step": plumb.max(ms) / steps, "kernel_ms": float(np.mean(main_ms)), "launches": launches, "clocks": clocks,
            "step_ms_median": plumb.max(float(np.median(step_ms))), "step_ms_best": plumb.max(float(np.min(step_ms)))}


DUMP_ROWS = 1 << 16        # CSR rows sampled by --dump-outputs
DUMP_SEED = 0
DUMP_BYTES = 64 << 20      # all files together, .npy headers included
DUMP_CHUNK = 1 << 22       # entries per pass of the whole-result sums (bounds their temporaries)


def dump_outputs(I, out_dir):
    """Write what the last device step computed, as the caller of interpolate() would receive it, under out_dir.

    The whole CSR of the default workload is ~2.4 GB, so a fixed seeded sample of DUMP_ROWS rows is written: their ids
    (rows), entry counts (row_nnz), element ids (indices), weights (data) and neumann weights (neumann).  totals holds
    sums over the whole result, so that a difference outside the sample still shows: [n_rows, n_cols, nnz, NaN count,
    nansum(data), nansum(|data|), nansum(data * (indices + 1)), nansum(neumann)], the entry sums taken DUMP_CHUNK
    entries at a time.  Every file is float64, and all of them together take at most DUMP_BYTES."""
    ctx, g = I._ctx, I.grid
    n_rows, n_cols = int(g.n_points), int(g.n_elems)
    indptr = np.empty(n_rows + 1, dtype=np.int32)
    neumann = np.empty(n_rows, dtype=np.float64)
    ctx.interpolate_fetch(indptr, None, None, neumann)
    nnz = int(indptr[-1])
    indices = np.empty(nnz, dtype=np.int32)
    data = np.empty(nnz, dtype=np.float64)
    ctx.interpolate_fetch(None, indices, data, None)
    perm = np.random.default_rng(DUMP_SEED).permutation(n_rows)
    k = min(n_rows, DUMP_ROWS)
    fixed = 8 * 8 + 6 * 256                 # totals, and six .npy headers (128 bytes each for 1-D arrays)
    while True:
        rows = np.sort(perm[:k])
        counts = (indptr[rows + 1] - indptr[rows]).astype(np.int64)
        if 16 * int(counts.sum()) + 24 * k + fixed <= DUMP_BYTES or k == 1:
            break
        k //= 2
    starts = indptr[rows].astype(np.int64)
    at = np.repeat(starts - (np.cumsum(counts) - counts), counts) + np.arange(int(counts.sum()))
    sums = np.zeros(4)                      # NaN count, nansum(data), nansum(|data|), nansum(data * (indices + 1))
    for b in range(0, nnz, DUMP_CHUNK):
        d, ix = data[b:b + DUMP_CHUNK], indices[b:b + DUMP_CHUNK]
        sums += [np.isnan(d).sum(), np.nansum(d), np.nansum(np.abs(d)), np.nansum(d * (ix + 1.0))]
    totals = [n_rows, n_cols, nnz, *sums, np.nansum(neumann)]
    out = {"rows": rows, "row_nnz": counts, "indices": indices[at], "data": data[at], "neumann": neumann[rows], "totals": totals}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    log(f"dumped {k} of {n_rows} rows ({int(counts.sum())} of {nnz} entries) to {out_dir}")


def timed_e2e_steps(I, plumb, method, steps, warmup):
    # warmup >= 2: the loop below holds the previous result while the next one is computed, so the pooled page-locked
    # output buffers ping-pong between two sets; both must exist before the clock starts (cudaHostAlloc of 2.5 GB ~ 1 s)
    def one():
        I.invalidate_inputs()
        return I.interpolate(VARIABLE, method)
    for _ in range(warmup):
        W, nv = one()
    plumb.barrier()
    I._ctx.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        W, nv = one()
    I._ctx.synchronize()
    dt = time.perf_counter() - t0
    plumb.barrier()
    # bytes actually copied per step, summed over the ranks (a GLS rank uploads the slice of the cell fields its
    # nodes read; with gather='host' a rank downloads its own rows, with gather='all' the whole CSR)
    h2d = plumb.sum(I.last_timings["h2d_input_bytes"])
    d2h = plumb.sum(I.last_timings["d2h_bytes"])
    nnz = W.nnz
    del W, nv
    return plumb.max(dt) / steps, int(h2d), int(d2h), nnz


def k4_breakdown(I, plumb, method):
    """The two collectives of the general (unplanned) path, timed alone on the device: counts + neumann all-gather,
    then the row-block all-gather-v (grouped in-place ncclBroadcast over NVLink)."""
    ctx = I._ctx
    I.set_gather("all")
    for _ in range(2):
        nnz = ctx.interpolate_count(method)
        ctx.interpolate_fetch(None, None, None, None)
    lo, hi = ctx.scalar("row_lo"), ctx.scalar("row_hi")
    ip = np.asarray(I.grid.esup_ptr)
    own = 12.0 * float(ip[hi] - ip[lo])          # upper bound of this rank's block (every esup entry kept)
    total = 12.0 * float(nnz)
    ms = plumb.max(ctx.timing_or("k4_gather"))
    recv = max(total - own, 0.0)
    return {"k4_gather_ms": ms, "k4_gather_counts_ms": plumb.max(ctx.timing_or("k4_gather_counts")),
            "nvlink_bytes_received_per_rank": recv, "nvlink_gbs_per_rank": recv / (ms * 1e-3) / 1e9 if ms > 0 else None,
            "note": "general two-pass path, collectives serialised after the kernels; the planned path needs no counts exchange"}


def roofline_block(I, method, kernel_ms, lo, hi, share_of, workload):
    nbytes, flops, n_proc = algorithmic_model(I, method, lo, hi)
    peak, peak_src = measured_peaks()
    achieved = nbytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    prof = profiled(WORKLOADS[workload][0] if workload in WORKLOADS else workload, method)
    traffic = prof["bytes"] * n_proc if "bytes" in prof else None
    out = {"bound": "hbm", "kernel": "k_gls_mf (largest size class)" if method == "gls" else f"k_{method}_tile",
           "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "traffic": traffic,
           "traffic_source": ("DRAM bytes per processed node of the committed `ncu --set full` capture of this kernel on the same mesh family "
                              "(profiles/roofline_traffic.json) x the processed nodes of the timed launch") if traffic is not None else None,
           "peak_source": peak_src, "algorithmic_bytes_per_launch": nbytes, "kernel_ms": kernel_ms, "processed_nodes_this_rank": n_proc}
    return out, flops, prof


def run_config(I, I_kwargs, comm, plumb, key, workload, methods, neumann_rate, steps):
    """A short run of another BASELINE config on the same GPUs (same Interpolator: one NCCL communicator per unique id):
    device-timed value + roofline + e2e per method."""
    kind, n, desc = WORKLOADS[workload]
    mesh = make_mesh(kind, n, neumann_rate)
    t0 = time.time()
    I.load_mesh(mesh_obj=mesh)
    t_load = time.time() - t0
    ctx, g = I._ctx, I.grid
    out = {"workload": desc + (f", neumann_rate={neumann_rate}" if neumann_rate != 0.5 else ""), "n_nodes": g.n_points,
           "n_cells": g.n_elems, "load_mesh_wall_s": t_load, "k1_device_ms": ctx.timing_or("k1"), "methods": {}}
    for mi, method in enumerate(methods):
        W, _ = I.interpolate(VARIABLE, method)
        nnz = W.nnz
        del W
        if comm.world > 1:
            I.set_gather("all")      # like the headline value: the step ends with the full CSR on every GPU
        r = timed_device_steps(I, plumb, method, steps, 3)
        I.set_gather(I_kwargs["gather"])
        lo, hi = ctx.scalar("row_lo"), ctx.scalar("row_hi")
        roof, _f, _p = roofline_block(I, method, r["kernel_ms"], lo, hi, (hi - lo) / max(g.n_points, 1), workload)
        m = {"value": g.n_points / (r["ms_per_step"] * 1e-3), "unit": "nodes/s", "ms_per_step": r["ms_per_step"],
             "kernel_ms": r["kernel_ms"], "nnz": nnz, "gpu_launches": r["launches"],
             "roofline": {k: roof[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "algorithmic_bytes_per_launch")}}
        e2e_s, h2d, d2h, _n = timed_e2e_steps(I, plumb, method, steps, 2)
        m["e2e"] = {"value": g.n_points / e2e_s, "unit": "nodes/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h}
        out["methods"][method] = m
    return out


def run_ours(args, rank, world):
    import ninpol_b200
    from ninpol_b200 import dist as nd
    kind, n, desc = WORKLOADS[args.workload]
    if args.n:
        n = args.n
        desc = f"{kind} n={n} (override)"
    plumb = Plumbing(rank, world)
    comm = nd.init_from_env() if world > 1 else nd.Comm(0, 1)
    t0 = time.time()
    mesh = make_mesh(kind, n)
    if rank == 0:
        log(f"mesh {desc}: generated in {time.time() - t0:.1f}s")
    e2e_gather = args.gather if world > 1 else "all"
    I_kwargs = {"gather": e2e_gather, "stream_chunks": args.stream_chunks}
    t0 = time.time()
    I = ninpol_b200.Interpolator(comm=comm, **I_kwargs)
    t_ctor = time.time() - t0
    t0 = time.time()
    I.load_mesh(mesh_obj=mesh)
    t_load = time.time() - t0
    ctx = I._ctx
    g = I.grid
    n_points, n_elems = g.n_points, g.n_elems
    host_phases = {k: round(I.last_timings.get(k, 0.0), 3) for k in ("load_mesh_process_s", "load_mesh_device_call_s", "load_mesh_data_s")}
    host_phases["constructor_s"] = round(t_ctor, 3)
    k1 = {k: ctx.timing_or(k) for k in ("k1", "k1_esup", "k1_esuel", "k1_faces", "k1_fsup", "k1_geom", "h2d_mesh")}
    if rank == 0:
        log(f"Interpolator() {t_ctor:.2f}s (CUDA context, NCCL communicator); load_mesh phases {host_phases}")
        log(f"load_mesh {t_load:.2f}s wall; device K1 {k1['k1']:.1f} ms (esup {k1['k1_esup']:.1f}, esuel {k1['k1_esuel']:.1f}, "
            f"faces {k1['k1_faces']:.1f}, fsup {k1['k1_fsup']:.1f}, geom {k1['k1_geom']:.1f}); H2D {k1['h2d_mesh']:.1f} ms")
    method = args.method
    try:
        W0, _ = I.interpolate(VARIABLE, method)      # stages the inputs, sets the partition
    except Exception as e:                          # /dev/shm too small on this box (every rank sees the same)
        if world > 1 and e2e_gather == "host" and "gather='host'" in str(e):
            e2e_gather = "all"
            I.set_gather("all")
            W0, _ = I.interpolate(VARIABLE, method)
        else:
            raise
    nnz = W0.nnz
    del W0
    warm = max(args.warmup, 3)
    sampler = ClockSampler(ctx.device) if rank == 0 else None
    # ---- value: device-timed, result on the device; N > 1: every rank ends up with the full CSR (NCCL gather), the
    #      step cut into 4 chunks per rank so that the gather of chunk k runs under the kernels of chunk k+1 ----
    dev_chunks = 1
    if world > 1:
        I.set_gather("all")
        dev_chunks = 4
    dev = timed_device_steps(I, plumb, method, args.steps, warm, sampler, chunks=dev_chunks)
    if args.dump_outputs and rank == 0:      # gather='all' above: rank 0 holds the whole result
        dump_outputs(I, args.dump_outputs)
    value = n_points / (dev["ms_per_step"] * 1e-3)
    lo, hi = ctx.scalar("row_lo"), ctx.scalar("row_hi")
    compute_only, k4, gather_after = None, None, None
    if world > 1:
        # the dominant kernel is timed on the un-chunked step (one launch per size class over the rank's whole range)
        ga = timed_device_steps(I, plumb, method, args.steps, 2, None, chunks=1)
        dev["kernel_ms"] = ga["kernel_ms"]
        gather_after = {"value": n_points / (ga["ms_per_step"] * 1e-3), "unit": "nodes/s", "ms_per_step": ga["ms_per_step"],
                        "note": "same step un-chunked: the NCCL gather starts after the last kernel (nothing overlaps it)"}
        k4 = k4_breakdown(I, plumb, method)
        I.set_gather("host")
        co = timed_device_steps(I, plumb, method, args.steps, 2)
        compute_only = {"value": n_points / (co["ms_per_step"] * 1e-3), "unit": "nodes/s", "ms_per_step": co["ms_per_step"],
                        "note": "same step with every row block left on the GPU that computed it (gather='host': no block crosses NVLink; "
                                "one 4-byte all-reduce per step tells every rank that no plan was voided)"}
    roof, flops, prof = roofline_block(I, method, dev["kernel_ms"], lo, hi, (hi - lo) / max(n_points, 1), args.workload)
    # ---- e2e through the public API, host buffers ----
    I.set_gather(e2e_gather)
    e2e_s, h2d, d2h, _n = timed_e2e_steps(I, plumb, method, args.steps, 2)
    e2e = {"value": n_points / e2e_s, "unit": "nodes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": e2e_s * 1e3,
           "api": (f"Interpolator({'comm=comm, gather=' + repr(e2e_gather) if world > 1 else ''}).interpolate(variable, method) after "
                   "invalidate_inputs() - the constructor's defaults: page-locked pooled outputs, inputs page-locked in place, 8 node chunks. "
                   "Per step: H2D of the flags (N > 1: of the slice of this rank's nodes; the ranks sum the slice checksums to learn that the resident row is unchanged) "
                   "and (GLS) of the permeability / diff_mag slices this rank's nodes read, kernels, D2H of the CSR; "
                   "uploads, kernels and downloads overlap chunk by chunk on separate streams. gather='host': every rank writes its rows into "
                   "one page-locked host mapping shared by the ranks (all PCIe links in parallel), one NCCL 1-int exchange closes the step; "
                   "gather='all': row blocks all-gathered over NCCL / NVLink, every rank downloads the whole CSR. Byte counts are sums over ranks.")}
    e2e_all = None
    if world > 1 and e2e_gather != "all":
        I.set_gather("all")
        s2, h2, d2, _n = timed_e2e_steps(I, plumb, method, max(2, args.steps // 4), 2)
        e2e_all = {"value": n_points / s2, "unit": "nodes/s", "ms_per_step": s2 * 1e3, "h2d_bytes_per_step": h2, "d2h_bytes_per_step": d2,
                   "api": "same, gather='all' (the constructor default): NCCL all-gather of the blocks, every rank returns the full CSR"}
        I.set_gather(e2e_gather)
    line = {
        "metric": f"node weights/sec ({method.upper()})", "value": value, "unit": "nodes/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": dev["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "method": method, "n_nodes": n_points, "n_cells": n_elems, "nnz": nnz,
                   "partition": f"nodes split into {world} contiguous cost-balanced ranges; mesh replicated; value: gather='all' (NCCL, "
                                f"4 chunks per rank so that the gather overlaps the kernels), e2e: gather='{e2e_gather}'" if world > 1 else "one GPU",
                   "cache": "inputs larger than L2 (working set >> 126 MB); no flush needed" if n_elems > 2_000_000 else
                            "small workload: L2-resident between iterations"},
        "step_ms_median": dev["step_ms_median"], "step_ms_best": dev["step_ms_best"],
        "e2e": e2e, "gpu_launches": dev["launches"], "clocks": dev["clocks"], "roofline": roof,
        "load_mesh": {"k1_device_ms": k1["k1"], "h2d_ms": k1["h2d_mesh"], "cells_per_s_device": n_elems / (k1["k1"] * 1e-3) if k1["k1"] else None,
                      "wall_s": plumb.max(t_load), "host_phases_s": host_phases, "breakdown_ms": k1,
                      "k1_roofline": {"bound": "hbm", "algorithmic_bytes": 292.0 * n_elems if kind == "tet" else None,
                                      "frac": (292.0 * n_elems / (k1["k1"] * 1e-3) / 1e9 / roof["peak"]) if (kind == "tet" and k1["k1"]) else None}},
    }
    if compute_only:
        line["device_compute_only"] = compute_only
        line["device_gather_after_kernels"] = gather_after
        line["k4"] = k4
    if e2e_all:
        line["e2e_gather_all"] = e2e_all
    if method == "gls":
        fp64_peak = ctx.measure_fp64_peak() if rank == 0 else 0.0
        ach_tf = flops / (dev["kernel_ms"] * 1e-3) / 1e12 if dev["kernel_ms"] > 0 else 0.0
        line["roofline"]["fp64"] = {
            "achieved_effective": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac_effective": ach_tf / fp64_peak if fp64_peak else None,
            "pipe_active": prof.get("counters", {}).get("fp64_pipe_active"), "warps_active": prof.get("counters", {}).get("warps_active"),
            "executed_mflop_per_node": prof.get("counters", {}).get("executed_mflop_per_node"),
            "flop_model": "EFFECTIVE rate: the dense one-RHS Householder model sum 2mn^2 - 2/3 n^3 + 4mn (m=E+3F+B, n=3E+1) divided by the time; the "
                          "multifrontal kernel executes ~10x fewer FLOPs than that model, so the pipe utilisation (pipe_active, from the committed "
                          "ncu capture) is the hardware-side figure",
            "peak_source": "measured live by this run: register-resident DFMA loop (npb_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
            "note": "GLS is bound by per-warp instruction latency, not HBM (SURVEY.md Q13); the HBM fraction is reported because the metric asks for it"}
    # ---- secondary methods on the same mesh (device-timed; the north star names IDW on this mesh) ----
    also = {}
    for m2 in [m for m in args.also.split(",") if m in ("idw", "ls", "gls") and m != method]:
        if world > 1:
            I.set_gather("host")     # rows stay on their owners: the step is this rank's kernels + the 1-int verdict exchange
        W2, _ = I.interpolate(VARIABLE, m2)
        del W2
        r2 = timed_device_steps(I, plumb, m2, args.steps, 3)
        roof2, _f, _p = roofline_block(I, m2, r2["kernel_ms"], lo, hi, (hi - lo) / max(n_points, 1), args.workload)
        step_bw = roof2["algorithmic_bytes_per_launch"] / (r2["ms_per_step"] * 1e-3) / 1e9
        also[m2] = {"value": n_points / (r2["ms_per_step"] * 1e-3), "unit": "nodes/s", "ms_per_step": r2["ms_per_step"],
                    "kernel_ms": r2["kernel_ms"], "gpu_launches": r2["launches"],
                    "roofline": {k: roof2[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "algorithmic_bytes_per_launch")},
                    "roofline_by_step_time": {"achieved": step_bw, "frac": step_bw / roof2["peak"],
                                              "note": "this rank's algorithmic bytes / the whole step (plan reuse, kernel, verdict) instead of the kernel alone"}}
        if world > 1:
            I.set_gather("all")
            r3 = timed_device_steps(I, plumb, m2, max(2, args.steps // 2), 2)
            also[m2]["with_nccl_gather"] = {"value": n_points / (r3["ms_per_step"] * 1e-3), "ms_per_step": r3["ms_per_step"],
                                            "note": "every rank ends with the full CSR: (world-1)/world of 12 B x nnz cross NVLink per rank"}
    if also:
        line["also"] = also
    I.set_gather(e2e_gather)
    # ---- the other BASELINE configs, short runs on the same GPUs ----
    if not args.no_configs:
        cfg = {}
        for key, wl, methods, rate in CONFIG_RUNS:
            if args.configs and key not in args.configs.split(","):
                continue
            try:
                cfg[key] = run_config(I, I_kwargs, comm, plumb, key, wl, methods, rate, args.config_steps)
            except Exception as e:   # a side run must never take the headline down
                cfg[key] = {"error": repr(e)}
            if rank == 0:
                log(f"config {key}: done")
        line["configs"] = cfg
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            base = time_reference(args.ref_workload, method, REF_REPEATS, 1)
            line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:  # the checker must never take the bench down
            line["cpu_baseline"] = {"value": None, "unit": "nodes/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}
    if rank == 0:
        emit(line)
    plumb.close()


_JSON_OUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else a library prints on fd 1 (NCCL's version
    banner, for one) was redirected to stderr in main()."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tet203", choices=sorted(WORKLOADS))
    ap.add_argument("--method", default="gls", choices=["gls", "idw", "ls"])
    ap.add_argument("--also", default="idw,ls", help="comma list of extra methods to time on the same mesh")
    ap.add_argument("--n", type=int, default=0, help="override the lattice size of the workload (debug)")
    ap.add_argument("--ref-workload", default=REF_WORKLOAD, choices=sorted(WORKLOADS),
                    help="what the reference arm / cpu_baseline time (default: config C2, Kuhn n=69)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the side runs of the other BASELINE configs")
    ap.add_argument("--configs", default="", help="comma list of config keys to run (default: all)")
    ap.add_argument("--config-steps", type=int, default=3)
    ap.add_argument("--gather", default="host", choices=["host", "all"],
                    help="N > 1, e2e: where the row blocks meet (host: shared host mapping; all: every GPU, over NCCL)")
    ap.add_argument("--stream-chunks", type=int, default=8, help="node chunks of the e2e pipeline (0 = plain count + fetch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="--impl ours: after the timed steps, write a seeded sample of the last step's result as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the result of this repository's arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            sys.exit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
