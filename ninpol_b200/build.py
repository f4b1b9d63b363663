"""Build recipe for libninpol_b200.so: explicit nvcc for sm_100a, in-tree output (the .so is
git-ignored but travels to the GPU box with the gpurun snapshot).

    python -m ninpol_b200.build [--force]

Bit-exact translation units (geometry, IDW/LS) are compiled with -fmad=false on top of their explicit
_rn intrinsics; everything carries -lineinfo so ncu's source page maps to the .cu files.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libninpol_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-ccbin", "/usr/bin/g++"]
EXTRA = os.environ.get("NPB_NVCC_EXTRA", "").split()   # experiments: e.g. -DLS_ECAP=1280 (use with --force)
UNITS = {
    "capi.cu": [],
    "scan.cu": [],
    "export.cu": [],
    "k1_connectivity.cu": [],
    "k1_geometry.cu": ["-fmad=false"],
    "k2_idw_ls.cu": ["-fmad=false"],
    "k2_idw_ls_tile.cu": ["-fmad=false"],
    "k2_gls.cu": [],
    "k2_gls_dense.cu": [],
    "k3_emit.cu": [],
    "k4_shard.cu": [],
    "pipeline.cu": [],
    "k5_apply.cu": ["-fmad=false"],
}


def _digest(paths, extra=()):
    """Content hash of the inputs of one build step.  Staleness is decided on content, not on mtimes: the
    gpurun snapshot does not preserve them, and a stale binary must never be tested against edited sources."""
    import hashlib
    h = hashlib.sha256()
    for p in sorted(paths):
        h.update(os.path.basename(p).encode())
        with open(p, "rb") as f:
            h.update(f.read())
    for e in extra:
        h.update(str(e).encode())
    return h.hexdigest()


def _stale(target, stamp_value):
    stamp = target + ".sha"
    if not os.path.exists(target) or not os.path.exists(stamp):
        return True
    with open(stamp) as f:
        return f.read().strip() != stamp_value


def _mark(target, stamp_value):
    with open(target + ".sha", "w") as f:
        f.write(stamp_value)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "ninpol_b200.h"))
    jobs = []
    objs = []
    stamps = []
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        cmd = [NVCC] + ARCH + COMMON + extra + EXTRA + ["-c", s, "-o", o]
        stamp = _digest([s] + headers, cmd)
        stamps.append(stamp)
        if force or _stale(o, stamp):
            jobs.append((cmd, o, stamp))

    def run(cmd):
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for " + cmd[-3])

    def compile_one(job):
        cmd, o, stamp = job
        run(cmd)
        _mark(o, stamp)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(compile_one, jobs))
    lib_stamp = _digest([], stamps)
    if jobs or force or _stale(LIB, lib_stamp):
        run([NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart", "-ldl", "-lpthread", "-ccbin", "/usr/bin/g++"])
        _mark(LIB, lib_stamp)
    return LIB


def is_current():
    """True when libninpol_b200.so was built from exactly the sources in the tree."""
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "ninpol_b200.h"))
    stamps = []
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        stamps.append(_digest([s] + headers, [NVCC] + ARCH + COMMON + extra + EXTRA + ["-c", s, "-o", o]))
    return not _stale(LIB, _digest([], stamps))


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
