"""ctypes binding of libninpol_b200.so (include/ninpol_b200.h).

This is the only way the Python host reaches the device; there is no PyTorch, no Triton and no CPU
fallback behind it: if the shared library is missing or no sm_100 GPU is usable, calls raise.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libninpol_b200.so")

METHOD_IDS = {"idw": 0, "ls": 1, "gls": 2}
UNIQUE_ID_BYTES = 128

_c_i64p = ctypes.POINTER(ctypes.c_int64)
_SIGNATURES = {
    "npb_version": (ctypes.c_int, []),
    "npb_last_error": (ctypes.c_char_p, []),
    "npb_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "npb_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "npb_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_comm_unique_id": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_comm_init": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "npb_set_partition": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]),
    "npb_set_gather": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "npb_comm_barrier": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_partition_elem_range": (ctypes.c_int, [ctypes.c_void_p, _c_i64p, _c_i64p]),
    "npb_set_cell_field_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]),
    "npb_load_mesh": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 9 + [ctypes.c_int]),
    "npb_load_mesh_strided": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int]
                              + [ctypes.c_void_p] * 8 + [ctypes.c_int]),
    "npb_grid_scalar": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, _c_i64p]),
    "npb_grid_array": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "npb_set_cell_field": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "npb_set_point_flags": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "npb_set_point_flags_f64": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "npb_set_point_flags_f64_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, _c_i64p]),
    "npb_interpolate_count": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, _c_i64p]),
    "npb_interpolate_fetch": (ctypes.c_int, [ctypes.c_void_p] * 5),
    "npb_interpolate_dense": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "npb_interpolate_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 6
                            + [ctypes.c_int64, _c_i64p, ctypes.POINTER(ctypes.c_int)]),
    "npb_interpolate_streamed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 6 + [ctypes.c_int64, _c_i64p]),
    "npb_apply": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "npb_apply_transpose": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "npb_timing": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double)]),
    "npb_launch_count": (ctypes.c_int, [ctypes.c_void_p, _c_i64p]),
    "npb_check_guards": (ctypes.c_int, [ctypes.c_void_p, _c_i64p, _c_i64p]),
    "npb_measure_fp64_peak": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "npb_measure_copy_bw": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_double)]),
    "npb_flush_l2": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    "npb_synchronize": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_timer_start": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_timer_stop": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "npb_host_alloc": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(ctypes.c_void_p)]),
    "npb_host_free": (ctypes.c_int, [ctypes.c_void_p]),
    "npb_host_register": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    "npb_host_unregister": (ctypes.c_int, [ctypes.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class NinpolB200Error(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen the in-tree shared library; fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NinpolB200Error(
                f"{LIB_PATH} not found: build it with `python -m ninpol_b200.build` (nvcc, sm_100a). "
                "ninpol_b200 has no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def check(rc):
    if rc != 0:
        msg = load_library().npb_last_error().decode("utf-8", "replace")
        raise NinpolB200Error(f"libninpol_b200 error {rc}: {msg}")


def device_count():
    n = ctypes.c_int(0)
    check(load_library().npb_device_count(ctypes.byref(n)))
    return n.value


def comm_unique_id():
    buf = ctypes.create_string_buffer(UNIQUE_ID_BYTES)
    check(load_library().npb_comm_unique_id(buf))
    return buf.raw


class Context:
    """One device context (one GPU, one stream)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.handle = ctypes.c_void_p()
        check(self.lib.npb_create(int(device), ctypes.byref(self.handle)))
        self.device = int(device)

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.npb_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- multi-GPU ---
    def comm_init(self, unique_id, rank, world):
        buf = ctypes.create_string_buffer(bytes(unique_id), UNIQUE_ID_BYTES)
        check(self.lib.npb_comm_init(self.handle, buf, int(rank), int(world)))

    def set_partition(self, bounds):
        b = np.ascontiguousarray(bounds, dtype=np.int64)
        check(self.lib.npb_set_partition(self.handle, _ptr(b), len(b)))

    def set_gather(self, mode):
        """'all': every rank receives the full CSR; 'root': rank 0 only, the others keep their row block."""
        check(self.lib.npb_set_gather(self.handle, {"all": 0, "root": 1, "host": 2}[mode]))

    def comm_barrier(self):
        check(self.lib.npb_comm_barrier(self.handle))

    def partition_elem_range(self):
        """Closed range of the element ids this rank's nodes touch (first > last when it owns no node)."""
        a, b = ctypes.c_int64(0), ctypes.c_int64(-1)
        check(self.lib.npb_partition_elem_range(self.handle, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    # --- K1 ---
    def load_mesh(self, dim, n_elems, n_points, conn, etype, npoel, nfael, lnofa, lpofa, nedel, lpoed, coords, build_edges):
        arrs = [np.ascontiguousarray(a, dtype=np.int64) for a in (conn, etype, npoel, nfael, lnofa, lpofa, nedel, lpoed)]
        coords = np.ascontiguousarray(coords, dtype=np.float64)
        assert arrs[0].ndim == 2 and arrs[0].shape[0] == n_elems and 1 <= arrs[0].shape[1] <= 8 and coords.shape == (n_points, 3)
        if arrs[0].shape[1] == 8:
            check(self.lib.npb_load_mesh(self.handle, int(dim), int(n_elems), int(n_points), *[_ptr(a) for a in arrs],
                                         _ptr(coords), int(bool(build_edges))))
        else:   # a single-type block as meshio holds it: [n_elems, nodes per element], no padding
            check(self.lib.npb_load_mesh_strided(self.handle, int(dim), int(n_elems), int(n_points), _ptr(arrs[0]),
                                                 int(arrs[0].shape[1]), *[_ptr(a) for a in arrs[1:]], _ptr(coords),
                                                 int(bool(build_edges))))

    def scalar(self, name):
        v = ctypes.c_int64(0)
        check(self.lib.npb_grid_scalar(self.handle, name.encode(), ctypes.byref(v)))
        return int(v.value)

    def array(self, name, shape, dtype):
        out = np.empty(shape, dtype=dtype)
        check(self.lib.npb_grid_array(self.handle, name.encode(), _ptr(out), out.nbytes))
        return out

    # --- per-variable inputs ---
    def set_cell_field(self, name, data):
        d = np.ascontiguousarray(data, dtype=np.float64).ravel()
        check(self.lib.npb_set_cell_field(self.handle, name.encode(), _ptr(d), d.size))

    def set_cell_field_range(self, name, data, first_elem, count):
        """`data` = the slice of the field that belongs to elements [first_elem, first_elem + count)."""
        d = np.ascontiguousarray(data, dtype=np.float64).ravel()
        per = 9 if name == "permeability" else 1
        assert d.size == per * count, (d.size, per, count)
        check(self.lib.npb_set_cell_field_range(self.handle, name.encode(), _ptr(d), int(first_elem), int(count)))

    def set_point_flags(self, flags):
        """int64 flags, or the float64 point-data row as it is (truncated on the device like `.astype(int)`)."""
        flags = np.asarray(flags)
        if flags.dtype == np.float64 and flags.flags.c_contiguous:
            check(self.lib.npb_set_point_flags_f64(self.handle, _ptr(flags), flags.size))
            return
        f = np.ascontiguousarray(flags, dtype=np.int64)
        check(self.lib.npb_set_point_flags(self.handle, _ptr(f), f.size))

    def set_point_flags_slice(self, flags, first, count):
        """Collective: upload flags[first:first + count] only (float64, contiguous); returns the checksum of the whole
        row summed over the ranks.  Equal to scalar('flags_checksum'): the resident row is still right."""
        part = flags[first:first + count]
        v = ctypes.c_int64(0)
        check(self.lib.npb_set_point_flags_f64_range(self.handle, _ptr(part) if count > 0 else None, int(first), int(count),
                                                     ctypes.byref(v)))
        return int(v.value)

    # --- K2 / K3 / K4 ---
    def interpolate_run(self, method, n_chunks, perm=None, diff_mag=None, indptr=None, indices=None, data=None, neumann=None):
        """Chunk pipeline over this rank's nodes (pipeline.cu).  Host arrays page-locked or None.  Returns
        (nnz, fell_back); fell_back = True (on every rank alike): nothing valid was written, run count + fetch."""
        nnz = ctypes.c_int64(0)
        fb = ctypes.c_int(0)
        cap = min(indices.size, data.size) if (indices is not None and data is not None) else 0
        check(self.lib.npb_interpolate_run(self.handle, METHOD_IDS[method], int(n_chunks), _ptr(perm), _ptr(diff_mag),
                                           _ptr(indptr), _ptr(indices), _ptr(data), _ptr(neumann), int(cap),
                                           ctypes.byref(nnz), ctypes.byref(fb)))
        return int(nnz.value), bool(fb.value)

    def interpolate_streamed(self, method, n_chunks, perm, diff_mag, indptr, indices, data, neumann):
        """Single-GPU pipeline with the internal two-pass fallback (pipeline.cu); all arrays page-locked."""
        nnz = ctypes.c_int64(0)
        check(self.lib.npb_interpolate_streamed(self.handle, METHOD_IDS[method], int(n_chunks),
                                                _ptr(perm) if perm is not None else None,
                                                _ptr(diff_mag) if diff_mag is not None else None,
                                                _ptr(indptr), _ptr(indices), _ptr(data), _ptr(neumann),
                                                int(min(indices.size, data.size)), ctypes.byref(nnz)))
        return int(nnz.value)

    def interpolate_dense(self, method, weights, neumann_ws):
        """The plug-in's dense outputs (weights [n_points, MX_ELEMENTS_PER_POINT], neumann_ws [n_points])."""
        assert weights.flags.c_contiguous and neumann_ws.flags.c_contiguous
        assert weights.dtype == np.float64 and neumann_ws.dtype == np.float64
        check(self.lib.npb_interpolate_dense(self.handle, METHOD_IDS[method], _ptr(weights), _ptr(neumann_ws)))

    def interpolate_count(self, method):
        nnz = ctypes.c_int64(0)
        check(self.lib.npb_interpolate_count(self.handle, METHOD_IDS[method], ctypes.byref(nnz)))
        return int(nnz.value)

    def interpolate_fetch(self, indptr, indices, data, neumann):
        check(self.lib.npb_interpolate_fetch(self.handle, _ptr(indptr), _ptr(indices), _ptr(data), _ptr(neumann)))

    def apply(self, method, values, out):
        """out[:] = W @ values with the CSR of `method` resident on the device (npb_apply).  values [n_elems, k] and
        out [n_points, k]: float64, C-contiguous (1-D: k = 1).  Collective when world > 1."""
        assert values.dtype == np.float64 and out.dtype == np.float64
        assert values.flags.c_contiguous and out.flags.c_contiguous
        k = 1 if values.ndim == 1 else int(values.shape[1])
        assert values.ndim in (1, 2) and out.ndim == values.ndim and out.shape[1:] == values.shape[1:]
        check(self.lib.npb_apply(self.handle, METHOD_IDS[method], _ptr(values), k, _ptr(out)))

    def apply_transpose(self, method, values, out):
        """out[:] = W.T @ values with the CSR of `method` resident on the device (npb_apply_transpose).  values
        [n_points, k] and out [n_elems, k]: float64, C-contiguous (1-D: k = 1).  One GPU only."""
        assert values.dtype == np.float64 and out.dtype == np.float64
        assert values.flags.c_contiguous and out.flags.c_contiguous
        k = 1 if values.ndim == 1 else int(values.shape[1])
        assert values.ndim in (1, 2) and out.ndim == values.ndim and out.shape[1:] == values.shape[1:]
        check(self.lib.npb_apply_transpose(self.handle, METHOD_IDS[method], _ptr(values), k, _ptr(out)))

    # --- measurement ---
    def timing(self, name):
        v = ctypes.c_double(0.0)
        check(self.lib.npb_timing(self.handle, name.encode(), ctypes.byref(v)))
        return float(v.value)

    def timing_or(self, name, default=0.0):
        v = ctypes.c_double(0.0)
        rc = self.lib.npb_timing(self.handle, name.encode(), ctypes.byref(v))
        return float(v.value) if rc == 0 else default

    def launch_count(self):
        v = ctypes.c_int64(0)
        check(self.lib.npb_launch_count(self.handle, ctypes.byref(v)))
        return int(v.value)

    def check_guards(self):
        """(guarded blocks, damaged blocks) — both 0 unless NPB_DEBUG_GUARDS=1 was set before the library's first use."""
        nb, nd = ctypes.c_int64(0), ctypes.c_int64(0)
        check(self.lib.npb_check_guards(self.handle, ctypes.byref(nb), ctypes.byref(nd)))
        return int(nb.value), int(nd.value)

    def measure_fp64_peak(self):
        v = ctypes.c_double(0.0)
        check(self.lib.npb_measure_fp64_peak(self.handle, ctypes.byref(v)))
        return float(v.value)

    def measure_copy_bw(self, nbytes=1 << 31):
        v = ctypes.c_double(0.0)
        check(self.lib.npb_measure_copy_bw(self.handle, int(nbytes), ctypes.byref(v)))
        return float(v.value)

    def flush_l2(self, nbytes=256 << 20):
        check(self.lib.npb_flush_l2(self.handle, int(nbytes)))

    def synchronize(self):
        check(self.lib.npb_synchronize(self.handle))

    def timer_start(self):
        check(self.lib.npb_timer_start(self.handle))

    def timer_stop(self):
        v = ctypes.c_double(0.0)
        check(self.lib.npb_timer_stop(self.handle, ctypes.byref(v)))
        return float(v.value)


class HostRegistration:
    """Keeps a numpy array page-locked in place (cudaHostRegister) for as long as this object lives."""

    def __init__(self, array):
        self.lib = load_library()
        self.array = array                       # keeps the memory alive
        self.ptr = ctypes.c_void_p(array.ctypes.data)
        check(self.lib.npb_host_register(self.ptr, array.nbytes))

    def release(self):
        if self.ptr is not None:
            self.lib.npb_host_unregister(self.ptr)
            self.ptr = None
            self.array = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class _PinnedOwner:
    """Owns one cudaHostAlloc block; numpy arrays made from it keep it alive through `.base`."""

    def __init__(self, nbytes, shape, dtype):
        self.lib = load_library()
        self.ptr = ctypes.c_void_p()
        check(self.lib.npb_host_alloc(int(nbytes), ctypes.byref(self.ptr)))
        self.__array_interface__ = {"shape": tuple(shape), "typestr": np.dtype(dtype).str,
                                    "data": (self.ptr.value, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr and self.ptr.value:
                self.lib.npb_host_free(self.ptr)
                self.ptr = ctypes.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype):
    """numpy array in page-locked host memory (full-rate PCIe copies); freed when the last view dies."""
    shape = (int(shape),) if np.ndim(shape) == 0 else tuple(int(x) for x in shape)
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    return np.asarray(_PinnedOwner(max(n, 1) * dtype.itemsize, shape, dtype))
