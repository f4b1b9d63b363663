"""Interpolator — drop-in for `ninpol.Interpolator` on one B200 (or one per process for multi-GPU).

Same constructor keywords, methods and attributes as the reference class
(ninpol/_interpolator/interpolator.pyx:35-670, interpolator.pxd:27-58):

    I = Interpolator(name="interpolator", logging=False, build_edges=False)
    I.load_mesh(mesh_obj=mesh)                       # or filename=... when meshio is installed
    W, neumann = I.interpolate("pressure", "gls")    # scipy CSR (n_nodes, n_elements), ndarray (n_nodes,)
    u_nodes = I.nodal_values("pressure", "gls")     # W @ u on the GPU, bit for bit; the weights stay resident
    g_cells = I.nodal_adjoint("pressure", "gls", g_nodes)   # W.T @ g on the GPU (one GPU), same weights, bit for bit
    I.supported_methods                              # {"gls": ..., "idw": ..., "ls": ...}

The host side only ingests the mesh object (vectorised numpy instead of the reference's per-item Python
loops, same outputs) and hands plain arrays to libninpol_b200.so through ctypes; connectivity,
geometry, the per-node weights and the CSR emit all run on the GPU.  There is no CPU fallback.
"""
import os
import struct
import pickle
import sys
import tempfile
import time

import numpy as np
import scipy.sparse as sp

from . import _capi
from . import dist as _dist
from . import element_tables as et
from .grid import Grid

DTYPE_I = np.int64
DTYPE_F = np.float64


class _Logger:
    """`[TYPE ] (HH:MM:SS) msg` lines like the reference Logger (logger.pyx:47-56); stdout only."""

    def __init__(self, name, logging=False):
        self.name, self.logging = name, logging

    def log(self, msg, kind="INFO"):
        if self.logging:
            print(f"[{kind:<5}] ({time.strftime('%H:%M:%S')}) {self.name}: {msg}", flush=True)


class _Method:
    """Host mirror of one interpolation plug-in (IDWInterpolation / LSInterpolation /
    GLSInterpolation).  `prepare` has the reference plug-in signature (idw.pxd:19-24, ls.pxd:20-25,
    gls.pxd:22-27): it fills the caller's dense zero-initialised `weights[n_target, MX_ELEMENTS_PER_POINT]`
    (column k of row p <-> esup[esup_ptr[p]+k]) and `neumann_ws[n_target]`."""

    def __init__(self, owner, method, logging=False):
        self._owner, self.method, self.logging = owner, method, logging
        self.logger = _Logger(method.upper(), logging)

    def prepare(self, grid, cells_data, points_data, faces_data, variable_to_index, variable, target_points,
                weights, neumann_ws):
        I = self._owner
        if grid is not I.grid:
            raise ValueError("this plug-in is bound to its Interpolator's grid")
        I._check_targets(target_points)
        n, mx = grid.n_points, grid.MX_ELEMENTS_PER_POINT
        w = np.asarray(weights)
        nw = np.asarray(neumann_ws)
        if w.shape != (n, mx) or nw.shape != (n,) or w.dtype != DTYPE_F or nw.dtype != DTYPE_F:
            raise ValueError(f"weights must be float64 [{n}, {mx}] and neumann_ws float64 [{n}] (interpolator.pyx:645-651)")
        I._weights_key = None              # the dense path below voids the resident CSR
        I._stage_inputs(self.method, variable, variable_to_index, cells_data, points_data)
        # the kernels' esup-indexed values go straight into the caller's dense rows (npb_interpolate_dense):
        # nothing is rebuilt from the zero-eliminated CSR
        wc = w if w.flags.c_contiguous else np.empty((n, mx), dtype=DTYPE_F)
        nc = nw if nw.flags.c_contiguous else np.empty(n, dtype=DTYPE_F)
        I._ctx.interpolate_dense(self.method, wc, nc)
        if wc is not w:
            w[...] = wc
        if nc is not nw:
            nw[...] = nc

    __call__ = prepare


class _PinnedPool:
    """Page-locked output buffers that are reused ONLY when nothing else refers to them any more.

    interpolate() hands out numpy views of cudaHostAlloc blocks (full-rate, overlappable device->host copies).  A
    block goes back into circulation when the arrays made from it - and the scipy matrix holding them - are gone,
    which the owner's reference count tells; as long as the caller keeps a result it is never overwritten, so the
    drop-in semantics of the reference (fresh arrays per call) hold while a loop that drops its previous result
    runs without allocating."""

    def __init__(self):
        self._blocks = {}   # name -> list of _PinnedOwner-backed base arrays

    def take(self, name, n, dtype):
        dtype = np.dtype(dtype)
        free = None
        for owner in self._blocks.setdefault(name, []):
            # references: the list, the loop variable and getrefcount's argument; a live view adds one.  A block more
            # than twice the request is not used: scipy copies index / data arrays that are views of a base more than
            # twice their size (sparse._sputils._prune_array), which would cost a full host copy per call
            if owner.dtype == dtype and n <= owner.size <= 2 * n + 64 and sys.getrefcount(owner) <= 3:
                if free is None or owner.size < free.size:
                    free = owner
        if free is None:
            free = _capi.pinned_empty(n + n // 16 + 16, dtype)
            # keep at most two idle generations per name: drop smaller unused blocks
            self._blocks[name] = [o for o in self._blocks[name] if sys.getrefcount(o) > 3 or n <= o.size <= 2 * n + 64][-3:]
            self._blocks[name].append(free)
        return free[:n]

    def clear(self):
        self._blocks = {}


class Interpolator:
    def __init__(self, name="interpolator", logging=False, build_edges=False, device=None, comm=None,
                 pinned_outputs=True, pin_inputs=True, gather="all", stream_chunks=8):
        # pinned_outputs=True (default): the CSR / neumann arrays returned by interpolate() are views of page-locked
        # blocks from a pool; a block is reused only once the caller has dropped every array made from it
        # (_PinnedPool), so results are never overwritten behind the caller's back.  False: plain numpy arrays.
        self.pinned_outputs = pinned_outputs
        self._pool = _PinnedPool()
        # pin_inputs=True (default): the per-variable host arrays (permeability, diff_mag, flags) are page-locked in
        # place (cudaHostRegister) the first time they are uploaded, so uploads run at the PCIe rate and overlap
        self.pin_inputs = pin_inputs
        self._registered = {}
        self._data_version = 0
        self.point_ordering = et.POINT_ORDERING
        self.is_grid_initialized = False
        self.build_edges = build_edges
        self.gls = _Method(self, "gls", logging)
        self.idw = _Method(self, "idw", logging)
        self.ls = _Method(self, "ls", logging)
        # same keys, same order as interpolator.pyx:60-64
        self.supported_methods = {"gls": self.gls.prepare, "idw": self.idw.prepare, "ls": self.ls.prepare}
        self.variable_to_index = {"points": {}, "cells": {}, "faces": {}}
        self.types_per_dimension = {k: list(v) for k, v in et.TYPES_PER_DIMENSION.items()}
        # per-variable rows; `cells_data` / `points_data` (the reference's [n_var, n*max_dim] arrays) are
        # materialised from them on first access — at 50M cells the dense form alone is >10 GB
        self._rows = {"cells": [], "points": []}
        self._dense = {"cells": np.zeros((1, 1), dtype=DTYPE_F), "points": np.zeros((1, 1), dtype=DTYPE_F)}
        self.cells_data_dimensions = np.zeros(1, dtype=DTYPE_I)
        self.points_data_dimensions = np.zeros(1, dtype=DTYPE_I)
        self.faces_data = np.zeros((1, 1), dtype=DTYPE_F)
        self.faces_data_dimensions = np.zeros(1, dtype=DTYPE_I)
        self.logging = logging
        self.logger = _Logger(name, logging)
        # the reference caches under tempfile.gettempdir() itself; a world-writable directory lets any user plant a
        # pickle, so the cache lives in a per-user 0700 directory below it (same file names inside)
        self.CACHE_PATH = self._private_cache_dir()
        self.mesh_obj = None
        self.grid = None
        self.points_coords = None
        # device side
        self.comm = comm if comm is not None else _dist.Comm(0, 1)
        if device is None:
            device = self.comm.local_rank if self.comm.world > 1 else 0
        self._ctx = _capi.Context(device)      # raises when the library or the GPU is missing
        # gather="all": every rank returns the full CSR; gather="root": rank 0 does, the other ranks
        # return the rows they own (other rows empty) and the blocks travel to rank 0 only;
        # gather="host": every rank copies its rows straight into one shared host mapping (/dev/shm), so the
        # full CSR assembles through all PCIe links at once and every rank returns views of it - valid
        # until any rank's next interpolate() / load_mesh()
        if gather not in ("all", "root", "host"):
            raise ValueError("gather must be 'all', 'root' or 'host'")
        self.gather = gather
        # stream_chunks=K > 0 (default 8): interpolate() runs as a pipeline over K chunks of this rank's nodes -
        # uploads of the GLS cell fields, the kernels, the NCCL gather and the downloads of the CSR blocks overlap
        # (npb_interpolate_run); results are bit-identical to the plain count + fetch path (stream_chunks=0)
        self.stream_chunks = int(stream_chunks)
        self.min_chunk_nodes = 200_000     # chunks only pay when each is long next to the launch / copy latencies
        # GLS uploads 80 B per cell and spends ~70 ns per node: its chunks pay from 50 k nodes on (2M-tet mesh: 27.9 ms in
        # one piece, 25.2 ms in six; profiles/r02_e2e_probe.log), and at 8 GPUs the two PCIe legs nothing hides get shorter
        self.min_chunk_nodes_gls = 50_000
        if self.comm.world > 1:
            self._ctx.comm_init(self.comm.unique_id, self.comm.rank, self.comm.world)
            self._ctx.set_gather(gather)
        self._staged = None
        self._pending_key = None
        self._partition_key = None
        self._flag_mask, self._flag_version, self._elem_range_key, self._elem_range = None, 0, None, (0, -1)
        self._shared, self._shared_reg, self._mesh_serial = None, None, 0
        # (method, variable, _data_version, _mesh_serial) of the CSR resident on the device, for nodal_values
        self._weights_key = None
        self.last_timings = {}

    def _dense_view(self, kind):
        if self._dense[kind] is None:
            rows = self._rows[kind]
            width = max(len(r) for r in rows) if rows else 1
            out = np.zeros((max(len(rows), 1), width), dtype=DTYPE_F)
            for i, r in enumerate(rows):
                out[i, :len(r)] = r
            self._dense[kind] = out
        return self._dense[kind]

    def _set_dense(self, kind, value):
        self._dense[kind] = value
        self._rows[kind] = list(value)
        self._data_version += 1      # whatever is resident on the device no longer matches
        self._staged = None

    cells_data = property(lambda self: self._dense_view("cells"), lambda self, v: self._set_dense("cells", v))
    points_data = property(lambda self: self._dense_view("points"), lambda self, v: self._set_dense("points", v))

    # ------------------------------------------------------------------------------------------
    # cache helpers (interpolator.pyx:93-111) — inputs-only pickle cache, file meshes only
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _private_cache_dir():
        uid = os.getuid() if hasattr(os, "getuid") else 0
        path = os.path.join(tempfile.gettempdir(), f"ninpol_b200-{uid}")
        try:
            os.makedirs(path, mode=0o700, exist_ok=True)
            st = os.stat(path)
            if (hasattr(os, "getuid") and st.st_uid != uid) or (st.st_mode & 0o077):
                os.chmod(path, 0o700)          # raises when the directory is somebody else's
                if os.stat(path).st_uid != uid:
                    raise PermissionError(path)
        except OSError:
            path = tempfile.mkdtemp(prefix="ninpol_b200-")   # private by construction
        return path

    @staticmethod
    def _source_stamp(filename):
        st = os.stat(filename)
        return (int(st.st_size), int(st.st_mtime_ns))

    def is_cached(self, filename):
        """Path of the cache of `filename` (interpolator.pyx:93-102: <basename><hex(size)>.pkl), or None.  The name
        alone does not identify a mesh (two files of equal name and size): the cache also records the source's size and
        modification time and is ignored when they differ."""
        if filename == "":
            return None
        little_hash = hex(os.path.getsize(filename))
        cache_name = filename.split(os.path.sep)[-1].split(".")[0] + little_hash + ".pkl"
        final_path = os.path.join(self.CACHE_PATH, cache_name)
        return final_path if os.path.exists(final_path) else None

    # ------------------------------------------------------------------------------------------
    # load_mesh (interpolator.pyx:168-252)
    # ------------------------------------------------------------------------------------------
    def load_mesh(self, filename="", mesh_obj=None):
        if filename == "" and mesh_obj is None:
            raise ValueError("Filename for the mesh or meshio.Mesh object must be provided.")
        t_begin = time.time()
        cached = self.is_cached(filename)
        cache = None
        if cached:
            with open(cached, "rb") as f:
                cache = pickle.load(f)
            if cache.get("source_stamp") != self._source_stamp(filename) or \
                    cache.get("source_path") != os.path.abspath(filename):
                cache, cached = None, None       # another file of the same name and size: rebuild
        if cached:
            self.logger.log("Loading mesh from cache")
            args = cache["grid"]
            ic = cache["interpolator"]
            self._set_dense("cells", ic["cells_data"])
            self._set_dense("points", ic["points_data"])
            self.cells_data_dimensions, self.points_data_dimensions = ic["cells_data_dimensions"], ic["points_data_dimensions"]
            self.faces_data, self.faces_data_dimensions = ic["faces_data"], ic["faces_data_dimensions"]
            self.variable_to_index, self.points_coords = ic["variable_to_index"], ic["points_coords"]
        else:
            if filename != "":
                self.logger.log(f"Reading mesh from {filename}")
                try:
                    import meshio
                except ImportError as e:
                    raise ImportError("reading mesh files needs the `meshio` package; pass mesh_obj= instead") from e
                self.mesh_obj = meshio.read(filename)
            else:
                self.logger.log("Using mesh object")
                self.mesh_obj = mesh_obj
            # a mesh file is cached with the reference's padded [n_elems, 8] table (make_cache); a mesh object
            # with a single cell block of the mesh's dimension goes to the device as it is
            args = self.process_mesh(self.mesh_obj, padded=(filename != ""))
            self.points_coords = np.asarray(self.mesh_obj.points, dtype=DTYPE_F)
        dim, n_elems, n_points, npoel, nfael, lnofa, lpofa, nedel, lpoed, connectivity, element_types = args[:11]
        coords = np.asarray(self.points_coords, dtype=DTYPE_F)
        if coords.shape[1] != 3:
            # the reference keeps 2-column coordinates as they are (grid.pyx:661-667) and then reads a
            # third column out of bounds in LS/GLS; the device layout is [n,3], zero padded
            c3 = np.zeros((coords.shape[0], 3), dtype=DTYPE_F)
            c3[:, :coords.shape[1]] = coords
            coords = c3
        t0 = time.time()
        self.last_timings["load_mesh_process_s"] = t0 - t_begin
        self._ctx.load_mesh(dim, n_elems, n_points, connectivity, element_types, npoel, nfael, lnofa, lpofa, nedel,
                            lpoed, coords, self.build_edges)
        self.last_timings["load_mesh_device_call_s"] = time.time() - t0
        self.grid = Grid(self._ctx, (npoel, nfael, lnofa, lpofa, nedel, lpoed), self.logging, self.build_edges)
        self.logger.log(f"Grid built in {time.time() - t0:.2f} seconds")
        self.last_timings["load_mesh_device_ms"] = self._ctx.timing_or("k1")
        self.last_timings["load_mesh_h2d_ms"] = self._ctx.timing_or("h2d_mesh")
        if not cached:
            t0 = time.time()
            self.variable_to_index = {"points": {}, "cells": {}, "faces": {}}
            if self.mesh_obj.cell_data:
                self.load_cell_data()
            else:
                self._set_dense("cells", np.zeros((1, 1), dtype=DTYPE_F))
                self.cells_data_dimensions = np.zeros(1, dtype=DTYPE_I)
            if self.mesh_obj.point_data:
                self.load_point_data()
            else:
                self._set_dense("points", np.zeros((1, 1), dtype=DTYPE_F))
                self.points_data_dimensions = np.zeros(1, dtype=DTYPE_I)
            self.logger.log(f"Data loaded in {time.time() - t0:.2f} seconds")
            self.last_timings["load_mesh_data_s"] = time.time() - t0
        self.is_grid_initialized = True
        self._pool.clear()        # blocks sized for the previous mesh (results still held by the caller stay alive)
        for reg in self._registered.values():
            reg.release()
        self._registered = {}
        self._staged = None
        self._pending_key = None
        self._data_version += 1
        self._partition_key = None
        self._shared, self._shared_reg = None, None      # gather="host": a new mapping per mesh
        self._mesh_serial += 1
        self._weights_key = None
        self.logger.log(f"Mesh loaded successfully: {n_points} points and {n_elems} elements.")
        if not cached and filename != "":
            little_hash = hex(os.path.getsize(filename))
            pkl_name = filename.split(os.path.sep)[-1].split(".")[0] + little_hash + ".pkl"
            final_path = os.path.join(self.CACHE_PATH, pkl_name)
            payload = self.make_cache(args)
            payload["source_stamp"] = self._source_stamp(filename)
            payload["source_path"] = os.path.abspath(filename)
            with open(final_path, "wb") as f:
                pickle.dump(payload, f)
            self.logger.log(f"Caching grid to {final_path}")

    def make_cache(self, args):
        return {"grid": tuple(args),
                "interpolator": {"cells_data": np.asarray(self.cells_data),
                                 "cells_data_dimensions": np.asarray(self.cells_data_dimensions),
                                 "points_data": np.asarray(self.points_data),
                                 "points_data_dimensions": np.asarray(self.points_data_dimensions),
                                 "faces_data": np.asarray(self.faces_data),
                                 "faces_data_dimensions": np.asarray(self.faces_data_dimensions),
                                 "variable_to_index": self.variable_to_index,
                                 "points_coords": np.asarray(self.points_coords)}}

    # ------------------------------------------------------------------------------------------
    # process_mesh (interpolator.pyx:255-369), vectorised
    # ------------------------------------------------------------------------------------------
    def process_mesh(self, mesh, padded=True):
        """Same tuple as the reference's process_mesh.  padded=False (internal): a mesh with ONE cell block of
        its dimension keeps that block's [n_elems, nodes-per-element] array instead of the -1 padded
        [n_elems, 8] copy (npb_load_mesh_strided takes it as it is)."""
        dim = 1
        for blk in mesh.cells:
            for dimension, names in self.types_per_dimension.items():
                if blk.type in names:
                    dim = max(dim, dimension)
        tables = et.tables_for_dim(dim, self.point_ordering)
        blocks = [b for b in mesh.cells if b.type in self.types_per_dimension[dim]]
        n_elems = int(sum(len(b.data) for b in blocks))
        n_points = int(np.asarray(mesh.points).shape[0])
        if not padded and len(blocks) == 1 and np.asarray(blocks[0].data).ndim == 2 and n_elems > 0:
            connectivity = np.ascontiguousarray(blocks[0].data, dtype=DTYPE_I)
            element_types = np.full(n_elems, self.point_ordering["elements"][blocks[0].type]["element_type"], dtype=DTYPE_I)
            return (dim, n_elems, n_points) + tuple(tables) + (connectivity, element_types, self.logging, self.build_edges)
        connectivity = -np.ones((n_elems, et.MAX_POINTS_PER_ELEMENT), dtype=DTYPE_I)
        element_types = -np.ones(n_elems, dtype=DTYPE_I)
        at = 0
        for b in blocks:
            d = np.asarray(b.data)
            connectivity[at:at + len(d), :d.shape[1]] = d
            element_types[at:at + len(d)] = self.point_ordering["elements"][b.type]["element_type"]
            at += len(d)
        return (dim, n_elems, n_points) + tuple(tables) + (connectivity, element_types, self.logging, self.build_edges)

    # ------------------------------------------------------------------------------------------
    # load_data / load_cell_data / load_point_data (interpolator.pyx:372-454), vectorised
    # ------------------------------------------------------------------------------------------
    def load_data(self, data_dict, data_type):
        """Row i of cells_data / points_data = variable i flattened (vectors item-major), zero padded to
        n_items * max_dim — same content as the reference's per-item Python loops (:403-419)."""
        n_items = self.grid.n_elems if data_type == "cells" else self.grid.n_points
        dims = np.zeros(len(data_dict), dtype=DTYPE_I)
        rows = [None] * len(data_dict)
        for index, variable in enumerate(data_dict):
            a = np.asarray(data_dict[variable])
            cur = a.shape[1] if a.ndim > 1 else 1
            self.variable_to_index[data_type][variable] = index
            dims[index] = cur
            if cur == 1:
                r = a[:n_items] if a.ndim == 1 else a[:n_items, 0]
            else:
                r = a[:n_items].reshape(-1)
            rows[index] = np.ascontiguousarray(r, dtype=DTYPE_F)
        kind = "cells" if data_type == "cells" else "points"
        self._rows[kind] = rows
        self._dense[kind] = None
        self._data_version += 1
        self._staged = None
        if data_type == "cells":
            self.cells_data_dimensions = dims
        else:
            self.points_data_dimensions = dims

    def _cell_data_by_type(self):
        """What `mesh_obj.cell_data_dict` holds (variable -> {cell type -> values}, types in first-appearance order,
        blocks of one type concatenated in block order), built from `cell_data` / `cells` without copying the array
        of a type that has a single block - meshio's property concatenates unconditionally, 4 GB at 50M cells."""
        mesh = self.mesh_obj
        blocks = getattr(mesh, "cells", None)
        cd = getattr(mesh, "cell_data", None)
        if blocks is None or not isinstance(cd, dict) or any(len(v) != len(blocks) for v in cd.values()):
            return mesh.cell_data_dict
        out = {}
        for variable, per_block in cd.items():
            by_type = {}
            for values, blk in zip(per_block, blocks):
                by_type.setdefault(blk.type, []).append(np.asarray(values))
            out[variable] = {t: (v[0] if len(v) == 1 else np.concatenate(v)) for t, v in by_type.items()}
        return out

    def load_cell_data(self):
        dim = self.grid.dim
        cell_data_dict = self._cell_data_by_type()
        cell_data = {}
        for variable in cell_data_dict:
            parts = [np.asarray(v) for t, v in cell_data_dict[variable].items() if t in self.types_per_dimension[dim]]
            # one block of the mesh's dimension (the common case): no copy of the user's array
            cell_data[variable] = parts[0] if len(parts) == 1 else (np.concatenate(parts) if parts else np.zeros(0))
            if variable == "permeability":
                cell_data["diff_mag"] = self.compute_diffusion_magnitude(cell_data["permeability"])
        self.load_data(cell_data, "cells")

    def load_point_data(self):
        self.load_data(self.mesh_obj.point_data, "points")

    def load_face_data(self, data_dict, face_connectivity=None):
        """interpolator.pyx:456-499 (scalar face data; optional remap through a user inpofa)."""
        n_faces = self.grid.n_faces
        face_to_grid = np.arange(n_faces, dtype=DTYPE_I)
        if face_connectivity is not None and len(face_connectivity) > 0 and np.asarray(face_connectivity).size > 0:
            A = np.ascontiguousarray(face_connectivity, dtype=DTYPE_I)
            B = np.ascontiguousarray(self.grid.inpofa, dtype=DTYPE_I)
            Av = A.view([("", A.dtype)] * A.shape[1]).ravel()
            Bv = B.view([("", B.dtype)] * B.shape[1]).ravel()
            order = np.argsort(Bv)
            face_to_grid = order[np.searchsorted(Bv[order], Av)]
        self.faces_data = np.zeros((len(data_dict), n_faces), dtype=DTYPE_F)
        self.faces_data_dimensions = np.zeros(len(data_dict), dtype=DTYPE_I)
        for i, variable in enumerate(data_dict):
            a = np.asarray(data_dict[variable])
            self.variable_to_index["faces"][variable] = i
            self.faces_data_dimensions[i] = a.shape[1] if a.ndim > 1 else 1
            self.faces_data[i] = a[face_to_grid].astype(DTYPE_F).reshape(n_faces, -1)[:, 0]

    @staticmethod
    def compute_diffusion_magnitude(permeability):
        """interpolator.pyx:501-509 as the RELEASE build evaluates it: `1 / 3` is C integer division
        (cdivision=True, setup.py:100-108), so det**0 == 1 and diff_mag = (1 - 3/tr K)^2 (SURVEY.md Q2).
        Element-wise, so large arrays are cut into slabs for a few threads (numpy releases the GIL): same values."""
        Ks = np.reshape(np.asarray(permeability, dtype=DTYPE_F), (len(permeability), 9))

        def slab(a, b):
            trKs = (Ks[a:b, 0] + Ks[a:b, 4]) + Ks[a:b, 8]          # np.trace order
            # 3 * det**0 == 3.0 exactly for every det (numpy: x**0 == 1, NaN and inf included)
            return (1 - (3.0 / trKs)) ** 2

        n = len(Ks)
        if n < (1 << 21):
            return slab(0, n)
        from concurrent.futures import ThreadPoolExecutor
        workers = max(1, min(8, os.cpu_count() or 1))
        step = -(-n // (4 * workers))
        out = np.empty(n, dtype=DTYPE_F)

        def run(a):
            out[a:a + step] = slab(a, min(n, a + step))

        with ThreadPoolExecutor(max_workers=workers) as ex:
            list(ex.map(run, range(0, n, step)))
        return out

    def get_dict(self):
        return {"point_ordering": self.point_ordering, "variable_to_index": self.variable_to_index,
                "cells_data": np.asarray(self.cells_data),
                "cells_data_dimensions": np.asarray(self.cells_data_dimensions),
                "points_data": np.asarray(self.points_data),
                "points_data_dimensions": np.asarray(self.points_data_dimensions)}

    def get_data(self, data_type, index, variable):
        kind = "cells" if data_type == "cells" else "points"
        if variable not in self.variable_to_index[kind]:
            raise ValueError(f"Variable '{variable}' not found in {kind} data.")
        src = self.cells_data if kind == "cells" else self.points_data
        return np.asarray(src[self.variable_to_index[kind][variable]])[index]

    # ------------------------------------------------------------------------------------------
    # interpolate (interpolator.pyx:549-629)
    # ------------------------------------------------------------------------------------------
    def _check_targets(self, target_points):
        n = self.grid.n_points
        tp = np.asarray(target_points)
        if len(tp) == 0:
            return
        if len(tp) != n or not np.array_equal(tp, np.arange(n)):
            # the reference indexes a (n_target, n_elems) matrix with global point ids and raises
            # ValueError from scipy for every strict subset (SURVEY.md Q6)
            raise ValueError("target_points subsets are not supported: the reference builds an inconsistent "
                             "(n_target, n_elems) matrix for them and fails in scipy; pass all nodes or nothing")

    def _stage_inputs(self, method, variable, variable_to_index, cells_data, points_data, defer_fields=False):
        """Uploads what the plug-in of `method` reads for `variable` (idw.pyx:27-28, ls.pyx:28-29,
        gls.pyx:47-59).  Missing names raise KeyError like the reference's dict lookups.
        defer_fields: the pipeline uploads permeability / diff_mag itself, slice by slice; returns them."""
        g = self.grid
        # resident inputs are identified by a data-version counter (bumped by load_mesh / load_data / the
        # cells_data / points_data setters), not by object identity
        own = cells_data is self._rows["cells"] and points_data is self._rows["points"]
        key = (method == "gls", variable, self._data_version) if own else None
        if method == "gls":
            permeability_index = variable_to_index["cells"]["permeability"]
            diff_mag_index = variable_to_index["cells"]["diff_mag"]
            flag_index = variable_to_index["points"]["neumann_flag_" + variable]
            variable_to_index["points"]["neumann_" + variable]   # looked up (KeyError) but dead (SURVEY.md Q3)
        else:
            flag_index = variable_to_index["points"]["neumann_flag_" + variable]
        if key is not None and self._staged == key:
            return None
        self._staged = None
        flags = np.asarray(points_data[flag_index])[:g.n_points]
        if flags.dtype == DTYPE_F and flags.flags.c_contiguous:
            flags = self._maybe_pin("neumann_flag", flags)     # truncated like .astype(int) on the device
        else:
            flags = flags.astype(DTYPE_I)
        h2d = None
        if (self.comm.world > 1 and flags.dtype == DTYPE_F and self._flag_mask is not None
                and self._partition_key == (method == "gls", self._flag_version, self._mesh_serial)):
            # a flag row is resident and the node ranges cut for it are current: upload only the slice of the nodes this
            # rank owns; the ranks add up the checksums of their slices.  Equal to the resident row's: it IS the resident
            # row, and the partition, the row plan and the other ranks' slices on this device all stand.
            lo, hi = int(self.partition_bounds[self.comm.rank]), int(self.partition_bounds[self.comm.rank + 1])
            if (self._ctx.set_point_flags_slice(flags, lo, hi - lo), int(flags.shape[0])) == self._flag_mask:
                h2d = (hi - lo) * flags.itemsize
        if h2d is None:
            self._ctx.set_point_flags(flags)
            h2d = flags.nbytes
        self._flags_host = flags
        if self.comm.world > 1 and h2d == flags.nbytes:
            # the node ranges depend on WHICH nodes are flagged (skipped nodes cost nothing): re-cut them only when that
            # set changed - cutting is a few numpy passes over all nodes, 150 ms at 8.5M nodes.  The flag kernel folds
            # the set into a 64-bit checksum on the device, so the test costs no pass over the array either.
            checksum = (self._ctx.scalar("flags_checksum"), int(flags.shape[0]))
            if checksum != self._flag_mask:
                self._flag_mask = checksum
                self._flag_version += 1
        self._set_partition(method)
        fields = None
        if method == "gls":
            perm = np.ascontiguousarray(np.asarray(cells_data[permeability_index])[:g.n_elems * 9], dtype=DTYPE_F)
            dm = np.ascontiguousarray(np.asarray(cells_data[diff_mag_index])[:g.n_elems], dtype=DTYPE_F)
            perm, dm = self._maybe_pin("permeability", perm, defer_fields), self._maybe_pin("diff_mag", dm, defer_fields)
            if defer_fields and self._is_registered("permeability", perm) and self._is_registered("diff_mag", dm):
                # the pipeline uploads them slice by slice, overlapped with the kernels; the key is set by the
                # caller once that call has succeeded
                self._pending_key = key
                self.last_timings["h2d_input_bytes"] = h2d    # + the slices, added by the pipeline
                return perm, dm
            if self.comm.world > 1:
                # a rank's nodes read the cell fields of the elements in their own esup rows only
                first, last = self._ctx.partition_elem_range()
                cnt = max(0, last - first + 1)
                self._ctx.set_cell_field_range("permeability", perm[9 * first:9 * (first + cnt)], first, cnt)
                self._ctx.set_cell_field_range("diff_mag", dm[first:first + cnt], first, cnt)
                h2d += 80 * cnt
            else:
                self._ctx.set_cell_field("permeability", perm)
                self._ctx.set_cell_field("diff_mag", dm)
                h2d += perm.nbytes + dm.nbytes
        self.last_timings["h2d_input_bytes"] = h2d
        self._staged = key                 # only now: every upload has succeeded
        self._pending_key = None
        return fields

    def _is_registered(self, name, arr):
        reg = self._registered.get(name)
        return reg is not None and reg.array is not None and reg.array.ctypes.data == arr.ctypes.data

    def _maybe_pin(self, name, arr, force=False):
        if not self.pin_inputs or (arr.nbytes < (8 << 20) and not force) or arr.nbytes == 0:
            return arr
        reg = self._registered.get(name)
        if reg is None or reg.array is None or reg.array.ctypes.data != arr.ctypes.data or reg.array.nbytes != arr.nbytes:
            if reg is not None:
                reg.release()
            try:
                self._registered[name] = _capi.HostRegistration(arr)
            except _capi.NinpolB200Error:
                self._registered.pop(name, None)     # not registrable (e.g. read-only mapping): staged copy
        return arr

    def set_gather(self, gather):
        """Switch between gather="all" and gather="root" on a live communicator (see __init__)."""
        if gather not in ("all", "root", "host"):
            raise ValueError("gather must be 'all', 'root' or 'host'")
        self.gather = gather
        self._weights_key = None           # npb_set_gather voids the resident CSR
        if self.comm.world > 1:
            self._ctx.set_gather(gather)

    def _shared_outputs(self):
        """The shared host mapping of gather="host" for the current mesh (created collectively on first use)."""
        if self._shared is not None:
            return self._shared
        g = self.grid
        token = bytes(self.comm.unique_id) + struct.pack("<q", self._mesh_serial)
        so = _dist.SharedOutputs(token, g.n_points, self._ctx.scalar("len_esup"))
        if not _dist.SharedOutputs.fits(so.nbytes):
            raise _capi.NinpolB200Error(f"gather='host' needs {so.nbytes >> 20} MiB in {so.DIR}; use gather='root'")
        if self.comm.rank == 0:
            so.create()
        self._ctx.comm_barrier()
        if self.comm.rank != 0:
            so.attach()
        self._ctx.comm_barrier()
        if self.comm.rank == 0:
            so.unlink()                     # the mapping lives on; the name is gone
        try:
            self._shared_reg = _capi.HostRegistration(so.buf)   # page-lock this process's view: full-rate DMA
        except _capi.NinpolB200Error:
            self._shared_reg = None
        self._shared = so
        return so

    def _ctx_has_fields(self):
        return self._ctx.scalar("have_cell_fields") != 0

    def invalidate_inputs(self):
        """Forget which per-variable inputs are resident on the device: the next interpolate() uploads
        the flags (and, for GLS, permeability + diff_mag) again from host memory, and nodal_values() / nodal_adjoint()
        recompute the weights."""
        self._staged = None
        self._weights_key = None

    def _set_partition(self, method):
        if self.comm.world == 1:
            return
        key = (method == "gls", self._flag_version, self._mesh_serial)
        if self._partition_key == key:
            return
        g = self.grid
        E = np.diff(np.asarray(g.esup_ptr))
        processed = ~((np.asarray(g.boundary_points) != 0) & (self._flags_host.astype(DTYPE_I) == 0))
        bounds = _dist.partition_nodes(_dist.node_cost(method, E, processed), self.comm.world)
        self._ctx.set_partition(bounds)
        self._partition_key = key
        self.partition_bounds = bounds

    def _out(self, name, n, dtype):
        if not self.pinned_outputs:
            return np.empty(n, dtype=dtype)
        return self._pool.take(name, n, dtype)

    def _run_pipeline(self, method, fields, fetch=True):
        """npb_interpolate_run: plan, then chunks of this rank's nodes through upload / compute / gather / download
        streams.  Returns None when the plan was voided (an exact-zero weight somewhere): the caller falls back to the
        two-pass path - every rank takes the same decision.  fetch=False: the CSR stays on the device (one GPU);
        returns its nnz."""
        g, ctx = self.grid, self._ctx
        n_points, cap = g.n_points, max(1, ctx.scalar("len_esup"))
        perm, dm = fields if fields is not None else (None, None)
        world = self.comm.world
        # every rank must cut the same number of chunks (the NCCL gather is chunked alike): the rule uses global sizes
        rule = min(self.min_chunk_nodes, self.min_chunk_nodes_gls) if method == "gls" else self.min_chunk_nodes
        chunks = max(1, min(self.stream_chunks, n_points // (max(1, rule) * world)))
        if not fetch:
            nnz, fell_back = ctx.interpolate_run(method, chunks, perm, dm)
            if fell_back:
                return None
            if perm is not None:
                self.last_timings["h2d_input_bytes"] += perm.nbytes + dm.nbytes
            self.last_timings.update({"streamed_ms": ctx.timing_or("streamed"), "nnz": nnz})
            return nnz
        if world > 1 and self.gather == "host":
            so = self._shared_outputs()
            ctx.comm_barrier()        # every rank is done with the arrays of the previous call
            pinned = self._shared_reg is not None
            arrays = (so.indptr, so.indices, so.data, so.neumann)
        else:
            arrays = (self._out("indptr", n_points + 1, np.int32), self._out("indices", cap, np.int32),
                      self._out("data", cap, np.float64), self._out("neumann", n_points, np.float64))
            pinned = self.pinned_outputs
        if pinned:
            nnz, fell_back = ctx.interpolate_run(method, chunks, perm, dm, *arrays)
        else:                         # pageable outputs: device-resident run, then the staged copies of fetch
            nnz, fell_back = ctx.interpolate_run(method, chunks, perm, dm)
            if not fell_back:
                ctx.interpolate_fetch(*arrays)
        if fell_back:
            return None
        indptr, indices, data, neumann = arrays
        if world > 1 and self.gather == "host":
            lo, hi = int(self.partition_bounds[self.comm.rank]), int(self.partition_bounds[self.comm.rank + 1])
            self.last_timings["d2h_bytes"] = 12 * int(so.indptr[hi] - so.indptr[lo]) + 12 * (hi - lo)   # this rank's rows
            out = (so.exact("indptr", n_points + 1), so.exact("indices", nnz), so.exact("data", nnz), so.exact("neumann", n_points))
        else:
            self.last_timings["d2h_bytes"] = indptr.nbytes + neumann.nbytes + 12 * nnz
            out = (indptr, indices[:nnz], data[:nnz], neumann)
        if perm is not None:
            if world > 1:
                if self._elem_range_key != self._partition_key:      # byte accounting only: one reduction per partition
                    self._elem_range, self._elem_range_key = ctx.partition_elem_range(), self._partition_key
                first, last = self._elem_range
                self.last_timings["h2d_input_bytes"] += 80 * max(0, last - first + 1)
            else:
                self.last_timings["h2d_input_bytes"] += perm.nbytes + dm.nbytes
        self.last_timings.update({"streamed_ms": ctx.timing_or("streamed"), "nnz": nnz})
        return out

    def _run(self, method, fetch=True):
        g = self.grid
        self._set_partition(method)
        if not fetch:
            # the two-pass count only: the rows stay on the device (world > 1: the ranks exchange row counts and
            # neumann entries, no CSR block); npb_apply writes them if the count left them unwritten
            nnz = self._ctx.interpolate_count(method)
            t = self._ctx.timing_or
            self.last_timings.update({"k2_ms": t("k2"), "k3_count_ms": t("k3_count"), "nnz": nnz})
            return nnz
        if self.comm.world > 1 and self.gather == "host":
            so = self._shared_outputs()
            self._ctx.comm_barrier()        # every rank is done with the arrays of the previous call
            nnz = self._ctx.interpolate_count(method)
            self._ctx.interpolate_fetch(so.indptr, so.indices, so.data, so.neumann)
            self._ctx.comm_barrier()        # every block has landed
            t = self._ctx.timing_or
            self.last_timings.update({"k2_ms": t("k2"), "k3_count_ms": t("k3_count"), "k3_fill_ms": t("k3_fill"),
                                      "k4_gather_ms": 0.0, "d2h_csr_ms": t("d2h_csr"), "nnz": nnz})
            lo, hi = int(self.partition_bounds[self.comm.rank]), int(self.partition_bounds[self.comm.rank + 1])
            self.last_timings["d2h_bytes"] = 12 * int(so.indptr[hi] - so.indptr[lo]) + 12 * (hi - lo)   # this rank's rows
            return (so.exact("indptr", g.n_points + 1), so.exact("indices", nnz), so.exact("data", nnz),
                    so.exact("neumann", g.n_points))
        nnz = self._ctx.interpolate_count(method)
        n_points = g.n_points
        indptr = self._out("indptr", n_points + 1, np.int32)
        indices = self._out("indices", nnz, np.int32)
        data = self._out("data", nnz, np.float64)
        neumann = self._out("neumann", n_points, np.float64)
        self._ctx.interpolate_fetch(indptr, indices, data, neumann)
        t = self._ctx.timing_or
        self.last_timings.update({"k2_ms": t("k2"), "k3_count_ms": t("k3_count"), "k3_fill_ms": t("k3_fill"),
                                  "k4_gather_ms": t("k4_gather") if self.comm.world > 1 else 0.0,
                                  "d2h_csr_ms": t("d2h_csr"), "nnz": nnz,
                                  "d2h_bytes": indptr.nbytes + indices.nbytes + data.nbytes + neumann.nbytes})
        return indptr, indices, data, neumann

    def interpolate(self, variable, method, target_points=np.array([], dtype=DTYPE_I)):
        self._check_call(variable, method)
        data_index = self.variable_to_index["cells"][variable]
        if self.cells_data_dimensions[data_index] > 1:
            raise ValueError(f"Variable '{variable}' has more than one dimension. Vector data not supported yet.")
        self._check_targets(target_points)
        self.logger.log(f"Interpolating variable '{variable}' using method '{method}'")
        indptr, indices, data, neumann = self._compute_weights(variable, method, fetch=True)
        g = self.grid
        # the device emitted canonical CSR (sorted, zero-free, int32 index arrays): no conversion, no copy
        W = sp.csr_matrix((data, indices, indptr), shape=(g.n_points, g.n_elems), copy=False)
        W.has_sorted_indices = True
        W.has_canonical_format = True
        return W, neumann

    def _check_call(self, variable, method):
        """The argument checks interpolate() and nodal_values() share (interpolator.pyx:549-560)."""
        if not self.is_grid_initialized:
            raise ValueError("Grid not initialized. Please load a mesh first.")
        if method not in self.supported_methods:
            raise ValueError(f"Method '{method}' not supported. Supported methods are: {list(self.supported_methods.keys())}")
        if variable not in self.variable_to_index["cells"]:
            raise ValueError(f"Variable '{variable}' not found in cells data. Point -> Cell interpolation not supported yet.")

    def _compute_weights(self, variable, method, fetch):
        """Stages the inputs of (method, variable) and computes the CSR: the chunk pipeline where it applies, else (or when
        an exact-zero weight voids its plan) the two-pass path.  fetch=True: returns the host arrays (indptr, indices, data,
        neumann).  fetch=False: the CSR stays on the device for npb_apply, nothing is downloaded; with world > 1 only the
        two-pass count runs, since the pipeline's gather = "all" would broadcast every block."""
        self._weights_key = None
        if fetch:
            piped = self.stream_chunks > 0 and not (self.comm.world > 1 and self.gather == "root")
        else:
            piped = self.stream_chunks > 0 and self.comm.world == 1
        fields = self._stage_inputs(method, variable, self.variable_to_index, self._rows["cells"], self._rows["points"],
                                    defer_fields=piped and self.pin_inputs)
        out = self._run_pipeline(method, fields, fetch) if piped else None
        if out is None:
            if fields is not None and not (self._ctx_has_fields()):
                # the pipeline never ran (or gave up before its uploads): stage the cell fields the classic way
                fields = None
                self._stage_inputs(method, variable, self.variable_to_index, self._rows["cells"], self._rows["points"])
            out = self._run(method, fetch)
        if getattr(self, "_pending_key", None) is not None:
            self._staged, self._pending_key = self._pending_key, None
        self._weights_key = (method, variable, self._data_version, self._mesh_serial)
        return out

    def nodal_values(self, variable, method, values=None):
        """Nodal values `W @ values`, where W is the CSR `interpolate(variable, method)` returns, computed on the GPU
        from the resident weights: bit-identical to scipy's product (NaN included), without the CSR ever leaving the
        device.  The weights stay resident between calls; a later call with the same (method, variable) and unchanged
        inputs only uploads `values`, runs one kernel and downloads the result.

        values: None (the cell data of `variable`: shape (n_elems,), or (n_elems, dim) for a vector variable, which
        this method accepts), or any real array of shape (n_elems,) or (n_elems, k), converted to float64 like scipy
        does.  Returns float64 of shape (n_points,) or (n_points, k).  With several GPUs every rank calls it and every
        rank receives the full result, in every gather mode."""
        self._check_call(variable, method)
        g = self.grid
        n_elems, n_points = g.n_elems, g.n_points
        if values is None:
            dim = int(self.cells_data_dimensions[self.variable_to_index["cells"][variable]])
            row = np.asarray(self._rows["cells"][self.variable_to_index["cells"][variable]], dtype=DTYPE_F)
            x = row[:n_elems * dim] if dim == 1 else row[:n_elems * dim].reshape(n_elems, dim)
        else:
            x = self._as_real_rows("nodal_values", values, n_elems)
        x = np.ascontiguousarray(x)
        if x.ndim == 2 and x.shape[1] == 0:
            return np.empty((n_points, 0), dtype=DTYPE_F)
        reused = self._resident_weights(variable, method)
        out = self._out("nodal", n_points * (1 if x.ndim == 1 else x.shape[1]), DTYPE_F)
        out = out.reshape((n_points,) + x.shape[1:])
        self._ctx.apply(method, x, out)
        t = self._ctx.timing_or
        self.last_timings.update({"nodal_h2d_ms": t("h2d_apply"), "nodal_apply_ms": t("apply"),
                                  "nodal_d2h_ms": t("d2h_apply"), "nodal_weights_reused": reused})
        return out

    def nodal_adjoint(self, variable, method, values):
        """The transposed product `W.T @ values`, where W is the CSR `interpolate(variable, method)` returns, computed on
        the GPU from the resident weights: bit-identical to scipy's product (NaN included).  It takes nodal values or
        sensitivities back to the cells: gradients through the nodal reconstruction (d f(W u) / du = W.T df/dy),
        transposed matrix-free solves, least-squares fits of a cell field to nodal data.  The weights are shared with
        nodal_values(): alternating the two on unchanged inputs computes them once.

        values: any real array of shape (n_points,) or (n_points, k), converted to float64 like scipy does.  Returns
        float64 of shape (n_elems,) or (n_elems, k).  One GPU only: with several ranks it raises NotImplementedError,
        since every rank holds only its own rows of W."""
        self._check_call(variable, method)
        if self.comm.world > 1:
            raise NotImplementedError("nodal_adjoint: the transposed product is single-GPU; every rank holds only its "
                                      "own rows of W")
        g = self.grid
        n_elems, n_points = g.n_elems, g.n_points
        y = np.ascontiguousarray(self._as_real_rows("nodal_adjoint", values, n_points))
        if y.ndim == 2 and y.shape[1] == 0:
            return np.empty((n_elems, 0), dtype=DTYPE_F)
        reused = self._resident_weights(variable, method)
        out = self._out("adjoint", n_elems * (1 if y.ndim == 1 else y.shape[1]), DTYPE_F)
        out = out.reshape((n_elems,) + y.shape[1:])
        self._ctx.apply_transpose(method, y, out)
        t = self._ctx.timing_or
        self.last_timings.update({"adjoint_h2d_ms": t("h2d_adjoint"), "adjoint_map_ms": t("adjoint_map"),
                                  "adjoint_apply_ms": t("adjoint"), "adjoint_d2h_ms": t("d2h_adjoint"),
                                  "adjoint_weights_reused": reused})
        return out

    @staticmethod
    def _as_real_rows(caller, values, n_rows):
        """values as float64 of shape (n_rows,) or (n_rows, k), the operand checks of nodal_values / nodal_adjoint."""
        if np.iscomplexobj(values):
            raise TypeError(f"{caller}: complex values are not supported; pass the real and imaginary parts "
                            "as separate columns")
        x = np.asarray(values, dtype=DTYPE_F)
        if x.ndim not in (1, 2) or x.shape[0] != n_rows:
            raise ValueError(f"{caller}: values must have shape ({n_rows},) or ({n_rows}, k), got {x.shape}")
        return x

    def _resident_weights(self, variable, method):
        """Makes the CSR of (method, variable) for the current inputs resident on the device, computing it only when
        the resident one is not that; returns True when it was reused."""
        reused = self._weights_key == (method, variable, self._data_version, self._mesh_serial)
        if not reused:
            self._compute_weights(variable, method, fetch=False)
        return reused
