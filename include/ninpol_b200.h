/*
 * ninpol_b200.h — C ABI of libninpol_b200.so: the sm_100a replacement for ninpol's nodal-interpolation
 * hot path (Interpolator.load_mesh -> Interpolator.interpolate).
 *
 * The reference is a Cython package with no C FFI of its own; the boundary this library replaces is
 * the set of `cdef` calls its Interpolator makes into Grid and into the IDW / LS / GLS plug-ins.  Each
 * entry point below names the reference interface it stands in for (paths relative to the reference
 * repository root).  Conventions:
 *   - plain C: opaque context pointer, raw host pointers + element counts, no framework types;
 *   - every function returns 0 on success, non-zero on error; npb_last_error() gives the message of the
 *     last failure on the calling thread;
 *   - host arrays are borrowed for the duration of the call only; device state lives in the context;
 *   - array dtypes/layouts on the host side are the reference's own (int64 ids, -1 padding, float64
 *     geometry, int32/float64 CSR exactly as scipy returns them), so results compare bit-for-bit;
 *   - one context drives one GPU on one CUDA stream; multi-GPU = one process (and context) per GPU.
 * There is no CPU fallback: every call fails with NPB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef NINPOL_B200_H
#define NINPOL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NPB_OK 0
#define NPB_ERR_ARG 1      /* bad argument / unknown name / call order                      */
#define NPB_ERR_CUDA 2     /* CUDA runtime failure or no usable device                      */
#define NPB_ERR_NCCL 3     /* NCCL failure or libnccl.so.2 not loadable                     */
#define NPB_ERR_RANGE 4    /* a count exceeds the 32-bit id range used on the device        */
#define NPB_ERR_STATE 5    /* e.g. interpolate before load_mesh, missing field              */

#define NPB_METHOD_IDW 0   /* ninpol/_methods/idw.pyx                                        */
#define NPB_METHOD_LS 1    /* ninpol/_methods/ls.pyx                                         */
#define NPB_METHOD_GLS 2   /* ninpol/_methods/gls.pyx                                        */

#define NPB_UNIQUE_ID_BYTES 128

typedef struct npb_ctx npb_ctx;

/* library */
int npb_version(void);
const char *npb_last_error(void);
int npb_device_count(int *count);

/* Context: owns one device, one stream, all device arrays.
 * Replaces: object construction in Interpolator.__cinit__ (ninpol/_interpolator/interpolator.pyx:37-91). */
int npb_create(int device, npb_ctx **ctx);
int npb_destroy(npb_ctx *ctx);

/* Multi-GPU wiring (one process per GPU).  Rank 0 calls npb_comm_unique_id and ships the 128 bytes to
 * the other ranks by any host channel; every rank then calls npb_comm_init.  NCCL is dlopen'ed here, so
 * single-GPU use needs no NCCL at all.  No reference counterpart (the reference is single-process,
 * SURVEY.md 2.2). */
int npb_comm_unique_id(void *id_out /* NPB_UNIQUE_ID_BYTES */);
int npb_comm_init(npb_ctx *ctx, const void *id, int rank, int world);
/* node ranges of all ranks: bounds[world+1], bounds[0]=0, bounds[world]=n_points, non-decreasing.
 * Default (never called, or world==1): this rank owns every node. */
int npb_set_partition(npb_ctx *ctx, const int64_t *bounds, int n_bounds);
/* Who receives the assembled CSR when world > 1: NPB_GATHER_ALL (default) all-gathers the row blocks to
 * every rank; NPB_GATHER_ROOT sends them to rank 0 only - the other ranks' npb_interpolate_count /
 * npb_interpolate_fetch then return their own row block (rows of other ranks empty, shape unchanged). */
#define NPB_GATHER_ALL 0
#define NPB_GATHER_ROOT 1
/* NPB_GATHER_HOST: no device-side gather of the blocks at all - npb_interpolate_count reports the global nnz
 * on every rank and npb_interpolate_fetch copies THIS RANK'S rows to their global positions in the arrays it
 * is given (indptr[lo..hi), indices / data [indptr[lo], indptr[hi]), neumann[lo..hi); the last rank also
 * writes indptr[n_points]).  When all ranks pass views of one shared host mapping, the full CSR assembles
 * in host memory through eight PCIe links in parallel; npb_comm_barrier separates the steps. */
#define NPB_GATHER_HOST 2
int npb_set_gather(npb_ctx *ctx, int mode);
/* All ranks of the communicator have reached this call and their streams are idle (a grouped 1-int
 * ncclBroadcast from every rank).  No-op when world == 1. */
int npb_comm_barrier(npb_ctx *ctx);
/* Closed range [first, last] of the element ids that occur in the node->element rows of this rank's node
 * range (after npb_set_partition): the only elements whose cell fields the rank's nodes read, so a rank
 * needs to upload just that slice (npb_set_cell_field_range).  first > last for an empty node range. */
int npb_partition_elem_range(npb_ctx *ctx, int64_t *first, int64_t *last);

/* K1 — connectivity + geometry on the device.
 * Replaces: Grid.__cinit__ + Grid.build + load_point_coords + calculate_centroids +
 * calculate_normal_faces, i.e. the calls at interpolator.pyx:194,204-207 into
 * ninpol/_interpolator/grid.pyx:47-140,142-231,233-267,304-525,661-809.  Arguments are the tuple
 * process_mesh returns (interpolator.pyx:363-369) plus the coordinates:
 *   connectivity  [n_elems, 8]  int64, -1 padded          element_types [n_elems] int64
 *   npoel[8] nfael[8] lnofa[8][6] lpofa[8][6][4] nedel[8] lpoed[8][12][2]   int64 tables
 *   coords        [n_points, 3] float64
 * build_edges != 0 additionally builds inpoed / inedel (grid.pyx:527-580). */
int npb_load_mesh(npb_ctx *ctx, int dim, int64_t n_elems, int64_t n_points, const int64_t *connectivity,
                  const int64_t *element_types, const int64_t *npoel, const int64_t *nfael, const int64_t *lnofa,
                  const int64_t *lpofa, const int64_t *nedel, const int64_t *lpoed, const double *coords,
                  int build_edges);
/* Same, with connectivity rows of conn_stride <= 8 nodes ([n_elems, conn_stride], no -1 padding needed up
 * to the widest element type present): a one-block mesh (all tets, all hexes ...) passes its meshio block as
 * it is and skips building and uploading the padded [n_elems, 8] array (3.2 GB at 50M cells). */
int npb_load_mesh_strided(npb_ctx *ctx, int dim, int64_t n_elems, int64_t n_points, const int64_t *connectivity,
                          int conn_stride, const int64_t *element_types, const int64_t *npoel, const int64_t *nfael,
                          const int64_t *lnofa, const int64_t *lpofa, const int64_t *nedel, const int64_t *lpoed,
                          const double *coords, int build_edges);

/* Grid attributes (grid.pxd:128-187).  Scalars: dim n_elems n_points n_faces n_edges
 * MX_ELEMENTS_PER_POINT MX_POINTS_PER_POINT MX_ELEMENTS_PER_FACE MX_FACES_PER_POINT, and the flat
 * lengths len_esup len_fsup len_esuf len_psup.  Arrays (reference dtype and shape, caller-allocated):
 * inpoel element_types esup esup_ptr psup psup_ptr esuel infael inpofa fsup fsup_ptr esuf esuf_ptr
 * boundary_faces boundary_points inpoed inedel (int64);  point_coords centroids faces_centers
 * normal_faces faces_areas (float64). */
int npb_grid_scalar(npb_ctx *ctx, const char *name, int64_t *out);
int npb_grid_array(npb_ctx *ctx, const char *name, void *out, int64_t capacity_bytes);

/* Per-variable inputs of the plug-ins.
 * Replaces: the cells_data / points_data rows the plug-ins look up through variable_to_index
 * (idw.pyx:27-28, ls.pyx:28-29, gls.pyx:47-59).  name is "permeability" (n = 9*n_elems, row-major 3x3
 * per element) or "diff_mag" (n = n_elems).  neumann_flag holds int64 truncations of the point data
 * (non-zero = Neumann node), exactly what `.astype(int)` yields in the reference. */
int npb_set_cell_field(npb_ctx *ctx, const char *name, const double *data, int64_t n);
/* Same, for the elements [first_elem, first_elem + n_elems_in_range) only: data holds 9 (permeability) or
 * 1 (diff_mag) values per element of the range.  Values of elements outside every uploaded range are
 * unspecified; a rank needs the range npb_partition_elem_range reports. */
int npb_set_cell_field_range(npb_ctx *ctx, const char *name, const double *data, int64_t first_elem,
                             int64_t n_elems_in_range);
int npb_set_point_flags(npb_ctx *ctx, const int64_t *neumann_flag, int64_t n_points);
/* Same, from the float64 point-data row itself: the `.astype(int)` truncation (NaN / inf -> non-zero, as
 * numpy casts them) happens on the device, which saves the host a pass over the array. */
int npb_set_point_flags_f64(npb_ctx *ctx, const double *neumann_flag, int64_t n_points);
/* Multi-GPU re-staging of a flag row that is expected to be unchanged (no reference counterpart): the rank uploads only
 * the slice [first, first + count) it owns; the slices of all ranks must tile [0, n_points).  *checksum = the checksum of
 * the whole row, summed over the ranks (collective: one 8-byte ncclAllReduce), in the form of the "flags_checksum" scalar.
 * Equal to the resident row's checksum: nothing else needs to move.  Different: call npb_set_point_flags_f64. */
int npb_set_point_flags_f64_range(npb_ctx *ctx, const double *flag_slice, int64_t first, int64_t count, int64_t *checksum);

/* K2 + K3 (+ K4) — weights and CSR.
 * Replaces: Interpolator.prepare_interpolator -> XInterpolation.prepare (interpolator.pyx:631-670;
 * idw.pyx:14-84, ls.pyx:21-135, gls.pyx:38-474) and the COO fill / COO->CSR / eliminate_zeros of
 * Interpolator.interpolate (interpolator.pyx:598-624), for target_points = all nodes.
 * npb_interpolate_count runs the weight kernels for this rank's node range, counts the surviving
 * entries per row, (multi-GPU: all-gathers the row counts), scans them into indptr and reports the
 * global nnz.  npb_interpolate_fetch fills indices/data/neumann at their global offsets, (multi-GPU:
 * all-gathers the row blocks over NCCL) and copies the full CSR + neumann vector into caller memory:
 *   indptr [n_points+1] int32, indices [nnz] int32, data [nnz] float64, neumann [n_points] float64.
 * Any output pointer may be NULL to skip that copy. */
int npb_interpolate_count(npb_ctx *ctx, int method, int64_t *nnz);
int npb_interpolate_fetch(npb_ctx *ctx, int32_t *indptr, int32_t *indices, double *data, double *neumann);

/* K5 — nodal values from the resident weights (no reference counterpart; the reference's callers multiply the CSR
 * by the cell field with scipy, `W @ u`).
 * out[p, c] = sum over the entries j of row p in ascending order of data[j] * values[indices[j], c], for c < n_cols,
 * using the CSR of `method` that the last npb_interpolate_count / npb_interpolate_run left on the device.  Each sum
 * starts at +0.0 and every product and addition is rounded on its own: bit-identical to scipy's csr_matvec(s).
 * values [n_elems, n_cols] and out [n_points, n_cols]: float64, row-major, host memory (pageable or page-locked).
 * NPB_ERR_STATE when no CSR of `method` is resident (c->counted false or c->method != method): every change of the
 * inputs (flags, cell fields, partition, gather mode, mesh, npb_interpolate_dense) voids it.  When world > 1 this is
 * collective: each rank reads only the rows of `values` its nodes refer to (npb_partition_elem_range), computes its
 * own rows, and the row blocks of the result are all-gathered, so every rank's `out` holds all n_points rows in every
 * gather mode; no CSR block moves between the GPUs or to the host.  Timings: "h2d_apply" "apply" "apply_gather"
 * "d2h_apply" (and "k3_fill" when the rows still had to be written). */
int npb_apply(npb_ctx *ctx, int method, const double *values, int64_t n_cols, double *out);

/* K5 — the transposed product from the resident weights: adjoints / gradients through the nodal reconstruction,
 * transposed matrix-free solves, least-squares fits of a cell field to nodal data (scipy: `W.T @ y`).
 * out[e, c] = sum over the entries (p, e) of W in ascending p of data[j] * values[p, c], for c < n_cols, using the CSR
 * of `method` that the last npb_interpolate_count / npb_interpolate_run left on the device.  Each sum starts at +0.0
 * and every product and addition is rounded on its own: bit-identical to scipy's csc_matvec(s) on the view W.T.
 * values [n_points, n_cols] and out [n_elems, n_cols]: float64, row-major, host memory (pageable or page-locked).
 * NPB_ERR_STATE when no CSR of `method` is resident, exactly as npb_apply.  NPB_ERR_STATE when world > 1: a rank holds
 * only its own rows, so the ordered sum of an element spans ranks; the transposed product is single-GPU.
 * The first call on a CSR builds a map of every element's (node, CSR position) slots (8 * spe bytes per element); it
 * is rebuilt whenever the CSR is rewritten or voided.  Timings: "h2d_adjoint" "adjoint_map" (0 when the map was
 * reused) "adjoint" "d2h_adjoint" (and "k3_fill" when the rows still had to be written). */
int npb_apply_transpose(npb_ctx *ctx, int method, const double *values, int64_t n_cols, double *out);

/* The plug-in's own output, for callers that sit where Interpolator.prepare_interpolator sits
 * (interpolator.pyx:631-670): dense weights [n_points, MX_ELEMENTS_PER_POINT] (row stride
 * MX_ELEMENTS_PER_POINT, column k of row p <-> esup[esup_ptr[p] + k], untouched entries 0) and neumann_ws
 * [n_points], exactly the two caller-allocated outputs of `XInterpolation.prepare(grid, cells_data,
 * points_data, faces_data, variable_to_index, variable, target_points, weights, neumann_ws)`
 * (idw.pxd:19-24, ls.pxd:20-25, gls.pxd:22-27), target_points = all nodes.  Single GPU. */
int npb_interpolate_dense(npb_ctx *ctx, int method, double *weights, double *neumann_ws);

/* The same result as npb_interpolate_count + npb_interpolate_fetch, computed as a pipeline over n_chunks
 * contiguous node chunks of THIS RANK's node range (one GPU: all nodes).  The CSR row lengths are planned before
 * the weights exist (a Dirichlet node emits nothing, every other node its whole node->element row), so every rank
 * knows the global indptr without any exchange and four streams overlap: upload of the cell-field slice chunk k+1
 * reads (GLS; perm_host / diff_mag_host = the full page-locked host arrays, or NULL to use the fields already set),
 * compute of chunk k at its final global offsets, (gather = NPB_GATHER_ALL) NCCL broadcast of chunk k to the peers,
 * download of the finished blocks into the caller's page-locked arrays (NPB_GATHER_HOST: this rank's rows at their
 * global positions of arrays shared by the ranks; otherwise the whole CSR).  Any of indptr / indices / data /
 * neumann may be NULL (device-resident result only: what bench.py's device-timed `value` measures); indices / data
 * hold `capacity` entries, capacity >= the planned nnz (<= grid scalar "len_esup").
 * *fell_back = 1 (identically on every rank) when some rank met an exact-zero weight - scipy's eliminate_zeros
 * would drop it, which voids the planned offsets - or a node star too large for the tile kernels: nothing valid was
 * written and the caller runs npb_interpolate_count + npb_interpolate_fetch instead.  Not for NPB_GATHER_ROOT.
 * No reference counterpart (host orchestration of interpolator.pyx:579-624 for a device behind PCIe / NVLink). */
int npb_interpolate_run(npb_ctx *ctx, int method, int n_chunks, const double *perm_host, const double *diff_mag_host,
                        int32_t *indptr, int32_t *indices, double *data, double *neumann, int64_t capacity,
                        int64_t *nnz, int *fell_back);
/* Round-1 entry point of the single-GPU pipeline: npb_interpolate_run with all four outputs required and the
 * two-pass fallback taken internally. */
int npb_interpolate_streamed(npb_ctx *ctx, int method, int n_chunks, const double *perm_host,
                             const double *diff_mag_host, int32_t *indptr, int32_t *indices, double *data,
                             double *neumann, int64_t capacity, int64_t *nnz);

/* Device-side timings (CUDA events on the context's stream) of the most recent calls, in ms.
 * Names: "k1" "k1_esup" "k1_esuel" "k1_faces" "k1_fsup" "k1_geom" "k2" "k3_count" "k3_fill" "k4_gather"
 * "h2d_mesh" "d2h_csr".  Replaces the clock_gettime stopwatches of grid.pyx:150-227 /
 * interpolator.pyx:608-668. */
int npb_timing(npb_ctx *ctx, const char *name, double *ms);
/* Number of this library's kernel launches since the context was created (bench.py's gpu_launches). */
int npb_launch_count(npb_ctx *ctx, int64_t *count);
/* Debug aid (no reference counterpart): with NPB_DEBUG_GUARDS=1 in the environment when the library is first used,
 * every device block the library allocates is followed by 64 guard bytes; this reads them all back.  n_blocks = guarded
 * blocks checked, n_damaged = blocks whose guard was overwritten (npb_last_error names one).  Both 0 when guards are off. */
int npb_check_guards(npb_ctx *ctx, int64_t *n_blocks, int64_t *n_damaged);

/* Measurement helpers used by bench.py for the roofline denominators that MEASURED_PEAKS.json lacks:
 * a register-resident DFMA loop (FP64 TFLOP/s) and a device copy (GB/s, read+write). */
int npb_measure_fp64_peak(npb_ctx *ctx, double *tflops);
int npb_measure_copy_bw(npb_ctx *ctx, int64_t bytes, double *gbs);
/* Writes `bytes` of device memory (an L2 flush between timed iterations). */
int npb_flush_l2(npb_ctx *ctx, int64_t bytes);
int npb_synchronize(npb_ctx *ctx);
/* CUDA-event stopwatch on the context's stream: start records an event, stop records a second one,
 * waits for it and returns the elapsed device time between the two in ms. */
int npb_timer_start(npb_ctx *ctx);
int npb_timer_stop(npb_ctx *ctx, double *ms);
/* Page-locked host memory for the CSR outputs / field inputs (full-rate PCIe copies). */
int npb_host_alloc(int64_t bytes, void **ptr);
int npb_host_free(void *ptr);
/* Page-lock / unlock caller-owned host memory in place (cudaHostRegister), so that the copies made from it
 * by npb_set_cell_field / npb_set_point_flags / npb_load_mesh run at the PCIe rate without staging. */
int npb_host_register(void *ptr, int64_t bytes);
int npb_host_unregister(void *ptr);

#ifdef __cplusplus
}
#endif
#endif /* NINPOL_B200_H */
