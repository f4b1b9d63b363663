// common.cuh — context, device-buffer bookkeeping and element tables shared by the translation units
// of libninpol_b200.so.  Device ids are int32 (every count the reference can index is < 2^31,
// SURVEY.md App. A.9), geometry is float64.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <map>
#include <string>
#include <vector>
#include "../../include/ninpol_b200.h"

typedef long long i64;

#define NPB_MX_PE 8
#define NPB_MX_FE 6
#define NPB_MX_PF 4
#define NPB_N_TYPES 8
#define NPB_MX_EE 12
// Doubles per centroid record on the device.  4 (32-byte records that never straddle two 32-byte sectors, pad
// stripped at export) was measured on B200 and is SLOWER than the packed 3: the gather misses L2 60 % of the time, so
// the extra 8 bytes per record cost more DRAM traffic than the straddling saves (IDW 0.685 -> 0.655 of the HBM roofline
// at 50M tets, LS 0.517 -> 0.502).
#define NPB_CSTRIDE 3

// element tables (reference utils/point_ordering.yaml via process_mesh, interpolator.pyx:274-330);
// passed to kernels by value -> lives in the constant bank.
struct ElemTables {
    int8_t npoel[NPB_N_TYPES];
    int8_t nfael[NPB_N_TYPES];
    int8_t lnofa[NPB_N_TYPES][NPB_MX_FE];
    int8_t lpofa[NPB_N_TYPES][NPB_MX_FE][NPB_MX_PF];
};
struct EdgeTables {
    int8_t nedel[NPB_N_TYPES];
    int8_t lpoed[NPB_N_TYPES][NPB_MX_EE][2];
};

void npb_set_error(const char *fmt, ...);

#define NPB_CUDA(call)                                                                            \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            npb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e__), __FILE__, __LINE__, #call); \
            return NPB_ERR_CUDA;                                                                  \
        }                                                                                         \
    } while (0)

#define NPB_TRY(call)                \
    do {                             \
        int r__ = (call);            \
        if (r__ != NPB_OK) return r__; \
    } while (0)

struct NcclApi;  // k4_shard.cu

struct NpbPendingTimer {
    std::string name;
    cudaEvent_t a, b;
    bool accumulate;
};

struct npb_ctx {
    std::vector<NpbPendingTimer> pending_timers;
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    i64 launches = 0;
    std::map<std::string, float> timings;
    std::vector<void *> owned;  // everything cudaMalloc'ed for the current mesh

    // ---- mesh (K1 outputs) ----
    bool mesh_loaded = false;
    int dim = 0;
    i64 n_elems = 0, n_points = 0, n_faces = 0, n_edges = 0;
    int spe = 8;  // row stride of inpoel on the device (4 for pure-tet/quad/tri meshes, else 8)
    int sfe = 6;  // row stride of esuel / infael on the device (4 or 6)
    i64 len_esup = 0, len_fsup = 0, len_esuf = 0, len_psup = 0;
    int mx_epp = 0, mx_fpp = 0, mx_epf = 0, mx_ppp = 0;
    ElemTables tab;
    EdgeTables etab;
    bool build_edges = false;
    int32_t *inpoel = nullptr;   // [n_elems, spe], -1 padded
    uint8_t *etype = nullptr;    // [n_elems]
    double *coords = nullptr;    // [n_points, 3]
    int32_t *esup_ptr = nullptr, *esup = nullptr;
    int32_t *esuel = nullptr, *infael = nullptr;  // [n_elems, sfe]
    int32_t *inpofa = nullptr;   // [n_faces, 4], -1 padded
    int2 *esuf2 = nullptr;       // [n_faces] (owner, other | -1)
    uint8_t *bface = nullptr, *bpoint = nullptr;
    int32_t *fsup_ptr = nullptr, *fsup = nullptr;
    int32_t *psup_ptr = nullptr, *psup = nullptr;
    i64 *inedel_d = nullptr, *inpoed_d = nullptr;   // edges, reference layout (int64), built when build_edges
    double *centroids = nullptr, *fcent = nullptr, *fnormal = nullptr, *farea = nullptr;

    // ---- per-variable inputs ----
    double *perm = nullptr, *diff_mag = nullptr;
    uint8_t *nflag = nullptr;
    bool have_perm = false, have_dm = false, have_flags = false;
    i64 flags_checksum = 0;      // which nodes are flagged, folded on the device (capi.cu)

    // ---- partition / communicator ----
    int rank = 0, world = 1;
    std::vector<i64> bounds;  // world+1
    i64 lo = 0, hi = 0;       // this rank's node range
    i64 wbase = 0;            // esup_ptr[lo]: origin of wbuf
    i64 wlen = 0;             // esup_ptr[hi] - esup_ptr[lo]
    NcclApi *nccl = nullptr;
    void *comm = nullptr;

    // ---- interpolate state ----
    int method = -1;
    bool counted = false;
    bool fused_failed[2] = {false, false};   // per method: the single-pass emit met an exact zero for the current inputs
    bool filled = false;         // indices / data already hold the CSR (fused path, or k3_fill done)
    // bumped at every write or voiding of the CSR rows (each counted / filled transition): what is derived from the CSR
    // (the transposed map below) records the generation it was built from and is rebuilt when it differs
    unsigned long long csr_gen = 1;
    i64 nnz = 0;
    i64 nnz_ret = 0, blk_off = 0;   // what count / fetch hand out: all of it, or this rank's row block (gather to root)
    int gather_mode = 0;            // NPB_GATHER_ALL / NPB_GATHER_ROOT
    double *wbuf = nullptr;      // final data values, esup-indexed, local node range
    size_t wbuf_cap = 0;
    int32_t *rowcnt = nullptr;   // [n_points + 1]
    int32_t *indptr = nullptr;   // [n_points + 1]
    double *neumann = nullptr;   // [n_points]
    int32_t *indices = nullptr;
    double *data = nullptr;
    size_t out_cap = 0;
    void *scratch = nullptr;     // staging of flag uploads, rebased indptr, edge sort temp storage
    size_t scratch_cap = 0;
    void *scan_tmp = nullptr, *part_tmp = nullptr;   // tile totals of the scans; per-block class histograms
    size_t scan_tmp_cap = 0, part_tmp_cap = 0;
    int32_t *node_list = nullptr;  // GLS work lists
    void *gls_ws = nullptr;
    size_t gls_ws_cap = 0;
    int *counters = nullptr;     // small device int array (work counters, flags)
    int *h_small = nullptr, *d_small = nullptr;   // 64 ints of mapped page-locked memory: counts a kernel hands to the host
                                                  // without a D2H copy (small copies queue behind bulk downloads on the copy engine)
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;  // npb_timer_start / stop
    void *stage[2] = {nullptr, nullptr};         // page-locked staging buffers for pageable host memory
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    cudaStream_t up_stream = nullptr, down_stream = nullptr, comm_stream = nullptr;   // pipeline.cu: upload / download / gather legs
    std::vector<cudaEvent_t> pipe_ev;
    // pipeline.cu: the optimistic row plan (c->indptr holds it while plan_kind != 0: 1 = IDW / LS, 2 = GLS)
    int plan_kind = 0;
    bool plan_failed[3] = {false, false, false};   // per method: an exact zero voided the plan for the current inputs (every
                                                   // rank saw the same verdict), so the next call goes straight to two passes
    i64 plan_nnz = 0;
    int plan_chunks = 0;                 // chunk table below is valid for this many chunks per rank
    std::vector<i64> chunk_node, chunk_nz;   // [world * K + 1] node / nnz boundaries of every rank's chunks
    std::vector<i64> chunk_efirst, chunk_elast;   // [K] element range this rank's chunk k reads (empty: not computed yet)
    bool gathered = false;               // indices / data / neumann of ALL ranks are on this device (gather = all)
    // npb_apply (k5_apply.cu): the values uploaded for this rank's rows and the result rows, [.., n_cols] row-major.
    // npb_apply_transpose uses the same two buffers by shape: apply_y holds its nodal input, apply_x its element output
    double *apply_x = nullptr, *apply_y = nullptr;
    size_t apply_x_cap = 0, apply_y_cap = 0;
    bool apply_range_ok = false;         // apply_first / apply_last hold npb_partition_elem_range for the current partition
    i64 apply_first = 0, apply_last = -1;
    // npb_apply_transpose: [n_elems, spe] (node, CSR position) slots of every element, built from the CSR of generation
    // tmap_gen (k5_tmap)
    int2 *tmap = nullptr;
    size_t tmap_cap = 0;
    unsigned long long tmap_gen = 0;
};

// ---- helpers implemented in capi.cu ----
int npb_alloc(npb_ctx *c, void **p, size_t bytes, bool owned_by_mesh = true);
int npb_ensure(void **p, size_t *cap, size_t bytes);
bool npb_is_pinned(const void *p);
int npb_h2d(npb_ctx *c, void *dst_dev, const void *src_host, size_t bytes);
int npb_d2h(npb_ctx *c, void *dst_host, const void *src_dev, size_t bytes);
struct NpbTimer {
    npb_ctx *c;
    const char *name;
    cudaEvent_t a, b;
    bool accumulate;
    NpbTimer(npb_ctx *c_, const char *n, bool accumulate_ = false);   // accumulate: add to timings[name]
    void stop_lazy();   // records the closing event only; the elapsed time is read when somebody asks (npb_resolve_timers):
                        // no host synchronisation on the hot path
    ~NpbTimer();   // an early (error) return must not leak the two events
    NpbTimer(const NpbTimer &) = delete;
    NpbTimer &operator=(const NpbTimer &) = delete;
    void stop();
};

// ---- scan.cu (CUB) ----
int npb_exclusive_scan_i32(npb_ctx *c, const int32_t *in, int32_t *out, i64 n);   // out may alias in
int npb_max_i32(npb_ctx *c, const int32_t *in, i64 n, int32_t *host_out);
int npb_partition_classes(npb_ctx *c, const uint8_t *cls, i64 lo, i64 hi, int32_t *out, int *host_starts /*[9 + 1]*/);
int npb_sort_pairs_u32(npb_ctx *c, const uint32_t *keys_in, uint32_t *keys_out, const uint32_t *vals_in, uint32_t *vals_out, i64 n);
int npb_propagate_heads(npb_ctx *c, uint2 *pairs, i64 n);

// ---- kernels' host drivers ----
int npb_k1_build(npb_ctx *c, const i64 *h_conn, int conn_stride, const i64 *h_types, const double *h_coords);
int npb_k1_geometry(npb_ctx *c);
int npb_k1_extras(npb_ctx *c);  // psup, edges
int npb_k2_idw_ls(npb_ctx *c, int method, i64 lo, i64 hi);
int npb_k2_idw_ls_fused(npb_ctx *c, int method, int *used);
int npb_k2_idw_ls_tiles(npb_ctx *c, int method, i64 lo, i64 hi, int *used);
int npb_ensure_out(npb_ctx *c, size_t n);
int npb_k2_gls(npb_ctx *c, i64 lo, i64 hi);
int npb_k3_fill(npb_ctx *c, i64 lo, i64 hi);
int npb_read_int(npb_ctx *c, const int *d_src, int *h_out);
void npb_resolve_timers(npb_ctx *c);   // turns the lazily stopped timers into timings[] entries (waits for their events)
__global__ void k_copy2_int(int *dst, const int *src);   // capi.cu: two ints, device -> mapped host block
__global__ void k_copy_int(int *dst, const int *src);    // capi.cu   // device int -> host through the mapped block + stream sync
int npb_minmax_i32(npb_ctx *c, const int32_t *in, i64 n, int32_t *h_min, int32_t *h_max);
int npb_k4_gather_counts(npb_ctx *c);
int npb_k4_gather_blocks(npb_ctx *c);
int npb_k4_gather_rows(npb_ctx *c, double *rows, i64 n_cols);
int npb_k5_apply(npb_ctx *c, i64 lo, i64 hi, const double *x, int64_t k, double *out);
int npb_k5_tmap(npb_ctx *c, int2 *map);
int npb_k5_apply_t(npb_ctx *c, const int2 *map, const double *y, int64_t k, double *out);
int npb_export_array(npb_ctx *c, const char *name, void *out, i64 cap);
// cudaMalloc'ed temporary that is freed when it goes out of scope (error returns included)
struct NpbTmp {
    void *p = nullptr;
    ~NpbTmp() { if (p) cudaFree(p); }
    NpbTmp() = default;
    NpbTmp(const NpbTmp &) = delete;
    NpbTmp &operator=(const NpbTmp &) = delete;
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 8); }
    template <class T> T *as() { return (T *)p; }
};

static inline unsigned npb_blocks(i64 n, int threads) { return (unsigned)((n + threads - 1) / threads); }
#define NPB_LAUNCH(c) ((c)->launches++)
