// pipeline.cu — interpolate() as a pipeline over node chunks, on one GPU or on every rank of a multi-GPU run.
//
// No reference counterpart: the reference computes on the host (ninpol/_interpolator/interpolator.pyx:579-624
// is the orchestration this replaces for a device that sits behind PCIe / NVLink).
//
// 1. PLAN.  CSR row lengths are known before the weights are: a Dirichlet node (and, for GLS, a node whose
//    faces are all boundary faces, gls.pyx:266-267) emits nothing, every other node emits its whole esup row,
//    unless a weight is exactly +-0.0 (scipy's eliminate_zeros would drop it).  One kernel + one scan give the
//    GLOBAL indptr on every rank with no exchange; it is cached until the flags or the mesh change.
// 2. CHUNKS.  This rank's node range is cut into contiguous chunks and four streams overlap:
//      upload    the slice of permeability / diff_mag chunk k+1 reads (GLS, from page-locked host memory);
//      compute   K2 (+ K3 for GLS) of chunk k, written at the planned global offsets; exact zeros and
//                row-count mismatches are counted on the device;
//      gather    (multi-GPU, gather = all) the chunk's block is broadcast to the peers over NCCL / NVLink;
//      download  the chunk's block into the caller's page-locked arrays (gather = host: this rank's rows at
//                their global positions of a host mapping shared by the ranks).
// 3. VERDICT.  If any rank met an exact zero (or a star too large for the tile kernels), every rank learns it
//    from one grouped 1-int broadcast and the caller re-runs the general two-pass path
//    (npb_interpolate_count / npb_interpolate_fetch).  Otherwise the arrays hold the final canonical CSR.
// Every node's weights come from the same kernels as in the two-pass path, so results are bit-identical to it.
#include <stdio.h>
#include <stdlib.h>
#include "gls_common.cuh"

int npb_k4_share_flags(npb_ctx *c, const int *d_bad2, int host_flag, int *any);
int npb_k4_bcast_chunk(npb_ctx *c, cudaStream_t st, const std::vector<i64> &node_lo, const std::vector<i64> &node_hi,
                       const std::vector<i64> &nz_lo, const std::vector<i64> &nz_hi, bool with_neumann);
int npb_k2_idw_ls_direct(npb_ctx *c, int method, i64 lo, i64 hi, int *used);
int npb_k3_fill_planned(npb_ctx *c, i64 lo, i64 hi, int *mismatch_counter);

// rowcnt-to-be of every node for the optimistic plan; neumann zeroed (IDW / LS never write it)
__global__ void k_plan(const int32_t *__restrict__ esup_ptr, const int32_t *__restrict__ fsup_ptr, const int32_t *__restrict__ fsup,
                       const int2 *__restrict__ esuf2, const uint8_t *__restrict__ bpoint, const uint8_t *__restrict__ nflag,
                       i64 n_points, int gls, int32_t *__restrict__ cnt, double *__restrict__ neumann)
{
    i64 p = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p > n_points) return;
    if (p == n_points) {
        cnt[p] = 0;
        return;
    }
    const bool bp = bpoint[p] != 0;
    bool skip = bp && !nflag[p];                       // idw.pyx:62, ls.pyx:61, gls.pyx:165
    if (gls && !skip && bp) {                          // only a boundary node has boundary faces
        const int fb = fsup_ptr[p], fe = fsup_ptr[p + 1];
        int nb = 0;
        for (int q = fb; q < fe; q++) nb += (esuf2[fsup[q]].y < 0) ? 1 : 0;
        if (nb >= fe - fb) skip = true;                // gls.pyx:266-267 -> zero row (Q8)
    }
    cnt[p] = skip ? 0 : esup_ptr[p + 1] - esup_ptr[p];
    neumann[p] = 0.0;
}

static int d2h_pieces(npb_ctx *c, cudaStream_t st, void *dst, const void *src, size_t bytes)
{
    // bulk downloads in 16 MB pieces: a small copy of another stream waits for one piece, not for the block
    const size_t piece = (size_t)16 << 20;
    for (size_t off = 0; off < bytes; off += piece) {
        size_t n = bytes - off < piece ? bytes - off : piece;
        NPB_CUDA(cudaMemcpyAsync((char *)dst + off, (const char *)src + off, n, cudaMemcpyDeviceToHost, st));
    }
    return NPB_OK;
}

static int ensure_streams(npb_ctx *c, int n_events)
{
    if (!c->up_stream) NPB_CUDA(cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking));
    if (!c->down_stream) NPB_CUDA(cudaStreamCreateWithFlags(&c->down_stream, cudaStreamNonBlocking));
    if (!c->comm_stream) NPB_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
    while ((int)c->pipe_ev.size() < n_events) {
        cudaEvent_t e;
        NPB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->pipe_ev.push_back(e);
    }
    return NPB_OK;
}

// the optimistic global indptr for `method` in c->indptr (cached: c->plan_kind)
static int ensure_plan(npb_ctx *c, int method)
{
    const int kind = method == NPB_METHOD_GLS ? 2 : 1;
    if (c->plan_kind == kind) return NPB_OK;
    cudaStream_t s = c->stream;
    const i64 np = c->n_points;
    c->plan_kind = 0;
    k_plan<<<npb_blocks(np + 1, 256), 256, 0, s>>>(c->esup_ptr, c->fsup_ptr, c->fsup, c->esuf2, c->bpoint, c->nflag, np,
                                                   kind == 2 ? 1 : 0, c->indptr, c->neumann);
    NPB_LAUNCH(c);
    NPB_TRY(npb_exclusive_scan_i32(c, c->indptr, c->indptr, np + 1));
    int32_t total = 0;
    NPB_TRY(npb_read_int(c, c->indptr + np, &total));
    c->plan_nnz = total;
    c->plan_kind = kind;
    c->plan_chunks = 0;   // chunk offsets belong to a plan
    return NPB_OK;
}

// node / nnz boundaries of every rank's chunks: chunk k of rank r = nodes [cb[r*K+k], cb[r*K+k+1]) when the
// boundary list is laid out rank-major (the last boundary of rank r is the first of rank r+1)
static int ensure_chunk_table(npb_ctx *c, int K)
{
    if (c->plan_chunks == K && (int)c->chunk_node.size() == c->world * K + 1) return NPB_OK;
    const int W = c->world;
    const std::vector<i64> old_nodes = c->chunk_node;
    c->chunk_node.assign((size_t)W * K + 1, 0);
    // Chunk sizes ramp up and down (weights 1, 2, 3, 3, ..., 3, 2): the upload of the first chunk and the download of
    // the last one are the two legs nothing can hide, so those chunks are the small ones.  Same rule on every rank.
    std::vector<i64> cum(K + 1, 0);
    for (int k = 0; k < K; k++) {
        const i64 wgt = K < 4 ? 1 : (k == 0 ? 1 : (k == 1 || k == K - 1) ? 2 : 3);
        cum[k + 1] = cum[k] + wgt;
    }
    for (int r = 0; r < W; r++) {
        const i64 a = c->bounds[r], n = c->bounds[r + 1] - a;
        for (int k = 0; k < K; k++) c->chunk_node[(size_t)r * K + k] = a + (n * cum[k]) / cum[K];
    }
    c->chunk_node[(size_t)W * K] = c->n_points;
    if (c->chunk_node != old_nodes) {   // the element ranges of the chunks follow the node boundaries, not the plan
        c->chunk_efirst.clear();
        c->chunk_elast.clear();
    }
    // one gather kernel would do; the table is tiny (W*K+1 <= 16*64+1) and read once per plan
    std::vector<int32_t> off((size_t)W * K + 1);
    for (size_t i = 0; i < off.size(); i++)
        NPB_CUDA(cudaMemcpyAsync(&off[i], c->indptr + c->chunk_node[i], sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    c->chunk_nz.assign(off.begin(), off.end());
    c->plan_chunks = K;
    return NPB_OK;
}

static void drain(npb_ctx *c)
{
    if (c->up_stream) cudaStreamSynchronize(c->up_stream);
    if (c->down_stream) cudaStreamSynchronize(c->down_stream);
    if (c->comm_stream) cudaStreamSynchronize(c->comm_stream);
    cudaStreamSynchronize(c->stream);
}

static int run_pipeline(npb_ctx *c, int method, int K, const double *perm_host, const double *diff_mag_host,
                        int32_t *indptr, int32_t *indices, double *data, double *neumann, int64_t capacity, int *fell_back)
{
    const bool gls = method == NPB_METHOD_GLS;
    const bool upload = gls && perm_host && diff_mag_host;
    const bool to_host = indptr || indices || data || neumann;
    const int W = c->world, R = c->rank;
    const bool host_gather = W > 1 && c->gather_mode == NPB_GATHER_HOST;
    const bool nccl_gather = W > 1 && c->gather_mode == NPB_GATHER_ALL;
    cudaStream_t s = c->stream;
    const i64 np = c->n_points;
    *fell_back = 0;

    NPB_TRY(ensure_plan(c, method));
    NPB_TRY(ensure_chunk_table(c, K));
    const i64 total = c->plan_nnz;
    if (to_host && total > capacity) {
        npb_set_error("npb_interpolate_run: capacity %lld is smaller than the planned nnz %lld", (long long)capacity, (long long)total);
        return NPB_ERR_ARG;
    }
    NPB_TRY(ensure_streams(c, 3 * K + 2));
    NPB_TRY(npb_ensure_out(c, (size_t)total));
    if (gls) NPB_TRY(npb_ensure((void **)&c->wbuf, &c->wbuf_cap, sizeof(double) * (size_t)(c->wlen > 0 ? c->wlen : 1)));
    c->counted = false;
    c->filled = false;
    c->csr_gen++;
    int *bad = c->counters + 45;   // [45] exact zeros (tile kernels), [46] row-count mismatches (planned emit)
    NPB_CUDA(cudaMemsetAsync(bad, 0, 2 * sizeof(int), s));
    cudaEvent_t ev_start = c->pipe_ev[3 * K], ev_side = c->pipe_ev[3 * K + 1];
    NPB_CUDA(cudaEventRecord(ev_start, s));
    NPB_CUDA(cudaStreamWaitEvent(c->up_stream, ev_start, 0));
    NPB_CUDA(cudaStreamWaitEvent(c->down_stream, ev_start, 0));
    NPB_CUDA(cudaStreamWaitEvent(c->comm_stream, ev_start, 0));

    const i64 *cn = c->chunk_node.data() + (size_t)R * K;   // this rank's chunk boundaries (K+1 entries)
    // element range each of this rank's chunks reads (GLS uploads)
    if (upload && (int)c->chunk_efirst.size() != K) {   // a property of the chunk table: computed once per table
        std::vector<i64> e_first(K, 0), e_last(K, -1);
        std::vector<int32_t> ptr(K + 1);
        for (int k = 0; k <= K; k++)
            NPB_CUDA(cudaMemcpyAsync(&ptr[k], c->esup_ptr + cn[k], sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        NPB_CUDA(cudaStreamSynchronize(s));
        for (int k = 0; k < K; k++) {
            int32_t mn = 0, mx = -1;
            NPB_TRY(npb_minmax_i32(c, c->esup + ptr[k], (i64)ptr[k + 1] - ptr[k], &mn, &mx));
            e_first[k] = mn;
            e_last[k] = mx;
        }
        c->chunk_efirst = e_first;
        c->chunk_elast = e_last;
    }
    const std::vector<i64> &e_first = c->chunk_efirst, &e_last = c->chunk_elast;
    if (upload) {
        if (!c->perm) NPB_TRY(npb_alloc(c, (void **)&c->perm, sizeof(double) * 9 * (size_t)c->n_elems));
        if (!c->diff_mag) NPB_TRY(npb_alloc(c, (void **)&c->diff_mag, sizeof(double) * (size_t)c->n_elems));
        c->have_perm = c->have_dm = false;   // until the last slice has landed
    }
    i64 ulo = 0, uhi = 0;   // resident element interval [ulo, uhi)
    auto enqueue_upload = [&](int k) -> int {
        if (upload && e_last[k] >= e_first[k]) {
            i64 a = e_first[k], b = e_last[k] + 1;
            i64 seg[2][2] = {{0, 0}, {0, 0}};
            if (uhi <= ulo) {
                seg[0][0] = a; seg[0][1] = b;
                ulo = a; uhi = b;
            } else {
                if (a < ulo) { seg[0][0] = a; seg[0][1] = ulo; ulo = a; }
                if (b > uhi) { seg[1][0] = uhi; seg[1][1] = b; uhi = b; }
            }
            for (int q = 0; q < 2; q++) {
                i64 n = seg[q][1] - seg[q][0];
                if (n <= 0) continue;
                NPB_CUDA(cudaMemcpyAsync(c->perm + 9 * seg[q][0], perm_host + 9 * seg[q][0], sizeof(double) * 9 * (size_t)n,
                                         cudaMemcpyHostToDevice, c->up_stream));
                NPB_CUDA(cudaMemcpyAsync(c->diff_mag + seg[q][0], diff_mag_host + seg[q][0], sizeof(double) * (size_t)n,
                                         cudaMemcpyHostToDevice, c->up_stream));
            }
        }
        NPB_CUDA(cudaEventRecord(c->pipe_ev[3 * k], c->up_stream));
        return NPB_OK;
    };

    // the row pointer is final as soon as the plan exists: it travels while the first chunk computes
    if (indptr) {
        if (host_gather) {
            const i64 a = c->lo, n = c->hi - c->lo + (R == W - 1 ? 1 : 0);
            if (n > 0) NPB_TRY(d2h_pieces(c, c->down_stream, indptr + a, c->indptr + a, sizeof(int32_t) * (size_t)n));
        } else
            NPB_TRY(d2h_pieces(c, c->down_stream, indptr, c->indptr, sizeof(int32_t) * (size_t)(np + 1)));
    }
    NPB_TRY(enqueue_upload(0));
    bool tiles_ok = true;
    for (int k = 0; k < K; k++) {
        const i64 a = cn[k], b = cn[k + 1];
        if (k + 1 < K) NPB_TRY(enqueue_upload(k + 1));
        NPB_CUDA(cudaStreamWaitEvent(s, c->pipe_ev[3 * k], 0));
        if (b > a) {
            if (gls) {
                NPB_TRY(npb_k2_gls(c, a, b));
                NPB_TRY(npb_k3_fill_planned(c, a, b, bad + 1));
            } else {
                int used = 0;
                NPB_TRY(npb_k2_idw_ls_direct(c, method, a, b, &used));
                if (!used) tiles_ok = false;
            }
        }
        NPB_CUDA(cudaEventRecord(c->pipe_ev[3 * k + 1], s));
        cudaEvent_t ready = c->pipe_ev[3 * k + 1];
        // what chunk step k makes final on this device: my chunk k, or (after the gather) chunk k of every rank
        std::vector<i64> nlo, nhi, zlo, zhi;
        if (nccl_gather) {
            for (int r = 0; r < W; r++) {
                nlo.push_back(c->chunk_node[(size_t)r * K + k]);
                nhi.push_back(c->chunk_node[(size_t)r * K + k + 1]);
                zlo.push_back(c->chunk_nz[(size_t)r * K + k]);
                zhi.push_back(c->chunk_nz[(size_t)r * K + k + 1]);
            }
            NPB_CUDA(cudaStreamWaitEvent(c->comm_stream, ready, 0));
            NPB_TRY(npb_k4_bcast_chunk(c, c->comm_stream, nlo, nhi, zlo, zhi, gls));
            NPB_CUDA(cudaEventRecord(c->pipe_ev[3 * k + 2], c->comm_stream));
            ready = c->pipe_ev[3 * k + 2];
        } else {
            nlo.push_back(a); nhi.push_back(b);
            zlo.push_back(c->chunk_nz[(size_t)R * K + k]);
            zhi.push_back(c->chunk_nz[(size_t)R * K + k + 1]);
        }
        if (to_host) {
            NPB_CUDA(cudaStreamWaitEvent(c->down_stream, ready, 0));
            for (size_t q = 0; q < nlo.size(); q++) {
                const i64 rows = nhi[q] - nlo[q], nk = zhi[q] - zlo[q];
                if (neumann && rows > 0) NPB_TRY(d2h_pieces(c, c->down_stream, neumann + nlo[q], c->neumann + nlo[q], sizeof(double) * (size_t)rows));
                if (indices && nk > 0) NPB_TRY(d2h_pieces(c, c->down_stream, indices + zlo[q], c->indices + zlo[q], sizeof(int32_t) * (size_t)nk));
                if (data && nk > 0) NPB_TRY(d2h_pieces(c, c->down_stream, data + zlo[q], c->data + zlo[q], sizeof(double) * (size_t)nk));
            }
        }
    }
    if (upload) {   // elements no node of this rank refers to: on one GPU keep the resident copy complete
        if (W == 1) {
            const i64 rest[2][2] = {{0, uhi > ulo ? ulo : c->n_elems}, {uhi > ulo ? uhi : c->n_elems, c->n_elems}};
            for (int q = 0; q < 2; q++) {
                i64 n = rest[q][1] - rest[q][0];
                if (n <= 0) continue;
                NPB_CUDA(cudaMemcpyAsync(c->perm + 9 * rest[q][0], perm_host + 9 * rest[q][0], sizeof(double) * 9 * (size_t)n,
                                         cudaMemcpyHostToDevice, c->up_stream));
                NPB_CUDA(cudaMemcpyAsync(c->diff_mag + rest[q][0], diff_mag_host + rest[q][0], sizeof(double) * (size_t)n,
                                         cudaMemcpyHostToDevice, c->up_stream));
            }
        }
        c->have_perm = true;
        c->have_dm = true;
    }
    // the compute stream joins the side streams, so that an event pair on it brackets the whole step
    for (cudaStream_t side : {c->up_stream, c->down_stream, c->comm_stream}) {
        NPB_CUDA(cudaEventRecord(ev_side, side));
        NPB_CUDA(cudaStreamWaitEvent(s, ev_side, 0));
    }
    // verdict: exact zeros / mismatches on this rank, shared with the peers (world > 1: the device-side counters go
    // straight into the all-reduce, one host synchronisation for the whole step)
    int any = tiles_ok ? 0 : 1;
    if (W > 1) {
        NPB_TRY(npb_k4_share_flags(c, bad, any, &any));
    } else {
        k_copy2_int<<<1, 1, 0, s>>>(c->d_small + 10, bad);
        NPB_LAUNCH(c);
        NPB_CUDA(cudaStreamSynchronize(s));
        if (c->h_small[10] != 0 || c->h_small[11] != 0) any = 1;
    }
    if (any) {
        *fell_back = 1;
        c->plan_failed[method] = true;
        c->plan_kind = 0;   // the two-pass path rewrites indptr
        return NPB_OK;
    }
    c->nnz = total;
    c->nnz_ret = total;
    c->blk_off = 0;
    c->method = method;
    c->counted = true;     // a later npb_interpolate_fetch copies these very arrays
    c->filled = true;
    c->csr_gen++;
    c->gathered = nccl_gather;
    return NPB_OK;
}

extern "C" int npb_interpolate_run(npb_ctx *c, int method, int n_chunks, const double *perm_host,
                                   const double *diff_mag_host, int32_t *indptr, int32_t *indices, double *data,
                                   double *neumann, int64_t capacity, int64_t *nnz, int *fell_back)
{
    if (!c || !nnz || !fell_back) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("Grid not initialized. Please load a mesh first.");
        return NPB_ERR_STATE;
    }
    if (method != NPB_METHOD_IDW && method != NPB_METHOD_LS && method != NPB_METHOD_GLS) {
        npb_set_error("unknown method id %d", method);
        return NPB_ERR_ARG;
    }
    if (c->world > 1 && c->gather_mode == NPB_GATHER_ROOT) {
        npb_set_error("npb_interpolate_run: gather = root uses npb_interpolate_count / npb_interpolate_fetch");
        return NPB_ERR_STATE;
    }
    if (!c->have_flags) {
        npb_set_error("neumann flags have not been set");
        return NPB_ERR_STATE;
    }
    const bool gls = method == NPB_METHOD_GLS;
    const bool upload = gls && perm_host && diff_mag_host;
    if (gls && !upload && (!c->have_perm || !c->have_dm)) {
        npb_set_error("GLS needs the 'permeability' and 'diff_mag' cell fields");
        return NPB_ERR_STATE;
    }
    for (const void *hp : {(const void *)indptr, (const void *)indices, (const void *)data, (const void *)neumann,
                           (const void *)(upload ? perm_host : nullptr), (const void *)(upload ? diff_mag_host : nullptr)})
        if (hp && !npb_is_pinned(hp)) {
            npb_set_error("npb_interpolate_run needs page-locked host arrays (npb_host_alloc / npb_host_register)");
            return NPB_ERR_ARG;
        }
    NPB_CUDA(cudaSetDevice(c->device));
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > 64) n_chunks = 64;
    if (c->plan_failed[method]) {   // same inputs -> same zeros: do not compute a result that will be discarded again
        *fell_back = 1;
        *nnz = 0;
        return NPB_OK;
    }
    NpbTimer tall(c, "streamed");
    int rc = run_pipeline(c, method, n_chunks, perm_host, diff_mag_host, indptr, indices, data, neumann, capacity, fell_back);
    if (rc != NPB_OK) {
        drain(c);   // nothing queued on the side streams may outlive the call: it targets caller buffers
        return rc;
    }
    tall.stop();
    *nnz = *fell_back ? 0 : c->nnz;
    return NPB_OK;
}

// round-1 name of the single-GPU pipeline; falls back to the two-pass path by itself
extern "C" int npb_interpolate_streamed(npb_ctx *c, int method, int n_chunks, const double *perm_host,
                                        const double *diff_mag_host, int32_t *indptr, int32_t *indices, double *data,
                                        double *neumann, int64_t capacity, int64_t *nnz)
{
    if (!c || !nnz || !indptr || !indices || !data || !neumann) return NPB_ERR_ARG;
    if (c->world != 1) {
        npb_set_error("npb_interpolate_streamed is the single-GPU entry point; use npb_interpolate_run");
        return NPB_ERR_STATE;
    }
    int fell_back = 0;
    NPB_TRY(npb_interpolate_run(c, method, n_chunks, perm_host, diff_mag_host, indptr, indices, data, neumann, capacity, nnz,
                                &fell_back));
    if (!fell_back) return NPB_OK;
    NPB_TRY(npb_interpolate_count(c, method, nnz));
    if (*nnz > capacity) {
        npb_set_error("npb_interpolate_streamed: capacity %lld too small for nnz %lld", (long long)capacity, (long long)*nnz);
        return NPB_ERR_ARG;
    }
    return npb_interpolate_fetch(c, indptr, indices, data, neumann);
}
