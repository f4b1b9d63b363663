// capi.cu — the extern "C" surface of libninpol_b200.so (include/ninpol_b200.h): context, error
// channel, mesh ingest, per-variable inputs, the interpolate count/fetch pair, timings, measurement
// helpers.  No kernels of the hot path live here; see k1_*.cu, k2_*.cu, k3_emit.cu, k4_shard.cu.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <thread>
#include "common.cuh"

static thread_local char g_err[1024] = "";

void npb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *npb_last_error(void) { return g_err; }
extern "C" int npb_version(void) { return 100; }

extern "C" int npb_device_count(int *count)
{
    if (!count) return NPB_ERR_ARG;
    *count = 0;
    NPB_CUDA(cudaGetDeviceCount(count));
    return NPB_OK;
}

// ---- guard words (debug aid; compute-sanitizer is not available on the pool) ----
// With NPB_DEBUG_GUARDS=1 every device block handed out by npb_alloc / npb_ensure is followed by 64 bytes of a known
// pattern; npb_check_guards reads them back.  A kernel that writes past the end of its buffer (the likeliest kind
// of bad access in the scatter / emit kernels) shows up in the GPU tests instead of corrupting a neighbour silently.
#include <map>
#include <mutex>
#define NPB_GUARD_BYTES 64
#define NPB_GUARD_BYTE 0xA5
static std::mutex g_guard_mu;
static std::map<void *, size_t> g_guard;   // block -> offset of its guard
static bool guards_on()
{
    static const bool on = [] { const char *e = getenv("NPB_DEBUG_GUARDS"); return e && e[0] == '1'; }();
    return on;
}
static int guard_arm(void *p, size_t offset)
{
    NPB_CUDA(cudaMemset((char *)p + offset, NPB_GUARD_BYTE, NPB_GUARD_BYTES));
    std::lock_guard<std::mutex> lk(g_guard_mu);
    g_guard[p] = offset;
    return NPB_OK;
}
void npb_guard_forget(void *p)
{
    if (!p || !guards_on()) return;
    std::lock_guard<std::mutex> lk(g_guard_mu);
    g_guard.erase(p);
}
extern "C" int npb_check_guards(npb_ctx *c, int64_t *n_blocks, int64_t *n_damaged)
{
    if (!c || !n_blocks || !n_damaged) return NPB_ERR_ARG;
    *n_blocks = *n_damaged = 0;
    if (!guards_on()) return NPB_OK;
    NPB_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lk(g_guard_mu);
    unsigned char h[NPB_GUARD_BYTES];
    for (auto &kv : g_guard) {
        NPB_CUDA(cudaMemcpy(h, (char *)kv.first + kv.second, NPB_GUARD_BYTES, cudaMemcpyDeviceToHost));
        bool ok = true;
        for (int i = 0; i < NPB_GUARD_BYTES; i++) ok = ok && h[i] == NPB_GUARD_BYTE;
        (*n_blocks)++;
        if (!ok) {
            (*n_damaged)++;
            npb_set_error("guard after device block %p (+%zu bytes) was overwritten", kv.first, kv.second);
        }
    }
    return NPB_OK;
}

int npb_alloc(npb_ctx *c, void **p, size_t bytes, bool owned_by_mesh)
{
    *p = nullptr;
    // 64 bytes of slack behind every block: guard mode arms its guard words there, and no kernel has been
    // audited for reads past the end of its inputs
    NPB_CUDA(cudaMalloc(p, bytes + 64));
    if (owned_by_mesh) c->owned.push_back(*p);
    if (guards_on()) NPB_TRY(guard_arm(*p, bytes));
    return NPB_OK;
}

int npb_ensure(void **p, size_t *cap, size_t bytes)
{
    if (*p && *cap >= bytes) return NPB_OK;
    if (*p) {
        npb_guard_forget(*p);
        NPB_CUDA(cudaFree(*p));
    }
    *p = nullptr;
    *cap = 0;
    if (guards_on()) {   // exact size + guard: the next larger request reallocates, so the guard follows the largest one
        NPB_CUDA(cudaMalloc(p, bytes + NPB_GUARD_BYTES));
        *cap = bytes;
        return guard_arm(*p, bytes);
    }
    size_t want = bytes + bytes / 8 + 256;
    NPB_CUDA(cudaMalloc(p, want));
    *cap = want;
    return NPB_OK;
}

__global__ void k_copy_int(int *dst, const int *src) { *dst = *src; }
__global__ void k_copy2_int(int *dst, const int *src)
{
    dst[0] = src[0];
    dst[1] = src[1];
}

int npb_read_int(npb_ctx *c, const int *d_src, int *h_out)
{
    k_copy_int<<<1, 1, 0, c->stream>>>(c->d_small + 8, d_src);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    *h_out = c->h_small[8];
    return NPB_OK;
}

NpbTimer::NpbTimer(npb_ctx *c_, const char *n, bool accumulate_) : c(c_), name(n), a(nullptr), b(nullptr), accumulate(accumulate_)
{
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, c->stream);
}
void NpbTimer::stop_lazy()
{
    if (!a) return;
    cudaEventRecord(b, c->stream);
    if (c->pending_timers.size() > 64) npb_resolve_timers(c);
    c->pending_timers.push_back({name, a, b, accumulate});
    a = b = nullptr;
}

void npb_resolve_timers(npb_ctx *c)
{
    for (auto &p : c->pending_timers) {
        float ms = 0.f;
        if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            if (p.accumulate)
                c->timings[p.name] += ms;
            else
                c->timings[p.name] = ms;
        }
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    c->pending_timers.clear();
}

NpbTimer::~NpbTimer()
{
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
}
void NpbTimer::stop()
{
    if (!a) return;
    cudaEventRecord(b, c->stream);
    cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    if (accumulate)
        c->timings[name] += ms;
    else
        c->timings[name] = ms;
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    a = b = nullptr;
}


// ------------------------------------------------------------------------------------------------
// Host <-> device copies for PAGEABLE caller memory (numpy arrays): staged through two page-locked
// buffers, the host-side memcpy of chunk i+1 (split over a few threads) overlapping the DMA of chunk i.
// cudaMemcpy on pageable memory does the same staging single-threaded at 6-10 GB/s; this reaches the
// PCIe rate.  Page-locked caller memory (npb_host_alloc) is detected and copied directly.
// ------------------------------------------------------------------------------------------------
#define NPB_STAGE_BYTES ((size_t)32 << 20)
#define NPB_STAGE_THREADS 4

static void par_memcpy(void *dst, const void *src, size_t n)
{
    if (n < ((size_t)4 << 20)) {
        memcpy(dst, src, n);
        return;
    }
    std::thread th[NPB_STAGE_THREADS];
    size_t part = (n + NPB_STAGE_THREADS - 1) / NPB_STAGE_THREADS;
    part = (part + 4095) & ~(size_t)4095;
    for (int t = 0; t < NPB_STAGE_THREADS; t++) {
        size_t b = (size_t)t * part;
        size_t len = b >= n ? 0 : (n - b < part ? n - b : part);
        th[t] = std::thread([=]() {
            if (len) memcpy((char *)dst + b, (const char *)src + b, len);
        });
    }
    for (int t = 0; t < NPB_STAGE_THREADS; t++) th[t].join();
}

bool npb_is_pinned(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

static int ensure_stage(npb_ctx *c)
{
    for (int i = 0; i < 2; i++)
        if (!c->stage[i]) {
            NPB_CUDA(cudaHostAlloc(&c->stage[i], NPB_STAGE_BYTES, cudaHostAllocDefault));
            NPB_CUDA(cudaEventCreateWithFlags(&c->stage_ev[i], cudaEventDisableTiming));
        }
    return NPB_OK;
}

int npb_h2d(npb_ctx *c, void *dst_dev, const void *src_host, size_t bytes)
{
    if (bytes == 0) return NPB_OK;
    if (bytes < ((size_t)8 << 20) || npb_is_pinned(src_host)) {
        NPB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, c->stream));
        return NPB_OK;
    }
    NPB_TRY(ensure_stage(c));
    int k = 0;
    for (size_t off = 0; off < bytes; off += NPB_STAGE_BYTES, k ^= 1) {
        size_t n = bytes - off < NPB_STAGE_BYTES ? bytes - off : NPB_STAGE_BYTES;
        NPB_CUDA(cudaEventSynchronize(c->stage_ev[k]));   // the DMA that last read this buffer is done
        par_memcpy(c->stage[k], (const char *)src_host + off, n);
        NPB_CUDA(cudaMemcpyAsync((char *)dst_dev + off, c->stage[k], n, cudaMemcpyHostToDevice, c->stream));
        NPB_CUDA(cudaEventRecord(c->stage_ev[k], c->stream));
    }
    return NPB_OK;
}

// blocking: returns when dst_host holds the data
int npb_d2h(npb_ctx *c, void *dst_host, const void *src_dev, size_t bytes)
{
    if (bytes == 0) return NPB_OK;
    if (bytes < ((size_t)8 << 20) || npb_is_pinned(dst_host)) {
        NPB_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, c->stream));
        NPB_CUDA(cudaStreamSynchronize(c->stream));
        return NPB_OK;
    }
    NPB_TRY(ensure_stage(c));
    size_t nchunks = (bytes + NPB_STAGE_BYTES - 1) / NPB_STAGE_BYTES;
    for (size_t i = 0; i <= nchunks; i++) {
        if (i < nchunks) {   // start the DMA of chunk i
            size_t off = i * NPB_STAGE_BYTES, n = bytes - off < NPB_STAGE_BYTES ? bytes - off : NPB_STAGE_BYTES;
            NPB_CUDA(cudaMemcpyAsync(c->stage[i & 1], (const char *)src_dev + off, n, cudaMemcpyDeviceToHost, c->stream));
            NPB_CUDA(cudaEventRecord(c->stage_ev[i & 1], c->stream));
        }
        if (i > 0) {         // drain chunk i-1 while chunk i is in flight
            size_t off = (i - 1) * NPB_STAGE_BYTES, n = bytes - off < NPB_STAGE_BYTES ? bytes - off : NPB_STAGE_BYTES;
            NPB_CUDA(cudaEventSynchronize(c->stage_ev[(i - 1) & 1]));
            par_memcpy((char *)dst_host + off, c->stage[(i - 1) & 1], n);
        }
    }
    return NPB_OK;
}

int npb_comm_destroy(npb_ctx *c);
int npb_psup_stats(npb_ctx *c);

static void free_mesh(npb_ctx *c)
{
    for (void *p : c->owned) {
        npb_guard_forget(p);
        cudaFree(p);
    }
    c->owned.clear();
    c->inpoel = c->esup_ptr = c->esup = c->esuel = c->infael = c->inpofa = c->fsup_ptr = c->fsup = nullptr;
    c->psup_ptr = c->psup = c->node_list = nullptr;
    c->inedel_d = c->inpoed_d = nullptr;
    c->n_edges = 0;
    c->etype = c->bface = c->bpoint = c->nflag = nullptr;
    c->esuf2 = nullptr;
    c->coords = c->centroids = c->fcent = c->fnormal = c->farea = c->perm = c->diff_mag = c->neumann = nullptr;
    c->rowcnt = c->indptr = nullptr;
    c->have_perm = c->have_dm = c->have_flags = false;
    c->fused_failed[0] = c->fused_failed[1] = false;
    c->mesh_loaded = false;
    c->counted = false;
    c->csr_gen++;
    c->plan_kind = 0;
    c->plan_chunks = 0;
    c->chunk_node.clear();
    c->chunk_efirst.clear();
    c->chunk_elast.clear();
    c->plan_failed[0] = c->plan_failed[1] = c->plan_failed[2] = false;
    c->apply_range_ok = false;
}

extern "C" int npb_create(int device, npb_ctx **out)
{
    if (!out) {
        npb_set_error("npb_create: null output");
        return NPB_ERR_ARG;
    }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        npb_set_error("no CUDA device available (%s); libninpol_b200 has no CPU fallback",
                      e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return NPB_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        npb_set_error("device %d out of range (have %d)", device, n);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    NPB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        npb_set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return NPB_ERR_CUDA;
    }
    npb_ctx *c = new npb_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    auto init = [&]() -> int {
        NPB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        NPB_CUDA(cudaMalloc(&c->counters, sizeof(int) * 128));
        NPB_CUDA(cudaMemset(c->counters, 0, sizeof(int) * 128));
        NPB_CUDA(cudaHostAlloc((void **)&c->h_small, sizeof(int) * 64, cudaHostAllocMapped));
        NPB_CUDA(cudaHostGetDevicePointer((void **)&c->d_small, c->h_small, 0));
        return NPB_OK;
    };
    int rc = init();
    if (rc != NPB_OK) {   // nothing half-built survives a failed create
        if (c->h_small) cudaFreeHost(c->h_small);
        if (c->counters) cudaFree(c->counters);
        if (c->stream) cudaStreamDestroy(c->stream);
        delete c;
        return rc;
    }
    *out = c;
    return NPB_OK;
}

extern "C" int npb_destroy(npb_ctx *c)
{
    if (!c) return NPB_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    npb_resolve_timers(c);
    npb_comm_destroy(c);
    free_mesh(c);
    if (c->wbuf) { npb_guard_forget(c->wbuf); cudaFree(c->wbuf); }
    if (c->indices) { npb_guard_forget(c->indices); cudaFree(c->indices); }
    if (c->data) { npb_guard_forget(c->data); cudaFree(c->data); }
    if (c->scratch) { npb_guard_forget(c->scratch); cudaFree(c->scratch); }
    if (c->scan_tmp) { npb_guard_forget(c->scan_tmp); cudaFree(c->scan_tmp); }
    if (c->part_tmp) { npb_guard_forget(c->part_tmp); cudaFree(c->part_tmp); }
    if (c->gls_ws) { npb_guard_forget(c->gls_ws); cudaFree(c->gls_ws); }
    if (c->apply_x) { npb_guard_forget(c->apply_x); cudaFree(c->apply_x); }
    if (c->apply_y) { npb_guard_forget(c->apply_y); cudaFree(c->apply_y); }
    if (c->tmap) { npb_guard_forget(c->tmap); cudaFree(c->tmap); }
    if (c->counters) cudaFree(c->counters);
    if (c->h_small) cudaFreeHost(c->h_small);
    for (int i = 0; i < 2; i++) {
        if (c->stage[i]) cudaFreeHost(c->stage[i]);
        if (c->stage_ev[i]) cudaEventDestroy(c->stage_ev[i]);
    }
    for (cudaEvent_t e : c->pipe_ev) cudaEventDestroy(e);
    if (c->up_stream) cudaStreamDestroy(c->up_stream);
    if (c->down_stream) cudaStreamDestroy(c->down_stream);
    if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
    if (c->ev_a) cudaEventDestroy(c->ev_a);
    if (c->ev_b) cudaEventDestroy(c->ev_b);
    cudaStreamDestroy(c->stream);
    delete c;
    return NPB_OK;
}

extern "C" int npb_synchronize(npb_ctx *c)
{
    if (!c) return NPB_ERR_ARG;
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// partition
// ------------------------------------------------------------------------------------------------
static int refresh_range(npb_ctx *c)
{
    if (c->bounds.size() != (size_t)c->world + 1) {
        // default: rank 0 .. world-1 get equal node counts
        c->bounds.resize(c->world + 1);
        for (int r = 0; r <= c->world; r++) c->bounds[r] = (c->n_points * r) / c->world;
    }
    c->lo = c->bounds[c->rank];
    c->hi = c->bounds[c->rank + 1];
    int32_t b[2] = {0, 0};
    NPB_CUDA(cudaMemcpyAsync(&b[0], c->esup_ptr + c->lo, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaMemcpyAsync(&b[1], c->esup_ptr + c->hi, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    c->wbase = b[0];
    c->wlen = (i64)b[1] - b[0];
    c->counted = false;
    c->csr_gen++;
    c->plan_chunks = 0;   // chunk boundaries follow the rank bounds
    c->apply_range_ok = false;
    return NPB_OK;
}

extern "C" int npb_set_partition(npb_ctx *c, const int64_t *bounds, int n_bounds)
{
    if (!c || !bounds) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_set_partition: no mesh loaded");
        return NPB_ERR_STATE;
    }
    if (n_bounds != c->world + 1 || bounds[0] != 0 || bounds[n_bounds - 1] != c->n_points) {
        npb_set_error("npb_set_partition: need %d bounds from 0 to n_points", c->world + 1);
        return NPB_ERR_ARG;
    }
    for (int r = 0; r < c->world; r++)
        if (bounds[r + 1] < bounds[r]) {
            npb_set_error("npb_set_partition: bounds must be non-decreasing");
            return NPB_ERR_ARG;
        }
    NPB_CUDA(cudaSetDevice(c->device));
    c->bounds.assign(bounds, bounds + n_bounds);
    return refresh_range(c);
}

extern "C" int npb_set_gather(npb_ctx *c, int mode)
{
    if (!c || (mode != NPB_GATHER_ALL && mode != NPB_GATHER_ROOT && mode != NPB_GATHER_HOST)) {
        npb_set_error("npb_set_gather: mode must be NPB_GATHER_ALL, NPB_GATHER_ROOT or NPB_GATHER_HOST");
        return NPB_ERR_ARG;
    }
    c->gather_mode = mode;
    c->counted = false;
    c->csr_gen++;
    return NPB_OK;
}

extern "C" int npb_partition_elem_range(npb_ctx *c, int64_t *first, int64_t *last)
{
    if (!c || !first || !last) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_partition_elem_range: no mesh loaded");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    int32_t ptr[2] = {0, 0};
    NPB_CUDA(cudaMemcpyAsync(&ptr[0], c->esup_ptr + c->lo, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaMemcpyAsync(&ptr[1], c->esup_ptr + c->hi, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    int32_t mn = 0, mx = -1;
    NPB_TRY(npb_minmax_i32(c, c->esup + ptr[0], (i64)ptr[1] - ptr[0], &mn, &mx));
    *first = mn;
    *last = mx;
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------------
extern "C" int npb_load_mesh(npb_ctx *c, int dim, int64_t n_elems, int64_t n_points, const int64_t *conn,
                             const int64_t *types, const int64_t *npoel, const int64_t *nfael, const int64_t *lnofa,
                             const int64_t *lpofa, const int64_t *nedel, const int64_t *lpoed, const double *coords,
                             int build_edges)
{
    return npb_load_mesh_strided(c, dim, n_elems, n_points, conn, NPB_MX_PE, types, npoel, nfael, lnofa, lpofa, nedel,
                                 lpoed, coords, build_edges);
}

extern "C" int npb_load_mesh_strided(npb_ctx *c, int dim, int64_t n_elems, int64_t n_points, const int64_t *conn,
                                     int conn_stride, const int64_t *types, const int64_t *npoel, const int64_t *nfael,
                                     const int64_t *lnofa, const int64_t *lpofa, const int64_t *nedel,
                                     const int64_t *lpoed, const double *coords, int build_edges)
{
    if (conn_stride < 1 || conn_stride > NPB_MX_PE) {
        npb_set_error("npb_load_mesh_strided: conn_stride must be in [1, %d]", NPB_MX_PE);
        return NPB_ERR_ARG;
    }
    if (!c || !conn || !types || !npoel || !nfael || !lnofa || !lpofa || !coords) {
        npb_set_error("npb_load_mesh: null argument");
        return NPB_ERR_ARG;
    }
    // same argument checks (and messages) as Grid.__cinit__, grid.pyx:55-60
    if (dim < 1) {
        npb_set_error("The number of dimensions must be greater than 0.");
        return NPB_ERR_ARG;
    }
    if (n_elems < 1) {
        npb_set_error("The number of elements must be greater than 0.");
        return NPB_ERR_ARG;
    }
    if (n_points < 1) {
        npb_set_error("The number of points must be greater than 0.");
        return NPB_ERR_ARG;
    }
    if (n_elems * NPB_MX_PE >= (1ll << 31) || n_points >= (1ll << 31) - 1) {
        npb_set_error("mesh too large for 32-bit device ids (n_elems=%lld, n_points=%lld)", (long long)n_elems,
                      (long long)n_points);
        return NPB_ERR_RANGE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    free_mesh(c);
    c->bounds.clear();
    c->dim = dim;
    c->n_elems = n_elems;
    c->n_points = n_points;
    c->build_edges = build_edges != 0;
    // tables; spe / sfe from the element types of this mesh dimension
    memset(&c->tab, 0, sizeof(c->tab));
    memset(&c->etab, 0, sizeof(c->etab));
    int mxp = 0, mxf = 0;
    for (int t = 0; t < NPB_N_TYPES; t++) {
        c->tab.npoel[t] = (int8_t)npoel[t];
        c->tab.nfael[t] = (int8_t)(nfael[t] < 0 ? 0 : nfael[t]);
        for (int f = 0; f < NPB_MX_FE; f++) {
            c->tab.lnofa[t][f] = (int8_t)(lnofa[t * NPB_MX_FE + f] < 0 ? 0 : lnofa[t * NPB_MX_FE + f]);
            for (int k = 0; k < NPB_MX_PF; k++) {
                int64_t v = lpofa[(t * NPB_MX_FE + f) * NPB_MX_PF + k];
                c->tab.lpofa[t][f][k] = (int8_t)(v < 0 ? 0 : v);
            }
        }
        if (nedel && lpoed) {
            c->etab.nedel[t] = (int8_t)(nedel[t] < 0 ? 0 : nedel[t]);
            for (int e = 0; e < NPB_MX_EE; e++)
                for (int k = 0; k < 2; k++) {
                    int64_t v = lpoed[(t * NPB_MX_EE + e) * 2 + k];
                    c->etab.lpoed[t][e][k] = (int8_t)(v < 0 ? 0 : v);
                }
        }
    }
    // device row strides from the element types that are actually present in the mesh
    bool present[NPB_N_TYPES] = {false, false, false, false, false, false, false, false};
    for (int64_t e = 0; e < n_elems; e++) {
        int64_t t = types[e];
        if (t < 0 || t >= NPB_N_TYPES || nfael[t] < 0) {
            npb_set_error("element %lld has type %lld, which is not a cell type of a %d-D mesh", (long long)e, (long long)t, dim);
            return NPB_ERR_ARG;
        }
        present[t] = true;
    }
    for (int t = 0; t < NPB_N_TYPES; t++) {
        if (present[t]) {
            if (npoel[t] > mxp) mxp = (int)npoel[t];
            if (nfael[t] > mxf) mxf = (int)nfael[t];
        }
    }
    c->spe = mxp <= 4 ? 4 : 8;
    c->sfe = mxf <= 4 ? 4 : 6;
    {   // the device indexes fsup / esuf / inpofa with int32 as well: bound their flat lengths by the present types
        int64_t fn = 0;   // max over present types of sum_f lnofa[t][f] (node incidences of an element's faces)
        for (int t = 0; t < NPB_N_TYPES; t++) {
            if (!present[t]) continue;
            int64_t sum = 0;
            for (int f = 0; f < c->tab.nfael[t]; f++) sum += c->tab.lnofa[t][f];
            if (sum > fn) fn = sum;
        }
        if (n_elems * fn >= (1ll << 31) || n_elems * (int64_t)mxf * NPB_MX_PF >= (1ll << 31)) {
            npb_set_error("mesh too large for 32-bit device ids: up to %lld node->face incidences (n_elems=%lld)",
                          (long long)(n_elems * fn), (long long)n_elems);
            return NPB_ERR_RANGE;
        }
    }
    if (mxp > conn_stride) {
        npb_set_error("npb_load_mesh_strided: conn_stride %d is smaller than the %d nodes of an element type present", conn_stride, mxp);
        return NPB_ERR_ARG;
    }
    int rc = npb_k1_build(c, (const i64 *)conn, conn_stride, (const i64 *)types, coords);
    if (rc != NPB_OK) {
        free_mesh(c);
        return rc;
    }
    NPB_TRY(npb_alloc(c, (void **)&c->rowcnt, sizeof(int32_t) * (n_points + 1)));
    NPB_TRY(npb_alloc(c, (void **)&c->indptr, sizeof(int32_t) * (n_points + 1)));
    NPB_TRY(npb_alloc(c, (void **)&c->neumann, sizeof(double) * n_points));
    NPB_TRY(npb_alloc(c, (void **)&c->nflag, (size_t)n_points));
    c->mesh_loaded = true;
    NPB_TRY(npb_k1_extras(c));
    return refresh_range(c);
}

extern "C" int npb_grid_scalar(npb_ctx *c, const char *name, int64_t *out)
{
    if (!c || !name || !out) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_grid_scalar: no mesh loaded");
        return NPB_ERR_STATE;
    }
    if (!strcmp(name, "MX_POINTS_PER_POINT") || !strcmp(name, "len_psup")) {
        NPB_CUDA(cudaSetDevice(c->device));
        NPB_TRY(npb_psup_stats(c));
    }
    struct { const char *n; i64 v; } tbl[] = {
        {"dim", c->dim}, {"n_elems", c->n_elems}, {"n_points", c->n_points}, {"n_faces", c->n_faces},
        {"n_edges", c->n_edges}, {"MX_ELEMENTS_PER_POINT", c->mx_epp}, {"MX_POINTS_PER_POINT", c->mx_ppp},
        {"MX_ELEMENTS_PER_FACE", c->mx_epf}, {"MX_FACES_PER_POINT", c->mx_fpp}, {"len_esup", c->len_esup},
        {"len_fsup", c->len_fsup}, {"len_esuf", c->len_esuf}, {"len_psup", c->len_psup},
        {"row_lo", c->lo}, {"row_hi", c->hi}, {"rank", c->rank}, {"world", c->world}, {"sm_count", c->sm_count},
        {"have_cell_fields", (c->have_perm && c->have_dm) ? 1 : 0}, {"plan_nnz", c->plan_nnz}, {"flags_checksum", c->flags_checksum},
    };
    for (auto &e : tbl)
        if (strcmp(e.n, name) == 0) {
            *out = e.v;
            return NPB_OK;
        }
    npb_set_error("npb_grid_scalar: unknown name '%s'", name);
    return NPB_ERR_ARG;
}

extern "C" int npb_grid_array(npb_ctx *c, const char *name, void *out, int64_t cap)
{
    if (!c || !name || !out) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_grid_array: no mesh loaded");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    return npb_export_array(c, name, out, cap);
}

// ------------------------------------------------------------------------------------------------
// per-variable inputs
// ------------------------------------------------------------------------------------------------
extern "C" int npb_set_cell_field(npb_ctx *c, const char *name, const double *data, int64_t n)
{
    if (!c || !name || !data) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_set_cell_field: no mesh loaded");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    if (strcmp(name, "permeability") == 0) {
        if (n != 9 * c->n_elems) {
            npb_set_error("permeability needs 9*n_elems = %lld values, got %lld", (long long)(9 * c->n_elems), (long long)n);
            return NPB_ERR_ARG;
        }
        if (!c->perm) NPB_TRY(npb_alloc(c, (void **)&c->perm, sizeof(double) * n));
        NPB_TRY(npb_h2d(c, c->perm, data, sizeof(double) * n));
        c->have_perm = true;
    } else if (strcmp(name, "diff_mag") == 0) {
        if (n != c->n_elems) {
            npb_set_error("diff_mag needs n_elems = %lld values, got %lld", (long long)c->n_elems, (long long)n);
            return NPB_ERR_ARG;
        }
        if (!c->diff_mag) NPB_TRY(npb_alloc(c, (void **)&c->diff_mag, sizeof(double) * n));
        NPB_TRY(npb_h2d(c, c->diff_mag, data, sizeof(double) * n));
        c->have_dm = true;
    } else {
        npb_set_error("npb_set_cell_field: unknown field '%s'", name);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    c->counted = false;
    c->csr_gen++;
    c->plan_failed[NPB_METHOD_GLS] = false;
    return NPB_OK;
}

extern "C" int npb_set_cell_field_range(npb_ctx *c, const char *name, const double *data, int64_t first_elem,
                                        int64_t n_elems_in_range)
{
    if (!c || !name || (!data && n_elems_in_range > 0)) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_set_cell_field_range: no mesh loaded");
        return NPB_ERR_STATE;
    }
    if (first_elem < 0 || n_elems_in_range < 0 || first_elem + n_elems_in_range > c->n_elems) {
        npb_set_error("npb_set_cell_field_range: elements [%lld, %lld) outside [0, %lld)", (long long)first_elem,
                      (long long)(first_elem + n_elems_in_range), (long long)c->n_elems);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    if (strcmp(name, "permeability") == 0) {
        if (!c->perm) NPB_TRY(npb_alloc(c, (void **)&c->perm, sizeof(double) * 9 * (size_t)c->n_elems));
        NPB_TRY(npb_h2d(c, c->perm + 9 * first_elem, data, sizeof(double) * 9 * (size_t)n_elems_in_range));
        c->have_perm = true;
    } else if (strcmp(name, "diff_mag") == 0) {
        if (!c->diff_mag) NPB_TRY(npb_alloc(c, (void **)&c->diff_mag, sizeof(double) * (size_t)c->n_elems));
        NPB_TRY(npb_h2d(c, c->diff_mag + first_elem, data, sizeof(double) * (size_t)n_elems_in_range));
        c->have_dm = true;
    } else {
        npb_set_error("npb_set_cell_field_range: unknown field '%s'", name);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    c->counted = false;
    c->csr_gen++;
    c->plan_failed[NPB_METHOD_GLS] = false;
    return NPB_OK;
}

// Both flag kernels also fold WHICH nodes are flagged into a 64-bit checksum: the wrapping sum, over the flagged nodes, of
// a mixed (splitmix64) image of the node id.  The host re-cuts the node partition only when it changes, without a pass
// over the array; being a sum, it can be formed slice by slice on different ranks (npb_set_point_flags_f64_range).
#define NPB_FLAG_MIX 0x9E3779B97F4A7C15ull
static int read_flag_checksum(npb_ctx *c);
__device__ __forceinline__ void flag_checksum(bool set, i64 i, unsigned long long *sum)
{
    unsigned long long v = 0ull;
    if (set) {
        v = (unsigned long long)(i + 1) * NPB_FLAG_MIX;
        v ^= v >> 30; v *= 0xBF58476D1CE4E5B9ull;
        v ^= v >> 27; v *= 0x94D049BB133111EBull;
        v ^= v >> 31;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(sum, v);
}

__global__ void k_flags(const i64 *__restrict__ in, i64 n, uint8_t *__restrict__ out, unsigned long long *__restrict__ sum)
{
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    bool set = false;
    if (i < n) {
        set = in[i] != 0;
        out[i] = set ? 1 : 0;
    }
    flag_checksum(set, i, sum);
}

extern "C" int npb_set_point_flags(npb_ctx *c, const int64_t *flag, int64_t n_points)
{
    if (!c || !flag) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_set_point_flags: no mesh loaded");
        return NPB_ERR_STATE;
    }
    if (n_points != c->n_points) {
        npb_set_error("neumann flags need n_points = %lld values, got %lld", (long long)c->n_points, (long long)n_points);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    // staged through the persistent scratch block: a cudaMalloc / cudaFree pair per call costs tens of
    // milliseconds once gigabytes of page-locked host memory are mapped
    NPB_TRY(npb_ensure(&c->scratch, &c->scratch_cap, sizeof(i64) * (size_t)n_points));
    i64 *tmp = (i64 *)c->scratch;
    NPB_TRY(npb_h2d(c, tmp, flag, sizeof(i64) * n_points));
    NPB_CUDA(cudaMemsetAsync(c->counters + 66, 0, sizeof(unsigned long long), c->stream));
    k_flags<<<npb_blocks(n_points, 256), 256, 0, c->stream>>>(tmp, n_points, c->nflag, (unsigned long long *)(c->counters + 66));
    NPB_LAUNCH(c);
    NPB_TRY(read_flag_checksum(c));
    c->have_flags = true;
    c->counted = false;
    c->csr_gen++;
    c->plan_kind = 0;     // row lengths depend on the flags
    c->plan_failed[0] = c->plan_failed[1] = c->plan_failed[2] = false;
    c->fused_failed[0] = c->fused_failed[1] = false;
    return NPB_OK;
}

__global__ void k_flags_f64(const double *__restrict__ in, i64 first, i64 n, uint8_t *__restrict__ out,
                            unsigned long long *__restrict__ sum)
{
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;   // local index: in[i] is node first + i
    bool set = false;
    if (i < n) {
        double f = in[i];
        // numpy's float64 -> int64 cast truncates toward zero; NaN / inf become INT64_MIN (non-zero)
        set = (f != f || (long long)f != 0);
        out[first + i] = set ? 1 : 0;
    }
    flag_checksum(set, first + i, sum);
}

static int read_flag_checksum(npb_ctx *c)
{
    unsigned long long h = 0;
    NPB_CUDA(cudaMemcpyAsync(&h, c->counters + 66, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    c->flags_checksum = (i64)(h >> 1);     // non-negative for the int64 scalar interface
    return NPB_OK;
}

extern "C" int npb_set_point_flags_f64(npb_ctx *c, const double *flag, int64_t n_points)
{
    if (!c || !flag) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("npb_set_point_flags_f64: no mesh loaded");
        return NPB_ERR_STATE;
    }
    if (n_points != c->n_points) {
        npb_set_error("neumann flags need n_points = %lld values, got %lld", (long long)c->n_points, (long long)n_points);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    NPB_TRY(npb_ensure(&c->scratch, &c->scratch_cap, sizeof(double) * (size_t)n_points));
    NPB_TRY(npb_h2d(c, c->scratch, flag, sizeof(double) * n_points));
    NPB_CUDA(cudaMemsetAsync(c->counters + 66, 0, sizeof(unsigned long long), c->stream));
    k_flags_f64<<<npb_blocks(n_points, 256), 256, 0, c->stream>>>((const double *)c->scratch, 0, n_points, c->nflag,
                                                                  (unsigned long long *)(c->counters + 66));
    NPB_LAUNCH(c);
    NPB_TRY(read_flag_checksum(c));
    c->have_flags = true;
    c->counted = false;
    c->csr_gen++;
    c->plan_kind = 0;     // row lengths depend on the flags
    c->plan_failed[0] = c->plan_failed[1] = c->plan_failed[2] = false;
    c->fused_failed[0] = c->fused_failed[1] = false;
    return NPB_OK;
}

int npb_k4_allreduce_u64(npb_ctx *c, unsigned long long *d_value);

// Multi-GPU re-staging of flags that are expected to be unchanged: this rank uploads only the slice [first, first + count)
// of the float64 flag row (the nodes it owns), the ranks add up the checksums of their slices, and *checksum is that
// total in the form of the "flags_checksum" scalar.  When it equals the checksum of the flags already resident, the
// other slices on this device are still right and nothing else needs to move (the row plan stays valid); otherwise the
// caller uploads the whole row with npb_set_point_flags_f64.  The slices of the ranks must tile [0, n_points).
extern "C" int npb_set_point_flags_f64_range(npb_ctx *c, const double *flag_slice, int64_t first, int64_t count, int64_t *checksum)
{
    if (!c || !checksum || (count > 0 && !flag_slice)) return NPB_ERR_ARG;
    if (!c->mesh_loaded || !c->have_flags) {
        npb_set_error("npb_set_point_flags_f64_range: a full flag row must have been set for this mesh first");
        return NPB_ERR_STATE;
    }
    if (first < 0 || count < 0 || first + count > c->n_points) {
        npb_set_error("npb_set_point_flags_f64_range: slice [%lld, %lld) outside [0, %lld)", (long long)first,
                      (long long)(first + count), (long long)c->n_points);
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    unsigned long long *sum = (unsigned long long *)(c->counters + 66);
    NPB_CUDA(cudaMemsetAsync(sum, 0, sizeof(unsigned long long), c->stream));
    if (count > 0) {
        NPB_TRY(npb_ensure(&c->scratch, &c->scratch_cap, sizeof(double) * (size_t)count));
        NPB_TRY(npb_h2d(c, c->scratch, flag_slice, sizeof(double) * (size_t)count));
        k_flags_f64<<<npb_blocks(count, 256), 256, 0, c->stream>>>((const double *)c->scratch, first, count, c->nflag, sum);
        NPB_LAUNCH(c);
    }
    if (c->world > 1) NPB_TRY(npb_k4_allreduce_u64(c, sum));
    unsigned long long h = 0;
    NPB_CUDA(cudaMemcpyAsync(&h, sum, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    *checksum = (i64)(h >> 1);
    if (*checksum != c->flags_checksum) {   // the flags changed somewhere: this device's copy is no longer trustworthy
        c->counted = false;
        c->csr_gen++;
        c->plan_kind = 0;
    }
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// K2 + K3 (+ K4)
// ------------------------------------------------------------------------------------------------
extern "C" int npb_interpolate_count(npb_ctx *c, int method, int64_t *nnz)
{
    if (!c || !nnz) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("Grid not initialized. Please load a mesh first.");
        return NPB_ERR_STATE;
    }
    if (method != NPB_METHOD_IDW && method != NPB_METHOD_LS && method != NPB_METHOD_GLS) {
        npb_set_error("unknown method id %d", method);
        return NPB_ERR_ARG;
    }
    if (!c->have_flags) {
        npb_set_error("neumann flags have not been set");
        return NPB_ERR_STATE;
    }
    if (method == NPB_METHOD_GLS && (!c->have_perm || !c->have_dm)) {
        npb_set_error("GLS needs the 'permeability' and 'diff_mag' cell fields");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    c->filled = false;
    c->csr_gen++;
    c->gathered = false;
    c->plan_kind = 0;     // this path rewrites indptr / neumann
    if (method != NPB_METHOD_GLS && !c->fused_failed[method]) {
        // fused K2+K3 (k2_idw_ls_tile.cu): final CSR in one pass unless a weight is an exact zero
        NpbTimer tm(c, "k2");
        int used = 0;
        NPB_TRY(npb_k2_idw_ls_fused(c, method, &used));
        tm.stop();
        if (!used && c->world == 1) c->fused_failed[method] = true;   // same inputs -> same zeros next time
        if (used) {
            c->timings["k3_count"] = 0.f;
            c->timings["k3_fill"] = 0.f;
            c->method = method;
            c->counted = true;
            c->filled = true;
            c->csr_gen++;
            c->nnz_ret = c->nnz;
            c->blk_off = 0;
            *nnz = c->nnz;
            return NPB_OK;
        }
    }
    NPB_TRY(npb_ensure((void **)&c->wbuf, &c->wbuf_cap, sizeof(double) * (size_t)(c->wlen > 0 ? c->wlen : 1)));
    {
        NpbTimer tm(c, "k2");
        if (method == NPB_METHOD_GLS)
            NPB_TRY(npb_k2_gls(c, c->lo, c->hi));
        else {
            int used = 0;
            NPB_TRY(npb_k2_idw_ls_tiles(c, method, c->lo, c->hi, &used));
            if (!used) {
                NPB_TRY(npb_k2_idw_ls(c, method, c->lo, c->hi));
                c->timings.erase("k2_main");
            }
        }
        tm.stop();
        npb_resolve_timers(c);
        if (method != NPB_METHOD_GLS && !c->timings.count("k2_main")) c->timings["k2_main"] = c->timings["k2"];
    }
    {
        NpbTimer tm(c, "k3_count");
        if (c->world > 1) {
            NpbTimer tg(c, "k4_gather_counts");
            NPB_TRY(npb_k4_gather_counts(c));
            tg.stop();
        }
        NPB_CUDA(cudaMemsetAsync(c->rowcnt + c->n_points, 0, sizeof(int32_t), s));
        NPB_TRY(npb_exclusive_scan_i32(c, c->rowcnt, c->indptr, c->n_points + 1));
        int32_t total = 0;
        NPB_CUDA(cudaMemcpyAsync(&total, c->indptr + c->n_points, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        tm.stop();
        c->nnz = total;
    }
    c->nnz_ret = c->nnz;
    c->blk_off = 0;
    if (c->world > 1 && c->gather_mode == NPB_GATHER_ROOT && c->rank != 0) {
        int32_t o[2] = {0, 0};
        NPB_CUDA(cudaMemcpyAsync(&o[0], c->indptr + c->lo, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        NPB_CUDA(cudaMemcpyAsync(&o[1], c->indptr + c->hi, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        NPB_CUDA(cudaStreamSynchronize(s));
        c->blk_off = o[0];
        c->nnz_ret = (i64)o[1] - o[0];
    }
    c->method = method;
    c->counted = true;
    c->csr_gen++;
    *nnz = c->nnz_ret;
    return NPB_OK;
}

int npb_ensure_out(npb_ctx *c, size_t n)
{
    size_t n1 = n > 0 ? n : 1;
    if (c->out_cap >= n1) return NPB_OK;
    if (c->indices) {
        npb_guard_forget(c->indices);
        NPB_CUDA(cudaFree(c->indices));
    }
    if (c->data) {
        npb_guard_forget(c->data);
        NPB_CUDA(cudaFree(c->data));
    }
    c->indices = nullptr;
    c->data = nullptr;
    c->out_cap = 0;
    size_t want = guards_on() ? n1 : n1 + n1 / 16 + 64;   // guard mode: exact capacity, guard right behind it
    NPB_CUDA(cudaMalloc(&c->indices, sizeof(int32_t) * want + NPB_GUARD_BYTES));
    NPB_CUDA(cudaMalloc(&c->data, sizeof(double) * want + NPB_GUARD_BYTES));
    c->out_cap = want;
    if (guards_on()) {
        NPB_TRY(guard_arm(c->indices, sizeof(int32_t) * want));
        NPB_TRY(guard_arm(c->data, sizeof(double) * want));
    }
    return NPB_OK;
}

__global__ void k_block_indptr(const int32_t *__restrict__ indptr, i64 n, int32_t lo, int32_t hi, int32_t *__restrict__ out)
{
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        int32_t v = indptr[i];
        out[i] = (v < lo ? lo : v > hi ? hi : v) - lo;
    }
}

extern "C" int npb_interpolate_fetch(npb_ctx *c, int32_t *indptr, int32_t *indices, double *data, double *neumann)
{
    if (!c) return NPB_ERR_ARG;
    if (!c->counted) {
        npb_set_error("npb_interpolate_fetch: call npb_interpolate_count first");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    if (!c->filled) {
        NPB_TRY(npb_ensure_out(c, (size_t)c->nnz));
        NpbTimer tm(c, "k3_fill");
        NPB_TRY(npb_k3_fill(c, c->lo, c->hi));
        tm.stop();
        c->filled = true;
        c->csr_gen++;
    }
    const bool host_gather = c->world > 1 && c->gather_mode == NPB_GATHER_HOST;
    if (c->world > 1 && !host_gather && !c->gathered) {
        NpbTimer tm(c, "k4_gather");
        NPB_TRY(npb_k4_gather_blocks(c));
        tm.stop();
    }
    if (host_gather) {
        // this rank's rows to their global positions of the (shared) host arrays
        NpbTimer tm(c, "d2h_csr");
        int32_t o[2] = {0, 0};
        NPB_TRY(npb_read_int(c, c->indptr + c->lo, &o[0]));
        NPB_TRY(npb_read_int(c, c->indptr + c->hi, &o[1]));
        const i64 rows = c->hi - c->lo, nk = (i64)o[1] - o[0];
        const i64 extra = (c->rank == c->world - 1) ? 1 : 0;   // the closing indptr entry
        if (indptr && rows + extra > 0) NPB_TRY(npb_d2h(c, indptr + c->lo, c->indptr + c->lo, sizeof(int32_t) * (size_t)(rows + extra)));
        if (indices && nk > 0) NPB_TRY(npb_d2h(c, indices + o[0], c->indices + o[0], sizeof(int32_t) * (size_t)nk));
        if (data && nk > 0) NPB_TRY(npb_d2h(c, data + o[0], c->data + o[0], sizeof(double) * (size_t)nk));
        if (neumann && rows > 0) NPB_TRY(npb_d2h(c, neumann + c->lo, c->neumann + c->lo, sizeof(double) * (size_t)rows));
        tm.stop();
        NPB_CUDA(cudaStreamSynchronize(s));
        return NPB_OK;
    }
    {
        NpbTimer tm(c, "d2h_csr");
        const bool block_only = c->world > 1 && c->gather_mode == NPB_GATHER_ROOT && c->rank != 0;
        if (indptr && block_only) {
            // this rank's rows only: indptr clamped to the block and rebased, rows of other ranks empty
            NPB_TRY(npb_ensure(&c->scratch, &c->scratch_cap, sizeof(int32_t) * (size_t)(c->n_points + 1)));
            k_block_indptr<<<npb_blocks(c->n_points + 1, 256), 256, 0, s>>>(c->indptr, c->n_points + 1, (int32_t)c->blk_off,
                                                                           (int32_t)(c->blk_off + c->nnz_ret),
                                                                           (int32_t *)c->scratch);
            NPB_LAUNCH(c);
            NPB_TRY(npb_d2h(c, indptr, c->scratch, sizeof(int32_t) * (c->n_points + 1)));
        } else if (indptr)
            NPB_TRY(npb_d2h(c, indptr, c->indptr, sizeof(int32_t) * (c->n_points + 1)));
        if (indices && c->nnz_ret > 0) NPB_TRY(npb_d2h(c, indices, c->indices + c->blk_off, sizeof(int32_t) * c->nnz_ret));
        if (data && c->nnz_ret > 0) NPB_TRY(npb_d2h(c, data, c->data + c->blk_off, sizeof(double) * c->nnz_ret));
        if (neumann) NPB_TRY(npb_d2h(c, neumann, c->neumann, sizeof(double) * c->n_points));
        tm.stop();
    }
    NPB_CUDA(cudaStreamSynchronize(s));
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// K5 — nodal values W @ values (and W.T @ values) from the CSR left on the device by the last count / run
// ------------------------------------------------------------------------------------------------
// the two-pass count (exact-zero fallback, or world > 1) leaves the rows unwritten: write them before a product
static int fill_rows_for_apply(npb_ctx *c)
{
    if (c->filled) return NPB_OK;
    NPB_TRY(npb_ensure_out(c, (size_t)c->nnz));
    NpbTimer tm(c, "k3_fill");
    NPB_TRY(npb_k3_fill(c, c->lo, c->hi));
    tm.stop_lazy();
    c->filled = true;
    c->csr_gen++;
    return NPB_OK;
}

extern "C" int npb_apply(npb_ctx *c, int method, const double *values, int64_t n_cols, double *out)
{
    if (!c || n_cols < 0 || (n_cols > 0 && (!values || !out))) return NPB_ERR_ARG;
    if (!c->counted || c->method != method) {
        npb_set_error("npb_apply: no weights of method %d are resident (run npb_interpolate_count or npb_interpolate_run "
                      "for the current inputs first)", method);
        return NPB_ERR_STATE;
    }
    if (n_cols == 0) return NPB_OK;
    NPB_CUDA(cudaSetDevice(c->device));
    NPB_TRY(fill_rows_for_apply(c));
    // this rank's nodes read the values of the elements in their esup rows only: upload that slice
    i64 first = 0, last = c->n_elems - 1;
    if (c->world > 1) {
        if (!c->apply_range_ok) {
            int64_t f = 0, l = -1;
            NPB_TRY(npb_partition_elem_range(c, &f, &l));
            c->apply_first = f;
            c->apply_last = l;
            c->apply_range_ok = true;
        }
        first = c->apply_first;
        last = c->apply_last;
    }
    const i64 n_up = last >= first ? last - first + 1 : 0;
    NPB_TRY(npb_ensure((void **)&c->apply_x, &c->apply_x_cap, sizeof(double) * (size_t)(c->n_elems * n_cols)));
    NPB_TRY(npb_ensure((void **)&c->apply_y, &c->apply_y_cap, sizeof(double) * (size_t)(c->n_points * n_cols)));
    {
        NpbTimer tm(c, "h2d_apply");
        NPB_TRY(npb_h2d(c, c->apply_x + first * n_cols, values + first * n_cols, sizeof(double) * (size_t)(n_up * n_cols)));
        tm.stop_lazy();
    }
    {
        NpbTimer tm(c, "apply");
        NPB_TRY(npb_k5_apply(c, c->lo, c->hi, c->apply_x, n_cols, c->apply_y));
        tm.stop_lazy();
    }
    if (c->world > 1) {
        NpbTimer tm(c, "apply_gather");
        NPB_TRY(npb_k4_gather_rows(c, c->apply_y, n_cols));
        tm.stop_lazy();
    }
    {
        NpbTimer tm(c, "d2h_apply");
        NPB_TRY(npb_d2h(c, out, c->apply_y, sizeof(double) * (size_t)(c->n_points * n_cols)));
        tm.stop();
    }
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    return NPB_OK;
}

// W.T @ values: one GPU only.  A rank holds only its own rows, so the ascending-node sum of an element would span ranks.
extern "C" int npb_apply_transpose(npb_ctx *c, int method, const double *values, int64_t n_cols, double *out)
{
    if (!c || n_cols < 0 || (n_cols > 0 && (!values || !out))) return NPB_ERR_ARG;
    if (c->world > 1) {
        npb_set_error("npb_apply_transpose: the transposed product is single-GPU (world is %d): every rank holds only its "
                      "own rows of W, and the ascending-node sum of an element spans ranks", c->world);
        return NPB_ERR_STATE;
    }
    if (!c->counted || c->method != method) {
        npb_set_error("npb_apply_transpose: no weights of method %d are resident (run npb_interpolate_count or "
                      "npb_interpolate_run for the current inputs first)", method);
        return NPB_ERR_STATE;
    }
    if (n_cols == 0) return NPB_OK;
    NPB_CUDA(cudaSetDevice(c->device));
    NPB_TRY(fill_rows_for_apply(c));
    if (c->tmap_gen != c->csr_gen) {
        NPB_TRY(npb_ensure((void **)&c->tmap, &c->tmap_cap, sizeof(int2) * (size_t)(c->n_elems * c->spe)));
        NpbTimer tm(c, "adjoint_map");
        NPB_TRY(npb_k5_tmap(c, c->tmap));
        tm.stop();   // synchronous: a reused map below records 0 with no pending timer left to overwrite it
        c->tmap_gen = c->csr_gen;
    } else {
        c->timings["adjoint_map"] = 0.f;
    }
    NPB_TRY(npb_ensure((void **)&c->apply_y, &c->apply_y_cap, sizeof(double) * (size_t)(c->n_points * n_cols)));
    NPB_TRY(npb_ensure((void **)&c->apply_x, &c->apply_x_cap, sizeof(double) * (size_t)(c->n_elems * n_cols)));
    {
        NpbTimer tm(c, "h2d_adjoint");
        NPB_TRY(npb_h2d(c, c->apply_y, values, sizeof(double) * (size_t)(c->n_points * n_cols)));
        tm.stop_lazy();
    }
    {
        NpbTimer tm(c, "adjoint");
        NPB_TRY(npb_k5_apply_t(c, c->tmap, c->apply_y, n_cols, c->apply_x));
        tm.stop_lazy();
    }
    {
        NpbTimer tm(c, "d2h_adjoint");
        NPB_TRY(npb_d2h(c, out, c->apply_x, sizeof(double) * (size_t)(c->n_elems * n_cols)));
        tm.stop();
    }
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// plug-in contract: dense weights[n_points, MX_ELEMENTS_PER_POINT] + neumann_ws, as XInterpolation.prepare
// leaves them (idw.pxd:19-24, ls.pxd:20-25, gls.pxd:22-27; caller-allocated, interpolator.pyx:645-651)
// ------------------------------------------------------------------------------------------------
__global__ void k_dense_rows(const int32_t *__restrict__ esup_ptr, const double *__restrict__ wbuf, i64 wbase,
                             const double *__restrict__ neumann, i64 n_points, int mx, double *__restrict__ out)
{
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_points * mx) return;
    i64 p = idx / mx;
    int k = (int)(idx - p * mx);
    int b = esup_ptr[p], e = esup_ptr[p + 1];
    // wbuf holds the CSR value w + neumann_ws (interpolator.pyx:618); the plug-in's own output is w.  IDW / LS
    // never write neumann_ws (it is +0.0), so this is exact for them; for GLS it is w to within one rounding
    out[idx] = (k < e - b) ? wbuf[(i64)b + k - wbase] - neumann[p] : 0.0;
}

extern "C" int npb_interpolate_dense(npb_ctx *c, int method, double *weights, double *neumann_ws)
{
    if (!c || !weights || !neumann_ws) return NPB_ERR_ARG;
    if (!c->mesh_loaded) {
        npb_set_error("Grid not initialized. Please load a mesh first.");
        return NPB_ERR_STATE;
    }
    if (method != NPB_METHOD_IDW && method != NPB_METHOD_LS && method != NPB_METHOD_GLS) {
        npb_set_error("unknown method id %d", method);
        return NPB_ERR_ARG;
    }
    if (c->world != 1) {
        npb_set_error("npb_interpolate_dense: the dense plug-in view is single-GPU only");
        return NPB_ERR_STATE;
    }
    if (!c->have_flags) {
        npb_set_error("neumann flags have not been set");
        return NPB_ERR_STATE;
    }
    if (method == NPB_METHOD_GLS && (!c->have_perm || !c->have_dm)) {
        npb_set_error("GLS needs the 'permeability' and 'diff_mag' cell fields");
        return NPB_ERR_STATE;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    c->counted = false;
    c->filled = false;
    c->csr_gen++;
    NPB_TRY(npb_ensure((void **)&c->wbuf, &c->wbuf_cap, sizeof(double) * (size_t)(c->wlen > 0 ? c->wlen : 1)));
    if (method == NPB_METHOD_GLS)
        NPB_TRY(npb_k2_gls(c, c->lo, c->hi));
    else {
        int used = 0;
        NPB_TRY(npb_k2_idw_ls_tiles(c, method, c->lo, c->hi, &used));
        if (!used) NPB_TRY(npb_k2_idw_ls(c, method, c->lo, c->hi));
    }
    const i64 total = c->n_points * (i64)c->mx_epp;
    NpbTmp dense;
    NPB_CUDA(dense.alloc(sizeof(double) * (size_t)total));
    if (total > 0) {
        k_dense_rows<<<npb_blocks(total, 256), 256, 0, s>>>(c->esup_ptr, c->wbuf, c->wbase, c->neumann, c->n_points, c->mx_epp,
                                                            dense.as<double>());
        NPB_LAUNCH(c);
        NPB_TRY(npb_d2h(c, weights, dense.p, sizeof(double) * (size_t)total));
    }
    NPB_TRY(npb_d2h(c, neumann_ws, c->neumann, sizeof(double) * (size_t)c->n_points));
    NPB_CUDA(cudaStreamSynchronize(s));
    return NPB_OK;
}

// ------------------------------------------------------------------------------------------------
// timings, launch count, measurement helpers
// ------------------------------------------------------------------------------------------------
extern "C" int npb_timing(npb_ctx *c, const char *name, double *ms)
{
    if (!c || !name || !ms) return NPB_ERR_ARG;
    npb_resolve_timers(c);
    auto it = c->timings.find(name);
    if (it == c->timings.end()) {
        npb_set_error("npb_timing: no timing named '%s'", name);
        return NPB_ERR_ARG;
    }
    *ms = it->second;
    return NPB_OK;
}

extern "C" int npb_timer_start(npb_ctx *c)
{
    if (!c) return NPB_ERR_ARG;
    NPB_CUDA(cudaSetDevice(c->device));
    if (!c->ev_a) {
        NPB_CUDA(cudaEventCreate(&c->ev_a));
        NPB_CUDA(cudaEventCreate(&c->ev_b));
    }
    NPB_CUDA(cudaEventRecord(c->ev_a, c->stream));
    return NPB_OK;
}

extern "C" int npb_timer_stop(npb_ctx *c, double *ms)
{
    if (!c || !ms || !c->ev_a) return NPB_ERR_ARG;
    NPB_CUDA(cudaEventRecord(c->ev_b, c->stream));
    NPB_CUDA(cudaEventSynchronize(c->ev_b));
    float f = 0.f;
    NPB_CUDA(cudaEventElapsedTime(&f, c->ev_a, c->ev_b));
    *ms = f;
    return NPB_OK;
}

extern "C" int npb_host_alloc(int64_t bytes, void **ptr)
{
    if (!ptr || bytes < 0) return NPB_ERR_ARG;
    *ptr = nullptr;
    NPB_CUDA(cudaHostAlloc(ptr, (size_t)(bytes > 0 ? bytes : 8), cudaHostAllocDefault));
    return NPB_OK;
}

extern "C" int npb_host_free(void *ptr)
{
    if (ptr) NPB_CUDA(cudaFreeHost(ptr));
    return NPB_OK;
}

extern "C" int npb_host_register(void *ptr, int64_t bytes)
{
    if (!ptr || bytes <= 0) return NPB_ERR_ARG;
    NPB_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault));
    return NPB_OK;
}

extern "C" int npb_host_unregister(void *ptr)
{
    if (ptr) NPB_CUDA(cudaHostUnregister(ptr));
    return NPB_OK;
}

extern "C" int npb_launch_count(npb_ctx *c, int64_t *count)
{
    if (!c || !count) return NPB_ERR_ARG;
    *count = c->launches;
    return NPB_OK;
}

// register-resident chains of dependent DFMAs, 8 independent chains per thread
__global__ void __launch_bounds__(256) k_dfma_peak(double *out, int iters)
{
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0, a6 = a0 + 6.0,
           a7 = a0 + 7.0;
    const double m = 0.999999, b = 1e-7;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
        a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int npb_measure_fp64_peak(npb_ctx *c, double *tflops)
{
    if (!c || !tflops) return NPB_ERR_ARG;
    NPB_CUDA(cudaSetDevice(c->device));
    int blocks = c->sm_count * 8, threads = 256, iters = 1 << 15;
    double *out = nullptr;
    NPB_CUDA(cudaMalloc(&out, sizeof(double) * (size_t)blocks * threads));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(a, c->stream);
        k_dfma_peak<<<blocks, threads, 0, c->stream>>>(out, iters);
        cudaEventRecord(b, c->stream);
        NPB_CUDA(cudaEventSynchronize(b));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        double tf = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    NPB_CUDA(cudaFree(out));
    *tflops = best;
    return NPB_OK;
}

__global__ void k_copy16(const int4 *__restrict__ in, int4 *__restrict__ out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = in[i];
}

extern "C" int npb_measure_copy_bw(npb_ctx *c, int64_t bytes, double *gbs)
{
    if (!c || !gbs || bytes < 1024) return NPB_ERR_ARG;
    NPB_CUDA(cudaSetDevice(c->device));
    size_t n = (size_t)bytes / 16;
    int4 *a = nullptr, *b = nullptr;
    NPB_CUDA(cudaMalloc(&a, n * 16));
    NPB_CUDA(cudaMalloc(&b, n * 16));
    NPB_CUDA(cudaMemsetAsync(a, 1, n * 16, c->stream));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        cudaEventRecord(e0, c->stream);
        k_copy16<<<c->sm_count * 16, 512, 0, c->stream>>>(a, b, n);
        cudaEventRecord(e1, c->stream);
        NPB_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double g = 2.0 * n * 16 / (ms * 1e-3) / 1e9;
        if (rep > 0 && g > best) best = g;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    NPB_CUDA(cudaFree(a));
    NPB_CUDA(cudaFree(b));
    *gbs = best;
    return NPB_OK;
}

__global__ void k_fill8(double *p, size_t n, double v)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

extern "C" int npb_flush_l2(npb_ctx *c, int64_t bytes)
{
    if (!c || bytes < 8) return NPB_ERR_ARG;
    NPB_CUDA(cudaSetDevice(c->device));
    NPB_TRY(npb_ensure(&c->scratch, &c->scratch_cap, (size_t)bytes));
    k_fill8<<<c->sm_count * 8, 512, 0, c->stream>>>((double *)c->scratch, (size_t)bytes / 8, 0.0);
    return NPB_OK;
}
