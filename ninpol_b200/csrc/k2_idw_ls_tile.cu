// k2_idw_ls_tile.cu — IDW / LS weights fused with the CSR emit (kernel groups K2 + K3), the
// HBM-roofline path for the two bit-exact methods.
//
// Same arithmetic as k2_idw_ls.cu (reference ninpol/_methods/idw.pyx:35-84, ls.pyx:33-135; evaluation
// order of SURVEY.md App. C, no FMA: -fmad=false plus _rn intrinsics), different mapping:
//   * a CTA owns a tile of NB consecutive nodes, i.e. ONE CONTIGUOUS slice of esup;
//   * phase A, one thread per esup ENTRY: coalesced read of esup, gather of the 24-byte centroid,
//     per-entry arithmetic (the IEEE sqrt / divide sequences that dominate the instruction count),
//     results staged in shared memory;
//   * phase B, one thread per NODE: the order-sensitive sequential sums of the reference (total
//     distance / the nine LS moments, Cramer's rule) over the staged values — this is what keeps the
//     result bit-identical to the serial CPU loops;
//   * phase C, one thread per entry again: final divide and coalesced stores of (index, value)
//     straight into the CSR arrays.
// CSR positions are known before the weights are: a Dirichlet node contributes no entries, every other
// node all of its esup row, unless a weight is exactly +-0.0 (scipy's eliminate_zeros would drop it,
// SURVEY.md Q5).  The kernels count such zeros; if there is any, the caller discards this result and
// takes the general two-pass path (k2_idw_ls.cu + k3_emit.cu).
#include <stdlib.h>
#include "common.cuh"

#define TILE_NB 64
#define TILE_T 256
#ifndef IDW_ECAP
#define IDW_ECAP 1536
#endif
#ifndef LS_ECAP
#define LS_ECAP 1408
#endif
#ifndef LS_ECAP_WIDE
#define LS_ECAP_WIDE 1024
#endif
#ifndef LS_NB_WIDE
#define LS_NB_WIDE 128
#endif
#define IDW_EPS ((double)1.0000000036274937e-15f) /* float32(1e-15), idw.pyx:53 */

struct TileArgs {
    const int32_t *esup_ptr, *esup;
    const uint8_t *bpoint, *nflag;
    const double *coords, *cent;
    const int32_t *indptr;
    int32_t *indices;
    double *data;
    int *zero_counter;
    double *neumann;
    double *wbuf;        // two-pass mode: values go to wbuf (esup-indexed from wbase) and rowcnt[p] = surviving entries
    int32_t *rowcnt;
    i64 wbase;
    i64 p_lo, p_hi;      // node range of this launch
    int nb, dim;
    int direct;          // 1: write the CSR at indptr[] positions and count exact zeros; 0: two-pass mode
};

// rowcnt[p] = entries node p will emit if no weight is an exact zero; neumann[p] = 0
__global__ void k_row_plan(const int32_t *__restrict__ esup_ptr, const uint8_t *__restrict__ bpoint,
                           const uint8_t *__restrict__ nflag, i64 n_points, int32_t *__restrict__ rowcnt,
                           double *__restrict__ neumann)
{
    i64 p = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p > n_points) return;
    if (p == n_points) {
        rowcnt[p] = 0;
        return;
    }
    bool proc = !(bpoint[p] && !nflag[p]);
    rowcnt[p] = proc ? esup_ptr[p + 1] - esup_ptr[p] : 0;
    neumann[p] = 0.0;
}


// MINB = resident CTAs asked for
template <int NBCAP, int MINB>
__global__ void __launch_bounds__(TILE_T, MINB) k_idw_tile(TileArgs a)
{
    __shared__ double s_r[IDW_ECAP + NBCAP];
    __shared__ int s_e[IDW_ECAP];
    __shared__ unsigned char s_rid[IDW_ECAP];
    __shared__ double s_x[NBCAP * 3], s_tot[NBCAP];
    __shared__ int s_ptr[NBCAP + 1], s_out[NBCAP], s_fz[NBCAP], s_cnt[NBCAP];
    __shared__ unsigned char s_proc[NBCAP];
    const int tid = threadIdx.x;
    const i64 ntiles = (a.p_hi - a.p_lo + a.nb - 1) / a.nb;
    for (i64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const i64 p0 = a.p_lo + tile * a.nb;
        const int nb = (int)min((i64)a.nb, a.p_hi - p0);
        if (tid <= nb) s_ptr[tid] = a.esup_ptr[p0 + tid];
        if (tid < nb) {
            i64 p = p0 + tid;
            s_proc[tid] = !(a.bpoint[p] && !a.nflag[p]);
            s_out[tid] = a.direct ? a.indptr[p] : 0;
            s_cnt[tid] = 0;
            s_x[3 * tid] = a.coords[p * 3];
            s_x[3 * tid + 1] = a.coords[p * 3 + 1];
            s_x[3 * tid + 2] = a.coords[p * 3 + 2];
        }
        __syncthreads();
        const int eb = s_ptr[0], ne = s_ptr[nb] - eb;
        if (tid < nb)
            for (int k = s_ptr[tid] - eb; k < s_ptr[tid + 1] - eb; k++) s_rid[k] = (unsigned char)tid;
        __syncthreads();
        // phase A: one thread per esup entry
        for (int i = tid; i < ne; i += TILE_T) {
            int node = s_rid[i];
            if (!s_proc[node]) continue;
            int e = a.esup[eb + i];
            s_e[i] = e;
            const double *cc = a.cent + (i64)e * NPB_CSTRIDE;
            double d0 = __dsub_rn(s_x[3 * node], cc[0]);
            double dist = __dadd_rn(0.0, __dmul_rn(d0, d0));
            if (a.dim > 1) {
                double d1 = __dsub_rn(s_x[3 * node + 1], cc[1]);
                dist = __dadd_rn(dist, __dmul_rn(d1, d1));
            }
            if (a.dim > 2) {
                double d2 = __dsub_rn(s_x[3 * node + 2], cc[2]);
                dist = __dadd_rn(dist, __dmul_rn(d2, d2));
            }
            // coincident centroid (idw.pyx:69): marked with -1 (a reciprocal distance is never negative)
            s_r[i + node] = (dist <= IDW_EPS) ? -1.0 : __ddiv_rn(1.0, __dsqrt_rn(dist));
        }
        __syncthreads();
        // phase B: one thread per node, sequential sum in esup order (idw.pyx:79)
        if (tid < nb && s_proc[tid]) {
            int b = s_ptr[tid] - eb + tid, E = s_ptr[tid + 1] - s_ptr[tid];
            double total = 0.0;
            int fz = -1;
            for (int k = 0; k < E; k++) {
                double v = s_r[b + k];
                if (v == -1.0) {
                    fz = k;
                    break;
                }
                total = __dadd_rn(total, v);
            }
            s_tot[tid] = total;
            s_fz[tid] = fz;
        }
        __syncthreads();
        // phase C: normalise and emit
        for (int i = tid; i < ne; i += TILE_T) {
            int node = s_rid[i];
            if (!s_proc[node]) {
                if (!a.direct) a.wbuf[(i64)eb + i - a.wbase] = 0.0;
                continue;
            }
            int k = i - (s_ptr[node] - eb);
            int fz = s_fz[node];
            double w;
            if (fz >= 0)
                w = (k == fz) ? 1.0 : 0.0;
            else
                w = __dadd_rn(__ddiv_rn(s_r[i + node], s_tot[node]), 0.0);
            if (a.direct) {
                i64 pos = (i64)s_out[node] + k;
                a.data[pos] = w;
                a.indices[pos] = s_e[i];
                if (w == 0.0) atomicAdd(a.zero_counter, 1);
            } else {
                a.wbuf[(i64)eb + i - a.wbase] = w;
                if (w != 0.0) atomicAdd(&s_cnt[node], 1);
            }
        }
        __syncthreads();
        if (!a.direct && tid < nb) {
            a.rowcnt[p0 + tid] = s_cnt[tid];
            a.neumann[p0 + tid] = 0.0;
        }
    }
}

#define M2(a, b) __dmul_rn(a, b)
#define S2(a, b) __dsub_rn(a, b)
#define A2(a, b) __dadd_rn(a, b)

// NBCAP = node capacity of a tile: 64 for stars of >= 22 elements (tets); 128 (with 1024 entries) for small
// stars such as the 8 hexes around a node, where 64 nodes would use a third of the entry capacity and leave
// 3/4 of the threads idle in phase B (hex 200^3: 1.53 -> 1.08 ms)
template <int ECAP, int NBCAP, int MINB>
__global__ void __launch_bounds__(TILE_T, MINB) k_ls_tile(TileArgs a)
{
    __shared__ double s_vx[ECAP + NBCAP], s_vy[ECAP + NBCAP], s_vz[ECAP + NBCAP];
    __shared__ int s_e[ECAP];
    __shared__ unsigned char s_rid[ECAP];
    __shared__ double s_x[NBCAP * 3], s_lam[NBCAP * 4];
    __shared__ int s_ptr[NBCAP + 1], s_out[NBCAP], s_cnt[NBCAP];
    __shared__ unsigned char s_proc[NBCAP], s_mode[NBCAP];
    const int tid = threadIdx.x;
    const i64 ntiles = (a.p_hi - a.p_lo + a.nb - 1) / a.nb;
    for (i64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const i64 p0 = a.p_lo + tile * a.nb;
        const int nb = (int)min((i64)a.nb, a.p_hi - p0);
        if (tid <= nb) s_ptr[tid] = a.esup_ptr[p0 + tid];
        if (tid < nb) {
            i64 p = p0 + tid;
            s_proc[tid] = !(a.bpoint[p] && !a.nflag[p]);
            s_out[tid] = a.direct ? a.indptr[p] : 0;
            s_cnt[tid] = 0;
            s_x[3 * tid] = a.coords[p * 3];
            s_x[3 * tid + 1] = a.coords[p * 3 + 1];
            s_x[3 * tid + 2] = a.coords[p * 3 + 2];
        }
        __syncthreads();
        const int eb = s_ptr[0], ne = s_ptr[nb] - eb;
        if (tid < nb)
            for (int k = s_ptr[tid] - eb; k < s_ptr[tid + 1] - eb; k++) s_rid[k] = (unsigned char)tid;
        __syncthreads();
        // phase A: v = centroid - x_v per entry (ls.pyx:65-67).  Memory-level parallelism first: the ids of all of
        // this thread's entries are fetched with independent loads, then the centroids in batches of MLP_B entries,
        // so a tile costs ~3 dependent global round trips instead of 2 per entry
        constexpr int KMAX = (ECAP + TILE_T - 1) / TILE_T;
        constexpr int MLP_B = 2;
        int ee[KMAX];
#pragma unroll
        for (int u = 0; u < KMAX; u++) {
            const int i = tid + u * TILE_T;
            ee[u] = (i < ne) ? a.esup[eb + i] : -1;
        }
#pragma unroll
        for (int u0 = 0; u0 < KMAX; u0 += MLP_B) {
            double c[MLP_B][3];
#pragma unroll
            for (int v = 0; v < MLP_B; v++) {
                const int u = u0 + v;
                if (u < KMAX && ee[u >= KMAX ? 0 : u] >= 0) {
                    const double *cc = a.cent + (i64)ee[u >= KMAX ? 0 : u] * NPB_CSTRIDE;
                    c[v][0] = cc[0]; c[v][1] = cc[1]; c[v][2] = cc[2];
                }
            }
#pragma unroll
            for (int v = 0; v < MLP_B; v++) {
                const int u = u0 + v;
                if (u >= KMAX || ee[u >= KMAX ? 0 : u] < 0) continue;
                const int i = tid + u * TILE_T;
                const int node = s_rid[i];
                s_e[i] = ee[u >= KMAX ? 0 : u];
                if (!s_proc[node]) continue;
                s_vx[i + node] = S2(c[v][0], s_x[3 * node]);
                s_vy[i + node] = S2(c[v][1], s_x[3 * node + 1]);
                s_vz[i + node] = S2(c[v][2], s_x[3 * node + 2]);
            }
        }
        __syncthreads();
        // phase B: per node, the nine moments summed in esup order, then Cramer's rule (ls.pyx:69-126)
        if (tid < nb && s_proc[tid]) {
            int b = s_ptr[tid] - eb + tid, E = s_ptr[tid + 1] - s_ptr[tid];
            double Ix = 0.0, Iy = 0.0, Iz = 0.0, Ixx = 0.0, Ixy = 0.0, Ixz = 0.0, Iyy = 0.0, Iyz = 0.0, Izz = 0.0;
            for (int k = 0; k < E; k++) {
                double vx = s_vx[b + k], vy = s_vy[b + k], vz = s_vz[b + k];
                Ix = A2(Ix, vx); Iy = A2(Iy, vy); Iz = A2(Iz, vz);
                Ixx = A2(Ixx, M2(vx, vx)); Ixy = A2(Ixy, M2(vx, vy)); Ixz = A2(Ixz, M2(vx, vz));
                Iyy = A2(Iyy, M2(vy, vy)); Iyz = A2(Iyz, M2(vy, vz)); Izz = A2(Izz, M2(vz, vz));
            }
            bool flat = (Iz == 0.0 && Izz == 0.0 && Ixz == 0.0 && Iyz == 0.0);
            if (flat) Izz = 1.0;
            double D = A2(A2(M2(Ixx, S2(M2(Iyy, Izz), M2(Iyz, Iyz))), M2(Ixy, S2(M2(Iyz, Ixz), M2(Ixy, Izz)))),
                          M2(Ixz, S2(M2(Ixy, Iyz), M2(Iyy, Ixz))));
            if (D == 0.0) {  // inverse-distance fallback (ls.pyx:88-102): total of 1/|v| in esup order
                double total = 0.0;
                for (int k = 0; k < E; k++) {
                    double vx = s_vx[b + k], vy = s_vy[b + k], vz = s_vz[b + k];
                    total = A2(total, __ddiv_rn(1.0, __dsqrt_rn(A2(A2(M2(vx, vx), M2(vy, vy)), M2(vz, vz)))));
                }
                s_lam[4 * tid + 3] = total;
                s_mode[tid] = 1;
            } else {
                // ls.pyx:105-106 repeats the test, but Izz is already 1.0 whenever it held: the reference
                // never reaches Izz = -1.0; restated literally
                if (Iz == 0.0 && Izz == 0.0 && Ixz == 0.0 && Iyz == 0.0) Izz = -1.0;
                double lx = __ddiv_rn(A2(A2(M2(Ix, S2(M2(Iyz, Iyz), M2(Iyy, Izz))), M2(Iy, S2(M2(Ixy, Izz), M2(Iyz, Ixz)))),
                                         M2(Iz, S2(M2(Iyy, Ixz), M2(Ixy, Iyz)))), D);
                double ly = __ddiv_rn(A2(A2(M2(Ix, S2(M2(Ixy, Izz), M2(Iyz, Ixz))), M2(Iy, S2(M2(Ixz, Ixz), M2(Ixx, Izz)))),
                                         M2(Iz, S2(M2(Ixx, Iyz), M2(Ixy, Ixz)))), D);
                double lz = __ddiv_rn(A2(A2(M2(Ix, S2(M2(Iyy, Ixz), M2(Ixy, Iyz))), M2(Iy, S2(M2(Ixx, Iyz), M2(Ixy, Ixz)))),
                                         M2(Iz, S2(M2(Ixy, Ixy), M2(Ixx, Iyy)))), D);
                s_lam[4 * tid] = lx;
                s_lam[4 * tid + 1] = ly;
                s_lam[4 * tid + 2] = lz;
                s_lam[4 * tid + 3] = A2(A2(A2((double)E, M2(lx, Ix)), M2(ly, Iy)), M2(lz, Iz));   // denom, ls.pyx:126
                s_mode[tid] = 0;
            }
        }
        __syncthreads();
        // phase C: weights (ls.pyx:127-135 / :95-102) and emit
        for (int i = tid; i < ne; i += TILE_T) {
            int node = s_rid[i];
            if (!s_proc[node]) {
                if (!a.direct) a.wbuf[(i64)eb + i - a.wbase] = 0.0;
                continue;
            }
            int k = i - (s_ptr[node] - eb);
            double vx = s_vx[i + node], vy = s_vy[i + node], vz = s_vz[i + node];
            double den = s_lam[4 * node + 3];
            double w;
            if (s_mode[node] == 0)
                w = A2(A2(A2(1.0, M2(s_lam[4 * node], vx)), M2(s_lam[4 * node + 1], vy)), M2(s_lam[4 * node + 2], vz));
            else
                w = __ddiv_rn(1.0, __dsqrt_rn(A2(A2(M2(vx, vx), M2(vy, vy)), M2(vz, vz))));
            w = A2(__ddiv_rn(w, den), 0.0);
            if (a.direct) {
                i64 pos = (i64)s_out[node] + k;
                a.data[pos] = w;
                a.indices[pos] = s_e[i];
                if (w == 0.0) atomicAdd(a.zero_counter, 1);
            } else {
                a.wbuf[(i64)eb + i - a.wbase] = w;
                if (w != 0.0) atomicAdd(&s_cnt[node], 1);
            }
        }
        __syncthreads();
        if (!a.direct && tid < nb) {
            a.rowcnt[p0 + tid] = s_cnt[tid];
            a.neumann[p0 + tid] = 0.0;
        }
    }
}

// nodes per tile; > TILE_NB selects the small-star LS variant (128 nodes x 1024 entries)
static int tile_nb(npb_ctx *c, int method)
{
    if (c->mx_epp <= 0) return 0;
    const char *force = getenv("NPB_FORCE_SIMPLE_IDW_LS");   // tests: exercise the thread-per-node kernels
    if (force && force[0] == '1') return 0;
    if (method == NPB_METHOD_IDW) {   // measured: 192-node IDW tiles are 25 % slower than 64-node ones on hex meshes
        int nb = IDW_ECAP / c->mx_epp;
        return nb > TILE_NB ? TILE_NB : nb;
    }
    int nb = LS_ECAP / c->mx_epp;
    if (nb > TILE_NB) {
        int nw = LS_ECAP_WIDE / c->mx_epp;
        return nw > LS_NB_WIDE ? LS_NB_WIDE : nw;
    }
    return nb > TILE_NB ? TILE_NB : nb;
}

static void tile_params(npb_ctx *c, TileArgs &a, int method, i64 lo, i64 hi, int direct)
{
    a.esup_ptr = c->esup_ptr; a.esup = c->esup; a.bpoint = c->bpoint; a.nflag = c->nflag; a.coords = c->coords;
    a.cent = c->centroids; a.indptr = c->indptr; a.indices = c->indices; a.data = c->data;
    a.zero_counter = c->counters + 45; a.neumann = c->neumann; a.wbuf = c->wbuf; a.rowcnt = c->rowcnt; a.wbase = c->wbase;
    a.p_lo = lo; a.p_hi = hi; a.nb = tile_nb(c, method); a.dim = c->dim; a.direct = direct;
}

static int tile_launch(npb_ctx *c, const TileArgs &a, int method)
{
    i64 ntiles = (a.p_hi - a.p_lo + a.nb - 1) / a.nb;
    int grid = (int)(ntiles < (i64)c->sm_count * 8 ? ntiles : (i64)c->sm_count * 8);
    if (grid < 1) return NPB_OK;
    NpbTimer tm(c, "k2_main");
    // LS loads the centroids in batches (k_ls_tile phase A): 0.39 -> 0.52 of the HBM roofline on 50M tets, 0.42 -> 0.50
    // on hex 200^3 against per-entry loads, which stay the faster choice for IDW (B200, DESIGN.md K2/K3).  LS asks for 4
    // resident CTAs: 4 of 46.8 KB fit an SM; 64 registers, no spills (5 would need <= 51)
    if (method == NPB_METHOD_IDW)
        k_idw_tile<TILE_NB, 7><<<grid, TILE_T, 0, c->stream>>>(a);
    else if (a.nb > TILE_NB)
        k_ls_tile<LS_ECAP_WIDE, LS_NB_WIDE, 4><<<grid, TILE_T, 0, c->stream>>>(a);
    else
        k_ls_tile<LS_ECAP, TILE_NB, 4><<<grid, TILE_T, 0, c->stream>>>(a);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaGetLastError());
    tm.stop_lazy();     // no host synchronisation between the tile kernel and whatever follows it on the stream
    return NPB_OK;
}

// Two-pass mode over this rank's node range: values to wbuf, surviving-entry counts to rowcnt.
// *used = 0 when a star is too large for a tile (the thread-per-node kernels of k2_idw_ls.cu take over).
int npb_k2_idw_ls_tiles(npb_ctx *c, int method, i64 lo, i64 hi, int *used)
{
    *used = 0;
    if (tile_nb(c, method) < 1) return NPB_OK;
    *used = 1;
    if (hi <= lo) return NPB_OK;
    TileArgs a;
    tile_params(c, a, method, lo, hi, 0);
    return tile_launch(c, a, method);
}

// Direct mode over a node range with c->indptr already holding the (optimistic) global plan and c->indices /
// c->data sized for it (pipeline.cu): exact zeros are counted in counters[45], which the caller reads.
int npb_k2_idw_ls_direct(npb_ctx *c, int method, i64 lo, i64 hi, int *used)
{
    *used = 0;
    if (tile_nb(c, method) < 1) return NPB_OK;
    *used = 1;
    if (hi <= lo) return NPB_OK;
    TileArgs a;
    tile_params(c, a, method, lo, hi, 1);
    return tile_launch(c, a, method);
}

// Single-pass mode: *used = 1 when indptr / indices / data / neumann hold the final CSR, 0 when the
// caller has to run the two-pass path instead (multi-GPU, oversized stars, or an exact-zero weight).
int npb_k2_idw_ls_fused(npb_ctx *c, int method, int *used)
{
    *used = 0;
    if (c->world != 1 || c->n_points <= 0 || tile_nb(c, method) < 1) return NPB_OK;
    cudaStream_t s = c->stream;
    i64 np = c->n_points;
    int *zero_counter = c->counters + 45;
    NPB_CUDA(cudaMemsetAsync(zero_counter, 0, sizeof(int), s));
    k_row_plan<<<npb_blocks(np + 1, 256), 256, 0, s>>>(c->esup_ptr, c->bpoint, c->nflag, np, c->rowcnt, c->neumann);
    NPB_LAUNCH(c);
    NPB_TRY(npb_exclusive_scan_i32(c, c->rowcnt, c->indptr, np + 1));
    int32_t total = 0;
    NPB_CUDA(cudaMemcpyAsync(&total, c->indptr + np, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    NPB_CUDA(cudaStreamSynchronize(s));
    NPB_TRY(npb_ensure_out(c, (size_t)total));
    TileArgs a;
    tile_params(c, a, method, 0, np, 1);
    NPB_TRY(tile_launch(c, a, method));
    int zeros = 0;
    NPB_CUDA(cudaMemcpyAsync(&zeros, zero_counter, sizeof(int), cudaMemcpyDeviceToHost, s));
    NPB_CUDA(cudaStreamSynchronize(s));
    if (zeros != 0) return NPB_OK;   // an exact zero would be dropped by eliminate_zeros: two-pass path
    c->nnz = total;
    *used = 1;
    return NPB_OK;
}
