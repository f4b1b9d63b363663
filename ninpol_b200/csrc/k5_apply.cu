// k5_apply.cu — nodal values from the resident weights (kernel group K5): out = W @ values on the device.
//
// No reference counterpart in the interpolator itself; it is what every caller does next (the reference's own
// accuracy check multiplies the CSR by the cell field with scipy).  The arithmetic is scipy's csr_matvec /
// csr_matvecs, bit for bit: every output element starts at +0.0 and adds data[j] * x[indices[j], c] over the entries
// of its row in ascending order, each product and each sum rounded on its own (no FMA, no reordering; this unit is
// built with -fmad=false on top of the explicit _rn intrinsics).
//
// Mapping: one thread owns one output element (p, c) and sums sequentially.  A CTA takes a run of consecutive rows;
// their CSR entries form one contiguous span, which is streamed through a shared-memory tile with coalesced loads;
// every thread then adds the part of its row that lies in the tile.  A row longer than the tile is simply spread over
// several tiles, in order.  values are row-major, so the threads of one row's columns gather adjacent doubles.
//
// The transposed product out = W.T @ y (k5_tmap + k5_apply_t, bottom of the file) is scipy's csc_matvec(s) on the
// free CSC view W.T: output element (e, c) starts at +0.0 and adds data[j] * y[p, c] over the entries (p, e) of W in
// ascending p.  The CSR is row-major by node, so those entries are found once through the element's own nodes and kept
// as a per-element map.
#include "common.cuh"
#include <climits>

#define K5_THREADS 256
#define K5_TILE 2048   // entries per staging tile: 8 KB of indices + 16 KB of data

// rows [lo, hi) of this launch; column block blockIdx.y covers columns [cb * blockIdx.y, + cb) of k.
__global__ void __launch_bounds__(K5_THREADS)
k5_apply_rows(const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices, const double *__restrict__ data,
              const double *__restrict__ x, i64 lo, i64 hi, int k, int cb, int rows_per_cta, double *__restrict__ out)
{
    __shared__ int32_t s_idx[K5_TILE];
    __shared__ double s_val[K5_TILE];
    const i64 r0 = lo + (i64)blockIdx.x * rows_per_cta;
    const i64 r1 = min(hi, r0 + rows_per_cta);
    const int t = threadIdx.x;
    const int c = (int)blockIdx.y * cb + t % cb;
    const i64 p = r0 + t / cb;
    const bool mine = t < rows_per_cta * cb && p < r1 && c < k;
    int b = 0, e = 0;
    if (mine) {
        b = indptr[p];
        e = indptr[p + 1];
    }
    const int span_b = indptr[r0], span_e = indptr[r1];
    double acc = 0.0;
    for (int t0 = span_b; t0 < span_e; t0 += K5_TILE) {
        const int n = min(K5_TILE, span_e - t0);
        for (int i = t; i < n; i += K5_THREADS) {
            s_idx[i] = indices[t0 + i];
            s_val[i] = data[t0 + i];
        }
        __syncthreads();
        const int jb = max(b, t0) - t0, je = min(e, t0 + n) - t0;
        int j = jb;
        // four gathers in flight ahead of the (sequential) sums
        for (; j + 4 <= je; j += 4) {
            const double x0 = x[(i64)s_idx[j] * k + c], x1 = x[(i64)s_idx[j + 1] * k + c];
            const double x2 = x[(i64)s_idx[j + 2] * k + c], x3 = x[(i64)s_idx[j + 3] * k + c];
            acc = __dadd_rn(acc, __dmul_rn(s_val[j], x0));
            acc = __dadd_rn(acc, __dmul_rn(s_val[j + 1], x1));
            acc = __dadd_rn(acc, __dmul_rn(s_val[j + 2], x2));
            acc = __dadd_rn(acc, __dmul_rn(s_val[j + 3], x3));
        }
        for (; j < je; j++) acc = __dadd_rn(acc, __dmul_rn(s_val[j], x[(i64)s_idx[j] * k + c]));
        __syncthreads();
    }
    if (mine) out[p * k + c] = acc;
}

// out[p, :] for the rows [lo, hi); x and out are device arrays with k doubles per element / per node
int npb_k5_apply(npb_ctx *c, i64 lo, i64 hi, const double *x, int64_t k, double *out)
{
    if (hi <= lo || k < 1) return NPB_OK;
    const int cb = (int)(k < K5_THREADS ? k : K5_THREADS);
    const int rows_per_cta = K5_THREADS / cb;
    const i64 ctas = (hi - lo + rows_per_cta - 1) / rows_per_cta;
    const i64 col_blocks = (k + cb - 1) / cb;
    if (ctas > 0x7fffffff || col_blocks > 65535) {
        npb_set_error("npb_apply: %lld rows x %lld columns exceed the launch grid", (long long)(hi - lo), (long long)k);
        return NPB_ERR_RANGE;
    }
    dim3 grid((unsigned)ctas, (unsigned)col_blocks);
    k5_apply_rows<<<grid, K5_THREADS, 0, c->stream>>>(c->indptr, c->indices, c->data, x, lo, hi, (int)k, cb, rows_per_cta, out);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaGetLastError());
    return NPB_OK;
}

// ---- transposed product: out = W.T @ y ----
//
// (p, e) is an entry of W only if p is a node of e (the rows come from esup), so the entries of column e are found by
// searching e in the rows of e's own nodes.  The map holds, for each element, spe slots (p, j): its nodes p in ascending
// order that have an entry in row p, with j the CSR position of that entry, compacted and padded with (-1, -1).  A node
// whose row has no entry for e (Dirichlet node, all-boundary-face GLS node, eliminated exact zero) gets no slot.

// one thread per element: sort its <= SPE node ids in registers, binary-search e in each node's (sorted) row
template <int SPE>
__global__ void __launch_bounds__(256)
k5_tmap(const int32_t *__restrict__ inpoel, const uint8_t *__restrict__ etype, ElemTables tab, i64 n_elems,
        const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices, int2 *__restrict__ map)
{
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_elems) return;
    const int npe = tab.npoel[etype[e]];
    int q[SPE];
#pragma unroll
    for (int s = 0; s < SPE; s++) q[s] = s < npe ? inpoel[e * SPE + s] : INT_MAX;
    // odd-even transposition sort: SPE rounds with fixed indices, so q never leaves the registers
#pragma unroll
    for (int r = 0; r < SPE; r++) {
#pragma unroll
        for (int s = r & 1; s + 1 < SPE; s += 2) {
            const int a = min(q[s], q[s + 1]), b = max(q[s], q[s + 1]);
            q[s] = a;
            q[s + 1] = b;
        }
    }
    int rb[SPE], re[SPE];
#pragma unroll
    for (int s = 0; s < SPE; s++) {
        rb[s] = s < npe ? indptr[q[s]] : 0;
        re[s] = s < npe ? indptr[q[s] + 1] : 0;
    }
    const int ei = (int)e;
    int2 *row = map + e * SPE;
    int n = 0;
#pragma unroll
    for (int s = 0; s < SPE; s++) {
        if (s < npe && (s == 0 || q[s] != q[s - 1])) {   // a node listed twice is searched once
            int lo = rb[s], hi = re[s];
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (indices[mid] < ei) lo = mid + 1;
                else hi = mid;
            }
            if (lo < re[s] && indices[lo] == ei) row[n++] = make_int2(q[s], lo);
        }
    }
    for (int s = n; s < SPE; s++) row[s] = make_int2(-1, -1);
}

// one thread per output element (e, c), mapped as k5_apply_rows maps (p, c): the k threads of an element read the same
// slots and adjacent doubles of y.  The gathers of all slots are written ahead of the (sequential, ascending-p) sums.
template <int SPE>
__global__ void __launch_bounds__(K5_THREADS)
k5_apply_t(const int2 *__restrict__ map, const double *__restrict__ data, const double *__restrict__ y, i64 n_elems,
           int k, int cb, int elems_per_cta, double *__restrict__ out)
{
    const int t = threadIdx.x;
    const int c = (int)blockIdx.y * cb + t % cb;
    const i64 e = (i64)blockIdx.x * elems_per_cta + t / cb;
    if (t >= elems_per_cta * cb || e >= n_elems || c >= k) return;
    const int4 *m4 = reinterpret_cast<const int4 *>(map + e * SPE);   // 8 * SPE bytes per element: 16-byte aligned
    int p[SPE], j[SPE];
#pragma unroll
    for (int s = 0; s < SPE / 2; s++) {
        const int4 v = m4[s];
        p[2 * s] = v.x;
        j[2 * s] = v.y;
        p[2 * s + 1] = v.z;
        j[2 * s + 1] = v.w;
    }
    // unpredicated gathers (a padding slot reads data[0] and y[0, c], which always exist, and adds nothing): no load waits
    // on a predicate.  At 32 registers ptxas still interleaves the last few loads with the first sums.
    double w[SPE], v[SPE];
#pragma unroll
    for (int s = 0; s < SPE; s++) {
        w[s] = data[max(j[s], 0)];
        v[s] = y[(i64)max(p[s], 0) * k + c];
    }
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < SPE; s++)
        if (p[s] >= 0) acc = __dadd_rn(acc, __dmul_rn(w[s], v[s]));
    out[e * k + c] = acc;
}

// the map of the CSR on the device: [n_elems, spe] int2
int npb_k5_tmap(npb_ctx *c, int2 *map)
{
    if (c->n_elems <= 0) return NPB_OK;
    const unsigned blocks = npb_blocks(c->n_elems, 256);
    if (c->spe == 4)
        k5_tmap<4><<<blocks, 256, 0, c->stream>>>(c->inpoel, c->etype, c->tab, c->n_elems, c->indptr, c->indices, map);
    else
        k5_tmap<8><<<blocks, 256, 0, c->stream>>>(c->inpoel, c->etype, c->tab, c->n_elems, c->indptr, c->indices, map);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaGetLastError());
    return NPB_OK;
}

// out[e, :] = (W.T @ y)[e, :] for all elements; y and out are device arrays with k doubles per node / per element
int npb_k5_apply_t(npb_ctx *c, const int2 *map, const double *y, int64_t k, double *out)
{
    if (c->n_elems <= 0 || k < 1) return NPB_OK;
    const int cb = (int)(k < K5_THREADS ? k : K5_THREADS);
    const int elems_per_cta = K5_THREADS / cb;
    const i64 ctas = (c->n_elems + elems_per_cta - 1) / elems_per_cta;
    const i64 col_blocks = (k + cb - 1) / cb;
    if (ctas > 0x7fffffff || col_blocks > 65535) {
        npb_set_error("npb_apply_transpose: %lld elements x %lld columns exceed the launch grid", (long long)c->n_elems,
                      (long long)k);
        return NPB_ERR_RANGE;
    }
    dim3 grid((unsigned)ctas, (unsigned)col_blocks);
    if (c->spe == 4)
        k5_apply_t<4><<<grid, K5_THREADS, 0, c->stream>>>(map, c->data, y, c->n_elems, (int)k, cb, elems_per_cta, out);
    else
        k5_apply_t<8><<<grid, K5_THREADS, 0, c->stream>>>(map, c->data, y, c->n_elems, (int)k, cb, elems_per_cta, out);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaGetLastError());
    return NPB_OK;
}
