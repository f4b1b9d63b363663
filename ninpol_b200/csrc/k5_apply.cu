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
#include "common.cuh"

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
