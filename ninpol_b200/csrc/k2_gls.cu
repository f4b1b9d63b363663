// k2_gls.cu — per-node GLS weight construction (kernel group K2, tolerance method).
//
// Replaces GLSInterpolation.GLS and its helpers (ninpol/_methods/gls.pyx:75-474): build_ks_sv_arrays
// (:234-249), build_ls_matrices (:252-356), set_neumann_rows (:374-416), solve_ls (:420-474, LAPACK
// DGELS on an (E+3F+B) x (3E+1) system with E right-hand sides, keeping only the last row of X).
//
// Algebra (SURVEY.md 3.3): with M = [A | c] (A = the 3E gradient columns, c = last column = 1 on the E
// element rows, 0 elsewhere) and r = c - A argmin_g |A g - c| the residual of ONE least-squares problem,
//     weights_i = X[3E, i] = r_i / |r|^2 = r_i / sum_j r_j          (i < E),
// so one QR of A with the single right-hand side c replaces the reference's E solves.  The all-zero
// rows the reference leaves for boundary faces (gls.pyx:340-344) do not change a least-squares
// solution and are not materialised.  Reproduced reference behaviour: Q3 (neumann[p] is the weight of
// the node's LAST element; the Neumann right-hand side is dead), Q4 (that value is added to every
// weight of the row), Q8 (all faces boundary -> zero row).
//
// Structure exploited: A is block sparse — 3 columns per element; an element row touches one block, the
// 3 rows of an interior face touch the two blocks of its elements, a Neumann row touches one block.
// The kernel runs a MULTIFRONTAL Householder QR per node, one warp per node, in three regimes:
//  1. leaf fronts, one per LANE: blocks none of whose neighbours is eliminated yet have a front of original
//     rows only (10 x (3 + 3 nn + 1), fixed sparsity); a greedy independent set of them is factored at
//     once, lane b doing block b entirely in registers and writing its 3 rows of R and its 7-row
//     contribution block straight to the slabs;
//  2. general fronts, one per WARP: the remaining blocks go in greedy minimum-degree order (adjacency as
//     per-lane bitmasks); the row groups containing the pivot are fetched into a dense front in shared
//     memory (cp.async), the 3 pivot columns are factored with lanes over rows (registers + shuffles), the
//     Householder vectors overwrite the panel columns of the front, and the three reflectors are applied
//     to the other columns in two passes (lanes over columns; narrow fronts put several rows on the lanes);
//  3. chained end game: a front's contribution block stays in place until the next pivot is known and the
//     next front is built around it when that pivot is its first column and brings no new column — every
//     step once the remaining blocks form a clique, i.e. the dense tall-skinny tail with most of the FLOPs.
// An interior node of the 50M-tet mesh (E=24, F=36) costs ~0.11 MFLOP this way instead of 1.19 MFLOP
// for a dense one-RHS QR (1.94 MFLOP in the reference) and ~35 k warp-instructions.  Back substitution
// through the stored R rows (leaf fronts again one per lane) gives g, then r_i = 1 - d_i . g_i.
//
// Memory: the front being factored and small tables live in shared memory (17.6 KB for an interior tet
// node); the row groups — original rows and contribution blocks — and the finished rows of R live in an
// append-only, L2-resident global slab per CTA.  One-warp CTAs, persistent, atomic work counter; 12 CTAs
// per SM for the interior-tet class (168 registers), 16 for smaller stars.  Fronts taller than the shared
// buffer are processed in row chunks (the 3 pivot rows of a chunk are carried into the next).  Nodes are
// bucketed into 7 size classes by star size; stars that do not fit (E > 64, a capacity overflow detected
// at run time) go to the dense global-memory kernel of k2_gls_dense.cu.  The kernel is latency / issue
// bound on this bookkeeping, not FP64 or HBM bound (SURVEY.md Q13, profiles/).
#include <stdlib.h>
#include <string.h>
#include "gls_common.cuh"

typedef unsigned long long u64;

#define MF_NCLASS 9          // 0 = skipped node, 1..7 = shared-memory classes, 8 = dense fallback
#define MF_SCAP 64           // max row groups merged into one front

struct MfClass {
    int fcap;   // front buffer in shared memory (doubles)
    int ecap;   // max elements around the node
    int fcap_f; // max faces around the node
    int acap;   // capacity (doubles) of the CTA's global row-group arena; the R slab has the same size
};
#define MF_CLASS_TABLE {{0, 0, 0, 0}, {640, 8, 14, 3072}, {640, 12, 22, 6144}, {768, 16, 30, 8192}, {1664, 24, 40, 12288}, \
                        {1664, 32, 56, 18432}, {2560, 48, 80, 32768}, {4096, 64, 112, 49152}, {0, 0, 0, 0}}
__constant__ MfClass c_mf[MF_NCLASS] = MF_CLASS_TABLE;
static const MfClass h_mf[MF_NCLASS] = MF_CLASS_TABLE;

// group table entries: original groups (<= ecap + fcap_f), leaf contribution blocks and re-entered survivors of the
// leaf phase (<= ecap together), one contribution block per general front (<= ecap)
__host__ __device__ __forceinline__ int mf_ngcap(const MfClass &k) { return ((3 * k.ecap + k.fcap_f + 7) / 8) * 8; }
__host__ __device__ __forceinline__ size_t mf_smem_bytes(const MfClass &k)
{
    size_t d = (size_t)k.fcap + 6 * (size_t)k.ecap;  // front, gvec, dvec
    size_t b = d * 8 + (size_t)mf_ngcap(k) * (8 + 4 + 2 + 1) + (size_t)k.ecap * (8 + 4 + 4);   // group table, R table
    b += (size_t)k.ecap * 4 + MF_SCAP * 4 + 64;                             // es, S list, colblk
    return (b + 15) & ~(size_t)15;
}

// per node: Dirichlet / Q8 nodes are finished here (zero row); the others get a size class.
// sig[k] / sig[MF_NCLASS + k]: smallest / largest star signature (E << 8 | F) seen in class k — equal when all stars of
// the class have the same size, which is when the team launch pays (npb_k2_gls).
__global__ void k_gls_classify(GlsArgs a, i64 lo, i64 hi, uint8_t *__restrict__ cls, int force_dense, int *__restrict__ sig)
{
    __shared__ int smin[MF_NCLASS], smax[MF_NCLASS];
    if (threadIdx.x < MF_NCLASS) {
        smin[threadIdx.x] = 0x7fffffff;
        smax[threadIdx.x] = 0;
    }
    __syncthreads();
    i64 p = lo + (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < hi) {
        int eb = a.esup_ptr[p], ee = a.esup_ptr[p + 1];
        int fb = a.fsup_ptr[p], fe = a.fsup_ptr[p + 1];
        int E = ee - eb, F = fe - fb;
        bool neu = a.nflag[p] != 0;
        int nb = 0;
        bool skip = (a.bpoint[p] && !neu);  // gls.pyx:165-166
        if (!skip) {
            for (int q = fb; q < fe; q++) nb += (a.esuf2[a.fsup[q]].y < 0) ? 1 : 0;
            if (nb >= F) skip = true;  // gls.pyx:266-267 + DGELS on a zero matrix -> zero weights (Q8)
        }
        if (skip) {
            double *w = a.wbuf + ((i64)eb - a.wbase);
            for (int k = 0; k < E; k++) w[k] = 0.0;
            a.rowcnt[p] = 0;
            a.neumann[p] = 0.0;
            cls[p] = 0;
        } else {
            int k = MF_NCLASS - 1;
            for (int q = 1; q < MF_NCLASS - 1 && !force_dense; q++)
                if (E <= c_mf[q].ecap && F <= c_mf[q].fcap_f) {
                    k = q;
                    break;
                }
            cls[p] = (uint8_t)k;
            const int sg = (min(E, 0xffff) << 8) | min(F, 255);
            atomicMin(&smin[k], sg);
            atomicMax(&smax[k], sg);
        }
    }
    __syncthreads();
    if (threadIdx.x < MF_NCLASS && smax[threadIdx.x] != 0) {
        atomicMin(&sig[threadIdx.x], smin[threadIdx.x]);
        atomicMax(&sig[MF_NCLASS + threadIdx.x], smax[threadIdx.x]);
    }
}

// hands the signature ranges to the host through the mapped block (read after the partition's synchronisation)
__global__ void k_gls_publish_sig(const int *__restrict__ sig, int *__restrict__ mapped)
{
    if (threadIdx.x < 2 * MF_NCLASS) mapped[threadIdx.x] = sig[threadIdx.x];
}

__device__ __forceinline__ u64 warp_or64(u64 v)
{
    unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v);
    unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
    return ((u64)hi << 32) | lo;
}
// 8-byte asynchronous global -> shared copy (LDGSTS): no register staging, no stall until the wait
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gmem_src)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ int nth_set_bit(u64 m, int n)  // index of the n-th (0-based) set bit
{
    for (int q = 0; q < n; q++) m &= m - 1;
    return __ffsll((long long)m) - 1;
}

struct MfWs {
    double *arena;   // global: row groups (original rows, contribution blocks), append-only
    double *front;   // shared: the dense front being factored
    double *gvec, *dvec;
    u64 *g_mask, *r_mask;
    int *g_off, *r_off, *r_meta;   // r_meta = piv | npiv << 8 | c << 16
    unsigned short *g_nr;
    unsigned char *g_ld;
    int *es;
    int *s_list;            // packed (gid | rowbase << 16)
    unsigned char *colblk;  // block id of every 3-column slot of the current front
};

__device__ __forceinline__ MfWs mf_carve(unsigned char *base, const MfClass &k, double *garena)
{
    MfWs w;
    int ng = mf_ngcap(k);
    w.arena = garena;
    w.front = (double *)base;
    w.gvec = w.front + k.fcap;
    w.dvec = w.gvec + 3 * k.ecap;
    w.g_mask = (u64 *)(w.dvec + 3 * k.ecap);
    w.r_mask = w.g_mask + ng;
    w.g_off = (int *)(w.r_mask + k.ecap);
    w.r_off = w.g_off + ng;
    w.r_meta = w.r_off + k.ecap;
    w.es = w.r_meta + k.ecap;
    w.s_list = w.es + k.ecap;
    w.g_nr = (unsigned short *)(w.s_list + MF_SCAP);
    w.g_ld = (unsigned char *)(w.g_nr + ng);
    w.colblk = w.g_ld + ng;                     // [64]
    return w;
}

// Closes the holes left by consumed groups in the (global) group arena: live table entries and their
// blocks slide down in table order, which equals arena order because entries are only ever appended.
// Keeps the slab region a CTA touches small enough that the resident CTAs' slabs stay in L2 (without it
// every contribution block ends up written to HBM once: 584 GB per pass over the 50M-tet mesh).
__device__ void mf_compact(MfWs &w, int &ng, int &top, int lane)
{
    int newng = 0, newtop = 0;
    for (int g0 = 0; g0 < ng; g0 += 32) {
        int g = g0 + lane;
        unsigned bal = __ballot_sync(0xffffffffu, g < ng && w.g_nr[g] > 0);
        while (bal) {
            int gi = g0 + __ffs(bal) - 1;
            bal &= bal - 1;
            u64 mk = w.g_mask[gi];
            int src = w.g_off[gi], nr = w.g_nr[gi], ld = w.g_ld[gi];
            int sz = nr * ld;
            if (src != newtop) {
                for (int i0 = 0; i0 < sz; i0 += 32) {
                    int i = i0 + lane;
                    double v = 0.0;
                    if (i < sz) v = w.arena[src + i];
                    __syncwarp();
                    if (i < sz) w.arena[newtop + i] = v;
                    __syncwarp();
                }
            }
            if (lane == 0) {
                w.g_mask[newng] = mk;
                w.g_off[newng] = newtop;
                w.g_nr[newng] = (unsigned short)nr;
                w.g_ld[newng] = (unsigned char)ld;
            }
            newtop += sz;
            newng++;
        }
    }
    __syncwarp();
    ng = newng;
    top = newtop;
}

// rows x cw block of the front (row stride sld) -> contiguous rows in the group arena; narrow blocks put
// several rows on the 32 lanes
__device__ __forceinline__ void mf_store_cb(const double *src, int sld, int rows, int cw, double *dst, int lane)
{
    const int L = cw > 16 ? 32 : cw > 8 ? 16 : cw > 4 ? 8 : cw > 2 ? 4 : cw > 1 ? 2 : 1;
    if (L < 32) {
        const int G = 32 / L, grp = lane / L, jl = lane & (L - 1);
        if (jl < cw) {
            src += grp * sld + jl;
            dst += grp * cw + jl;
            for (int r = grp; r < rows; r += G) {
                *dst = *src;
                src += G * sld;
                dst += G * cw;
            }
        }
    } else {
        for (int j = lane; j < cw; j += 32) {
            const double *sp = src + j;
            double *dp = dst + j;
            for (int r = 0; r < rows; r++) {
                *dp = *sp;
                sp += sld;
                dp += cw;
            }
        }
    }
}

#define MF_RPL 3   // front rows per lane in the panel factorisation: fronts of up to 96 rows
#ifndef MF_APPLY_UNROLL
#define MF_APPLY_UNROLL 4
#endif
#define MF_PRAGMA_(x) _Pragma(#x)
#define MF_PRAGMA(x) MF_PRAGMA_(x)
#define MF_UNROLL_APPLY MF_PRAGMA(unroll MF_APPLY_UNROLL)
#ifdef MF_HH_NOINLINE
#define MF_HH_INLINE __noinline__
#else
#define MF_HH_INLINE __forceinline__
#endif

// Householder scalars of one column: alpha = -sign(x0) |x|, beta = 2 / |v|^2 with v = x - alpha e1, and
// rinv = 1 / alpha (kept on the diagonal of R for the back substitution).  sqrt and 1/alpha come from one
// rsqrt plus a Newton step instead of the IEEE sqrt and divide sequences.
// MUFU seeds (upper-word approximations, ~20 bits) for 1/sqrt(x) and 1/x; refined below with Newton steps.
__device__ __forceinline__ double rsqrt_seed(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
__device__ __forceinline__ double rcp_seed(double x)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
__device__ MF_HH_INLINE void hh_scalars(double sigma, double x0, double &alpha, double &beta, double &rinv)
{
    if (sigma == 0.0) {   // zero column: identity reflector, zero pivot (NaN takes the normal path and propagates)
        alpha = 0.0;
        beta = 0.0;
        rinv = 0.0;
        return;
    }
    // sqrt(sigma), 1/sqrt(sigma) and 1/(sigma + |x0| sqrt(sigma)) from two hardware seeds and Newton steps:
    // a third of the instructions of the IEEE rsqrt / reciprocal sequences, accurate to an ulp or two
    const double h = 0.5 * sigma;
    double y = rsqrt_seed(sigma);
    y = y * fma(-h * y, y, 1.5);
    y = y * fma(-h * y, y, 1.5);
    double sq = sigma * y;
    sq = fma(fma(-sq, sq, sigma), 0.5 * y, sq);   // sq -> sqrt(sigma)
    const double rs = fma(fma(-sq, y, 1.0), y, y); // rs -> 1 / sq
    alpha = (x0 >= 0.0) ? -sq : sq;
    rinv = (x0 >= 0.0) ? -rs : rs;
    const double den = fma(fabs(x0), sq, sigma);   // sigma - x0 * alpha
    double r = rcp_seed(den);
    r = r * fma(-den, r, 2.0);
    r = r * fma(-den, r, 2.0);
    r = fma(fma(-den, r, 1.0), r, r);
    beta = r;
}

// returns 0 on success, 1 when the star does not fit this class (caller reroutes it to the dense kernel)
// Team mode (experimental, k_gls_mf_team): the warps of one CTA keep loosely in step, front by front, so that they run
// the same stretch of the 150 KB kernel body at the same time and share its instruction fetches.  No barrier: a warp
// that is ahead of the slowest live warp by more than `slack` fronts naps for a bounded number of rounds.
struct MfTeam {
    volatile unsigned *prog;   // shared: fronts started so far, one counter per warp (0xffffffff: warp has left)
    int warp, team, slack, spins;
    unsigned step;
};

template <bool TEAM>
__device__ int mf_node(const GlsArgs &a, int p, unsigned char *smem, const MfClass &kc, double *rslab, double *garena, int flags,
                       MfTeam *tm = nullptr)
{
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    MfWs w = mf_carve(smem, kc, garena);
    const int eb = a.esup_ptr[p], E = a.esup_ptr[p + 1] - eb;
    const int fb = a.fsup_ptr[p], F = a.fsup_ptr[p + 1] - fb;
    const bool neu = a.nflag[p] != 0;
    const double xv0 = a.coords[(i64)p * 3 + 0], xv1 = a.coords[(i64)p * 3 + 1], xv2 = a.coords[(i64)p * 3 + 2];
    const int ngcap = mf_ngcap(kc);

    // ---- setup: esup row, element groups ----
    // The original rows (element rows, face groups, Neumann rows) are built in the SHARED front buffer, which is idle
    // until the first general front: the lane-per-leaf phase reads them from there, and only the groups it leaves
    // behind (the element rows of the non-leaf blocks on a closed star) move on to the global arena.  Keeps ~0.85 k
    // doubles per node out of the L2-resident slab and takes the global round trips out of the leaf phase.
    for (int i = lane; i < E; i += 32) w.es[i] = a.esup[eb + i];
    __syncwarp();
    int n_if = 0;
    for (int f0 = 0; f0 < F; f0 += 32) {
        int fi = f0 + lane;
        bool interior = false;
        if (fi < F) interior = a.esuf2[a.fsup[fb + fi]].y >= 0;
        n_if += __popc(__ballot_sync(FULL, interior));
    }
    const int n_bf = F - n_if;
    const int off_if = 4 * E, off_bf = 4 * E + 21 * n_if;
    const int orig_len = off_bf + (neu ? 4 * n_bf : 0);
    const bool orig_in_smem = orig_len <= kc.fcap;
    double *orig = orig_in_smem ? w.front : w.arena;
    for (int i = lane; i < E; i += 32) {
        const double *cc = a.cent + (i64)w.es[i] * NPB_CSTRIDE;
        double d0 = cc[0] - xv0, d1 = cc[1] - xv1, d2 = cc[2] - xv2;
        w.dvec[3 * i] = d0; w.dvec[3 * i + 1] = d1; w.dvec[3 * i + 2] = d2;
        double *row = orig + 4 * i;                       // [ d^T | 1 ]   gls.pyx:268-281
        row[0] = d0; row[1] = d1; row[2] = d2; row[3] = 1.0;
        w.g_mask[i] = 1ull << i;
        w.g_off[i] = 4 * i;
        w.g_nr[i] = 1;
        w.g_ld[i] = 4;
    }
    // ---- face groups (gls.pyx:291-356) and Neumann groups (:394-416) ----
    int if_seen = 0, bf_seen = 0;
    for (int f0 = 0; f0 < F; f0 += 32) {
        int fi = f0 + lane;
        int face = -1;
        int2 e2 = make_int2(-1, -1);
        if (fi < F) {
            face = a.fsup[fb + fi];
            e2 = a.esuf2[face];
        }
        bool interior = (fi < F) && e2.y >= 0;
        bool boundary = (fi < F) && e2.y < 0;
        unsigned mi = __ballot_sync(FULL, interior);
        unsigned mb = __ballot_sync(FULL, boundary);
        unsigned below = (1u << lane) - 1u;
        if (interior) {
            int j = if_seen + __popc(mi & below);
            int I1 = 0, I2 = 0;
            for (int k = 0; k < E; k++) {
                int ek = w.es[k];
                if (ek == e2.x) I1 = k;
                if (ek == e2.y) I2 = k;
            }
            const double *Nn = a.fnormal + (i64)face * 3;
            const double *xs = a.fcent + (i64)face * 3;
            double N0 = Nn[0], N1 = Nn[1], N2 = Nn[2];
            double t0 = xv0 - xs[0], t1 = xv1 - xs[1], t2 = xv2 - xs[2];                     // T1 = x_v - x_S
            double c0 = gls_cross(N1, t2, N2, t1), c1 = gls_cross(N2, t0, N0, t2), c2 = gls_cross(N0, t1, N1, t0);   // T2 = N x T1
            double eta = fmax(fmax(0.0, a.diff_mag[e2.x]), a.diff_mag[e2.y]);
            double tau = pow(gls_norm3(c0, c1, c2), -eta);
            const double *K1 = a.perm + (i64)e2.x * 9;
            const double *K2 = a.perm + (i64)e2.y * 9;
            // columns in ascending block order: the owner (smaller element id) has the smaller local index
            double s1 = -1.0, s2 = 1.0;
            int lo_i = I1, hi_i = I2;
            if (I2 < I1) { lo_i = I2; hi_i = I1; s1 = 1.0; s2 = -1.0; const double *t = K1; K1 = K2; K2 = t; }
            double *r1 = orig + off_if + 21 * j;      // 3 rows x (3 + 3 + rhs)
            double *r2 = r1 + 7, *r3 = r2 + 7;
            const double tc0 = __dmul_rn(tau, c0), tc1 = __dmul_rn(tau, c1), tc2 = __dmul_rn(tau, c2);
#pragma unroll
            for (int q = 0; q < 3; q++) {
                r1[q] = s1 * gls_kn(K1 + 3 * q, N0, N1, N2);
                r1[3 + q] = s2 * gls_kn(K2 + 3 * q, N0, N1, N2);
            }
            r2[0] = s1 * t0; r2[1] = s1 * t1; r2[2] = s1 * t2; r2[3] = s2 * t0; r2[4] = s2 * t1; r2[5] = s2 * t2;
            r3[0] = s1 * tc0; r3[1] = s1 * tc1; r3[2] = s1 * tc2;
            r3[3] = s2 * tc0; r3[4] = s2 * tc1; r3[5] = s2 * tc2;
            r1[6] = 0.0; r2[6] = 0.0; r3[6] = 0.0;
            int g = E + j;
            w.g_mask[g] = (1ull << lo_i) | (1ull << hi_i);
            w.g_off[g] = off_if + 21 * j;
            w.g_nr[g] = 3;
            w.g_ld[g] = 7;
        }
        if (boundary && neu) {
            int j = bf_seen + __popc(mb & below);
            int Ik = 0;
            for (int k = 0; k < E; k++)
                if (w.es[k] == e2.x) Ik = k;
            const double *Nn = a.fnormal + (i64)face * 3;
            const double *K1 = a.perm + (i64)e2.x * 9;
            double N0 = Nn[0], N1 = Nn[1], N2 = Nn[2];
            double *rr = orig + off_bf + 4 * j;
#pragma unroll
            for (int q = 0; q < 3; q++) rr[q] = -gls_kn(K1 + 3 * q, N0, N1, N2);
            rr[3] = 0.0;
            int g = E + n_if + j;
            w.g_mask[g] = 1ull << Ik;
            w.g_off[g] = off_bf + 4 * j;
            w.g_nr[g] = 1;
            w.g_ld[g] = 4;
        }
        if_seen += __popc(mi);
        bf_seen += __popc(mb);
    }
    int ng = E + n_if + (neu ? n_bf : 0);
    const int ng_orig = ng;
    int top = orig_in_smem ? 0 : orig_len;   // the global arena starts empty when the original rows live in shared memory
    __syncwarp();

    // ---- adjacency bitmasks: lane b owns blocks b and b + 32 ----
    u64 adjA = 0, adjB = 0;
    {
        u64 *adj = reinterpret_cast<u64 *>(w.gvec);   // [E], free until the back substitution
        for (int i = lane; i < E; i += 32) adj[i] = 1ull << i;
        __syncwarp();
        for (int g = E + lane; g < ng; g += 32) {   // groups 0..E-1 are the element rows: one block each
            const u64 mk = w.g_mask[g];
            u64 m = mk;
            atomicOr((unsigned long long *)&adj[__ffsll((long long)m) - 1], mk);
            m &= m - 1;
            if (m) atomicOr((unsigned long long *)&adj[__ffsll((long long)m) - 1], mk);
        }
        __syncwarp();
        if (lane < E) adjA = adj[lane];
        if (lane + 32 < E) adjB = adj[lane + 32];
        __syncwarp();
    }
    u64 alive = (E >= 64) ? ~0ull : ((1ull << E) - 1ull);
    int nR = 0, rtop = 0;   // R rows written so far (entries / doubles in the global slab)
    int n_leaf = 0;         // the first n_leaf entries of the R table are leaf fronts

    // ---- leaf fronts, one per LANE ----
    // A block none of whose neighbours has been eliminated has a front made of original rows only: its
    // element row and its <= 3 face groups (3 rows coupling it to one neighbour, or one Neumann row),
    // 10 x (3 + 3 nn + 1) with a fixed sparsity.  Such blocks are pairwise independent when no two are
    // adjacent, so a greedy independent set of them (12 of the 24 tets around an interior node of the
    // Kuhn mesh) is eliminated at once: lane b factors the front of block b entirely in registers and
    // writes its 3 rows of R and its 7-row contribution block straight to the slabs.
    if (!(flags & 1) && ng - E <= 64) {
        u64 *fmask = w.r_mask;   // free until the first rows of R are recorded
        for (int i = lane; i < E; i += 32) fmask[i] = 0ull;
        __syncwarp();
        for (int g = E + lane; g < ng; g += 32) {   // atomicOr: the result does not depend on the order
            u64 mk = w.g_mask[g];
            const u64 bit = 1ull << (g - E);
            atomicOr((unsigned long long *)&fmask[__ffsll((long long)mk) - 1], bit);
            mk &= mk - 1;
            if (mk) atomicOr((unsigned long long *)&fmask[__ffsll((long long)mk) - 1], bit);
        }
        __syncwarp();
        const int b = lane;
        u64 fm = (b < E) ? fmask[b] : 0ull;
        __syncwarp();
        const int nf = __popcll(fm);
        bool elig = b < E && nf <= 3;
        int gk[3], nbk[3], offk[3];
        bool valid[3], intr[3];
        u64 Upl = 0;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            valid[k] = elig && k < nf;
            gk[k] = E + (valid[k] ? __ffsll((long long)fm) - 1 : 0);
            fm &= fm - 1;
            const u64 other = valid[k] ? (w.g_mask[gk[k]] & ~(1ull << b)) : 0ull;
            intr[k] = other != 0;
            nbk[k] = intr[k] ? __ffsll((long long)other) - 1 : 0;
            offk[k] = valid[k] ? w.g_off[gk[k]] : 0;
            if (intr[k] && ((Upl >> nbk[k]) & 1ull)) elig = false;   // two faces shared with one neighbour
            if (intr[k]) Upl |= 1ull << nbk[k];
        }
        // greedy independent set in index order (what minimum degree picks on a closed star)
        unsigned rem = __ballot_sync(FULL, elig), chosen = 0;
        {
            const unsigned nbm = (unsigned)Upl;
            while (rem) {
                const int bb = __ffs(rem) - 1;
                chosen |= 1u << bb;
                rem &= ~(__shfl_sync(FULL, nbm, bb) | (1u << bb));
            }
        }
        const bool mine = (chosen >> lane) & 1u;
        const int nn = __popcll(Upl);
        const int c = 3 * nn + 4, cw = c - 3;
        const int cbsz = (mine && nn > 0) ? 7 * cw : 0, rsz = mine ? 3 * c : 0;
        int cb_incl = cbsz, r_incl = rsz;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t1 = __shfl_up_sync(FULL, cb_incl, o), t2 = __shfl_up_sync(FULL, r_incl, o);
            if (lane >= o) { cb_incl += t1; r_incl += t2; }
        }
        const int cb_tot = __shfl_sync(FULL, cb_incl, 31), r_tot = __shfl_sync(FULL, r_incl, 31);
        const unsigned hascb = __ballot_sync(FULL, mine && nn > 0);
        if (ng + __popc(hascb) > ngcap || top + cb_tot > kc.acap || rtop + r_tot > kc.acap) return 1;
        if (mine) {
            const unsigned below = (1u << lane) - 1u;
            double *Rr = rslab + rtop + (r_incl - rsz);
            double *CB = w.arena + top + (cb_incl - cbsz);
            double a0[10], a1[10], a2[10];
            a0[0] = w.dvec[3 * b]; a1[0] = w.dvec[3 * b + 1]; a2[0] = w.dvec[3 * b + 2];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                // own columns come second when the neighbour has the smaller index
                const double *src = orig + offk[k] + ((intr[k] && nbk[k] < b) ? 3 : 0);
                const int ld = intr[k] ? 7 : 4;
#pragma unroll
                for (int r = 0; r < 3; r++) {
                    const bool has = valid[k] && (intr[k] || r == 0);
                    a0[1 + 3 * k + r] = has ? src[r * ld] : 0.0;
                    a1[1 + 3 * k + r] = has ? src[r * ld + 1] : 0.0;
                    a2[1 + 3 * k + r] = has ? src[r * ld + 2] : 0.0;
                }
            }
            double alpha0, beta0, alpha1, beta1, alpha2, beta2, ri0, ri1, ri2;
            {
                double sg = 0.0;
#pragma unroll
                for (int q = 0; q < 10; q++) sg += a0[q] * a0[q];
                hh_scalars(sg, a0[0], alpha0, beta0, ri0);
                a0[0] -= alpha0;
                double t1 = 0.0, t2 = 0.0;
#pragma unroll
                for (int q = 0; q < 10; q++) { t1 += a0[q] * a1[q]; t2 += a0[q] * a2[q]; }
                t1 *= beta0; t2 *= beta0;
#pragma unroll
                for (int q = 0; q < 10; q++) { a1[q] -= t1 * a0[q]; a2[q] -= t2 * a0[q]; }
            }
            const double r01 = a1[0], r02 = a2[0];
            a1[0] = 0.0; a2[0] = 0.0;
            {
                double sg = 0.0;
#pragma unroll
                for (int q = 1; q < 10; q++) sg += a1[q] * a1[q];
                hh_scalars(sg, a1[1], alpha1, beta1, ri1);
                a1[1] -= alpha1;
                double t2 = 0.0;
#pragma unroll
                for (int q = 1; q < 10; q++) t2 += a1[q] * a2[q];
                t2 *= beta1;
#pragma unroll
                for (int q = 1; q < 10; q++) a2[q] -= t2 * a1[q];
            }
            const double r12 = a2[1];
            a2[1] = 0.0;
            double d10 = 0.0, d20 = 0.0, d21 = 0.0;
            {
                double sg = 0.0;
#pragma unroll
                for (int q = 2; q < 10; q++) sg += a2[q] * a2[q];
                hh_scalars(sg, a2[2], alpha2, beta2, ri2);
                a2[2] -= alpha2;
#pragma unroll
                for (int q = 0; q < 10; q++) { d10 += a1[q] * a0[q]; d20 += a2[q] * a0[q]; d21 += a2[q] * a1[q]; }
            }
            Rr[0] = ri0; Rr[1] = r01; Rr[2] = r02;
            Rr[c] = 0.0; Rr[c + 1] = ri1; Rr[c + 2] = r12;
            Rr[2 * c] = 0.0; Rr[2 * c + 1] = 0.0; Rr[2 * c + 2] = ri2;
            // the neighbours' columns: three nonzeros each before the reflections, dense after
#pragma unroll
            for (int k = 0; k < 3; k++) {
                if (!intr[k]) continue;
                const int slot = 1 + __popcll(Upl & ((1ull << nbk[k]) - 1ull));
                const double *src = orig + offk[k] + ((nbk[k] < b) ? 0 : 3);
#pragma unroll
                for (int q = 0; q < 3; q++) {
                    const double n0 = src[q], n1 = src[7 + q], n2 = src[14 + q];
                    const double w0 = a0[1 + 3 * k] * n0 + a0[2 + 3 * k] * n1 + a0[3 + 3 * k] * n2;
                    const double w1 = a1[1 + 3 * k] * n0 + a1[2 + 3 * k] * n1 + a1[3 + 3 * k] * n2;
                    const double w2 = a2[1 + 3 * k] * n0 + a2[2 + 3 * k] * n1 + a2[3 + 3 * k] * n2;
                    const double s0 = beta0 * w0;
                    const double s1 = beta1 * (w1 - d10 * s0);
                    const double s2 = beta2 * (w2 - d20 * s0 - d21 * s1);
                    double *rcol = Rr + 3 * slot + q, *ccol = CB + 3 * (slot - 1) + q;
#pragma unroll
                    for (int r = 0; r < 10; r++) {
                        double o = (r == 1 + 3 * k) ? n0 : (r == 2 + 3 * k) ? n1 : (r == 3 + 3 * k) ? n2 : 0.0;
                        double v = o - (a0[r] * s0 + a1[r] * s1 + a2[r] * s2);
                        if (r < 3) rcol[r * c] = v;
                        else ccol[(r - 3) * cw] = v;
                    }
                }
            }
            {   // right-hand side: e_0 before the reflections
                const double s0 = beta0 * a0[0];
                const double s1 = beta1 * (-d10 * s0);
                const double s2 = beta2 * (-d20 * s0 - d21 * s1);
#pragma unroll
                for (int r = 0; r < 10; r++) {
                    double v = (r == 0 ? 1.0 : 0.0) - (a0[r] * s0 + a1[r] * s1 + a2[r] * s2);
                    if (r < 3) Rr[r * c + c - 1] = v;
                    else if (nn > 0) CB[(r - 3) * cw + cw - 1] = v;
                }
            }
            // tables: consumed groups, the new contribution block, the rows of R
            w.g_nr[b] = 0;
#pragma unroll
            for (int k = 0; k < 3; k++)
                if (valid[k]) w.g_nr[gk[k]] = 0;
            if (nn > 0) {
                const int gi = ng + __popc(hascb & below);
                w.g_mask[gi] = Upl;
                w.g_off[gi] = top + (cb_incl - cbsz);
                w.g_nr[gi] = 7;
                w.g_ld[gi] = (unsigned char)cw;
            }
            const int ri = nR + __popc(chosen & below);
            w.r_mask[ri] = Upl | (1ull << b);
            w.r_off[ri] = rtop + (r_incl - rsz);
            w.r_meta[ri] = b | (3 << 8) | (c << 16);
        }
        __syncwarp();
        // adjacency: the neighbours of every eliminated leaf become a clique
        const u64 Ufull = mine ? (Upl | (1ull << b)) : 0ull;
        for (unsigned cm = chosen; cm; cm &= cm - 1) {
            const int bb = __ffs(cm) - 1;
            const u64 Ub = __shfl_sync(FULL, Ufull, bb);
            const u64 keep = ~(1ull << bb);
            if (((Ub >> lane) & 1ull) && lane != bb) adjA = (adjA | Ub) & keep;
            if ((Ub >> (lane + 32)) & 1ull) adjB = (adjB | Ub) & keep;
        }
        alive &= ~(u64)chosen;
        top += cb_tot;
        ng += __popc(hascb);
        nR += __popc(chosen);
        n_leaf = nR;
        rtop += r_tot;
        __syncwarp();
    }

    // ---- original groups that survived the leaf phase leave the front buffer for the global arena ----
    // They are re-entered at the END of the group table, so that table order stays arena order (mf_compact relies on it).
    if (orig_in_smem) {
        for (int g0 = 0; g0 < ng_orig; g0 += 32) {
            const int g = g0 + lane;
            int sz = 0, src_off = 0, nr = 0, gld = 0;
            u64 mk = 0;
            if (g < ng_orig && w.g_nr[g] > 0) {
                nr = w.g_nr[g];
                gld = w.g_ld[g];
                sz = nr * gld;
                src_off = w.g_off[g];
                mk = w.g_mask[g];
            }
            int incl = sz;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const int tot = __shfl_sync(FULL, incl, 31);
            const unsigned live = __ballot_sync(FULL, sz > 0);
            if (top + tot > kc.acap || ng + __popc(live) > ngcap) return 1;
            if (sz > 0) {
                const int dst = top + incl - sz;
                for (int q = 0; q < sz; q++) w.arena[dst + q] = orig[src_off + q];
                const int gi = ng + __popc(live & ((1u << lane) - 1u));
                w.g_mask[gi] = mk;
                w.g_off[gi] = dst;
                w.g_nr[gi] = (unsigned short)nr;
                w.g_ld[gi] = (unsigned char)gld;
                w.g_nr[g] = 0;
            }
            top += tot;
            ng += __popc(live);
        }
        __syncwarp();
    }

    // ---- elimination ----
    // The contribution block of a front stays where it is (rows >= 3, columns >= 3 of the front) until the
    // next pivot is known: when that pivot is the block's first column and brings no new column - every
    // step of the dense end game, where the remaining blocks form a clique - the next front is built in
    // place around it and only the new rows are fetched; otherwise it is flushed to the group arena.
    int ch_rows = 0, ch_off = 0, ch_ld = 0;
    u64 ch_mask = 0;
    while (alive) {
        if (TEAM) {
            tm->step++;
            if (lane == 0) tm->prog[tm->warp] = tm->step;
            for (int spin = 0; spin < tm->spins; spin++) {
                unsigned mn = 0xffffffffu;
                if (lane < tm->team) mn = tm->prog[lane];
                mn = __reduce_min_sync(FULL, mn);
                if (tm->step <= mn + (unsigned)tm->slack) break;
                __nanosleep(64);
            }
        }
        // (a) minimum-degree pivot block
        unsigned keyA = ((alive >> lane) & 1ull) ? (unsigned)((__popcll(adjA) << 8) | lane) : 0xffffffffu;
        unsigned keyB = ((alive >> (lane + 32)) & 1ull) ? (unsigned)((__popcll(adjB) << 8) | (lane + 32)) : 0xffffffffu;
        unsigned key = __reduce_min_sync(FULL, keyA < keyB ? keyA : keyB);
        const int piv = (int)(key & 0xffu);
        const u64 pbit = 1ull << piv;
        // rescue for stars whose contribution blocks outgrow the slab: close the holes left by consumed groups
        // (regular stars never get here; compacting eagerly would cut HBM write-back traffic but costs ~9 % time)
        if (top > (kc.acap / 4) * 3) {
            mf_compact(w, ng, top, lane);
        }
        // (b) row groups containing the pivot block
        int nS = 0, rho = 0;
        u64 U = 0;
        for (int g0 = 0; g0 < ng; g0 += 32) {
            int g = g0 + lane;
            bool in = false;
            int nr = 0;
            u64 mk = 0;
            if (g < ng) {
                nr = w.g_nr[g];
                mk = w.g_mask[g];
                in = nr > 0 && (mk & pbit);
            }
            unsigned bal = __ballot_sync(FULL, in);
            if (bal == 0) continue;
            int pos = nS + __popc(bal & ((1u << lane) - 1u));
            if (in && pos < MF_SCAP) w.s_list[pos] = g;
            nS += __popc(bal);
            rho += __reduce_add_sync(FULL, in ? nr : 0);
            U |= warp_or64(in ? mk : 0ull);
        }
        bool inplace = false;
        if (ch_rows > 0) {
            const bool has = (ch_mask & pbit) != 0;
            if (has && (ch_mask & (pbit - 1ull)) == 0 && (U & ~ch_mask) == 0 && nS <= MF_SCAP)
                inplace = ch_rows + rho <= min(32 * MF_RPL, (kc.fcap - ch_off) / ch_ld);
            if (inplace) {
                U = ch_mask;
            } else {
                const int cwp = 3 * __popcll(ch_mask) + 1;
                if (ng + 1 > ngcap || top + ch_rows * cwp > kc.acap) return 1;
                mf_store_cb(w.front + ch_off, ch_ld, ch_rows, cwp, w.arena + top, lane);
                if (lane == 0) {
                    w.g_mask[ng] = ch_mask;
                    w.g_off[ng] = top;
                    w.g_nr[ng] = (unsigned short)ch_rows;
                    w.g_ld[ng] = (unsigned char)cwp;
                    if (has && nS < MF_SCAP) w.s_list[nS] = ng;
                }
                if (has) {
                    nS++;
                    U |= ch_mask;
                    rho += ch_rows;
                }
                top += ch_rows * cwp;
                ng++;
                __syncwarp();
            }
        }
        const u64 Up = U & ~pbit;
        const int c = 3 * __popcll(U) + 1;
        // (c) capacity checks: group table, R slab; the front is processed in chunks of at most `rcap` rows
        const int ld = inplace ? ch_ld : ((c + 1) & ~1);   // even row stride
        const int rcap = inplace ? ch_rows + rho : min(32 * MF_RPL, kc.fcap / ld);
        const int La = c > 16 ? 32 : c > 8 ? 16 : c > 4 ? 8 : 4, Ga = 32 / La;   // assembly: lanes per front row
        if (nS > MF_SCAP || (!inplace && rcap < 8) || rtop + 3 * c > kc.acap) return 1;
        // block id of every column slot: slot 0 = pivot, then the other blocks ascending
        if ((Up >> lane) & 1ull) w.colblk[1 + __popcll(Up & ((1ull << lane) - 1ull))] = (unsigned char)lane;
        if ((Up >> (lane + 32)) & 1ull) w.colblk[1 + __popcll(Up & ((1ull << (lane + 32)) - 1ull))] = (unsigned char)(lane + 32);
        if (lane == 0) w.colblk[0] = (unsigned char)piv;
        __syncwarp();
        double *Fm = inplace ? w.front + ch_off : w.front;
        const bool par = inplace && (ch_off & 1);   // odd offset: the (v1, v2) pair is the 16-byte aligned one
        const unsigned front_s = (unsigned)__cvta_generic_to_shared(Fm);
        int t_next = 0, r_done = 0; // next group of the S list / rows of it already taken
        int carry = inplace ? ch_rows : 0;   // rows already in the front: the chained block / the previous chunk's pivot rows
        ch_rows = 0;
        int npiv = 0;
        double fri0 = 0.0, fri1 = 0.0, fri2 = 0.0;   // 1 / alpha of the last chunk's pivots
#ifdef MF_ZERO_FIRST
        int rho_left = rho;   // rows of the S list not assembled yet
#else
        (void)rho;
#endif
        for (bool last = false; !last;) {
            // (d) assemble one chunk: lanes over front columns [pivot block | other blocks ascending | rhs]
            int rho_c = carry;
#ifdef MF_ZERO_FIRST
            {   // the rows this chunk assembles are cleared at once; the groups then copy only the entries they have
                const int fill = min(rcap - carry, rho_left) * ld;
                rho_left -= min(rcap - carry, rho_left);
                double *z = Fm + carry * ld;
                for (int i = lane; i < fill; i += 32) z[i] = 0.0;
                __syncwarp();
            }
#endif
            while (t_next < nS && rho_c < rcap) {
                const int g = w.s_list[t_next] & 0xffff;
                const u64 mk = w.g_mask[g];
                const int nr = w.g_nr[g], gld = w.g_ld[g];
                const int take = min(nr - r_done, rcap - rho_c);
                const double *gsrc = w.arena + w.g_off[g] + r_done * gld;
                // fronts of <= 16 columns: La lanes per row, Ga rows per step
                for (int j0 = 0; j0 < c; j0 += 32) {
                    const int j = (La == 32) ? j0 + lane : (lane & (La - 1));
                    const int r0 = (La == 32) ? 0 : lane / La;
                    if (j >= c) continue;
                    const bool is_rhs = (j == c - 1);
                    const int blk = is_rhs ? 0 : w.colblk[j / 3];
                    const bool has = is_rhs || ((mk >> blk) & 1ull);
                    const int sc = is_rhs ? 3 * __popcll(mk) : 3 * __popcll(mk & ((1ull << blk) - 1ull)) + j % 3;
                    if (has) {
                        const double *src = gsrc + sc + r0 * gld;
                        unsigned ds = front_s + (unsigned)(((rho_c + r0) * ld + j) * 8);
                        for (int r = r0; r < take; r += Ga) {
                            // row groups live in global memory: all copies of a chunk are in flight at once
                            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(ds), "l"(src) : "memory");
                            src += Ga * gld;
                            ds += (unsigned)(Ga * ld * 8);
                        }
                    }
#ifndef MF_ZERO_FIRST
                    else {
                        double *dst = Fm + (rho_c + r0) * ld + j;
                        for (int r = r0; r < take; r += Ga) {
                            *dst = 0.0;
                            dst += Ga * ld;
                        }
                    }
#endif
                }
                rho_c += take;
                r_done += take;
                if (r_done == nr) {
                    t_next++;
                    r_done = 0;
                }
            }
            last = (t_next >= nS);
            cp_async_wait_all();
            __syncwarp();
            // (e) panel: Householder on the three pivot columns, lanes over rows, entries in registers
            double a0[MF_RPL], a1[MF_RPL], a2[MF_RPL];
#pragma unroll
            for (int q = 0; q < MF_RPL; q++) {
                int r = lane + 32 * q;
                bool ok = r < rho_c;
                a0[q] = ok ? Fm[r * ld + 0] : 0.0;
                a1[q] = ok ? Fm[r * ld + 1] : 0.0;
                a2[q] = ok ? Fm[r * ld + 2] : 0.0;
            }
            double alpha0, beta0, alpha1, beta1, alpha2, beta2, d10, d20, d21, ri0, ri1, ri2;
            {
                double sg = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) sg += a0[q] * a0[q];
                sg = warp_sum(sg);
                double x00 = __shfl_sync(FULL, a0[0], 0);
                hh_scalars(sg, x00, alpha0, beta0, ri0);
                if (lane == 0) a0[0] = x00 - alpha0;                  // a0 now holds v0
                double t1 = 0.0, t2 = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) { t1 += a0[q] * a1[q]; t2 += a0[q] * a2[q]; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { t1 += __shfl_xor_sync(FULL, t1, o); t2 += __shfl_xor_sync(FULL, t2, o); }
                t1 *= beta0; t2 *= beta0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) { a1[q] -= t1 * a0[q]; a2[q] -= t2 * a0[q]; }
            }
            double r01 = __shfl_sync(FULL, a1[0], 0), r02 = __shfl_sync(FULL, a2[0], 0);
            {
                if (lane == 0) a1[0] = 0.0;                           // rows above the pivot do not take part
                double sg = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) sg += a1[q] * a1[q];
                sg = warp_sum(sg);
                double x11 = __shfl_sync(FULL, a1[0], 1);
                hh_scalars(sg, x11, alpha1, beta1, ri1);
                if (lane == 1) a1[0] = x11 - alpha1;                  // a1 now holds v1
                if (lane == 0) a2[0] = 0.0;
                double t2 = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) t2 += a1[q] * a2[q];
                t2 = warp_sum(t2) * beta1;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) a2[q] -= t2 * a1[q];
            }
            double r12 = __shfl_sync(FULL, a2[0], 1);
            {
                if (lane == 1) a2[0] = 0.0;
                double sg = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) sg += a2[q] * a2[q];
                sg = warp_sum(sg);
                double x22 = __shfl_sync(FULL, a2[0], 2);
                hh_scalars(sg, x22, alpha2, beta2, ri2);
                if (lane == 2) a2[0] = x22 - alpha2;                  // a2 now holds v2
                d10 = 0.0; d20 = 0.0; d21 = 0.0;
#pragma unroll
                for (int q = 0; q < MF_RPL; q++) { d10 += a1[q] * a0[q]; d20 += a2[q] * a0[q]; d21 += a2[q] * a1[q]; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    d10 += __shfl_xor_sync(FULL, d10, o);
                    d20 += __shfl_xor_sync(FULL, d20, o);
                    d21 += __shfl_xor_sync(FULL, d21, o);
                }
            }
            // the Householder vectors overwrite the panel columns of the front (LAPACK style); the pivot rows'
            // panel entries of R are put back after the update
#pragma unroll
            for (int q = 0; q < MF_RPL; q++) {
                int r = lane + 32 * q;
                if (r < rho_c) {
                    Fm[r * ld] = a0[q];
                    Fm[r * ld + 1] = a1[q];
                    Fm[r * ld + 2] = a2[q];
                }
            }
            __syncwarp();
            // (f) apply the three reflections to the other columns: two passes over the rows.  Narrow fronts
            //     (<= 16 other columns: the tall-skinny end game) split the rows over 2..32 lane groups
            const int cw3 = c - 3;
            const int po = par ? 1 : 0, so = par ? 0 : 2;   // aligned pair of v entries / the single one
            // lanes per group: the power of two covering the columns; G = 32 / L groups take rows g, g + G, ...
            const int L = cw3 > 16 ? 32 : cw3 > 8 ? 16 : cw3 > 4 ? 8 : cw3 > 2 ? 4 : cw3 > 1 ? 2 : 1;
            if (L < 32 && cw3 > 0) {
                const int G = 32 / L, grp = lane / L, jl = lane & (L - 1);
                const bool act = jl < cw3;
                const int j = 3 + (act ? jl : 0);
                const int step = G * ld;
                double wa = 0.0, wb = 0.0, wc = 0.0;
                {
                    const double *vp = Fm + grp * ld;
MF_UNROLL_APPLY
                    for (int r = grp; r < rho_c; r += G) {
                        double f = vp[j];
                        double2 va = *reinterpret_cast<const double2 *>(vp + po);
                        double vc = vp[so];
                        wa += va.x * f; wb += va.y * f; wc += vc * f;
                        vp += step;
                    }
                }
                for (int o = L; o < 32; o <<= 1) {
                    wa += __shfl_xor_sync(FULL, wa, o);
                    wb += __shfl_xor_sync(FULL, wb, o);
                    wc += __shfl_xor_sync(FULL, wc, o);
                }
                const double w0 = par ? wc : wa, w1 = par ? wa : wb, w2 = par ? wb : wc;
                double s0 = beta0 * w0;
                double s1 = beta1 * (w1 - d10 * s0);
                double s2 = beta2 * (w2 - d20 * s0 - d21 * s1);
                const double ca = par ? s1 : s0, cb = par ? s2 : s1, cc = par ? s0 : s2;
                if (act) {
                    double *vp = Fm + grp * ld;
MF_UNROLL_APPLY
                    for (int r = grp; r < rho_c; r += G) {
                        double2 va = *reinterpret_cast<const double2 *>(vp + po);
                        double vc = vp[so];
                        vp[j] = vp[j] - (va.x * ca + va.y * cb + vc * cc);
                        vp += step;
                    }
                }
            } else
            for (int j0 = 3; j0 < c; j0 += 32) {
                int j = j0 + lane;
                if (j >= c) continue;
                double wa = 0.0, wb = 0.0, wc = 0.0;
                {
                    const double *fp = Fm + j;
                    const double *vp = Fm;
MF_UNROLL_APPLY
                    for (int r = 0; r < rho_c; r++) {
                        double f = *fp;
                        double2 va = *reinterpret_cast<const double2 *>(vp + po);
                        double vc = vp[so];
                        wa += va.x * f; wb += va.y * f; wc += vc * f;
                        fp += ld; vp += ld;
                    }
                }
                const double w0 = par ? wc : wa, w1 = par ? wa : wb, w2 = par ? wb : wc;
                double s0 = beta0 * w0;
                double s1 = beta1 * (w1 - d10 * s0);
                double s2 = beta2 * (w2 - d20 * s0 - d21 * s1);
                const double ca = par ? s1 : s0, cb = par ? s2 : s1, cc = par ? s0 : s2;
                {
                    double *fp = Fm + j;
                    const double *vp = Fm;
MF_UNROLL_APPLY
                    for (int r = 0; r < rho_c; r++) {
                        double2 va = *reinterpret_cast<const double2 *>(vp + po);
                        double vc = vp[so];
                        *fp = *fp - (va.x * ca + va.y * cb + vc * cc);
                        fp += ld; vp += ld;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) {
                Fm[0] = alpha0; Fm[1] = r01; Fm[2] = r02;
                if (rho_c > 1) { Fm[ld] = 0.0; Fm[ld + 1] = alpha1; Fm[ld + 2] = r12; }
                if (rho_c > 2) { Fm[2 * ld] = 0.0; Fm[2 * ld + 1] = 0.0; Fm[2 * ld + 2] = alpha2; }
            }
            __syncwarp();
            fri0 = ri0; fri1 = ri1; fri2 = ri2;
            // (g) rows below the pivot rows (columns of the other blocks + rhs) are appended to the group arena
            //     as a new contribution block; the pivot rows stay in the front for the next chunk, or go to
            //     the R slab after the last one
            npiv = rho_c < 3 ? rho_c : 3;
            const int left = rho_c - npiv;
            const bool keep = left > 0 && Up != 0;
            if (keep && last) {   // stays in the front until the next pivot is known
                ch_rows = left;
                ch_off = (int)(Fm - w.front) + npiv * ld + 3;
                ch_ld = ld;
                ch_mask = Up;
            } else if (keep) {
                const int cw = c - 3;
                if (ng + 1 > ngcap || top + left * cw > kc.acap) return 1;
                mf_store_cb(Fm + npiv * ld + 3, ld, left, cw, w.arena + top, lane);
                if (lane == 0) {
                    w.g_mask[ng] = Up;
                    w.g_off[ng] = top;
                    w.g_nr[ng] = (unsigned short)left;
                    w.g_ld[ng] = (unsigned char)cw;
                }
                top += left * cw;
                ng++;
            }
            carry = npiv;
            __syncwarp();
        }
        for (int t = lane; t < nS; t += 32) w.g_nr[w.s_list[t] & 0xffff] = 0;   // consumed
        // R rows to the slab; the diagonal carries 1 / alpha so that the back substitution has no divisions
        for (int j = lane; j < c; j += 32) {
            double v0 = Fm[j], v1 = Fm[ld + j], v2 = Fm[2 * ld + j];
            if (j == 0) v0 = fri0;
            if (j == 1) v1 = fri1;
            if (j == 2) v2 = fri2;
            rslab[rtop + j] = v0;
            if (npiv > 1) rslab[rtop + c + j] = v1;
            if (npiv > 2) rslab[rtop + 2 * c + j] = v2;
        }
        if (lane == 0) {
            w.r_mask[nR] = U;
            w.r_off[nR] = rtop;
            w.r_meta[nR] = piv | (npiv << 8) | (c << 16);
        }
        nR++;
        rtop += npiv * c;
        // (h) adjacency update: the neighbours of the pivot become a clique
        if ((Up >> lane) & 1ull) adjA = (adjA | U) & ~pbit;
        if ((Up >> (lane + 32)) & 1ull) adjB = (adjB | U) & ~pbit;
        alive &= ~pbit;
        __syncwarp();
    }

    // ---- back substitution through the R rows, newest first (slab copied back into the free arena) ----
    __syncwarp();
    const bool r_in_smem = rtop <= kc.fcap;
    if (r_in_smem) {
        for (int i = lane; i < rtop; i += 32) cp_async8(w.front + i, rslab + i);
        cp_async_wait_all();
    }
    const double *Rbase = r_in_smem ? w.front : rslab;
    for (int i = lane; i < 3 * E; i += 32) w.gvec[i] = 0.0;
    __syncwarp();
    for (int g = nR - 1; g >= n_leaf; g--) {
        const int meta = w.r_meta[g];
        const int piv = meta & 0xff, npiv = (meta >> 8) & 0xff, c = meta >> 16;
        const u64 Up = w.r_mask[g] & ~(1ull << piv);
        const double *R = Rbase + w.r_off[g];
        double p0 = 0.0, p1 = 0.0, p2 = 0.0;
        for (int j0 = 3; j0 < c - 1; j0 += 32) {
            int j = j0 + lane;
            if (j < c - 1) {
                int blk = nth_set_bit(Up, (j - 3) / 3);
                double gj = w.gvec[3 * blk + (j - 3) % 3];
                p0 += R[j] * gj;
                if (npiv > 1) p1 += R[c + j] * gj;
                if (npiv > 2) p2 += R[2 * c + j] * gj;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            p0 += __shfl_xor_sync(FULL, p0, o);
            p1 += __shfl_xor_sync(FULL, p1, o);
            p2 += __shfl_xor_sync(FULL, p2, o);
        }
        if (lane == 0) {
            double g0 = 0.0, g1 = 0.0, g2 = 0.0;   // the diagonal of R holds 1 / alpha (0 for a zero pivot)
            if (npiv > 2) g2 = (R[2 * c + c - 1] - p2) * R[2 * c + 2];
            if (npiv > 1) g1 = (R[c + c - 1] - p1 - R[c + 2] * g2) * R[c + 1];
            g0 = (R[c - 1] - p0 - R[1] * g1 - R[2] * g2) * R[0];
            w.gvec[3 * piv] = g0;
            w.gvec[3 * piv + 1] = g1;
            w.gvec[3 * piv + 2] = g2;
        }
        __syncwarp();
    }
    // leaf fronts: their unknowns depend on non-leaf blocks only, so all of them are solved at once, one per lane
    if (lane < n_leaf) {
        const int meta = w.r_meta[lane];
        const int piv = meta & 0xff, c = meta >> 16;
        u64 Up = w.r_mask[lane] & ~(1ull << piv);
        const double *R = Rbase + w.r_off[lane];
        double p0 = 0.0, p1 = 0.0, p2 = 0.0;
        for (int j = 3; Up; j += 3, Up &= Up - 1) {
            const double *gb = w.gvec + 3 * (__ffsll((long long)Up) - 1);
#pragma unroll
            for (int q = 0; q < 3; q++) {
                const double gj = gb[q];
                p0 += R[j + q] * gj;
                p1 += R[c + j + q] * gj;
                p2 += R[2 * c + j + q] * gj;
            }
        }
        const double g2 = (R[2 * c + c - 1] - p2) * R[2 * c + 2];
        const double g1 = (R[c + c - 1] - p1 - R[c + 2] * g2) * R[c + 1];
        const double g0 = (R[c - 1] - p0 - R[1] * g1 - R[2] * g2) * R[0];
        w.gvec[3 * piv] = g0;
        w.gvec[3 * piv + 1] = g1;
        w.gvec[3 * piv + 2] = g2;
    }
    __syncwarp();
    // ---- residual on the element rows, weights, CSR values ----
    double *wo = a.wbuf + ((i64)eb - a.wbase);
    double part = 0.0;
    for (int i = lane; i < E; i += 32) {
        double ri = 1.0 - (w.dvec[3 * i] * w.gvec[3 * i] + w.dvec[3 * i + 1] * w.gvec[3 * i + 1] + w.dvec[3 * i + 2] * w.gvec[3 * i + 2]);
        w.front[i] = ri;
        part += ri;
    }
    double tot = warp_sum(part);
    // r_i = 1 - d_i . g_i and sum_i r_i lose digits to cancellation when the system is nearly consistent (residuals
    // << 1, or of mixed sign: one-sided stars, typically 2-D Neumann boundary nodes; in 3-D r_i ~ 1 and the statistic
    // below sits at 2.0 - 2.9).  Such nodes go to the dense kernel, which forms r through the reflectors (k2_gls_dense.cu).
    double rmx = 0.0;
    for (int i = lane; i < E; i += 32) rmx = fmax(rmx, fabs(w.front[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmx = fmax(rmx, __shfl_xor_sync(FULL, rmx, o));
    if (!(1.0 / rmx + (double)E / fabs(tot) <= 4.0)) return 1;
    __syncwarp();
    double nv = neu ? w.front[E - 1] / tot : 0.0;   // gls.pyx:470-472 (Q3)
    int cnt = 0;
    for (int i = lane; i < E; i += 32) {
        double v = w.front[i] / tot + nv;           // interpolator.pyx:618 (Q4)
        wo[i] = v;
        cnt += (v != 0.0) ? 1 : 0;
    }
    cnt = __reduce_add_sync(FULL, cnt);
    if (lane == 0) {
        a.rowcnt[p] = cnt;
        a.neumann[p] = nv;
    }
    __syncwarp();
    return 0;
}

// persistent: one warp per CTA; nodes handed out through an atomic counter; stars that do not fit are
// appended to the overflow list for the dense kernel
template <int MINBLOCKS>
__global__ void __launch_bounds__(32, MINBLOCKS)
k_gls_mf(GlsArgs a, const int32_t *__restrict__ list, int count, int *__restrict__ counter, int klass,
         int32_t *__restrict__ overflow, int *__restrict__ n_overflow, double *__restrict__ slabs, int flags)
{
    extern __shared__ __align__(16) unsigned char smem_mf[];
    const MfClass kc = c_mf[klass];
    double *rslab = slabs + (size_t)blockIdx.x * kc.acap * 2;   // per CTA: R slab, then the group arena
    double *garena = rslab + kc.acap;
    while (true) {
        int i = 0;
        if (threadIdx.x == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= count) break;
        int p = list[i];
        int rc = mf_node<false>(a, p, smem_mf, kc, rslab, garena, flags);
        __syncwarp();
        if (rc != 0 && threadIdx.x == 0) overflow[atomicAdd(n_overflow, 1)] = p;
    }
}

// Team launch: up to WARPS one-node warps per CTA (blockDim.x / 32 of them), one CTA per SM, loosely in step (see MfTeam).
// WARPS only sets the register budget (12: 168 registers, 16: 128), like MINBLOCKS of k_gls_mf.
template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS, 1)
k_gls_mf_team(GlsArgs a, const int32_t *__restrict__ list, int count, int *__restrict__ counter, int klass,
              int32_t *__restrict__ overflow, int *__restrict__ n_overflow, double *__restrict__ slabs, int flags,
              int smem_per_warp, int slack, int spins)
{
    extern __shared__ __align__(16) unsigned char smem_mf[];
    const MfClass kc = c_mf[klass];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, team = blockDim.x >> 5;
    MfTeam tm;
    tm.prog = (volatile unsigned *)smem_mf;
    tm.warp = warp; tm.team = team; tm.slack = slack; tm.spins = spins; tm.step = 0;
    if (lane == 0) tm.prog[warp] = 0;
    __syncthreads();
    unsigned char *my = smem_mf + 128 + (size_t)warp * smem_per_warp;
    double *rslab = slabs + ((size_t)blockIdx.x * team + warp) * kc.acap * 2;
    double *garena = rslab + kc.acap;
    while (true) {
        int i = 0;
        if (lane == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= count) break;
        int p = list[i];
        int rc = mf_node<true>(a, p, my, kc, rslab, garena, flags, &tm);
        __syncwarp();
        if (rc != 0 && lane == 0) overflow[atomicAdd(n_overflow, 1)] = p;
    }
    if (lane == 0) tm.prog[warp] = 0xffffffffu;   // the others no longer wait for this warp
}

int npb_k2_gls(npb_ctx *c, i64 lo, i64 hi)
{
    if (hi <= lo) return NPB_OK;
    npb_resolve_timers(c);   // a lazily stopped "k2_main" of an earlier IDW / LS launch must not land on top of this pass's
    cudaStream_t s = c->stream;
    GlsArgs a;
    a.esup_ptr = c->esup_ptr; a.esup = c->esup; a.fsup_ptr = c->fsup_ptr; a.fsup = c->fsup; a.esuf2 = c->esuf2;
    a.bpoint = c->bpoint; a.nflag = c->nflag; a.coords = c->coords; a.cent = c->centroids; a.fcent = c->fcent;
    a.fnormal = c->fnormal; a.perm = c->perm; a.diff_mag = c->diff_mag; a.wbuf = c->wbuf; a.rowcnt = c->rowcnt;
    a.neumann = c->neumann; a.wbase = c->wbase;
    i64 nloc = hi - lo;
    if (!c->node_list) {
        // [0, n): work list of the current class; [n, 2n): overflow list; then n bytes of classes
        NPB_TRY(npb_alloc(c, (void **)&c->node_list, sizeof(int32_t) * 2 * (size_t)c->n_points + (size_t)c->n_points));
    }
    int32_t *overflow = c->node_list + c->n_points;
    uint8_t *cls = (uint8_t *)(c->node_list + 2 * c->n_points);
    int *n_overflow = c->counters + 40;
    NPB_CUDA(cudaMemsetAsync(n_overflow, 0, sizeof(int), s));
    const char *force = getenv("NPB_FORCE_GLS_DENSE");   // tests: exercise the dense fallback kernel
    // 2-D meshes: every star is a small, nearly consistent system (weights up to +-150, residual << 1): all of them
    // take the dense kernel, which forms the residual through the reflectors (see k2_gls_dense.cu)
    const int force_dense = ((force && force[0] == '1') || c->dim == 2) ? 1 : 0;
    int *sig = c->counters + 70;   // [2 * MF_NCLASS]: min / max star signature per class
    NPB_CUDA(cudaMemsetAsync(sig, 0x7f, sizeof(int) * MF_NCLASS, s));
    NPB_CUDA(cudaMemsetAsync(sig + MF_NCLASS, 0, sizeof(int) * MF_NCLASS, s));
    k_gls_classify<<<npb_blocks(nloc, 256), 256, 0, s>>>(a, lo, hi, cls, force_dense, sig);
    NPB_LAUNCH(c);
    k_gls_publish_sig<<<1, 32, 0, s>>>(sig, c->d_small + 44);
    NPB_LAUNCH(c);
    // test switch, read once per pass (the tests flip it between calls of one process)
    const char *noleaf = getenv("NPB_GLS_NO_LEAF");   // every front through the general loop
    const int mf_flags = (noleaf && noleaf[0] == '1') ? 1 : 0;
    float main_ms = 0.f;
    static const char *cls_names[MF_NCLASS] = {"", "k2_gls_c1", "k2_gls_c2", "k2_gls_c3", "k2_gls_c4", "k2_gls_c5", "k2_gls_c6", "k2_gls_c7", "k2_gls_dense"};
    for (int k = 1; k < MF_NCLASS; k++) c->timings.erase(cls_names[k]);
    int n_dense_direct = 0;
    // work lists of all classes at once: a stable partition of [lo, hi) by class (scan.cu), one host round trip
    int starts[MF_NCLASS + 1];
    NPB_TRY(npb_partition_classes(c, cls, lo, hi, c->node_list, starts));
    for (int k = 1; k < MF_NCLASS - 1; k++) {
        const int count = starts[k + 1] - starts[k];
        if (count == 0) continue;
        const int32_t *list = c->node_list + starts[k];
        int *counter = c->counters + 20 + k;
        NPB_CUDA(cudaMemsetAsync(counter, 0, sizeof(int), s));
        NpbTimer tk(c, cls_names[k]);
        int smem = (int)mf_smem_bytes(h_mf[k]);
        // resident warps per SM are bounded by shared memory; the launch bound follows it so that small
        // stars trade registers for residency (16: 128 registers, 12: 168)
        int per_sm = (int)((227 * 1024) / (smem + 1024));
        if (per_sm > 32) per_sm = 32;
        const int variant = per_sm >= 16 ? 16 : 12;
        const int vregs = variant == 16 ? 128 : 168;
        if (per_sm > 65536 / (32 * vregs)) per_sm = 65536 / (32 * vregs);
        int grid = c->sm_count * per_sm;
        if (grid > count) grid = count;
        NPB_TRY(npb_ensure(&c->gls_ws, &c->gls_ws_cap, sizeof(double) * (size_t)grid * h_mf[k].acap * 2));
        // Team launch (the warps of an SM in one CTA, loosely in step, so that they share instruction fetches): pays
        // when the stars of the class are all alike - every node then runs the same instruction stream (structured
        // tets: -9 %) - and costs when they differ (mixed mesh: +20 %), so it is taken for the 168-register classes
        // whose smallest and largest star signature coincide.  NPB_GLS_TEAM = "off" | "slack[,spins]" overrides (tests, A/B).
        const char *team = getenv("NPB_GLS_TEAM");
        const bool uniform_stars = c->h_small[44 + k] == c->h_small[44 + MF_NCLASS + k];
        bool team_on = variant == 12 && per_sm == 12 && uniform_stars && count >= 12 * 64;
        int slack = 1, spins = 16;
        if (team) {
            team_on = strcmp(team, "off") != 0 && per_sm >= 2 && per_sm <= 32;
            slack = atoi(team);
            const char *comma = strchr(team, ',');
            if (comma) spins = atoi(comma + 1);
        }
        if (team_on) {
            const int tsmem = 128 + per_sm * smem;
            grid = c->sm_count;
            if ((i64)grid * per_sm > count) grid = (count + per_sm - 1) / per_sm;
            NPB_TRY(npb_ensure(&c->gls_ws, &c->gls_ws_cap, sizeof(double) * (size_t)grid * per_sm * h_mf[k].acap * 2));
            if (variant == 16) {
                NPB_CUDA(cudaFuncSetAttribute(k_gls_mf_team<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, tsmem));
                k_gls_mf_team<16><<<grid, 32 * per_sm, tsmem, s>>>(a, list, count, counter, k, overflow, n_overflow,
                                                                  (double *)c->gls_ws, mf_flags, smem, slack, spins);
            } else {
                NPB_CUDA(cudaFuncSetAttribute(k_gls_mf_team<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, tsmem));
                k_gls_mf_team<12><<<grid, 32 * per_sm, tsmem, s>>>(a, list, count, counter, k, overflow, n_overflow,
                                                                  (double *)c->gls_ws, mf_flags, smem, slack, spins);
            }
        } else if (variant == 16) {
            NPB_CUDA(cudaFuncSetAttribute(k_gls_mf<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k_gls_mf<16><<<grid, 32, smem, s>>>(a, list, count, counter, k, overflow, n_overflow, (double *)c->gls_ws, mf_flags);
        } else {
            NPB_CUDA(cudaFuncSetAttribute(k_gls_mf<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k_gls_mf<12><<<grid, 32, smem, s>>>(a, list, count, counter, k, overflow, n_overflow, (double *)c->gls_ws, mf_flags);
        }
        NPB_LAUNCH(c);
        NPB_CUDA(cudaGetLastError());
        tk.stop();
        if (c->timings[cls_names[k]] > main_ms) main_ms = c->timings[cls_names[k]];
    }
    // dense fallback: stars classified as too large, then whatever overflowed at run time
    {
        NpbTimer tk(c, cls_names[MF_NCLASS - 1]);
        n_dense_direct = starts[MF_NCLASS] - starts[MF_NCLASS - 1];
        NPB_TRY(npb_gls_dense(c, a, c->node_list + starts[MF_NCLASS - 1], n_dense_direct));
        int h_over = 0;
        NPB_TRY(npb_read_int(c, n_overflow, &h_over));
        NPB_TRY(npb_gls_dense(c, a, overflow, h_over));
        tk.stop();
        c->timings["gls_dense_nodes"] = (float)(n_dense_direct + h_over);
        if (c->timings[cls_names[MF_NCLASS - 1]] > main_ms && (n_dense_direct + h_over) > 0) main_ms = c->timings[cls_names[MF_NCLASS - 1]];
    }
    c->timings["k2_main"] = main_ms;
    return NPB_OK;
}
