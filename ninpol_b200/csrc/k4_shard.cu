// k4_shard.cu — node-partitioned sharding across the GPUs of one box (kernel group K4).
//
// No reference counterpart (the reference is one process, SURVEY.md 2.2).  Every rank holds the whole
// mesh (K1 runs redundantly, cheaper than broadcasting it) and computes the CSR rows of one contiguous
// node range; the row blocks are then all-gathered over NCCL (NVLink 5 / NVSwitch) straight into their
// final positions: first the per-row counts and the neumann entries, then — once the scanned indptr
// gives every block its global offset — the indices and data blocks.  Variable-size all-gather is
// expressed as one grouped set of in-place ncclBroadcast calls, one per owner rank.
// NCCL is dlopen'ed so that single-GPU use does not need it.
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>
#include "common.cuh"

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi g_nccl;

static int load_nccl()
{
    if (g_nccl.handle) return NPB_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *n : names) {
        h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) {
        npb_set_error("cannot dlopen libnccl.so.2: %s", dlerror());
        return NPB_ERR_NCCL;
    }
#define SYM(field, name)                                                     \
    *(void **)(&g_nccl.field) = dlsym(h, name);                              \
    if (!g_nccl.field) {                                                     \
        npb_set_error("libnccl lacks symbol %s", name);                      \
        return NPB_ERR_NCCL;                                                 \
    }
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(Broadcast, "ncclBroadcast")
    SYM(AllReduce, "ncclAllReduce")
    SYM(Send, "ncclSend")
    SYM(Recv, "ncclRecv")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    g_nccl.handle = h;
    return NPB_OK;
}

#define NPB_NCCL(call)                                                                         \
    do {                                                                                       \
        ncclResult_t r__ = (call);                                                             \
        if (r__ != ncclSuccess) {                                                              \
            npb_set_error("NCCL error %s at %s:%d", g_nccl.GetErrorString(r__), __FILE__, __LINE__); \
            return NPB_ERR_NCCL;                                                               \
        }                                                                                      \
    } while (0)

extern "C" int npb_comm_unique_id(void *id_out)
{
    static_assert(sizeof(ncclUniqueId) == NPB_UNIQUE_ID_BYTES, "ncclUniqueId size");
    if (!id_out) {
        npb_set_error("npb_comm_unique_id: null output");
        return NPB_ERR_ARG;
    }
    NPB_TRY(load_nccl());
    ncclUniqueId id;
    NPB_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return NPB_OK;
}

extern "C" int npb_comm_init(npb_ctx *c, const void *id, int rank, int world)
{
    if (!c || !id || world < 1 || rank < 0 || rank >= world) {
        npb_set_error("npb_comm_init: bad arguments");
        return NPB_ERR_ARG;
    }
    NPB_CUDA(cudaSetDevice(c->device));
    if (world == 1) {
        c->rank = 0;
        c->world = 1;
        return NPB_OK;
    }
    NPB_TRY(load_nccl());
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    ncclComm_t comm;
    NPB_NCCL(g_nccl.CommInitRank(&comm, world, uid, rank));
    c->comm = comm;
    c->nccl = &g_nccl;
    c->rank = rank;
    c->world = world;
    return NPB_OK;
}

int npb_comm_destroy(npb_ctx *c)
{
    if (c->comm && c->nccl) c->nccl->CommDestroy((ncclComm_t)c->comm);
    c->comm = nullptr;
    return NPB_OK;
}

extern "C" int npb_comm_barrier(npb_ctx *c)
{
    if (!c) return NPB_ERR_ARG;
    if (c->world == 1) return NPB_OK;
    NPB_CUDA(cudaSetDevice(c->device));
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    int *buf = c->counters + 48;   // 16 ints: one per rank (world <= 16 on one box)
    if (c->world > 16) {
        npb_set_error("npb_comm_barrier: world > 16 not supported");
        return NPB_ERR_ARG;
    }
    NPB_NCCL(api->GroupStart());
    for (int r = 0; r < c->world; r++) NPB_NCCL(api->Broadcast(buf + r, buf + r, 1, ncclInt32, r, comm, c->stream));
    NPB_NCCL(api->GroupEnd());
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    return NPB_OK;
}

// all-gather of rowcnt[lo_r:hi_r] and neumann[lo_r:hi_r] from their owners
int npb_k4_gather_counts(npb_ctx *c)
{
    if (c->world == 1) return NPB_OK;
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    NPB_NCCL(api->GroupStart());
    for (int r = 0; r < c->world; r++) {
        i64 b = c->bounds[r], n = c->bounds[r + 1] - b;
        if (n <= 0) continue;
        NPB_NCCL(api->Broadcast(c->rowcnt + b, c->rowcnt + b, (size_t)n, ncclInt32, r, comm, c->stream));
        NPB_NCCL(api->Broadcast(c->neumann + b, c->neumann + b, (size_t)n, ncclFloat64, r, comm, c->stream));
    }
    NPB_NCCL(api->GroupEnd());
    return NPB_OK;
}

// all-gather of the indices / data row blocks; nnz offsets of the blocks come from the scanned indptr
int npb_k4_gather_blocks(npb_ctx *c)
{
    if (c->world == 1) return NPB_OK;
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    std::vector<int32_t> off(c->world + 1);
    for (int r = 0; r <= c->world; r++)
        NPB_CUDA(cudaMemcpyAsync(&off[r], c->indptr + c->bounds[r], sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    NPB_NCCL(api->GroupStart());
    if (c->gather_mode == NPB_GATHER_ROOT) {
        // gather-v to rank 0: the other ranks keep (and later hand out) their own row block only
        for (int r = 1; r < c->world; r++) {
            i64 b = off[r], n = (i64)off[r + 1] - off[r];
            if (n <= 0) continue;
            if (c->rank == 0) {
                NPB_NCCL(api->Recv(c->indices + b, (size_t)n, ncclInt32, r, comm, c->stream));
                NPB_NCCL(api->Recv(c->data + b, (size_t)n, ncclFloat64, r, comm, c->stream));
            } else if (c->rank == r) {
                NPB_NCCL(api->Send(c->indices + b, (size_t)n, ncclInt32, 0, comm, c->stream));
                NPB_NCCL(api->Send(c->data + b, (size_t)n, ncclFloat64, 0, comm, c->stream));
            }
        }
    } else {
        // all-gather-v as one group of point-to-point transfers: my block to every peer, every peer's block to its
        // final position here.  Through NVSwitch all 2 (world - 1) transfers of a rank run at once; the grouped
        // in-place ncclBroadcasts used before serialise per root (measured 272 GB/s per rank at 8 GPUs).
        const i64 mb = off[c->rank], mn = (i64)off[c->rank + 1] - off[c->rank];
        for (int r = 0; r < c->world; r++) {
            if (r == c->rank) continue;
            i64 b = off[r], n = (i64)off[r + 1] - off[r];
            if (mn > 0) {
                NPB_NCCL(api->Send(c->indices + mb, (size_t)mn, ncclInt32, r, comm, c->stream));
                NPB_NCCL(api->Send(c->data + mb, (size_t)mn, ncclFloat64, r, comm, c->stream));
            }
            if (n > 0) {
                NPB_NCCL(api->Recv(c->indices + b, (size_t)n, ncclInt32, r, comm, c->stream));
                NPB_NCCL(api->Recv(c->data + b, (size_t)n, ncclFloat64, r, comm, c->stream));
            }
        }
    }
    NPB_NCCL(api->GroupEnd());
    return NPB_OK;
}

// all-gather of the row blocks of a [n_points, n_cols] float64 array (npb_apply's result): rank r owns the rows
// [bounds[r], bounds[r + 1]).  One group of ncclSend / ncclRecv, as in npb_k4_gather_blocks, whatever the gather mode:
// the result is n_points * n_cols doubles, small next to the CSR.
int npb_k4_gather_rows(npb_ctx *c, double *rows, i64 n_cols)
{
    if (c->world == 1) return NPB_OK;
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    const i64 mb = c->bounds[c->rank] * n_cols, mn = (c->bounds[c->rank + 1] - c->bounds[c->rank]) * n_cols;
    NPB_NCCL(api->GroupStart());
    for (int r = 0; r < c->world; r++) {
        if (r == c->rank) continue;
        const i64 b = c->bounds[r] * n_cols, n = (c->bounds[r + 1] - c->bounds[r]) * n_cols;
        if (mn > 0) NPB_NCCL(api->Send(rows + mb, (size_t)mn, ncclFloat64, r, comm, c->stream));
        if (n > 0) NPB_NCCL(api->Recv(rows + b, (size_t)n, ncclFloat64, r, comm, c->stream));
    }
    NPB_NCCL(api->GroupEnd());
    return NPB_OK;
}

// Every rank contributes one int; *any = 1 when some rank's is non-zero: ONE 4-byte ncclAllReduce (sum) on the
// compute stream - the only exchange of a planned IDW / LS step - whose result comes back through the mapped block.
__global__ void k_fold_flags(int *dst, const int *bad2, int host_flag) { *dst = (bad2[0] != 0 || bad2[1] != 0 || host_flag != 0) ? 1 : 0; }

// d_bad2: two device counters of this rank (exact zeros, row-length mismatches); host_flag: a condition the host
// already knows.  *any = 1 when any rank has any of them set.
int npb_k4_share_flags(npb_ctx *c, const int *d_bad2, int host_flag, int *any)
{
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    int *buf = c->counters + 47;
    k_fold_flags<<<1, 1, 0, c->stream>>>(buf, d_bad2, host_flag);
    NPB_LAUNCH(c);
    NPB_NCCL(api->AllReduce(buf, buf, 1, ncclInt32, ncclSum, comm, c->stream));
    k_copy_int<<<1, 1, 0, c->stream>>>(c->d_small + 16, buf);
    NPB_LAUNCH(c);
    NPB_CUDA(cudaStreamSynchronize(c->stream));
    *any = c->h_small[16] != 0 ? 1 : 0;
    return NPB_OK;
}

// wrapping 64-bit sum over the ranks, in place, on the compute stream (the flag-slice checksums of capi.cu)
int npb_k4_allreduce_u64(npb_ctx *c, unsigned long long *d_value)
{
    if (c->world == 1) return NPB_OK;
    NcclApi *api = c->nccl;
    NPB_NCCL(api->AllReduce(d_value, d_value, 1, ncclUint64, ncclSum, (ncclComm_t)c->comm, c->stream));
    return NPB_OK;
}

// One chunk step of the pipelined all-gather-v: rank r owns nodes [node_lo[r], node_hi[r]) = CSR entries
// [nz_lo[r], nz_hi[r]); every rank receives every block at its final position (one group of ncclSend / ncclRecv on `st`).
int npb_k4_bcast_chunk(npb_ctx *c, cudaStream_t st, const std::vector<i64> &node_lo, const std::vector<i64> &node_hi,
                       const std::vector<i64> &nz_lo, const std::vector<i64> &nz_hi, bool with_neumann)
{
    if (c->world == 1) return NPB_OK;
    NcclApi *api = c->nccl;
    ncclComm_t comm = (ncclComm_t)c->comm;
    NPB_NCCL(api->GroupStart());
    const int me = c->rank;
    const i64 my_rows = node_hi[me] - node_lo[me], my_nk = nz_hi[me] - nz_lo[me];
    for (int r = 0; r < c->world; r++) {
        if (r == me) continue;
        const i64 rows = node_hi[r] - node_lo[r], nk = nz_hi[r] - nz_lo[r];
        if (with_neumann && my_rows > 0) NPB_NCCL(api->Send(c->neumann + node_lo[me], (size_t)my_rows, ncclFloat64, r, comm, st));
        if (my_nk > 0) {
            NPB_NCCL(api->Send(c->indices + nz_lo[me], (size_t)my_nk, ncclInt32, r, comm, st));
            NPB_NCCL(api->Send(c->data + nz_lo[me], (size_t)my_nk, ncclFloat64, r, comm, st));
        }
        if (with_neumann && rows > 0) NPB_NCCL(api->Recv(c->neumann + node_lo[r], (size_t)rows, ncclFloat64, r, comm, st));
        if (nk > 0) {
            NPB_NCCL(api->Recv(c->indices + nz_lo[r], (size_t)nk, ncclInt32, r, comm, st));
            NPB_NCCL(api->Recv(c->data + nz_lo[r], (size_t)nk, ncclFloat64, r, comm, st));
        }
    }
    NPB_NCCL(api->GroupEnd());
    return NPB_OK;
}
