// NCCL inside the library (include/tecount.h: tec_comm_*, tec_bulk_allreduce, tec_sc_exchange, tec_sc_allgather_triples).
//
// Where the path has an exchange step (SURVEY.md 8e) the library issues the collective itself, on its own stream, over
// its own device buffers: the bulk counter block (one all-reduce of n_ensg + 8 counters), the single-cell survivors
// (all-to-all by owner rank = grouped send / receive of the packed records), the small all-reduces of tec_sc_finalize
// (bundle boundaries, per-cell counts, presence table, statistics) and the final triples (all-gather + merge).  No host
// round trip per collective and no Python in the control plane; the caller only carries the 128-byte unique id
// from rank 0 to the other ranks once (any transport: te_counter_b200/dist.py uses torch.distributed).
//
// NCCL is bound at run time (dlopen of libnccl.so.2: the copy the process already has -- PyTorch's -- or the system's),
// so libtecount.so has no link-time dependency on it and single-GPU users never load it.
#pragma once
#include "context.cuh"
#include <dlfcn.h>
#include <nccl.h>

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string why;

    bool load() {
        if (handle) return true;
        // TEC_NCCL_LIB (a path) first, then the copy this process already mapped (PyTorch's), then the search path.  The
        // order matters in a process that imports torch later: the loader reuses a mapped libnccl.so.2 by name, and
        // an older system copy would leave libtorch_cuda.so with unresolved symbols.
        const char* env = getenv("TEC_NCCL_LIB");
        if (env && *env) handle = dlopen(env, RTLD_NOW | RTLD_LOCAL);
        if (!handle) handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL | RTLD_NOLOAD);
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (handle) break;
            handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
        }
        if (!handle) { why = std::string("libnccl.so.2 not found: ") + (dlerror() ? dlerror() : ""); return false; }
#define TEC_NCCL_SYM(field, name) \
        *(void**)(&field) = dlsym(handle, name); \
        if (!field) { why = std::string("NCCL symbol missing: ") + name; handle = nullptr; return false; }
        TEC_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
        TEC_NCCL_SYM(CommInitRank, "ncclCommInitRank")
        TEC_NCCL_SYM(CommDestroy, "ncclCommDestroy")
        TEC_NCCL_SYM(AllReduce, "ncclAllReduce")
        TEC_NCCL_SYM(AllGather, "ncclAllGather")
        TEC_NCCL_SYM(Send, "ncclSend")
        TEC_NCCL_SYM(Recv, "ncclRecv")
        TEC_NCCL_SYM(GroupStart, "ncclGroupStart")
        TEC_NCCL_SYM(GroupEnd, "ncclGroupEnd")
        TEC_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef TEC_NCCL_SYM
        return true;
    }
};
static NcclApi g_nccl;

#define TEC_NCCL(call)                                                                              \
    do {                                                                                            \
        ncclResult_t r_ = (call);                                                                   \
        if (r_ != ncclSuccess) {                                                                    \
            ctx->err = std::string(#call) + ": " + g_nccl.GetErrorString(r_);                       \
            return TEC_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

extern "C" int tec_comm_unique_id(tec_ctx* ctx, void* id, int32_t capacity) {
    if (!ctx) return TEC_ERR_ARG;
    if (!id || capacity < (int32_t)sizeof(ncclUniqueId)) TEC_FAIL(TEC_ERR_ARG, "tec_comm_unique_id: the buffer must hold TEC_COMM_ID_BYTES bytes");
    if (!g_nccl.load()) TEC_FAIL(TEC_ERR_UNSUPPORTED, "tec_comm_unique_id: " + g_nccl.why);
    ncclUniqueId u;
    TEC_NCCL(g_nccl.GetUniqueId(&u));
    memcpy(id, &u, sizeof(u));
    return TEC_OK;
}

extern "C" int tec_comm_destroy(tec_ctx* ctx) {
    if (!ctx) return TEC_ERR_ARG;
    if (ctx->comm) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        g_nccl.CommDestroy((ncclComm_t)ctx->comm);
    }
    ctx->comm = nullptr;
    ctx->comm_rank = 0;
    ctx->comm_world = 1;
    return TEC_OK;
}

extern "C" int tec_comm_init(tec_ctx* ctx, const void* id, int32_t rank, int32_t world) {
    if (!ctx) return TEC_ERR_ARG;
    if (!id || world < 1 || rank < 0 || rank >= world) TEC_FAIL(TEC_ERR_ARG, "tec_comm_init: bad arguments");
    if (!g_nccl.load()) TEC_FAIL(TEC_ERR_UNSUPPORTED, "tec_comm_init: " + g_nccl.why);
    tec_comm_destroy(ctx);
    TEC_CUDA(cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclComm_t c = nullptr;
    TEC_NCCL(g_nccl.CommInitRank(&c, world, u, rank));
    ctx->comm = c;
    ctx->comm_rank = rank;
    ctx->comm_world = world;
    return TEC_OK;
}

extern "C" int tec_comm_info(tec_ctx* ctx, int32_t* rank, int32_t* world) {
    if (!ctx) return TEC_ERR_ARG;
    if (rank) *rank = ctx->comm_rank;
    if (world) *world = ctx->comm ? ctx->comm_world : 1;
    return TEC_OK;
}

// all-reduce in place on the library's stream; dtype 0 u32, 1 u64, 2 i64; op 0 sum, 1 min, 2 max
static int comm_allreduce(tec_ctx* ctx, void* dev, int64_t count, int dtype, int op) {
    if (!ctx->comm || count <= 0) return TEC_OK;
    const ncclDataType_t dt = dtype == 0 ? ncclUint32 : dtype == 1 ? ncclUint64 : ncclInt64;
    const ncclRedOp_t ro = op == 0 ? ncclSum : op == 1 ? ncclMin : ncclMax;
    TEC_NCCL(g_nccl.AllReduce(dev, dev, (size_t)count, dt, ro, (ncclComm_t)ctx->comm, ctx->stream));
    return TEC_OK;
}

// Sum of every rank's bulk counter block (n_ensg counters + TEC_BULK_NSTATS statistics [+ row counters]), in place, ordered behind the
// pushes on the library's stream: tec_bulk_finish then returns the job's result on every rank.
extern "C" int tec_bulk_allreduce(tec_ctx* ctx) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->bulk_active) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_allreduce: tec_bulk_begin not called");
    if (ctx->bank_pending) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_allreduce: a paired-end range count waits for tec_bulk_keep_bank");
    if (ctx->name_held) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_allreduce: rows of a read-name range wait for tec_bulk_name_partition_dev");
    if (!ctx->comm) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_allreduce: tec_comm_init not called");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (int rc = name_flush(ctx)) return rc;
    return comm_allreduce(ctx, ctx->d_counts, (int64_t)ctx->bulk_words(), 1, 0);
}
