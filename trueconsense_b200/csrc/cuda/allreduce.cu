// allreduce.cu — the one collective of the path: summing per-rank count tables when an
// ultra-deep single sample is sharded by read range (SURVEY.md §8e).  Counts are additive int32,
// so the result is bit-identical to the single-GPU table.  The table is ~1 MB (L = 29,903) to
// ~6 MB (L = 197 k): latency-bound on NVLink/NVSwitch, one ncclAllReduce.
//
// NCCL is resolved at run time from the library the host layer created the communicator with
// (TC_NCCL_LIB, default "libnccl.so.2"), so libtcb200.so itself has no link-time NCCL dependency.
#include <dlfcn.h>
#include <stdlib.h>

#include "tc_common.cuh"

typedef int (*nccl_allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*nccl_errstr_fn)(int);

static nccl_allreduce_fn g_allreduce = nullptr;
static nccl_errstr_fn g_errstr = nullptr;

static int nccl_resolve(tc_ctx* ctx) {
    if (!g_allreduce) {
        const char* path = getenv("TC_NCCL_LIB");
        void* h = dlopen(path && *path ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return tc_fail(ctx, TC_ERR_ARG, "cannot load NCCL (%s): %s", path ? path : "libnccl.so.2", dlerror());
        g_allreduce = (nccl_allreduce_fn)dlsym(h, "ncclAllReduce");
        g_errstr = (nccl_errstr_fn)dlsym(h, "ncclGetErrorString");
        if (!g_allreduce) return tc_fail(ctx, TC_ERR_ARG, "ncclAllReduce not found in the NCCL library");
    }
    return TC_OK;
}

TC_API int tc_allreduce_counts(tc_ctx_t* ctx, int32_t* counts_dev, int64_t n_elems, void* comm, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!counts_dev || n_elems < 0 || !comm) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (!tc_is_device_ptr(counts_dev)) return tc_fail(ctx, TC_ERR_ARG, "tc_allreduce_counts needs a device pointer");
    TC_CUDA(cudaSetDevice(ctx->device));
    int rc = nccl_resolve(ctx);
    if (rc) return rc;
    const int nccl_int32 = 2, nccl_sum = 0;
    int r = g_allreduce(counts_dev, counts_dev, (size_t)n_elems, nccl_int32, nccl_sum, comm, (cudaStream_t)stream);
    if (r != 0) return tc_fail(ctx, TC_ERR_CUDA, "ncclAllReduce failed: %s", g_errstr ? g_errstr(r) : "?");
    return TC_OK;
}

// ---- the shard's pileup and the sum in one enqueue -------------------------------------------------------------------
// The pad row of the table (row 7, all zero by contract) carries one word of the collective: "this rank's status block
// holds an error".  Summed with the counts, every rank learns whether ANY shard needs the slow road, without a second
// collective and without a synchronisation between the pileup and the sum.
__global__ void rr_flag_kernel(const tc_status* st, int32_t* pad0) { *pad0 = st->err != 0 ? 1 : 0; }

struct rr_host { tc_status st; int32_t any_err; };

// one shard pass in flight: what its finish needs, its pinned result block, and the chain's graph (keyed like a sample's)
struct tc_rr_slot {
    int state;                      // 0 free, 1 enqueued
    rr_host* host;                  // pinned
    cudaEvent_t done;
    tc_reads_t reads; int32_t ref_len; tc_pileup_params_t p; int32_t* counts; void* comm; void* stream;
    tc_pileup_pending pend;         // of the run that was enqueued eagerly or captured: a replay is that run again
    tc_graph_cache graph;
};

static int rr_slots(tc_ctx* ctx) {
    if (ctx->rr) return TC_OK;
    tc_rr_slot* sl = (tc_rr_slot*)calloc(2, sizeof(tc_rr_slot));
    if (!sl) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
    for (int i = 0; i < 2; ++i) {
        cudaError_t e = cudaMallocHost((void**)&sl[i].host, 256);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl[i].done, cudaEventDisableTiming);
        if (e != cudaSuccess) { free(sl); return tc_cuda_fail(ctx, e, "shard pass slot"); }
    }
    ctx->rr = sl;
    return TC_OK;
}

void tc_rr_slots_free(tc_ctx* ctx) {
    if (!ctx->rr) return;
    for (int i = 0; i < 2; ++i) {
        if (ctx->rr[i].host) cudaFreeHost(ctx->rr[i].host);
        if (ctx->rr[i].done) cudaEventDestroy(ctx->rr[i].done);
        tc_graph_destroy(ctx->rr[i].graph);
    }
    free(ctx->rr);
    ctx->rr = nullptr;
}

static int rr_chain(tc_ctx* ctx, tc_rr_slot& sl, cudaStream_t s) {
    const int L = sl.ref_len;
    int rc = tc_pileup_enqueue(ctx, &sl.reads, L, &sl.p, sl.counts, s, &sl.pend);
    if (rc) return rc;
    int32_t* pad0 = sl.counts + (size_t)(TC_NROWS - 1) * L;
    rr_flag_kernel<<<1, 1, 0, s>>>(sl.pend.d_status, pad0);
    TC_LAUNCH_CHECK();
    const int nccl_int32 = 2, nccl_sum = 0;
    // rows 0..6 and the flag word: the rest of the pad row stays out of the collective
    const int r = g_allreduce(sl.counts, sl.counts, (size_t)(TC_NROWS - 1) * L + 1, nccl_int32, nccl_sum, sl.comm, s);
    if (r != 0) return tc_fail(ctx, TC_ERR_CUDA, "ncclAllReduce failed: %s", g_errstr ? g_errstr(r) : "?");
    ctx->launches++;
    TC_D2H(&sl.host->st, sl.pend.d_status, sizeof(tc_status), s);
    TC_D2H(&sl.host->any_err, pad0, sizeof(int32_t), s);
    TC_CUDA(cudaMemsetAsync(pad0, 0, sizeof(int32_t), s));
    return TC_OK;
}

TC_API int tc_pileup_counts_allreduce_enqueue(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p,
                                              int32_t* counts, void* comm, void* stream, int32_t* ticket) {
    if (!ctx) return TC_ERR_ARG;
    if (!reads || !p || !counts || !comm || !ticket || ref_len <= 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (!tc_is_device_ptr(counts)) return tc_fail(ctx, TC_ERR_ARG, "tc_pileup_counts_allreduce needs a device pointer for the table");
    static_assert(sizeof(rr_host) <= 256, "pinned result block");
    TC_CUDA(cudaSetDevice(ctx->device));
    int rc = nccl_resolve(ctx);
    if (rc) return rc;
    rc = rr_slots(ctx);
    if (rc) return rc;
    const int slot = ctx->rr_next;
    tc_rr_slot& sl = ctx->rr[slot];
    if (sl.state != 0) return tc_fail(ctx, TC_ERR_ARG, "two shard passes are in flight on this context already: finish one first");
    cudaStream_t s = (cudaStream_t)stream;
    sl.reads = *reads; sl.ref_len = ref_len; sl.p = *p; sl.counts = counts; sl.comm = comm; sl.stream = stream;

    unsigned char key[256];
    int kn = 0;
    auto put = [&](const void* q, size_t bytes) { memcpy(key + kn, q, bytes); kn += (int)bytes; };
    put(reads, sizeof(*reads)); put(&ref_len, 4); put(p, sizeof(*p)); put(&counts, sizeof(counts)); put(&comm, sizeof(comm));
    put(&ctx->buf_epoch, 8); put(&ctx->timing, 4);
    static_assert(sizeof(tc_reads_t) + 4 + sizeof(tc_pileup_params_t) + 16 + 12 <= 256, "shard key");
    rc = tc_graph_run(ctx, sl.graph, key, kn, tc_reads_all_device(reads), [&](cudaStream_t cs) { return rr_chain(ctx, sl, cs); }, s);
    if (rc) return rc;
    TC_CUDA(cudaEventRecord(sl.done, s));
    sl.state = 1;
    ctx->rr_next = slot ^ 1;
    *ticket = slot;
    return TC_OK;
}

TC_API int tc_pileup_counts_allreduce_finish(tc_ctx_t* ctx, int32_t ticket) {
    if (!ctx) return TC_ERR_ARG;
    if (ticket < 0 || ticket > 1 || !ctx->rr || ctx->rr[ticket].state == 0) return tc_fail(ctx, TC_ERR_ARG, "bad ticket");
    TC_CUDA(cudaSetDevice(ctx->device));
    tc_rr_slot& sl = ctx->rr[ticket];
    sl.state = 0;
    TC_CUDA(cudaEventSynchronize(sl.done));                 // the one synchronisation of the pass
    rr_host h;
    memcpy(&h, sl.host, sizeof(h));
    cudaStream_t s = (cudaStream_t)sl.stream;
    const int L = sl.ref_len;
    if (h.any_err != 0) {
        // some rank's shard did not go through: every rank takes the separate calls (which handle the kernel variants) and
        // makes the same collective call whatever its own outcome, so nobody waits for a rank that failed
        sl.graph.key_len = 0;
        const int prc = tc_pileup_counts(ctx, &sl.reads, L, &sl.p, sl.counts, sl.stream);
        if (prc) TC_CUDA(cudaMemsetAsync(sl.counts, 0, sizeof(int32_t) * TC_NROWS * (size_t)L, s));
        char keep[sizeof(ctx->err)];
        if (prc) memcpy(keep, ctx->err, sizeof(keep));
        const int arc = tc_allreduce_counts(ctx, sl.counts, (int64_t)TC_NROWS * L, sl.comm, sl.stream);
        if (prc) { memcpy(ctx->err, keep, sizeof(keep)); return prc; }
        return arc;
    }
    return tc_pileup_settle(ctx, h.st, sl.pend, &sl.reads, L, &sl.p, sl.counts, s, nullptr);
}

TC_API int tc_pileup_counts_allreduce(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p,
                                      int32_t* counts, void* comm, void* stream) {
    int32_t ticket = -1;
    const int rc = tc_pileup_counts_allreduce_enqueue(ctx, reads, ref_len, p, counts, comm, stream, &ticket);
    if (rc) return rc;
    return tc_pileup_counts_allreduce_finish(ctx, ticket);
}
