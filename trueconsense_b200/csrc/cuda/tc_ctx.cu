// tc_ctx.cu — context lifecycle, error text, grow-only device buffers, host<->device staging.
#include <stdarg.h>
#include <stdlib.h>

#include <thread>

#include "tc_common.cuh"

static char g_create_err[512] = "";
void tc_sample_slots_free(tc_ctx* ctx);     // sample.cu
void tc_rr_slots_free(tc_ctx* ctx);         // allreduce.cu

int tc_fail(tc_ctx* ctx, int code, const char* fmt, ...) {
    char* dst = ctx ? ctx->err : g_create_err;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}

int tc_cuda_fail(tc_ctx* ctx, cudaError_t e, const char* what) {
    return tc_fail(ctx, TC_ERR_CUDA, "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
}

void* tc_dev_buf(tc_ctx* ctx, int slot, size_t bytes) {
    tc_buf* b = ctx->bank ? &ctx->bank[slot] : &ctx->bufs[slot];
    if (bytes == 0) bytes = 16;
    if (b->cap >= bytes) return b->p;
    if (b->p) { cudaFree(b->p); b->p = NULL; b->cap = 0; }
    size_t cap = bytes + bytes / 8 + 256;       // a little slack so slowly growing inputs do not realloc every call
    cap = (cap + 255) & ~(size_t)255;
    void* p = NULL;
    cudaError_t e = cudaMalloc(&p, cap);
    if (e != cudaSuccess) {
        tc_fail(ctx, TC_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(e));
        cudaGetLastError();
        return NULL;
    }
    b->p = p; b->cap = cap;
    ctx->buf_epoch++;
    return p;
}

bool tc_is_device_ptr(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Large uploads from PAGEABLE host memory (numpy arrays, a mapped BAM file).  cudaMemcpyAsync stages such a copy through
// the driver's own pinned buffer on the calling thread: ~11 GB/s measured for a 92 MB file, a fifth of the link.  Here the
// source is cut into 8 MB chunks; four host threads copy a wave of four chunks into pinned ring slots while the previous
// wave's slots are on their way over PCIe (two sets of four slots), so the link sees pinned memory only and the host copy
// runs at several cores' memory bandwidth.  Returns when every chunk has been ENQUEUED: the source may be released then,
// exactly as with the plain call.
constexpr size_t TC_RING_CHUNK = 8u << 20;
constexpr int TC_RING_SLOTS = 8;
constexpr size_t TC_RING_MIN = 24u << 20;

static bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

static int stage_pageable(tc_ctx* ctx, void* d, const void* p, size_t bytes, cudaStream_t s) {
    if (!ctx->ring) {
        TC_CUDA(cudaMallocHost(&ctx->ring, TC_RING_CHUNK * TC_RING_SLOTS));
        for (int i = 0; i < TC_RING_SLOTS; ++i) TC_CUDA(cudaEventCreateWithFlags(&ctx->ring_ev[i], cudaEventDisableTiming));
    }
    const size_t n_chunks = (bytes + TC_RING_CHUNK - 1) / TC_RING_CHUNK;
    const int wave = TC_RING_SLOTS / 2;
    for (size_t c0 = 0, w = 0; c0 < n_chunks; c0 += wave, ++w) {
        const int n = (int)((n_chunks - c0) < (size_t)wave ? (n_chunks - c0) : (size_t)wave);
        const int base = (int)(w & 1) * wave;
        std::thread th[TC_RING_SLOTS / 2];
        for (int k = 0; k < n; ++k) {
            TC_CUDA(cudaEventSynchronize(ctx->ring_ev[base + k]));          // the copy that used this slot two waves ago
            const size_t off = (c0 + k) * TC_RING_CHUNK;
            const size_t len = bytes - off < TC_RING_CHUNK ? bytes - off : TC_RING_CHUNK;
            char* slot = (char*)ctx->ring + (size_t)(base + k) * TC_RING_CHUNK;
            const char* src = (const char*)p + off;
            if (k + 1 < n) th[k] = std::thread([=] { memcpy(slot, src, len); });
            else memcpy(slot, src, len);                                     // the calling thread takes the last one
        }
        for (int k = 0; k + 1 < n; ++k) th[k].join();
        for (int k = 0; k < n; ++k) {
            const size_t off = (c0 + k) * TC_RING_CHUNK;
            const size_t len = bytes - off < TC_RING_CHUNK ? bytes - off : TC_RING_CHUNK;
            TC_CUDA(cudaMemcpyAsync((char*)d + off, (char*)ctx->ring + (size_t)(base + k) * TC_RING_CHUNK, len, cudaMemcpyHostToDevice, s));
            TC_CUDA(cudaEventRecord(ctx->ring_ev[base + k], s));
        }
    }
    return TC_OK;
}

// host -> device into a caller-chosen place (part of a larger buffer): the ring for large pageable sources, a plain async copy otherwise
int tc_h2d(tc_ctx* ctx, void* d, const void* p, size_t bytes, cudaStream_t s) {
    if (!bytes) return TC_OK;
    if (bytes >= TC_RING_MIN && is_pageable(p)) {
        const int rc = stage_pageable(ctx, d, p, bytes, s);
        if (rc) return rc;
    } else {
        TC_CUDA(cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, s));
    }
    ctx->h2d_bytes += (int64_t)bytes;
    return TC_OK;
}

const void* tc_stage_in(tc_ctx* ctx, int slot, const void* p, size_t bytes, cudaStream_t s, int* rc) {
    *rc = TC_OK;
    if (!p) return NULL;
    if (tc_is_device_ptr(p)) return p;
    void* d = tc_dev_buf(ctx, slot, bytes);
    if (!d) { *rc = TC_ERR_NOMEM; return NULL; }
    if (bytes) {
        if (bytes >= TC_RING_MIN && is_pageable(p)) {
            *rc = stage_pageable(ctx, d, p, bytes, s);
            if (*rc) return NULL;
        } else {
            cudaError_t e = cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) { *rc = tc_cuda_fail(ctx, e, "cudaMemcpyAsync H2D"); return NULL; }
        }
        ctx->h2d_bytes += (int64_t)bytes;
    }
    return d;
}

// 16-bit (len << 4 | op) entries to the 32-bit ones the kernels read: 8 per thread and step (the buffers are 16-byte aligned
// and padded by tc_dev_buf)
__global__ void widen_cigar_kernel(const uint16_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n) {
    const int64_t n8 = n / 8;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 v = reinterpret_cast<const uint4*>(in)[i];
        reinterpret_cast<uint4*>(out)[2 * i] = make_uint4(v.x & 0xffffu, v.x >> 16, v.y & 0xffffu, v.y >> 16);
        reinterpret_cast<uint4*>(out)[2 * i + 1] = make_uint4(v.z & 0xffffu, v.z >> 16, v.w & 0xffffu, v.w >> 16);
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(n - 8 * n8)) out[8 * n8 + threadIdx.x] = in[8 * n8 + threadIdx.x];
}

// 2-bit SEQ transport -> the 4-bit one-hot words the kernels read.  Base j of a word sits in nibble (j even: high, odd: low) of
// byte j / 2, as in BAM: one byte of seq2 (4 bases) becomes two bytes of seq4 through a 256-entry table.  Flat over the words
// (four per thread: one 8-byte load, one 16-byte store); the zero padding behind every read's last base is a second, tiny
// kernel over the reads.  (One warp per read with the padding folded in measured 0.5 ms for 100 M words: short rows of 50
// words keep neither the lanes nor the memory pipe busy.)
__global__ void __launch_bounds__(256) widen_seq_kernel(const uint16_t* __restrict__ seq2, int64_t n_words, uint32_t* __restrict__ seq4) {
    __shared__ uint16_t lut[256];
    {
        const uint32_t h = threadIdx.x;
        const uint32_t c0 = h & 3u, c1 = (h >> 2) & 3u, c2 = (h >> 4) & 3u, c3 = (h >> 6) & 3u;
        lut[h] = (uint16_t)((((1u << c0) << 4) | (1u << c1)) | ((((1u << c2) << 4) | (1u << c3)) << 8));
    }
    __syncthreads();
    const int64_t n4 = n_words / 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const uint2 v = reinterpret_cast<const uint2*>(seq2)[i];
        uint4 o;
        o.x = (uint32_t)lut[v.x & 0xffu] | ((uint32_t)lut[(v.x >> 8) & 0xffu] << 16);
        o.y = (uint32_t)lut[(v.x >> 16) & 0xffu] | ((uint32_t)lut[v.x >> 24] << 16);
        o.z = (uint32_t)lut[v.y & 0xffu] | ((uint32_t)lut[(v.y >> 8) & 0xffu] << 16);
        o.w = (uint32_t)lut[(v.y >> 16) & 0xffu] | ((uint32_t)lut[v.y >> 24] << 16);
        reinterpret_cast<uint4*>(seq4)[i] = o;
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(n_words - 4 * n4)) {
        const uint32_t h = seq2[4 * n4 + threadIdx.x];
        seq4[4 * n4 + threadIdx.x] = (uint32_t)lut[h & 0xffu] | ((uint32_t)lut[h >> 8] << 16);
    }
}
__global__ void pad_seq_kernel(const uint32_t* __restrict__ seq_off, const int32_t* __restrict__ l_seq, int64_t n_reads, uint32_t* __restrict__ seq4) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const uint32_t w0 = seq_off[r], w1 = seq_off[r + 1];
    if (w1 == w0) return;
    const int valid = l_seq[r] - 8 * (int)(w1 - 1 - w0);        // bases of the read's last word that exist
    if (valid >= 8) return;
    uint32_t keep = 0;
    for (int j = 0; j < valid; ++j) keep |= 0xfu << (8 * (j >> 1) + ((j & 1) ? 0 : 4));
    seq4[w1 - 1] &= keep;
}
__global__ void patch_seq_kernel(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ val, int64_t n, uint32_t* __restrict__ seq4) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) seq4[idx[k]] = val[k];
}

int tc_resolve_reads(tc_ctx* ctx, const tc_reads_t* in, dreads* out, int need, cudaStream_t s) {
    if (!in) return tc_fail(ctx, TC_ERR_ARG, "reads is NULL");
    if (in->n_reads < 0 || in->n_seq_words < 0 || in->n_cigar_ops < 0) return tc_fail(ctx, TC_ERR_ARG, "negative sizes in tc_reads_t");
    if (in->n_reads >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 reads in one batch; shard the input");
    int64_t n = in->n_reads;
    memset(out, 0, sizeof(*out));
    out->n = n;
    if (n == 0) return TC_OK;
    if (!in->pos || !in->flag || !in->l_seq || !in->seq_off || !in->cigar_off || (!in->cigar && !in->cigar16 && in->n_cigar_ops) ||
        (!in->seq4 && !in->seq2 && in->n_seq_words))
        return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t: a required array is NULL");
    int rc;
#define STAGE(field, slot, type, count)                                                              \
    out->field = (const type*)tc_stage_in(ctx, slot, in->field, sizeof(type) * (size_t)(count), s, &rc); \
    if (rc) return rc;
    STAGE(pos, SLOT_POS, int32_t, n)
    STAGE(flag, SLOT_FLAG, uint16_t, n)
    STAGE(l_seq, SLOT_LSEQ, int32_t, n)
    STAGE(seq_off, SLOT_SEQOFF, uint32_t, n + 1)
    STAGE(cigar_off, SLOT_CIGOFF, uint32_t, n + 1)
#define STAGE_OR_DEFER(field, slot, type, count, defer)                                               \
    if ((need & (defer)) && in->field && !tc_is_device_ptr(in->field)) {                                \
        out->field = (const type*)tc_dev_buf(ctx, slot, sizeof(type) * (size_t)(count));                \
        if (!out->field) return TC_ERR_NOMEM;                                                           \
    } else { STAGE(field, slot, type, count) }
    if (in->seq2 && in->n_seq_words && !tc_is_device_ptr(in->seq2) && (!in->seq4 || !tc_is_device_ptr(in->seq4)) &&
        !((need & DEFER_SEQ) && in->seq4)) {
        // compact transport: 2 bits per base over the link (+ the words that hold something else), widened behind it
        if (in->n_seq_exc < 0 || (in->n_seq_exc > 0 && (!in->seq_exc_idx || !in->seq_exc_val)))
            return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t: seq2 without its exception list");
        const uint16_t* s2 = (const uint16_t*)tc_stage_in(ctx, SLOT_SEQ2, in->seq2, sizeof(uint16_t) * (size_t)in->n_seq_words, s, &rc);
        if (rc) return rc;
        const uint32_t* ei = (const uint32_t*)tc_stage_in(ctx, SLOT_SEQ_EXC_IDX, in->seq_exc_idx, 4 * (size_t)in->n_seq_exc, s, &rc); if (rc) return rc;
        const uint32_t* ev = (const uint32_t*)tc_stage_in(ctx, SLOT_SEQ_EXC_VAL, in->seq_exc_val, 4 * (size_t)in->n_seq_exc, s, &rc); if (rc) return rc;
        uint32_t* s4 = (uint32_t*)tc_dev_buf(ctx, SLOT_SEQ4, sizeof(uint32_t) * (size_t)in->n_seq_words);
        if (!s4) return TC_ERR_NOMEM;
        widen_seq_kernel<<<ctx->sm_count * 8, 256, 0, s>>>(s2, in->n_seq_words, s4);
        TC_LAUNCH_CHECK();
        pad_seq_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(out->seq_off, out->l_seq, n, s4);
        TC_LAUNCH_CHECK();
        if (in->n_seq_exc > 0) {
            patch_seq_kernel<<<(unsigned)((in->n_seq_exc + 255) / 256), 256, 0, s>>>(ei, ev, in->n_seq_exc, s4);
            TC_LAUNCH_CHECK();
        }
        out->seq4 = s4;
    } else {
        if (!in->seq4 && in->n_seq_words) return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t: seq4 is NULL and seq2 is not a host array");
        STAGE_OR_DEFER(seq4, SLOT_SEQ4, uint32_t, in->n_seq_words, DEFER_SEQ)
    }
    if (in->cigar16 && in->n_cigar_ops && !tc_is_device_ptr(in->cigar16) && (!in->cigar || !tc_is_device_ptr(in->cigar)) &&
        !((need & DEFER_CIGAR) && in->cigar)) {
        // compact transport: 2 bytes per operation over the link, widened behind it
        const uint16_t* c16 = (const uint16_t*)tc_stage_in(ctx, SLOT_CIGAR16, in->cigar16, sizeof(uint16_t) * (size_t)in->n_cigar_ops, s, &rc);
        if (rc) return rc;
        uint32_t* c32 = (uint32_t*)tc_dev_buf(ctx, SLOT_CIGAR, sizeof(uint32_t) * (size_t)in->n_cigar_ops);
        if (!c32) return TC_ERR_NOMEM;
        const int64_t n8 = (in->n_cigar_ops + 7) / 8;
        const int grid = (int)((n8 + 255) / 256 < (int64_t)ctx->sm_count * 8 ? (n8 + 255) / 256 : (int64_t)ctx->sm_count * 8);
        widen_cigar_kernel<<<grid, 256, 0, s>>>(c16, c32, in->n_cigar_ops);
        TC_LAUNCH_CHECK();
        out->cigar = c32;
    } else {
        if (!in->cigar && in->n_cigar_ops) return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t: cigar is NULL and cigar16 is not a host array");
        STAGE_OR_DEFER(cigar, SLOT_CIGAR, uint32_t, in->n_cigar_ops, DEFER_CIGAR)
    }
    if (in->mapq) { STAGE(mapq, SLOT_MAPQ, uint8_t, n) }
    if (need & NEED_QUAL) {
        if (!in->qual && in->n_seq_words) return tc_fail(ctx, TC_ERR_ARG, "this pass applies a base-quality filter but reads->qual is NULL");
        STAGE_OR_DEFER(qual, SLOT_QUAL, uint8_t, 8 * in->n_seq_words, DEFER_QUAL)
    } else if (in->qual && tc_is_device_ptr(in->qual)) {
        out->qual = in->qual;
    }
    if ((need & NEED_MATE) && in->qname_hash && in->mpos && in->isize) {       // all three or none
        STAGE_OR_DEFER(qname_hash, SLOT_QHASH, uint64_t, n, DEFER_MATE)
        STAGE_OR_DEFER(mpos, SLOT_MPOS, int32_t, n, DEFER_MATE)
        STAGE_OR_DEFER(isize, SLOT_ISIZE, int32_t, n, DEFER_MATE)
    }
#undef STAGE_OR_DEFER
#undef STAGE
    return TC_OK;
}

// ---------------------------------------------------------------- C-ABI: lifecycle
TC_API int tc_abi_version(void) { return TC_ABI_VERSION; }

TC_API int tc_ctx_create(int device, tc_ctx_t** out) {
    if (!out) return tc_fail(NULL, TC_ERR_ARG, "out is NULL");
    *out = NULL;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return tc_fail(NULL, TC_ERR_NO_DEVICE, "no CUDA device available (%s); there is no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0) {
        e = cudaGetDevice(&device);
        if (e != cudaSuccess) return tc_cuda_fail(NULL, e, "cudaGetDevice");
    }
    if (device >= n) return tc_fail(NULL, TC_ERR_ARG, "device %d out of range (%d devices)", device, n);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return tc_cuda_fail(NULL, e, "cudaSetDevice");
    tc_ctx* ctx = (tc_ctx*)calloc(1, sizeof(tc_ctx));
    if (!ctx) return tc_fail(NULL, TC_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { free(ctx); return tc_cuda_fail(NULL, e, "cudaGetDeviceProperties"); }
    ctx->sm_count = prop.multiProcessorCount;
    if (prop.major < 10) {
        int rc = tc_fail(NULL, TC_ERR_NO_DEVICE, "device %d is sm_%d%d; this library holds sm_100a code only", device, prop.major, prop.minor);
        free(ctx);
        return rc;
    }
    e = cudaMallocHost(&ctx->host_status, 256);
    if (e != cudaSuccess) { free(ctx); return tc_cuda_fail(NULL, e, "cudaMallocHost"); }
    *out = ctx;
    return TC_OK;
}

TC_API int tc_ctx_destroy(tc_ctx_t* ctx) {
    if (!ctx) return TC_OK;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < SLOT_COUNT; ++i)
        if (ctx->bufs[i].p) cudaFree(ctx->bufs[i].p);
    tc_rr_slots_free(ctx);
    if (ctx->aux[0]) { for (int i = 0; i < 4; ++i) cudaStreamDestroy(ctx->aux[i]); for (int i = 0; i < 5; ++i) cudaEventDestroy(ctx->aux_ev[i]); }
    if (ctx->ring) { cudaFreeHost(ctx->ring); for (int i = 0; i < 8; ++i) cudaEventDestroy(ctx->ring_ev[i]); }
    if (ctx->host_status) cudaFreeHost(ctx->host_status);
    if (ctx->host_scratch) cudaFreeHost(ctx->host_scratch);
    if (ctx->ev0) { cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); }
    tc_sample_slots_free(ctx);
    free(ctx);
    return TC_OK;
}

TC_API int tc_transfer_bytes(const tc_ctx_t* ctx, int64_t* h2d, int64_t* d2h) {
    if (!ctx) return TC_ERR_ARG;
    if (h2d) *h2d = ctx->h2d_bytes;
    if (d2h) *d2h = ctx->d2h_bytes;
    return TC_OK;
}

TC_API int tc_ctx_set_timing(tc_ctx_t* ctx, int enabled) {
    if (!ctx) return TC_ERR_ARG;
    TC_CUDA(cudaSetDevice(ctx->device));
    if (enabled && !ctx->ev0) {
        TC_CUDA(cudaEventCreate(&ctx->ev0));
        TC_CUDA(cudaEventCreate(&ctx->ev1));
    }
    ctx->timing = enabled ? 1 : 0;
    ctx->ev_valid = 0;
    return TC_OK;
}

TC_API float tc_last_pileup_kernel_ms(tc_ctx_t* ctx) {
    if (ctx && ctx->finished_ms > 0.0f) { const float ms = ctx->finished_ms; ctx->finished_ms = -1.0f; return ms; }     // of the sample finished last
    if (!ctx || !ctx->ev_valid) return -1.0f;
    float ms = -1.0f;
    if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.0f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) { cudaGetLastError(); return -1.0f; }
    return ms;
}

TC_API const char* tc_last_error(const tc_ctx_t* ctx) { return ctx ? ctx->err : g_create_err; }

TC_API int64_t tc_launch_count(const tc_ctx_t* ctx) { return ctx ? ctx->launches : 0; }

TC_API int tc_reads_upload(tc_ctx_t* ctx, const tc_reads_t* host, tc_reads_t* dev, void* stream) {
    if (!ctx || !host || !dev) return tc_fail(ctx, TC_ERR_ARG, "NULL argument");
    TC_CUDA(cudaSetDevice(ctx->device));
    dreads d;
    int need = (host->qual ? NEED_QUAL : 0) | NEED_MATE;        // (arrays that are NULL in *host are not copied)
    int rc = tc_resolve_reads(ctx, host, &d, need, (cudaStream_t)stream);
    if (rc) return rc;
    *dev = *host;
    dev->pos = d.pos; dev->flag = d.flag; dev->mapq = d.mapq; dev->l_seq = d.l_seq; dev->seq_off = d.seq_off;
    dev->cigar_off = d.cigar_off; dev->seq4 = d.seq4; dev->qual = d.qual; dev->cigar = d.cigar;
    dev->qname_hash = d.qname_hash; dev->mpos = d.mpos; dev->isize = d.isize;
    dev->cigar16 = nullptr;
    dev->seq2 = nullptr; dev->seq_exc_idx = nullptr; dev->seq_exc_val = nullptr; dev->n_seq_exc = 0;
    return TC_OK;
}

TC_API int tc_download(tc_ctx_t* ctx, void* dst_host, const void* src_dev, int64_t bytes, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (bytes < 0 || (bytes > 0 && (!dst_host || !src_dev))) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (bytes == 0) return TC_OK;
    TC_CUDA(cudaSetDevice(ctx->device));
    TC_D2H(dst_host, src_dev, (size_t)bytes, (cudaStream_t)stream);
    TC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return TC_OK;
}
