// bamwrite.cu — the decoded records written back as a BAM file image: BGZF members compressed on the device.
//
// After a decode the context holds the final records (payload + refID offsets, in the order the passes read them: clipped,
// sorted).  tc_bam_write_records turns them into the bytes of a BAM file as htslib frames one, so samtools, htslib and this
// library's own readers take it:
//   bamw_size_kernel       every record's 4 + block_size; a cub exclusive sum gives its offset behind the header
//   bamw_gather_kernel     one warp per record: the record copied into one contiguous stream behind the header (the lanes
//                          share 4-byte stores, bamrec.cuh's warp_copy), its bin recomputed as reg2bin(pos, end)
//   bgzf_deflate_kernel    one member per CTA: the header's members (at most 0xff00 bytes each, as bam_hdr_write flushes
//                          behind the header), then the records' from a fresh member on, cut every 0xff00 bytes.  The
//                          compressor is deflate_core.cuh's (dynamic Huffman, a stored block when that is smaller), the
//                          whole member in shared memory; the member's gzip header with the BC subfield, CRC-32 and ISIZE
//   bgzf_compact_kernel    the members' sizes summed (cub) and the members copied back to back, the 28-byte EOF member last
// Nothing here writes a buffer the read arrays, the payload or the record offsets of a decode live in: the reads stay valid.
#include <cub/device/device_scan.cuh>

#include "bamrec.cuh"
#include "deflate_core.cuh"
#include "tc_common.cuh"

namespace {

constexpr int REC_WARPS = 8;                    // records per 256-thread block
constexpr int DEFLATE_THREADS = 512;
constexpr long long MEMBER_STRIDE = 65536 + 64; // a member's slot: its 18-byte gzip header at +2, the stream at +20 (4-aligned)
constexpr int STREAM_AT = 20;
constexpr int BGZF_HEADER = 18, BGZF_TRAILER = 8, BGZF_EOF_BYTES = 28;
constexpr long long MEMBER_MAX = tcdef::MEMBER_MAX;

__constant__ uint8_t BGZF_EOF[BGZF_EOF_BYTES] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

__global__ void __launch_bounds__(256) bamw_size_kernel(const uint8_t* __restrict__ u, const long long* __restrict__ rec, long long n,
                                                        unsigned long long* size) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) size[i] = 4ull + ld32(u + rec[i] + BAM_BLOCK_SIZE);
}

__global__ void __launch_bounds__(256) bamw_gather_kernel(const uint8_t* __restrict__ u, const long long* __restrict__ rec, long long n,
                                                          const unsigned long long* __restrict__ off, uint8_t* __restrict__ out) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const uint8_t* r = u + rec[i];
    uint8_t* w = out + off[i] - BAM_BLOCK_SIZE;             // the output record's refID field
    const uint32_t n_cig = ld16(r + BAM_N_CIGAR_OP);
    const uint8_t* cig = bam_cigar(r);
    long long span = 0;
    for (uint32_t k = lane; k < n_cig; k += 32) {
        const uint32_t c = ld32(cig + 4ull * k);
        if (op_consumes_ref(c & 15u)) span += c >> 4;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) span += __shfl_xor_sync(0xffffffffu, span, o);
    const long long pos = (int32_t)ld32(r + BAM_POS);
    const uint32_t bin = reg2bin(pos, pos + (span > 0 ? span : 1));
    warp_copy(w + BAM_BLOCK_SIZE, r + BAM_BLOCK_SIZE, 4u + ld32(r + BAM_BLOCK_SIZE), lane);
    __syncwarp();
    if (lane == 0) { w[BAM_BIN] = (uint8_t)bin; w[BAM_BIN + 1] = (uint8_t)(bin >> 8); }
}

// member m: the header's members [0, n_hm), then the records' (the stream's bytes [n_header, n_total))
__device__ __forceinline__ void member_range(long long m, long long n_header, long long n_total, long long n_hm, long long& start, int& len) {
    if (m < n_hm) start = m * MEMBER_MAX;
    else start = n_header + (m - n_hm) * MEMBER_MAX;
    const long long end = m < n_hm ? n_header : n_total;
    len = (int)(end - start < MEMBER_MAX ? end - start : MEMBER_MAX);
}

__global__ void __launch_bounds__(DEFLATE_THREADS, 1) bgzf_deflate_kernel(const uint8_t* __restrict__ raw, long long n_header, long long n_total,
                                                                          long long n_hm, uint8_t* __restrict__ members,
                                                                          unsigned long long* __restrict__ msize) {
    extern __shared__ __align__(16) uint8_t smem[];
    tcdef::member_smem& s = *reinterpret_cast<tcdef::member_smem*>(smem);
    const long long m = blockIdx.x;
    long long start;
    int n;
    member_range(m, n_header, n_total, n_hm, start, n);
    for (int i = threadIdx.x; i < n; i += blockDim.x) s.in[i] = raw[start + i];
    __syncthreads();
    uint8_t* slot = members + m * MEMBER_STRIDE;
    tcdef::deflate_member(s, n, reinterpret_cast<uint32_t*>(slot + STREAM_AT), blockDim.x, threadIdx.x);
    const int c = s.t.out_bytes;
    const uint32_t bsize = (uint32_t)(BGZF_HEADER + c + BGZF_TRAILER - 1);
    uint8_t* h = slot + STREAM_AT - BGZF_HEADER;
    if (threadIdx.x < BGZF_HEADER) {
        const uint8_t head[16] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0};
        h[threadIdx.x] = threadIdx.x < 16 ? head[threadIdx.x] : (uint8_t)(bsize >> (8 * (threadIdx.x - 16)));
    } else if (threadIdx.x < BGZF_HEADER + BGZF_TRAILER) {
        const int k = threadIdx.x - BGZF_HEADER;
        const uint32_t v = k < 4 ? s.t.crc : (uint32_t)n;
        slot[STREAM_AT + c + k] = (uint8_t)(v >> (8 * (k & 3)));
    }
    if (threadIdx.x == 0) msize[m] = bsize + 1ull;
}

__global__ void __launch_bounds__(256) bgzf_compact_kernel(const uint8_t* __restrict__ members, const unsigned long long* __restrict__ msize,
                                                           const unsigned long long* __restrict__ moff, long long n_members,
                                                           uint8_t* __restrict__ image) {
    const long long m = blockIdx.x;
    if (m == n_members) {
        if (threadIdx.x < BGZF_EOF_BYTES) image[moff[m] + threadIdx.x] = BGZF_EOF[threadIdx.x];
        return;
    }
    const uint8_t* src = members + m * MEMBER_STRIDE + STREAM_AT - BGZF_HEADER;
    uint8_t* dst = image + moff[m];
    const uint32_t n = (uint32_t)msize[m];
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

}  // namespace

TC_API int tc_bam_write_records(tc_ctx_t* ctx, const uint8_t* header, int64_t n_header, const uint8_t* payload, int64_t n_bytes,
                                const int64_t* rec_off, int64_t n_reads, const uint8_t** image_dev, int64_t* image_bytes,
                                int64_t* n_members, float* t_ms, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (n_header < 0 || (n_header > 0 && !header) || n_reads < 0 || n_bytes < 0 || (n_reads > 0 && (!payload || !rec_off)) ||
        !image_dev || !image_bytes || !n_members)
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    *image_dev = nullptr; *image_bytes = 0; *n_members = 0;
    cudaEvent_t ev[6] = {};
    if (t_ms) for (auto& e : ev) TC_CUDA(cudaEventCreate(&e));
    int rc = TC_OK;
    const size_t n = (size_t)n_reads;
    const uint8_t* u = nullptr;
    const long long* rec = nullptr;
    unsigned long long* d_off = nullptr;
    long long n_rec_bytes = 0;
    unsigned long long* h = (unsigned long long*)ctx->host_status;
    if (t_ms) TC_CUDA(cudaEventRecord(ev[0], s));
    if (n) {
        u = (const uint8_t*)tc_stage_in(ctx, SLOT_BAMW_PAYLOAD, payload, (size_t)n_bytes, s, &rc); if (rc) return rc;
        rec = (const long long*)tc_stage_in(ctx, SLOT_BAMW_REC, rec_off, 8 * n, s, &rc); if (rc) return rc;
        unsigned long long* d_size = (unsigned long long*)tc_dev_buf(ctx, SLOT_BAMW_WORK, 16 * (n + 1));
        if (!d_size) return TC_ERR_NOMEM;
        d_off = d_size + n + 1;
        TC_CUDA(cudaMemsetAsync(d_size + n, 0, 8, s));
        bamw_size_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(u, rec, n_reads, d_size);
        TC_LAUNCH_CHECK();
        size_t tmp_bytes = 0;
        TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_size, d_off, (int)(n + 1), s));
        void* d_tmp = tc_dev_buf(ctx, SLOT_BAMW_TMP, tmp_bytes + 16);
        if (!d_tmp) return TC_ERR_NOMEM;
        TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_size, d_off, (int)(n + 1), s));
        ctx->launches++;
        TC_D2H(h, d_off + n, 8, s);
        if (t_ms) TC_CUDA(cudaEventRecord(ev[1], s));
        TC_CUDA(cudaStreamSynchronize(s));
        n_rec_bytes = (long long)h[0];
    } else if (t_ms) {
        TC_CUDA(cudaEventRecord(ev[1], s));
    }
    // the uncompressed stream: the header, then the records
    const long long n_total = n_header + n_rec_bytes;
    const long long n_hm = (n_header + MEMBER_MAX - 1) / MEMBER_MAX, n_rm = (n_rec_bytes + MEMBER_MAX - 1) / MEMBER_MAX;
    const long long nm = n_hm + n_rm;
    uint8_t* d_raw = (uint8_t*)tc_dev_buf(ctx, SLOT_BAMW_RAW, (size_t)n_total + 64);
    uint8_t* d_members = (uint8_t*)tc_dev_buf(ctx, SLOT_BAMW_MEMBERS, (size_t)(nm > 0 ? nm : 1) * MEMBER_STRIDE + 16 * (size_t)(nm + 1) * 2);
    uint8_t* d_image = (uint8_t*)tc_dev_buf(ctx, SLOT_BAMW_IMAGE, (size_t)nm * 65536 + BGZF_EOF_BYTES + 64);
    if (!d_raw || !d_members || !d_image) return TC_ERR_NOMEM;
    unsigned long long* d_msize = (unsigned long long*)(d_members + (size_t)(nm > 0 ? nm : 1) * MEMBER_STRIDE);
    unsigned long long* d_moff = d_msize + nm + 1;
    if (t_ms) TC_CUDA(cudaEventRecord(ev[2], s));
    if (n_header) { rc = tc_h2d(ctx, d_raw, header, (size_t)n_header, s); if (rc) return rc; }
    if (n) {
        bamw_gather_kernel<<<(unsigned)((n + REC_WARPS - 1) / REC_WARPS), 32 * REC_WARPS, 0, s>>>(u, rec, n_reads, d_off, d_raw + n_header);
        TC_LAUNCH_CHECK();
    }
    if (t_ms) TC_CUDA(cudaEventRecord(ev[3], s));
    TC_CUDA(cudaMemsetAsync(d_msize + nm, 0, 8, s));
    if (nm) {
        const int smem = (int)sizeof(tcdef::member_smem);
        TC_CUDA(cudaFuncSetAttribute(bgzf_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        bgzf_deflate_kernel<<<(unsigned)nm, DEFLATE_THREADS, smem, s>>>(d_raw, n_header, n_total, n_hm, d_members, d_msize);
        TC_LAUNCH_CHECK();
    }
    if (t_ms) TC_CUDA(cudaEventRecord(ev[4], s));
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_msize, d_moff, (int)(nm + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_BAMW_TMP, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_msize, d_moff, (int)(nm + 1), s));
    ctx->launches++;
    bgzf_compact_kernel<<<(unsigned)(nm + 1), 256, 0, s>>>(d_members, d_msize, d_moff, nm, d_image);
    TC_LAUNCH_CHECK();
    if (t_ms) TC_CUDA(cudaEventRecord(ev[5], s));
    TC_D2H(h, d_moff + nm, 8, s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (t_ms) {
        float a = 0, b = 0, c = 0, d = 0;
        cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&b, ev[2], ev[3]);
        cudaEventElapsedTime(&c, ev[3], ev[4]); cudaEventElapsedTime(&d, ev[4], ev[5]);
        t_ms[0] = a + b; t_ms[1] = c; t_ms[2] = d;
        for (auto& e : ev) cudaEventDestroy(e);
    }
    *image_dev = d_image;
    *image_bytes = (int64_t)h[0] + BGZF_EOF_BYTES;
    *n_members = nm;
    return TC_OK;
}
