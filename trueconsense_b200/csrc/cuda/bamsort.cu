// bamsort.cu — a BAM's records in coordinate order, for input that is not coordinate-sorted (aligner output, a
// queryname-sorted file).
//
// Only the record offsets move: tc_bam_records_to_reads and tc_bam_contig_ranges read every record through rec_off, so
// handing them the offsets in coordinate order yields the sorted read arrays without a second copy of the payload.
//   bam_sort_key_kernel   one thread per record: refID, pos and FLAG -> the 64-bit key of samtools' default coordinate
//                         order (bam_sort.c bam1_cmp_core: refID, pos, then forward before reverse); whether the records are
//                         already sorted by (refID, pos); refID / pos outside what a placed record may hold
//   cub::DeviceRadixSort  keys + offsets, stable (ties keep file order: samtools' stable merge), over the key bits the
//                         header's reference count can set — skipped when the records are sorted already
#include <cub/device/device_radix_sort.cuh>

#include "tc_common.cuh"

namespace {

__device__ __forceinline__ uint32_t ld32(const uint8_t* p) {       // records start at any byte
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

struct sort_status {
    int unsorted;                   // some record sorts before its predecessor by (refID, pos)
    int pad;
    unsigned long long bad;         // smallest index of a record with refID outside [0, n_ref) or pos < -1 (~0: none)
};

__global__ void __launch_bounds__(256) bam_sort_key_kernel(const uint8_t* __restrict__ u, const long long* __restrict__ rec, long long n,
                                                           int n_ref, unsigned long long* __restrict__ key, sort_status* st) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int bad_order = 0;
    if (i < n) {
        const uint8_t* r = u + rec[i];
        const int32_t tid = (int32_t)ld32(r), pos = (int32_t)ld32(r + 4);
        const uint32_t reverse = (ld32(r + 12) >> 20) & 1u;            // FLAG (bytes 14-15) & 0x10
        if (tid < 0 || tid >= n_ref || pos < -1) atomicMin(&st->bad, (unsigned long long)i);
        // refID < 2^31 - 1 and pos + 1 < 2^31: both fields fit (refID above bit 32, pos + 1 in bits 1..31, the strand in bit 0)
        key[i] = ((unsigned long long)(uint32_t)tid << 32) | ((unsigned long long)(uint32_t)(pos + 1) << 1) | reverse;
        if (i > 0) {
            const uint8_t* q = u + rec[i - 1];
            const int32_t ptid = (int32_t)ld32(q), ppos = (int32_t)ld32(q + 4);
            bad_order = (tid < ptid) || (tid == ptid && pos < ppos);
        }
    }
    if (__ballot_sync(0xffffffffu, bad_order) && (threadIdx.x & 31) == 0) atomicExch(&st->unsorted, 1);
}

}  // namespace

TC_API int tc_bam_sort_records(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                               int32_t n_ref, const uint8_t** payload_dev, const int64_t** rec_sorted_dev, int32_t* reordered,
                               void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!payload_dev || !rec_sorted_dev || !reordered || n_reads < 0 || n_bytes < 0 || n_ref < 0 || (n_reads > 0 && (!payload || !rec_off)))
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n_reads >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 reads in one batch; shard the input");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    *payload_dev = payload; *rec_sorted_dev = rec_off; *reordered = 0;
    const size_t n = (size_t)n_reads;
    if (n == 0) return TC_OK;
    int rc;
    const uint8_t* u = (const uint8_t*)tc_stage_in(ctx, SLOT_BAM_PAYLOAD, payload, (size_t)n_bytes, s, &rc); if (rc) return rc;
    const long long* rec = (const long long*)tc_stage_in(ctx, SLOT_BAM_REC, rec_off, 8 * n, s, &rc); if (rc) return rc;
    *payload_dev = u; *rec_sorted_dev = (const int64_t*)rec;
    // keys in, keys out (8 bytes each per record), the status block
    unsigned long long* d_keys = (unsigned long long*)tc_dev_buf(ctx, SLOT_TMP_A, 16 * n + sizeof(sort_status) + 64);
    if (!d_keys) return TC_ERR_NOMEM;
    sort_status* d_st = (sort_status*)(d_keys + 2 * n);
    TC_CUDA(cudaMemsetAsync(d_st, 0, sizeof(sort_status), s));
    TC_CUDA(cudaMemsetAsync(&d_st->bad, 0xff, 8, s));
    bam_sort_key_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(u, rec, n_reads, n_ref, d_keys, d_st);
    TC_LAUNCH_CHECK();
    sort_status* h = (sort_status*)ctx->host_status;
    TC_D2H(h, d_st, sizeof(sort_status), s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (h->bad != ~0ull)
        return tc_fail(ctx, TC_ERR_RANGE, "BAM record %llu (of the %lld placed ones, in file order): refID outside the header's %d references or pos < -1",
                       h->bad, (long long)n_reads, n_ref);
    if (!h->unsorted) return TC_OK;
    // the refID part of the key spans bit_width(n_ref - 1) bits: a single-reference file sorts 32 bits, not 64
    int end_bit = 32;
    for (uint32_t m = (uint32_t)(n_ref - 1); m; m >>= 1) ++end_bit;
    long long* d_sorted = (long long*)tc_dev_buf(ctx, SLOT_BAM_REC_SORTED, 8 * n);
    if (!d_sorted) return TC_ERR_NOMEM;
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys + n, rec, d_sorted, (int)n, 0, end_bit, s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys + n, rec, d_sorted, (int)n, 0, end_bit, s));
    ctx->launches++;
    // the offsets are complete on return (the caller may read them on another stream, and the sort's time is its own)
    TC_CUDA(cudaStreamSynchronize(s));
    *rec_sorted_dev = (const int64_t*)d_sorted;
    *reordered = 1;
    return TC_OK;
}
