// contigs.cu — every reference of a multi-reference BAM in one device pass.
//
// The references lie side by side in one coordinate space: reference k occupies the global columns
// [base[k], base[k] + len[k]), base being the exclusive prefix sum of the lengths.  Two small passes put the reads there:
//   contig_ranges_kernel  one thread per record reads its refID and writes the boundaries where it changes:
//                         first_read[k] .. first_read[k+1]-1 are the reads of reference k (records are in file order)
//   contig_shift_kernel   one thread per read: its reference span (the CIGAR ops bam_meta_kernel counts), the range check
//                         the single-reference pileup makes for that read on its own reference, then pos += base[k] and,
//                         for a mate on the same reference, mpos += base[k] (-1 and -2 stay: the mate-overlap emulation
//                         keeps pairing only mates of one reference)
// Pileup, insertion candidates and ExtractInserts then run unchanged over the concatenated coordinates: no read of one
// reference covers a column of another.  tc_call_contigs (call.cu) keeps the X-runs of the call table inside their reference.
#include <algorithm>
#include <vector>

#include "tc_common.cuh"

namespace {

__device__ __forceinline__ int32_t ld_i32(const uint8_t* p) {     // records start at any byte
    return (int32_t)((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24));
}

__global__ void __launch_bounds__(256) contig_ranges_kernel(const uint8_t* __restrict__ u, const long long* __restrict__ rec, long long n,
                                                            int n_ref, int32_t* __restrict__ first_read, int* __restrict__ err) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int tid = ld_i32(u + rec[i]);
    const int prev = i > 0 ? ld_i32(u + rec[i - 1]) : -1;
    if (tid < 0 || tid >= n_ref) { atomicCAS(err, 0, TC_ERR_RANGE); return; }
    if (tid < prev) { atomicCAS(err, 0, TC_ERR_UNSORTED); return; }
    for (int k = max(prev, -1) + 1; k <= tid; ++k) first_read[k] = (int32_t)i;        // references tid and the empty ones before it
    if (i == n - 1)
        for (int k = tid + 1; k <= n_ref; ++k) first_read[k] = (int32_t)n;
}

struct shift_args {
    int32_t* pos; int32_t* mpos; const uint16_t* flag; const uint32_t* cigar_off; const uint32_t* cigar; long long n;
    const int32_t* first_read; const int32_t* base; int n_ref;
    unsigned long long* bad;        // smallest index of a read outside its reference (~0: none)
};

__global__ void __launch_bounds__(256) contig_shift_kernel(shift_args a) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.n) return;
    int lo = 0, hi = a.n_ref - 1;               // the last reference k with first_read[k] <= r (empty references share it)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(a.first_read + mid) <= r) lo = mid; else hi = mid - 1;
    }
    const int b = __ldg(a.base + lo), len = __ldg(a.base + lo + 1) - b;
    long long span = 0;
    for (uint32_t k = a.cigar_off[r]; k < a.cigar_off[r + 1]; ++k) {
        const uint32_t c = a.cigar[k], op = c & 15u;
        if (op == OP_M || op == OP_D || op == OP_N || op == OP_EQ || op == OP_X) span += (long long)(c >> 4);
    }
    int p = a.pos[r];
    if (!(a.flag[r] & 4u)) {
        // what tc_pileup_counts refuses for this read on its own reference (TC_ERR_RANGE)
        if (p < 0 || p >= len || (long long)p + span > len) { atomicMin(a.bad, (unsigned long long)r); return; }
    } else {
        // unmapped reads are dropped by every pass; kept inside their reference so that the order stays sorted
        p = min(max(p, 0), max(len - 1, 0));
    }
    a.pos[r] = b + p;
    if (a.mpos) {
        const int m = a.mpos[r];
        if (m >= 0) a.mpos[r] = (int32_t)((uint32_t)m + (uint32_t)b);
    }
}

// a host or device array of n int32 values on the host (tmp receives a device array)
const int32_t* host_view(tc_ctx* ctx, const int32_t* p, size_t n, int32_t* tmp, cudaStream_t s, int* rc) {
    *rc = TC_OK;
    if (!tc_is_device_ptr(p)) return p;
    cudaError_t e = cudaMemcpyAsync(tmp, p, 4 * n, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { *rc = tc_cuda_fail(ctx, e, "reading a boundary array"); return nullptr; }
    ctx->d2h_bytes += (int64_t)(4 * n);
    return tmp;
}

}  // namespace

TC_API int tc_bam_contig_ranges(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                                int32_t n_ref, int32_t* first_read, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!first_read || n_ref <= 0 || n_reads < 0 || n_bytes < 0 || (n_reads > 0 && (!payload || !rec_off)))
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n_reads >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 reads in one batch; shard the input");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)n_reads, out_bytes = 4 * ((size_t)n_ref + 1);
    const bool out_dev = tc_is_device_ptr(first_read);
    // [status int] [pad] [first_read: n_ref + 1]
    int32_t* d_buf = (int32_t*)tc_dev_buf(ctx, SLOT_CONTIG_B, 16 + out_bytes);
    if (!d_buf) return TC_ERR_NOMEM;
    int32_t* d_fr = out_dev ? first_read : d_buf + 4;
    TC_CUDA(cudaMemsetAsync(d_buf, 0, 16, s));
    TC_CUDA(cudaMemsetAsync(d_fr, 0, out_bytes, s));
    if (n > 0) {
        int rc;
        const uint8_t* u = (const uint8_t*)tc_stage_in(ctx, SLOT_BAM_PAYLOAD, payload, (size_t)n_bytes, s, &rc); if (rc) return rc;
        const long long* rec = (const long long*)tc_stage_in(ctx, SLOT_BAM_REC, rec_off, 8 * n, s, &rc); if (rc) return rc;
        contig_ranges_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(u, rec, n_reads, n_ref, d_fr, d_buf);
        TC_LAUNCH_CHECK();
    }
    int32_t* h = (int32_t*)ctx->host_status;
    TC_D2H(h, d_buf, 4, s);
    if (!out_dev) TC_D2H(first_read, d_fr, out_bytes, s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (h[0] == TC_ERR_UNSORTED) return tc_fail(ctx, TC_ERR_UNSORTED, "Unsorted input. Pileup aborts");
    if (h[0]) return tc_fail(ctx, h[0], "a record's refID lies outside the header's %d references", n_ref);
    return TC_OK;
}

TC_API int tc_reads_to_contig_coords(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t n_ref, const int32_t* ref_len,
                                     const int32_t* first_read, int32_t* contig_start, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!reads || !ref_len || !first_read || n_ref <= 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    const int64_t n = reads->n_reads;
    if (n < 0 || n >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "bad read count %lld", (long long)n);
    if (n > 0 && (!reads->pos || !reads->flag || !reads->cigar_off || !reads->cigar || !tc_is_device_ptr(reads->pos) ||
                  !tc_is_device_ptr(reads->flag) || !tc_is_device_ptr(reads->cigar_off) || !tc_is_device_ptr(reads->cigar) ||
                  (reads->mpos && !tc_is_device_ptr(reads->mpos))))
        return tc_fail(ctx, TC_ERR_ARG, "the reads must be device-resident (pos, flag, cigar_off, cigar and mpos, if given)");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    const size_t m = (size_t)n_ref + 1;
    // host copies of the lengths and boundaries, and the bases
    std::vector<int32_t> len_v(n_ref), fr_v(m), base(m);
    int rc;
    const int32_t* hlen = host_view(ctx, ref_len, (size_t)n_ref, len_v.data(), s, &rc); if (rc) return rc;
    const int32_t* hfr = host_view(ctx, first_read, m, fr_v.data(), s, &rc); if (rc) return rc;
    int64_t total = 0;
    for (int32_t k = 0; k < n_ref; ++k) {
        if (hlen[k] < 0) return tc_fail(ctx, TC_ERR_ARG, "reference %d has a negative length", k);
        base[k] = (int32_t)total;
        total += hlen[k];
        if (total > (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "the references' lengths add up to more than 2^31-1 columns");
        if (hfr[k + 1] < hfr[k]) return tc_fail(ctx, TC_ERR_ARG, "first_read must not decrease");
    }
    base[n_ref] = (int32_t)total;
    if (hfr[0] != 0 || hfr[n_ref] != n) return tc_fail(ctx, TC_ERR_ARG, "first_read must run from 0 to n_reads (%lld)", (long long)n);
    if (contig_start && !tc_is_device_ptr(contig_start)) memcpy(contig_start, base.data(), 4 * m);
    // device: [base: m] [first_read: m] [pad] [bad: 8 bytes]
    const size_t bad_at = (2 * m + 1) & ~(size_t)1;
    int32_t* d = (int32_t*)tc_dev_buf(ctx, SLOT_CONTIG_C, 4 * bad_at + 16);
    if (!d) return TC_ERR_NOMEM;
    rc = tc_h2d(ctx, d, base.data(), 4 * m, s); if (rc) return rc;
    rc = tc_h2d(ctx, d + m, hfr, 4 * m, s); if (rc) return rc;
    if (contig_start && tc_is_device_ptr(contig_start))
        TC_CUDA(cudaMemcpyAsync(contig_start, d, 4 * m, cudaMemcpyDeviceToDevice, s));
    if (n == 0) return TC_OK;
    unsigned long long* d_bad = (unsigned long long*)(d + bad_at);
    TC_CUDA(cudaMemsetAsync(d_bad, 0xff, 8, s));
    shift_args a;
    a.pos = const_cast<int32_t*>(reads->pos); a.mpos = const_cast<int32_t*>(reads->mpos); a.flag = reads->flag;
    a.cigar_off = reads->cigar_off; a.cigar = reads->cigar; a.n = n;
    a.first_read = d + m; a.base = d; a.n_ref = n_ref; a.bad = d_bad;
    contig_shift_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    uint64_t* h = (uint64_t*)ctx->host_status;
    TC_D2H(h, d_bad, 8, s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (h[0] != ~0ull) {
        const int64_t r = (int64_t)h[0];
        int32_t* hp = (int32_t*)(h + 1);
        TC_D2H(hp, reads->pos + r, 4, s);   // the failing thread wrote nothing: still the coordinate on its own reference
        TC_CUDA(cudaStreamSynchronize(s));
        int k = (int)(std::upper_bound(hfr, hfr + n_ref, (int32_t)r) - hfr) - 1;
        return tc_fail(ctx, TC_ERR_RANGE, "read %lld (file order) at %d runs outside reference %d (length %d); "
                       "the reads before it have been moved, decode the batch again", (long long)r, hp[0], k, hlen[k]);
    }
    return TC_OK;
}
