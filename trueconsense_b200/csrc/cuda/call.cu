// call.cu — kernel (4): the per-position consensus / IUPAC call.
//
// One thread per reference position restates, on the seven counters of that position,
//   GetDistribution + GetNucleotide   TrueConsense/Sequences.py:119-165
//   IsAmbiguous and helpers           TrueConsense/Ambig.py:102-228
//   MinorityDel                       TrueConsense/Events.py:85-106
//   the ListInserts threshold         TrueConsense/Events.py:25-36
// and emits the candidate table (tc_call_table_t) the sequential walk of
// Sequences.BuildConsensus reads.  A second, single-CTA kernel turns the PRIMARY_X flags into
// len(WalkForward(p)) for every p (Sequences.py:44-52) with a reverse segmented scan.
//
// The percentage tests are IEEE-double (count / cov) * 100 with division and multiplication
// rounded separately, exactly like CPython's float arithmetic: __ddiv_rn / __dmul_rn / __dsub_rn
// keep ptxas from contracting anything (the file is also built with --fmad=false).  Integer
// cross-multiplication gives different answers at the thresholds (SURVEY.md §4.3: 55/45 at
// coverage 100 is not ambiguous, 6/5 at coverage 10 is).
#include <stdlib.h>

#include "tc_common.cuh"

__device__ __forceinline__ double pct(int c, int cov) { return __dmul_rn(__ddiv_rn((double)c, (double)cov), 100.0); }
__device__ __forceinline__ bool within(double a, double b, double maxdist) { return fabs(__dsub_rn(a, b)) <= maxdist; }

// letters indexed 0..4 = A,T,C,G,X in the reference's dict order; tie-break by the letter's
// ASCII value (Sequences.py:137-140 sorts (count, letter) tuples)
struct ranked5 { int cnt[5]; char let[5]; };

__device__ __forceinline__ void rank5(const int c[5], ranked5& r) {
    // rank of letter i = how many letters beat it: larger count, or equal count and larger ASCII
    const int asc[5] = {'A', 'T', 'C', 'G', 'X'};
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        int beat = 0;
#pragma unroll
        for (int j = 0; j < 5; ++j)
            if (j != i && (c[j] > c[i] || (c[j] == c[i] && asc[j] > asc[i]))) ++beat;
#pragma unroll
        for (int k = 0; k < 5; ++k)
            if (beat == k) { r.cnt[k] = c[i]; r.let[k] = (char)asc[i]; }
    }
}

// Ambig.py:18-99: the IUPAC code of a set of 2 or 3 distinct letters out of A,C,G,T
__device__ __forceinline__ char iupac_of_mask(int m) {
    // bit0 A, bit1 C, bit2 G, bit3 T
    switch (m) {
        case 0x3: return 'M'; case 0x5: return 'R'; case 0x9: return 'W'; case 0x6: return 'S';
        case 0xA: return 'Y'; case 0xC: return 'K'; case 0x7: return 'V'; case 0xB: return 'H';
        case 0xD: return 'D'; case 0xE: return 'B'; default: return 0;
    }
}
__device__ __forceinline__ int letter_bit(char l) { return l == 'A' ? 1 : l == 'C' ? 2 : l == 'G' ? 4 : l == 'T' ? 8 : 0; }

// Ambig.py:179-228
__device__ __forceinline__ char is_ambiguous(const char let[4], const int cnt[4], int cov, double maxdist) {
    if (cov == 0) return 0;
    if (let[0] == 'X' || let[1] == 'X') return 0;
    double p1 = pct(cnt[0], cov), p2 = pct(cnt[1], cov), p3 = pct(cnt[2], cov), p4 = pct(cnt[3], cov);
    if (!within(p1, p2, maxdist)) return 0;                                     // AmbiguityType: None
    if (within(p1, p3, maxdist) && within(p2, p3, maxdist)) {
        if (within(p1, p4, maxdist) && within(p2, p4, maxdist) && within(p3, p4, maxdist)) return 'N';   // type 4
        if (let[2] == 'X') return 'N';                                          // type 3 with X in the top three
        return iupac_of_mask(letter_bit(let[0]) | letter_bit(let[1]) | letter_bit(let[2]));
    }
    return iupac_of_mask(letter_bit(let[0]) | letter_bit(let[1]));              // type 2
}

struct call_args {
    const int32_t* counts; int L;
    int mincov; int include_ambig; double maxdist, mdel_pct, ins_pct;
    uint8_t* call_char; uint8_t* flags; int32_t* xrun; uint8_t* rank_letter; int32_t* rank_count; uint8_t* ambig_char;
};

__global__ void __launch_bounds__(256) call_kernel(call_args a) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.L) return;
    const size_t L = (size_t)a.L;
    const int cov = a.counts[TC_ROW_COV * L + p];
    int c[5];
    c[0] = a.counts[TC_ROW_A * L + p]; c[1] = a.counts[TC_ROW_T * L + p]; c[2] = a.counts[TC_ROW_C * L + p];
    c[3] = a.counts[TC_ROW_G * L + p]; c[4] = a.counts[TC_ROW_X * L + p];
    const int ins = a.counts[TC_ROW_I * L + p];
    ranked5 r;
    rank5(c, r);
    char amb = is_ambiguous(r.let, r.cnt, cov, a.maxdist);
    unsigned f = 0;
    if (cov < a.mincov) f |= TC_CF_LOWCOV;
    if (cov > a.mincov) f |= TC_CF_COV_GT_MINCOV;
    if (cov == 0) f |= TC_CF_ZERO_COV;
    if (r.let[0] == 'X') f |= TC_CF_PRIMARY_X;
    if (cov != 0 && pct(c[4], cov) >= a.mdel_pct) f |= TC_CF_MINORITY_DEL;                       // Events.py:102-106
    if (!(cov < a.mincov) && cov != 0 && ins != 0 && pct(ins, cov) > a.ins_pct) f |= TC_CF_INS_CANDIDATE;   // Events.py:29-36
    if (amb) f |= TC_CF_AMBIG;
    char ch;
    if (r.let[0] != 'X') {
        if (a.include_ambig && amb) ch = amb;
        else ch = (r.cnt[0] < a.mincov) ? (char)(r.let[0] | 0x20) : r.let[0];
    } else {
        ch = (r.cnt[1] < a.mincov) ? (char)(r.let[1] | 0x20) : r.let[1];
    }
    if (a.call_char) a.call_char[p] = (uint8_t)ch;
    a.flags[p] = (uint8_t)f;
    if (a.ambig_char) a.ambig_char[p] = (uint8_t)amb;
    if (a.rank_letter) {
#pragma unroll
        for (int k = 0; k < 4; ++k) a.rank_letter[k * L + p] = (uint8_t)r.let[k];
    }
    if (a.rank_count) {
#pragma unroll
        for (int k = 0; k < 4; ++k) a.rank_count[k * L + p] = r.cnt[k];
    }
}

// xrun[j] = number of consecutive PRIMARY_X positions starting at j+1.  One CTA; thread t owns a
// contiguous chunk, scans it backwards, thread 0 chains the chunk carries, chunks patch their tails.
// len(WalkForward(p)) (Sequences.py:44-52) = consecutive positions after p whose rank-1 letter is X
//                                           = nn(p + 1) - (p + 1),  nn(k) = first position >= k that is not X (L if none).
// nn is a reverse min-scan.  xrun_local_kernel scans inside blocks of XR_BLOCK positions (coalesced, warp
// shuffles) and leaves every block's first non-X position; xrun_apply_kernel looks up the blocks to the
// right for runs that leave their block.  Both are ordinary multi-CTA kernels: no serial pass over L.
// Several references side by side (tc_call_contigs): a run stops at the end of its own reference, so xrun_apply_kernel
// clamps nn to that end — the first non-X position at or after k, if it lies beyond the end, means every position from
// k to the end is X.  The local scan needs no boundaries.
constexpr int XR_BLOCK = 256;

__global__ void __launch_bounds__(XR_BLOCK) xrun_local_kernel(const uint8_t* __restrict__ flags, int32_t* __restrict__ nn_local,
                                                              int32_t* __restrict__ block_first, int L) {
    __shared__ int wmin[XR_BLOCK / 32];
    const int j = blockIdx.x * XR_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int INF = 0x7fffffff;
    int v = (j < L && !(flags[j] & TC_CF_PRIMARY_X)) ? j : INF;
    // suffix minimum inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v = min(v, t); }
    if (lane == 0) wmin[warp] = v;
    __syncthreads();
    int later = INF;
    for (int w = warp + 1; w < XR_BLOCK / 32; ++w) later = min(later, wmin[w]);
    v = min(v, later);
    if (j < L) nn_local[j] = v;                 // first non-X position in [j, end of block), INF if none
    if (threadIdx.x == 0) block_first[blockIdx.x] = v;
}

// the end (exclusive) of the reference holding position j: contig_start[n] = L, references may be empty
__device__ __forceinline__ int contig_end(const int32_t* __restrict__ contig_start, int n, int j) {
    int lo = 0, hi = n - 1;                     // the last reference k with contig_start[k] <= j
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(contig_start + mid) <= j) lo = mid; else hi = mid - 1;
    }
    return __ldg(contig_start + lo + 1);
}

// contig_start: NULL (one reference) or the n_contigs + 1 boundaries of the references
__global__ void __launch_bounds__(XR_BLOCK) xrun_apply_kernel(uint8_t* __restrict__ flags, const int32_t* __restrict__ nn_local,
                                                              const int32_t* __restrict__ block_first, int32_t* __restrict__ xrun, int L, int n_blocks,
                                                              const int32_t* __restrict__ contig_start, int n_contigs) {
    __shared__ int right_s;
    const int INF = 0x7fffffff;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {     // first non-X position in any block to the right (L if none)
        int best = INF;
        for (int b0 = blockIdx.x + 1; b0 < n_blocks && best == INF; b0 += 32) {
            const int v = b0 + lane < n_blocks ? block_first[b0 + lane] : INF;
            const unsigned has = __ballot_sync(0xffffffffu, v != INF);
            if (has) best = __shfl_sync(0xffffffffu, v, __ffs(has) - 1);
        }
        if (lane == 0) right_s = best == INF ? L : best;
    }
    __syncthreads();
    const int j = blockIdx.x * XR_BLOCK + threadIdx.x;
    if (j >= L) return;
    const int k = j + 1;                        // nn(k)
    int nn;
    if (k >= L) nn = L;
    else if (k < (blockIdx.x + 1) * XR_BLOCK) { const int v = nn_local[k]; nn = v == INF ? right_s : v; }
    else {                                      // k is the first position of the next block
        const int v = block_first[blockIdx.x + 1];
        if (v != INF) nn = v;
        else {                                  // rare: the whole next block is X — look further right
            nn = L;
            for (int b2 = blockIdx.x + 2; b2 < n_blocks; ++b2) { const int w = block_first[b2]; if (w != INF) { nn = w; break; } }
        }
    }
    const int end = contig_start ? contig_end(contig_start, n_contigs, j) : L;
    nn = min(nn, end);
    xrun[j] = nn - k;
    if (nn == end) flags[j] |= TC_CF_XRUN_OFF_END;
}

__global__ void is_ambiguous_kernel(const uint8_t* __restrict__ letters, const int32_t* __restrict__ cnts,
                                    const int32_t* __restrict__ cov, int64_t n, double maxdist, uint8_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    char let[4]; int cnt[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { let[k] = (char)letters[k * n + i]; cnt[k] = cnts[k * n + i]; }
    out[i] = (uint8_t)is_ambiguous(let, cnt, cov[i], maxdist);
}

// INS_CANDIDATE positions (1-based): appended in any order by a multi-CTA pass (candidates are rare), then
// put in ascending order by a rank sort over the few that exist
__global__ void list_candidates_kernel(const uint8_t* __restrict__ flags, int L, int32_t* __restrict__ out, int cap, int32_t* __restrict__ n_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < L && (flags[j] & TC_CF_INS_CANDIDATE)) {
        const int slot = atomicAdd(n_out, 1);
        if (slot < cap) out[slot] = j + 1;
    }
}

__global__ void rank_sort_kernel(const int32_t* __restrict__ in, const int32_t* __restrict__ n_in, int cap, int32_t* __restrict__ out) {
    const int n = min(*n_in, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int v = in[i];
        int rank = 0;
        for (int k = 0; k < n; ++k) rank += in[k] < v;       // positions are distinct
        out[rank] = v;
    }
}

// ---------------------------------------------------------------- C-ABI
// tc_call and tc_call_contigs: d_contig_start is NULL (one reference) or the n_contigs + 1 boundaries in device memory
static int call_table(tc_ctx_t* ctx, const int32_t* counts, int32_t ref_len, const int32_t* d_contig_start, int32_t n_contigs,
                      const tc_call_params_t* p, const tc_call_table_t* t, cudaStream_t s) {
    const size_t L = (size_t)ref_len;
    int rc;
    call_args a;
    a.counts = (const int32_t*)tc_stage_in(ctx, SLOT_COUNTS, counts, sizeof(int32_t) * TC_NROWS * L, s, &rc);
    if (rc) return rc;
    a.L = ref_len; a.mincov = p->mincov; a.include_ambig = p->include_ambig;
    a.maxdist = p->ambig_maxdist; a.mdel_pct = p->minority_del_pct; a.ins_pct = p->insert_pct;
    struct out_t { void* user; void* dev; size_t bytes; int slot; };
    out_t outs[6] = {
        {t->call_char, nullptr, L, SLOT_CALL_A}, {t->flags, nullptr, L, SLOT_CALL_B}, {t->xrun, nullptr, 4 * L, SLOT_CALL_C},
        {t->rank_letter, nullptr, 4 * L, SLOT_CALL_D}, {t->rank_count, nullptr, 16 * L, SLOT_CALL_E}, {t->ambig_char, nullptr, L, SLOT_CALL_F}};
    for (int i = 0; i < 6; ++i) {
        bool need = outs[i].user != nullptr || i == 1;     // flags feed the xrun kernel
        if (!need) continue;
        if (outs[i].user && tc_is_device_ptr(outs[i].user)) outs[i].dev = outs[i].user;
        else { outs[i].dev = tc_dev_buf(ctx, outs[i].slot, outs[i].bytes); if (!outs[i].dev) return TC_ERR_NOMEM; }
    }
    a.call_char = (uint8_t*)outs[0].dev; a.flags = (uint8_t*)outs[1].dev; a.xrun = (int32_t*)outs[2].dev;
    a.rank_letter = (uint8_t*)outs[3].dev; a.rank_count = (int32_t*)outs[4].dev; a.ambig_char = (uint8_t*)outs[5].dev;
    call_kernel<<<(unsigned)((L + 255) / 256), 256, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    if (a.xrun) {
        const int n_blocks = (ref_len + XR_BLOCK - 1) / XR_BLOCK;
        int32_t* nn_local = (int32_t*)tc_dev_buf(ctx, SLOT_SEGS, 4 * (L + (size_t)n_blocks) + 64);
        if (!nn_local) return TC_ERR_NOMEM;
        int32_t* block_first = nn_local + L;
        xrun_local_kernel<<<n_blocks, XR_BLOCK, 0, s>>>(a.flags, nn_local, block_first, ref_len);
        TC_LAUNCH_CHECK();
        xrun_apply_kernel<<<n_blocks, XR_BLOCK, 0, s>>>(a.flags, nn_local, block_first, a.xrun, ref_len, n_blocks, d_contig_start, n_contigs);
        TC_LAUNCH_CHECK();
    }
    bool any_host = false;
    for (int i = 0; i < 6; ++i) {
        if (outs[i].user && outs[i].dev != outs[i].user) {
            TC_D2H(outs[i].user, outs[i].dev, outs[i].bytes, s);
            any_host = true;
        }
    }
    if (any_host) TC_CUDA(cudaStreamSynchronize(s));
    return TC_OK;
}

TC_API int tc_call(tc_ctx_t* ctx, const int32_t* counts, int32_t ref_len, const tc_call_params_t* p,
                   const tc_call_table_t* t, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!counts || !p || !t) return tc_fail(ctx, TC_ERR_ARG, "NULL argument");
    if (ref_len <= 0) return tc_fail(ctx, TC_ERR_ARG, "ref_len must be positive");
    TC_CUDA(cudaSetDevice(ctx->device));
    return call_table(ctx, counts, ref_len, nullptr, 0, p, t, (cudaStream_t)stream);
}

TC_API int tc_call_contigs(tc_ctx_t* ctx, const int32_t* counts, int32_t total_len, int32_t n, const int32_t* contig_start,
                           const tc_call_params_t* p, const tc_call_table_t* t, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!counts || !p || !t || !contig_start) return tc_fail(ctx, TC_ERR_ARG, "NULL argument");
    if (total_len <= 0 || n <= 0) return tc_fail(ctx, TC_ERR_ARG, "total_len and the number of references must be positive");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    // the boundaries are checked on the host (a device array is read back: n + 1 integers) and kept on the device
    const size_t bytes = 4 * ((size_t)n + 1);
    const bool on_dev = tc_is_device_ptr(contig_start);
    const int32_t* h = contig_start;
    int32_t* tmp = nullptr;
    if (on_dev) {
        tmp = (int32_t*)malloc(bytes);
        if (!tmp) return tc_fail(ctx, TC_ERR_NOMEM, "host memory for %d boundaries", n + 1);
        cudaError_t e = cudaMemcpyAsync(tmp, contig_start, bytes, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { free(tmp); return tc_cuda_fail(ctx, e, "reading contig_start"); }
        ctx->d2h_bytes += (int64_t)bytes;
        h = tmp;
    }
    int bad = h[0] != 0 || h[n] != total_len;
    for (int32_t k = 0; k < n && !bad; ++k) bad = h[k + 1] < h[k];
    free(tmp);
    if (bad) return tc_fail(ctx, TC_ERR_ARG, "contig_start must rise from 0 to total_len (%d) in %d steps", total_len, n);
    int rc;
    const int32_t* d_cs = (const int32_t*)tc_stage_in(ctx, SLOT_CONTIG_A, contig_start, bytes, s, &rc);
    if (rc) return rc;
    return call_table(ctx, counts, total_len, d_cs, n, p, t, s);
}

TC_API int tc_is_ambiguous(tc_ctx_t* ctx, const uint8_t* letters, const int32_t* cnts, const int32_t* cov, int64_t n,
                           double maxdist, uint8_t* out_char, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!letters || !cnts || !cov || !out_char || n < 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n == 0) return TC_OK;
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const uint8_t* dl = (const uint8_t*)tc_stage_in(ctx, SLOT_TMP_A, letters, 4 * (size_t)n, s, &rc); if (rc) return rc;
    const int32_t* dc = (const int32_t*)tc_stage_in(ctx, SLOT_TMP_B, cnts, 16 * (size_t)n, s, &rc); if (rc) return rc;
    const int32_t* dv = (const int32_t*)tc_stage_in(ctx, SLOT_TMP_C, cov, 4 * (size_t)n, s, &rc); if (rc) return rc;
    bool out_dev = tc_is_device_ptr(out_char);
    uint8_t* d_out = out_dev ? out_char : (uint8_t*)tc_dev_buf(ctx, SLOT_CALL_F, (size_t)n);
    if (!d_out) return TC_ERR_NOMEM;
    is_ambiguous_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dl, dc, dv, n, maxdist, d_out);
    TC_LAUNCH_CHECK();
    if (!out_dev) {
        TC_D2H(out_char, d_out, (size_t)n, s);
        TC_CUDA(cudaStreamSynchronize(s));
    }
    return TC_OK;
}

// INS_CANDIDATE positions, ascending, left on the device together with their number: [unordered: cap] [count] [sorted: cap]
int tc_candidates_enqueue(tc_ctx* ctx, const uint8_t* d_flags, int32_t ref_len, int32_t cap, int32_t** d_count, int32_t** d_sorted, cudaStream_t s) {
    int32_t* d_buf = (int32_t*)tc_dev_buf(ctx, SLOT_TMP_B, 4 * (2 * (size_t)cap + 1) + 64);
    if (!d_buf) return TC_ERR_NOMEM;
    int32_t* d_cnt = d_buf + cap;
    TC_CUDA(cudaMemsetAsync(d_cnt, 0, 4, s));
    list_candidates_kernel<<<(unsigned)((ref_len + 255) / 256), 256, 0, s>>>(d_flags, ref_len, d_buf, cap, d_cnt);
    TC_LAUNCH_CHECK();
    rank_sort_kernel<<<32, 256, 0, s>>>(d_buf, d_cnt, cap, d_cnt + 1);
    TC_LAUNCH_CHECK();
    *d_count = d_cnt; *d_sorted = d_cnt + 1;
    return TC_OK;
}

TC_API int tc_list_insert_candidates(tc_ctx_t* ctx, const uint8_t* flags, int32_t ref_len, int32_t* cand_pos, int32_t cap,
                                     int32_t* n_out, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!flags || !cand_pos || !n_out || ref_len <= 0 || cap < 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const uint8_t* df = (const uint8_t*)tc_stage_in(ctx, SLOT_TMP_A, flags, (size_t)ref_len, s, &rc); if (rc) return rc;
    int32_t *d_cnt, *d_sorted;
    rc = tc_candidates_enqueue(ctx, df, ref_len, cap, &d_cnt, &d_sorted, s);
    if (rc) return rc;
    // the count and the first candidates come back in one copy (there are rarely more than a handful)
    const int first = cap < 63 ? cap : 63;
    TC_D2H(ctx->host_status, d_cnt, 4 * (size_t)(1 + first), s);
    TC_CUDA(cudaStreamSynchronize(s));
    const int32_t n = *(int32_t*)ctx->host_status;
    *n_out = n;
    if (n > cap) return tc_fail(ctx, TC_ERR_CAPACITY, "%d insertion candidates, capacity %d", n, cap);
    if (n > 0) {
        if (tc_is_device_ptr(cand_pos)) {
            TC_CUDA(cudaMemcpyAsync(cand_pos, d_sorted, 4 * (size_t)n, cudaMemcpyDeviceToDevice, s));
            TC_CUDA(cudaStreamSynchronize(s));
        } else if (n <= first) {
            memcpy(cand_pos, (int32_t*)ctx->host_status + 1, 4 * (size_t)n);
        } else {
            TC_D2H(cand_pos, d_sorted, 4 * (size_t)n, s);
            TC_CUDA(cudaStreamSynchronize(s));
        }
    }
    return TC_OK;
}
