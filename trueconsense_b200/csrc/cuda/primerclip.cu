// primerclip.cu — amplicon primers soft-clipped off aligned BAM records (what `samtools ampliconclip --soft-clip` does
// before `samtools sort`), records in, records out.  The rule is DESIGN §4's; oracle/primer_clip.py restates it.
//
// The clip sits between the record index (or the SAM conversion) and tc_bam_sort_records: the clipped records land in a
// payload buffer of their own with their refID offsets in input order, and sorting, parsing and the contig ranges run on
// them unchanged.
//   primer tables (host)   per reference: the primers by start with a running max of the end, by end with a running min of
//                          the start from the right — one binary search per read end finds whether a primer matches and the
//                          column the clip reaches
//   clip_plan_kernel       one warp per record: the CIGAR 32 ops at a time (warp scans of the reference and query lengths,
//                          ballots for the op each cut falls on) -> the record's new size, pos, FLAG, bin and edit descriptor
//   cub exclusive sum      new sizes -> output offsets
//   clip_pack_kernel       one warp per record: fixed fields, name, the new CIGAR, then SEQ / QUAL / optional fields copied
//                          with the lanes sharing 4-byte words
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <vector>

#include "bamrec.cuh"
#include "tc_common.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int REC_WARPS = 8;            // records per 256-thread block

__device__ __forceinline__ bool is_clip(uint32_t op) { return op == OP_S || op == OP_H; }
__device__ __forceinline__ uint32_t query_len(uint32_t c) {          // M, I, S, =, X
    const uint32_t op = c & 15u;
    return ((0x193u >> op) & 1u) ? (c >> 4) : 0u;
}
__device__ __forceinline__ uint32_t ref_len(uint32_t c) { return op_consumes_ref(c & 15u) ? (c >> 4) : 0u; }

// per reference r the primers [first[r], first[r + 1]): starts ascending with the running max of the ends, ends ascending with
// the running min of the starts from the right
struct primer_tables {
    const int32_t* first; const int32_t* by_start; const int32_t* max_end; const int32_t* by_end; const int32_t* min_start;
};

// what clip_plan_kernel leaves for clip_pack_kernel
struct clip_plan {
    int32_t pos;
    uint32_t flag_bin;          // new FLAG | bin << 16
    uint32_t n_cig;             // new number of ops
    uint32_t edit;              // 1 left end clipped, 2 right end clipped (0: the record is copied as it is, FLAG patched)
    int32_t lead, trail;        // the body: ops [lead, trail) between the leading and the trailing H / S ops
    int32_t kl, kr;             // the first and the last body op kept
    uint32_t dl, dr;            // lengths cut off the front of op kl and off the back of op kr
    uint32_t sl, sr;            // the new soft clips' lengths (old S + clipped query bases)
};

struct clip_args {
    const uint8_t* u; const long long* rec; long long n;
    primer_tables t; int n_ref; int tol; int both;
    clip_plan* plan; unsigned long long* size;          // size[n + 1]: the new record sizes, block_size included; size[n] = 0
    const unsigned long long* off;
    uint8_t* out; long long* rec_out;
    unsigned long long* status;         // [0] first record over 65535 ops (~0: none), [1..4] left, right, unmapped, columns,
                                        // [5] first record whose CIGAR the rule does not cover (~0: none)
};

__device__ __forceinline__ int upper_bound(const int32_t* a, int lo, int hi, long long v) {     // first index in [lo, hi) with a[i] > v
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((long long)__ldg(a + mid) <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// inclusive warp scan
__device__ __forceinline__ long long warp_scan(long long v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(FULL, v, o);
        if (lane >= o) v += y;
    }
    return v;
}

__device__ void plan_record(const clip_args& a, long long i, int lane, unsigned long long* acc) {
    const uint8_t* r = a.u + a.rec[i];
    const int32_t tid = (int32_t)ld32(r + BAM_REF_ID);
    const long long p = (int32_t)ld32(r + BAM_POS);
    const uint32_t n_cig = ld16(r + BAM_N_CIGAR_OP), flag = ld16(r + BAM_FLAG);
    const uint8_t* cig = bam_cigar(r);
    const unsigned long long size = 4ull + ld32(r + BAM_BLOCK_SIZE);
    clip_plan pl;
    pl.pos = (int32_t)p; pl.flag_bin = flag | (ld16(r + BAM_BIN) << 16); pl.n_cig = n_cig; pl.edit = 0;
    // the span, whether a match op occurs, where the body begins and ends, whether an op has length 0, how many H / S ops
    long long span = 0;
    bool any_match = false, zero_len = false;
    int lead = -1, trail = -1, n_clip = 0;
    for (uint32_t b = 0; b < n_cig; b += 32) {
        const uint32_t k = b + lane;
        const uint32_t c = k < n_cig ? ld32(cig + 4ull * k) : (uint32_t)OP_S;
        span += ref_len(c);
        any_match |= __any_sync(FULL, op_is_match(c & 15u) && k < n_cig);
        zero_len |= __any_sync(FULL, k < n_cig && (c >> 4) == 0);
        n_clip += __popc(__ballot_sync(FULL, k < n_cig && is_clip(c & 15u)));
        const unsigned body = __ballot_sync(FULL, k < n_cig && !is_clip(c & 15u));
        if (body) {
            if (lead < 0) lead = (int)b + __ffs(body) - 1;
            trail = (int)b + 32 - __clz(body);
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) span += __shfl_xor_sync(FULL, span, o);
    const bool eligible = tid >= 0 && !(flag & 4u) && any_match;
    // the rule's walk is defined for CIGARs as the SAM spec has them: H / S only at the ends, no op of length 0
    if (eligible && (zero_len || n_clip != lead + (int)n_cig - trail)) {
        if (lane == 0) {
            atomicMin(&a.status[5], (unsigned long long)i);
            a.plan[i] = pl;
            a.size[i] = size;
        }
        return;
    }
    const long long q = p + span - 1;
    long long E = 0, S = 0;
    bool left = false, right = false;
    if (eligible && tid < a.n_ref) {
        const int f0 = __ldg(a.t.first + tid), f1 = __ldg(a.t.first + tid + 1);
        if (f1 > f0) {
            const bool rev = flag & 16u;
            if (a.both || !rev) {       // s - t <= p < e: among the primers with s <= p + t the largest e, when it lies behind p
                const int k = upper_bound(a.t.by_start, f0, f1, p + a.tol);
                if (k > f0) { E = __ldg(a.t.max_end + k - 1); left = E > p; }
            }
            if (a.both || rev) {        // s <= q < e + t: among the primers with e > q - t the smallest s, when it lies at or before q
                const int j = upper_bound(a.t.by_end, f0, f1, q - a.tol);
                if (j < f1) { S = __ldg(a.t.min_start + j); right = S <= q; }
            }
        }
    }
    if (left || right) {
        // left: the first match op whose end lies behind E is kept (cut in front when it starts before E); every op before it goes
        int kl = lead; long long l_start = p; uint32_t cl = 0, dl = 0;
        if (left) {
            long long rb = p, qb = 0;
            kl = -1;
            for (int b = lead; b < trail && kl < 0; b += 32) {
                const int k = b + lane;
                const uint32_t c = k < trail ? ld32(cig + 4ull * k) : 0u;
                const long long rl = ref_len(c), ql = query_len(c);
                const long long r_end = rb + warp_scan(rl, lane), q_end = qb + warp_scan(ql, lane);
                const unsigned hit = __ballot_sync(FULL, k < trail && op_is_match(c & 15u) && r_end > E);
                if (hit) {
                    const int src = __ffs(hit) - 1;
                    kl = b + src;
                    const long long kr_start = __shfl_sync(FULL, r_end - rl, src), kq_start = __shfl_sync(FULL, q_end - ql, src);
                    dl = (uint32_t)(kr_start < E ? E - kr_start : 0);
                    l_start = kr_start + dl;
                    cl = (uint32_t)(kq_start + dl);
                }
                rb = __shfl_sync(FULL, r_end, 31); qb = __shfl_sync(FULL, q_end, 31);
            }
        }
        // right: the mirror image, from the end
        int kr = trail - 1; long long r_end_new = q + 1; uint32_t cr = 0, dr = 0;
        if (right) {
            long long re = q + 1, qe = 0;
            kr = -1;
            for (int b = trail - 1; b >= lead && kr < 0; b -= 32) {
                const int k = b - lane;
                const uint32_t c = k >= lead ? ld32(cig + 4ull * k) : 0u;
                const long long rl = ref_len(c), ql = query_len(c);
                const long long r_start = re - warp_scan(rl, lane), q_start = qe + warp_scan(ql, lane);
                const unsigned hit = __ballot_sync(FULL, k >= lead && op_is_match(c & 15u) && r_start < S);
                if (hit) {
                    const int src = __ffs(hit) - 1;
                    kr = b - src;
                    const long long k_end = __shfl_sync(FULL, r_start + rl, src), kq = __shfl_sync(FULL, q_start - ql, src);
                    dr = (uint32_t)(k_end > S ? k_end - S : 0);
                    r_end_new = k_end - dr;
                    cr = (uint32_t)(kq + dr);
                }
                re = __shfl_sync(FULL, r_start, 31); qe = __shfl_sync(FULL, q_start, 31);
            }
        }
        const bool full = kl < 0 || kr < 0 || kl > kr || (kl == kr && l_start >= r_end_new);
        if (full) {
            pl.flag_bin |= 4u;
            if (lane == 0) atomicAdd(&acc[2], 1ull);
        } else {
            uint32_t n_new = (uint32_t)(kr - kl + 1);
            uint32_t sl = 0, sr = 0;
            if (left) {
                for (int k = 0; k < lead; ++k) {
                    const uint32_t c = ld32(cig + 4ull * k);
                    if ((c & 15u) == OP_H) ++n_new; else sl += c >> 4;
                }
                sl += cl;
                n_new += sl > 0;
            } else n_new += (uint32_t)lead;
            if (right) {
                for (int k = trail; k < (int)n_cig; ++k) {
                    const uint32_t c = ld32(cig + 4ull * k);
                    if ((c & 15u) == OP_H) ++n_new; else sr += c >> 4;
                }
                sr += cr;
                n_new += sr > 0;
            } else n_new += n_cig - (uint32_t)trail;
            pl.pos = (int32_t)l_start;
            pl.flag_bin = (pl.flag_bin & 0xffffu) | (reg2bin(l_start, r_end_new) << 16);
            pl.n_cig = n_new;
            pl.edit = (left ? 1u : 0u) | (right ? 2u : 0u);
            pl.lead = lead; pl.trail = trail; pl.kl = kl; pl.kr = kr; pl.dl = dl; pl.dr = dr; pl.sl = sl; pl.sr = sr;
            if (lane == 0) {
                if (n_new > 65535u) atomicMin(&a.status[0], (unsigned long long)i);
                if (left) atomicAdd(&acc[0], 1ull);
                if (right) atomicAdd(&acc[1], 1ull);
                atomicAdd(&acc[3], (unsigned long long)((l_start - p) + (q + 1 - r_end_new)));
            }
        }
    }
    if (lane == 0) {
        a.plan[i] = pl;
        a.size[i] = size + 4ull * pl.n_cig - 4ull * n_cig;
    }
}

__global__ void __launch_bounds__(256) clip_plan_kernel(clip_args a) {
    __shared__ unsigned long long acc[4];           // this block's left, right, fully clipped records and columns
    if (threadIdx.x < 4) acc[threadIdx.x] = 0;
    __syncthreads();
    const long long i = (long long)blockIdx.x * REC_WARPS + (threadIdx.x >> 5);
    if (i < a.n) plan_record(a, i, threadIdx.x & 31, acc);
    __syncthreads();
    if (threadIdx.x < 4 && acc[threadIdx.x]) atomicAdd(&a.status[1 + threadIdx.x], acc[threadIdx.x]);
}

__global__ void __launch_bounds__(256) clip_pack_kernel(clip_args a) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= a.n) return;
    const uint8_t* r = a.u + a.rec[i];
    const unsigned long long o = a.off[i];     // the output record's block_size
    uint8_t* w = a.out + o - BAM_BLOCK_SIZE;
    const clip_plan pl = a.plan[i];
    const uint32_t old_size = 4u + ld32(r + BAM_BLOCK_SIZE);
    if (lane == 0) a.rec_out[i] = (long long)o - BAM_BLOCK_SIZE;
    if (!pl.edit) {
        warp_copy(w + BAM_BLOCK_SIZE, r + BAM_BLOCK_SIZE, old_size, lane);
        __syncwarp();
        if (lane == 0) { w[BAM_FLAG] = (uint8_t)pl.flag_bin; w[BAM_FLAG + 1] = (uint8_t)(pl.flag_bin >> 8); }
        return;
    }
    const uint32_t l_name = r[BAM_L_READ_NAME], n_old = ld16(r + BAM_N_CIGAR_OP);
    const uint8_t* cig = bam_cigar(r);
    const uint32_t new_size = old_size + 4u * pl.n_cig - 4u * n_old;
    // the fixed fields one 32-bit word per lane: 0 block_size, 1 refID, 2 pos, 3 l_read_name | MAPQ | bin, 4 n_cigar_op | FLAG,
    // 5 l_seq, 6 next refID, 7 next pos, 8 tlen.  block_size, pos, bin and n_cigar_op are patched; the rest and the name stay
    if (lane < 9) {
        uint32_t x = ld32(r + BAM_BLOCK_SIZE + 4 * lane);
        if (lane == 0) x = new_size - 4u;
        else if (lane == 2) x = (uint32_t)pl.pos;
        else if (lane == 3) x = (x & 0xffffu) | (pl.flag_bin & 0xffff0000u);
        else if (lane == 4) x = pl.n_cig | (x & 0xffff0000u);
        st32(w + BAM_BLOCK_SIZE + 4 * lane, x);
    }
    for (uint32_t j = lane; j < l_name; j += 32) w[BAM_READ_NAME + j] = r[BAM_READ_NAME + j];
    uint8_t* nc = w + BAM_READ_NAME + l_name;
    // leading section, then the body ops kl..kr (kl cut at its front, kr at its back), then the trailing section
    uint32_t at = 0;
    if (pl.edit & 1u) {
        if (lane == 0)
            for (int k = 0; k < pl.lead; ++k) {
                const uint32_t c = ld32(cig + 4ull * k);
                if ((c & 15u) == OP_H) st32(nc + 4ull * at++, c);
            }
        at = __shfl_sync(FULL, at, 0);
        if (pl.sl) { if (lane == 0) st32(nc + 4ull * at, pl.sl << 4 | OP_S); ++at; }
    } else {
        for (int k = lane; k < pl.lead; k += 32) st32(nc + 4ull * k, ld32(cig + 4ull * k));
        at = (uint32_t)pl.lead;
    }
    for (int k = pl.kl + lane; k <= pl.kr; k += 32) {
        uint32_t c = ld32(cig + 4ull * k);
        uint32_t len = c >> 4;
        if (k == pl.kl) len -= pl.dl;
        if (k == pl.kr) len -= pl.dr;
        st32(nc + 4ull * (at + (uint32_t)(k - pl.kl)), len << 4 | (c & 15u));
    }
    at += (uint32_t)(pl.kr - pl.kl + 1);
    const uint32_t n_old_i = n_old;
    if (pl.edit & 2u) {
        if (pl.sr) { if (lane == 0) st32(nc + 4ull * at, pl.sr << 4 | OP_S); ++at; }
        if (lane == 0)
            for (uint32_t k = (uint32_t)pl.trail; k < n_old_i; ++k) {
                const uint32_t c = ld32(cig + 4ull * k);
                if ((c & 15u) == OP_H) st32(nc + 4ull * at++, c);
            }
    } else {
        for (uint32_t k = (uint32_t)pl.trail + lane; k < n_old_i; k += 32) st32(nc + 4ull * (at + k - (uint32_t)pl.trail), ld32(cig + 4ull * k));
    }
    // SEQ, QUAL and the optional fields as they are
    const uint32_t tail_off = BAM_READ_NAME + l_name + 4u * n_old;
    warp_copy(nc + 4ull * pl.n_cig, r + tail_off, old_size - 4u - tail_off, lane);
}

}  // namespace

TC_API int tc_bam_clip_primers(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                               int32_t n_ref, const int32_t* primer_ref, const int32_t* primer_start, const int32_t* primer_end,
                               int32_t n_primers, int32_t tolerance, uint32_t mode, const uint8_t** payload_dev, int64_t* n_bytes_out,
                               const int64_t** rec_off_dev, tc_clip_stats_t* stats, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!payload_dev || !n_bytes_out || !rec_off_dev || !stats || n_reads < 0 || n_bytes < 0 || n_ref < 0 || n_primers < 0 ||
        tolerance < 0 || (mode & ~1u) || (n_reads > 0 && (!payload || !rec_off)) ||
        (n_primers > 0 && (!primer_ref || !primer_start || !primer_end)))
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n_reads >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 reads in one batch; shard the input");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    memset(stats, 0, sizeof(*stats));
    *payload_dev = payload; *n_bytes_out = n_bytes; *rec_off_dev = rec_off;
    // the primers on the host (rows in device memory are copied on `s`), checked, then the search tables
    const size_t np = (size_t)n_primers;
    std::vector<int32_t> pr(np), ps(np), pe(np);
    if (np) {
        const int32_t* src[3] = {primer_ref, primer_start, primer_end};
        int32_t* dst[3] = {pr.data(), ps.data(), pe.data()};
        bool on_dev = false;
        for (int k = 0; k < 3; ++k) {
            if (tc_is_device_ptr(src[k])) {
                TC_D2H(dst[k], src[k], 4 * np, s);
                on_dev = true;
            } else {
                memcpy(dst[k], src[k], 4 * np);
            }
        }
        if (on_dev) TC_CUDA(cudaStreamSynchronize(s));
    }
    for (size_t k = 0; k < np; ++k)
        if (pr[k] < 0 || pr[k] >= n_ref || ps[k] < 0 || pe[k] <= ps[k])
            return tc_fail(ctx, TC_ERR_ARG, "primer %zu: reference %d of %d, [%d, %d): needs a reference of the header and 0 <= start < end",
                           k, pr[k], n_ref, ps[k], pe[k]);
    const size_t nr = (size_t)n_ref;
    std::vector<int32_t> tab(nr + 1 + 4 * np);
    int32_t* first = tab.data();
    int32_t *by_start = first + nr + 1, *max_end = by_start + np, *by_end = max_end + np, *min_start = by_end + np;
    std::vector<int32_t> idx(np);
    for (size_t k = 0; k < np; ++k) { idx[k] = (int32_t)k; ++first[pr[k] + 1]; }
    for (size_t r = 0; r < nr; ++r) first[r + 1] += first[r];
    std::sort(idx.begin(), idx.end(), [&](int32_t x, int32_t y) { return pr[x] != pr[y] ? pr[x] < pr[y] : ps[x] < ps[y]; });
    for (size_t k = 0; k < np; ++k) {
        const int32_t j = idx[k];
        by_start[k] = ps[j];
        max_end[k] = (k > 0 && (size_t)first[pr[j]] < k) ? std::max(max_end[k - 1], pe[j]) : pe[j];
    }
    std::sort(idx.begin(), idx.end(), [&](int32_t x, int32_t y) { return pr[x] != pr[y] ? pr[x] < pr[y] : pe[x] < pe[y]; });
    for (size_t k = np; k-- > 0;) {
        const int32_t j = idx[k];
        by_end[k] = pe[j];
        min_start[k] = (k + 1 < np && (size_t)first[pr[j] + 1] > k + 1) ? std::min(min_start[k + 1], ps[j]) : ps[j];
    }
    const size_t n = (size_t)n_reads;
    if (n == 0) return TC_OK;
    int rc;
    const uint8_t* u = (const uint8_t*)tc_stage_in(ctx, SLOT_BAM_PAYLOAD, payload, (size_t)n_bytes, s, &rc); if (rc) return rc;
    const long long* rec = (const long long*)tc_stage_in(ctx, SLOT_BAM_REC, rec_off, 8 * n, s, &rc); if (rc) return rc;
    // one work buffer: plans, sizes and offsets (n + 1 each), the status block, the tables
    const size_t plan_b = (sizeof(clip_plan) * n + 15) & ~(size_t)15, size_b = 8 * (n + 1), st_b = 64;
    const size_t tab_b = 4 * tab.size();
    uint8_t* d_work = (uint8_t*)tc_dev_buf(ctx, SLOT_CLIP_PLAN, plan_b + 2 * size_b + st_b + tab_b);
    // the output: every record grows by at most two ops (one soft clip at each end)
    uint8_t* d_out = (uint8_t*)tc_dev_buf(ctx, SLOT_CLIP_PAYLOAD, (size_t)n_bytes + 8 * n + 64);
    long long* d_rec = (long long*)tc_dev_buf(ctx, SLOT_CLIP_REC, 8 * n);
    if (!d_work || !d_out || !d_rec) return TC_ERR_NOMEM;
    clip_args a;
    memset(&a, 0, sizeof(a));
    a.u = u; a.rec = rec; a.n = n_reads; a.n_ref = n_ref; a.tol = tolerance; a.both = (int)(mode & 1u);
    a.plan = (clip_plan*)d_work;
    a.size = (unsigned long long*)(d_work + plan_b);
    unsigned long long* d_off = (unsigned long long*)(d_work + plan_b + size_b);
    a.off = d_off;
    a.status = (unsigned long long*)(d_work + plan_b + 2 * size_b);
    const int32_t* d_tab = (const int32_t*)(d_work + plan_b + 2 * size_b + st_b);
    a.t.first = d_tab; a.t.by_start = d_tab + nr + 1; a.t.max_end = a.t.by_start + np; a.t.by_end = a.t.max_end + np;
    a.t.min_start = a.t.by_end + np;
    a.out = d_out; a.rec_out = d_rec;
    rc = tc_h2d(ctx, (void*)d_tab, tab.data(), tab_b, s); if (rc) return rc;
    TC_CUDA(cudaMemsetAsync(a.size + n, 0, 8, s));
    TC_CUDA(cudaMemsetAsync(a.status, 0, 48, s));
    TC_CUDA(cudaMemsetAsync(a.status, 0xff, 8, s));
    TC_CUDA(cudaMemsetAsync(a.status + 5, 0xff, 8, s));
    const unsigned blocks = (unsigned)((n + REC_WARPS - 1) / REC_WARPS);
    clip_plan_kernel<<<blocks, 32 * REC_WARPS, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, a.size, d_off, (int)(n + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.size, d_off, (int)(n + 1), s));
    ctx->launches++;
    clip_pack_kernel<<<blocks, 32 * REC_WARPS, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    unsigned long long* h = (unsigned long long*)ctx->host_status;
    TC_D2H(h, a.status, 48, s);
    TC_D2H(h + 6, d_off + n, 8, s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (h[5] != ~0ull)
        return tc_fail(ctx, TC_ERR_ARG, "BAM record %llu (of %lld, in input order): the CIGAR has an op of length 0, or an H / S op "
                       "between other ops; primers cannot be clipped off it", h[5], (long long)n_reads);
    if (h[0] != ~0ull)
        return tc_fail(ctx, TC_ERR_ARG, "BAM record %llu (of %lld, in input order): the clipped CIGAR has more than 65535 operations",
                       h[0], (long long)n_reads);
    stats->n_left = (int64_t)h[1]; stats->n_right = (int64_t)h[2]; stats->n_unmapped = (int64_t)h[3]; stats->n_columns = (int64_t)h[4];
    *payload_dev = d_out; *n_bytes_out = (int64_t)h[6]; *rec_off_dev = (const int64_t*)d_rec;
    return TC_OK;
}
