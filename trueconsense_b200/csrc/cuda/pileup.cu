// pileup.cu — kernel (1) CIGAR-walk pileup and kernel (3) depth.
//
// Replaces htslib's pileup engine + pysam's get_query_sequences + the reference's per-string
// classifier (TrueConsense/indexing.py:100-143).  What one (read, column) pair contributes is
// decided from the CIGAR alone (SURVEY.md Appendix A.3/A.4 boiled down to counters):
//   coverage  every column of every M,=,X,D,N op                     (indexing.py:117)
//   A/T/C/G   M,=,X columns whose 4-bit base code is exactly 1/8/2/4  (indexing.py:120-127)
//   X         D columns, except the last column of a D that is followed by an insertion
//             (that entry reads "*+n..." and is not equal to "*")       (indexing.py:118)
//   I         the last column of an M,=,X,D,N op followed by I (or by P then I)   (indexing.py:130)
// Coverage is not counted per base: the kernel adds +1/-1 at the two ends of every read's
// reference span into a difference array and a scan turns it into the coverage row — that
// is also all of kernel (3).
//
// Variant 1 ("scatter", the north_star's design): reads are cut into chunks of consecutive
// (start-sorted) reads; a CTA stages the counters of the reference window its chunk starts in,
// in shared memory, one warp walks one read with its lanes spread over the columns of each CIGAR
// op (so the shared atomics of a warp hit 32 different banks), and flushes the window to HBM.
#include "pileup.cuh"

#define SC_W      2048      // window columns staged per CTA
#define SC_ROWS   8         // cov(diff), A, T, C, G, X, I, per-entry coverage
#define SC_CHUNK  256       // reads per chunk
#define SC_THREADS 256

template <bool PER_ENTRY_COV>
__global__ void __launch_bounds__(SC_THREADS) pileup_scatter_kernel(pileup_args a, int n_chunks) {
    extern __shared__ int32_t sm[];                               // [SC_ROWS][SC_W]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = SC_THREADS / 32;
    const int L = a.L;
    for (int chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        const int64_t r0 = (int64_t)chunk * SC_CHUNK;
        const int64_t r1 = min(a.r.n, r0 + SC_CHUNK);
        const int base = a.r.pos[r0] & ~31;
        for (int i = threadIdx.x; i < SC_ROWS * SC_W; i += SC_THREADS) sm[i] = 0;
        __syncthreads();

        auto add = [&](int row, int col, int v) {
            int j = col - base;
            if (j >= 0 && j < SC_W) atomicAdd(&sm[row * SC_W + j], v);
            else if (row == 0) atomicAdd(&a.diff[col], v);
            else if (row == 7) atomicAdd(&a.counts[col], v);
            else atomicAdd(&a.counts[(size_t)row * L + col], v);
        };

        for (int64_t r = r0 + warp; r < r1; r += nwarps) {
            if (lane == 0 && r > 0 && a.r.pos[r] < a.r.pos[r - 1]) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
            if (!read_passes(a, r)) continue;
            const int start = a.r.pos[r];
            const uint32_t c0 = a.r.cigar_off[r];
            const int n = (int)(a.r.cigar_off[r + 1] - c0);
            const uint32_t* __restrict__ cig = a.r.cigar + c0;
            const uint32_t* __restrict__ seqw = a.r.seq4 + a.r.seq_off[r];
            const uint8_t* __restrict__ ql = (a.min_bq > 0) ? a.r.qual + 8ull * a.r.seq_off[r] : nullptr;
            const int lq = a.r.l_seq[r];
            if (start < 0 || start >= L) { if (lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_RANGE); continue; }
            int x = start, y = 0;
            for (int k = 0; k < n; ++k) {                         // every lane walks the same ops
                const uint32_t c = cig[k];
                const uint32_t op = c & 15u;
                const int l = (int)(c >> 4);
                if (!op_consumes_ref(op)) {
                    if (op == OP_I || op == OP_S) y += l;
                    continue;
                }
                if (x + l > L) { if (lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_RANGE); break; }
                const int indel = peek_indel(cig, n, k);
                const bool match = op_is_match(op);
                for (int j = lane; j < l; j += 32) {
                    const int col = x + j;
                    const bool last = (j == l - 1);
                    const int q = match ? y + j : y;
                    if (a.min_bq > 0) {                           // pysam pileup_base_qual_skip
                        int qv = (q < lq) ? (int)ql[q] : 0;
                        if (qv < a.min_bq) continue;
                    }
                    if (PER_ENTRY_COV) add(7, col, 1);
                    if (match) {
                        uint32_t code = (q < lq) ? seq_code(seqw, q) : 15u;
                        int row = code_row(code);
                        if (row > 0) add(row, col, 1);
                    } else if (op == OP_D) {
                        if (!(last && indel > 0)) add(TC_ROW_X, col, 1);
                    }
                    if (last && indel > 0) add(TC_ROW_I, col, 1);
                }
                if (match) y += l;
                x += l;
            }
            if (lane == 0) {
                if (!PER_ENTRY_COV && x > start) { add(0, start, 1); add(0, x, -1); }
                if (x == start) atomicAdd(&a.status->n_zero_span, 1);
                atomicMax(&a.status->max_span, x - start);
            }
        }
        __syncthreads();
        // flush the window: coalesced over columns, only non-zero cells touch HBM
        for (int i = threadIdx.x; i < SC_ROWS * SC_W; i += SC_THREADS) {
            int v = sm[i];
            if (v == 0) continue;
            int row = i / SC_W, col = base + (i % SC_W);
            if (row == 0) { if (col <= L) atomicAdd(&a.diff[col], v); }
            else if (row == 7) { if (col < L) atomicAdd(&a.counts[col], v); }
            else if (col < L) atomicAdd(&a.counts[(size_t)row * L + col], v);
        }
        __syncthreads();
    }
}

// Inclusive scan of the difference array into the coverage row, plus its maximum, as two small multi-CTA kernels
// (a single CTA streaming L elements was the largest fixed cost of a small sample):
//   cov_block_kernel   every CTA scans its 4096 columns locally and leaves its total
//   cov_apply_kernel   every CTA adds the totals of the CTAs before it (a handful: L / 4096), tracks the maximum and —
//                      when `xi` is given (variant 3 / 4: packed X | I event counters per column) — unpacks those
//                      into rows X and I of the count table that `cov` is row 0 of.
constexpr int COV_BLOCK = 4096;

__global__ void __launch_bounds__(1024) cov_block_kernel(const int32_t* __restrict__ diff, int32_t* __restrict__ cov, int L,
                                                         int32_t* __restrict__ block_total) {
    __shared__ int warp_sums[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i0 = blockIdx.x * COV_BLOCK + threadIdx.x * 4;
    int v[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) v[t] = (i0 + t < L) ? diff[i0 + t] : 0;
    v[1] += v[0]; v[2] += v[1]; v[3] += v[2];
    int s = v[3];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
    if (lane == 31) warp_sums[warp] = s;
    __syncthreads();
    if (warp == 0) {
        int w = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const int prefix = (warp > 0 ? warp_sums[warp - 1] : 0) + (s - v[3]);
#pragma unroll
    for (int t = 0; t < 4; ++t) if (i0 + t < L) cov[i0 + t] = prefix + v[t];
    if (threadIdx.x == 1023) block_total[blockIdx.x] = prefix + v[3];
}

__global__ void __launch_bounds__(1024) cov_apply_kernel(int32_t* __restrict__ cov, int L, const int32_t* __restrict__ block_total,
                                                         tc_status* status, const unsigned long long* __restrict__ xi) {
    __shared__ int carry_s;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {
        int c = 0;
        for (int b = lane; b < (int)blockIdx.x; b += 32) c += block_total[b];
#pragma unroll
        for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) carry_s = c;
    }
    __syncthreads();
    const int carry = carry_s;
    const int i0 = blockIdx.x * COV_BLOCK + threadIdx.x * 4;
    int vmax = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (i0 + t < L) {
            const int c = cov[i0 + t] + carry;
            cov[i0 + t] = c;
            vmax = max(vmax, c);
            if (xi) {
                const unsigned long long e = xi[i0 + t];
                cov[(size_t)TC_ROW_X * L + i0 + t] = (int32_t)(uint32_t)e;
                cov[(size_t)TC_ROW_I * L + i0 + t] = (int32_t)(uint32_t)(e >> 32);
            }
        }
    }
    for (int o = 16; o; o >>= 1) vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if (lane == 0 && vmax > 0) atomicMax(&status->max_cov, vmax);
}

static int coverage_scan(tc_ctx* ctx, const int32_t* d_diff, int32_t* d_cov, int L, tc_status* d_status, const unsigned long long* xi,
                         cudaStream_t s) {
    const int nb = (L + COV_BLOCK - 1) / COV_BLOCK;
    int32_t* totals = (int32_t*)tc_dev_buf(ctx, SLOT_COV_TOTALS, 4 * (size_t)nb + 16);
    if (!totals) return TC_ERR_NOMEM;
    cov_block_kernel<<<nb, 1024, 0, s>>>(d_diff, d_cov, L, totals);
    TC_LAUNCH_CHECK();
    cov_apply_kernel<<<nb, 1024, 0, s>>>(d_cov, L, totals, d_status, xi);
    TC_LAUNCH_CHECK();
    return TC_OK;
}

// kernel (3) on its own: one thread per read adds its span ends to the difference array
__global__ void depth_diff_kernel(pileup_args a) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.r.n) return;
    if (a.span_out) a.span_out[r] = -1;
    if (r > 0 && a.r.pos[r] < a.r.pos[r - 1]) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
    if (!read_passes(a, r)) return;
    int start = a.r.pos[r];
    if (start < 0 || start >= a.L) { atomicCAS(&a.status->err, 0, TC_ERR_RANGE); return; }
    int span = 0;
    for (uint32_t k = a.r.cigar_off[r]; k < a.r.cigar_off[r + 1]; ++k) {
        uint32_t c = a.r.cigar[k];
        if (op_consumes_ref(c & 15u)) span += (int)(c >> 4);
    }
    if (a.span_out) a.span_out[r] = span;
    if (start + span > a.L) { atomicCAS(&a.status->err, 0, TC_ERR_RANGE); return; }
    if (span > 0) { atomicAdd(&a.diff[start], 1); atomicAdd(&a.diff[start + span], -1); }
    else atomicAdd(&a.status->n_zero_span, 1);
    atomicMax(&a.status->max_span, span);
}


// the same for long CIGARs (hundreds of ops per read): one warp per read, coalesced loads, a warp sum
__global__ void depth_diff_warp_kernel(pileup_args a) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= a.r.n) return;
    const bool passes = read_passes(a, r);
    const int start = a.r.pos[r];
    const bool inside = start >= 0 && start < a.L;
    int span = 0;
    if (passes && inside)
        for (uint32_t k = a.r.cigar_off[r] + lane; k < a.r.cigar_off[r + 1]; k += 32) {
            const uint32_t c = __ldg(a.r.cigar + k);
            if (op_consumes_ref(c & 15u)) span += (int)(c >> 4);
        }
    span = __reduce_add_sync(0xffffffffu, span);
    if (lane != 0) return;
    if (a.span_out) a.span_out[r] = (passes && inside) ? span : -1;
    if (r > 0 && start < a.r.pos[r - 1]) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
    if (!passes) return;
    if (!inside) { atomicCAS(&a.status->err, 0, TC_ERR_RANGE); return; }
    if (start + span > a.L) { atomicCAS(&a.status->err, 0, TC_ERR_RANGE); return; }
    if (span > 0) { atomicAdd(&a.diff[start], 1); atomicAdd(&a.diff[start + span], -1); }
    else atomicAdd(&a.status->n_zero_span, 1);
    atomicMax(&a.status->max_span, span);
}

static void launch_depth_diff(const pileup_args& a, int64_t n_cigar_ops, cudaStream_t s) {
    if (n_cigar_ops > 64 * a.r.n) depth_diff_warp_kernel<<<(unsigned)((a.r.n * 32 + 255) / 256), 256, 0, s>>>(a);
    else depth_diff_kernel<<<(unsigned)((a.r.n + 255) / 256), 256, 0, s>>>(a);
}

template <bool PER_ENTRY_COV>
static int launch_scatter(tc_ctx* ctx, const pileup_args& a, cudaStream_t s) {
    const int n_chunks = (int)((a.r.n + SC_CHUNK - 1) / SC_CHUNK);
    const size_t smem = sizeof(int32_t) * SC_ROWS * SC_W;
    TC_CUDA(cudaFuncSetAttribute(pileup_scatter_kernel<PER_ENTRY_COV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pileup_scatter_kernel<PER_ENTRY_COV><<<min(n_chunks, ctx->sm_count * 3), SC_THREADS, smem, s>>>(a, n_chunks);
    TC_LAUNCH_CHECK();
    return TC_OK;
}

// timing on: the events around the pileup kernel (inside a graph capture they become external event nodes)
static cudaError_t timing_event(tc_ctx* ctx, cudaEvent_t e, cudaStream_t s) {
    return ctx->timing ? cudaEventRecordWithFlags(e, s, ctx->in_capture ? cudaEventRecordExternal : cudaEventRecordDefault) : cudaSuccess;
}

static int fetch_status(tc_ctx* ctx, tc_status* d_status, tc_status* out, cudaStream_t s) {
    TC_D2H(ctx->host_status, d_status, sizeof(tc_status), s);
    TC_CUDA(cudaStreamSynchronize(s));
    memcpy(out, ctx->host_status, sizeof(tc_status));
    return TC_OK;
}

static int status_to_rc(tc_ctx* ctx, const tc_status& st, const tc_pileup_params_t* p) {
    if (st.err == TC_ERR_UNSORTED) return tc_fail(ctx, TC_ERR_UNSORTED, "Unsorted input. Pileup aborts");
    if (st.err == TC_ERR_RANGE) return tc_fail(ctx, TC_ERR_RANGE, "a read starts or ends outside [0, ref_len)");
    if (st.err) return tc_fail(ctx, st.err, "device-side failure %d", st.err);
    // htslib drops reads at push time once more than max_depth are live (bam_plp_set_maxcnt).  The bulk
    // kernels do not emulate that order-dependent rule; they prove it cannot bind instead: at any push
    // the live set is within the reads covering the previous column plus those starting at this one.
    if (p->max_depth > 0 && 2ll * st.max_cov + st.n_zero_span + 1 > p->max_depth)
        return tc_fail(ctx, TC_ERR_DEPTH_CAP, "coverage %d could reach max_depth %lld: the pileup depth cap may bind and is not emulated by the bulk kernel",
                       st.max_cov, (long long)p->max_depth);
    return TC_OK;
}

static int check_common(tc_ctx* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p, const void* out) {
    if (!ctx) return TC_ERR_ARG;
    if (!reads || !p || !out) return tc_fail(ctx, TC_ERR_ARG, "NULL argument");
    if (ref_len <= 0) return tc_fail(ctx, TC_ERR_ARG, "ref_len must be positive");
    return TC_OK;
}

// A pass's filters, and its status block and coverage difference array [L + 1] in one buffer under one memset.  with_xi (the
// pileup): behind them the packed X | I event counters of variants 3 / 4, one 64-bit word per column.
static int init_pass(tc_ctx* ctx, const tc_pileup_params_t* p, int32_t L, bool with_xi, cudaStream_t s, pileup_args& a) {
    const size_t diff_words = ((size_t)L + 2) & ~(size_t)1;        // keeps the X | I words 8-byte aligned
    const size_t bytes = sizeof(tc_status) + sizeof(int32_t) * diff_words + (with_xi ? 8 * ((size_t)L + 1) : 0);
    uint8_t* head = (uint8_t*)tc_dev_buf(ctx, SLOT_DIFF, bytes);
    if (!head) return TC_ERR_NOMEM;
    TC_CUDA(cudaMemsetAsync(head, 0, bytes, s));
    a.status = (tc_status*)head;
    a.diff = (int32_t*)(head + sizeof(tc_status));
    a.xi = with_xi ? (unsigned long long*)(a.diff + diff_words) : nullptr;
    a.L = L; a.flag_filter = p->flag_filter; a.min_mapq = p->min_mapq; a.min_bq = p->min_base_quality; a.ignore_orphans = p->ignore_orphans;
    return TC_OK;
}

// The plan of one attempt.  rung 0: p->kernel, and for 0 the scatter kernel under a base-quality filter or with seq4 / cigar not
// 16-byte aligned, else variant 4 when the caller's span bound fits no window of variant 3, else variant 3.  rung 3 / 4 / 1 (the
// fallback ladder, tc_pileup_settle): that variant.  Coverage ends, span statistics and the sortedness / range checks take a span
// pass, one thread per read, unless variant 3 does them while it walks the CIGARs (the caller's bound fits its windows).
static int pileup_plan_of(tc_ctx* ctx, const tc_pileup_params_t* p, const pileup_args& a, int rung, pileup_plan* plan) {
    const bool per_entry = p->min_base_quality > 0, fits = a.span_hint > 0 && warp_geometry(a.span_hint) != 0;
    int v = rung ? rung : p->kernel;
    if (v == 0) v = (per_entry || !tc_pileup_warp_supported(a)) ? 1 : (a.span_hint > 0 && !fits) ? 4 : 3;
    if (v != 1 && v != 3 && v != 4) return tc_fail(ctx, TC_ERR_ARG, "unknown pileup kernel variant %d", v);
    if (v != 1 && per_entry) return tc_fail(ctx, TC_ERR_ARG, "the bit-parallel kernels have no base-quality filter; use kernel=1");
    if (v != 1 && !tc_pileup_warp_supported(a)) return tc_fail(ctx, TC_ERR_ARG, "the bit-parallel kernels need 16-byte aligned seq4 / cigar arrays; use kernel=1");
    *plan = {v, v == 4 || (v == 3 && !fits), v == 4};
    return TC_OK;
}

// Everything of one attempt up to (not including) the read-back of the status block: memsets, the span pass if the plan has
// one, the pileup kernel, the coverage scan.  `counts` may be a host pointer (the table is then built in a context buffer).
int tc_pileup_enqueue(tc_ctx* ctx, const tc_reads_t* reads, int32_t L, const tc_pileup_params_t* p, int32_t* counts, cudaStream_t s,
                      tc_pileup_pending* pend, int rung, int grid) {
    const bool per_entry = p->min_base_quality > 0;
    pileup_args a = {};
    int rc = tc_resolve_reads(ctx, reads, &a.r, per_entry ? NEED_QUAL : 0, s);
    if (rc) return rc;
    const bool out_dev = tc_is_device_ptr(counts);
    int32_t* d_counts = out_dev ? counts : (int32_t*)tc_dev_buf(ctx, SLOT_COUNTS, sizeof(int32_t) * TC_NROWS * (size_t)L);
    if (!d_counts) return TC_ERR_NOMEM;
    TC_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(int32_t) * TC_NROWS * (size_t)L, s));
    rc = init_pass(ctx, p, L, true, s, a);
    if (rc) return rc;
    a.counts = d_counts;
    a.span_hint = reads->max_ref_span > 0 ? reads->max_ref_span : 0;
    pileup_plan plan;
    rc = pileup_plan_of(ctx, p, a, rung, &plan);
    if (rc) return rc;
    if (a.r.n > 0) {
        TC_CUDA(timing_event(ctx, ctx->ev0, s));
        if (plan.span_pass) {
            a.span_hint = 0;        // variant 3 reads the longest span the pass leaves in the status block
            a.span_out = plan.span_out ? (int32_t*)tc_dev_buf(ctx, SLOT_SPAN_END, sizeof(int32_t) * (size_t)a.r.n) : nullptr;
            if (plan.span_out && !a.span_out) return TC_ERR_NOMEM;
            launch_depth_diff(a, reads->n_cigar_ops, s);
            TC_LAUNCH_CHECK();
        }
        rc = plan.variant == 4 ? tc_pileup_long_launch(ctx, a, s)
           : plan.variant == 3 ? tc_pileup_warp_launch(ctx, a, s, grid)
           : per_entry ? launch_scatter<true>(ctx, a, s) : launch_scatter<false>(ctx, a, s);
        if (rc) return rc;
        TC_CUDA(timing_event(ctx, ctx->ev1, s));
        if (ctx->timing) ctx->ev_valid = 1;
    }
    rc = per_entry ? TC_OK : coverage_scan(ctx, a.diff, d_counts, L, a.status, plan.variant != 1 ? a.xi : nullptr, s);
    if (rc) return rc;
    pend->d_status = a.status; pend->d_counts = d_counts; pend->plan = plan; pend->out_dev = out_dev ? 1 : 0; pend->n_reads = a.r.n;
    return TC_OK;
}

// one attempt enqueued and read back: the table when the caller's is on the host, then the status block
static int pileup_attempt(tc_ctx* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p, int32_t* counts,
                          cudaStream_t s, int rung, tc_pileup_pending* pend, tc_status* st) {
    int rc = tc_pileup_enqueue(ctx, reads, ref_len, p, counts, s, pend, rung);
    if (rc) return rc;
    if (!pend->out_dev) TC_D2H(counts, pend->d_counts, sizeof(int32_t) * TC_NROWS * (size_t)ref_len, s);
    return fetch_status(ctx, pend->d_status, st, s);
}

// The host side of a pileup once its status block has come back.  With kernel == 0 a batch the bit-parallel kernels decline
// (TC_ERR_CAPACITY) goes down the fallback ladder, each rung enqueued, read back and settled in turn:
//   3 -> 4   the span pass (no bound was given) found a read too long for every window of variant 3: cut into pieces
//   3 -> 1   anything else variant 3 declines (pads, zero-length ops, an op of 4096+ bases, a read beyond the staging buffers)
//   4 -> 1   anything the long-read split or its pieces decline; the scatter kernel (1) carries htslib's full look-ahead state
// Then, for the attempt that went through: errors, the depth-cap proof and the caller's span bound.
int tc_pileup_settle(tc_ctx* ctx, tc_status st, tc_pileup_pending pend, const tc_reads_t* reads, int32_t ref_len,
                     const tc_pileup_params_t* p, int32_t* counts, cudaStream_t s, int* redone) {
    while (st.err == TC_ERR_CAPACITY && p->kernel == 0 && pend.plan.variant != 1) {
        const int next = (pend.plan.variant == 3 && pend.plan.span_pass && warp_geometry(st.max_span) == 0) ? 4 : 1;
        if (redone) *redone = 1;
        int rc = pileup_attempt(ctx, reads, ref_len, p, counts, s, next, &pend, &st);
        if (rc == TC_ERR_CAPACITY && next == 4) rc = pileup_attempt(ctx, reads, ref_len, p, counts, s, 1, &pend, &st);   // too many pieces
        if (rc) return rc;
    }
    if (st.err == TC_ERR_CAPACITY)
        return tc_fail(ctx, TC_ERR_CAPACITY, "a read exceeds the bit-parallel kernels' windows or staging buffers; use kernel=1 (or 0)");
    if (p->min_base_quality > 0) {
        // coverage was counted entry by entry, so max_cov is not the live depth; fall back to the
        // trivial bound (every read live at once)
        st.max_cov = 0;
        if (p->max_depth > 0 && pend.n_reads + 1 > p->max_depth && st.err == 0)
            return tc_fail(ctx, TC_ERR_DEPTH_CAP, "%lld reads with a base-quality filter: the depth cap %lld may bind and is not emulated by the bulk kernel",
                           (long long)pend.n_reads, (long long)p->max_depth);
    }
    if (st.err == 0 && reads->max_ref_span > 0 && st.max_span > reads->max_ref_span)
        return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t.max_ref_span = %d but a read spans %d reference columns", reads->max_ref_span, st.max_span);
    const int rc = status_to_rc(ctx, st, p);
    // a flag filter hides reads from this pass: the bound then only holds for the reads that passed, not for another pass's
    if (rc == TC_OK && reads->max_ref_span > 0 && (p->flag_filter & ~4u) == 0 && p->min_mapq <= 0 && !p->ignore_orphans) {
        ctx->span_ok_cigar = reads->cigar; ctx->span_ok_off = reads->cigar_off; ctx->span_ok_n = reads->n_reads;
        ctx->span_ok_ops = reads->n_cigar_ops; ctx->span_ok_bound = reads->max_ref_span;
    }
    return rc;
}

TC_API int tc_pileup_counts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p,
                            int32_t* counts, void* stream) {
    int rc = check_common(ctx, reads, ref_len, p, counts);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    tc_pileup_pending pend; tc_status st;
    rc = pileup_attempt(ctx, reads, ref_len, p, counts, s, 0, &pend, &st);
    if (rc) return rc;
    return tc_pileup_settle(ctx, st, pend, reads, ref_len, p, counts, s, nullptr);
}

TC_API int tc_depth(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t L, const tc_pileup_params_t* p,
                    int32_t* depth, void* stream) {
    int rc = check_common(ctx, reads, L, p, depth);
    if (rc) return rc;
    if (p->min_base_quality > 0) return tc_fail(ctx, TC_ERR_ARG, "tc_depth counts whole spans; it is only the coverage column when min_base_quality == 0");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    pileup_args a = {};
    // the depth pass reads pos, flag, mapq and the CIGARs only
    dreads& d = a.r;
    d.n = reads->n_reads;
    if (d.n > 0) {
        if (!reads->pos || !reads->flag || !reads->cigar_off || (!reads->cigar && reads->n_cigar_ops)) return tc_fail(ctx, TC_ERR_ARG, "tc_reads_t: a required array is NULL");
        d.pos = (const int32_t*)tc_stage_in(ctx, SLOT_POS, reads->pos, 4 * (size_t)d.n, s, &rc); if (rc) return rc;
        d.flag = (const uint16_t*)tc_stage_in(ctx, SLOT_FLAG, reads->flag, 2 * (size_t)d.n, s, &rc); if (rc) return rc;
        d.cigar_off = (const uint32_t*)tc_stage_in(ctx, SLOT_CIGOFF, reads->cigar_off, 4 * (size_t)(d.n + 1), s, &rc); if (rc) return rc;
        d.cigar = (const uint32_t*)tc_stage_in(ctx, SLOT_CIGAR, reads->cigar, 4 * (size_t)reads->n_cigar_ops, s, &rc); if (rc) return rc;
        if (reads->mapq) { d.mapq = (const uint8_t*)tc_stage_in(ctx, SLOT_MAPQ, reads->mapq, (size_t)d.n, s, &rc); if (rc) return rc; }
    }
    const bool out_dev = tc_is_device_ptr(depth);
    int32_t* d_depth = out_dev ? depth : (int32_t*)tc_dev_buf(ctx, SLOT_COUNTS, sizeof(int32_t) * (size_t)L);
    if (!d_depth) return TC_ERR_NOMEM;
    rc = init_pass(ctx, p, L, false, s, a);
    if (rc) return rc;
    if (d.n > 0) {
        launch_depth_diff(a, reads->n_cigar_ops, s);
        TC_LAUNCH_CHECK();
    }
    rc = coverage_scan(ctx, a.diff, d_depth, L, a.status, nullptr, s);
    if (rc) return rc;
    if (!out_dev) TC_D2H(depth, d_depth, sizeof(int32_t) * (size_t)L, s);
    tc_status st;
    rc = fetch_status(ctx, a.status, &st, s);
    if (rc) return rc;
    return status_to_rc(ctx, st, p);
}
