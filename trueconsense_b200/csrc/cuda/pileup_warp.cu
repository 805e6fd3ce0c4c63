// pileup_warp.cu — variant 3 of the pileup kernel: barrier-free, one warp = one stream of reads.
//
// Same bit-parallel idea as variant 2 (pileup_swar.cu): BAM's base codes are one-hot (A=1, C=2, G=4,
// T=8), so once a read's bases sit on the reference grid as 4-bit codes, counting A/C/G/T per column
// is a positional popcount down the reads — a Harley-Seal carry-save tree of LOP3s into bit-sliced
// counters that live in registers.  What changed is everything around it (profiles/r1_v24_swar.md:
// 70 % of variant 2's instructions were divergent CIGAR / shift-change handling, at 8 warps per SM
// behind CTA-wide barriers):
//
//   partition   the start-sorted reads are cut into one contiguous range per warp of the grid (one
//               CTA per SM, all resident); a warp never synchronises with another warp.
//   window      a warp keeps its counters for the 8*WC reference columns [w0, w0 + 8*WC); reads are
//               taken 32 at a time while their starts stay inside [w0, w0 + slack), slack = 8*WC -
//               (longest reference span) - 8, so every column they touch is inside the window.  When a
//               read starts beyond it the counters are flushed to HBM (one red.add per non-zero cell)
//               and the window moves.  Deep data flushes once per thousands of reads.
//   stage       the packed SEQ words and CIGAR ops of the <= 32 reads are contiguous in HBM: one lane requests the two
//               ranges as TMA bulk copies (cp.async.bulk) that complete on the warp's mbarrier — SEQ to its place,
//               the raw CIGAR ops into the rows, idle and all zero at that point — and the next sub-tile's ranges
//               as two bulk L2 prefetches.  Then, in place: SEQ words byte-swapped to "first base in the top
//               nibble", codes that are not one-hot (N, IUPAC) cleared (3 ops per word to detect), CIGAR ops packed
//               to 16 bits (length < 4096 inside a window), the rows cleared again.  (LDG.128 + STS remains for the
//               1024-column geometry and for a batch's last sub-tile.)
//   emit        one lane per read, walk and expansion fused (emit_phase): lanes stay in step on
//               chunks of match ops — the part of an M/=/X op inside CW consecutive 8-column row words —
//               consuming the I / D / S op in front of it first (deletion columns and insertion anchors,
//               sparse, go to packed 64-bit global counters with one red.global.add), then CW + 1 source
//               words, CW funnel shifts under the op's shift D (query index = column + D), head / tail
//               masks, CW red.shared.or into the lane's own row.  Nothing is written to be re-read.
//   phases      the lanes' rows cover 256 columns only (32 x 33 words per warp whatever the window width):
//               a window of 512 / 1024 columns is walked in 2 / 4 PHASES — every lane runs until its read
//               reaches the phase's last column (chunks are cut there), the rows are summed into that
//               phase's counters and cleared, and the walk resumes from the registers it stopped in.  The
//               kernel's speed is proportional to the warps resident per SM (measured: 6 / 8 / 10 / 12
//               warps -> 1.06 / 0.80 / 0.70 / 0.60 ms), shared memory is what limits them, and rows of
//               the full window width were 44 % of a warp's slice.
//   column sum  lane j owns row word j of the phase: 32 rows go through two 16-input carry-save trees
//               into the bit-sliced counters (4 + HI planes per word, in registers across sub-tiles).
//   span pass   when the caller bounds the longest reference span (tc_reads_t.max_ref_span) the kernel also
//               checks sort order and range and adds the two ends of every read's span to the coverage
//               difference array (combined inside the warp with match.any) — no separate pass over the CIGARs.
//   declined    sub-tiles with pads, zero-length ops, or an op of 4096+ bases that matters raise
//               TC_ERR_CAPACITY (such CIGARs are legal and essentially never seen); what runs next is the
//               fallback ladder of tc_pileup_settle (pileup.cu).
#include <limits.h>

#include "pileup_smem.cuh"

namespace {

using namespace tcsm;
constexpr int HI_PLANES = 7;            // bit-sliced planes above "eights": 15 + 16*127 = 2047 reads per run
constexpr int RUN_CAP = 2047;
#ifndef TC_CHUNK_WORDS
#define TC_CHUNK_WORDS 6
#endif
constexpr int CHUNK_WORDS = TC_CHUNK_WORDS;     // row words per emitted chunk of a match op
#ifndef TC_MAX_WARPS
#define TC_MAX_WARPS 24                         // 80 registers per thread (short reads: 24 warps fit the 256-column geometry)
#endif
#ifndef TC_CIG_PER_WC
#define TC_CIG_PER_WC 15
#endif
#ifndef TC_SEQ_PER_WC
#define TC_SEQ_PER_WC 26
#endif
#ifndef TC_TMA_STAGING
#define TC_TMA_STAGING 1                        // 1: sub-tiles are staged with cp.async.bulk (TMA), 0: with LDG.128 + STS
#endif
#ifndef TC_STAGE_UNROLL
#define TC_STAGE_UNROLL 4
#endif
#ifndef TC_PHASE_WORDS
#define TC_PHASE_WORDS 32                       // 32: 256-column phases; 0: one phase (rows as wide as the window)
#endif
#ifndef TC_WALK_STEPS
#define TC_WALK_STEPS 1                         // 1: a D1 / I1 behind a match op takes the walk's short path; 0: the generic op branch
#endif
template <int WC> struct geom {
    static constexpr int ROWW = WC * 8;             // window width in reference columns
    static constexpr int PW = (TC_PHASE_WORDS > 0 && TC_PHASE_WORDS < WC) ? TC_PHASE_WORDS : WC;   // row words (8 columns each) per phase
    static constexpr int NPH = WC / PW;             // phases
    static constexpr int NW = WC / 32;              // window words owned by one lane in the column sum
    static constexpr int RS = PW + 1;               // padded row stride (words)
    static constexpr int SEQ_PAD = 4;               // zero words in front of the staged SEQ stream
    static constexpr int SEQ_CAP = WC * TC_SEQ_PER_WC;   // staged SEQ words per sub-tile (26: WC=64 holds 32 reads of 416 bases; longer reads make shorter sub-tiles)
    static constexpr int CIG_CAP = WC * TC_CIG_PER_WC;   // staged CIGAR ops per sub-tile (16 bits each)
    static constexpr int SEQ_WORDS = SEQ_PAD + SEQ_CAP + 8;
    static constexpr int CIG_WORDS = CIG_CAP / 2 + 4;
    static constexpr int WARP_WORDS = 32 * RS + SEQ_WORDS + CIG_WORDS;
    // + 2 words per warp: its mbarrier (TMA staging)
    static constexpr int WARPS = (227 * 1024 / 4) / (WARP_WORDS + 2) > TC_MAX_WARPS ? TC_MAX_WARPS : (227 * 1024 / 4) / (WARP_WORDS + 2);
    // the raw CIGAR ops of a sub-tile land in the rows (idle while staging) before they are packed to 16 bits
    static constexpr bool TMA = TC_TMA_STAGING && (CIG_CAP + 4 <= 32 * RS);
};

extern __shared__ __align__(16) uint32_t smem[];

// A lane's walk over its read, resumable between phases.
struct lane_walk {
    uint32_t cp, cend;      // shared addresses of the next op and of the end of the read's ops (16 bits each)
    uint32_t c0, c1;        // the next two ops, fetched ahead of their use
    uint32_t prev;          // what the op before the current one was: bit 1 = it consumed the reference, bit 0 = it was a deletion
    int x, y, rem;          // window column, query index, columns left of the match op being emitted
};

// One phase of the walk (no pads, no zero-length ops: those sub-tiles are declined), walk and expansion fused, no
// descriptors.  One lane = one read; lanes are kept in step on CHUNKS of match ops: a chunk is the part of an M/=/X
// op that falls into CW consecutive row words (at most 8 * CW - (x & 7) columns; CW = 6 measured best on ONT-like
// reads, 4 and 8 within 3 %) and in front of the phase's last column xlim.  Per iteration a lane first consumes at
// most one op that is not a match (typically the I or D between two match ops: the sparse X / I events) and starts
// the match op behind it — straight-line code for the common "M I M D M" shape; a second op in a row that is not a
// match (S I, D I, ...) simply waits for the next iteration — then emits one chunk: CW + 1 source words, CW funnel
// shifts under the op's shift D (query index = column + D), head / tail masks, CW red.shared.or into its own row.
// rowp: shared address of the lane's row minus the phase's first word; sq: shared address of the read's first staged
// SEQ word; lq: l_seq (reads without SEQ have had their match ops turned into reference skips).  Returns whether any
// lane did anything (the rows are then summed).
// STEPS: a 1-base D or I right behind a match op (92 % of the match ops of ONT-like reads, profiles/walk_shapes.json) takes
// a short path that sets exactly what the generic branch would, without classifying the op.
template <int ROWW, int CW, bool LIMIT, bool STEPS>
__device__ __forceinline__ bool emit_phase(lane_walk& s, const int lq, const uint32_t rowp, const int xlim,
                                           unsigned long long* xi, const int xi_n, const uint32_t sq, int* err) {
    bool any_iter = false;
    // LIMIT: the phase ends at column xlim (otherwise it runs to the end of the reads and xlim plays no part)
    while (__any_sync(FULL, (s.cp < s.cend || s.rem > 0) && (!LIMIT || s.x < xlim))) {
        any_iter = true;
        if (s.rem == 0 && s.cp < s.cend && (!LIMIT || s.x < xlim)) {
            uint32_t c = s.c0;
            uint32_t fl = op_flags(c & 15u);
            if (!(fl & 1u)) {
                if (STEPS && c - ((1u << 4) | OP_I) < 2u && s.prev == 2u) {
                    // D1 (0x12): +1 X on column x, x + 1; I1 (0x11): +1 I on its anchor x - 1 (a match column), y + 1
                    const uint32_t si = c & 1u;
                    red_xi_if(true, xi, (uint32_t)min(s.x - (int)si, xi_n - 1), si ^ 1u, si);
                    s.x += (int)(si ^ 1u);
                    s.y += (int)si;
                    s.prev = 3u * (si ^ 1u);
                } else {
                    const uint32_t op = c & 15u;
                    const int l = (int)(c >> 4);
                    // X / I events: a deletion's first column counts +1 X; an insertion counts +1 I on its anchor column
                    // x-1 — and -1 X there when that column belongs to a deletion (it reads "*+n..", not "*").  Without
                    // zero-length ops the anchor exists whenever the previous op consumed the reference; a column past
                    // the reference is clamped (such a read is a TC_ERR_RANGE, the counts are void).
                    const bool is_d = (op == OP_D);
                    const bool ev = is_d || (op == OP_I && (s.prev & 2u));
                    const uint32_t col = (uint32_t)min(is_d ? s.x : s.x - 1, xi_n - 1);
                    const uint32_t pd = s.prev & 1u;
                    // one 64-bit add per event: +1 X, +1 I, or "+1 I, -1 X" (2^32 - 1; exact modulo 2^64)
                    red_xi_if(ev, xi, col, is_d ? 1u : 0u - pd, (is_d ? 1u : pd) ^ 1u);
                    if (is_d && l > 1) for (int k = s.x + 1; k < min(s.x + l, xi_n); ++k) red_xi_if(true, xi, (uint32_t)k, 1u, 0u);
                    s.prev = (fl & 2u) | (is_d ? 1u : 0u);
                    if (fl & 2u) s.x += l;
                    if (fl & 4u) s.y += l;
                }
                s.cp += 2;
                c = s.c1;
                fl = op_flags(c & 15u);
            }
            if ((fl & 1u) && s.cp < s.cend) {
                const int l = (int)(c >> 4);
                // beyond the window, or a CIGAR that consumes more query than SEQ holds: the scatter kernel's business
                if (s.x + l > ROWW || s.y + l > lq) { atomicCAS(err, 0, TC_ERR_CAPACITY); s.cp = s.cend; }
                else { s.rem = l; s.cp += 2; }
            }
            s.c0 = lds16(s.cp); s.c1 = lds16(s.cp + 2);
        }
        __syncwarp();           // lanes leave the part above at different points: emit the chunks together
        if (s.rem > 0 && (!LIMIT || s.x < xlim)) {
            const int x = s.x;
            const int kb = x & 7;
            const int cl = LIMIT ? min(min(s.rem, 8 * CW - kb), xlim - x) : min(s.rem, 8 * CW - kb);
            {
                const int q0 = (x - kb) + (s.y - x);                // query index under the first column of row word x >> 3
                const uint32_t src = sq + (uint32_t)((q0 >> 3) << 2);
                const int sh4 = (q0 & 7) << 2;
                uint32_t w[CW + 1];
#pragma unroll
                for (int j = 0; j <= CW; ++j) w[j] = lds(src + 4 * j);
                const int rem4 = 4 * (kb + cl);                     // 4 * columns from the first row word's start to the chunk's end
                const uint32_t ro = rowp + (uint32_t)((x >> 3) << 2);
                reds_or(ro, __funnelshift_l(w[1], w[0], sh4) & (0xffffffffu >> (4 * kb)) & ~__funnelshift_rc(0xffffffffu, 0u, rem4));
                // words behind the chunk's end get an empty mask and are not written
#pragma unroll
                for (int j = 1; j < CW; ++j)
                    reds_or(ro + 4 * j, __funnelshift_l(w[j + 1], w[j], sh4) & ~__funnelshift_rc(0xffffffffu, 0u, max(rem4 - 32 * j, 0)));
            }
            s.x += cl; s.y += cl; s.rem -= cl;
            s.prev = 2u;
        }
    }
    return any_iter;
}

template <int WC, bool PIECES>
__global__ void __launch_bounds__(geom<WC>::WARPS * 32, 1) warp_pileup_kernel(pileup_args a) {
    using G = geom<WC>;
    constexpr int ROWW = G::ROWW, RS = G::RS, NW = G::NW, NPH = G::NPH, PW = G::PW, KW = G::PW / 32;
    const int lane = threadIdx.x & 31;
    const int L = a.L;
    // pieces of a batch the long-read split declined: some records were never written (lr_finish_kernel)
    if (PIECES && a.status->err) return;

    // which geometry handles this batch: the narrowest whose slack is usable (warp_geometry, pileup.cuh)
    // the longest reference span: the caller's bound (tc_reads_t.max_ref_span) or what the span pass found
    // (PIECES: the "reads" are pieces of at most PIECE_COLS columns; the span pass ran over the real reads)
    const bool fold = !PIECES && a.span_hint > 0;   // no span pass ran: this kernel also does its checks and the coverage ends
    const int ms = PIECES ? PIECE_COLS : ((max(fold ? a.span_hint : a.status->max_span, 1) + 7) & ~7);
    // 256-column windows (short reads: half the shared memory per warp, more warps per SM), 512 or 1024
    const int slack32 = (256 - ms - 8) & ~7, slack64 = (512 - ms - 8) & ~7, slack128 = (1024 - ms - 8) & ~7;
    const bool mine = (WC == 32) ? (slack32 >= MIN_SLACK)
                    : (WC == 64) ? (slack32 < MIN_SLACK && slack64 >= MIN_SLACK) : (slack64 < MIN_SLACK);
    if (!mine) return;
    const int slack = (WC == 32) ? slack32 : (WC == 64) ? slack64 : slack128;
    if (slack < MIN_SLACK) {
        if (threadIdx.x == 0 && blockIdx.x == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY);
        return;
    }

    // the warp's slice of shared memory, as shared-window byte addresses
    const uint32_t rows = (uint32_t)__cvta_generic_to_shared(smem) + 4u * (threadIdx.x >> 5) * G::WARP_WORDS;   // [32][RS]
    const uint32_t seq_s = rows + 4u * 32 * RS;                 // seq_s + 4 * SEQ_PAD <-> SEQ word sbase_al
    const uint32_t cig_s = seq_s + 4u * G::SEQ_WORDS;
    for (int i = lane; i < 32 * RS; i += 32) sts(rows + 4 * i, 0u);
    if (lane < G::SEQ_PAD) sts(seq_s + 4 * lane, 0u);
    // the warp's mbarrier sits behind all slices
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(smem) + 4u * G::WARPS * G::WARP_WORDS + 8u * (threadIdx.x >> 5);
    uint32_t tma_parity = 0;
    if (G::TMA && lane == 0) { mbar_init(mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncwarp();

    const int64_t n_reads = PIECES ? a.n_pieces : a.r.n;
    const int64_t n_seq_words = (int64_t)a.r.seq_off[a.r.n];
    const int64_t n_ops_total = PIECES ? 0 : (int64_t)a.r.cigar_off[a.r.n];
    const int64_t gw = (int64_t)blockIdx.x * G::WARPS + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * G::WARPS;
    int64_t r = gw * n_reads / n_warps;
    const int64_t r_end = (gw + 1) * n_reads / n_warps;

    uint32_t ones[NW], twos[NW], fours[NW], eights[NW], hi[NW][HI_PLANES];
#pragma unroll
    for (int j = 0; j < NW; ++j) {
        ones[j] = twos[j] = fours[j] = eights[j] = 0;
#pragma unroll
        for (int p = 0; p < HI_PLANES; ++p) hi[j][p] = 0;
    }
    int w0 = INT_MIN, run_reads = 0;
    const uint32_t row = rows + 4u * lane * RS;
    int prev_pos = (fold && r > 0 && r < r_end) ? a.r.pos[r - 1] : INT_MIN;     // sort-order check across sub-tiles
    int my_max_span = 0, my_zero_span = 0;

    auto flush = [&]() {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NW; ++j) {
            uint32_t planes[4 + HI_PLANES];
            planes[0] = ones[j]; planes[1] = twos[j]; planes[2] = fours[j]; planes[3] = eights[j];
#pragma unroll
            for (int p = 0; p < HI_PLANES; ++p) planes[4 + p] = hi[j][p];
            uint32_t any = 0;
#pragma unroll
            for (int p = 0; p < 4 + HI_PLANES; ++p) any |= planes[p];
            if (any) {
#pragma unroll 4
                for (int bit = 0; bit < 32; ++bit) {
                    if (!((any >> bit) & 1u)) continue;
                    int v = 0;
#pragma unroll
                    for (int p = 0; p < 4 + HI_PLANES; ++p) v |= (int)((planes[p] >> bit) & 1u) << p;
                    const int colr = w0 + 8 * (lane + 32 * j) + (7 - (bit >> 2));
                    const int cls = bit & 3;     // bit 0 A, 1 C, 2 G, 3 T (BAM codes 1,2,4,8)
                    const int crow = cls == 0 ? TC_ROW_A : cls == 1 ? TC_ROW_C : cls == 2 ? TC_ROW_G : TC_ROW_T;
                    if (colr < L) atomicAdd(&a.counts[(size_t)crow * L + colr], v);
                }
            }
            ones[j] = twos[j] = fours[j] = eights[j] = 0;
#pragma unroll
            for (int p = 0; p < HI_PLANES; ++p) hi[j][p] = 0;
        }
        __syncwarp();
    };

    while (r < r_end) {
        const int nmax = (int)min((int64_t)32, r_end - r);
        const bool valid = lane < nmax;
        const int64_t ri = r + (valid ? lane : 0);
        int p, lq, n, nops_lane, y0 = 0;
        bool passes = true, declined = false;
        uint32_t big = 0;               // OR of the staged CIGAR words: >= OP_BIG <=> some op does not fit 16 bits
        uint32_t cs, sq_lane;
        if constexpr (PIECES) {
            // ---- pieces of long reads: one record per lane, gathered through the start-sorted order
            const tc_piece* pc = a.pieces + a.piece_order[ri];
            const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(pc)), m1 = __ldg(reinterpret_cast<const uint4*>(pc) + 1);
            p = (int)m0.x; lq = (int)m1.y; y0 = (int)m1.z;
            passes = p < L;
            const uint32_t so = m0.y, co = m0.z;
            nops_lane = (int)m0.w;
            const int p0 = __shfl_sync(FULL, p, 0);
            const bool fresh = (w0 == INT_MIN);
            if (fresh) w0 = max(p0, 0) & ~7;
            // every piece is staged on its own, as 16-byte vectors from the aligned-down start of its words / ops
            const int sv = (int)(((so & 3u) + m1.x + 3u) >> 2), cv = (int)(((co & 3u) + m0.w + 3u) >> 2);
            int s_inc = valid ? sv : 0, c_inc = valid ? cv : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int ts = __shfl_up_sync(FULL, s_inc, o), tc = __shfl_up_sync(FULL, c_inc, o);
                if (lane >= o) { s_inc += ts; c_inc += tc; }
            }
            const bool inwin = p >= w0 && p - w0 < slack;
            const bool fits = valid && inwin && 4 * s_inc <= G::SEQ_CAP && 4 * c_inc <= G::CIG_CAP;
            const unsigned fm = __ballot_sync(FULL, fits);
            n = (fm == FULL) ? 32 : __ffs(~fm) - 1;
            n = min(n, RUN_CAP - run_reads);
            if (n == 0) {
                const bool inwin0 = __shfl_sync(FULL, (int)inwin, 0) != 0;
                if ((!inwin0 && !fresh) || run_reads >= RUN_CAP) {
                    flush();
                    w0 = INT_MIN; run_reads = 0;
                    continue;
                }
                if (lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY);     // one piece larger than the staging buffers
                r += 1;
                continue;
            }
            const uint32_t sdst = seq_s + 4u * G::SEQ_PAD + 16u * (uint32_t)(s_inc - sv);
            const uint32_t cdst = cig_s + 8u * (uint32_t)(c_inc - cv);
            // TMA staging: every lane asks for its own piece's words and ops as bulk copies (SEQ to its place, the raw ops
            // into the rows) that complete on the warp's mbarrier — the whole gather in flight at once
            const int64_t sb_p = (int64_t)(so & ~3u);
            const bool tma_p = G::TMA && __all_sync(FULL, lane >= n || sb_p + 4ll * sv <= n_seq_words);
            if (tma_p) {
                const int s_tot = __shfl_sync(FULL, s_inc, n - 1), c_tot = __shfl_sync(FULL, c_inc, n - 1);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_expect_tx(mbar, 16u * (uint32_t)(s_tot + c_tot));
                __syncwarp();
                if (lane < n) {
                    tma_bulk_g2s(sdst, a.r.seq4 + sb_p, 16u * (uint32_t)sv, mbar);
                    if (cv > 0) tma_bulk_g2s(rows + 16u * (uint32_t)(c_inc - cv), a.r.cigar + (co & ~3u), 16u * (uint32_t)cv, mbar);
                }
                mbar_wait(mbar, tma_parity);
                tma_parity ^= 1u;
                const uint32_t sbase = seq_s + 4u * G::SEQ_PAD;
                for (int i = lane; i < s_tot; i += 32) {
                    uint4 v = lds4(sbase + 16 * i);
                    if (multibit(v.x) | multibit(v.y) | multibit(v.z) | multibit(v.w)) {
                        v.x = clear_multibit(v.x); v.y = clear_multibit(v.y); v.z = clear_multibit(v.z); v.w = clear_multibit(v.w);
                    }
                    v.x = __byte_perm(v.x, 0, 0x0123); v.y = __byte_perm(v.y, 0, 0x0123);
                    v.z = __byte_perm(v.z, 0, 0x0123); v.w = __byte_perm(v.w, 0, 0x0123);
                    sts4(sbase + 16 * i, v);
                }
                for (int i = lane; i < c_tot; i += 32) {
                    const uint4 v0 = lds4(rows + 16 * i);
                    big |= v0.x | v0.y | v0.z | v0.w;
                    sts2(cig_s + 8 * i, pack_ops(v0.x, v0.y), pack_ops(v0.z, v0.w));
                    sts4(rows + 16 * i, make_uint4(0u, 0u, 0u, 0u));
                }
            } else {
                if (lane < n) {
                    const int64_t sb = (int64_t)(so & ~3u);
                    // a piece's words and ops are a gather (the pieces of a sub-tile come from 32 different reads): the loads
                    // go out four at a time before any of them is consumed — one at a time, their latencies were half of
                    // this kernel's stall samples
                    constexpr int SB = 4;           // loads in flight per lane (8 spill)
                    const bool whole = sb + 4ll * sv <= n_seq_words;        // (the last words of the batch: do not read past the array)
                    for (int v0 = 0; v0 < sv; v0 += SB) {
                        uint4 q[SB];
    #pragma unroll
                        for (int u = 0; u < SB; ++u) {
                            const int v = v0 + u;
                            if (v < sv) {
                                if (whole) q[u] = __ldg(reinterpret_cast<const uint4*>(a.r.seq4 + sb) + v);
                                else {
                                    q[u].x = sb + 4 * v + 0 < n_seq_words ? __ldg(a.r.seq4 + sb + 4 * v + 0) : 0u;
                                    q[u].y = sb + 4 * v + 1 < n_seq_words ? __ldg(a.r.seq4 + sb + 4 * v + 1) : 0u;
                                    q[u].z = sb + 4 * v + 2 < n_seq_words ? __ldg(a.r.seq4 + sb + 4 * v + 2) : 0u;
                                    q[u].w = sb + 4 * v + 3 < n_seq_words ? __ldg(a.r.seq4 + sb + 4 * v + 3) : 0u;
                                }
                            }
                        }
    #pragma unroll
                        for (int u = 0; u < SB; ++u) {
                            const int v = v0 + u;
                            if (v < sv) {
                                if (multibit(q[u].x) | multibit(q[u].y) | multibit(q[u].z) | multibit(q[u].w)) {
                                    q[u].x = clear_multibit(q[u].x); q[u].y = clear_multibit(q[u].y); q[u].z = clear_multibit(q[u].z); q[u].w = clear_multibit(q[u].w);
                                }
                                q[u].x = __byte_perm(q[u].x, 0, 0x0123); q[u].y = __byte_perm(q[u].y, 0, 0x0123);
                                q[u].z = __byte_perm(q[u].z, 0, 0x0123); q[u].w = __byte_perm(q[u].w, 0, 0x0123);
                                sts4(sdst + 16 * v, q[u]);
                            }
                        }
                    }
                    // the piece-CIGAR buffer is padded to whole vectors behind its last op
                    const uint4* csrc = reinterpret_cast<const uint4*>(a.r.cigar + (co & ~3u));
                    for (int v0 = 0; v0 < cv; v0 += 4) {
                        uint4 q[4];
    #pragma unroll
                        for (int u = 0; u < 4; ++u) if (v0 + u < cv) q[u] = __ldg(csrc + v0 + u);
    #pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (v0 + u < cv) {
                                big |= q[u].x | q[u].y | q[u].z | q[u].w;
                                sts2(cdst + 8 * (v0 + u), pack_ops(q[u].x, q[u].y), pack_ops(q[u].z, q[u].w));
                            }
                    }
                }
            }
            __syncwarp();
            cs = cdst + 2u * (co & 3u);
            // an op of 4096+ bases (pileup_long.cu drops leading clips; a trailing one is harmless): set right below
            if (__any_sync(FULL, big >= OP_BIG)) {
                if (lane < n) {
                    bool after_sat = false;
                    for (uint32_t k = 0; k < m0.w; ++k) {
                        const uint32_t c = __ldg(a.r.cigar + co + k), op = c & 15u;
                        if (c >= OP_BIG) {
                            if (op == OP_H) sts16(cs + 2 * k, (1u << 4) | OP_H);
                            else if (op == OP_S) { sts16(cs + 2 * k, S_SATURATED); after_sat = true; }
                            else declined = true;
                        } else if (after_sat && op_flags(op) != 0u) declined = true;       // the query index behind the clip is unknown
                    }
                }
                __syncwarp();
            }
            sq_lane = sdst + 4u * (so & 3u);
        } else {
            // ---- metadata of the next (up to) 32 reads, one per lane
            p = a.r.pos[ri];
            const uint32_t so = a.r.seq_off[ri], so_next = a.r.seq_off[ri + 1];
            const uint32_t co = a.r.cigar_off[ri], co_next = a.r.cigar_off[ri + 1];
            const uint32_t flg = a.r.flag[ri];
            lq = a.r.l_seq[ri];
            passes = !(flg & (a.flag_filter | 4u)) && !(a.ignore_orphans && (flg & 1u) && !(flg & 2u));
            if (a.min_mapq > 0 && a.r.mapq && (int)a.r.mapq[ri] < a.min_mapq) passes = false;
            if (p >= L) {       // starts past the reference: TC_ERR_RANGE (the span pass says so; without one, here) — never walked
                if (fold && valid && passes) atomicCAS(&a.status->err, 0, TC_ERR_RANGE);
                passes = false;
            }
            const int p0 = __shfl_sync(FULL, p, 0);
            const bool fresh = (w0 == INT_MIN);
            if (fresh) w0 = max(p0, 0) & ~7;
            const uint32_t sbase_al = __shfl_sync(FULL, so, 0) & ~3u;
            const uint32_t cbase_al = __shfl_sync(FULL, co, 0) & ~3u;
            const bool inwin = p >= w0 && p - w0 < slack;
            const bool fits = valid && inwin && (so_next - sbase_al + 1 <= (uint32_t)G::SEQ_CAP) && (co_next - cbase_al <= (uint32_t)G::CIG_CAP);
            const unsigned fm = __ballot_sync(FULL, fits);
            n = (fm == FULL) ? 32 : __ffs(~fm) - 1;
            n = min(n, RUN_CAP - run_reads);
            if (n == 0) {
                const bool inwin0 = __shfl_sync(FULL, (int)inwin, 0) != 0;
                if ((!inwin0 && !fresh) || run_reads >= RUN_CAP) {      // the window (or the counters' range) is used up
                    flush();
                    w0 = INT_MIN; run_reads = 0;
                    continue;
                }
                // a negative position (TC_ERR_RANGE), or one read larger than the staging buffers
                if (inwin0 && lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY);
                if (fold && lane == 0) {
                    if (p0 < prev_pos) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
                    if (p0 < 0 && passes) atomicCAS(&a.status->err, 0, TC_ERR_RANGE);
                }
                prev_pos = p0;
                r += 1;
                continue;
            }

            // ---- stage SEQ words [sbase_al, send) and CIGAR ops [cbase_al, cend)
            {
                const uint32_t send = __shfl_sync(FULL, so_next, n - 1) + 1;        // one word of look-ahead for the funnel shift
                const int nv = (int)((send - sbase_al + 3) >> 2);
                const uint32_t cend = __shfl_sync(FULL, co_next, n - 1);
                const int ncv = (int)((cend - cbase_al + 3) >> 2);
                uint32_t dirty = 0;          // dirty: bit t <=> the lane's t-th vector holds a code that is not one-hot
                const uint32_t sdst = seq_s + 4u * G::SEQ_PAD;
                uint32_t exmin = 1u;         // pads and zero-length ops: min over the ops of min((op ^ P), len) is 0 exactly when one is present
                // TMA staging: the two contiguous ranges are requested as bulk copies (SEQ to its place, the raw CIGAR ops
                // into the rows, which are idle and all zero here) — every byte of the sub-tile is in flight at once and no
                // register holds any of it.  (The last sub-tile of a batch, whose vectors may reach past the arrays, and
                // the 1024-column geometry, whose ops do not fit the rows, take the LDG path below.)
                const bool use_tma = G::TMA && (int64_t)sbase_al + 4ll * nv <= n_seq_words && (int64_t)cbase_al + 4ll * ncv <= n_ops_total;
                if (use_tma) {
                    fence_proxy_async();        // the warp's earlier accesses to these buffers come before the copies' writes
                    __syncwarp();
                    if (lane == 0) {
                        mbar_expect_tx(mbar, 16u * (uint32_t)(nv + ncv));
                        tma_bulk_g2s(sdst, a.r.seq4 + sbase_al, 16u * (uint32_t)nv, mbar);
                        if (ncv > 0) tma_bulk_g2s(rows, a.r.cigar + cbase_al, 16u * (uint32_t)ncv, mbar);
                    }
                }
                // the next sub-tile starts where this one ends and is about as large: pull its lines (and the
                // metadata lines two sub-tiles ahead) towards L2 while this one is being processed
                {
                    const int64_t s_lo = ((int64_t)send - 1) & ~3ll, s_len = (int64_t)send - sbase_al;
                    const int64_t c_lo = (int64_t)cend & ~3ll, c_len = (int64_t)cend - cbase_al;
                    if (lane == 0) {        // two bulk prefetches instead of one prefetch instruction per 128-byte line
                        const int64_t sw = min(s_len + 4, n_seq_words - s_lo) & ~3ll, cw = min(c_len + 4, n_ops_total - c_lo) & ~3ll;
                        if (sw > 0) prefetch_l2_bulk(a.r.seq4 + s_lo, (uint32_t)(4 * sw));
                        if (cw > 0) prefetch_l2_bulk(a.r.cigar + c_lo, (uint32_t)(4 * cw));
                    }
                    const int64_t rm = r + n + 64;
                    if (rm < n_reads) {
                        if (lane == 0) prefetch_l2(a.r.pos + rm);
                        if (lane == 1) prefetch_l2(a.r.seq_off + rm);
                        if (lane == 2) prefetch_l2(a.r.cigar_off + rm);
                        if (lane == 3) prefetch_l2(a.r.l_seq + rm);
                        if (lane == 4) prefetch_l2(a.r.flag + rm);
                    }
                }
                if (use_tma) {
                    mbar_wait(mbar, tma_parity);
                    tma_parity ^= 1u;
                    // SEQ in place: one-hot check (codes that are not are cleared at once: rare), first base to the top nibble
                    for (int i = lane; i < nv; i += 32) {
                        uint4 v = lds4(sdst + 16 * i);
                        if (multibit(v.x) | multibit(v.y) | multibit(v.z) | multibit(v.w)) {
                            v.x = clear_multibit(v.x); v.y = clear_multibit(v.y); v.z = clear_multibit(v.z); v.w = clear_multibit(v.w);
                        }
                        v.x = __byte_perm(v.x, 0, 0x0123); v.y = __byte_perm(v.y, 0, 0x0123);
                        v.z = __byte_perm(v.z, 0, 0x0123); v.w = __byte_perm(v.w, 0, 0x0123);
                        sts4(sdst + 16 * i, v);
                    }
                    // CIGAR ops: rows -> 16 bits each in their place; the rows are cleared again
                    for (int i = lane; i < ncv; i += 32) {
                        const uint4 v0 = lds4(rows + 16 * i);
                        exmin = min(exmin, min(min(op_exotic_min(v0.x), op_exotic_min(v0.y)), min(op_exotic_min(v0.z), op_exotic_min(v0.w))));
                        big |= v0.x | v0.y | v0.z | v0.w;
                        sts2(cig_s + 8 * i, pack_ops(v0.x, v0.y), pack_ops(v0.z, v0.w));
                        sts4(rows + 16 * i, make_uint4(0u, 0u, 0u, 0u));
                    }
                } else {
                    if ((int64_t)sbase_al + 4ll * nv <= n_seq_words) {
                        const uint4* src = reinterpret_cast<const uint4*>(a.r.seq4 + sbase_al);
                        int t = 0;
                        constexpr int SU = TC_STAGE_UNROLL;     // vectors in flight per lane
                        for (int i = lane; i < nv; i += 32 * SU, t += SU) {
                            uint4 v[SU];
        #pragma unroll
                            for (int u = 0; u < SU; ++u) if (i + 32 * u < nv) v[u] = __ldg(src + i + 32 * u);
        #pragma unroll
                            for (int u = 0; u < SU; ++u) if (i + 32 * u < nv) {
                                const uint32_t z = multibit(v[u].x) | multibit(v[u].y) | multibit(v[u].z) | multibit(v[u].w);
                                dirty |= (z != 0 ? 1u : 0u) << (t + u);
                                v[u].x = __byte_perm(v[u].x, 0, 0x0123); v[u].y = __byte_perm(v[u].y, 0, 0x0123);
                                v[u].z = __byte_perm(v[u].z, 0, 0x0123); v[u].w = __byte_perm(v[u].w, 0, 0x0123);
                                sts4(sdst + 16 * (i + 32 * u), v[u]);
                            }
                        }
                    } else {            // the last sub-tile of the batch: do not read past the array
                        int t = 0;
                        for (int i = lane; i < nv; i += 32, ++t) {
                            uint32_t w[4];
        #pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int64_t wi = (int64_t)sbase_al + 4 * i + u;
                                w[u] = wi < n_seq_words ? __ldg(a.r.seq4 + wi) : 0u;
                            }
                            const uint32_t z = multibit(w[0]) | multibit(w[1]) | multibit(w[2]) | multibit(w[3]);
                            dirty |= (z != 0 ? 1u : 0u) << t;
        #pragma unroll
                            for (int u = 0; u < 4; ++u) sts(sdst + 16 * i + 4 * u, __byte_perm(w[u], 0, 0x0123));
                        }
                    }
                    // CIGAR ops, packed to 16 bits.  Pads and zero-length ops: min over the ops of min((op ^ P), len) is 0
                    // exactly when one is present
                    if ((int64_t)cbase_al + 4ll * ncv <= n_ops_total) {
                        const uint4* csrc = reinterpret_cast<const uint4*>(a.r.cigar + cbase_al);
                        for (int i = lane; i < ncv; i += 64) {
                            uint4 v0 = __ldg(csrc + i), v1 = make_uint4(16u, 16u, 16u, 16u);
                            const bool b1 = i + 32 < ncv;
                            if (b1) v1 = __ldg(csrc + i + 32);
                            exmin = min(exmin, min(min(op_exotic_min(v0.x), op_exotic_min(v0.y)), min(op_exotic_min(v0.z), op_exotic_min(v0.w))));
                            exmin = min(exmin, min(min(op_exotic_min(v1.x), op_exotic_min(v1.y)), min(op_exotic_min(v1.z), op_exotic_min(v1.w))));
                            big |= v0.x | v0.y | v0.z | v0.w | v1.x | v1.y | v1.z | v1.w;
                            sts2(cig_s + 8 * i, pack_ops(v0.x, v0.y), pack_ops(v0.z, v0.w));
                            if (b1) sts2(cig_s + 8 * (i + 32), pack_ops(v1.x, v1.y), pack_ops(v1.z, v1.w));
                        }
                    } else {
                        for (int i = lane; i < 4 * ncv; i += 32) {
                            const int64_t oi = (int64_t)cbase_al + i;
                            const uint32_t c = oi < n_ops_total ? __ldg(a.r.cigar + oi) : 16u;
                            exmin = min(exmin, op_exotic_min(c));
                            big |= c;
                            sts16(cig_s + 2 * i, c);
                        }
                    }
                }
                declined = exmin == 0u;
                __syncwarp();
                // an op of 4096+ bases (rare: a long clip): hard clips count for nothing, a soft clip saturates (fine when
                // nothing that consumes the query or the reference follows), anything else is declined
                if (__any_sync(FULL, big >= OP_BIG)) {
                    if (lane < n) {
                        bool after_sat = false;
                        for (uint32_t k = co; k < co_next; ++k) {
                            const uint32_t c = __ldg(a.r.cigar + k), op = c & 15u;
                            if (c >= OP_BIG) {
                                if (op == OP_H) sts16(cig_s + 2 * (k - cbase_al), (1u << 4) | OP_H);
                                else if (op == OP_S) { sts16(cig_s + 2 * (k - cbase_al), S_SATURATED); after_sat = true; }
                                else declined = true;
                            } else if (after_sat && op_flags(op) != 0u) declined = true;       // the query index behind the clip is unknown
                        }
                    }
                    __syncwarp();
                }
                // some base is N / IUPAC (rare in real reads): clear those codes — they only count towards coverage.
                // Only the vectors that hold one are revisited, one per lane and iteration.
                while (__any_sync(FULL, dirty != 0)) {
                    if (dirty) {
                        const int t = __ffs(dirty) - 1;
                        dirty &= dirty - 1;
                        const uint32_t q = sdst + 16 * (lane + 32 * t);
                        uint4 v = lds4(q);
                        v.x = clear_multibit(v.x); v.y = clear_multibit(v.y); v.z = clear_multibit(v.z); v.w = clear_multibit(v.w);
                        sts4(q, v);
                    }
                }
                __syncwarp();
            }
            cs = cig_s + 2u * (co - cbase_al);
            nops_lane = (int)(co_next - co);
            sq_lane = seq_s + 4u * G::SEQ_PAD + 4u * (so - sbase_al);
        }
        // ---- walk
        const bool act = lane < n && passes;
        const int nops = act ? nops_lane : 0;
        const int x0 = p - w0;
        const uint32_t sq = act ? sq_lane : seq_s + 4u * G::SEQ_PAD;
        if (!act) cs = cig_s;           // lanes without a read still run the loops' first fetch: keep it inside the slice
        // reads without SEQ ('*': every base reads 'N' — coverage and events only; rare): their match ops become
        // reference skips of the same length, and the walk below needs no special case
        if (__any_sync(FULL, act && lq == 0)) {
            if (act && lq == 0)
                for (int k = 0; k < nops; ++k) {
                    const uint32_t c = lds16(cs + 2 * k);
                    if (op_flags(c & 15u) & 1u) sts16(cs + 2 * k, (c & ~15u) | OP_N);
                }
            __syncwarp();
        }
        // pads, zero-length ops or an over-long op somewhere in the sub-tile: declined (the batch goes to the scatter kernel)
        const bool skip = __any_sync(FULL, declined);
        if (skip && lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY);
        lane_walk st;
        st.cp = cs; st.cend = cs + 2u * (uint32_t)(skip ? 0 : nops);
        st.c0 = lds16(cs); st.c1 = lds16(cs + 2);
        st.prev = 0; st.x = x0; st.y = y0; st.rem = 0;
        // ---- phases: walk up to the phase's last column, then sum the rows into the phase's counters
#pragma unroll
        for (int ph = 0; ph < NPH; ++ph) {
            const int xlim = (ph == NPH - 1) ? INT_MAX : 8 * PW * (ph + 1);      // the last phase runs to the end of the reads
            const bool did = emit_phase<ROWW, CHUNK_WORDS, (NPH > 1), (TC_WALK_STEPS != 0 && !PIECES)>(st, lq, row - 4u * PW * ph, xlim, a.xi + w0, L - w0, sq, &a.status->err);
            __syncwarp();
            if (!did) continue;
            // column sum: lane owns row words lane + 32 k of the phase, all 32 rows
#pragma unroll
            for (int k = 0; k < KW; ++k) {
                const int j = ph * KW + k;
                const uint32_t col = rows + 4u * (lane + 32 * k);
#pragma unroll
                for (int blk = 0; blk < 2; ++blk) {
                    if (blk * 16 < n) {
                        uint32_t xw[16];
#pragma unroll
                        for (int q = 0; q < 16; ++q) { xw[q] = lds(col + 4u * (blk * 16 + q) * RS); sts(col + 4u * (blk * 16 + q) * RS, 0u); }
                        uint32_t twosA, twosB, foursA, foursB, eightsA, eightsB, sixteens;
                        csa(twosA, ones[j], ones[j], xw[0], xw[1]);
                        csa(twosB, ones[j], ones[j], xw[2], xw[3]);
                        csa(foursA, twos[j], twos[j], twosA, twosB);
                        csa(twosA, ones[j], ones[j], xw[4], xw[5]);
                        csa(twosB, ones[j], ones[j], xw[6], xw[7]);
                        csa(foursB, twos[j], twos[j], twosA, twosB);
                        csa(eightsA, fours[j], fours[j], foursA, foursB);
                        csa(twosA, ones[j], ones[j], xw[8], xw[9]);
                        csa(twosB, ones[j], ones[j], xw[10], xw[11]);
                        csa(foursA, twos[j], twos[j], twosA, twosB);
                        csa(twosA, ones[j], ones[j], xw[12], xw[13]);
                        csa(twosB, ones[j], ones[j], xw[14], xw[15]);
                        csa(foursB, twos[j], twos[j], twosA, twosB);
                        csa(eightsB, fours[j], fours[j], foursA, foursB);
                        csa(sixteens, eights[j], eights[j], eightsA, eightsB);
                        uint32_t carry = sixteens;
#pragma unroll
                        for (int pl = 0; pl < HI_PLANES; ++pl) { const uint32_t t = hi[j][pl] & carry; hi[j][pl] ^= carry; carry = t; }
                    }
                }
            }
            __syncwarp();
        }
        const int x_end = st.x;

        // ---- without a span pass: sort order, range, span statistics and the two ends of every read's span in the
        // coverage difference array (adds to the same column are combined inside the warp first)
        if (fold) {
            int pprev = __shfl_up_sync(FULL, p, 1);
            if (lane == 0) pprev = prev_pos;
            if (lane < n && p < pprev) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
            prev_pos = __shfl_sync(FULL, p, n - 1);
            const int span = act ? x_end - x0 : 0;
            const bool bad = act && (p >= L || p + span > L);
            if (bad) atomicCAS(&a.status->err, 0, TC_ERR_RANGE);
            const bool has = act && span > 0 && !bad;
            my_max_span = max(my_max_span, span);
            my_zero_span += (act && span == 0) ? 1 : 0;
            const unsigned g0 = __match_any_sync(FULL, has ? p : -1 - lane);
            if (has && (__ffs(g0) - 1) == lane) atomicAdd(&a.diff[p], __popc(g0));
            const unsigned g1 = __match_any_sync(FULL, has ? p + span : -1 - lane);
            if (has && (__ffs(g1) - 1) == lane) atomicAdd(&a.diff[p + span], -__popc(g1));
        }

        r += n;
        run_reads += n;
    }
    if (run_reads > 0) flush();
    if (fold) {
        my_max_span = __reduce_max_sync(FULL, my_max_span);
        my_zero_span = __reduce_add_sync(FULL, my_zero_span);
        if (lane == 0) {
            if (my_max_span > 0) atomicMax(&a.status->max_span, my_max_span);
            if (my_zero_span > 0) atomicAdd(&a.status->n_zero_span, my_zero_span);
        }
    }
}

}  // namespace

bool tc_pileup_warp_supported(const pileup_args& a) {
    return (((uintptr_t)a.r.seq4 | (uintptr_t)a.r.cigar) & 15u) == 0;
}

template <int WC, bool PIECES>
static int launch_geom(tc_ctx* ctx, const pileup_args& a, cudaStream_t s, int grid = 0) {
    using G = geom<WC>;
    const size_t smem = sizeof(uint32_t) * (size_t)(G::WARP_WORDS + 2) * G::WARPS;
    const uint32_t bit = 1u << ((WC == 32 ? 0 : WC == 64 ? 1 : 2) + (PIECES ? 3 : 0));
    if (!(ctx->warp_attr_set & bit)) {
        TC_CUDA(cudaFuncSetAttribute(warp_pileup_kernel<WC, PIECES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->warp_attr_set |= bit;
    }
    warp_pileup_kernel<WC, PIECES><<<grid > 0 ? grid : ctx->sm_count, G::WARPS * 32, smem, s>>>(a);
    TC_LAUNCH_CHECK();
    return TC_OK;
}

// Without a span bound all geometries are enqueued: each reads the longest reference span the span pass left in
// a.status and returns at once unless it is the one that fits (no host round trip in between).  With the caller's
// bound the host knows which one that is.
int tc_pileup_warp_launch(tc_ctx* ctx, const pileup_args& a, cudaStream_t s, int grid) {
    if (a.span_hint > 0) {
        const int wc = warp_geometry(a.span_hint);
        if (wc == 32) return launch_geom<32, false>(ctx, a, s, grid);
        if (wc == 64) return launch_geom<64, false>(ctx, a, s, grid);
        return launch_geom<128, false>(ctx, a, s, grid);      // (too long for it too: the kernel declines the batch)
    }
    int rc = launch_geom<32, false>(ctx, a, s, grid);
    if (rc) return rc;
    rc = launch_geom<64, false>(ctx, a, s, grid);
    if (rc) return rc;
    return launch_geom<128, false>(ctx, a, s, grid);
}

// pieces of long reads (pileup_long.cu): always the 512-column geometry
int tc_pileup_warp_launch_pieces(tc_ctx* ctx, const pileup_args& a, cudaStream_t s) { return launch_geom<64, true>(ctx, a, s); }
