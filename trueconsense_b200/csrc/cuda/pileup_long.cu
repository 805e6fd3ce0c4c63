// pileup_long.cu — long reads for pileup variant 3.
//
// The warp kernel (pileup_warp.cu) keeps a read's whole alignment inside one 512- or 1024-column window, so a
// read may span at most ~950 reference columns.  Longer reads (10-kb long reads, BASELINE config 5) are cut
// into PIECES here: the reference is divided into cells of PIECE_COLS columns and the part of an alignment
// inside one cell becomes a piece that looks like a short read —
//     position, the SEQ word holding its first query base (+ the base's index inside that word), the query
//     length left from there, and its own CIGAR: the read's ops over the cell, the op crossing a cell border
//     split in two.  Ops that consume no reference (I, S, H) stay with the piece of the reference-consuming op in
//     front of them, so "an insertion counts on the last column before it" never looks across a cut.
// SEQ is not copied: pieces point into the read's own packed bases.  Pieces are then ordered by start column
// (cub radix sort) and the same kernel runs over them in its PIECES mode (records gathered through the order,
// every piece staged on its own).  Coverage, span statistics and the sort / range checks come from the span
// pass over the real reads, as always.
//
//   lr_count_kernel   one thread per read: pieces and piece-CIGAR ops the read will produce (from its span, which the
//                     span pass left behind)
//   exclusive sums    cub::DeviceScan -> where each read's pieces / ops go
//   lr_split_kernel   one warp per read, one lane per segment of ops: piece CIGARs and the records of the pieces' starts
//   lr_finish_kernel  one thread per piece: its op / SEQ word counts (it ends where the next piece starts)
//   radix sort        piece start columns -> processing order
//   warp_pileup_kernel<64, PIECES>
// Reads with pads, zero-length ops or no SEQ are not cut: TC_ERR_CAPACITY (the fallback ladder: tc_pileup_settle, pileup.cu).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "pileup.cuh"

namespace {

__device__ __forceinline__ int ref_span_of(const pileup_args& a, int64_t r) {
    int span = 0;
    for (uint32_t k = a.r.cigar_off[r]; k < a.r.cigar_off[r + 1]; ++k) {
        const uint32_t c = a.r.cigar[k];
        if (op_consumes_ref(c & 15u)) span += (int)(c >> 4);
    }
    return span;
}

// pieces per read = cells its span touches; ops per read <= its own ops + one extra per cut, padded to whole
// 16-byte vectors per piece (+3 ops each) so that a piece's ops can be staged as vectors
__global__ void lr_count_kernel(pileup_args a, uint32_t* __restrict__ n_pieces, uint32_t* __restrict__ n_ops) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.r.n) return;
    uint32_t np = 0, no = 0;
    const int pos = a.r.pos[r];
    if (read_passes(a, r) && pos >= 0 && pos < a.L) {
        const int span = a.span_out ? a.span_out[r] : ref_span_of(a, r);      // the span pass has walked the CIGARs already
        if (span > 0) {
            np = (uint32_t)((pos + span - 1) / PIECE_COLS - pos / PIECE_COLS + 1);
            no = (a.r.cigar_off[r + 1] - a.r.cigar_off[r]) + np * 8u;      // + cut ops, vector padding, alignment slack
        }
    }
    n_pieces[r] = np;
    n_ops[r] = (no + 3u) & ~3u;
}

// One warp per read, one lane per SEGMENT of consecutive ops (1/32 of the read's ops, between LR_SEG_MIN and LR_SEG_MAX) (a thread walking the 600 ops of a 10-kb read alone
// is a serial chain: 0.39 ms for 49 k reads, however its loads are arranged).  Three short walks per lane:
//   sums    reference / query bases and emitted ops of the segment     -> warp scan: (x, y) at the segment's first op
//   cuts    cell borders strictly inside the segment's ops (each adds an op) -> warp scan: the segment's first op slot
//   emit    the segment's piece-CIGAR ops and the records of the pieces that OPEN in it (start column, first SEQ word,
//           first op slot).  A piece ends where the next one starts, possibly in another lane's segment: its op and SEQ
//           word counts are filled in by lr_finish_kernel from the next piece's record (or the read's end state).
// Clips in front of the first aligned base are dropped (a soft clip only moves the query index), so pieces never carry an
// over-long leading clip into the pileup kernel's 16-bit op staging.
constexpr int LR_SEG_MAX = 64;       // ops per lane and round at most (2048 ops per round); shorter CIGARs are spread over all 32 lanes
constexpr int LR_SEG_MIN = 4;
constexpr int LR_WARPS = 4;
constexpr uint32_t LR_PAD_OP = 0x10u | OP_H;        // a no-op hard clip

__global__ void __launch_bounds__(LR_WARPS * 32) lr_split_kernel(pileup_args a, const uint32_t* __restrict__ piece_base, const uint32_t* __restrict__ ops_base,
                                tc_piece* __restrict__ pieces, uint32_t* __restrict__ pcig, int32_t* __restrict__ piece_pos,
                                uint32_t* __restrict__ end_w, uint32_t* __restrict__ end_y) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * LR_WARPS + (threadIdx.x >> 5);
    if (r >= a.r.n) return;                                     // whole warps leave together
    if (piece_base[r + 1] == piece_base[r]) return;
    const int lq = a.r.l_seq[r];
    if (lq == 0) { if (lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY); return; }        // SEQ '*': scatter kernel only
    const uint32_t sbeg = a.r.seq_off[r];
    const uint32_t k0 = a.r.cigar_off[r], k1 = a.r.cigar_off[r + 1];
    const int pos = a.r.pos[r];
    const int first_cell = pos / PIECE_COLS;
    const uint32_t pbase = piece_base[r], wbase = ops_base[r];
    const uint32_t* __restrict__ cig = a.r.cigar;
    int cx = pos, cy = 0;               // state in front of the round's first op (the same in every lane)
    uint32_t cw = wbase;
    const uint32_t seg = min((uint32_t)LR_SEG_MAX, max((uint32_t)LR_SEG_MIN, (k1 - k0 + 31u) / 32u));
    for (uint32_t kr = k0; kr < k1; kr += 32u * seg) {
        const uint32_t s0 = min(kr + (uint32_t)lane * seg, k1), s1 = min(s0 + seg, k1);
        // ---- sums; the read's leading clips (only in front of the very first op that is not a clip) are dropped
        uint32_t lead = 0;              // dropped ops at the start of this segment
        int ref = 0, qry = 0, emitted = 0, lead_qry = 0;      // lead_qry: bases of the dropped soft clips
        bool bad = false;
        {
            bool leading = (s0 == k0);
            for (uint32_t k = s0; k < s1; ++k) {
                const uint32_t c = __ldg(cig + k), op = c & 15u;
                const int l = (int)(c >> 4);
                if (op == OP_P || l == 0 || op > OP_X) bad = true;
                if (leading && (op == OP_H || op == OP_S)) { ++lead; if (op == OP_S) lead_qry += l; } else { leading = false; ++emitted; }
                if (op_consumes_ref(op)) ref += l;
                if (op_is_match(op) || op == OP_I || op == OP_S) qry += l;
            }
            // a read whose whole first segment is clips: not worth a general rule
            if (s0 == k0 && lead == s1 - s0 && s1 < k1) bad = true;
        }
        if (__any_sync(FULL, bad)) { if (lane == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY); return; }      // pads, zero-length ops: scatter kernel only
        int xs = ref, ys = qry;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int tx = __shfl_up_sync(FULL, xs, o), ty = __shfl_up_sync(FULL, ys, o);
            if (lane >= o) { xs += tx; ys += ty; }
        }
        const int tot_ref = __shfl_sync(FULL, xs, 31), tot_qry = __shfl_sync(FULL, ys, 31);
        xs = cx + xs - ref; ys = cy + ys - qry;         // exclusive
        // ---- cuts: cell borders strictly inside an op of the segment
        int cuts = 0;
        {
            int x = xs;
            for (uint32_t k = s0; k < s1; ++k) {
                const uint32_t c = __ldg(cig + k), op = c & 15u;
                if (op_consumes_ref(op)) {
                    const int l = (int)(c >> 4);
                    cuts += (x + l - 1) / PIECE_COLS - x / PIECE_COLS;
                    x += l;
                }
            }
        }
        int ws = emitted + cuts;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, ws, o);
            if (lane >= o) ws += t;
        }
        const int tot_out = __shfl_sync(FULL, ws, 31);
        uint32_t w = cw + (uint32_t)(ws - emitted - cuts);
        // ---- emit
        if (s0 < s1) {
            int x = xs, y = ys + lead_qry;
            bool open = w > wbase;                      // something was emitted before: a piece is open
            bool has_ref = x > pos;
            int cell_end = (has_ref && x % PIECE_COLS == 0) ? x : (x / PIECE_COLS + 1) * PIECE_COLS;     // a cut is pending on a border
            auto open_piece = [&]() {
                tc_piece pc;
                const int yw = y >> 3;
                const uint32_t pi = pbase + (uint32_t)(x / PIECE_COLS - first_cell);
                pc.pos = x; pc.seq_beg = sbeg + (uint32_t)yw; pc.cig_beg = w; pc.cig_n = 0; pc.seq_n = 0;
                pc.lq = lq - 8 * yw; pc.y0 = y & 7; pc.pad = (int32_t)r;     // the read, for lr_finish_kernel
                pieces[pi] = pc;
                piece_pos[pi] = x;
                open = true;
            };
            for (uint32_t k = s0 + lead; k < s1; ++k) {
                const uint32_t c = __ldg(cig + k), op = c & 15u;
                int l = (int)(c >> 4);
                if (!op_consumes_ref(op)) {
                    // I / S / H stay with the piece of the reference-consuming op in front of them; a leading
                    // insertion opens the first piece
                    if (!open) open_piece();
                    pcig[w++] = c;
                    if (op == OP_I || op == OP_S) y += l;
                    continue;
                }
                const bool match = op_is_match(op);
                while (l > 0) {
                    if (x == cell_end) {            // the next column belongs to the next cell: cut here
                        if (open && has_ref) { open = false; has_ref = false; }
                        cell_end += PIECE_COLS;
                    }
                    if (!open) open_piece();
                    const int take = min(l, cell_end - x);
                    pcig[w++] = ((uint32_t)take << 4) | op;
                    has_ref = true;
                    x += take; l -= take;
                    if (match) y += take;
                }
            }
            if (s1 == k1) {                                   // the read's last segment: its end state, and padding behind its ops
                end_w[r] = w; end_y[r] = (uint32_t)y;
                pcig[w] = LR_PAD_OP; pcig[w + 1] = LR_PAD_OP; pcig[w + 2] = LR_PAD_OP;
            }
        }
        cx += tot_ref; cy += tot_qry; cw += (uint32_t)tot_out;
    }
}

// op and SEQ word counts of every piece: it ends where the next piece of its read starts, or with the read
__global__ void lr_finish_kernel(pileup_args a, const uint32_t* __restrict__ piece_base, tc_piece* __restrict__ pieces, int64_t n_pieces,
                                 const uint32_t* __restrict__ end_w, const uint32_t* __restrict__ end_y) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pieces) return;
    // a read the split declined (no SEQ, a pad) has no piece records or end state: the batch is void, nothing to finish
    // (tests/test_pileup_edges.py: reads without SEQ or with a pad in front of variant 4 once the slab held other pieces)
    if (a.status->err) return;
    const int32_t rd = pieces[p].pad;
    const uint32_t sbeg = a.r.seq_off[rd];
    const bool last = (uint32_t)(p + 1) == piece_base[rd + 1];
    const uint32_t w_close = last ? end_w[rd] : pieces[p + 1].cig_beg;
    const int y_close = last ? (int)end_y[rd] : (int)(8u * (pieces[p + 1].seq_beg - sbeg)) + pieces[p + 1].y0;
    const int yw = (int)(pieces[p].seq_beg - sbeg);
    pieces[p].cig_n = w_close - pieces[p].cig_beg;
    pieces[p].seq_n = (uint32_t)((y_close - 8 * yw + 7) / 8 + 1);
}

__global__ void lr_iota_kernel(uint32_t* __restrict__ idx, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (uint32_t)i;
}

}  // namespace

int tc_pileup_long_launch(tc_ctx* ctx, const pileup_args& a0, cudaStream_t s) {
    pileup_args a = a0;
    const int64_t n = a.r.n;
    // per read: pieces and ops, then exclusive sums (n + 1 entries so that [r + 1] - [r] is the count)
    uint32_t* cnt = (uint32_t*)tc_dev_buf(ctx, SLOT_SEGS, 4 * 4 * ((size_t)n + 1) + 64);
    if (!cnt) return TC_ERR_NOMEM;
    uint32_t* n_pieces = cnt; uint32_t* n_ops = cnt + (n + 1); uint32_t* piece_base = cnt + 2 * (n + 1); uint32_t* ops_base = cnt + 3 * (n + 1);
    TC_CUDA(cudaMemsetAsync(cnt, 0, 4 * 2 * ((size_t)n + 1), s));
    lr_count_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a, n_pieces, n_ops);
    TC_LAUNCH_CHECK();
    size_t tmp_bytes = 0, tmp2 = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, n_pieces, piece_base, (int)(n + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_C, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, n_pieces, piece_base, (int)(n + 1), s));
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, n_ops, ops_base, (int)(n + 1), s));
    ctx->launches += 2;
    uint32_t* totals = (uint32_t*)ctx->host_status;        // pinned: the two copies do not wait for the stream one by one
    TC_CUDA(cudaMemcpyAsync(&totals[0], piece_base + n, 4, cudaMemcpyDeviceToHost, s));
    TC_CUDA(cudaMemcpyAsync(&totals[1], ops_base + n, 4, cudaMemcpyDeviceToHost, s));
    TC_CUDA(cudaStreamSynchronize(s));
    ctx->d2h_bytes += 8;
    const size_t NP = totals[0], NO = totals[1];
    if (NP == 0) return TC_OK;
    if (NP >= 0x7fffffffull) return tc_fail(ctx, TC_ERR_CAPACITY, "too many pieces (%zu)", NP);
    // pieces, their start columns (sort keys), the order, the piece CIGARs
    uint8_t* slab = (uint8_t*)tc_dev_buf(ctx, SLOT_TILES, NP * (sizeof(tc_piece) + 4 * 4) + 4 * (NO + 8) + 256);
    if (!slab) return TC_ERR_NOMEM;
    tc_piece* pieces = (tc_piece*)slab;
    int32_t* key_in = (int32_t*)(pieces + NP); int32_t* key_out = key_in + NP;
    uint32_t* idx_in = (uint32_t*)(key_out + NP); uint32_t* idx_out = idx_in + NP;
    uint32_t* pcig = idx_out + NP;
    pcig = (uint32_t*)(((uintptr_t)pcig + 15) & ~(uintptr_t)15);
    // n_pieces / n_ops are spent after the scans: they take the reads' end states (op slot, query index)
    lr_split_kernel<<<(unsigned)((n + LR_WARPS - 1) / LR_WARPS), LR_WARPS * 32, 0, s>>>(a, piece_base, ops_base, pieces, pcig, key_in, n_pieces, n_ops);
    TC_LAUNCH_CHECK();
    lr_finish_kernel<<<(unsigned)((NP + 255) / 256), 256, 0, s>>>(a, piece_base, pieces, (int64_t)NP, n_pieces, n_ops);
    TC_LAUNCH_CHECK();
    lr_iota_kernel<<<(unsigned)((NP + 255) / 256), 256, 0, s>>>(idx_in, (int64_t)NP);
    TC_LAUNCH_CHECK();
    int bits = 1;
    while ((1ll << bits) < (long long)a.L + 1 && bits < 31) ++bits;
    TC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp2, key_in, key_out, idx_in, idx_out, (int)NP, 0, bits, s));
    void* d_tmp2 = tc_dev_buf(ctx, SLOT_TMP_C, (tmp2 > tmp_bytes ? tmp2 : tmp_bytes) + 16);
    if (!d_tmp2) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp2, tmp2, key_in, key_out, idx_in, idx_out, (int)NP, 0, bits, s));
    ctx->launches++;
    a.pieces = pieces; a.piece_order = idx_out; a.n_pieces = (int64_t)NP;
    a.r.cigar = pcig;
    a.span_hint = 0;
    return tc_pileup_warp_launch_pieces(ctx, a, s);
}
