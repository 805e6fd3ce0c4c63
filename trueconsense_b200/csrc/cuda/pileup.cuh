// pileup.cuh — arguments shared by the pileup kernel variants.
#pragma once
#include "tc_common.cuh"

// A piece of a long read: the part of its alignment inside one cell of PIECE_COLS reference columns, made to look
// like a short read (pileup_long.cu builds them; pileup_warp.cu consumes them in its PIECES mode)
struct tc_piece {
    int32_t pos;            // first reference column of the piece
    uint32_t seq_beg;       // SEQ word holding the piece's first query base
    uint32_t cig_beg;       // first op in the piece-CIGAR buffer
    uint32_t cig_n;         // ops
    uint32_t seq_n;         // SEQ words to stage (with one word of look-ahead)
    int32_t lq;             // query bases from seq_beg's first nibble to the end of the read
    int32_t y0;             // query index of the piece's first base, relative to seq_beg's first nibble (0..7)
    int32_t pad;
};
#ifndef TC_PIECE_COLS
#define TC_PIECE_COLS 400
#endif
constexpr int PIECE_COLS = TC_PIECE_COLS;         // a multiple of 8, at most 440 (the 512-column window minus its slack)

// Variant 3 keeps a read's whole alignment inside a window of 8 * WC reference columns (WC = 32, 64 or 128 words) and takes
// reads while their starts stay within the window's first `slack` = 8 * WC - (longest span, rounded up to 8) - 8 columns; a
// slack below MIN_SLACK is not worth a window.
constexpr int MIN_SLACK = 64;

// The narrowest window (WC) for reads spanning at most `max_span` columns; 0 when the span is too long for any window (the
// reads are then cut into pieces, variant 4).  warp_pileup_kernel makes the same choice on the device from the span pass.
constexpr int warp_geometry(int max_span) {
    const int ms = (max_span + 7) & ~7;
    for (int wc = 32; wc <= 128; wc *= 2)
        if (((8 * wc - ms - 8) & ~7) >= MIN_SLACK) return wc;
    return 0;
}

struct pileup_args {
    dreads r;
    int32_t L;
    uint32_t flag_filter;
    int32_t min_mapq, min_bq, ignore_orphans;
    int32_t* counts;        // [8][L]
    int32_t* diff;          // [L+1]
    tc_status* status;
    int32_t span_hint;      // tc_reads_t.max_ref_span (0 = unknown: a span pass finds it)
    int32_t* span_out;      // [n] optional: the span pass leaves every read's reference span here (-1: filtered / out of range)
    // PIECES mode of variant 3 (long reads): pieces in order of start column; r.cigar is then the piece-CIGAR buffer
    unsigned long long* xi; // [L] variant 3: packed X (low 32 bits) | I (high 32 bits) event counters per column
    const tc_piece* pieces;
    const uint32_t* piece_order;
    int64_t n_pieces;
};

__device__ __forceinline__ bool read_passes(const pileup_args& a, int64_t r) {
    uint32_t fl = a.r.flag[r];
    if (fl & (a.flag_filter | 4u)) return false;                 // htslib always drops UNMAP
    if (a.min_mapq > 0 && a.r.mapq && (int)a.r.mapq[r] < a.min_mapq) return false;
    if (a.ignore_orphans && (fl & 1u) && !(fl & 2u)) return false;
    return true;
}


// variant 3 (pileup_warp.cu): barrier-free warp-per-read-stream SWAR kernel; fills every row except coverage
int tc_pileup_warp_launch(tc_ctx* ctx, const pileup_args& a, cudaStream_t s);
bool tc_pileup_warp_supported(const pileup_args& a);

// long reads (pileup_long.cu): cut every read into pieces of <= PIECE_COLS columns and run variant 3 over the pieces
int tc_pileup_long_launch(tc_ctx* ctx, const pileup_args& a, cudaStream_t s);
int tc_pileup_warp_launch_pieces(tc_ctx* ctx, const pileup_args& a, cudaStream_t s);

