// bamrec.cuh — the BAM record layout (SAM spec §4.2), for the device code that reads or writes records.
//
// Every record offset on the device (rec_off, as tc_bam_index_records, tc_sam_to_bam_records, tc_bam_clip_primers and
// tc_bam_sort_records hand it on) points at the record's refID field, so the offsets below count from there; block_size
// lies in front of it.  Records start at any byte: fields are loaded and stored a byte at a time, little-endian.
#pragma once

#include <cstdint>

constexpr int BAM_BLOCK_SIZE = -4;      // uint32: the record's bytes behind this field
constexpr int BAM_REF_ID = 0;           // int32
constexpr int BAM_POS = 4;              // int32, 0-based
constexpr int BAM_L_READ_NAME = 8;      // uint8, the NUL included
constexpr int BAM_MAPQ = 9;             // uint8
constexpr int BAM_BIN = 10;             // uint16
constexpr int BAM_N_CIGAR_OP = 12;      // uint16
constexpr int BAM_FLAG = 14;            // uint16
constexpr int BAM_L_SEQ = 16;           // uint32
constexpr int BAM_NEXT_REF_ID = 20;     // int32
constexpr int BAM_NEXT_POS = 24;        // int32
constexpr int BAM_TLEN = 28;            // int32
constexpr int BAM_READ_NAME = 32;       // l_read_name bytes, then n_cigar_op uint32 ops, SEQ, QUAL, optional fields

__device__ __forceinline__ uint32_t ld16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t ld32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ void st32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24);
}

// the CIGAR ops of the record whose refID field is at r
__device__ __forceinline__ const uint8_t* bam_cigar(const uint8_t* r) { return r + BAM_READ_NAME + r[BAM_L_READ_NAME]; }

// record i (refID tid, pos pos) sorts before record i - 1 by (refID, pos); false for i = 0
__device__ __forceinline__ bool bam_out_of_order(const uint8_t* u, const long long* rec, long long i, int32_t tid, int32_t pos) {
    if (i == 0) return false;
    const uint8_t* q = u + rec[i - 1];
    const int32_t ptid = (int32_t)ld32(q + BAM_REF_ID), ppos = (int32_t)ld32(q + BAM_POS);
    return tid < ptid || (tid == ptid && pos < ppos);
}

// htslib's hts_reg2bin(beg, end, 14, 5)
__device__ __forceinline__ uint32_t reg2bin(long long beg, long long end) {
    --end;
    if (beg >> 14 == end >> 14) return (uint32_t)(4681 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (uint32_t)(585 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (uint32_t)(73 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (uint32_t)(9 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (uint32_t)(1 + (beg >> 26));
    return 0;
}

// n bytes from s to d, the lanes sharing them: 4-byte stores wherever d is aligned (s may lie at any byte: two aligned
// loads and a funnel shift; every word loaded holds at least one byte of the source)
static __device__ void warp_copy(uint8_t* d, const uint8_t* s, uint32_t n, int lane) {
    const uint32_t head = (uint32_t)((4u - ((uintptr_t)d & 3u)) & 3u) < n ? (uint32_t)((4u - ((uintptr_t)d & 3u)) & 3u) : n;
    if ((uint32_t)lane < head) d[lane] = s[lane];
    d += head; s += head; n -= head;
    const uint32_t words = n >> 2, sh = (uint32_t)((uintptr_t)s & 3u);
    uint32_t* dw = reinterpret_cast<uint32_t*>(d);
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(s - sh);
    if (sh == 0) {
        for (uint32_t j = lane; j < words; j += 32) dw[j] = sw[j];
    } else {
        for (uint32_t j = lane; j < words; j += 32) dw[j] = __funnelshift_r(sw[j], sw[j + 1], 8 * sh);
    }
    for (uint32_t j = 4 * words + lane; j < n; j += 32) d[j] = s[j];
}
