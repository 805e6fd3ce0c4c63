// samparse.cu — SAM text (an aligner's output as it is written) -> BAM records in device memory.
//
// The records land where tc_bgzf_inflate + tc_bam_index_records leave a BAM's: a payload buffer and the offsets of the placed
// records' refID fields.  Sorting (tc_bam_sort_records), parsing (tc_bam_records_to_reads) and the contig ranges then run
// unchanged, so a SAM file yields the read arrays its BAM counterpart yields, byte for byte.
//   sam_line_count_kernel  4 KiB tiles of the text, 16-byte loads: '\n' per tile; cub's exclusive sum -> each tile's first line
//   sam_line_emit_kernel   the same tiles again: where every line starts (a block scan numbers the newlines inside a tile)
//   sam_meta_kernel        one warp per line: the 11 mandatory fields (ballots over 32-byte strides), their values checked
//                          and converted, RNAME / RNEXT looked up in the header's names, the record's size; the first bad
//                          line (atomicMin over line << 8 | reason)
//   exclusive sums         record sizes -> payload offsets; placed flags -> record numbers
//   sam_pack_kernel        one warp per placed line writes its record: fixed fields, name, CIGAR ops, SEQ nibbles, QUAL - 33
// The BAM `bin` field (left 0) and the optional fields are not produced: nothing downstream reads them.
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <utility>
#include <vector>

#include "bamrec.cuh"
#include "tc_common.cuh"

namespace {

constexpr int LI_THREADS = 256, LI_VEC = 16, LI_TILE = LI_THREADS * LI_VEC;
constexpr unsigned FULL = 0xffffffffu;
constexpr int LINE_WARPS = 8;           // lines per 256-thread block of the meta / pack kernels

enum sam_reason {
    R_NONE = 0, R_FIELDS, R_QNAME, R_FLAG, R_RNAME, R_POS, R_MAPQ, R_CIGAR, R_CIGAR_OPS, R_RNEXT, R_PNEXT, R_TLEN, R_EMPTY_FIELD,
    R_CIGAR_SEQ, R_QUAL_SEQ, R_QUAL_CHAR, R_EMPTY_LINE, R_HEADER, R_CG, R_LONG, R_COUNT
};
const char* const REASON_TEXT[R_COUNT] = {
    "",
    "fewer than 11 tab-separated fields",
    "QNAME must hold 1 to 254 characters",
    "FLAG is not a number in 0..65535",
    "RNAME names no reference of the header",
    "POS is not a number in 0..2147483647",
    "MAPQ is not a number in 0..255",
    "bad CIGAR: each operation is a length in 1..268435455 followed by one of MIDNSHP=X",
    "more than 65535 CIGAR operations (BAM's n_cigar_op is 16 bits)",
    "RNEXT is not '=', '*' or a reference of the header",
    "PNEXT is not a number in 0..2147483647",
    "TLEN is not a number in -2147483648..2147483647",
    "SEQ or QUAL is empty (write '*' for none)",
    "CIGAR and SEQ lengths differ",
    "QUAL and SEQ lengths differ",
    "QUAL character below '!'",
    "empty line",
    "header line after the first record",
    "the CIGAR is kept in a CG:B tag behind a <l_seq>S<n>N placeholder (more than 65535 operations): not supported",
    "line longer than 2^31 - 16 bytes",
};

// what sam_meta_kernel leaves for sam_pack_kernel (76 bytes a line)
struct sam_meta {
    int32_t tab[11];            // field f ends at tab[f] (relative to the line's start; tab[10]: QUAL's end), starts at tab[f-1] + 1
    int32_t tid, pos, mtid, mpos, tlen;
    uint32_t flag_mapq;         // FLAG | MAPQ << 16
    uint32_t n_cig;
    int32_t l_seq;
};
static_assert(sizeof(sam_meta) == 76, "the per-line buffer layout of tc_sam_to_bam_records rounds this array up to 16 bytes");

struct ref_table {              // the header's names: FNV-1a hashes sorted, each with its reference; the names to compare
    const unsigned long long* hash; const long long* off; const int32_t* idx; const uint8_t* names; int n;
};

struct sam_args {
    const uint8_t* u; const long long* ls; long long n_lines;
    ref_table refs;
    sam_meta* meta; unsigned long long* size; uint32_t* placed;
    const unsigned long long* off; const uint32_t* rank;
    uint8_t* out; long long* rec;
    unsigned long long* status;     // [0] first bad line << 8 | reason (~0: none), [1] SEQ words, [2] CIGAR ops, [3] records
};

__host__ __device__ __forceinline__ unsigned long long fnv1a(const uint8_t* s, long long n) {
    unsigned long long h = 1469598103934665603ull;
    for (long long i = 0; i < n; ++i) { h ^= s[i]; h *= 1099511628211ull; }
    return h;
}

// 16 bytes from p on, as four little-endian words; bytes at or behind n read as 0 (never a '\n' nor a tab)
__device__ __forceinline__ void load16(const uint8_t* u, long long p, long long n, uint32_t w[4]) {
    if (p + 16 <= n) {
        const uint4 v = *reinterpret_cast<const uint4*>(u + p);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        return;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t x = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) if (p + 4 * i + j < n) x |= (uint32_t)u[p + 4 * i + j] << (8 * j);
        w[i] = x;
    }
}

__device__ __forceinline__ unsigned newlines16(const uint32_t w[4]) {
    unsigned c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) c += __popc(__vcmpeq4(w[i], 0x0a0a0a0au)) >> 3;
    return c;
}

__global__ void __launch_bounds__(LI_THREADS) sam_line_count_kernel(const uint8_t* __restrict__ u, long long n,
                                                                    unsigned long long* __restrict__ tile_count) {
    typedef cub::BlockReduce<unsigned, LI_THREADS> reduce_t;
    __shared__ typename reduce_t::TempStorage tmp;
    uint32_t w[4];
    load16(u, (long long)blockIdx.x * LI_TILE + threadIdx.x * LI_VEC, n, w);
    const unsigned total = reduce_t(tmp).Sum(newlines16(w));
    if (threadIdx.x == 0) tile_count[blockIdx.x] = total;
}

// ls[0] = 0, ls[k + 1] = the byte behind line k's '\n'; a last line without one ends at n: ls[n_lines] = n + 1
__global__ void __launch_bounds__(LI_THREADS) sam_line_emit_kernel(const uint8_t* __restrict__ u, long long n,
                                                                   const unsigned long long* __restrict__ tile_first,
                                                                   long long* __restrict__ ls) {
    typedef cub::BlockScan<unsigned, LI_THREADS> scan_t;
    __shared__ typename scan_t::TempStorage tmp;
    const long long p = (long long)blockIdx.x * LI_TILE + threadIdx.x * LI_VEC;
    uint32_t w[4];
    load16(u, p, n, w);
    unsigned before;
    scan_t(tmp).ExclusiveSum(newlines16(w), before);
    long long idx = (long long)tile_first[blockIdx.x] + before;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (((w[j >> 2] >> (8 * (j & 3))) & 0xffu) == '\n') ls[1 + idx++] = p + j + 1;
    if (p <= n - 1 && n - 1 < p + 16 && u[n - 1] != '\n') ls[1 + idx] = n + 1;
    if (blockIdx.x == 0 && threadIdx.x == 0) ls[0] = 0;
}

__device__ __forceinline__ bool is_digit(unsigned c) { return c - '0' < 10u; }

__device__ __forceinline__ int op_of(unsigned c) {
    switch (c) {
        case 'M': return OP_M; case 'I': return OP_I; case 'D': return OP_D; case 'N': return OP_N; case 'S': return OP_S;
        case 'H': return OP_H; case 'P': return OP_P; case '=': return OP_EQ; case 'X': return OP_X;
        default: return -1;
    }
}

// decimal digits [s, e) -> *v; false when empty, not all digits, or above max
__device__ bool parse_dec(const uint8_t* s, const uint8_t* e, unsigned long long max, unsigned long long* v) {
    if (s >= e) return false;
    unsigned long long x = 0;
    for (; s < e; ++s) {
        const unsigned d = *s - '0';
        if (d > 9u) return false;
        x = x * 10 + d;
        if (x > max) return false;
    }
    *v = x;
    return true;
}

// the reference a name [s, s + n) is (-1: none): binary search over the hashes, then the bytes compared
__device__ int ref_lookup(const ref_table& t, const uint8_t* s, long long n) {
    const unsigned long long h = fnv1a(s, n);
    int lo = 0, hi = t.n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (t.hash[mid] < h) lo = mid + 1; else hi = mid;
    }
    for (; lo < t.n && t.hash[lo] == h; ++lo) {
        const int r = t.idx[lo];
        const long long b = t.off[r], len = t.off[r + 1] - b;
        if (len != n) continue;
        long long i = 0;
        while (i < n && t.names[b + i] == s[i]) ++i;
        if (i == n) return r;
    }
    return -1;
}

// the CIGAR operation a non-digit byte at p ends: its code and length, read over the digits in front of it.  False when it is
// not one of MIDNSHP=X, has no digits, or its length lies outside 1..2^28 - 1
__device__ __forceinline__ bool cigar_op_at(const uint8_t* u, long long cb, long long p, uint32_t* code, uint32_t* len) {
    const int op = op_of(u[p]);
    long long s = p;
    while (s > cb && is_digit(u[s - 1])) --s;
    unsigned long long v;
    if (op < 0 || !parse_dec(u + s, u + p, 0x0fffffffull, &v) || v == 0) return false;
    *code = (uint32_t)op; *len = (uint32_t)v;
    return true;
}

__device__ __forceinline__ bool query_op(uint32_t op) { return op == OP_M || op == OP_I || op == OP_S || op == OP_EQ || op == OP_X; }

// one line, all lanes of the warp (the small fields are parsed by every lane alike: no broadcasts).  Returns the reason the
// line is refused (R_NONE: it converts); *rec: the line is a record (not the empty last line)
__device__ int meta_line(const sam_args& a, long long k, int lane, int* tabs, uint32_t* cig2, unsigned long long* size,
                         int* placed, unsigned long long* words, unsigned long long* ops, int* rec) {
    const uint8_t* u = a.u;
    const long long b = a.ls[k], e = a.ls[k + 1] - 1;
    *size = 0; *placed = 0; *words = 0; *ops = 0; *rec = 0;
    if (e == b) return k + 1 < a.n_lines ? R_EMPTY_LINE : R_NONE;
    *rec = 1;
    if (e - b > 0x7ffffff0ll) return R_LONG;
    if (u[b] == '@') return R_HEADER;
    const unsigned lt = (1u << lane) - 1u;
    int nt = 0;
    bool qual_low = false;
    for (long long p0 = b; p0 < e && nt < 11; p0 += 32) {
        const long long p = p0 + lane;
        const unsigned c = p < e ? u[p] : 0u;
        const unsigned m = __ballot_sync(FULL, c == '\t');
        const int f = nt + __popc(m & lt);          // the field this byte lies in (a tab: the field it ends)
        if (c == '\t') { if (f < 11) tabs[f] = (int)(p - b); }
        else if (f == 10 && p < e && c < 33u) qual_low = true;
        nt += __popc(m);
    }
    qual_low = __any_sync(FULL, qual_low);
    if (nt < 10) return R_FIELDS;
    if (nt == 10 && lane == 0) tabs[10] = (int)(e - b);
    __syncwarp();
#define FS(f) (b + ((f) ? tabs[(f) - 1] + 1 : 0))
#define FE(f) (b + tabs[f])
    const long long l_qname = FE(0) - b;
    if (l_qname < 1 || l_qname > 254) return R_QNAME;
    unsigned long long v;
    if (!parse_dec(u + FS(1), u + FE(1), 65535, &v)) return R_FLAG;
    const uint32_t flag = (uint32_t)v;
    int tid = -1;
    if (!(FE(2) - FS(2) == 1 && u[FS(2)] == '*')) {
        tid = ref_lookup(a.refs, u + FS(2), FE(2) - FS(2));
        if (tid < 0) return R_RNAME;
    }
    if (!parse_dec(u + FS(3), u + FE(3), 0x7fffffff, &v)) return R_POS;
    const int32_t pos = (int32_t)v - 1;
    if (!parse_dec(u + FS(4), u + FE(4), 255, &v)) return R_MAPQ;
    const uint32_t mapq = (uint32_t)v;
    // CIGAR: every lane takes one byte of a 32-byte stride; a non-digit ends an operation
    const long long cb = FS(5), ce = FE(5);
    uint32_t n_cig = 0;
    unsigned long long qlen = 0;
    if (!(ce - cb == 1 && u[cb] == '*')) {
        if (ce == cb || is_digit(u[ce - 1])) return R_CIGAR;
        bool bad = false;
        for (long long p0 = cb; p0 < ce; p0 += 32) {
            const long long p = p0 + lane;
            const bool ends = p < ce && !is_digit(u[p]);
            const unsigned m = __ballot_sync(FULL, ends);
            if (ends) {
                uint32_t op, len;
                if (!cigar_op_at(u, cb, p, &op, &len)) bad = true;
                else {
                    if (query_op(op)) qlen += len;
                    const uint32_t j = n_cig + __popc(m & lt);
                    if (j < 2) cig2[j] = len << 4 | op;
                }
            }
            n_cig += __popc(m);
        }
        if (__any_sync(FULL, bad)) return R_CIGAR;
#pragma unroll
        for (int o = 16; o; o >>= 1) qlen += __shfl_xor_sync(FULL, qlen, o);
        if (n_cig > 65535u) return R_CIGAR_OPS;
    }
    int mtid;
    if (FE(6) - FS(6) == 1 && u[FS(6)] == '=') mtid = tid;
    else if (FE(6) - FS(6) == 1 && u[FS(6)] == '*') mtid = -1;
    else {
        mtid = ref_lookup(a.refs, u + FS(6), FE(6) - FS(6));
        if (mtid < 0) return R_RNEXT;
    }
    if (!parse_dec(u + FS(7), u + FE(7), 0x7fffffff, &v)) return R_PNEXT;
    const int32_t mpos = (int32_t)v - 1;
    {
        const long long tb = FS(8), te = FE(8);
        const bool neg = te > tb && u[tb] == '-', plus = te > tb && u[tb] == '+';
        if (!parse_dec(u + tb + (neg || plus), u + te, neg ? 0x80000000ull : 0x7fffffffull, &v)) return R_TLEN;
    }
    const int32_t tlen = (int32_t)(u[FS(8)] == '-' ? (uint32_t)(0u - (uint32_t)v) : (uint32_t)v);
    const long long sb = FS(9), se = FE(9), qb = FS(10), qe = FE(10);
    if (se == sb || qe == qb) return R_EMPTY_FIELD;
    const bool seq_star = se - sb == 1 && u[sb] == '*', qual_star = qe - qb == 1 && u[qb] == '*';
    const long long l_seq = seq_star ? 0 : se - sb;
    if (n_cig && !seq_star && qlen != (unsigned long long)l_seq) return R_CIGAR_SEQ;
    if (!qual_star && qe - qb != l_seq) return R_QUAL_SEQ;
    if (!qual_star && qual_low) return R_QUAL_CHAR;
    __syncwarp();
    if (tid >= 0 && n_cig == 2 && l_seq > 0 && nt > 10) {
        // the placeholder the BAM route refuses too (bgzf.cu record_valid): <l_seq>S<n>N with the real CIGAR in CG:B
        const uint32_t c0 = cig2[0], c1 = cig2[1];
        if ((c0 & 15u) == OP_S && (c0 >> 4) == (uint32_t)l_seq && (c1 & 15u) == OP_N) {
            bool cg = false;
            for (long long p0 = qe + 1; p0 < e; p0 += 32) {
                const long long p = p0 + lane;
                if (p + 4 <= e && u[p - 1] == '\t' && u[p] == 'C' && u[p + 1] == 'G' && u[p + 2] == ':' && u[p + 3] == 'B') cg = true;
            }
            if (__any_sync(FULL, cg)) return R_CG;
        }
    }
    if (lane == 0) {
        sam_meta& m = a.meta[k];
        for (int f = 0; f < 11; ++f) m.tab[f] = tabs[f];
        m.tid = tid; m.pos = pos; m.mtid = mtid; m.mpos = mpos; m.tlen = tlen;
        m.flag_mapq = flag | mapq << 16; m.n_cig = n_cig; m.l_seq = (int32_t)l_seq;
    }
#undef FS
#undef FE
    if (tid >= 0) {
        *placed = 1;
        *size = 36ull + (unsigned long long)(l_qname + 1) + 4ull * n_cig + (unsigned long long)((l_seq + 1) / 2 + l_seq);
        *words = (unsigned long long)((l_seq + 7) / 8);
        *ops = n_cig;
    }
    return R_NONE;
}

__global__ void __launch_bounds__(256) sam_meta_kernel(sam_args a) {
    __shared__ int tabs[LINE_WARPS][12];
    __shared__ uint32_t cig2[LINE_WARPS][2];
    __shared__ unsigned long long acc[3];          // this block's SEQ words, CIGAR ops and records
    if (threadIdx.x < 3) acc[threadIdx.x] = 0;
    __syncthreads();
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long k = (long long)blockIdx.x * LINE_WARPS + w;
    if (k < a.n_lines) {
        unsigned long long size, words, ops;
        int placed, rec;
        const int reason = meta_line(a, k, lane, tabs[w], cig2[w], &size, &placed, &words, &ops, &rec);
        if (lane == 0) {
            a.size[k] = reason ? 0 : size;
            a.placed[k] = reason ? 0 : placed;
            if (reason) atomicMin(&a.status[0], ((unsigned long long)k << 8) | (unsigned)reason);
            else if (rec) { atomicAdd(&acc[0], words); atomicAdd(&acc[1], ops); atomicAdd(&acc[2], 1ull); }
        }
    }
    __syncthreads();
    if (threadIdx.x < 3 && acc[threadIdx.x]) atomicAdd(&a.status[1 + threadIdx.x], acc[threadIdx.x]);
}

// htslib's seq_nt16 rule: "=ACMGRSVTWYHKDBN" in either case -> 0..15, anything else 15
__device__ uint8_t nt16_of(unsigned c) {
    if (c >= 'a' && c <= 'z') c -= 32;
    switch (c) {
        case '=': return 0; case 'A': return 1; case 'C': return 2; case 'M': return 3; case 'G': return 4; case 'R': return 5;
        case 'S': return 6; case 'V': return 7; case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11;
        case 'K': return 12; case 'D': return 13; case 'B': return 14;
        default: return 15;
    }
}

__global__ void __launch_bounds__(256) sam_pack_kernel(sam_args a) {
    __shared__ uint8_t nt16[256];
    nt16[threadIdx.x] = nt16_of(threadIdx.x);
    __syncthreads();
    const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= a.n_lines || !a.placed[k]) return;
    const uint8_t* u = a.u;
    const sam_meta& m = a.meta[k];
    const long long b = a.ls[k];
    const unsigned long long o = a.off[k];     // the record's block_size
    uint8_t* r = a.out + o - BAM_BLOCK_SIZE;
    const uint32_t l_name = (uint32_t)m.tab[0] + 1, n_cig = m.n_cig, l_seq = (uint32_t)m.l_seq;
    if (lane == 0) a.rec[a.rank[k]] = (long long)o - BAM_BLOCK_SIZE;
    // the fixed fields one 32-bit word per lane: 0 block_size, 1 refID, 2 pos, 3 l_read_name | MAPQ | bin, 4 n_cigar_op | FLAG,
    // 5 l_seq, 6 next refID, 7 next pos, 8 tlen
    if (lane < 9) {
        const unsigned long long size = a.off[k + 1] - o;       // placed: the next offset is this record's end
        uint32_t x;
        switch (lane) {
            case 0: x = (uint32_t)(size - 4); break;
            case 1: x = (uint32_t)m.tid; break;
            case 2: x = (uint32_t)m.pos; break;
            case 3: x = l_name | ((m.flag_mapq >> 16) << 8); break;        // l_read_name, MAPQ, bin (0)
            case 4: x = n_cig | ((m.flag_mapq & 0xffffu) << 16); break;
            case 5: x = l_seq; break;
            case 6: x = (uint32_t)m.mtid; break;
            case 7: x = (uint32_t)m.mpos; break;
            default: x = (uint32_t)m.tlen; break;
        }
        st32(r + BAM_BLOCK_SIZE + 4 * lane, x);
    }
    uint8_t* nm = r + BAM_READ_NAME;
    for (uint32_t j = lane; j < l_name; j += 32) nm[j] = j + 1 < l_name ? u[b + j] : 0;
    uint8_t* cg = nm + l_name;
    if (n_cig) {
        const long long cb = b + m.tab[4] + 1, ce = b + m.tab[5];
        const unsigned lt = (1u << lane) - 1u;
        uint32_t base = 0;
        for (long long p0 = cb; p0 < ce; p0 += 32) {
            const long long p = p0 + lane;
            const bool ends = p < ce && !is_digit(u[p]);
            const unsigned msk = __ballot_sync(FULL, ends);
            if (ends) {
                uint32_t op = 0, len = 0;
                cigar_op_at(u, cb, p, &op, &len);           // checked by sam_meta_kernel
                st32(cg + 4ull * (base + __popc(msk & lt)), len << 4 | op);
            }
            base += __popc(msk);
        }
    }
    uint8_t* sq = cg + 4ull * n_cig;
    const uint32_t sbytes = (l_seq + 1) / 2;
    const uint8_t* s = u + b + m.tab[8] + 1;
    for (uint32_t j = lane; j < sbytes; j += 32) {
        const uint32_t hi = nt16[s[2 * j]], lo = 2 * j + 1 < l_seq ? nt16[s[2 * j + 1]] : 0u;
        sq[j] = (uint8_t)(hi << 4 | lo);
    }
    uint8_t* ql = sq + sbytes;
    const uint8_t* q = u + b + m.tab[9] + 1;
    const bool qual_star = m.tab[10] - m.tab[9] - 1 == 1 && q[0] == '*';
    for (uint32_t j = lane; j < l_seq; j += 32) ql[j] = qual_star ? 0xffu : (uint8_t)(q[j] - 33);
}

double seconds_since(std::chrono::steady_clock::time_point t) {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t).count();
}

}  // namespace

TC_API int tc_sam_to_bam_records(tc_ctx_t* ctx, const uint8_t* text, int64_t n_bytes, int64_t first_line_off, int64_t first_line_no,
                                 int32_t n_ref, const char* ref_names, const int64_t* ref_name_off, const uint8_t** payload_dev,
                                 int64_t* n_payload, const int64_t** rec_off_dev, int64_t* n_placed, int64_t* n_records,
                                 int64_t* n_lines, int64_t* err, double* t_steps, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (n_bytes < 0 || first_line_off < 0 || first_line_off > n_bytes || (n_bytes > first_line_off && !text) || n_ref < 0 ||
        (n_ref > 0 && (!ref_names || !ref_name_off)) || !payload_dev || !n_payload || !rec_off_dev || !n_placed || !n_records ||
        !n_lines || !err)
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    *payload_dev = nullptr; *n_payload = 0; *rec_off_dev = nullptr; *n_placed = 0; *n_records = 0; *n_lines = 0;
    err[0] = err[1] = 0;
    if (t_steps) t_steps[0] = t_steps[1] = t_steps[2] = 0;
    const long long nb = n_bytes - first_line_off;
    if (nb == 0) return TC_OK;
    auto t0 = std::chrono::steady_clock::now();
    int rc;
    // the header's names for the device: sorted hashes, offsets, references, bytes
    std::vector<std::pair<unsigned long long, int32_t>> hv((size_t)n_ref);
    for (int32_t i = 0; i < n_ref; ++i) {
        if (ref_name_off[i + 1] < ref_name_off[i]) return tc_fail(ctx, TC_ERR_ARG, "bad reference name offsets");
        hv[i] = {fnv1a((const uint8_t*)ref_names + ref_name_off[i], ref_name_off[i + 1] - ref_name_off[i]), i};
    }
    std::sort(hv.begin(), hv.end());
    const size_t nr = (size_t)n_ref, names_bytes = n_ref ? (size_t)ref_name_off[n_ref] : 0;
    std::vector<uint8_t> tab(8 * nr + 8 * (nr + 1) + 4 * nr + names_bytes + 8);
    for (size_t i = 0; i < nr; ++i) {
        memcpy(tab.data() + 8 * i, &hv[i].first, 8);
        memcpy(tab.data() + 8 * nr + 8 * (nr + 1) + 4 * i, &hv[i].second, 4);
    }
    if (n_ref) {
        memcpy(tab.data() + 8 * nr, ref_name_off, 8 * (nr + 1));
        memcpy(tab.data() + 8 * nr + 8 * (nr + 1) + 4 * nr, ref_names, names_bytes);
    }
    uint8_t* d_tab = (uint8_t*)tc_dev_buf(ctx, SLOT_SAM_REFS, tab.size());
    if (!d_tab) return TC_ERR_NOMEM;
    rc = tc_h2d(ctx, d_tab, tab.data(), tab.size(), s); if (rc) return rc;
    // the text behind the header (16-byte loads: a device source at another alignment is copied)
    const uint8_t* body = text + first_line_off;
    const uint8_t* u;
    if (tc_is_device_ptr(body) && ((uintptr_t)body & 15u) == 0) u = body;
    else if (tc_is_device_ptr(body)) {
        uint8_t* d = (uint8_t*)tc_dev_buf(ctx, SLOT_SAM_TEXT, (size_t)nb);
        if (!d) return TC_ERR_NOMEM;
        TC_CUDA(cudaMemcpyAsync(d, body, (size_t)nb, cudaMemcpyDeviceToDevice, s));
        u = d;
    } else {
        u = (const uint8_t*)tc_stage_in(ctx, SLOT_SAM_TEXT, body, (size_t)nb, s, &rc);
        if (rc) return rc;
    }
    TC_CUDA(cudaStreamSynchronize(s));
    if (t_steps) t_steps[0] = seconds_since(t0);
    t0 = std::chrono::steady_clock::now();
    // line index
    const size_t n_tiles = (size_t)((nb + LI_TILE - 1) / LI_TILE);
    unsigned long long* d_tiles = (unsigned long long*)tc_dev_buf(ctx, SLOT_TMP_A, 16 * (n_tiles + 1));
    if (!d_tiles) return TC_ERR_NOMEM;
    unsigned long long* d_tile_first = d_tiles + (n_tiles + 1);
    TC_CUDA(cudaMemsetAsync(d_tiles + n_tiles, 0, 8, s));
    sam_line_count_kernel<<<(unsigned)n_tiles, LI_THREADS, 0, s>>>(u, nb, d_tiles);
    TC_LAUNCH_CHECK();
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_tiles, d_tile_first, (int)(n_tiles + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_tiles, d_tile_first, (int)(n_tiles + 1), s));
    ctx->launches++;
    unsigned long long* h = (unsigned long long*)ctx->host_status;
    TC_D2H(h, d_tile_first + n_tiles, 8, s);
    TC_D2H((uint8_t*)(h + 1), u + nb - 1, 1, s);
    TC_CUDA(cudaStreamSynchronize(s));
    const long long nl = (long long)h[0] + (((const uint8_t*)(h + 1))[0] != '\n');
    if (nl >= 0x7fffffffll) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 lines in one SAM file; split the input");
    const size_t n = (size_t)nl;
    long long* d_ls = (long long*)tc_dev_buf(ctx, SLOT_SAM_LINES, 8 * (n + 1));
    if (!d_ls) return TC_ERR_NOMEM;
    sam_line_emit_kernel<<<(unsigned)n_tiles, LI_THREADS, 0, s>>>(u, nb, d_tile_first, d_ls);
    TC_LAUNCH_CHECK();
    TC_CUDA(cudaStreamSynchronize(s));
    if (t_steps) t_steps[1] = seconds_since(t0);
    t0 = std::chrono::steady_clock::now();
    // per line: meta, record size, placed flag (one more, zero, entry each so that the exclusive sums end with the totals),
    // payload offset, record number; the status block
    const size_t n1 = n + 1;
    const size_t meta_b = (sizeof(sam_meta) * n + 15) & ~(size_t)15, size_b = 8 * n1, off_b = 8 * n1, placed_b = (4 * n1 + 7) & ~(size_t)7, rank_b = placed_b;
    uint8_t* d_meta = (uint8_t*)tc_dev_buf(ctx, SLOT_SAM_META, meta_b + size_b + off_b + placed_b + rank_b + 64);
    if (!d_meta) return TC_ERR_NOMEM;
    sam_args a;
    memset(&a, 0, sizeof(a));
    a.u = u; a.ls = d_ls; a.n_lines = nl;
    a.refs.hash = (const unsigned long long*)d_tab; a.refs.off = (const long long*)(d_tab + 8 * nr);
    a.refs.idx = (const int32_t*)(d_tab + 8 * nr + 8 * (nr + 1)); a.refs.names = d_tab + 8 * nr + 8 * (nr + 1) + 4 * nr; a.refs.n = n_ref;
    a.meta = (sam_meta*)d_meta;
    a.size = (unsigned long long*)(d_meta + meta_b);
    unsigned long long* d_off = (unsigned long long*)(d_meta + meta_b + size_b);
    a.placed = (uint32_t*)(d_meta + meta_b + size_b + off_b);
    uint32_t* d_rank = (uint32_t*)(d_meta + meta_b + size_b + off_b + placed_b);
    a.status = (unsigned long long*)(d_meta + meta_b + size_b + off_b + placed_b + rank_b);
    a.off = d_off; a.rank = d_rank;
    TC_CUDA(cudaMemsetAsync(a.size + n, 0, 8, s));
    TC_CUDA(cudaMemsetAsync(a.placed + n, 0, 4, s));
    TC_CUDA(cudaMemsetAsync(a.status, 0, 32, s));
    TC_CUDA(cudaMemsetAsync(a.status, 0xff, 8, s));
    const unsigned line_blocks = (unsigned)((n + LINE_WARPS - 1) / LINE_WARPS);
    sam_meta_kernel<<<line_blocks, 32 * LINE_WARPS, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    size_t tmp1 = 0, tmp2 = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp1, a.size, d_off, (int)n1, s));
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp2, a.placed, d_rank, (int)n1, s));
    tmp_bytes = std::max(tmp1, tmp2);
    d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.size, d_off, (int)n1, s));
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.placed, d_rank, (int)n1, s));
    ctx->launches += 2;
    TC_D2H(h, a.status, 32, s);
    TC_D2H(h + 4, d_off + n, 8, s);
    TC_D2H((uint32_t*)(h + 5), d_rank + n, 4, s);
    TC_CUDA(cudaStreamSynchronize(s));
    *n_lines = nl;
    if (h[0] != ~0ull) {
        const int reason = (int)(h[0] & 0xff);
        err[0] = first_line_no + (int64_t)(h[0] >> 8);
        err[1] = reason;
        return tc_fail(ctx, TC_ERR_ARG, "line %lld: %s", (long long)err[0], reason < R_COUNT ? REASON_TEXT[reason] : "bad line");
    }
    if (h[1] > 0xffffffffull || h[2] > 0xffffffffull)
        return tc_fail(ctx, TC_ERR_ARG, "more than 2^32 SEQ words or CIGAR operations in one SAM file; split the input");
    const unsigned long long payload_bytes = h[4];
    const uint32_t placed = *(const uint32_t*)(h + 5);
    *n_records = (int64_t)h[3];
    if (placed) {
        a.out = (uint8_t*)tc_dev_buf(ctx, SLOT_BAM_PAYLOAD, (size_t)payload_bytes + 64);
        a.rec = (long long*)tc_dev_buf(ctx, SLOT_BAM_REC, 8 * (size_t)placed);
        if (!a.out || !a.rec) return TC_ERR_NOMEM;
        sam_pack_kernel<<<line_blocks, 32 * LINE_WARPS, 0, s>>>(a);
        TC_LAUNCH_CHECK();
        TC_CUDA(cudaStreamSynchronize(s));
        *payload_dev = a.out; *rec_off_dev = (const int64_t*)a.rec;
    }
    *n_payload = (int64_t)payload_bytes; *n_placed = placed;
    if (t_steps) t_steps[2] = seconds_since(t0);
    return TC_OK;
}
