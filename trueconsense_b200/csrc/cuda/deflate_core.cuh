// deflate_core.cuh — raw DEFLATE (RFC 1951) of ONE BGZF member (at most 0xff00 bytes) by ONE CTA, as one dynamic-Huffman
// block, or a stored block when that is smaller.
//
// The member is compressed in phases separated by barriers.  Every phase is a loop over thread indices in which no two
// threads write the same location with different values (or only combine through max, add or or, whose result does not
// depend on the order), so the bytes are a function of the input alone: not of timing, of the order of atomics or of the
// launch geometry.  `deflate_member` runs the phases: on the device every thread of the CTA calls it and the phases are
// separated by __syncthreads(); on the host (tests/native/deflate_harness.cpp, checked against zlib by the CPU suite) one
// thread runs each phase for every thread index in turn.  Both produce the same bytes.
//
//   find     rounds of ROUND positions: position i hashes its next 4 bytes; its candidate is the nearest earlier position of
//            its 32-aligned group with the same hash (a warp's __match_any_sync), else the hash table's entry as it stood
//            before the round (the latest position of an earlier round).  Then every position of the round enters the table
//            (a max: the latest wins).  The candidate is one position at most 32 768 bytes back, or none: single-probe.
//   parse    the member cut into NSEG segments, one serial greedy walk each: a candidate whose bytes match for at least
//            MIN_MATCH is taken (up to 258 bytes, not across the segment's end), else a literal.  The symbols overwrite the
//            candidates in place.  Meanwhile other threads take the CRC-32 of each segment (inflate_core.cuh's table).
//   codes    symbol histograms; code lengths by in-place minimum-redundancy (Moffat-Katajainen) over the symbols sorted by
//            (frequency, index), limited to 15 bits (7 for the code-length alphabet) by moving leaves down (miniz's
//            rule); canonical codes; the code-length sequence run-length coded with 16 / 17 / 18.
//   emit     bits per segment, their offsets by a scan, and every segment's bits or-ed into the zeroed output words.
#pragma once
#include <stdint.h>

#include "inflate_core.cuh"

namespace tcdef {

constexpr int MEMBER_MAX = 0xff00;      // uncompressed bytes of a member (htslib's BGZF_BLOCK_SIZE)
constexpr int IN_BYTES = 65536;
constexpr int HASH_BITS = 14;
constexpr int HASH_SIZE = 1 << HASH_BITS;
constexpr int ROUND = 512;              // positions whose candidates are found together
constexpr int NSEG = 64;                // serial parse walks per member
constexpr int MIN_MATCH = 4, MAX_MATCH = 258, WINDOW = 32768;
constexpr uint16_t NONE = 0xffff;
constexpr uint16_t MATCH_BIT = 0x8000;  // parsed symbol: MATCH_BIT | (length - 3), the distance in the next entry; 0: a literal
constexpr int N_LIT = 286, N_DIST = 30, N_CL = 19;
constexpr int MAX_BITS = 15, MAX_CL_BITS = 7;

struct tables {
    uint32_t lfreq[N_LIT], dfreq[N_DIST], cfreq[N_CL];
    uint16_t lcode[N_LIT], dcode[N_DIST], ccode[N_CL];
    uint8_t llen[N_LIT], dlen[N_DIST], clen[N_CL];
    uint16_t lsorted[N_LIT], dsorted[N_DIST];       // used symbols by (frequency, index)
    uint16_t rle[N_LIT + N_DIST];                   // code-length sequence: symbol | extra << 5
    uint32_t crc_tab[256];
    uint32_t seg_bits[NSEG + 1];                    // bits of each segment's symbols, then their exclusive sum
    uint32_t seg_crc[NSEG];
    uint32_t work[N_LIT];                           // the code-length builder's scratch
    int n_rle, hlit, hdist, hclen;
    uint32_t header_bits, total_bits, crc;
    int stored, out_bytes;
};

struct member_smem {
    uint8_t in[IN_BYTES];
    uint16_t sym[MEMBER_MAX];                       // candidates, then the parsed symbols
    union {
        uint16_t head[HASH_SIZE];                   // find: the latest position of each hash
        tables t;                                   // from the parse on
    };
};
static_assert(sizeof(tables) <= sizeof(uint16_t) * HASH_SIZE, "tables overlay the hash table");

TCI_HD uint32_t hash4(const uint8_t* p) {
    const uint32_t x = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    return (x * 2654435761u) >> (32 - HASH_BITS);
}
TCI_HD int msb(uint32_t x) {
#ifdef __CUDA_ARCH__
    return 31 - __clz(x);
#else
    return 31 - __builtin_clz(x);
#endif
}
// length 3..258 -> symbol 257..285, extra bits, their value
TCI_HD void len_code(int len, int& sym, int& nb, int& extra) {
    if (len == 258) { sym = 285; nb = 0; extra = 0; return; }
    if (len < 11) { sym = 254 + len; nb = 0; extra = 0; return; }
    const int l = len - 3;
    nb = msb((uint32_t)l) - 2;
    sym = 257 + 4 * (nb + 1) + ((l >> nb) - 4);
    extra = l & ((1 << nb) - 1);
}
// distance 1..32768 -> symbol 0..29, extra bits, their value
TCI_HD void dist_code(int dist, int& sym, int& nb, int& extra) {
    const int d = dist - 1;
    if (d < 4) { sym = d; nb = 0; extra = 0; return; }
    const int m = msb((uint32_t)d);
    nb = m - 1;
    sym = 2 * m + ((d >> nb) & 1);
    extra = d & ((1 << nb) - 1);
}
TCI_HD uint32_t bit_reverse(uint32_t code, int len) {
    uint32_t r = 0;
    for (int k = 0; k < len; ++k) r |= ((code >> k) & 1u) << (len - 1 - k);
    return r;
}
TCI_HD void seg_range(int n, int s, int& s0, int& s1) {
    const int per = (n + NSEG - 1) / NSEG;
    s0 = s * per < n ? s * per : n;
    s1 = s0 + per < n ? s0 + per : n;
}

// ---------------------------------------------------------------- find
TCI_HD void find_init(member_smem& s, int tid, int nt) {
    for (int h = tid; h < HASH_SIZE; h += nt) s.head[h] = NONE;
}
// candidates of the round's positions (nt a multiple of 32: a warp holds a 32-aligned group of positions)
TCI_HD void find_round(member_smem& s, int n, int r, int tid, int nt) {
    for (int i = r * ROUND + tid; i < (r + 1) * ROUND; i += nt) {
        const bool valid = i + 4 <= n;
        const uint32_t h = valid ? hash4(s.in + i) : 0u;
        int near = -1;
#ifdef __CUDA_ARCH__
        const int lane = i & 31;
        const unsigned peers = __match_any_sync(0xffffffffu, valid ? h : 0x80000000u | (unsigned)lane);
        const unsigned lower = peers & ((1u << lane) - 1u);
        if (valid && lower) near = i - lane + msb(lower);
#else
        if (valid)
            for (int j = i - 1; j >= (i & ~31); --j)
                if (j + 4 <= n && hash4(s.in + j) == h) { near = j; break; }
#endif
        if (i >= n) continue;
        int c = near >= 0 ? near : (valid ? (int)s.head[h] : (int)NONE);
        if (c == (int)NONE || i - c > WINDOW) c = NONE;
        s.sym[i] = (uint16_t)c;
    }
}
TCI_HD void find_insert(member_smem& s, int n, int r, int tid, int nt) {
    for (int i = r * ROUND + tid; i < (r + 1) * ROUND && i + 4 <= n; i += nt) {
        uint16_t* a = &s.head[hash4(s.in + i)];
#ifdef __CUDA_ARCH__
        unsigned short old = *a;
        while (old == NONE || old < (unsigned short)i) {
            const unsigned short prev = atomicCAS((unsigned short*)a, old, (unsigned short)i);
            if (prev == old) break;
            old = prev;
        }
#else
        if (*a == NONE || *a < i) *a = (uint16_t)i;
#endif
    }
}

// ---------------------------------------------------------------- parse (threads 0..NSEG-1) and CRC pieces (NSEG..2 NSEG-1)
TCI_HD void parse_and_crc(member_smem& s, int n, int tid, int nt) {
    for (int k = tid; k < 2 * NSEG; k += nt) {
        int s0, s1;
        seg_range(n, k % NSEG, s0, s1);
        if (k >= NSEG) {
            uint32_t c = 0xffffffffu;
            for (int p = s0; p < s1; ++p) c = s.t.crc_tab[(c ^ s.in[p]) & 0xffu] ^ (c >> 8);
            s.t.seg_crc[k - NSEG] = c ^ 0xffffffffu;
            continue;
        }
        int p = s0;
        while (p < s1) {
            const int c = s.sym[p];
            int len = 0;
            if (c != NONE) {
                const int lim = s1 - p < MAX_MATCH ? s1 - p : MAX_MATCH;
                while (len < lim && s.in[c + len] == s.in[p + len]) ++len;
            }
            if (len >= MIN_MATCH) {
                s.sym[p] = (uint16_t)(MATCH_BIT | (len - 3));
                s.sym[p + 1] = (uint16_t)(p - c);
                p += len;
            } else {
                s.sym[p] = 0;
                ++p;
            }
        }
    }
}

// ---------------------------------------------------------------- codes
TCI_HD void add_u32(uint32_t* a, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicAdd(a, v);
#else
    *a += v;
#endif
}

TCI_HD void tables_init(member_smem& s, int tid, int nt) {
    for (int k = tid; k < 256; k += nt) s.t.crc_tab[k] = tcinf::crc_table_entry((uint32_t)k);
    for (int k = tid; k < N_LIT; k += nt) s.t.lfreq[k] = 0;
    for (int k = tid; k < N_DIST; k += nt) s.t.dfreq[k] = 0;
}

// the symbols of segment k, in order: f(literal byte, length, distance) with length 0 for a literal
template <class F>
TCI_HD void walk_segment(const member_smem& s, int n, int k, F f) {
    int s0, s1;
    seg_range(n, k, s0, s1);
    for (int p = s0; p < s1;) {
        const uint16_t v = s.sym[p];
        if (v & MATCH_BIT) {
            const int len = (v & 0xff) + 3;
            f(0, len, (int)s.sym[p + 1]);
            p += len;
        } else {
            f((int)s.in[p], 0, 0);
            ++p;
        }
    }
}

TCI_HD void histogram(member_smem& s, int n, int tid, int nt) {
    for (int k = tid; k < NSEG; k += nt)
        walk_segment(s, n, k, [&](int lit, int len, int dist) {
            if (!len) { add_u32(&s.t.lfreq[lit], 1u); return; }
            int sym, nb, ex;
            len_code(len, sym, nb, ex);
            add_u32(&s.t.lfreq[sym], 1u);
            dist_code(dist, sym, nb, ex);
            add_u32(&s.t.dfreq[sym], 1u);
        });
}

// a code needs two symbols at least (a single code of one bit is not complete): unused ones from index 0 up are added
TCI_HD void at_least_two(uint32_t* f, int nsym) {
    int used = 0;
    for (int i = 0; i < nsym; ++i) used += f[i] != 0;
    for (int i = 0; used < 2 && i < nsym; ++i)
        if (!f[i]) { f[i] = 1; ++used; }
}

TCI_HD void codes_prepare(member_smem& s, int tid, int nt) {
    (void)nt;
    if (tid != 0) return;
    s.t.lfreq[256] = 1;                                         // end of block
    at_least_two(s.t.lfreq, N_LIT);
    at_least_two(s.t.dfreq, N_DIST);
}

// the used symbols of both alphabets ordered by (frequency, index): every symbol finds its own rank
TCI_HD void codes_rank(member_smem& s, int tid, int nt) {
    for (int t = tid; t < N_LIT + N_DIST; t += nt) {
        const bool lit = t < N_LIT;
        const uint32_t* f = lit ? s.t.lfreq : s.t.dfreq;
        const int n = lit ? N_LIT : N_DIST, x = lit ? t : t - N_LIT;
        if (!f[x]) continue;
        int rank = 0;
        for (int u = 0; u < n; ++u) rank += f[u] && (f[u] < f[x] || (f[u] == f[x] && u < x));
        (lit ? s.t.lsorted : s.t.dsorted)[rank] = (uint16_t)x;
    }
}

// code lengths of the n used symbols `sorted` (ascending frequency) limited to `limit` bits; `a`: n words of scratch
TCI_HD void huff_lengths(const uint32_t* freq, const uint16_t* sorted, int n, int limit, uint8_t* len, int nsym, uint32_t* a) {
    for (int i = 0; i < nsym; ++i) len[i] = 0;
    if (n == 0) return;
    for (int i = 0; i < n; ++i) a[i] = freq[sorted[i]];
    if (n == 1) {
        a[0] = 1;
    } else {
        // Moffat & Katajainen, in place: a[] becomes the depth of every leaf
        a[0] += a[1];
        int root = 0, leaf = 2;
        for (int next = 1; next < n - 1; ++next) {
            if (leaf >= n || a[root] < a[leaf]) { a[next] = a[root]; a[root++] = (uint32_t)next; }
            else a[next] = a[leaf++];
            if (leaf >= n || (root < next && a[root] < a[leaf])) { a[next] += a[root]; a[root++] = (uint32_t)next; }
            else a[next] += a[leaf++];
        }
        a[n - 2] = 0;
        for (int next = n - 3; next >= 0; --next) a[next] = a[a[next]] + 1;
        int avbl = 1, used = 0, dpth = 0;
        root = n - 2;
        int next = n - 1;
        while (avbl > 0) {
            while (root >= 0 && (int)a[root] == dpth) { ++used; --root; }
            while (avbl > used) { a[next--] = (uint32_t)dpth; --avbl; }
            avbl = 2 * used;
            ++dpth;
            used = 0;
        }
    }
    // depths -> counts per length, the longest moved up to `limit`, then leaves moved down until the code is complete
    int count[33];
    for (int l = 0; l <= 32; ++l) count[l] = 0;
    for (int i = 0; i < n; ++i) count[a[i] < 32u ? a[i] : 32]++;
    for (int l = limit + 1; l <= 32; ++l) { count[limit] += count[l]; count[l] = 0; }
    uint32_t total = 0;
    for (int l = limit; l > 0; --l) total += (uint32_t)count[l] << (limit - l);
    while (total > (1u << limit)) {
        count[limit]--;
        for (int l = limit - 1; l > 0; --l)
            if (count[l]) { count[l]--; count[l + 1] += 2; break; }
        total--;
    }
    // the most frequent symbols get the shortest codes
    int j = n;
    for (int l = 1; l <= limit; ++l)
        for (int c = count[l]; c > 0; --c) len[sorted[--j]] = (uint8_t)l;
}

// canonical codes, bit-reversed for the LSB-first stream
TCI_HD void canonical(const uint8_t* len, uint16_t* code, int nsym) {
    int bl[MAX_BITS + 1], next[MAX_BITS + 1];
    for (int b = 0; b <= MAX_BITS; ++b) bl[b] = 0;
    for (int i = 0; i < nsym; ++i) bl[len[i]]++;
    bl[0] = 0;
    int c = 0;
    for (int b = 1; b <= MAX_BITS; ++b) { c = (c + bl[b - 1]) << 1; next[b] = c; }
    for (int i = 0; i < nsym; ++i)
        if (len[i]) code[i] = (uint16_t)bit_reverse((uint32_t)next[len[i]]++, len[i]);
}

TCI_HD int cl_extra_bits(int sym) { return sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0; }

// order of the code-length code lengths in the header
TCI_HD int cl_order(int i) {
    const int j = i - 4;
    return i < 3 ? 16 + i : (i == 3 ? 0 : ((j & 1) ? 7 - (j >> 1) : 8 + (j >> 1)));
}

TCI_HD void codes_build(member_smem& s, int tid, int nt) {
    (void)nt;
    if (tid != 0) return;
    tables& t = s.t;
    int nl = 0, nd = 0;
    for (int i = 0; i < N_LIT; ++i) nl += t.lfreq[i] != 0;
    for (int i = 0; i < N_DIST; ++i) nd += t.dfreq[i] != 0;
    huff_lengths(t.lfreq, t.lsorted, nl, MAX_BITS, t.llen, N_LIT, t.work);
    huff_lengths(t.dfreq, t.dsorted, nd, MAX_BITS, t.dlen, N_DIST, t.work);
    canonical(t.llen, t.lcode, N_LIT);
    canonical(t.dlen, t.dcode, N_DIST);
    int hlit = N_LIT, hdist = N_DIST;
    while (hlit > 257 && !t.llen[hlit - 1]) --hlit;
    while (hdist > 1 && !t.dlen[hdist - 1]) --hdist;
    t.hlit = hlit; t.hdist = hdist;
    // the code lengths of both alphabets as one sequence, runs coded with 16 (repeat the previous 3-6 times), 17 (3-10
    // zeros) and 18 (11-138 zeros)
    const int total = hlit + hdist;
    int nr = 0;
    for (int k = 0; k < N_CL; ++k) t.cfreq[k] = 0;
    for (int i = 0; i < total;) {
        const int v = i < hlit ? t.llen[i] : t.dlen[i - hlit];
        int run = 1;
        while (i + run < total && (i + run < hlit ? t.llen[i + run] : t.dlen[i + run - hlit]) == v) ++run;
        i += run;
        if (v == 0) {
            while (run >= 11) { const int r = run < 138 ? run : 138; t.rle[nr++] = (uint16_t)(18 | (r - 11) << 5); t.cfreq[18]++; run -= r; }
            if (run >= 3) { t.rle[nr++] = (uint16_t)(17 | (run - 3) << 5); t.cfreq[17]++; run = 0; }
        } else {
            t.rle[nr++] = (uint16_t)v; t.cfreq[v]++; --run;
            while (run >= 3) { const int r = run < 6 ? run : 6; t.rle[nr++] = (uint16_t)(16 | (r - 3) << 5); t.cfreq[16]++; run -= r; }
        }
        while (run-- > 0) { t.rle[nr++] = (uint16_t)v; t.cfreq[v]++; }
    }
    t.n_rle = nr;
    at_least_two(t.cfreq, N_CL);
    // 19 symbols: ordered by insertion
    uint16_t cs[N_CL];
    int nc = 0;
    for (int x = 0; x < N_CL; ++x) {
        if (!t.cfreq[x]) continue;
        int j = nc++;
        while (j > 0 && t.cfreq[cs[j - 1]] > t.cfreq[x]) { cs[j] = cs[j - 1]; --j; }
        cs[j] = (uint16_t)x;
    }
    huff_lengths(t.cfreq, cs, nc, MAX_CL_BITS, t.clen, N_CL, t.work);
    canonical(t.clen, t.ccode, N_CL);
    int hclen = N_CL;
    while (hclen > 4 && !t.clen[cl_order(hclen - 1)]) --hclen;
    t.hclen = hclen;
    uint32_t bits = 3 + 5 + 5 + 4 + 3 * (uint32_t)hclen;
    for (int k = 0; k < nr; ++k) bits += t.clen[t.rle[k] & 31] + cl_extra_bits(t.rle[k] & 31);
    t.header_bits = bits;
}

// ---------------------------------------------------------------- emit
TCI_HD void seg_bits(member_smem& s, int n, int tid, int nt) {
    for (int k = tid; k < NSEG; k += nt) {
        uint32_t bits = 0;
        walk_segment(s, n, k, [&](int lit, int len, int dist) {
            if (!len) { bits += s.t.llen[lit]; return; }
            int sym, nb, ex;
            len_code(len, sym, nb, ex);
            bits += s.t.llen[sym] + nb;
            dist_code(dist, sym, nb, ex);
            bits += s.t.dlen[sym] + nb;
        });
        s.t.seg_bits[k] = bits;
    }
}

// offsets of the segments' bits, the block's size, stored or not, the member's CRC-32
TCI_HD void decide(member_smem& s, int n, int tid, int nt) {
    (void)nt;
    if (tid != 0) return;
    tables& t = s.t;
    uint32_t at = t.header_bits;
    for (int k = 0; k <= NSEG; ++k) {
        const uint32_t b = k < NSEG ? t.seg_bits[k] : 0;
        t.seg_bits[k] = at;
        at += b;
    }
    t.total_bits = at + t.llen[256];
    const int dyn = (int)((t.total_bits + 7) / 8);
    t.stored = dyn > n + 5;
    t.out_bytes = t.stored ? n + 5 : dyn;
    // the pieces all have the same length except the ones at the end: one power of x serves those
    const int per = (n + NSEG - 1) / NSEG;
    const uint32_t xp = tcinf::crc_x8nmodp((uint64_t)per);
    uint32_t crc = 0;
    for (int k = 0; k < NSEG; ++k) {
        int s0, s1;
        seg_range(n, k, s0, s1);
        if (s1 == s0) continue;
        crc = s1 - s0 == per ? tcinf::crc_multmodp(xp, crc) ^ t.seg_crc[k] : tcinf::crc_combine(crc, t.seg_crc[k], (uint64_t)(s1 - s0));
    }
    t.crc = crc;
}

TCI_HD void zero_out(member_smem& s, uint32_t* out, int tid, int nt) {
    if (s.t.stored) return;
    const int words = (int)((s.t.total_bits + 31) / 32);
    for (int w = tid; w < words; w += nt) out[w] = 0;
}

struct bitw {
    uint32_t* w;
    uint32_t wi;
    uint64_t acc;
    int nb;
};
TCI_HD void or_word(uint32_t* a, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicOr(a, v);
#else
    *a |= v;
#endif
}
TCI_HD void bw_init(bitw& b, uint32_t* w, uint32_t bitpos) { b.w = w; b.wi = bitpos >> 5; b.nb = (int)(bitpos & 31u); b.acc = 0; }
TCI_HD void bw_put(bitw& b, uint32_t v, int n) {          // n <= 16
    b.acc |= (uint64_t)v << b.nb;
    b.nb += n;
    if (b.nb >= 32) { or_word(&b.w[b.wi++], (uint32_t)b.acc); b.acc >>= 32; b.nb -= 32; }
}
TCI_HD void bw_flush(bitw& b) { if (b.nb > 0) or_word(&b.w[b.wi], (uint32_t)b.acc); }

TCI_HD void emit(member_smem& s, int n, uint32_t* out, int tid, int nt) {
    const tables& t = s.t;
    if (t.stored) {
        uint8_t* o = (uint8_t*)out;
        if (tid == 0) { o[0] = 1; o[1] = (uint8_t)n; o[2] = (uint8_t)(n >> 8); o[3] = (uint8_t)~n; o[4] = (uint8_t)(~n >> 8); }
        for (int i = tid; i < n; i += nt) o[5 + i] = s.in[i];
        return;
    }
    for (int k = tid; k <= NSEG; k += nt) {
        bitw b;
        if (k == NSEG) {                                        // the block's header and its end
            bw_init(b, out, 0);
            bw_put(b, 1u | (2u << 1), 3);                       // BFINAL, dynamic Huffman
            bw_put(b, (uint32_t)(t.hlit - 257), 5);
            bw_put(b, (uint32_t)(t.hdist - 1), 5);
            bw_put(b, (uint32_t)(t.hclen - 4), 4);
            for (int i = 0; i < t.hclen; ++i) bw_put(b, t.clen[cl_order(i)], 3);
            for (int i = 0; i < t.n_rle; ++i) {
                const int sym = t.rle[i] & 31;
                bw_put(b, t.ccode[sym], t.clen[sym]);
                if (cl_extra_bits(sym)) bw_put(b, (uint32_t)(t.rle[i] >> 5), cl_extra_bits(sym));
            }
            bw_flush(b);
            bw_init(b, out, t.seg_bits[NSEG]);
            bw_put(b, t.lcode[256], t.llen[256]);
            bw_flush(b);
            continue;
        }
        bw_init(b, out, t.seg_bits[k]);
        walk_segment(s, n, k, [&](int lit, int len, int dist) {
            if (!len) { bw_put(b, t.lcode[lit], t.llen[lit]); return; }
            int sym, nb, ex;
            len_code(len, sym, nb, ex);
            bw_put(b, t.lcode[sym], t.llen[sym]);
            if (nb) bw_put(b, (uint32_t)ex, nb);
            dist_code(dist, sym, nb, ex);
            bw_put(b, t.dcode[sym], t.dlen[sym]);
            if (nb) bw_put(b, (uint32_t)ex, nb);
        });
        bw_flush(b);
    }
}

// ---------------------------------------------------------------- the member
// s.in[0 .. n) holds the member's bytes (n <= MEMBER_MAX).  Writes the raw DEFLATE stream to `out` (4-byte aligned, room
// for n + 8 bytes); afterwards s.t.out_bytes is its length and s.t.crc the CRC-32 of the input.  Device: every thread of the CTA calls this with its own tid (nt = blockDim.x, a multiple of 32).  Host: one
// call runs every thread index of each phase in turn.
#ifdef __CUDA_ARCH__
#define TCD_PHASE(...) do { __VA_ARGS__; __syncthreads(); } while (0)
#else
#define TCD_PHASE(...) do { for (int tid = 0; tid < nt; ++tid) { __VA_ARGS__; } } while (0)
#endif
TCI_HD void deflate_member(member_smem& s, int n, uint32_t* out, int nt, int tid_dev) {
#ifdef __CUDA_ARCH__
    const int tid = tid_dev;
#else
    (void)tid_dev;
#endif
    TCD_PHASE(find_init(s, tid, nt));
    for (int r = 0; r * ROUND < n; ++r) {
        TCD_PHASE(find_round(s, n, r, tid, nt));
        TCD_PHASE(find_insert(s, n, r, tid, nt));
    }
    TCD_PHASE(tables_init(s, tid, nt));
    TCD_PHASE(parse_and_crc(s, n, tid, nt));
    TCD_PHASE(histogram(s, n, tid, nt));
    TCD_PHASE(codes_prepare(s, tid, nt));
    TCD_PHASE(codes_rank(s, tid, nt));
    TCD_PHASE(codes_build(s, tid, nt));
    TCD_PHASE(seg_bits(s, n, tid, nt));
    TCD_PHASE(decide(s, n, tid, nt));
    TCD_PHASE(zero_out(s, out, tid, nt));
    TCD_PHASE(emit(s, n, out, tid, nt));
}
#undef TCD_PHASE

}  // namespace tcdef
