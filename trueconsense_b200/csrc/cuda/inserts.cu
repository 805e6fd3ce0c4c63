// inserts.cu — kernel (2): the insertion caller, TrueConsense/Events.py:47-82 (ExtractInserts).
//
// For every candidate position the reference piles up one column with pysam's DEFAULT arguments
// (Events.py:66): samtools stepper (flag filter 0x704, orphans skipped), max_depth 8000,
// min_base_quality 13; upper-cases the strings and takes collections.Counter's mode (ties: first
// encountered).  Here every candidate column c owns the slots [off, off + (hi - lo)) of an entry table,
// one slot per read whose start lies in (c - longest span, c], and the work is spread over the whole
// GPU in tiles of INS_TILE reads:
//   select   (ins_select_kernel, one CTA per tile) reads the region fetch would return and the stepper
//            would pass; for each the CIGAR walk to the column, the base-quality test and a 63-bit key
//            hashing exactly the characters pysam would print, upper-cased (head character, sign and
//            length of the indel, inserted bases); per tile: number of selected reads, last selected read.
//   admit    (ins_admit_kernel, one CTA per tile) htslib's depth cap (bam_plp_push: a read is dropped
//            when it starts on the column the engine is waiting to emit and more than max_depth reads
//            are live) reduces, for a single-column fetch where every fetched read is still live, to
//            "admitted  <=>  first selected read at its start coordinate, or fewer than max_depth
//            selected reads before it": a rank from the tile prefix; slots that are not admitted
//            entries get the sentinel key.
//   count    (ins_count_kernel, one CTA per candidate) the keys are counted in a shared-memory hash table
//            (count, first slot); the largest count wins, ties go to the key first encountered in file
//            order.  Every entry is then compared character by character with the first entry of its
//            key, so a hash collision is reported (TC_ERR_RANGE) and can never silently change a count.
//            A column with more distinct strings than the table holds falls back to the sorted form:
//            cub::DeviceSegmentedRadixSort (stable) + run-length encoding (ins_mode_kernel).
//   pair     (ins_pair_kernel, one CTA per candidate, only with a base-quality filter) htslib's mate-overlap quality
//            rewriting (pysam's default ignore_overlaps=True: sam.c overlap_push / overlap_remove /
//            tweak_overlap_quality).  The reads pushed for this column and those the depth cap dropped are grouped by
//            QNAME hash in a shared-memory table; per name a tiny automaton in file order replays htslib's hash table
//            (store the first mate, pair it with the next alignment of that name, forget it when a capped read of that
//            name goes by); for every pair one thread replays tweak_overlap_quality's walk over the two CIGARs and
//            keeps what it does to the two base qualities this column tests.  Then the quality test, and the
//            admitted entries are counted.
#include <cub/device/device_segmented_radix_sort.cuh>

#include <memory>
#include <new>

#include "tc_common.cuh"

constexpr int INS_TILE = 256;               // reads per tile == threads per CTA of the select / admit kernels
constexpr uint64_t KEY_NONE = ~0ull;        // slot without an admitted entry (real keys have bit 63 clear)
constexpr int INS_TBL = 4096;               // hash table slots per candidate column (count kernel)
constexpr int INS_BASES_FIXED = 64;         // inserted characters returned with the call itself

struct ins_args {
    dreads r;
    const int32_t* cand;            // [n_cand] 1-based positions
    int n_cand;                     // their number — or, with n_cand_dev, the capacity the buffers were sized for
    const int32_t* n_cand_dev;      // not NULL: the number of candidates lives on the device (tc_pileup_call_inserts: the list comes
                                    // straight from the call kernel's flags, nothing is read back in between)
    uint32_t flag_filter; int min_mapq, min_bq, ignore_orphans; long long max_depth;
    int32_t span_hint;              // > 0: caller's upper bound of the longest reference span (tc_reads_t.max_ref_span)
    int32_t* range;                 // [n_cand][2] lo, hi read indices: the reads with pos in (c - longest span, c]
    uint32_t* range_off;            // [n_cand][4] seq_off[lo], seq_off[hi], cigar_off[lo], cigar_off[hi]
    const int64_t* seg_off;         // [n_cand+1] slot offsets; read r of candidate ci owns slot seg_off[ci] + r - lo
    const int32_t* tile_cand;       // [n_tiles] candidate of every tile
    const int32_t* tile_first;      // [n_cand+1] first tile of every candidate
    int32_t* tile_sel;              // [n_tiles] selected reads in the tile
    int32_t* tile_last;             // [n_tiles] last selected read of the tile, -1 if none
    uint64_t* ent_key; int32_t* ent_indel; int32_t* ent_qpos; uint8_t* ent_head;
    uint8_t* ent_sel;               // bit 0: selected (fetched and passed by the stepper), bit 1: yields an entry (before the base-quality
                                    // test when min_bq > 0: ins_pair_kernel applies it), bit 2: admitted by the depth cap
    uint8_t* ent_q;                 // quality of the base the entry's quality test reads
    uint8_t* pair_q; unsigned long long pair_cap; unsigned long long* pair_bump;   // scratch for the rewritten quality strings of paired reads
    int olap_mode;                  // mate-overlap rewriting: 0 htslib >= 1.13, 1 off, 2 htslib <= 1.12 (tc_pileup_params_t.reserved bits 8-9)
    int32_t* seg_count;             // [n_cand] admitted entries
    int32_t* pair_any;              // [n_cand] some selected read of the column is one of a proper pair (else ins_pair_kernel has nothing to pair)
    int32_t* overflow;              // [1] some column had more distinct keys than INS_TBL holds
    const int32_t* layout;          // device-built layout (ins_layout_kernel): [0] tiles, [1] slots, [2] 1 = did not fit; NULL: host-built
    uint8_t* bases_fixed;           // [n_cand][INS_BASES_FIXED] inserted characters of each winner (longer ones: ins_bases_kernel)
    tc_status* status;
};

__device__ __forceinline__ int ins_ncand(const ins_args& a) { return a.n_cand_dev ? min(*a.n_cand_dev, a.n_cand) : a.n_cand; }

// longest reference span when the caller gave no bound: one thread per read (also checks the sort order)
__global__ void max_span_kernel(dreads r, tc_status* status) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int span = 0;
    if (i < r.n) {
        if (i > 0 && r.pos[i] < r.pos[i - 1]) atomicCAS(&status->err, 0, TC_ERR_UNSORTED);
        for (uint32_t k = r.cigar_off[i]; k < r.cigar_off[i + 1]; ++k) {
            uint32_t c = r.cigar[k];
            if (op_consumes_ref(c & 15u)) span += (int)(c >> 4);
        }
    }
    span = __reduce_max_sync(0xffffffffu, span);
    if ((threadIdx.x & 31) == 0 && span > 0) atomicMax(&status->max_span, span);
}

// reads that can overlap column c: pos in (c - max_span, c].  One warp per candidate; each lower bound is a
// 32-ary search (every round the lanes probe 32 evenly spaced reads): 5 rounds for 2 M reads instead of 21.
__device__ __forceinline__ int warp_lower_bound(const int32_t* __restrict__ pos, int64_t n, int v, int lane) {
    int64_t lo = 0, hi = n;                 // the first read with pos >= v (n if none) lies in [lo, hi]
    while (hi > lo) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t i = lo + (int64_t)lane * step;
        const bool ge = i >= hi || pos[i] >= v;         // a probe past the interval counts as "not smaller"
        const unsigned m = __ballot_sync(0xffffffffu, ge);
        if (m == 0u) { lo = lo + 31 * step + 1; continue; }     // every probe is smaller: the answer lies behind the last one
        const int first = __ffs(m) - 1;
        if (first == 0) return (int)lo;
        hi = min(hi, lo + (int64_t)first * step);       // this probe is >= v ...
        lo = lo + (int64_t)(first - 1) * step + 1;      // ... the one before it is smaller
    }
    return (int)lo;
}

__global__ void cand_range_kernel(ins_args a) {
    const int ci = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (ci >= ins_ncand(a)) return;
    const int c = a.cand[ci] - 1;
    const int ms = max(a.span_hint > 0 ? a.span_hint : a.status->max_span, 1);
    const int lo = warp_lower_bound(a.r.pos, a.r.n, c - ms + 1, lane);
    const int hi = max(lo, warp_lower_bound(a.r.pos, a.r.n, c + 1, lane));
    if (lane == 0) {
        a.range[2 * ci] = lo;
        a.range[2 * ci + 1] = hi;
        a.range_off[4 * ci] = a.r.seq_off[lo]; a.range_off[4 * ci + 1] = a.r.seq_off[hi];
        a.range_off[4 * ci + 2] = a.r.cigar_off[lo]; a.range_off[4 * ci + 3] = a.r.cigar_off[hi];
    }
}

__device__ __forceinline__ uint64_t mix_key(uint64_t h, uint64_t v) {
    h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    return h;
}

// the character pysam prints for base code `code` on a read of the given strand, upper-cased
__device__ __forceinline__ char base_char_upper(uint32_t code, bool rev) {
    const char nt16[17] = "=ACMGRSVTWYHKDBN";
    if (code == 0) return rev ? ',' : '.';      // strand_mark_char maps '=' to '.' / ','
    return nt16[code];
}

__device__ __forceinline__ char ins_char(const ins_args& a, uint32_t read, int qpos, int j, bool rev) {
    const int lq = a.r.l_seq[read];
    const int q = qpos + j;
    if (q >= lq) return 'N';
    return base_char_upper(seq_code(a.r.seq4 + a.r.seq_off[read], q), rev);
}

// what pysam prints for query base q of a read, as a 5-bit symbol: the BAM code, 15 ('N') past the end of SEQ,
// 16 for a reverse-strand '=' (printed ',' where the forward strand prints '.').  Equal symbols <=> equal characters.
struct read_syms {
    const uint32_t* w; int lq; bool rev;
    __device__ __forceinline__ uint32_t sym(int q) const {
        if (q >= lq) return 15u;
        const uint32_t code = seq_code(w, q);
        return (code == 0 && rev) ? 16u : code;
    }
};
__device__ __forceinline__ read_syms read_syms_of(const ins_args& a, uint32_t read) {
    read_syms rs;
    rs.w = a.r.seq4 + a.r.seq_off[read]; rs.lq = a.r.l_seq[read]; rs.rev = (a.r.flag[read] & 16u) != 0;
    return rs;
}

// The slot / tile layout built on the device, so that the ranges need not travel to the host first: slot offsets
// and first tiles per candidate (serial, a handful of candidates), then the candidate of every tile.  When the
// layout does not fit the buffers the host sized speculatively, layout[2] says so and no tile runs.
__global__ void __launch_bounds__(256) ins_layout_kernel(ins_args a, int64_t* __restrict__ seg_off, int32_t* __restrict__ tile_first,
                                                         int32_t* __restrict__ tile_cand, int32_t* __restrict__ layout, int64_t slot_cap, int tile_cap,
                                                         const tc_status* __restrict__ pileup_status, int32_t* __restrict__ rb_extra) {
    __shared__ int n_tiles_s;
    const int n_cand = ins_ncand(a);
    // device-side candidates: their number and positions, and the pileup's status block, travel back with the results
    if (rb_extra) {
        if (threadIdx.x == 0) rb_extra[TC_RB_EXTRA_NCAND] = *a.n_cand_dev;
        if (threadIdx.x < 16) rb_extra[TC_RB_EXTRA_STATUS + threadIdx.x] = pileup_status ? reinterpret_cast<const int32_t*>(pileup_status)[threadIdx.x] : 0;
        for (int i = threadIdx.x; i < n_cand; i += blockDim.x) rb_extra[TC_RB_EXTRA_CAND + i] = a.cand[i];
    }
    if (threadIdx.x == 0) {
        int64_t off = 0; int64_t tiles = 0;
        for (int i = 0; i < n_cand; ++i) {
            seg_off[i] = off; tile_first[i] = (int32_t)min(tiles, (int64_t)0x7fffffff);
            const int64_t len = a.range[2 * i + 1] - a.range[2 * i];
            off += len; tiles += (len + INS_TILE - 1) / INS_TILE;
        }
        seg_off[n_cand] = off; tile_first[n_cand] = (int32_t)min(tiles, (int64_t)0x7fffffff);
        const bool fits = off <= slot_cap && tiles <= tile_cap && !(a.n_cand_dev && *a.n_cand_dev > a.n_cand);
        layout[0] = fits ? (int32_t)tiles : 0;
        layout[1] = (int32_t)min(off, (int64_t)0x7fffffff);
        layout[2] = fits ? 0 : 1;
        n_tiles_s = fits ? (int)tiles : 0;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < n_tiles_s; t += blockDim.x) {
        int lo = 0, hi = n_cand - 1;            // last candidate whose first tile is <= t
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (tile_first[mid] <= t) lo = mid; else hi = mid - 1; }
        tile_cand[t] = lo;
    }
}

// select: one thread per read of the candidate's range
__global__ void __launch_bounds__(INS_TILE) ins_select_kernel(ins_args a) {
    __shared__ int wlast[INS_TILE / 32];
    const int tile = blockIdx.x;
    if (a.layout && tile >= a.layout[0]) return;
    const int ci = a.tile_cand[tile];
    const int c = a.cand[ci] - 1;
    const int lo = a.range[2 * ci], hi = a.range[2 * ci + 1];
    const int r = lo + (tile - a.tile_first[ci]) * INS_TILE + threadIdx.x;
    bool sel = false, emit = false, proper = false;
    if (r < hi) {
        const int pos = a.r.pos[r];
        if (r > 0 && pos < a.r.pos[r - 1]) atomicCAS(&a.status->err, 0, TC_ERR_UNSORTED);
        const uint32_t fl = a.r.flag[r];
        const bool pass = !(fl & (a.flag_filter | 4u)) && !(a.min_mapq > 0 && a.r.mapq && (int)a.r.mapq[r] < a.min_mapq) &&
                          !(a.ignore_orphans && (fl & 1u) && !(fl & 2u));
        int indel = 0, qpos = 0, qv = 0; char head = 0; uint64_t key = KEY_NONE;
        if (pass) {
            // CIGAR walk up to the column.  BAI query: pos < c+1 && endpos > c, where a read without reference
            // span has endpos = pos + 1
            const uint32_t c0 = a.r.cigar_off[r];
            const int n = (int)(a.r.cigar_off[r + 1] - c0);
            const uint32_t* cig = a.r.cigar + c0;
            const bool rev = (fl & 16u) != 0;
            const int lq = a.r.l_seq[r];
            int x = pos, y = 0;
            bool found = false;
            for (int k = 0; k < n; ++k) {
                const uint32_t cc = cig[k]; const uint32_t op = cc & 15u; const int l = (int)(cc >> 4);
                if (!op_consumes_ref(op)) { if (op == OP_I || op == OP_S) y += l; continue; }
                if (c < x + l) {
                    found = true;
                    const bool match = op_is_match(op);
                    qpos = match ? y + (c - x) : y;
                    if (c == x + l - 1) indel = peek_indel(cig, n, k);
                    qv = (qpos < lq) ? (int)a.r.qual[8ull * a.r.seq_off[r] + qpos] : 0;
                    if (qv >= a.min_bq || a.min_bq > 0) {      // with a filter: decided after the mate-overlap rewriting
                        emit = true;
                        if (match) head = (qpos < lq) ? base_char_upper(seq_code(a.r.seq4 + a.r.seq_off[r], qpos), rev) : 'N';
                        else head = (op == OP_N) ? (rev ? '<' : '>') : '*';
                    }
                    break;
                }
                if (op_is_match(op)) y += l;
                x += l;
            }
            // a read without reference span is only linked into htslib's list when it sits on the column; it never
            // yields an entry, and it counts towards the live total like any selected read
            sel = found || (x == pos && pos == c);
            if (emit) {
                const read_syms rs = read_syms_of(a, r);
                bool exact = false;
                if (indel <= 8 && indel > -8192) {
                    // the whole string fits the key: bit 62 = exact, bit 61 = 0, head character (7 bits), indel + 8192,
                    // 5 bits per inserted character (BAM code; 16 = the ',' a reverse-strand '=' prints as) —
                    // equal keys <=> equal strings, no verification needed
                    exact = true;
                    key = (1ull << 62) | ((uint64_t)((uint8_t)head & 127u) << 54) | ((uint64_t)(uint32_t)(indel + 8192) << 40);
                    for (int j = 1; j <= indel; ++j) key |= (uint64_t)rs.sym(qpos + j) << (5 * (j - 1));
                } else if (indel <= 12) {
                    // 9..12 inserted characters at 4 bits each (bit 61 = 1), unless one of them is a reverse-strand '='
                    exact = true;
                    key = (3ull << 61) | ((uint64_t)((uint8_t)head & 127u) << 54) | ((uint64_t)(uint32_t)indel << 48);
                    for (int j = 1; j <= indel; ++j) {
                        const uint32_t sy = rs.sym(qpos + j);
                        exact = exact && sy < 16u;
                        key |= (uint64_t)(sy & 15u) << (4 * (j - 1));
                    }
                }
                if (!exact) {
                    key = mix_key(0x7463696e73ull, (uint64_t)(uint8_t)head);
                    key = mix_key(key, (uint64_t)(uint32_t)indel);
                    for (int j = 1; j <= indel; ++j) key = mix_key(key, (uint64_t)(uint8_t)ins_char(a, r, qpos, j, rev));
                    key &= 0x3fffffffffffffffull;       // hashed: bit 62 clear, verified entry by entry in the count
                }
            }
        }
        const int64_t slot = a.seg_off[ci] + (r - lo);
        a.ent_key[slot] = key; a.ent_indel[slot] = indel; a.ent_qpos[slot] = qpos; a.ent_head[slot] = (uint8_t)head;
        a.ent_sel[slot] = (uint8_t)((sel ? 1 : 0) | (emit ? 2 : 0));
        a.ent_q[slot] = (uint8_t)qv;
        proper = sel && (fl & 2u);
    }
    if (__syncthreads_or(proper) && threadIdx.x == 0) a.pair_any[ci] = 1;
    const int nsel = __syncthreads_count(sel);
    int last = __reduce_max_sync(0xffffffffu, sel ? r : -1);
    if ((threadIdx.x & 31) == 0) wlast[threadIdx.x >> 5] = last;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 0; w < INS_TILE / 32; ++w) last = max(last, wlast[w]);
        a.tile_sel[tile] = nsel;
        a.tile_last[tile] = last;
    }
}

// admit: the depth cap, from the rank of every selected read among the candidate's selected reads
__global__ void __launch_bounds__(INS_TILE) ins_admit_kernel(ins_args a) {
    __shared__ int wsum[INS_TILE / 32], wlast[INS_TILE / 32];
    __shared__ long long base_s;
    __shared__ int prev_s;
    const int tile = blockIdx.x;
    if (a.layout && tile >= a.layout[0]) return;
    const int ci = a.tile_cand[tile];
    const int lo = a.range[2 * ci], hi = a.range[2 * ci + 1];
    const int t0 = a.tile_first[ci];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp == 0) {        // selected reads and last selected read of the candidate's earlier tiles
        long long base = 0; int prev = -1;
        for (int t = t0 + lane; t < tile; t += 32) { base += a.tile_sel[t]; prev = max(prev, a.tile_last[t]); }
#pragma unroll
        for (int o = 16; o; o >>= 1) { base += __shfl_xor_sync(0xffffffffu, base, o); prev = max(prev, __shfl_xor_sync(0xffffffffu, prev, o)); }
        if (lane == 0) { base_s = base; prev_s = prev; }
    }
    const int r = lo + (tile - t0) * INS_TILE + threadIdx.x;
    const int64_t slot = a.seg_off[ci] + (r - lo);
    const uint8_t es = r < hi ? a.ent_sel[slot] : 0;
    const bool sel = (es & 1) != 0, emit = (es & 2) != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, sel);
    int m = sel ? r : -1;       // nearest selected read at or before this one, within the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, m, o); if (lane >= o) m = max(m, t); }
    int prev = __shfl_up_sync(0xffffffffu, m, 1);
    if (lane == 0) prev = -1;
    if (lane == 31) wlast[warp] = m;
    if (lane == 0) wsum[warp] = __popc(bal);
    __syncthreads();
    long long rank = base_s + __popc(bal & ((1u << lane) - 1));
    prev = max(prev, prev_s);
    for (int w = 0; w < warp; ++w) { rank += wsum[w]; prev = max(prev, wlast[w]); }
    bool admitted = false;
    if (sel) {
        const bool first_at_start = prev < 0 || a.r.pos[prev] != a.r.pos[r];
        admitted = first_at_start || rank < a.max_depth;
    }
    if (a.min_bq > 0) {         // the quality test (after the mate-overlap rewriting) and the count: ins_pair_kernel
        if (r < hi && admitted) a.ent_sel[slot] = (uint8_t)(es | 4);
        return;
    }
    if (emit && !admitted) a.ent_key[slot] = KEY_NONE;
    const int n_adm = __syncthreads_count(emit && admitted);
    if (threadIdx.x == 0 && n_adm) atomicAdd(&a.seg_count[ci], n_adm);
}

// ---------------------------------------------------------------- mate overlaps (htslib sam.c)
// khash.h __ac_Wang_hash: which mate keeps its qualities is drawn from it (htslib >= 1.13)
__device__ __forceinline__ uint32_t wang_hash(uint32_t key) {
    key += ~(key << 15); key ^= (key >> 10); key += (key << 3); key ^= (key >> 6); key += ~(key << 11); key ^= (key >> 16);
    return key;
}

// cigar_iref2iseq_set / cigar_iref2iseq_next: walk to the first / next M,=,X base
struct cwalk { const uint32_t* cig; const uint32_t* end; long long icig, iseq, iref; };

__device__ int iref2iseq_set(cwalk& w, long long pos) {
    if (pos < 0) return -1;
    w.icig = 0; w.iseq = 0; w.iref = 0;
    while (w.cig < w.end) {
        const uint32_t cig = *w.cig & 15u; const long long ncig = (long long)(*w.cig >> 4);
        if (cig == OP_S) { w.cig++; w.iseq += ncig; w.icig = 0; continue; }
        if (cig == OP_H || cig == OP_P) { w.cig++; w.icig = 0; continue; }
        if (cig == OP_M || cig == OP_EQ || cig == OP_X) {
            pos -= ncig;
            if (pos < 0) { w.icig = ncig + pos; w.iseq += w.icig; w.iref += w.icig; return 0; }
            w.cig++; w.iseq += ncig; w.icig = 0; w.iref += ncig;
            continue;
        }
        if (cig == OP_I) { w.cig++; w.iseq += ncig; w.icig = 0; continue; }
        if (cig == OP_D || cig == OP_N) { pos -= ncig; if (pos < 0) pos = 0; w.cig++; w.icig = 0; w.iref += ncig; continue; }
        return -2;
    }
    w.iseq = -1;
    return -1;
}

__device__ int iref2iseq_next(cwalk& w) {
    while (w.cig < w.end) {
        const uint32_t cig = *w.cig & 15u; const long long ncig = (long long)(*w.cig >> 4);
        if (cig == OP_M || cig == OP_EQ || cig == OP_X) {
            if (w.icig >= ncig - 1) { w.icig = -1; w.cig++; continue; }
            w.iseq++; w.icig++; w.iref++;
            return 0;
        }
        if (cig == OP_D || cig == OP_N) { w.cig++; w.iref += ncig; w.icig = -1; continue; }
        if (cig == OP_I || cig == OP_S) { w.cig++; w.iseq += ncig; w.icig = -1; continue; }
        if (cig == OP_H || cig == OP_P) { w.cig++; w.icig = -1; continue; }
        return -2;
    }
    w.iseq = -1; w.iref = -1;
    return -1;
}

// tweak_overlap_quality(a, b), a the first-arrived read, replayed literally on scratch copies aq / bq of the two reads' base
// qualities.  (Only two of the rewritten values matter to a column, but htslib's catch-up around deletions can visit a
// base twice and then rewrites it from the already rewritten value opposite it — so the whole state is carried.)
__device__ void tweak_pair(const ins_args& a, uint32_t ra, uint32_t rb, uint8_t* aq, uint8_t* bq, int mode) {
    const uint32_t* a_first = a.r.cigar + a.r.cigar_off[ra]; const uint32_t* b_first = a.r.cigar + a.r.cigar_off[rb];
    cwalk wa = {a_first, a.r.cigar + a.r.cigar_off[ra + 1], 0, 0, 0}, wb = {b_first, a.r.cigar + a.r.cigar_off[rb + 1], 0, 0, 0};
    const long long apos = a.r.pos[ra], bpos = a.r.pos[rb], alq = a.r.l_seq[ra], blq = a.r.l_seq[rb];
    long long iref = bpos;
    int a_ret = iref2iseq_set(wa, iref - apos);
    if (a_ret < 0) return;
    int b_ret = iref2iseq_set(wb, iref - bpos);
    if (b_ret < 0) return;
    int amul = 1, bmul = 0;
    if (mode == 0) { if (wang_hash((uint32_t)a.r.qname_hash[ra]) & 1u) { amul = 1; bmul = 0; } else { amul = 0; bmul = 1; } }
    for (;;) {
        while (a_ret >= 0 && wa.iref >= 0 && wa.iref < iref - apos) a_ret = iref2iseq_next(wa);
        if (a_ret < 0) break;
        if (iref < wa.iref + apos) iref = wa.iref + apos;
        while (b_ret >= 0 && wb.iref >= 0 && wb.iref < iref - bpos) b_ret = iref2iseq_next(wb);
        if (b_ret < 0) break;
        if (iref < wb.iref + bpos) iref = wb.iref + bpos;
        iref++;
        if (wa.iref + apos != wb.iref + bpos) {
            if (mode != 0) continue;            // htslib <= 1.12: only positions both reads match
            if (wa.iref + apos < wb.iref + bpos && wb.cig > b_first && (*(wb.cig - 1) & 15u) == OP_D) {
                bool done = false;
                do {        // a deletion in b: a catches up, its bases under the deletion are down-weighted
                    if (wa.iseq < alq) aq[wa.iseq] = amul ? (uint8_t)((int)aq[wa.iseq] * 4 / 5) : (uint8_t)0;
                    a_ret = iref2iseq_next(wa);
                    if (a_ret < 0) { done = true; break; }
                } while (wa.iref + apos < wb.iref + bpos);
                if (done) return;
            } else if (wa.cig > a_first && (*(wa.cig - 1) & 15u) == OP_D) {
                bool done = false;
                do {
                    if (wb.iseq < blq) bq[wb.iseq] = bmul ? (uint8_t)((int)bq[wb.iseq] * 4 / 5) : (uint8_t)0;
                    b_ret = iref2iseq_next(wb);
                    if (b_ret < 0) { done = true; break; }
                } while (wb.iref + bpos < wa.iref + apos);
                if (done) return;
            } else continue;
        }
        if (wa.iseq >= alq || wb.iseq >= blq) return;
        const int oa = aq[wa.iseq], ob = bq[wb.iseq];
        int na, nb;
        if (seq_code(a.r.seq4 + a.r.seq_off[ra], (int)wa.iseq) == seq_code(a.r.seq4 + a.r.seq_off[rb], (int)wb.iseq)) {
            const int sum = min(oa + ob, 200);
            na = amul * sum; nb = bmul * sum;
        } else if (mode == 0) {
            if (oa > ob) { na = oa * 4 / 5; nb = 0; }
            else if (oa < ob) { nb = ob * 4 / 5; na = 0; }
            else { na = amul * (oa * 4 / 5); nb = bmul * (ob * 4 / 5); }
        } else {
            if (oa >= ob) { na = oa * 4 / 5; nb = 0; } else { nb = ob * 4 / 5; na = 0; }
        }
        aq[wa.iseq] = (uint8_t)na; bq[wb.iseq] = (uint8_t)nb;
    }
}

constexpr int PAIR_TBL = 16384;             // QNAME groups per candidate column (pushed reads <= max_depth + distinct starts)

// overlap_push's conditions on a pushed read: a proper pair whose mate is mapped on this reference and can overlap
__device__ bool olap_eligible(const ins_args& a, uint32_t r) {
    const uint32_t fl = a.r.flag[r];
    if ((fl & 8u) || !(fl & 2u)) return false;
    const int mp = a.r.mpos[r];
    if (mp == -2) return false;                         // the mate is on another reference
    long long isz = a.r.isize[r]; if (isz < 0) isz = -isz;
    if (isz >= 2ll * a.r.l_seq[r]) {                    // "no overlap possible, unless some wild cigar"
        int end = a.r.pos[r];
        for (uint32_t k = a.r.cigar_off[r]; k < a.r.cigar_off[r + 1]; ++k) { const uint32_t c = a.r.cigar[k]; if (op_consumes_ref(c & 15u)) end += (int)(c >> 4); }
        if (mp >= end) return false;
    }
    return true;
}

// One CTA per candidate.  Events of the column in file order: a pushed read (selected and admitted, with a reference
// span) or a read the depth cap dropped (htslib calls overlap_remove on it: whatever is stored under its name is
// forgotten).  They are grouped by QNAME hash; per group the automaton of htslib's olap_hash.
__global__ void __launch_bounds__(1024) ins_pair_kernel(ins_args a) {
    extern __shared__ __align__(16) unsigned char pair_smem[];
    unsigned int* tmin = reinterpret_cast<unsigned int*>(pair_smem);        // [PAIR_TBL] first event of the group + 1 (0: empty)
    unsigned int* tmax = tmin + PAIR_TBL;                                   // [PAIR_TBL] last event + 1
    unsigned short* tcnt = reinterpret_cast<unsigned short*>(tmax + PAIR_TBL);  // [PAIR_TBL] events
    __shared__ int over_s, nadm_s;
    const int ci = blockIdx.x;
    if (ci >= ins_ncand(a)) return;
    if (a.layout && a.layout[2]) return;
    const int64_t off = a.seg_off[ci];
    const int lo = a.range[2 * ci];
    const int n = a.range[2 * ci + 1] - lo;
    const bool pairing = a.olap_mode != 1 && a.r.qname_hash && a.r.mpos && a.r.isize && a.pair_any[ci];
    if (threadIdx.x == 0) { over_s = 0; nadm_s = 0; }
    if (pairing) {
        for (int i = threadIdx.x; i < PAIR_TBL; i += blockDim.x) { tmin[i] = 0u; tmax[i] = 0u; tcnt[i] = 0; }
        __syncthreads();
        // an event: pushed (bits 0 and 2, a reference span: its entry bit or a later column) or capped (bit 0 without bit 2)
        auto is_event = [&](int i, bool& push) -> bool {
            const uint8_t es = a.ent_sel[off + i];
            if (!(es & 1)) return false;
            if (!(es & 4)) { push = false; return true; }
            push = true;
            return true;
        };
        // pass 1: the pushed reads of proper pairs open the groups (at most max_depth + a few of them); pass 2: the reads the
        // depth cap dropped only JOIN the group of their name, if there is one (a deep unpaired sample drops tens of thousands
        // of reads per column: none of them may take a table slot)
        for (int pass = 0; pass < 2; ++pass) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                bool push;
                if (!is_event(i, push) || push != (pass == 0)) continue;
                const uint32_t r = (uint32_t)(lo + i);
                if (push && !(a.r.flag[r] & 2u)) continue;          // never in the table, never paired
                const unsigned long long k = a.r.qname_hash[r];
                unsigned h = (unsigned)(k ^ (k >> 31)) & (PAIR_TBL - 1);
                int probes = 0;
                for (;;) {
                    const unsigned cur = push ? atomicCAS(&tmin[h], 0u, (unsigned)i + 1u) : tmin[h];
                    if (cur == 0u && !push) break;                  // no pushed read of that name
                    if (cur == 0u || a.r.qname_hash[lo + cur - 1] == k) {
                        atomicMin(&tmin[h], (unsigned)i + 1u); atomicMax(&tmax[h], (unsigned)i + 1u);
                        // (16-bit counter: an atomic on the containing word)
                        atomicAdd(reinterpret_cast<unsigned int*>(tcnt) + (h >> 1), (h & 1) ? 0x10000u : 1u);
                        break;
                    }
                    h = (h + 1) & (PAIR_TBL - 1);
                    if (++probes >= PAIR_TBL * 3 / 4) { over_s = 1; break; }
                }
            }
            __syncthreads();
        }
        __syncthreads();
        if (over_s) { if (threadIdx.x == 0) atomicCAS(&a.status->err, 0, TC_ERR_CAPACITY); return; }
        for (int h = threadIdx.x; h < PAIR_TBL; h += blockDim.x) {
            const int cnt = tcnt[h];
            if (cnt < 2) continue;
            const int first = (int)tmin[h] - 1, last = (int)tmax[h] - 1;
            const unsigned long long k = a.r.qname_hash[lo + first];
            int stored = -1;
            int seen = 0;
            for (int i = first; i <= last && seen < cnt; i = (cnt == 2 && i == first) ? last : i + 1) {
                bool push;
                if (!is_event(i, push)) continue;
                const uint32_t r = (uint32_t)(lo + i);
                if (a.r.qname_hash[r] != k || (push && !(a.r.flag[r] & 2u))) continue;
                ++seen;
                if (!push) { stored = -1; continue; }                       // overlap_remove by name
                if (!olap_eligible(a, r)) continue;
                // a read without reference span is never linked (sel without a span: no overlap_push)
                bool has_span = false;
                for (uint32_t q = a.r.cigar_off[r]; q < a.r.cigar_off[r + 1] && !has_span; ++q) { const uint32_t c = a.r.cigar[q]; has_span = op_consumes_ref(c & 15u) && (c >> 4) > 0; }
                if (!has_span) continue;
                if (stored < 0) {
                    const int mp = a.r.mpos[r];
                    if (mp >= a.r.pos[r] || ((a.r.flag[r] & 1u) && mp == -1)) stored = i;     // the mate is still to arrive
                    continue;
                }
                // pair (stored, i): tweak_overlap_quality on scratch copies of the two quality strings, then the two values the
                // column tests
                const int64_t sa = off + stored, sb = off + i;
                const uint32_t ra = (uint32_t)(lo + stored);
                const int la = a.r.l_seq[ra], lb = a.r.l_seq[r];
                const unsigned long long at = atomicAdd(a.pair_bump, (unsigned long long)(la + lb));
                if (at + (unsigned long long)(la + lb) <= a.pair_cap) {
                    uint8_t* aq = a.pair_q + at; uint8_t* bq = aq + la;
                    const uint8_t* ga = a.r.qual + 8ull * a.r.seq_off[ra]; const uint8_t* gb = a.r.qual + 8ull * a.r.seq_off[r];
                    for (int q = 0; q < la; ++q) aq[q] = ga[q];
                    for (int q = 0; q < lb; ++q) bq[q] = gb[q];
                    tweak_pair(a, ra, r, aq, bq, a.olap_mode);
                    if ((a.ent_sel[sa] & 2) && a.ent_qpos[sa] < la) a.ent_q[sa] = aq[a.ent_qpos[sa]];
                    if ((a.ent_sel[sb] & 2) && a.ent_qpos[sb] < lb) a.ent_q[sb] = bq[a.ent_qpos[sb]];
                } else atomicOr(a.overflow, 2);         // the scratch is too small: the host sizes it from pair_bump and runs again
                stored = -1;
            }
        }
        __syncthreads();
    }
    // the quality test and the count of admitted entries
    int mine = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const uint8_t es = a.ent_sel[off + i];
        const bool ok = (es & 6) == 6 && (int)a.ent_q[off + i] >= a.min_bq;
        if (!ok) a.ent_key[off + i] = KEY_NONE;
        mine += ok ? 1 : 0;
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&nadm_s, mine);
    __syncthreads();
    if (threadIdx.x == 0) a.seg_count[ci] = nadm_s;
}

__device__ __forceinline__ bool same_entry(const ins_args& a, int lo, int64_t off, uint32_t e1, uint32_t e2) {
    if (a.ent_head[e1] != a.ent_head[e2] || a.ent_indel[e1] != a.ent_indel[e2]) return false;
    const int indel = a.ent_indel[e1];
    if (indel <= 0) return true;
    const read_syms s1 = read_syms_of(a, (uint32_t)(lo + (int64_t)e1 - off)), s2 = read_syms_of(a, (uint32_t)(lo + (int64_t)e2 - off));
    const int q1 = a.ent_qpos[e1], q2 = a.ent_qpos[e2];
    for (int j = 1; j <= indel; ++j)
        if (s1.sym(q1 + j) != s2.sym(q2 + j)) return false;
    return true;
}

// printed character of a 5-bit symbol (read_syms::sym): "=ACMGRSVTWYHKDBN"[code], '.' / ',' for '='
__device__ __forceinline__ uint8_t sym_char(uint32_t sym) {
    if (sym == 0u) return (uint8_t)'.';
    if (sym == 16u) return (uint8_t)',';
    const unsigned long long t = sym < 8u ? 0x565352474d43413dull : 0x4e42444b48595754ull;
    return (uint8_t)(t >> (8u * (sym & 7u)));
}

__device__ __forceinline__ void write_call(const ins_args& a, int ci, int m, unsigned long long best, tc_insert_call_t* calls) {
    const int64_t off = a.seg_off[ci];
    tc_insert_call_t out;
    out.pos = a.cand[ci]; out.n_entries = m; out.mode_count = 0; out.first_read = -1; out.head = 0; out.indel = 0; out.bases_off = -1;
    if (m > 0) {
        const uint32_t e = (uint32_t)off + (uint32_t)(0xffffffffull - (best & 0xffffffffull));
        out.mode_count = (int32_t)(best >> 32);
        out.first_read = (int32_t)(a.range[2 * ci] + (int64_t)e - off);
        out.head = a.ent_head[e];
        out.indel = a.ent_indel[e];
        out.bases_off = (int64_t)e;         // entry id for now; the host turns it into a buffer offset
        if (out.indel > 0 && out.indel <= INS_BASES_FIXED) {
            const read_syms rs = read_syms_of(a, (uint32_t)out.first_read);
            const int q = a.ent_qpos[e];
            for (int j = 1; j <= out.indel; ++j) a.bases_fixed[(size_t)ci * INS_BASES_FIXED + j - 1] = sym_char(rs.sym(q + j));
        }
    }
    calls[ci] = out;
}

// count: one CTA per candidate, keys counted in a shared-memory hash table (linear probing)
__global__ void __launch_bounds__(1024) ins_count_kernel(ins_args a, tc_insert_call_t* __restrict__ calls) {
    extern __shared__ __align__(16) unsigned char ins_smem[];
    unsigned long long* tkey = reinterpret_cast<unsigned long long*>(ins_smem);     // [INS_TBL]
    unsigned int* tcnt = reinterpret_cast<unsigned int*>(tkey + INS_TBL);           // [INS_TBL]
    unsigned int* tfirst = tcnt + INS_TBL;                                          // [INS_TBL] first slot (file order) of the key
    __shared__ unsigned long long best_s;
    __shared__ int over_s, hashed_s;
    const int ci = blockIdx.x;
    if (ci >= ins_ncand(a)) return;
    if (a.layout && a.layout[2]) return;        // the speculative layout did not fit: the host sizes it and runs again
    const int64_t off = a.seg_off[ci];
    const int lo = a.range[2 * ci];
    const int n = a.range[2 * ci + 1] - lo;
    for (int i = threadIdx.x; i < INS_TBL; i += blockDim.x) { tkey[i] = KEY_NONE; tcnt[i] = 0; tfirst[i] = 0xffffffffu; }
    if (threadIdx.x == 0) { best_s = 0ull; over_s = 0; hashed_s = 0; }
    __syncthreads();
    // four keys per thread are in flight at a time (the loop is bound by the latency of these loads)
    for (int base = 0; base < n; base += 4 * (int)blockDim.x) {
        unsigned long long kk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * (int)blockDim.x + (int)threadIdx.x;
            kk[u] = i < n ? a.ent_key[off + i] : KEY_NONE;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * (int)blockDim.x + (int)threadIdx.x;
            const unsigned long long k = kk[u];
            // lanes holding the same key insert once (most entries of a column print the same string)
            const unsigned grp = __match_any_sync(0xffffffffu, k);
            if (k == KEY_NONE || (__ffs(grp) - 1) != (int)(threadIdx.x & 31)) continue;
            if (!(k >> 62)) hashed_s = 1;       // a hashed key (an insertion longer than 12): entries get verified below
            unsigned h = (unsigned)(k ^ (k >> 29)) & (INS_TBL - 1);
            int probes = 0;
            for (;;) {
                const unsigned long long old = atomicCAS(&tkey[h], KEY_NONE, k);
                if (old == KEY_NONE || old == k) { atomicAdd(&tcnt[h], (unsigned)__popc(grp)); atomicMin(&tfirst[h], (unsigned)i); break; }
                h = (h + 1) & (INS_TBL - 1);
                if (++probes >= INS_TBL * 7 / 8) { over_s = 1; break; }
            }
        }
    }
    __syncthreads();
    if (over_s) { if (threadIdx.x == 0) atomicOr(a.overflow, 1); return; }
    // hashed keys (insertions longer than 12): every entry against the first entry of its key
    if (hashed_s)
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned long long k = a.ent_key[off + i];
        if (k == KEY_NONE || (k >> 62)) continue;      // exact keys need no check
        unsigned h = (unsigned)(k ^ (k >> 29)) & (INS_TBL - 1);
        while (tkey[h] != k) h = (h + 1) & (INS_TBL - 1);
        const unsigned f = tfirst[h];
        if (f != (unsigned)i && !same_entry(a, lo, off, (uint32_t)(off + f), (uint32_t)(off + i))) atomicCAS(&a.status->err, 0, TC_ERR_RANGE);
    }
    unsigned long long best = 0ull;
    for (int i = threadIdx.x; i < INS_TBL; i += blockDim.x)
        if (tcnt[i]) best = max(best, ((unsigned long long)tcnt[i] << 32) | (0xffffffffull - (unsigned long long)tfirst[i]));
    atomicMax(&best_s, best);
    __syncthreads();
    if (threadIdx.x == 0) write_call(a, ci, a.seg_count[ci], best_s, calls);
}

// sorted form of the count: one CTA per candidate over its radix-sorted keys (KEY_NONE slots sort last)
__global__ void __launch_bounds__(1024) ins_mode_kernel(ins_args a, const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sidx,
                                                        tc_insert_call_t* __restrict__ calls) {
    __shared__ unsigned long long best_s;
    const int ci = blockIdx.x;
    const int64_t off = a.seg_off[ci];
    const int lo_read = a.range[2 * ci];
    const int m = a.seg_count[ci];
    if (threadIdx.x == 0) best_s = 0ull;
    __syncthreads();
    unsigned long long best = 0ull;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const uint64_t k = skey[off + i];
        // run head = first element with this key
        int lo = 0, hi = i;
        while (lo < hi) { int mid = (lo + hi) >> 1; if (skey[off + mid] < k) lo = mid + 1; else hi = mid; }
        const int head = lo;
        if (head != i) {
            if (!(k >> 62) && !same_entry(a, lo_read, off, sidx[off + head], sidx[off + i])) atomicCAS(&a.status->err, 0, TC_ERR_RANGE);
        } else {
            int l2 = i, h2 = m;
            while (l2 < h2) { int mid = (l2 + h2) >> 1; if (skey[off + mid] <= k) l2 = mid + 1; else h2 = mid; }
            unsigned long long cnt = (unsigned long long)(l2 - i);
            // stable sort: the head of a run is its earliest entry in file order
            unsigned long long first = (unsigned long long)(sidx[off + i] - (uint32_t)off);
            unsigned long long v = (cnt << 32) | (0xffffffffull - first);
            best = max(best, v);
        }
    }
    atomicMax(&best_s, best);
    __syncthreads();
    if (threadIdx.x == 0) write_call(a, ci, m, best_s, calls);
}

__global__ void iota_kernel(uint32_t* __restrict__ idx, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (uint32_t)i;
}

__global__ void ins_bases_kernel(ins_args a, const tc_insert_call_t* __restrict__ calls, const int64_t* __restrict__ entry_of,
                                 uint8_t* __restrict__ bases) {
    const int ci = blockIdx.x;
    const tc_insert_call_t c = calls[ci];
    if (c.indel <= INS_BASES_FIXED) return;
    const uint32_t e = (uint32_t)entry_of[ci];
    const uint32_t r = (uint32_t)c.first_read;
    const bool rev = (a.r.flag[r] & 16u) != 0;
    for (int j = threadIdx.x; j < c.indel; j += blockDim.x) bases[c.bases_off + j] = (uint8_t)ins_char(a, r, a.ent_qpos[e], j + 1, rev);
}

// ---------------------------------------------------------------- host side, shared by both drivers
// The results block: status, device-built layout, overflow flags, pair-scratch bump; with_extra (the chained form) the
// candidate count, the pileup's status and the candidates; then seg_count / pair_any, the calls and their inserted
// characters.  n_cand: the candidates, or the capacity the chained form enqueues for.
static ins_block ins_block_of(int n_cand, bool with_extra) {
    static_assert(sizeof(tc_status) <= 64, "tc_status outgrew its place in the results block");
    ins_block b;
    b.layout = 64; b.over = 80; b.bump = 88;
    b.extra = with_extra ? 128 : 0;
    b.seg = with_extra ? b.extra + 4 * (TC_RB_EXTRA_CAND + (size_t)n_cand) : 96;
    b.calls = b.seg + ((4 * (2 * (size_t)n_cand + 2) + 15) & ~(size_t)15);
    b.fixed = b.calls + sizeof(tc_insert_call_t) * (size_t)n_cand;
    b.bytes = b.fixed + (size_t)n_cand * INS_BASES_FIXED;
    return b;
}

// One slab (SLOT_INS_D) for T entry slots and NT tiles: keys, indel, qpos, head, sel, quality per slot; tile tables;
// per-candidate offsets.  The pair scratch, the per-candidate words of the results block and p's filter fields.
static int ins_bind(tc_ctx* ctx, ins_args& a, uint8_t* d_rb, const ins_block& rb, size_t T, size_t NT, int n_cand, const tc_pileup_params_t* p) {
    const size_t bytes = T * (8 + 4 + 4 + 1 + 1 + 1) + NT * 12 + ((size_t)n_cand + 1) * 16 + 256 + 16;
    uint8_t* slab = (uint8_t*)tc_dev_buf(ctx, SLOT_INS_D, bytes);
    if (!slab) return TC_ERR_NOMEM;
    a.ent_key = (uint64_t*)slab;
    int64_t* d_off = (int64_t*)(a.ent_key + T);
    a.seg_off = d_off;
    a.ent_indel = (int32_t*)(d_off + n_cand + 1); a.ent_qpos = a.ent_indel + T;
    int32_t* d_tcand = a.ent_qpos + T; int32_t* d_tfirst = d_tcand + NT;
    a.tile_cand = d_tcand; a.tile_first = d_tfirst;
    a.tile_sel = d_tfirst + n_cand + 1; a.tile_last = a.tile_sel + NT;
    a.ent_head = (uint8_t*)(a.tile_last + NT); a.ent_sel = a.ent_head + T; a.ent_q = a.ent_sel + T;
    a.seg_count = (int32_t*)(d_rb + rb.seg); a.pair_any = a.seg_count + n_cand + 1; a.overflow = (int32_t*)(d_rb + rb.over);
    a.bases_fixed = d_rb + rb.fixed;
    if (ctx->pair_cap <= 0) ctx->pair_cap = 1 << 22;
    a.pair_bump = (unsigned long long*)(d_rb + rb.bump); a.pair_cap = (unsigned long long)ctx->pair_cap;
    a.pair_q = (uint8_t*)tc_dev_buf(ctx, SLOT_INS_F, (size_t)ctx->pair_cap);
    if (!a.pair_q) return TC_ERR_NOMEM;
    a.flag_filter = p->flag_filter; a.min_mapq = p->min_mapq; a.min_bq = p->min_base_quality; a.ignore_orphans = p->ignore_orphans;
    a.olap_mode = (p->reserved >> 8) & 3;
    a.max_depth = p->max_depth > 0 ? p->max_depth : (1ll << 62);
    return TC_OK;
}

// the slot / tile layout built on the device into the bound buffers (T slots, NT tiles); rb.extra: the chained form's extra section
static int ins_layout_dev(tc_ctx* ctx, ins_args& a, uint8_t* d_rb, const ins_block& rb, size_t T, size_t NT, const tc_status* pileup_status,
                          cudaStream_t s) {
    int32_t* d_layout = (int32_t*)(d_rb + rb.layout);
    a.layout = d_layout;
    ins_layout_kernel<<<1, 256, 0, s>>>(a, const_cast<int64_t*>(a.seg_off), const_cast<int32_t*>(a.tile_first), const_cast<int32_t*>(a.tile_cand),
                                        d_layout, (int64_t)T, (int)NT, pileup_status, rb.extra ? (int32_t*)(d_rb + rb.extra) : nullptr);
    TC_LAUNCH_CHECK();
    return TC_OK;
}

// select and admit over `tiles` tiles, the mate-overlap pass when a base-quality filter applies, then (d_calls not NULL) the
// hash count; the last two over `grid` candidates
static int ins_enqueue_count(tc_ctx* ctx, const ins_args& a, unsigned tiles, int grid, tc_insert_call_t* d_calls, cudaStream_t s) {
    if (tiles) {
        ins_select_kernel<<<tiles, INS_TILE, 0, s>>>(a);
        TC_LAUNCH_CHECK();
        ins_admit_kernel<<<tiles, INS_TILE, 0, s>>>(a);
        TC_LAUNCH_CHECK();
    }
    if (a.min_bq > 0) {
        const size_t smem = (size_t)PAIR_TBL * 10;
        if (!(ctx->ins_attr_set & 2)) {
            TC_CUDA(cudaFuncSetAttribute(ins_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ctx->ins_attr_set |= 2;
        }
        ins_pair_kernel<<<grid, 1024, smem, s>>>(a);
        TC_LAUNCH_CHECK();
    }
    if (d_calls) {
        const size_t smem = (size_t)INS_TBL * 16;
        if (!(ctx->ins_attr_set & 1)) {
            TC_CUDA(cudaFuncSetAttribute(ins_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ctx->ins_attr_set |= 1;
        }
        ins_count_kernel<<<grid, 1024, smem, s>>>(a, d_calls);
        TC_LAUNCH_CHECK();
    }
    return TC_OK;
}

static int ins_check_status(tc_ctx* ctx, const tc_status& st) {
    if (st.err == TC_ERR_UNSORTED) return tc_fail(ctx, TC_ERR_UNSORTED, "Unsorted input. Pileup aborts");
    if (st.err) return tc_fail(ctx, st.err, "insertion key collision or device-side failure %d", st.err);
    return TC_OK;
}

// Every call's offset into the caller's `bases` (-1 without inserted characters), and the winners' inserted characters
// placed there from `fixed` ([n][INS_BASES_FIXED]); an insertion longer than INS_BASES_FIXED gets its offset only.  *need_out:
// the bytes all insertions take.
static int ins_place_bases(tc_ctx* ctx, tc_insert_call_t* calls, int n, const uint8_t* fixed, uint8_t* bases, int64_t bases_cap,
                           int64_t* need_out = nullptr) {
    int64_t need = 0;
    for (int i = 0; i < n; ++i) {
        if (calls[i].indel > 0) { calls[i].bases_off = need; need += calls[i].indel; } else calls[i].bases_off = -1;
    }
    if (need_out) *need_out = need;
    if (need > 0 && (!bases || need > bases_cap)) return tc_fail(ctx, TC_ERR_CAPACITY, "bases buffer too small: need %lld bytes", (long long)need);
    for (int i = 0; i < n; ++i)
        if (calls[i].indel > 0 && calls[i].indel <= INS_BASES_FIXED)
            memcpy(bases + calls[i].bases_off, fixed + (size_t)i * INS_BASES_FIXED, (size_t)calls[i].indel);
    return TC_OK;
}

// Ranges [r[stride * i], r[stride * i + 1]) of ascending candidates ascend too: merge the overlapping ones and hand every
// stretch to copy(first, length) once.
template <class T, class F>
static int ins_stage_merged(const T* r, int stride, int n, F copy) {
    int i = 0;
    while (i < n) {
        const T b0 = r[stride * i];
        T b1 = r[stride * i + 1];
        int j = i + 1;
        while (j < n && r[stride * j] <= b1) { if (r[stride * j + 1] > b1) b1 = r[stride * j + 1]; ++j; }
        if (b1 != b0) {
            const int rc = copy((size_t)b0, (size_t)(b1 - b0));
            if (rc) return rc;
        }
        i = j;
    }
    return TC_OK;
}

static int ins_copy(tc_ctx* ctx, const void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s, const char* what) {
    const cudaError_t e = cudaMemcpyAsync(const_cast<void*>(dst), src, bytes, kind, s);
    return e == cudaSuccess ? TC_OK : tc_cuda_fail(ctx, e, what);
}

static int ins_sync(tc_ctx* ctx, cudaStream_t s, const char* what) {
    const cudaError_t e = cudaStreamSynchronize(s);
    return e == cudaSuccess ? TC_OK : tc_cuda_fail(ctx, e, what);
}

template <class T>
static std::unique_ptr<T[]> host_array(size_t n) { return std::unique_ptr<T[]>(new (std::nothrow) T[n > 0 ? n : 1]); }

TC_API int tc_extract_inserts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const int32_t* cand_pos, int32_t n_cand,
                              const tc_pileup_params_t* p, tc_insert_call_t* calls, uint8_t* bases, int64_t bases_cap, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!reads || !p || (n_cand > 0 && (!cand_pos || !calls)) || n_cand < 0 || ref_len <= 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n_cand == 0) return TC_OK;
    if (tc_is_device_ptr(cand_pos) || tc_is_device_ptr(calls) || (bases && tc_is_device_ptr(bases)))
        return tc_fail(ctx, TC_ERR_ARG, "tc_extract_inserts takes host pointers for cand_pos / calls / bases");
    for (int i = 0; i < n_cand; ++i)
        if (cand_pos[i] < 1 || cand_pos[i] > ref_len) return tc_fail(ctx, TC_ERR_ARG, "candidate position %d outside 1..%d", cand_pos[i], ref_len);
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    auto upload = [&](const void* d, const void* h, size_t bytes, const char* what) {
        const int rc = ins_copy(ctx, d, h, bytes, cudaMemcpyHostToDevice, s, what);
        if (rc == TC_OK) ctx->h2d_bytes += (int64_t)bytes;
        return rc;
    };
    // Every pass runs from the start.  A pass runs again when the pair scratch overflowed (sized from its bump), or when the
    // speculative layout did not fit (sized for next time) or a column needs the sorted form: then with the layout built on
    // the host (reserved bit 0).
    tc_pileup_params_t q = *p;
    for (;;) {
        ins_args a;
        memset(&a, 0, sizeof(a));
        // Host-resident SEQ / QUAL / CIGAR are staged range by range once the candidate ranges are known: this pass
        // reads them only for the reads over the candidate columns, and QUAL alone is 8x the packed bases.  (Without a
        // span bound the CIGARs of all reads are needed first, so they are staged in full.)
        // the caller's span bound is only trusted when tc_pileup_counts has verified it for these very arrays; a bound that is too
        // small would silently narrow the range of reads fetched for a column
        const bool bounded = reads->max_ref_span > 0 && ctx->span_ok_bound == reads->max_ref_span && ctx->span_ok_cigar == reads->cigar &&
                             ctx->span_ok_off == reads->cigar_off && ctx->span_ok_n == reads->n_reads && ctx->span_ok_ops == reads->n_cigar_ops;
        const int stage = NEED_QUAL | NEED_MATE | DEFER_SEQ | DEFER_QUAL | DEFER_MATE | (bounded ? DEFER_CIGAR : 0);
        const bool host_seq = reads->seq4 && !tc_is_device_ptr(reads->seq4);
        const bool host_qual = reads->qual && !tc_is_device_ptr(reads->qual);
        const bool host_cig = bounded && reads->cigar && !tc_is_device_ptr(reads->cigar);
        const bool host_mate = reads->qname_hash && reads->mpos && reads->isize && !tc_is_device_ptr(reads->qname_hash);
        int rc = tc_resolve_reads(ctx, reads, &a.r, stage, s);
        if (rc) return rc;
        const int64_t n = a.r.n;
        for (int i = 0; i < n_cand; ++i) { calls[i].pos = cand_pos[i]; calls[i].n_entries = 0; calls[i].mode_count = 0; calls[i].first_read = -1; calls[i].head = 0; calls[i].indel = 0; calls[i].bases_off = -1; }
        if (n == 0) return TC_OK;
        const ins_block rb = ins_block_of(n_cand, false);
        uint8_t* d_rb = (uint8_t*)tc_dev_buf(ctx, SLOT_INS_E, rb.bytes + 16);
        int32_t* d_cand = (int32_t*)tc_dev_buf(ctx, SLOT_INS_A, 4 * (size_t)n_cand);
        int32_t* d_range = (int32_t*)tc_dev_buf(ctx, SLOT_INS_B, 24 * (size_t)n_cand);       // [n_cand][2] ranges, then [n_cand][4] offsets
        if (!d_rb || !d_cand || !d_range) return TC_ERR_NOMEM;
        a.status = (tc_status*)d_rb;
        TC_CUDA(cudaMemsetAsync(d_rb, 0, rb.calls, s));
        TC_CUDA(cudaMemcpyAsync(d_cand, cand_pos, 4 * (size_t)n_cand, cudaMemcpyHostToDevice, s));
        ctx->h2d_bytes += 4 * (int64_t)n_cand;
        a.span_hint = bounded ? reads->max_ref_span : 0;
        if (a.span_hint == 0) {
            max_span_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a.r, a.status);
            TC_LAUNCH_CHECK();
        }
        a.cand = d_cand; a.n_cand = n_cand; a.range = d_range; a.range_off = (uint32_t*)(d_range + 2 * (size_t)n_cand);
        cand_range_kernel<<<(n_cand + 3) / 4, 128, 0, s>>>(a);
        TC_LAUNCH_CHECK();
        // Layout of the entry slots.  With everything resident on the device and the hash count, the layout is built
        // on the device into buffers sized from the last calls (no read-back of the ranges, one synchronisation per
        // call); otherwise — host arrays to stage range by range, the sorted form, or a layout that did not fit — on
        // the host from the ranges.
        const bool spec = !(host_seq || host_qual || host_cig || host_mate) && q.kernel != 2 && !(q.reserved & 1);
        if (ctx->ins_slot_cap <= 0) ctx->ins_slot_cap = 1 << 16;     // grows to twice the largest layout seen
        std::unique_ptr<int64_t[]> h_off;
        std::unique_ptr<int32_t[]> h_tfirst, h_tcand;
        int64_t total = ctx->ins_slot_cap;
        int n_tiles = (int)(total / INS_TILE) + n_cand + 1;
        if (!spec) {
            auto h_range = host_array<int32_t>(6 * (size_t)n_cand);
            h_off = host_array<int64_t>((size_t)n_cand + 1);
            h_tfirst = host_array<int32_t>((size_t)n_cand + 1);
            if (!h_range || !h_off || !h_tfirst) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
            if ((rc = ins_copy(ctx, h_range.get(), d_range, 24 * (size_t)n_cand, cudaMemcpyDeviceToHost, s, "range readback")) ||
                (rc = ins_sync(ctx, s, "range readback")))
                return rc;
            ctx->d2h_bytes += 24 * (int64_t)n_cand;
            // QNAME hash, PNEXT, TLEN of the reads over the candidate columns (read index ranges); SEQ + QUAL word ranges; CIGAR op ranges
            if (host_mate)
                rc = ins_stage_merged(h_range.get(), 2, n_cand, [&](size_t b0, size_t len) {
                    int e = upload(a.r.qname_hash + b0, reads->qname_hash + b0, 8 * len, "QNAME hash range upload");
                    if (!e) e = upload(a.r.mpos + b0, reads->mpos + b0, 4 * len, "PNEXT range upload");
                    if (!e) e = upload(a.r.isize + b0, reads->isize + b0, 4 * len, "TLEN range upload");
                    return e;
                });
            const uint32_t* ho = (const uint32_t*)(h_range.get() + 2 * (size_t)n_cand);
            if (!rc && (host_seq || host_qual))
                rc = ins_stage_merged(ho, 4, n_cand, [&](size_t b0, size_t len) {
                    int e = host_seq ? upload(a.r.seq4 + b0, reads->seq4 + b0, 4 * len, "SEQ range upload") : TC_OK;
                    if (!e && host_qual) e = upload(a.r.qual + 8 * b0, reads->qual + 8 * b0, 8 * len, "QUAL range upload");
                    return e;
                });
            if (!rc && host_cig)
                rc = ins_stage_merged(ho + 2, 4, n_cand,
                                      [&](size_t b0, size_t len) { return upload(a.r.cigar + b0, reads->cigar + b0, 4 * len, "CIGAR range upload"); });
            if (rc) return rc;
            h_off[0] = 0; h_tfirst[0] = 0;
            for (int i = 0; i < n_cand; ++i) {
                const int64_t len = h_range[2 * i + 1] - h_range[2 * i];
                h_off[i + 1] = h_off[i] + len;
                h_tfirst[i + 1] = h_tfirst[i] + (int32_t)((len + INS_TILE - 1) / INS_TILE);
            }
            total = h_off[n_cand];
            n_tiles = h_tfirst[n_cand];
            if (total >= 0x7fffffffll) return tc_fail(ctx, TC_ERR_CAPACITY, "too many candidate column entries (%lld)", (long long)total);
            h_tcand = host_array<int32_t>((size_t)n_tiles);
            if (!h_tcand) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
            for (int i = 0; i < n_cand; ++i) for (int t = h_tfirst[i]; t < h_tfirst[i + 1]; ++t) h_tcand[t] = i;
        }
        const size_t T = (size_t)(total > 0 ? total : 1), NT = (size_t)(n_tiles > 0 ? n_tiles : 1);
        if ((rc = ins_bind(ctx, a, d_rb, rb, T, NT, n_cand, &q))) return rc;
        tc_insert_call_t* d_calls = (tc_insert_call_t*)(d_rb + rb.calls);
        if (spec) rc = ins_layout_dev(ctx, a, d_rb, rb, T, NT, nullptr, s);
        else if (!(rc = upload(a.seg_off, h_off.get(), 8 * ((size_t)n_cand + 1), "offset upload")) &&
                 !(rc = upload(a.tile_first, h_tfirst.get(), 4 * ((size_t)n_cand + 1), "tile table upload")) && n_tiles)
            rc = upload(a.tile_cand, h_tcand.get(), 4 * (size_t)n_tiles, "tile table upload");
        if (rc) return rc;
        const bool sorted_form = q.kernel == 2;
        if ((rc = ins_enqueue_count(ctx, a, (unsigned)n_tiles, n_cand, sorted_form ? nullptr : d_calls, s))) return rc;
        int32_t h_over = 0;
        unsigned long long h_bump = 0;
        int32_t h_layout[3] = {0, 0, 0};
        const size_t calls_bytes = sizeof(tc_insert_call_t) * (size_t)n_cand, fixed_bytes = (size_t)n_cand * INS_BASES_FIXED;
        auto h_fixed = host_array<uint8_t>(fixed_bytes);
        if (!h_fixed) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
        // the results block comes back in one copy through pinned memory (copies into the caller's pageable buffers
        // would each wait for the stream)
        if (rb.bytes <= TC_HOST_SCRATCH) {
            const uint8_t* pin = (const uint8_t*)ctx->host_scratch;
            if ((rc = ins_copy(ctx, pin, d_rb, rb.bytes, cudaMemcpyDeviceToHost, s, "results readback")) || (rc = ins_sync(ctx, s, "results readback")))
                return rc;
            memcpy(ctx->host_status, pin, sizeof(tc_status));
            memcpy(h_layout, pin + rb.layout, 12); memcpy(&h_over, pin + rb.over, 4); memcpy(&h_bump, pin + rb.bump, 8);
            memcpy(calls, pin + rb.calls, calls_bytes); memcpy(h_fixed.get(), pin + rb.fixed, fixed_bytes);
        } else if ((rc = ins_copy(ctx, &h_over, a.overflow, 4, cudaMemcpyDeviceToHost, s, "overflow readback")) ||
                   (rc = ins_copy(ctx, &h_bump, a.pair_bump, 8, cudaMemcpyDeviceToHost, s, "overflow readback")) ||
                   (spec && (rc = ins_copy(ctx, h_layout, a.layout, 12, cudaMemcpyDeviceToHost, s, "layout readback"))) ||
                   (rc = ins_copy(ctx, calls, d_calls, calls_bytes, cudaMemcpyDeviceToHost, s, "insert calls readback")) ||
                   (rc = ins_copy(ctx, h_fixed.get(), a.bases_fixed, fixed_bytes, cudaMemcpyDeviceToHost, s, "inserted bases readback")) ||
                   (rc = ins_copy(ctx, ctx->host_status, a.status, sizeof(tc_status), cudaMemcpyDeviceToHost, s, "status readback")) ||
                   (rc = ins_sync(ctx, s, "insert calls readback"))) {
            return rc;
        }
        ctx->d2h_bytes += (int64_t)(sizeof(tc_insert_call_t) + INS_BASES_FIXED) * n_cand + (int64_t)sizeof(tc_status) + 4;
        if (sorted_form) h_over &= 2;
        if (h_over & 2) {
            // the scratch for the rewritten quality strings of overlapping mates was too small: size it and run again
            ctx->pair_cap = 2 * (int64_t)h_bump + 4096;
            continue;
        }
        if (spec) {
            if (h_layout[2] || h_over) {
                // the layout did not fit the speculative buffers (size them for next time), or a column needs the sorted
                // form: run again with the layout built on the host
                if (h_layout[2]) ctx->ins_slot_cap = 2 * (int64_t)h_layout[1] + 4096;
                q.reserved |= 1;
                continue;
            }
            total = h_layout[1];
        }
        if (sorted_form || h_over) {
            // radix sort + run-length encoding over the same slots
            uint8_t* slab2 = (uint8_t*)tc_dev_buf(ctx, SLOT_INS_C, T * (8 + 4 + 4) + 64);
            if (!slab2) return TC_ERR_NOMEM;
            uint64_t* d_skey = (uint64_t*)slab2; uint32_t* d_idx = (uint32_t*)(d_skey + T); uint32_t* d_sidx = d_idx + T;
            int64_t* d_off = const_cast<int64_t*>(a.seg_off);
            iota_kernel<<<(unsigned)((T + 255) / 256), 256, 0, s>>>(d_idx, (int64_t)total);
            TC_LAUNCH_CHECK();
            size_t tmp_bytes = 0;
            cudaError_t e = cub::DeviceSegmentedRadixSort::SortPairs(nullptr, tmp_bytes, a.ent_key, d_skey, d_idx, d_sidx, (int64_t)total, n_cand,
                                                                     d_off, d_off + 1, 0, 64, s);
            if (e != cudaSuccess) return tc_cuda_fail(ctx, e, "cub sort sizing");
            void* d_tmp = tc_dev_buf(ctx, SLOT_INS_G, tmp_bytes + 16);
            if (!d_tmp) return TC_ERR_NOMEM;
            e = cub::DeviceSegmentedRadixSort::SortPairs(d_tmp, tmp_bytes, a.ent_key, d_skey, d_idx, d_sidx, (int64_t)total, n_cand, d_off,
                                                         d_off + 1, 0, 64, s);
            if (e != cudaSuccess) return tc_cuda_fail(ctx, e, "cub segmented radix sort");
            ctx->launches++;
            ins_mode_kernel<<<n_cand, 1024, 0, s>>>(a, d_skey, d_sidx, d_calls);
            TC_LAUNCH_CHECK();
            if ((rc = ins_copy(ctx, calls, d_calls, calls_bytes, cudaMemcpyDeviceToHost, s, "insert calls readback")) ||
                (rc = ins_copy(ctx, h_fixed.get(), a.bases_fixed, fixed_bytes, cudaMemcpyDeviceToHost, s, "inserted bases readback")) ||
                (rc = ins_copy(ctx, ctx->host_status, a.status, sizeof(tc_status), cudaMemcpyDeviceToHost, s, "status readback")) ||
                (rc = ins_sync(ctx, s, "insert calls readback")))
                return rc;
        }
        tc_status st; memcpy(&st, ctx->host_status, sizeof(st));
        if ((rc = ins_check_status(ctx, st))) return rc;
        // lay the winners' inserted characters out in the caller's buffer: up to INS_BASES_FIXED characters came back
        // with the call; longer insertions (rare) are fetched by one more small kernel
        auto h_entry = host_array<int64_t>((size_t)n_cand);
        if (!h_entry) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
        int64_t n_long = 0;
        for (int i = 0; i < n_cand; ++i) { h_entry[i] = calls[i].bases_off; n_long += calls[i].indel > INS_BASES_FIXED; }
        int64_t need = 0;
        if ((rc = ins_place_bases(ctx, calls, n_cand, h_fixed.get(), bases, bases_cap, &need)) || n_long == 0) return rc;
        uint8_t* d_bases = (uint8_t*)tc_dev_buf(ctx, SLOT_TMP_A, (size_t)need);
        int64_t* d_entry = (int64_t*)tc_dev_buf(ctx, SLOT_TMP_B, 8 * (size_t)n_cand);
        auto h_long = host_array<uint8_t>((size_t)need);
        if (!d_bases || !d_entry || !h_long) return TC_ERR_NOMEM;
        const char* what = "inserted bases readback";
        if ((rc = ins_copy(ctx, d_entry, h_entry.get(), 8 * (size_t)n_cand, cudaMemcpyHostToDevice, s, what)) ||
            (rc = ins_copy(ctx, d_calls, calls, calls_bytes, cudaMemcpyHostToDevice, s, what)))
            return rc;
        ins_bases_kernel<<<n_cand, 128, 0, s>>>(a, d_calls, d_entry, d_bases);
        TC_LAUNCH_CHECK();
        if (!(rc = ins_copy(ctx, h_long.get(), d_bases, (size_t)need, cudaMemcpyDeviceToHost, s, what))) rc = ins_sync(ctx, s, what);
        ctx->d2h_bytes += need;
        if (rc) return rc;
        for (int i = 0; i < n_cand; ++i)
            if (calls[i].indel > INS_BASES_FIXED) memcpy(bases + calls[i].bases_off, h_long.get() + calls[i].bases_off, (size_t)calls[i].indel);
        return TC_OK;
    }
}


// ---------------------------------------------------------------- candidates that never leave the device
// tc_pileup_call_inserts (sample.cu): the candidate list is what the call kernel flagged; its length is only known on
// the device.  Everything is enqueued for up to `cap` candidates into buffers sized from earlier calls, and ONE block
// of results travels back: the insertion calls, the candidate list, and the pileup's status.  Whatever does not fit this
// speculative layout (more candidates than cap, more entry slots than the buffers hold, a column with thousands of
// distinct strings, an insertion longer than INS_BASES_FIXED characters) is reported as TC_ERR_CAPACITY in `fit` and the
// caller runs tc_extract_inserts with the list it got back.
int tc_inserts_enqueue_dev(tc_ctx* ctx, const tc_reads_t* reads, const int32_t* d_cand, const int32_t* d_ncand, int cap,
                           const tc_pileup_params_t* p, const tc_status* d_pileup_status, void* host_block, cudaStream_t s, tc_ins_pending* pend) {
    ins_args a;
    memset(&a, 0, sizeof(a));
    memset(pend, 0, sizeof(*pend));
    int rc = tc_resolve_reads(ctx, reads, &a.r, NEED_QUAL | NEED_MATE, s);       // every array is a device pointer already: nothing is copied
    if (rc) return rc;
    const int64_t n = a.r.n;
    const ins_block rb = ins_block_of(cap, true);
    if (rb.bytes > TC_HOST_SCRATCH) return tc_fail(ctx, TC_ERR_ARG, "candidate capacity %d too large for the pinned results block", cap);
    uint8_t* d_rb = (uint8_t*)tc_dev_buf(ctx, SLOT_INS_E, rb.bytes + 16);
    int32_t* d_range = (int32_t*)tc_dev_buf(ctx, SLOT_INS_B, 24 * (size_t)cap);
    if (!d_rb || !d_range) return TC_ERR_NOMEM;
    TC_CUDA(cudaMemsetAsync(d_rb, 0, rb.calls, s));
    a.span_hint = reads->max_ref_span > 0 ? reads->max_ref_span : 0;
    a.status = (tc_status*)d_rb;
    if (a.span_hint == 0 && n > 0) {
        max_span_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a.r, a.status);
        TC_LAUNCH_CHECK();
    }
    a.cand = d_cand; a.n_cand = cap; a.n_cand_dev = d_ncand; a.range = d_range; a.range_off = (uint32_t*)(d_range + 2 * (size_t)cap);
    cand_range_kernel<<<(cap + 3) / 4, 128, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    if (ctx->ins_slot_cap <= 0) ctx->ins_slot_cap = 1 << 16;
    const size_t T = (size_t)ctx->ins_slot_cap, NT = T / INS_TILE + (size_t)cap + 1;
    if ((rc = ins_bind(ctx, a, d_rb, rb, T, NT, cap, p)) || (rc = ins_layout_dev(ctx, a, d_rb, rb, T, NT, d_pileup_status, s))) return rc;
    if (n > 0 && (rc = ins_enqueue_count(ctx, a, (unsigned)NT, cap, (tc_insert_call_t*)(d_rb + rb.calls), s))) return rc;
    TC_CUDA(cudaMemcpyAsync(host_block, d_rb, rb.bytes, cudaMemcpyDeviceToHost, s));
    ctx->d2h_bytes += (int64_t)rb.bytes;
    pend->rb = rb; pend->cap = cap; pend->n_reads = n;
    return TC_OK;
}

// After the sample's event has completed: unpack its results block.  *fit = 0 when the speculative layout
// did not hold everything (cands / n_cand are valid all the same whenever n_cand <= cap).
int tc_inserts_finish_dev(tc_ctx* ctx, const tc_ins_pending* pend, const void* host_block, tc_status* pileup_status, int32_t* cands, int32_t* n_cand,
                          tc_insert_call_t* calls, uint8_t* bases, int64_t bases_cap, int* fit) {
    const uint8_t* pin = (const uint8_t*)host_block;
    const ins_block& rb = pend->rb;
    const int32_t* extra = (const int32_t*)(pin + rb.extra);
    tc_status st; memcpy(&st, pin, sizeof(st));
    memcpy(pileup_status, extra + TC_RB_EXTRA_STATUS, sizeof(tc_status));
    int32_t layout[3]; memcpy(layout, pin + rb.layout, 12);
    int32_t over; memcpy(&over, pin + rb.over, 4);
    const int n = extra[TC_RB_EXTRA_NCAND];
    *n_cand = n;
    *fit = 1;
    if (n > pend->cap) { *fit = 0; return TC_OK; }
    memcpy(cands, extra + TC_RB_EXTRA_CAND, 4 * (size_t)n);
    if (layout[2]) { ctx->ins_slot_cap = 2 * (int64_t)layout[1] + 4096; *fit = 0; return TC_OK; }
    if (over & 2) { unsigned long long bump; memcpy(&bump, pin + rb.bump, 8); ctx->pair_cap = 2 * (int64_t)bump + 4096; }
    if (over) { *fit = 0; return TC_OK; }
    if (const int rc = ins_check_status(ctx, st)) return rc;
    memcpy(calls, pin + rb.calls, sizeof(tc_insert_call_t) * (size_t)n);
    for (int i = 0; i < n; ++i) {
        if (pend->n_reads == 0) { calls[i].pos = cands[i]; calls[i].n_entries = 0; calls[i].mode_count = 0; calls[i].first_read = -1; calls[i].head = 0; calls[i].indel = 0; }
        if (calls[i].indel > INS_BASES_FIXED) { *fit = 0; return TC_OK; }       // rare: the separate call fetches long insertions
    }
    return ins_place_bases(ctx, calls, n, pin + rb.fixed, bases, bases_cap);
}
