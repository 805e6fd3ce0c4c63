// bgzf.cu — the BAM file as it lies on disk -> its uncompressed payload and the offsets of its records, on the device.
//
// The step in front of bamparse.cu, and the last piece of pysam's reader (TrueConsense/indexing.py:6-19 `Readbam`, :96)
// that ran on the host: htslib's bgzf.c inflates every <= 64 KiB BGZF member with zlib and checks its CRC-32, then
// bam_read1 hops from record to record.  Sixteen host cores inflate ~2.8 GB/s of payload (bench.py host_decode); a deep
// sample is a gigabyte and more.  Here the host only walks the member headers (csrc/host/bamio.c tc_bgzf_map: one header
// per member) and ships the file's bytes as they are — fewer than the payload — and the device does the rest:
//
//   bgzf_inflate_kernel   one member per warp (Huffman decoding is a serial walk of a bit stream; the members are independent):
//                         inflate_core.cuh's decoder, first-level tables in shared memory.  All 32 lanes run the same chain on
//                         the same values — an instruction costs one issue slot however many lanes are active — and share what is
//                         data-parallel: match copies (32 bytes per step) and table fills.  Thousands of members in flight; the
//                         kernel is bound by issue slots, and with one chain per warp resident warps are what fills them.
//   bgzf_crc_kernel       one WARP per member: every lane the CRC-32 of 1/32 of the member's payload, the 32 pieces
//                         combined by multiplication in GF(2)[x] / p(x) (zlib's crc32_combine), compared with the member's
//                         stored CRC.  htslib fails on a CRC mismatch: so does this.
//   bam_chain_*           the hop over the records without a sequential pass: the payload is cut into 64 KiB chunks; every
//                         chunk looks for the first offset that reads like a record (sizes consistent with block_size,
//                         refID / pos within the header's references, a printable NUL-terminated name, CIGAR op codes
//                         <= 8, and the record behind it plausible too) and follows the records from there to the chunk's
//                         end.  That guess is then PROVEN: the chunk holding the header's end starts at the true first
//                         record, and a chunk is on the chain exactly if the chain of the chunk before it ends on its own
//                         start — by induction every offset emitted is a true record start.  Chunks the chain jumps over
//                         (a record longer than a chunk) and guesses that do not link up are resolved by one thread
//                         walking the chunk table; a chain that cannot be closed is an error (the caller then takes the
//                         host reader, which names the broken record).  Records are validated as csrc/host/bamio.c does.
//
// Result: payload + record offsets resident in the context's buffers, exactly what tc_bam_payload hands to
// tc_bam_records_to_reads — which takes device pointers as they are.
#include <cub/device/device_scan.cuh>

#include "bamrec.cuh"
#include "inflate_core.cuh"
#include "tc_common.cuh"

namespace {

using namespace tcinf;

constexpr unsigned long long NO_ERROR = ~0ull;

// first failing member: (member index << 8 | code), smallest wins
__device__ __forceinline__ void report(unsigned long long* status, long long member, int code) {
    atomicMin(status, ((unsigned long long)member << 8) | (unsigned long long)code);
}

// One member per WARP.  Thirty-two members per warp (a lane each) was measured first: the lanes of a warp run different code
// paths at every symbol (literal, match, refill, table build) and do not reconverge — 32 x serialised, 269 ms for 2348 members
// against 10.3 ms with one member per warp (then one lane; now all lanes in step on the same member: 13.9 -> 13.3 ms with the
// upload, 42.4 -> 40.2 ms for 11 724 members).
constexpr int INFLATE_WARPS = 8;


// MIN_CTAS: 2 = up to 128 registers (16 warps per SM, the fastest single member); 4 = capped at 64 (32 warps
// per SM: a file with more members than the SMs hold at 16 warps is bound by issue slots, and every warp is one lane: 51.7 -> 42.0 ms
// for 11 724 members, 14.0 -> 14.8 ms for 2346)
template <int MIN_CTAS>
__global__ void __launch_bounds__(32 * INFLATE_WARPS, MIN_CTAS) bgzf_inflate_kernel(const uint8_t* __restrict__ file, const tc_bgzf_block_t* __restrict__ blk,
                                                                          long long m0, long long n_blk, uint8_t* __restrict__ payload,
                                                                          unsigned long long* status) {
    __shared__ __align__(16) uint16_t tables[INFLATE_WARPS][LUT_SIZE + DLUT_SIZE];
    const int w = threadIdx.x >> 5;
    const long long m = m0 + (long long)blockIdx.x * INFLATE_WARPS + w;
    if (m >= m0 + n_blk) return;
    const int lane = threadIdx.x & 31;
    huff hl, hd;
    uint8_t lens[LENS_SIZE];
    const tc_bgzf_block_t b = blk[m];
    // (the tables' shared address pinned in a register: re-deriving it from %tid at every look-up was 3 % of the instructions)
    uint32_t lut_s = (uint32_t)__cvta_generic_to_shared(tables[w]);
    asm volatile("" : "+r"(lut_s));
    uint16_t* lut = (uint16_t*)__cvta_shared_to_generic((size_t)lut_s);
    const int rc = inflate_block<32>(file + b.coff, b.csize, payload + b.uoff, b.usize, lut, lut + LUT_SIZE, hl, hd, lens, lane);
    if (rc && lane == 0) report(status, m, rc);
}

constexpr int CRC_ERR = 32;

__global__ void __launch_bounds__(256) bgzf_crc_kernel(const uint8_t* __restrict__ file, const tc_bgzf_block_t* __restrict__ blk, long long m0,
                                                       long long n_blk, const uint8_t* __restrict__ payload, unsigned long long* status) {
    __shared__ uint32_t tab[256];
    tab[threadIdx.x] = crc_table_entry(threadIdx.x);
    __syncthreads();
    const long long m = m0 + (((long long)blockIdx.x * 256 + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (m >= m0 + n_blk) return;
    const tc_bgzf_block_t b = blk[m];
    const uint32_t per = ((uint32_t)b.usize + 31u) / 32u;
    const uint32_t s0 = min(per * lane, (uint32_t)b.usize), s1 = min(s0 + per, (uint32_t)b.usize);
    const uint8_t* p = payload + b.uoff;
    uint32_t c = 0xffffffffu;
    for (uint32_t i = s0; i < s1; ++i) c = tab[(c ^ p[i]) & 0xffu] ^ (c >> 8);
    c ^= 0xffffffffu;
    uint32_t len = s1 - s0;
    // every lane's piece has the same length `per` except the tail's: one power of x per level serves all pairs whose
    // right-hand side is whole; the others compute their own
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const uint32_t oc = __shfl_down_sync(0xffffffffu, c, s), ol = __shfl_down_sync(0xffffffffu, len, s);
        if ((lane & (2 * s - 1)) == 0) { c = crc_combine(c, oc, ol); len += ol; }
    }
    if (lane == 0 && c != ld32(file + b.coff + b.csize)) report(status, m, CRC_ERR);
}

// ---------------------------------------------------------------- the records
constexpr int CHUNK = 65536;

struct chain_args {
    const uint8_t* u; long long n;              // payload
    long long first;                            // offset of the first record's block_size (behind the header)
    int n_ref; const int32_t* ref_len;
    long long n_chunks;
    long long* S; long long* E;                 // per chunk: chosen start (-1: none), where its chain leaves the chunk (n: the end)
    uint8_t* on;                                // per chunk: on the chain (written by the resolver when the chunks do not simply link up)
    long long* ctl;                             // [0] first chunk that does not link to its successor, [1] mode (0 range, 1 `on`), [2] error
    uint32_t* counts;                           // per chunk: placed records
    unsigned long long* totals;                 // [0] records, [1] placed, [2] SEQ words, [3] CIGAR ops, [4] first invalid record's offset + 1
    long long* rec_off; const uint32_t* offs;
};

// what a record's first 36 bytes and the sizes they give must satisfy (the host reader's checks, bamio.c scan_payload)
__device__ __forceinline__ bool record_valid(const uint8_t* u, long long n, long long q, uint32_t* bs_out) {
    if (q + 4 > n) return false;
    const uint32_t bs = ld32(u + q);
    *bs_out = bs;
    if (bs < 32u || bs > 0x7fffffffu || q + 4 + (long long)bs > n) return false;
    const uint8_t* r = u + q - BAM_BLOCK_SIZE;
    const uint32_t l_name = r[BAM_L_READ_NAME], n_cig = ld16(r + BAM_N_CIGAR_OP), l_seq = ld32(r + BAM_L_SEQ);
    const long long need = (long long)BAM_READ_NAME + l_name + 4ll * n_cig + ((long long)l_seq + 1) / 2 + (long long)l_seq;
    if (l_seq > 0x7fffffffu || need > (long long)bs || l_name < 1u) return false;
    if (r[BAM_READ_NAME + l_name - 1] != 0) return false;
    const int32_t refid = (int32_t)ld32(r + BAM_REF_ID);
    if (refid >= 0 && n_cig == 2) {             // the CG-tag placeholder of a CIGAR with more than 65535 operations: not expanded
        const uint8_t* cg = bam_cigar(r);
        const uint32_t c0 = ld32(cg), c1 = ld32(cg + 4);
        if ((c0 & 15u) == 4u && (c0 >> 4) == l_seq && (c1 & 15u) == 3u && l_seq > 0) return false;
    }
    return true;
}

// "reads like a record": the guess a chunk starts its chain from (proven or discarded afterwards)
__device__ bool record_plausible(const chain_args& a, long long q) {
    if (q + 36 > a.n) return false;
    uint32_t bs;
    if (!record_valid(a.u, a.n, q, &bs)) return false;
    const uint8_t* r = a.u + q - BAM_BLOCK_SIZE;
    const int32_t refid = (int32_t)ld32(r + BAM_REF_ID), pos = (int32_t)ld32(r + BAM_POS);
    const int32_t mrefid = (int32_t)ld32(r + BAM_NEXT_REF_ID), mpos = (int32_t)ld32(r + BAM_NEXT_POS);
    if (refid < -1 || refid >= a.n_ref || mrefid < -1 || mrefid >= a.n_ref || pos < -1 || mpos < -1) return false;
    if (refid >= 0 && pos > a.ref_len[refid]) return false;
    const uint32_t l_name = r[BAM_L_READ_NAME], n_cig = ld16(r + BAM_N_CIGAR_OP);
    for (uint32_t k = 0; k + 1 < l_name; ++k)
        if (r[BAM_READ_NAME + k] < 33 || r[BAM_READ_NAME + k] > 126) return false;
    for (uint32_t k = 0; k < n_cig; ++k)
        if ((r[BAM_READ_NAME + l_name + 4 * k] & 15u) > 8u) return false;
    return true;
}

// follow the records from q to the first one that starts at or behind `hi` (sizes only: validation is the counting pass's).
// Returns that offset; a.n when the records end with the payload (fewer than 4 bytes left); a.n + 1 when they do not form
// a chain (a block_size below 32, or a record running over the payload's end) — a value that links to nothing.
__device__ long long chain_exit(const chain_args& a, long long q, long long hi) {
    while (q < hi && q + 4 <= a.n) {
        const uint32_t bs = ld32(a.u + q);
        if (bs < 32u || bs > 0x7fffffffu) return a.n + 1;
        q += 4 + (long long)bs;
    }
    if (q + 4 <= a.n) return q;
    return q > a.n ? a.n + 1 : a.n;
}

__global__ void __launch_bounds__(128) bam_chain_start_kernel(chain_args a) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chunks) return;
    const long long lo = c * CHUNK, hi = min(lo + CHUNK, a.n);
    const long long anchor = a.first / CHUNK;
    long long s = -1;
    if (c == anchor) s = a.first < a.n ? a.first : -1;
    else if (c > anchor) {
        for (long long q = lo; q < hi; ++q) {
            if (!record_plausible(a, q)) continue;
            const long long nx = q + 4 + (long long)ld32(a.u + q);
            if (nx + 4 > a.n || record_plausible(a, nx)) { s = q; break; }
        }
    }
    a.S[c] = s;
    long long e = a.n;
    if (s >= 0) e = chain_exit(a, s, hi);
    a.E[c] = e;
}

// link[c]: chunk c's chain ends exactly on chunk c + 1's start.  The first chunk from the anchor on that does not link:
__global__ void __launch_bounds__(128) bam_chain_link_kernel(chain_args a) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long anchor = a.first / CHUNK;
    if (c >= a.n_chunks || c < anchor) return;
    const bool link = a.S[c] >= 0 && c + 1 < a.n_chunks && a.E[c] == a.S[c + 1];
    if (!link) atomicMin((unsigned long long*)&a.ctl[0], (unsigned long long)c);
}

// one thread: either the chunks from the anchor to T link up and T's chain runs to the payload's end (the common case:
// nothing to do), or the chunk table is walked: from a chunk on the chain to the chunk its chain ends in, whose start
// must be that very offset
__global__ void bam_chain_resolve_kernel(chain_args a) {
    const long long anchor = a.first / CHUNK;
    if (a.first >= a.n) { a.ctl[1] = 0; a.ctl[0] = anchor - 1; return; }      // no record at all
    const long long T = a.ctl[0];
    if (T >= 0 && T < a.n_chunks && a.S[T] >= 0 && a.E[T] == a.n) { a.ctl[1] = 0; return; }
    a.ctl[1] = 1;
    long long c = anchor;
    for (;;) {
        if (a.S[c] < 0) { a.ctl[2] = 1; return; }
        a.on[c] = 1;
        const long long e = a.E[c];
        if (e == a.n) return;
        if (e > a.n) { a.ctl[2] = 2; return; }
        const long long c2 = e / CHUNK;
        if (c2 <= c || c2 >= a.n_chunks || a.S[c2] != e) {
            // the guess of chunk c2 was not the record the chain arrives at: the chain is the truth — restart c2 from it
            if (c2 <= c || c2 >= a.n_chunks) { a.ctl[2] = 3; return; }
            a.S[c2] = e;
            a.E[c2] = chain_exit(a, e, min((c2 + 1) * (long long)CHUNK, a.n));
        }
        c = c2;
    }
}

__device__ __forceinline__ bool chunk_on_chain(const chain_args& a, long long c) {
    const long long anchor = a.first / CHUNK;
    if (a.ctl[1]) return a.on[c] != 0;
    return c >= anchor && c <= a.ctl[0];
}

// validate and count (WRITE = false), then emit the offsets of the placed records' refID fields (WRITE = true)
template <bool WRITE>
__global__ void __launch_bounds__(128) bam_chain_walk_kernel(chain_args a) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chunks) return;
    uint32_t kept = 0, total = 0;
    unsigned long long words = 0, ops = 0;
    if (chunk_on_chain(a, c)) {
        const long long hi = min((c + 1) * (long long)CHUNK, a.n);
        long long q = a.S[c];
        long long* out = WRITE ? a.rec_off + a.offs[c] : nullptr;
        while (q < hi && q + 4 <= a.n) {
            uint32_t bs;
            if (!WRITE && !record_valid(a.u, a.n, q, &bs)) { atomicMin(&a.totals[4], (unsigned long long)q + 1ull); break; }
            if (WRITE) bs = ld32(a.u + q);
            const uint8_t* r = a.u + q - BAM_BLOCK_SIZE;
            if ((int32_t)ld32(r + BAM_REF_ID) >= 0) {
                if (WRITE) out[kept] = q - BAM_BLOCK_SIZE;
                else { words += (ld32(r + BAM_L_SEQ) + 7u) / 8u; ops += ld16(r + BAM_N_CIGAR_OP); }
                ++kept;
            }
            ++total;
            q += 4 + (long long)bs;
        }
    }
    if (!WRITE) {
        a.counts[c] = kept;
        if (total) { atomicAdd(&a.totals[0], (unsigned long long)total); atomicAdd(&a.totals[1], (unsigned long long)kept);
                     atomicAdd(&a.totals[2], words); atomicAdd(&a.totals[3], ops); }
    }
}

}  // namespace

TC_API int tc_bgzf_inflate(tc_ctx_t* ctx, const uint8_t* file, int64_t file_bytes, const tc_bgzf_block_t* blocks, int64_t n_blocks,
                           int64_t payload_bytes, const uint8_t** payload_dev, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!file || file_bytes <= 0 || !blocks || n_blocks <= 0 || payload_bytes < 0 || !payload_dev) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    *payload_dev = nullptr;
    // the index came from the file's own headers: every member inside the file, the payload offsets a running sum
    int64_t uoff = 0;
    for (int64_t i = 0; i < n_blocks; ++i) {
        const tc_bgzf_block_t& b = blocks[i];
        if (b.coff < 0 || b.csize < 0 || b.usize < 0 || b.usize > 65536 || b.coff + b.csize + 8 > file_bytes || b.uoff != uoff)
            return tc_fail(ctx, TC_ERR_ARG, "BGZF member %lld of the index lies outside the file or the payload", (long long)i);
        uoff += b.usize;
    }
    if (uoff != payload_bytes) return tc_fail(ctx, TC_ERR_ARG, "the members inflate to %lld bytes, not %lld", (long long)uoff, (long long)payload_bytes);
    int rc;
    const bool trace = getenv("TC_TRACE") != nullptr;       // stage times to stderr (diagnostics)
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    if (trace) { for (auto& e : ev) cudaEventCreate(&e); cudaEventRecord(ev[0], s); }
    // (the bit reader fetches aligned 16-byte vectors: up to 15 bytes in front of a stream — the member's own 18-byte
    // header — and behind it — its CRC, ISIZE and the next header; the buffer is padded behind the file's end)
    const tc_bgzf_block_t* d_blk = (const tc_bgzf_block_t*)tc_stage_in(ctx, SLOT_BGZF_BLOCKS, blocks, sizeof(tc_bgzf_block_t) * (size_t)n_blocks, s, &rc);
    if (rc) return rc;
    uint8_t* d_payload = (uint8_t*)tc_dev_buf(ctx, SLOT_BAM_PAYLOAD, (size_t)payload_bytes + 64);
    unsigned long long* d_status = (unsigned long long*)tc_dev_buf(ctx, SLOT_STATUS, 64);
    if (!d_payload || !d_status) return TC_ERR_NOMEM;
    TC_CUDA(cudaMemsetAsync(d_status, 0xff, 8, s));
    const bool file_dev = tc_is_device_ptr(file);
    uint8_t* d_file = file_dev ? (uint8_t*)file : (uint8_t*)tc_dev_buf(ctx, SLOT_BGZF_FILE, (size_t)file_bytes + 64);
    if (!d_file) return TC_ERR_NOMEM;
    if (trace) cudaEventRecord(ev[1], s);
    // A large file goes in four groups of members: the host copies group g + 1 into the staging ring while the device inflates
    // group g, each group's kernels on a side stream of its own behind its upload (a member's decode is a serial chain of ~9 ms
    // whatever the group's size: kernels queued on one stream would wait for one another; four streams share the SMs).  A small
    // file is one group: its time is the upload plus that one chain, and nothing overlaps with a chain.
    constexpr int N_SIDE = 4;
    if (!ctx->aux[0]) {
        for (int i = 0; i < N_SIDE; ++i) TC_CUDA(cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking));
        for (int i = 0; i < N_SIDE + 1; ++i) TC_CUDA(cudaEventCreateWithFlags(&ctx->aux_ev[i], cudaEventDisableTiming));
    }
    const int n_groups = (file_bytes >= (128ll << 20) && n_blocks >= 4 * N_SIDE) ? N_SIDE : 1;
    const int64_t group_bytes = (file_bytes + n_groups - 1) / n_groups;
    int64_t sent = 0;               // file bytes [0, sent) are on their way
    int g = 0;
    for (int64_t g0 = 0; g0 < n_blocks; ++g) {
        int64_t g1 = g0 + 1;
        if (g + 1 >= n_groups) g1 = n_blocks;
        else while (g1 < n_blocks && blocks[g1].coff + blocks[g1].csize + 8 - sent <= group_bytes) ++g1;
        // (32 bytes more than the group's last member: the vectors a bit reader fetches behind a stream's end stay inside what was sent)
        int64_t end = g1 == n_blocks ? file_bytes : blocks[g1 - 1].coff + blocks[g1 - 1].csize + 8 + 32;
        if (end > file_bytes) end = file_bytes;
        if (!file_dev && end > sent) {
            rc = tc_h2d(ctx, d_file + sent, file + sent, (size_t)(end - sent), s);
            if (rc) return rc;
            sent = end;
        }
        cudaStream_t side = ctx->aux[g % N_SIDE];
        TC_CUDA(cudaEventRecord(ctx->aux_ev[N_SIDE], s));           // everything up to this group's bytes (and the status block's reset)
        TC_CUDA(cudaStreamWaitEvent(side, ctx->aux_ev[N_SIDE], 0));
        const int64_t n = g1 - g0;
        const unsigned grid = (unsigned)((n + INFLATE_WARPS - 1) / INFLATE_WARPS);
        if (n_blocks > (int64_t)ctx->sm_count * 16) bgzf_inflate_kernel<4><<<grid, 32 * INFLATE_WARPS, 0, side>>>(d_file, d_blk, g0, n, d_payload, d_status);
        else bgzf_inflate_kernel<2><<<grid, 32 * INFLATE_WARPS, 0, side>>>(d_file, d_blk, g0, n, d_payload, d_status);
        TC_LAUNCH_CHECK();
        bgzf_crc_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, side>>>(d_file, d_blk, g0, n, d_payload, d_status);
        TC_LAUNCH_CHECK();
        g0 = g1;
    }
    for (int i = 0; i < N_SIDE && i < g; ++i) {                     // the caller's stream continues behind the side streams
        TC_CUDA(cudaEventRecord(ctx->aux_ev[i], ctx->aux[i]));
        TC_CUDA(cudaStreamWaitEvent(s, ctx->aux_ev[i], 0));
    }
    if (trace) cudaEventRecord(ev[2], s);
    unsigned long long* h = (unsigned long long*)ctx->host_status;
    TC_D2H(h, d_status, 8, s);
    if (trace) cudaEventRecord(ev[3], s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (trace) {
        float t01 = 0, t12 = 0, t23 = 0;
        cudaEventElapsedTime(&t01, ev[0], ev[1]); cudaEventElapsedTime(&t12, ev[1], ev[2]); cudaEventElapsedTime(&t23, ev[2], ev[3]);
        fprintf(stderr, "[tc_bgzf_inflate] %lld members, %lld -> %lld bytes: member index %.3f ms, upload + inflate + crc (in groups) %.3f ms, read-back %.3f ms\n",
                (long long)n_blocks, (long long)file_bytes, (long long)payload_bytes, t01, t12, t23);
        for (auto& e : ev) cudaEventDestroy(e);
    }
    if (h[0] != NO_ERROR) {
        const int code = (int)(h[0] & 0xff);
        return tc_fail(ctx, TC_ERR_ARG, code == CRC_ERR ? "BGZF member %lld: CRC-32 mismatch" : "BGZF member %lld does not inflate (code %d)",
                       (long long)(h[0] >> 8), code);
    }
    *payload_dev = d_payload;
    return TC_OK;
}

TC_API int tc_bam_index_records(tc_ctx_t* ctx, const uint8_t* payload_dev, int64_t n_bytes, int64_t first_record, int32_t n_ref,
                                const int32_t* ref_len, const int64_t** rec_off_dev, int64_t* n_placed, int64_t* n_records, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!payload_dev || n_bytes < 0 || first_record < 0 || first_record > n_bytes || n_ref < 0 || (n_ref > 0 && !ref_len) || !rec_off_dev || !n_placed || !n_records)
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (!tc_is_device_ptr(payload_dev)) return tc_fail(ctx, TC_ERR_ARG, "tc_bam_index_records needs the payload in device memory (tc_bgzf_inflate)");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    *rec_off_dev = nullptr; *n_placed = 0; *n_records = 0;
    if (first_record + 4 > n_bytes) return TC_OK;           // a header and nothing behind it
    chain_args a;
    memset(&a, 0, sizeof(a));
    int rc;
    a.u = payload_dev; a.n = n_bytes; a.first = first_record; a.n_ref = n_ref;
    a.ref_len = (const int32_t*)tc_stage_in(ctx, SLOT_TMP_C, ref_len, 4 * (size_t)(n_ref > 0 ? n_ref : 1), s, &rc); if (rc) return rc;
    a.n_chunks = (n_bytes + CHUNK - 1) / CHUNK;
    const size_t nc = (size_t)a.n_chunks;
    // S, E (8 bytes each), counts + offs (4 + 4, one more entry), on (1), ctl (3 x 8), totals (5 x 8)
    const size_t bytes = 16 * nc + 8 * (nc + 1) + ((nc + 7) & ~(size_t)7) + 64 + 64;
    uint8_t* d = (uint8_t*)tc_dev_buf(ctx, SLOT_TMP_A, bytes);
    if (!d) return TC_ERR_NOMEM;
    a.S = (long long*)d; a.E = a.S + nc;
    a.counts = (uint32_t*)(a.E + nc); uint32_t* d_offs = a.counts + (nc + 1);
    a.on = (uint8_t*)(d_offs + (nc + 1));
    a.ctl = (long long*)(a.on + ((nc + 7) & ~(size_t)7));
    a.totals = (unsigned long long*)(a.ctl + 8);
    a.offs = d_offs;
    TC_CUDA(cudaMemsetAsync(a.counts, 0, bytes - 16 * nc, s));
    TC_CUDA(cudaMemsetAsync(&a.ctl[0], 0xff, 8, s));                // "no chunk fails to link" = the largest value
    TC_CUDA(cudaMemsetAsync(&a.totals[4], 0xff, 8, s));
    const unsigned grid = (unsigned)((nc + 127) / 128);
    bam_chain_start_kernel<<<grid, 128, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    bam_chain_link_kernel<<<grid, 128, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    bam_chain_resolve_kernel<<<1, 1, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    bam_chain_walk_kernel<false><<<grid, 128, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, a.counts, d_offs, (int)(nc + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.counts, d_offs, (int)(nc + 1), s));
    ctx->launches++;
    long long* h = (long long*)ctx->host_status;
    TC_D2H(h, a.ctl, 24, s);
    TC_D2H(h + 3, a.totals, 40, s);
    TC_CUDA(cudaStreamSynchronize(s));
    if (h[2] != 0) return tc_fail(ctx, TC_ERR_ARG, "the BAM records do not form a chain (resolver code %lld): the payload is corrupt", h[2]);
    const unsigned long long* tot = (const unsigned long long*)(h + 3);
    if (tot[4] != NO_ERROR) return tc_fail(ctx, TC_ERR_ARG, "corrupt BAM record at payload offset %lld", (long long)(tot[4] - 1));
    if (tot[2] > 0xffffffffull || tot[3] > 0xffffffffull || tot[1] >= 0x7fffffffull)
        return tc_fail(ctx, TC_ERR_ARG, "more than 2^32 SEQ words or CIGAR operations (or 2^31-1 reads) in one BAM; shard the input");
    *n_records = (int64_t)tot[0]; *n_placed = (int64_t)tot[1];
    if (tot[1] == 0) return TC_OK;
    a.rec_off = (long long*)tc_dev_buf(ctx, SLOT_BAM_REC, 8 * (size_t)tot[1]);
    if (!a.rec_off) return TC_ERR_NOMEM;
    bam_chain_walk_kernel<true><<<grid, 128, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    *rec_off_dev = (const int64_t*)a.rec_off;
    return TC_OK;
}
