// tc_common.cuh — context, error handling, staging and small device helpers shared by the
// kernels behind include/trueconsense_b200.h.  sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <functional>

#include "trueconsense_b200.h"

#define TC_API extern "C" __attribute__((visibility("default")))

// grow-only device buffers owned by a context
enum tc_slot {
    SLOT_POS = 0, SLOT_FLAG, SLOT_MAPQ, SLOT_LSEQ, SLOT_SEQOFF, SLOT_CIGOFF, SLOT_SEQ4, SLOT_QUAL, SLOT_CIGAR,
    SLOT_QHASH, SLOT_MPOS, SLOT_ISIZE,
    SLOT_COUNTS, SLOT_DIFF, SLOT_STATUS, SLOT_SPAN_END, SLOT_CALL_A, SLOT_CALL_B, SLOT_CALL_C, SLOT_CALL_D,
    SLOT_CALL_E, SLOT_CALL_F, SLOT_INS_A, SLOT_INS_B, SLOT_INS_C, SLOT_INS_D, SLOT_INS_E, SLOT_INS_F, SLOT_INS_G,
    SLOT_TMP_A, SLOT_TMP_B, SLOT_TMP_C, SLOT_TILES, SLOT_SEGS, SLOT_COV_TOTALS, SLOT_BAM_PAYLOAD, SLOT_BAM_REC, SLOT_CIGAR16, SLOT_SEQ2, SLOT_SEQ_EXC_IDX, SLOT_SEQ_EXC_VAL, SLOT_BGZF_FILE, SLOT_BGZF_BLOCKS,
    SLOT_CONTIG_A, SLOT_CONTIG_B, SLOT_CONTIG_C, SLOT_BAM_REC_SORTED, SLOT_SAM_TEXT, SLOT_SAM_LINES, SLOT_SAM_META, SLOT_SAM_REFS,
    SLOT_CLIP_PLAN, SLOT_CLIP_PAYLOAD, SLOT_CLIP_REC,
    SLOT_COUNT
};

struct tc_buf { void* p; size_t cap; };

constexpr size_t TC_HOST_SCRATCH = 64 * 1024;
struct tc_status;
struct pileup_plan {            // one attempt at the count table (pileup_plan_of, pileup.cu)
    int variant;                // 1 scatter, 3 warp streams, 4 long reads cut into pieces for the warp streams
    bool span_pass;             // a pass over the CIGARs finds the spans first (else variant 3 checks them itself)
    bool span_out;              // ... and leaves every read's span for variant 4's split
};
struct tc_pileup_pending {      // what tc_pileup_settle needs once the status block is on the host
    tc_status* d_status; int32_t* d_counts; pileup_plan plan; int out_dev; int64_t n_reads;
};

struct tc_ctx {
    int device;
    int sm_count;
    char err[512];
    int64_t launches;
    int64_t h2d_bytes, d2h_bytes;
    tc_buf bufs[SLOT_COUNT];
    int ins_attr_set;       // ins_count_kernel's shared-memory attribute has been set
    uint32_t warp_attr_set; // ... and those of the warp_pileup_kernel instances (one bit each)
    void* host_status;      // pinned, 256 bytes
    void* host_scratch;     // pinned, TC_HOST_SCRATCH bytes: small results come back here in truly asynchronous copies
                            // (a cudaMemcpyAsync into pageable memory waits for the stream)
    int timing;             // bracket the pileup kernel with events
    cudaEvent_t ev0, ev1;
    int ev_valid;
    // the span bound (tc_reads_t.max_ref_span) tc_pileup_counts verified last, and for which arrays: tc_extract_inserts
    // trusts a bound only when it is this one — otherwise it finds the longest span itself
    const void* span_ok_cigar; const void* span_ok_off; int64_t span_ok_n, span_ok_ops; int32_t span_ok_bound;
    int64_t pair_cap;       // tc_extract_inserts: bytes of scratch for the rewritten quality strings of overlapping mates; grows on demand
    int64_t ins_slot_cap;   // tc_extract_inserts: entry slots its speculative (no read-back) layout may use; grows on demand
    struct tc_sample_slot* samples;     // [2] samples in flight (tc_sample_enqueue / tc_sample_finish), allocated on first use
    int sample_next;
    int64_t buf_epoch;      // bumped whenever a context buffer is (re)allocated: captured graphs hold the old addresses
    cudaStream_t cap_stream;    // the stream sample graphs are captured on (a user's legacy default stream cannot be captured)
    int in_capture;         // timing events inside a capture are recorded as external event nodes
    float finished_ms;      // timing on: pileup-kernel duration of the sample tc_sample_finish returned last (< 0: none)
    // tc_pileup_counts_allreduce_enqueue / _finish: two shard passes in flight (allreduce.cu), each slot with its own graph
    struct tc_rr_slot* rr; int rr_next;
    // staging ring for large uploads from pageable memory (tc_stage_in): TC_RING_SLOTS pinned buffers of TC_RING_CHUNK bytes
    void* ring; cudaEvent_t ring_ev[8];
    cudaStream_t aux[4]; cudaEvent_t aux_ev[5];      // tc_bgzf_inflate: groups of members inflate on two side streams behind their upload
};

// device-side status block written by kernels, read back once per call
struct tc_status {
    int err;            // first TC_ERR_* raised on the device (0 = none)
    int max_cov;        // maximum of the coverage row
    int n_zero_span;    // reads with no reference span
    int max_span;       // longest reference span
    unsigned long long aligned; // pileup entries produced (coverage sum) — bookkeeping
    int reserved[10];
};

int tc_fail(tc_ctx* ctx, int code, const char* fmt, ...);
int tc_cuda_fail(tc_ctx* ctx, cudaError_t e, const char* what);
void* tc_dev_buf(tc_ctx* ctx, int slot, size_t bytes);       // NULL on failure (ctx->err set)
bool tc_is_device_ptr(const void* p);
// returns a device pointer for `p` (n bytes): p itself if it already is one, else a staged copy in `slot`
const void* tc_stage_in(tc_ctx* ctx, int slot, const void* p, size_t bytes, cudaStream_t s, int* rc);

#define TC_CUDA(call)                                                       \
    do {                                                                    \
        cudaError_t e__ = (call);                                           \
        if (e__ != cudaSuccess) return tc_cuda_fail(ctx, e__, #call);       \
    } while (0)

// device -> host copy with byte accounting
#define TC_D2H(dst, src, bytes, s)                                                            \
    do {                                                                                      \
        TC_CUDA(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, (s)));          \
        ctx->d2h_bytes += (int64_t)(bytes);                                                   \
    } while (0)

#define TC_LAUNCH_CHECK()                                                   \
    do {                                                                    \
        ctx->launches++;                                                    \
        cudaError_t e__ = cudaGetLastError();                               \
        if (e__ != cudaSuccess) return tc_cuda_fail(ctx, e__, "kernel launch"); \
    } while (0)

// device view of a read batch (device pointers only)
struct dreads {
    int64_t n;
    const int32_t* pos; const uint16_t* flag; const uint8_t* mapq; const int32_t* l_seq;
    const uint32_t* seq_off; const uint32_t* cigar_off; const uint32_t* seq4; const uint8_t* qual;
    const uint32_t* cigar; const uint64_t* qname_hash; const int32_t* mpos; const int32_t* isize;
};

// which arrays a pass needs on the device
#define NEED_QUAL  1
#define NEED_MATE  2
// host-resident seq4 / cigar / qual: give them full-size device buffers but copy nothing — the caller stages
// only the ranges its pass will read (tc_extract_inserts: the reads over the candidate columns)
#define DEFER_SEQ   4
#define DEFER_CIGAR 8
#define DEFER_QUAL  16
#define DEFER_MATE  32
int tc_resolve_reads(tc_ctx* ctx, const tc_reads_t* in, dreads* out, int need, cudaStream_t s);

// ---- pieces of the entry points that only ENQUEUE (tc_pileup_call_inserts chains them without a host round trip)
// rung: the variant of the fallback ladder to run; 0 the first attempt (p->kernel, or for 0 the library's choice)
int tc_pileup_enqueue(tc_ctx* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* p, int32_t* counts, cudaStream_t s,
                      tc_pileup_pending* pend, int rung = 0);
// redone (may be NULL): set to 1 when the batch went down the fallback ladder, i.e. another variant rebuilt the table
int tc_pileup_settle(tc_ctx* ctx, tc_status st, tc_pileup_pending pend, const tc_reads_t* reads, int32_t ref_len,
                     const tc_pileup_params_t* p, int32_t* counts, cudaStream_t s, int* redone);
int tc_h2d(tc_ctx* ctx, void* d, const void* p, size_t bytes, cudaStream_t s);
bool tc_reads_all_device(const tc_reads_t* r);     // every array of the batch already in device memory
int tc_candidates_enqueue(tc_ctx* ctx, const uint8_t* d_flags, int32_t ref_len, int32_t cap, int32_t** d_count, int32_t** d_sorted, cudaStream_t s);
// ExtractInserts' results block: one memset in front, one copy back.  Offsets in bytes; ins_block_of (inserts.cu) lays it out.
struct ins_block {
    size_t layout;      // int32[3] device-built layout: tiles, slots, 1 = did not fit
    size_t over;        // int32 overflow flags: 1 a column needs the sorted form, 2 the pair scratch was too small
    size_t bump;        // uint64 pair-scratch bump
    size_t extra;       // chained form only (else 0): candidate count, pileup status, candidates (TC_RB_EXTRA_*)
    size_t seg;         // int32 seg_count[n_cand + 1], then pair_any[n_cand + 1]
    size_t calls;       // tc_insert_call_t[n_cand]
    size_t fixed;       // uint8[n_cand][INS_BASES_FIXED] inserted characters of each winner
    size_t bytes;       // the whole block
};
// int32 words of the chained form's extra section
constexpr int TC_RB_EXTRA_NCAND = 0, TC_RB_EXTRA_STATUS = 16, TC_RB_EXTRA_CAND = 32;
struct tc_ins_pending { ins_block rb; int cap; int64_t n_reads; };
int tc_inserts_enqueue_dev(tc_ctx* ctx, const tc_reads_t* reads, const int32_t* d_cand, const int32_t* d_ncand, int cap,
                           const tc_pileup_params_t* p, const tc_status* d_pileup_status, void* host_block, cudaStream_t s, tc_ins_pending* pend);
int tc_inserts_finish_dev(tc_ctx* ctx, const tc_ins_pending* pend, const void* host_block, tc_status* pileup_status, int32_t* cands, int32_t* n_cand,
                          tc_insert_call_t* calls, uint8_t* bases, int64_t bases_cap, int* fit);
// A chain of enqueues as a CUDA graph, keyed by everything it depends on: the first run with a key is eager (and
// allocates), the second is captured (when can_capture and TC_NO_GRAPH is unset), later ones replay.  A failed capture
// runs the chain eagerly and tries again next time.
struct tc_graph_cache {
    unsigned char key[512]; int key_len, seen;
    cudaGraphExec_t exec; int64_t g_launches, g_d2h;        // what one replay adds to the context's counters
};
int tc_graph_run(tc_ctx* ctx, tc_graph_cache& g, const unsigned char* key, int key_len, bool can_capture,
                 const std::function<int(cudaStream_t)>& chain, cudaStream_t s);
void tc_graph_destroy(tc_graph_cache& g);
// a sample in flight
struct tc_sample_slot {
    int state;                      // 0 free, 1 chained and enqueued, 2 to be run through the separate calls at finish time
    void* host_block;               // pinned, TC_HOST_SCRATCH bytes: this sample's results block
    cudaEvent_t done, t0, t1;       // t0 / t1: around this sample's pileup kernel when the context's timing is on
    int timed;
    tc_reads_t reads; int32_t ref_len; tc_pileup_params_t pp, ip; tc_call_params_t cp; int32_t* counts; tc_call_table_t table; void* stream;
    tc_pileup_pending pend; tc_ins_pending ipend;
    tc_graph_cache graph;           // one launch per sample instead of ~25 (kernels, memsets, the results copy)
};

// ---------------------------------------------------------------- device helpers
enum { OP_M = 0, OP_I = 1, OP_D = 2, OP_N = 3, OP_S = 4, OP_H = 5, OP_P = 6, OP_EQ = 7, OP_X = 8 };

__device__ __forceinline__ bool op_consumes_ref(uint32_t op) {
    // M, D, N, =, X  -> bits 0,2,3,7,8
    return (0x18Du >> op) & 1u;
}
__device__ __forceinline__ bool op_is_match(uint32_t op) { return (0x181u >> op) & 1u; }          // M, =, X
__device__ __forceinline__ bool op_consumes_query_skip(uint32_t op) { return op == OP_I || op == OP_S; }

// 4-bit base code q of a read whose packed words start at w (BAM byte stream inside the words)
__device__ __forceinline__ uint32_t seq_code(const uint32_t* __restrict__ w, int q) {
    uint32_t word = __ldg(w + (q >> 3));
    uint32_t byte = (word >> (8 * ((q >> 1) & 3))) & 0xffu;
    return (q & 1) ? (byte & 15u) : (byte >> 4);
}

// count-table row of a base code: A=1, C=2, G=4, T=8 -> rows A,C,G,T ; anything else -> -1
__device__ __forceinline__ int code_row(uint32_t code) {
    // TC_ROW_A=1, TC_ROW_T=2, TC_ROW_C=3, TC_ROW_G=4
    switch (code) {
        case 1: return TC_ROW_A;
        case 2: return TC_ROW_C;
        case 4: return TC_ROW_G;
        case 8: return TC_ROW_T;
        default: return -1;
    }
}

// indel reported on the last column of reference-consuming op k (htslib resolve_cigar2's peek)
__device__ __forceinline__ int peek_indel(const uint32_t* __restrict__ cig, int n, int k) {
    if (k + 1 >= n) return 0;
    uint32_t op = cig[k] & 15u;
    uint32_t c2 = cig[k + 1];
    uint32_t op2 = c2 & 15u;
    int indel = 0;
    if (op2 == OP_D && op != OP_D) {
        indel = -(int)(c2 >> 4);
        for (int j = k + 2; j < n; ++j) {
            uint32_t c = cig[j];
            if ((c & 15u) == OP_D) indel -= (int)(c >> 4); else break;
        }
    } else if (op2 == OP_I) {
        indel = (int)(c2 >> 4);
        for (int j = k + 2; j < n; ++j) {
            uint32_t c = cig[j]; uint32_t o = c & 15u;
            if (o == OP_I) indel += (int)(c >> 4);
            else if (o != OP_P) break;
        }
    } else if (op2 == OP_P && k + 2 < n) {
        int l3 = 0;
        for (int j = k + 2; j < n; ++j) {
            uint32_t c = cig[j]; uint32_t o = c & 15u;
            if (o == OP_I) l3 += (int)(c >> 4);
            else if (op_consumes_ref(o)) break;
        }
        if (l3 > 0) indel = l3;
    }
    return indel;
}
