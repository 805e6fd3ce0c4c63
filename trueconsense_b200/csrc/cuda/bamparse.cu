// bamparse.cu — BAM records -> the flat read arrays of tc_reads_t, on the device.
//
// The step in front of the hot path: pysam's reader at TrueConsense/indexing.py:96 (SURVEY.md §8f rank 2).  The host inflates
// the BGZF blocks on all its cores and hops over the records once (csrc/host/bamio.c: tc_bam_payload — sequential by nature,
// every record says how long it is); the raw payload and the record offsets travel to the device ONCE and everything else
// happens here:
//   bam_meta_kernel   one thread per record: the fixed fields (refID, pos, MAPQ, FLAG, l_seq, next refID / pos, tlen), the two
//                     QNAME hashes, the reference span from the CIGAR, the words / ops the record will occupy; sort order,
//                     contig and span statistics
//   exclusive sums    cub::DeviceScan -> seq_off, cigar_off
//   bam_pack_kernel   one warp per record: CIGAR ops, SEQ bytes into 32-bit-word aligned slots (zero padded), QUAL bytes
// Result: the same arrays csrc/host/bamio.c's tc_bam_read fills (tests compare them byte for byte), resident in the context's
// read buffers like after tc_reads_upload — the CPU never touches a record's body.
#include <cub/device/device_scan.cuh>

#include "bamrec.cuh"
#include "tc_common.cuh"

namespace {

struct bam_args {
    const uint8_t* u; const long long* rec; long long n;
    int32_t* pos; uint16_t* flag; uint8_t* mapq; int32_t* l_seq; uint32_t* seq_n; uint32_t* cig_n;
    uint64_t* qname_hash; int32_t* mpos; int32_t* isize;
    const uint32_t* seq_off; const uint32_t* cigar_off; uint32_t* seq4; uint8_t* qual; uint32_t* cigar;
    tc_bam_stats_t* stats;
};

__global__ void __launch_bounds__(256) bam_meta_kernel(bam_args a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long span = 0;
    int bad_order = 0, other_contig = 0;
    if (i < a.n) {
        const uint8_t* r = a.u + a.rec[i];
        const int32_t tid = (int32_t)ld32(r + BAM_REF_ID), pos = (int32_t)ld32(r + BAM_POS);
        const uint32_t l_name = r[BAM_L_READ_NAME], n_cig = ld16(r + BAM_N_CIGAR_OP), l_seq = ld32(r + BAM_L_SEQ);
        const int32_t mtid = (int32_t)ld32(r + BAM_NEXT_REF_ID);
        a.pos[i] = pos; a.mapq[i] = r[BAM_MAPQ]; a.flag[i] = (uint16_t)ld16(r + BAM_FLAG); a.l_seq[i] = (int32_t)l_seq;
        // tc_reads_t.mpos: PNEXT, -2 when the mate maps to another reference
        a.mpos[i] = (mtid >= 0 && mtid != tid) ? -2 : (int32_t)ld32(r + BAM_NEXT_POS);
        a.isize[i] = (int32_t)ld32(r + BAM_TLEN);
        // low 32 bits: khash's X31 string hash (htslib keys its mate-overlap table with it), high 32: folded FNV-1a — as bamio.c
        const uint8_t* name = r + BAM_READ_NAME;
        uint32_t h = name[0];
        unsigned long long f = 1469598103934665603ull;
        for (uint32_t k = 0; k + 1 < l_name && name[k]; ++k) {
            if (k) h = (h << 5) - h + name[k];
            f ^= name[k]; f *= 1099511628211ull;
        }
        a.qname_hash[i] = ((unsigned long long)((uint32_t)(f >> 32) ^ (uint32_t)f) << 32) | h;
        const uint8_t* cg = name + l_name;
        for (uint32_t k = 0; k < n_cig; ++k) {
            const uint32_t c = ld32(cg + 4 * k);
            if (op_consumes_ref(c & 15u)) span += (long long)(c >> 4);
        }
        a.seq_n[i] = (l_seq + 7) / 8; a.cig_n[i] = n_cig;
        bad_order = bam_out_of_order(a.u, a.rec, i, tid, pos);
        other_contig = tid != (int32_t)ld32(a.u + a.rec[0] + BAM_REF_ID);
    }
    const long long wspan = __reduce_max_sync(0xffffffffu, (int)min(span, (long long)0x7fffffff));
    unsigned long long wsum = (unsigned long long)span;
#pragma unroll
    for (int o = 16; o; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    const unsigned any_bad = __ballot_sync(0xffffffffu, bad_order), any_other = __ballot_sync(0xffffffffu, other_contig);
    if ((threadIdx.x & 31) == 0) {
        if (wsum) atomicAdd(&a.stats->aligned_bases, wsum);
        if (wspan) atomicMax(&a.stats->max_ref_span, (int)wspan);
        if (any_bad) atomicExch(&a.stats->unsorted, 1);
        if (any_other) atomicExch(&a.stats->multi_contig, 1);
    }
}

// one warp per record; destination words / bytes are written whole (the padding behind the last base is zero, like calloc's)
__global__ void __launch_bounds__(256) bam_pack_kernel(bam_args a) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= a.n) return;
    const uint8_t* r = a.u + a.rec[i];
    const uint32_t n_cig = ld16(r + BAM_N_CIGAR_OP), l_seq = ld32(r + BAM_L_SEQ);
    const uint8_t* cg = bam_cigar(r);
    const uint8_t* sq = cg + 4 * (size_t)n_cig;
    const uint32_t sbytes = (l_seq + 1) / 2;
    const uint8_t* ql = sq + sbytes;
    const uint32_t co = a.cigar_off[i], so = a.seq_off[i], words = a.seq_off[i + 1] - so;
    for (uint32_t k = lane; k < n_cig; k += 32) a.cigar[co + k] = ld32(cg + 4 * (size_t)k);
    for (uint32_t w = lane; w < words; w += 32) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) { const uint32_t j = 4 * w + b; if (j < sbytes) v |= (uint32_t)sq[j] << (8 * b); }
        a.seq4[so + w] = v;
    }
    // QUAL: 8 bytes per SEQ word, written as 32-bit words
    uint32_t* qd = reinterpret_cast<uint32_t*>(a.qual + 8ull * so);
    for (uint32_t w = lane; w < 2 * words; w += 32) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) { const uint32_t j = 4 * w + b; if (j < l_seq) v |= (uint32_t)ql[j] << (8 * b); }
        qd[w] = v;
    }
}

}  // namespace

TC_API int tc_bam_records_to_reads(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                                   tc_reads_t* dev, tc_bam_stats_t* stats, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!dev || !stats || n_reads < 0 || n_bytes < 0 || (n_reads > 0 && (!payload || !rec_off))) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (n_reads >= (int64_t)0x7fffffff) return tc_fail(ctx, TC_ERR_ARG, "more than 2^31-1 reads in one batch; shard the input");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    memset(dev, 0, sizeof(*dev));
    memset(stats, 0, sizeof(*stats));
    stats->sorted = 1;
    const size_t n = (size_t)n_reads;
    if (n == 0) return TC_OK;
    int rc;
    bam_args a;
    memset(&a, 0, sizeof(a));
    a.u = (const uint8_t*)tc_stage_in(ctx, SLOT_BAM_PAYLOAD, payload, (size_t)n_bytes, s, &rc); if (rc) return rc;
    a.rec = (const long long*)tc_stage_in(ctx, SLOT_BAM_REC, rec_off, 8 * n, s, &rc); if (rc) return rc;
    a.n = n_reads;
    a.pos = (int32_t*)tc_dev_buf(ctx, SLOT_POS, 4 * n); a.flag = (uint16_t*)tc_dev_buf(ctx, SLOT_FLAG, 2 * n);
    a.mapq = (uint8_t*)tc_dev_buf(ctx, SLOT_MAPQ, n); a.l_seq = (int32_t*)tc_dev_buf(ctx, SLOT_LSEQ, 4 * n);
    a.qname_hash = (uint64_t*)tc_dev_buf(ctx, SLOT_QHASH, 8 * n); a.mpos = (int32_t*)tc_dev_buf(ctx, SLOT_MPOS, 4 * n);
    a.isize = (int32_t*)tc_dev_buf(ctx, SLOT_ISIZE, 4 * n);
    uint32_t* d_seq_off = (uint32_t*)tc_dev_buf(ctx, SLOT_SEQOFF, 4 * (n + 1));
    uint32_t* d_cig_off = (uint32_t*)tc_dev_buf(ctx, SLOT_CIGOFF, 4 * (n + 1));
    // sizes per record (one more, zero, entry so that the exclusive sums end with the totals), the stats block, cub's scratch
    uint32_t* d_sizes = (uint32_t*)tc_dev_buf(ctx, SLOT_TMP_A, 8 * (n + 1) + sizeof(tc_bam_stats_t) + 64);
    if (!a.pos || !a.flag || !a.mapq || !a.l_seq || !a.qname_hash || !a.mpos || !a.isize || !d_seq_off || !d_cig_off || !d_sizes) return TC_ERR_NOMEM;
    a.seq_n = d_sizes; a.cig_n = d_sizes + (n + 1);
    a.stats = (tc_bam_stats_t*)(d_sizes + 2 * (n + 1));
    TC_CUDA(cudaMemsetAsync(d_sizes, 0, 8 * (n + 1) + sizeof(tc_bam_stats_t), s));
    bam_meta_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    size_t tmp_bytes = 0;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, a.seq_n, d_seq_off, (int)(n + 1), s));
    void* d_tmp = tc_dev_buf(ctx, SLOT_TMP_B, tmp_bytes + 16);
    if (!d_tmp) return TC_ERR_NOMEM;
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.seq_n, d_seq_off, (int)(n + 1), s));
    TC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a.cig_n, d_cig_off, (int)(n + 1), s));
    ctx->launches += 2;
    // the totals size the big arrays: one small read-back
    uint32_t* h = (uint32_t*)ctx->host_status;
    TC_D2H(h, d_seq_off + n, 4, s);
    TC_D2H(h + 1, d_cig_off + n, 4, s);
    TC_D2H(h + 2, a.stats, sizeof(tc_bam_stats_t), s);
    TC_CUDA(cudaStreamSynchronize(s));
    const size_t n_words = h[0], n_ops = h[1];
    // (totals beyond 32 bits wrap: the host's hop over the records has summed them already and refuses such a batch)
    a.seq_off = d_seq_off; a.cigar_off = d_cig_off;
    a.seq4 = (uint32_t*)tc_dev_buf(ctx, SLOT_SEQ4, 4 * n_words + 16);
    a.qual = (uint8_t*)tc_dev_buf(ctx, SLOT_QUAL, 8 * n_words + 16);
    a.cigar = (uint32_t*)tc_dev_buf(ctx, SLOT_CIGAR, 4 * n_ops + 16);
    if (!a.seq4 || !a.qual || !a.cigar) return TC_ERR_NOMEM;
    bam_pack_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, s>>>(a);
    TC_LAUNCH_CHECK();
    memcpy(stats, h + 2, sizeof(*stats));
    stats->sorted = stats->unsorted ? 0 : 1;
    stats->n_seq_words = (int64_t)n_words; stats->n_cigar_ops = (int64_t)n_ops;
    dev->n_reads = n_reads; dev->n_seq_words = (int64_t)n_words; dev->n_cigar_ops = (int64_t)n_ops;
    dev->pos = a.pos; dev->flag = a.flag; dev->mapq = a.mapq; dev->l_seq = a.l_seq; dev->seq_off = d_seq_off; dev->cigar_off = d_cig_off;
    dev->seq4 = a.seq4; dev->qual = a.qual; dev->cigar = a.cigar; dev->qname_hash = a.qname_hash; dev->mpos = a.mpos; dev->isize = a.isize;
    dev->max_ref_span = stats->max_ref_span;
    return TC_OK;
}
