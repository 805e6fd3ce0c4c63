/*
 * trueconsense_b200.h — C-ABI of the B200 pileup-and-call hot path.
 *
 * This is the drop-in boundary for the path TrueConsense implements in
 *   TrueConsense/indexing.py:75-154   (BuildIndex: whole-BAM pileup -> count table)
 *   TrueConsense/Events.py:5-82       (ListInserts / ExtractInserts)
 *   TrueConsense/Coverage.py:1-34     (coverage column)
 *   TrueConsense/Sequences.py:119-165 (GetNucleotide / GetDistribution ranking)
 *   TrueConsense/Ambig.py:102-228     (IsAmbiguous and helpers)
 *   TrueConsense/Events.py:85-106     (MinorityDel)
 * The reference has no FFI of its own (it is pure Python on top of pysam/htslib); the
 * entry points below are what a ctypes binding inside those modules would call
 * (INTEGRATION.md shows the stubs).  Plain pointers and sizes only; every pointer
 * argument may be a host pointer (pageable or pinned) or a device pointer — the
 * library asks the CUDA runtime which (cudaPointerGetAttributes) and stages host
 * buffers through context-owned device memory.  All work is enqueued on `stream`
 * (a cudaStream_t passed as void*; NULL = the legacy default stream).  Calls that
 * return results to HOST memory synchronise the stream before returning; calls whose
 * outputs are device pointers return as soon as the work is enqueued.
 *
 * Thread-safety: a tc_ctx_t may be used by one thread at a time; different
 * contexts are independent.  The reference calls BuildIndex from a pool thread
 * (TrueConsense/TrueConsense.py:225-226), so every entry point sets the CUDA
 * device of its context itself.
 *
 * A pass covers one reference (contig); a BAM with several is called in one pass by placing its references side by side
 * (tc_bam_contig_ranges, tc_reads_to_contig_coords, tc_call_contigs below).
 *
 * There is no CPU fallback anywhere behind this ABI: without a CUDA device
 * tc_ctx_create fails with TC_ERR_NO_DEVICE.
 */
#ifndef TRUECONSENSE_B200_H
#define TRUECONSENSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TC_ABI_VERSION 3

/* ---- error codes (0 = success, negative = failure) ---- */
#define TC_OK              0
#define TC_ERR_CUDA       -1  /* a CUDA runtime call failed; see tc_last_error() */
#define TC_ERR_ARG        -2  /* bad argument (NULL pointer, negative size, ...) */
#define TC_ERR_UNSORTED   -3  /* reads are not sorted by position (htslib: "Unsorted input. Pileup aborts") */
#define TC_ERR_DEPTH_CAP  -4  /* the max_depth cap of the full-file pileup could bind; not emulated in bulk */
#define TC_ERR_NOMEM      -5
#define TC_ERR_NO_DEVICE  -6
#define TC_ERR_RANGE      -7  /* an offset / CIGAR walks outside its buffer */
#define TC_ERR_CAPACITY   -8  /* caller-provided output buffer too small */

/* ---- count table: int32 counts[TC_NROWS][ref_len], row-major planes ----
 * Rows 0..6 are the seven columns of the reference's index frame in its own order
 * (indexing.py:134: coverage, A, T, C, G, X, I); row 7 is padding so one position's
 * plane stride stays a multiple of 32 bytes. Column j is reference position j+1. */
enum {
    TC_ROW_COV = 0, TC_ROW_A = 1, TC_ROW_T = 2, TC_ROW_C = 3, TC_ROW_G = 4,
    TC_ROW_X = 5, TC_ROW_I = 6, TC_ROW_PAD = 7, TC_NROWS = 8
};

/* ---- flat read arrays (what the BAM decoder produces; BAM field names) ----
 * Reads are in file order and must be sorted by `pos` (coordinate-sorted BAM, one contig — or several references moved
 * side by side by tc_reads_to_contig_coords).
 * seq4 uses BAM's own packing (high nibble first, codes "=ACMGRSVTWYHKDBN"), but every
 * read starts on a 32-bit word boundary: read i occupies words seq_off[i] .. seq_off[i+1]-1,
 * the byte stream inside those words is the BAM byte stream.  QUAL shares the same
 * offsets: base q of read i is qual[8*seq_off[i] + q].  A read with l_seq == 0 (SEQ '*')
 * has no words.  cigar uses BAM's encoding (len<<4 | op, ops MIDNSHP=X = 0..8); read i
 * owns cigar[cigar_off[i] .. cigar_off[i+1]-1]. */
typedef struct tc_reads {
    int64_t n_reads;
    int64_t n_seq_words;        /* total 32-bit words in seq4 (== seq_off[n_reads]) */
    int64_t n_cigar_ops;        /* total CIGAR ops (== cigar_off[n_reads]) */
    const int32_t*  pos;        /* [n]   0-based leftmost reference coordinate */
    const uint16_t* flag;       /* [n]   BAM FLAG */
    const uint8_t*  mapq;       /* [n]   MAPQ */
    const int32_t*  l_seq;      /* [n]   query length (0 when SEQ is '*') */
    const uint32_t* seq_off;    /* [n+1] word offsets into seq4 (and /8 byte offsets into qual) */
    const uint32_t* cigar_off;  /* [n+1] op offsets into cigar */
    const uint32_t* seq4;       /* [n_seq_words] */
    const uint8_t*  qual;       /* [8*n_seq_words] phred bytes; may be NULL when no pass reads QUAL */
    const uint32_t* cigar;      /* [n_cigar_ops] */
    /* mate information, read by tc_extract_inserts' emulation of htslib's mate-overlap quality rewriting (pysam's default
     * ignore_overlaps=True, Events.py:66); all three NULL: no rewriting */
    const uint64_t* qname_hash; /* [n] a hash of QNAME, equal for all alignments of a template; its low 32 bits should be htslib's
                                   own string hash of the name (khash X31: h = c0; h = 31 h + c) — which mate keeps its qualities
                                   is drawn from it */
    const int32_t*  mpos;       /* [n] PNEXT (0-based); -1 if unavailable, -2 if the mate maps to another reference */
    const int32_t*  isize;      /* [n] TLEN */
    /* optional: an upper bound of the longest reference span (sum of M,=,X,D,N lengths) of any read, which a
     * BAM decoder knows for free; 0 = unknown (the library then finds it with one more pass over the CIGARs).
     * tc_pileup_counts verifies the bound while it walks the CIGARs and fails with TC_ERR_ARG if it is too small. */
    int32_t max_ref_span;
    int32_t reserved;
    /* optional compact transport of the CIGARs: the same n_cigar_ops operations as 16-bit (len << 4 | op) entries, offered
     * only when every operation is shorter than 4096 (the producer checks; the entries then equal the 32-bit ones).  When
     * both arrays sit in host memory the library copies this one — half the bytes over PCIe — and widens it on the device.
     * `cigar` may be NULL when this is given. */
    const uint16_t* cigar16;
    /* optional compact transport of SEQ: two bits per base (A C G T = 0 1 2 3), one 16-bit entry per seq4 word with the same
     * offsets — entry w holds the 8 bases of seq4[w], base j of the word in bits 2j+1:2j — plus the list of the words that hold
     * anything else than A / C / G / T over their valid bases (N, IUPAC codes, '='): seq_exc_idx (ascending word indices) and
     * seq_exc_val (those seq4 words as they are).  A decoder has both forms for free (tc_host.h: tc_seq2_pack).  When SEQ sits
     * in host memory the library copies seq2 and the exceptions — half the bytes — and rebuilds seq4 on the device, zero padding
     * included.  `seq4` may be NULL when this is given. */
    const uint16_t* seq2;
    const uint32_t* seq_exc_idx;
    const uint32_t* seq_exc_val;
    int64_t         n_seq_exc;
} tc_reads_t;

/* ---- pileup filters: the arguments of pysam's AlignmentFile.pileup() that the
 * reference passes (indexing.py:100) or leaves at their defaults (Events.py:66) ---- */
typedef struct tc_pileup_params {
    uint32_t flag_filter;       /* reads with (flag & flag_filter) != 0 are skipped. BuildIndex: 0x4 (htslib
                                   always drops UNMAP); ExtractInserts: 0x4|0x100|0x200|0x400 */
    int32_t  min_mapq;          /* reads with mapq < min_mapq are skipped (both call sites: 0) */
    int32_t  min_base_quality;  /* entries with qual < this are skipped. BuildIndex: 0; ExtractInserts: 13 */
    int32_t  ignore_orphans;    /* skip PAIRED && !PROPER_PAIR reads. BuildIndex (nofilter): 0; ExtractInserts: 1 */
    int64_t  max_depth;         /* BuildIndex: 10000000; ExtractInserts: 8000 */
    int32_t  kernel;            /* 0 = library's choice; 1 = scatter (smem atomics); 3 = bit-parallel, one warp per read stream;
                                   4 = long reads: cut into pieces, then 3 */
    int32_t  reserved;          /* bit 0: used by the library when it re-enters itself (pass 0).  Bits 8-9, only read with a base-quality
                                   filter: mate-overlap quality rewriting — 0 = as htslib >= 1.13 does it (pysam 0.23.3 bundles 1.21),
                                   1 = off (pysam's ignore_overlaps=False), 2 = as htslib <= 1.12 did (the first mate keeps its quality) */
} tc_pileup_params_t;

/* ---- per-position call table (struct of arrays, each of length ref_len) ----
 * Everything Sequences.BuildConsensus (Sequences.py:179-318) reads per position. */
#define TC_CF_LOWCOV        0x01  /* cov <  mincov           (Sequences.py:191) */
#define TC_CF_PRIMARY_X     0x02  /* rank-1 letter is 'X'    (Sequences.py:210,277) */
#define TC_CF_MINORITY_DEL  0x04  /* (X/cov)*100 >= 15       (Events.py:100-106); 0 when cov == 0 */
#define TC_CF_INS_CANDIDATE 0x08  /* ListInserts test        (Events.py:25-36) */
#define TC_CF_COV_GT_MINCOV 0x10  /* cov >  mincov (strict)  (Sequences.py:311, ORFs.py:139) */
#define TC_CF_XRUN_OFF_END  0x20  /* the X-run after this position reaches ref_len: WalkForward
                                     (Sequences.py:44-52) would raise KeyError(ref_len+1) */
#define TC_CF_ZERO_COV      0x40  /* cov == 0: MinorityDel here raises ZeroDivisionError (Events.py:102) */
#define TC_CF_AMBIG         0x80  /* IsAmbiguous(...)[0]     (Ambig.py:179-228) */

typedef struct tc_call_table {
    uint8_t* call_char;     /* the character the walk appends when it takes the plain branch:
                               rank-1 != 'X': ambiguity char if include_ambig && ambiguous, else rank-1 letter,
                                              lower-case when its count < mincov (Sequences.py:269-275);
                               rank-1 == 'X': rank-2 letter, lower-case when its count < mincov (Sequences.py:283-291) */
    uint8_t* flags;         /* TC_CF_* */
    int32_t* xrun;          /* len(WalkForward(index, p)): consecutive positions after p whose rank-1 is 'X' */
    uint8_t* rank_letter;   /* [4][ref_len]  GetNucleotide(index,p,k) letters for k=1..4 ('A','T','C','G','X') */
    int32_t* rank_count;    /* [4][ref_len]  ... and their counts */
    uint8_t* ambig_char;    /* IsAmbiguous(...)[1] as ASCII, 0 when not ambiguous */
} tc_call_table_t;

typedef struct tc_call_params {
    int32_t mincov;
    int32_t include_ambig;      /* IncludeAmbig of BuildConsensus */
    double  ambig_maxdist;      /* 10  (Ambig.py:156) */
    double  minority_del_pct;   /* 15  (Events.py:104) */
    double  insert_pct;         /* 55  (Events.py:36) */
} tc_call_params_t;

/* ---- result of the ExtractInserts emulation for one candidate position ---- */
typedef struct tc_insert_call {
    int32_t pos;            /* 1-based position, the reference's dict key */
    int32_t n_entries;      /* strings in the column after all filters (0: pysam returns "" -> (None, None)) */
    int32_t mode_count;     /* multiplicity of the modal upper-cased string */
    int32_t first_read;     /* index of the read that contributed its first occurrence */
    int32_t head;           /* ASCII of the modal string's first character (already upper-cased) */
    int32_t indel;          /* >0 "+n<bases>", <0 "-n" followed by n 'N', 0 no suffix */
    int64_t bases_off;      /* offset of the n inserted characters in the bases buffer (indel > 0) */
} tc_insert_call_t;

typedef struct tc_ctx tc_ctx_t;

/* ---- lifecycle ---- */
int  tc_abi_version(void);
/* device < 0: current device.  Fails with TC_ERR_NO_DEVICE when no CUDA device is usable. */
int  tc_ctx_create(int device, tc_ctx_t** out);
int  tc_ctx_destroy(tc_ctx_t* ctx);
/* text of the last failure on this context (or of the last failed tc_ctx_create when ctx == NULL) */
const char* tc_last_error(const tc_ctx_t* ctx);
/* number of kernel launches this context has issued so far (bench.py's gpu_launches) */
int64_t tc_launch_count(const tc_ctx_t* ctx);
/* Measurement aid (no counterpart in the reference): when enabled, tc_pileup_counts brackets its
 * dominant kernel (the pileup kernel proper, without memsets / scan / copies) with CUDA events on
 * the launching stream; tc_last_pileup_kernel_ms returns the duration of the most recent one (after tc_sample_finish:
 * of the sample that call finished). */
/* bytes this context has copied host->device / device->host so far (bench.py's e2e accounting) */
int  tc_transfer_bytes(const tc_ctx_t* ctx, int64_t* h2d, int64_t* d2h);
int  tc_ctx_set_timing(tc_ctx_t* ctx, int enabled);
float tc_last_pileup_kernel_ms(tc_ctx_t* ctx);

/* Copy a host read batch into context-owned device memory and fill *dev with device
 * pointers (valid until the next tc_reads_upload on this context or tc_ctx_destroy).
 * Arrays that are NULL in *host stay NULL.  Already-device pointers are passed through. */
int  tc_reads_upload(tc_ctx_t* ctx, const tc_reads_t* host, tc_reads_t* dev, void* stream);

/* Copy `bytes` from device memory (e.g. an array of a device-resident tc_reads_t) to the host; synchronises the stream. */
int  tc_download(tc_ctx_t* ctx, void* dst_host, const void* src_dev, int64_t bytes, void* stream);

/* ---- BAM records -> read arrays on the device: the reader half of pysam.AlignmentFile at indexing.py:96 ----
 * payload: the BAM's uncompressed stream (the concatenated payload of its BGZF blocks), host or device memory;
 * rec_off[n_reads]: for every record to keep, in file order, the offset of its refID field (block_size sits 4 bytes in
 * front) — what the host's one sequential hop over the records yields (libtchost.so: tc_bam_payload inflates on all cores and
 * hops).  The device parses the fixed fields, hashes the names, walks the CIGARs and packs SEQ / QUAL / CIGAR into
 * context-owned buffers; *dev receives device pointers (valid until the next tc_reads_upload / tc_bam_records_to_reads on this
 * context), exactly the arrays a host-side decode + tc_reads_upload would give.  The caller has validated the records'
 * sizes (tc_bam_payload does).  Synchronises the stream once. */
typedef struct tc_bam_stats {
    unsigned long long aligned_bases;   /* sum over the kept reads of M,=,X,D,N lengths */
    int32_t max_ref_span;
    int32_t unsorted;                   /* some record sorts before its predecessor by (refID, pos) */
    int32_t multi_contig;               /* records of more than one reference */
    int32_t sorted;                     /* !unsorted */
    int64_t n_seq_words, n_cigar_ops;
} tc_bam_stats_t;
int  tc_bam_records_to_reads(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                             tc_reads_t* dev, tc_bam_stats_t* stats, void* stream);

/* Coordinate order for a BAM's records (what `samtools sort` would give). payload / rec_off as tc_bam_records_to_reads
 * takes them (host or device); *payload_dev and *rec_sorted_dev feed tc_bam_records_to_reads and tc_bam_contig_ranges.
 * Records already sorted by (refID, pos) keep their order (*reordered = 0). TC_ERR_RANGE: refID outside [0, n_ref) or
 * pos < -1. Synchronises the stream once (twice when it reorders: the sorted offsets are complete on return).
 * The order otherwise: refID, then pos, then forward strand before reverse (FLAG 0x10), then file order (a stable radix sort
 * over 64-bit keys).  Host inputs are staged once into the context's payload / record buffers; the sorted offsets live in a
 * buffer of their own that neither tc_bam_records_to_reads nor tc_bam_contig_ranges writes, valid until the next call that
 * decodes a BAM on this context.  n_reads == 0: the inputs are handed back as they are. */
int  tc_bam_sort_records(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                         int32_t n_ref, const uint8_t** payload_dev, const int64_t** rec_sorted_dev, int32_t* reordered,
                         void* stream);

/* ---- amplicon primers soft-clipped off the aligned records (samtools ampliconclip --soft-clip; the rule: DESIGN §4) ----
 * payload / rec_off as tc_bam_sort_records takes them (host or device).  The primers: n_primers rows of 0-based half-open
 * [primer_start, primer_end) on reference primer_ref (host or device; 0 <= start < end, refs in [0, n_ref), else TC_ERR_ARG).
 * tolerance >= 0; mode bit 0: check both ends of every read (else only the 5' end: left for forward, right for reverse reads).
 * A placed, mapped record with an M / = / X op whose checked end lies under a primer loses those reference columns to a soft
 * clip (pos, CIGAR, n_cigar_op, block_size and bin change); a record left without a match op is marked unmapped (FLAG 0x4,
 * pos and CIGAR as they were).  Every other byte is copied.  *payload_dev / *rec_off_dev: the records in input order in a
 * context buffer of their own (distinct from the payload, record and sorted-offset buffers; valid until the next decode on this
 * context), *n_bytes_out their bytes; they feed tc_bam_sort_records, tc_bam_records_to_reads and tc_bam_contig_ranges as they
 * are.  stats: records clipped on the left / on the right (that stay mapped), records fully clipped, reference columns removed.
 * TC_ERR_ARG naming the record: a clipped CIGAR of more than 65535 ops; a mapped record with an M / = / X op whose CIGAR has
 * an op of length 0 or an H / S op between other ops (the SAM spec allows neither).  Synchronises the stream once (twice
 * when the primer rows are in device memory: they are read back first).
 * n_reads == 0: the inputs are handed back as they are (*payload_dev = payload, which may be host memory, *n_bytes_out =
 * n_bytes, *rec_off_dev = rec_off). */
typedef struct tc_clip_stats { int64_t n_left, n_right, n_unmapped, n_columns; } tc_clip_stats_t;
int  tc_bam_clip_primers(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                         int32_t n_ref, const int32_t* primer_ref, const int32_t* primer_start, const int32_t* primer_end,
                         int32_t n_primers, int32_t tolerance, uint32_t mode /* bit 0: both ends */,
                         const uint8_t** payload_dev, int64_t* n_bytes_out, const int64_t** rec_off_dev,
                         tc_clip_stats_t* stats, void* stream);

/* ---- SAM text straight from the aligner -> BAM records on the device ----
 * text[0 .. n_bytes): the SAM file (host or device memory); its records begin at first_line_off, which is file line
 * first_line_no (1-based) — the caller has read the '@' header lines and hands over the @SQ names in header order:
 * ref_names holds them concatenated, reference k is ref_names[ref_name_off[k] .. ref_name_off[k+1]).  Only the body travels
 * to the device (large pageable sources through the staging ring).  Every line becomes the BAM record `samtools view -b`
 * would write for it, without `bin` (0) and without optional fields; lines with RNAME '*' are dropped like
 * tc_bam_index_records drops refID -1.  *payload_dev / *rec_off_dev: the placed records and their refID offsets in file
 * order, as tc_bam_index_records leaves them (feed tc_bam_sort_records, tc_bam_records_to_reads, tc_bam_contig_ranges; valid
 * until the next call that decodes a BAM or SAM on this context); *n_payload their bytes; *n_records every record,
 * *n_placed the kept ones; *n_lines the lines of the body.
 * A malformed line (fewer than 11 fields, a number out of range, an unknown RNAME / RNEXT, a bad CIGAR, CIGAR / SEQ or QUAL /
 * SEQ lengths that differ, a QUAL character below '!', an empty line before the last, an '@' line, more than 65535 CIGAR
 * ops, a CG:B placeholder CIGAR): TC_ERR_ARG, the message "line <k>: <reason>" for the first such line; err[0] = k (1-based
 * in the file), err[1] = the reason's code.  t_steps (may be NULL): host seconds of the upload, the line index and the
 * conversion.  Synchronises the stream. */
int  tc_sam_to_bam_records(tc_ctx_t* ctx, const uint8_t* text, int64_t n_bytes, int64_t first_line_off, int64_t first_line_no,
                           int32_t n_ref, const char* ref_names, const int64_t* ref_name_off, const uint8_t** payload_dev,
                           int64_t* n_payload, const int64_t** rec_off_dev, int64_t* n_placed, int64_t* n_records,
                           int64_t* n_lines, int64_t err[2], double* t_steps, void* stream);

/* ---- the BAM file as it lies on disk: inflate and record index on the GPU ----
 * Replaces htslib's bgzf reader and bam_read1 under pysam (reference: indexing.py:6-19 `Readbam`, :96).  The host maps
 * the file and walks the BGZF member headers (tc_host.h: tc_bgzf_map — one header per member); the file's bytes travel as
 * they are, fewer than the payload.
 *
 * tc_bgzf_inflate: every member inflated by one device thread (RFC 1951: stored, fixed and dynamic blocks), its CRC-32
 * checked by one warp; *payload_dev = the uncompressed payload in a context buffer (valid until the next call that
 * decodes a BAM on this context).  TC_ERR_ARG names the first member that does not inflate or fails its CRC, like htslib.
 *
 * tc_bam_index_records: the offsets of the placed records' refID fields (refID >= 0), in file order — what the host reader's
 * sequential hop produces — found in parallel over 64 KiB chunks of the payload and PROVEN by linking every chunk's chain
 * of records to the next chunk's start from the header's end on (bgzf.cu).  `first_record`: payload offset behind the
 * header (the caller parses the header: it needs the reference names anyway); `ref_len`: the header's reference lengths
 * (host or device).  Records are validated as the host reader does (sizes against block_size, NUL-terminated name, the
 * CG-tag placeholder refused): TC_ERR_ARG then; the host reader (tc_bam_payload) names the record.
 * The results feed tc_bam_records_to_reads, which takes device pointers as they are. */
#ifndef TC_BGZF_BLOCK_T
#define TC_BGZF_BLOCK_T
typedef struct tc_bgzf_block { int64_t coff; int32_t csize; int32_t usize; int64_t uoff; } tc_bgzf_block_t;
#endif
int  tc_bgzf_inflate(tc_ctx_t* ctx, const uint8_t* file, int64_t file_bytes, const tc_bgzf_block_t* blocks, int64_t n_blocks,
                     int64_t payload_bytes, const uint8_t** payload_dev, void* stream);
int  tc_bam_index_records(tc_ctx_t* ctx, const uint8_t* payload_dev, int64_t n_bytes, int64_t first_record, int32_t n_ref,
                          const int32_t* ref_len, const int64_t** rec_off_dev, int64_t* n_placed, int64_t* n_records, void* stream);

/* ---- (1) pileup: replaces pysam pileup + parse_query_sequences, indexing.py:100-143 ----
 * counts: int32[TC_NROWS][ref_len] (host or device), fully overwritten, zero rows for uncovered
 * positions (indexing.py:147-151).  Reads starting at or beyond ref_len are an error (TC_ERR_RANGE). */
int  tc_pileup_counts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len,
                      const tc_pileup_params_t* params, int32_t* counts, void* stream);

/* ---- (3) depth: the `coverage` column alone (Coverage.py:1-34 reads it), as a difference
 * array over read spans + inclusive scan.  depth: int32[ref_len].  Only valid for
 * min_base_quality == 0 (every entry of a span counts); otherwise TC_ERR_ARG. */
int  tc_depth(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len,
              const tc_pileup_params_t* params, int32_t* depth, void* stream);

/* ---- (4) per-position call: Sequences.py:119-165 + Ambig.py + Events.py:25-36,85-106 ----
 * counts as produced by tc_pileup_counts (or an overridden index).  Any member of *table may be NULL. */
int  tc_call(tc_ctx_t* ctx, const int32_t* counts, int32_t ref_len,
             const tc_call_params_t* params, const tc_call_table_t* table, void* stream);

/* ---- several references side by side (a segmented genome, a panel of references) ----
 * In a multi-reference pass reference k occupies the global columns [contig_start[k], contig_start[k+1]) of one count table
 * of total_len columns (contig_start: the exclusive prefix sum of the references' lengths, contig_start[n] = total_len).
 * tc_pileup_counts, tc_list_insert_candidates and tc_extract_inserts run over total_len as they are; these three entry
 * points are what such a pass needs besides them (every column of reference k then holds what a pass over reference k
 * alone computes for it).
 *
 * tc_bam_contig_ranges: first_read[n_ref + 1] (host or device) from the records tc_bam_records_to_reads parses (payload and
 * rec_off as it takes them, host or device): the reads of reference k are first_read[k] .. first_read[k+1]-1.  One thread
 * per record reads its refID.  TC_ERR_UNSORTED when the refIDs decrease, TC_ERR_RANGE for a refID outside [0, n_ref).
 * Synchronises the stream. */
int  tc_bam_contig_ranges(tc_ctx_t* ctx, const uint8_t* payload, int64_t n_bytes, const int64_t* rec_off, int64_t n_reads,
                          int32_t n_ref, int32_t* first_read, void* stream);

/* tc_reads_to_contig_coords: moves device-resident reads (tc_reads_upload, tc_bam_records_to_reads) to the global columns
 * IN PLACE: pos += contig_start[k] for the reads of reference k (first_read as above, ref_len[n_ref]: the lengths the
 * pileup of each reference takes, host or device), and mpos likewise when it is >= 0 (-1 and -2 stay).  A mapped read
 * with pos < 0, pos >= ref_len[k] or pos + reference span > ref_len[k] is TC_ERR_RANGE (what tc_pileup_counts over that
 * reference alone says; the message names the read and the reference's index) — the reads before it are moved by then,
 * so the batch must be decoded again.  Unmapped reads (FLAG 0x4, dropped by every pass) are kept inside their
 * reference.  TC_ERR_ARG when the lengths add up to more than INT32_MAX.  contig_start[n_ref + 1] (host or device, may
 * be NULL) receives the boundaries.  Calling it twice on the same arrays moves them twice: the caller keeps track.
 * Synchronises the stream. */
int  tc_reads_to_contig_coords(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t n_ref, const int32_t* ref_len,
                               const int32_t* first_read, int32_t* contig_start, void* stream);

/* tc_call_contigs: tc_call over a count table of total_len columns holding n references (contig_start[n + 1], host or
 * device): every column as tc_call computes it, except that a run of X positions (xrun) never crosses into the next
 * reference and TC_CF_XRUN_OFF_END marks the runs that reach their own reference's end.  tc_call is the case n == 1. */
int  tc_call_contigs(tc_ctx_t* ctx, const int32_t* counts, int32_t total_len, int32_t n, const int32_t* contig_start,
                     const tc_call_params_t* params, const tc_call_table_t* table, void* stream);

/* IsAmbiguous on n independent columns given already-ranked (letter,count) tuples
 * (Ambig.py:179): letters uint8[4][n], cnts int32[4][n], cov int32[n] -> out_char uint8[n] (0 = not ambiguous). */
int  tc_is_ambiguous(tc_ctx_t* ctx, const uint8_t* letters, const int32_t* cnts, const int32_t* cov,
                     int64_t n, double maxdist, uint8_t* out_char, void* stream);

/* ---- (2) insertions: ExtractInserts, Events.py:47-82, for n_cand 1-based positions ----
 * For every candidate the column at pos-1 is piled up under `params` (the pysam defaults of
 * Events.py:66: samtools stepper, min_base_quality 13, max_depth 8000), every entry becomes a
 * fixed-width key (head char, indel, packed inserted bases), keys are counted (shared-memory hash
 * table per column; params->kernel == 2, or a column with thousands of distinct strings: radix sort +
 * run-length encoding) and the most common upper-cased string (ties: first encountered,
 * collections.Counter.most_common) is returned.  calls: [n_cand]; bases: char buffer of
 * bases_cap bytes receiving the inserted characters of each modal string. */
int  tc_extract_inserts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len,
                        const int32_t* cand_pos, int32_t n_cand, const tc_pileup_params_t* params,
                        tc_insert_call_t* calls, uint8_t* bases, int64_t bases_cap, void* stream);

/* Positions (1-based, ascending) with TC_CF_INS_CANDIDATE set; returns their number in *n_out
 * (cand_pos capacity `cap`; TC_ERR_CAPACITY if more). */
int  tc_list_insert_candidates(tc_ctx_t* ctx, const uint8_t* flags, int32_t ref_len,
                               int32_t* cand_pos, int32_t cap, int32_t* n_out, void* stream);

/* ---- one enqueue per sample: (1) -> (4) -> candidates -> (2) chained on the device ----
 * What TrueConsense.py:225-252 runs as separate steps (BuildIndex, then BuildConsensus -> ListInserts -> ExtractInserts),
 * for device-resident reads (tc_reads_upload, QUAL included): tc_pileup_counts (params `pileup`) into counts,
 * tc_call (`call`) into *table, the TC_CF_INS_CANDIDATE positions, and tc_extract_inserts (`inserts`) for exactly those —
 * with no host round trip in between and ONE synchronisation at the end.  counts and every non-NULL member of *table
 * must be device pointers (table->flags is required).  calls[calls_cap] / bases[bases_cap] are host buffers;
 * *n_calls receives the number of candidates (calls[i].pos ascending).  Results and errors are those of the separate
 * calls in that order; inputs the chained form does not take (host arrays, a base-quality filter in `pileup`, more
 * than 256 candidates, ...) run through the separate calls internally. */
int  tc_pileup_call_inserts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* pileup,
                            const tc_call_params_t* call, const tc_pileup_params_t* inserts, int32_t* counts,
                            const tc_call_table_t* table, tc_insert_call_t* calls, int32_t calls_cap, int32_t* n_calls,
                            uint8_t* bases, int64_t bases_cap, void* stream);

/* The same in two halves, so that the host's share of one sample (unpacking the results, preparing the next call) hides
 * behind the device's work on the next: tc_sample_enqueue returns as soon as everything is enqueued, tc_sample_finish
 * waits for that sample only.  At most two samples may be in flight on a context, enqueued on the same stream; the reads,
 * counts and table buffers of a sample must stay valid (and untouched by the caller) until its tc_sample_finish returns. */
int  tc_sample_enqueue(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* pileup,
                       const tc_call_params_t* call, const tc_pileup_params_t* inserts, int32_t* counts,
                       const tc_call_table_t* table, void* stream, int32_t* ticket);
int  tc_sample_finish(tc_ctx_t* ctx, int32_t ticket, tc_insert_call_t* calls, int32_t calls_cap, int32_t* n_calls,
                      uint8_t* bases, int64_t bases_cap);

/* ---- multi-GPU: read-range sharding (ultra-deep single sample) ----
 * Sum the count tables of all ranks in place.  `comm` is an ncclComm_t created by the caller
 * (the Python host layer creates it from a unique id exchanged over torch.distributed). */
int  tc_allreduce_counts(tc_ctx_t* ctx, int32_t* counts_dev, int64_t n_elems, void* comm, void* stream);

/* One rank's part of a read-range sharded sample in ONE enqueue: tc_pileup_counts of this rank's shard into `counts_dev`
 * (device, int32[8][ref_len]) followed by the sum over all ranks, with a single synchronisation at the end instead of one
 * between the pileup and the collective; from the second call with the same buffers on the chain is replayed as a CUDA
 * graph (the NCCL kernel included).  Collective-safe: the shards' status blocks travel with the sum, so when any rank's
 * shard needs another kernel variant or fails, EVERY rank repeats the pass through the separate calls and makes the same
 * collective calls; the failing rank then returns its error.  `params->max_depth` applies to the shard: pass 0 and prove the
 * cap on the summed coverage (host layer: sharding.check_depth_cap).  Results equal tc_pileup_counts + tc_allreduce_counts.
 * Replaces, per shard, the reference's indexing.py:96-143 (BuildIndex over the whole BAM). */
int  tc_pileup_counts_allreduce(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* params,
                                int32_t* counts_dev, void* comm, void* stream);
/* The same in two halves, so that the host's part of pass i (and a caller's reading of its table) hides behind the
 * device's work on pass i + 1: at most two passes in flight on a context, on the same stream, each with its own table;
 * reads and table stay untouched until the pass's finish returns.  Every rank must enqueue and finish in the same order. */
int  tc_pileup_counts_allreduce_enqueue(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* params,
                                        int32_t* counts_dev, void* comm, void* stream, int32_t* ticket);
int  tc_pileup_counts_allreduce_finish(tc_ctx_t* ctx, int32_t ticket);

#ifdef __cplusplus
}
#endif
#endif /* TRUECONSENSE_B200_H */
