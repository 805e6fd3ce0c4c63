// sample.cu — one enqueue per sample: pileup -> call -> insertion candidates -> ExtractInserts chained on the device.
//
// The reference runs these as separate Python steps (TrueConsense/TrueConsense.py:225-252: BuildIndex, then
// Sequences.BuildConsensus -> Events.ListInserts -> Events.ExtractInserts), and the separate entry points of this
// library mirror them — each returning host-visible results, i.e. each ending in a synchronisation: the pileup's status
// block, the candidate list, the insertion calls.  On a sample whose pileup takes half a millisecond those three round
// trips were a quarter of the step (VERDICT r1: 0.195 ms of 0.715).  Here nothing is read back in between: the
// candidate list and its length stay on the device, ExtractInserts runs its device-layout driver (D, inserts.cu) for up
// to TC_SAMPLE_MAX_CAND candidates, and ONE block of results comes back — insertion calls, candidate positions, pileup
// status — behind one synchronisation.  Whatever D cannot hold here (more candidates, more entry slots, a column with
// thousands of distinct strings, a pair scratch too small, an insertion of more than 64 characters) goes to
// tc_extract_inserts with the candidate list that came back, and a batch the bit-parallel pileup kernel declines to the
// separate entry points, with identical results.
#include "tc_common.cuh"

constexpr int TC_SAMPLE_MAX_CAND = 256;

bool tc_reads_all_device(const tc_reads_t* r) {
    if (r->n_reads == 0) return true;
    return tc_is_device_ptr(r->pos) && tc_is_device_ptr(r->flag) && tc_is_device_ptr(r->l_seq) && tc_is_device_ptr(r->seq_off) &&
           tc_is_device_ptr(r->cigar_off) && (!r->n_seq_words || (tc_is_device_ptr(r->seq4) && tc_is_device_ptr(r->qual))) &&
           (!r->n_cigar_ops || tc_is_device_ptr(r->cigar)) && (!r->mapq || tc_is_device_ptr(r->mapq));
}

void tc_graph_destroy(tc_graph_cache& g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g.exec = nullptr;
}

int tc_graph_run(tc_ctx* ctx, tc_graph_cache& g, const unsigned char* key, int key_len, bool can_capture,
                 const std::function<int(cudaStream_t)>& chain, cudaStream_t s) {
    const bool same = g.key_len == key_len && memcmp(g.key, key, (size_t)key_len) == 0;
    if (!same) {
        tc_graph_destroy(g);
        memcpy(g.key, key, (size_t)key_len); g.key_len = key_len; g.seen = 0;
    }
    if (same && g.exec) {
        // the same chain with the same buffers again: replay
        TC_CUDA(cudaGraphLaunch(g.exec, s));
        ctx->launches += g.g_launches; ctx->d2h_bytes += g.g_d2h;
        return TC_OK;
    }
    if (!same || g.seen < 1 || !can_capture || getenv("TC_NO_GRAPH")) {
        const int rc = chain(s);
        if (rc) return rc;
        g.seen++;
        return TC_OK;
    }
    // second time: every buffer exists (the eager run allocated them) — capture the chain and launch it as a graph
    if (!ctx->cap_stream) TC_CUDA(cudaStreamCreateWithFlags(&ctx->cap_stream, cudaStreamNonBlocking));
    const int64_t l0 = ctx->launches, d0 = ctx->d2h_bytes, epoch0 = ctx->buf_epoch;
    TC_CUDA(cudaStreamBeginCapture(ctx->cap_stream, cudaStreamCaptureModeRelaxed));
    ctx->in_capture = 1;
    int rc = chain(ctx->cap_stream);
    ctx->in_capture = 0;
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(ctx->cap_stream, &graph);
    if (rc == TC_OK && ce == cudaSuccess && graph && ctx->buf_epoch == epoch0) {
        const cudaError_t ie = cudaGraphInstantiate(&g.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { g.exec = nullptr; return tc_cuda_fail(ctx, ie, "cudaGraphInstantiate"); }
        g.g_launches = ctx->launches - l0; g.g_d2h = ctx->d2h_bytes - d0;
        TC_CUDA(cudaGraphLaunch(g.exec, s));
        return TC_OK;
    }
    // something in the chain could not be captured (or a buffer grew): run it eagerly, try again next time
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    ctx->launches = l0; ctx->d2h_bytes = d0;
    if (rc && rc != TC_ERR_CUDA) return rc;
    g.key_len = 0;
    return chain(s);
}

// the separate entry points in sequence (any input the chained form does not take)
static int sample_unchained(tc_ctx* ctx, const tc_reads_t* reads, int32_t L, const tc_pileup_params_t* pp, const tc_call_params_t* cp,
                            const tc_pileup_params_t* ip, int32_t* counts, const tc_call_table_t* table, bool pileup_done,
                            tc_insert_call_t* calls, int32_t calls_cap, int32_t* n_calls, uint8_t* bases, int64_t bases_cap, void* stream) {
    int rc = pileup_done ? TC_OK : tc_pileup_counts(ctx, reads, L, pp, counts, stream);
    if (rc) return rc;
    rc = tc_call(ctx, counts, L, cp, table, stream);
    if (rc) return rc;
    int32_t* cand = (int32_t*)malloc(4 * (size_t)(calls_cap > 0 ? calls_cap : 1));
    if (!cand) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
    rc = tc_list_insert_candidates(ctx, table->flags, L, cand, calls_cap, n_calls, stream);
    if (rc == TC_OK && *n_calls > 0) rc = tc_extract_inserts(ctx, reads, L, cand, *n_calls, ip, calls, bases, bases_cap, stream);
    free(cand);
    return rc;
}

// SMs the pileup kernel leaves free while the other sample's tail may still be running.  The kernel holds one CTA of 227 KiB
// of shared memory on every SM it gets, so no tail kernel fits beside it: with a full grid the tail of sample i waits for the
// whole pileup of sample i + 1.  With k SMs left to it, the tail runs under that pileup, which takes about
// sm_count / (sm_count - k) times as long.  k from a sweep on one B200 (scripts/overlap_sweep.py, profiles/overlap_sweep.json).
// TC_OVERLAP_SMS overrides it for such measurements; a negative value runs every tail behind its head on the caller's stream.
constexpr int TC_OVERLAP_SMS = 4;

static int overlap_sms() {
    const char* e = getenv("TC_OVERLAP_SMS");
    return e && *e ? atoi(e) : TC_OVERLAP_SMS;
}

static int sample_slots(tc_ctx* ctx) {
    if (ctx->samples) return TC_OK;
    tc_sample_slot* sl = (tc_sample_slot*)calloc(2, sizeof(tc_sample_slot));
    if (!sl) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
    int least = 0, greatest = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&least, &greatest);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaMallocHost(&sl[i].host_block, TC_HOST_SCRATCH);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl[i].done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl[i].head_done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreate(&sl[i].t0);
        if (e == cudaSuccess) e = cudaEventCreate(&sl[i].t1);
        // non-blocking: a caller on the legacy default stream would otherwise serialise the tail with the next head again;
        // the highest priority: the tail's CTAs go to the SMs the next pileup leaves free ahead of anything pending
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&sl[i].tail_stream, cudaStreamNonBlocking, greatest);
    }
    if (e != cudaSuccess) { free(sl); return tc_cuda_fail(ctx, e, "sample slot"); }
    ctx->samples = sl;
    return TC_OK;
}

void tc_sample_slots_free(tc_ctx* ctx) {
    if (!ctx->samples) return;
    for (int i = 0; i < 2; ++i) {
        tc_sample_slot& sl = ctx->samples[i];
        if (sl.tail_stream) { cudaStreamSynchronize(sl.tail_stream); cudaStreamDestroy(sl.tail_stream); }
        if (sl.host_block) cudaFreeHost(sl.host_block);
        if (sl.done) { cudaEventDestroy(sl.done); cudaEventDestroy(sl.head_done); cudaEventDestroy(sl.t0); cudaEventDestroy(sl.t1); }
        tc_graph_destroy(sl.head);
        tc_graph_destroy(sl.tail);
        for (int b = 0; b < SLOT_COUNT; ++b)
            if (sl.bufs[b].p) cudaFree(sl.bufs[b].p);
    }
    free(ctx->samples);
    ctx->samples = nullptr;
    if (ctx->cap_stream) { cudaStreamDestroy(ctx->cap_stream); ctx->cap_stream = nullptr; }
}

// everything the enqueued work depends on: the same key means the same kernels with the same arguments
static int sample_key(const tc_ctx* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* pp, const tc_call_params_t* cp,
                      const tc_pileup_params_t* ip, const int32_t* counts, const tc_call_table_t* table, int grid, unsigned char* key) {
    int n = 0;
    auto put = [&](const void* p, size_t bytes) { memcpy(key + n, p, bytes); n += (int)bytes; };
    put(reads, sizeof(*reads)); put(&ref_len, 4); put(pp, sizeof(*pp)); put(cp, sizeof(*cp)); put(ip, sizeof(*ip));
    put(&counts, sizeof(counts)); put(table, sizeof(*table));
    put(&ctx->buf_epoch, 8); put(&ctx->ins_slot_cap, 8); put(&ctx->pair_cap, 8); put(&ctx->timing, 4); put(&grid, 4);
    return n;
}
static_assert(sizeof(tc_reads_t) + 4 + 2 * sizeof(tc_pileup_params_t) + sizeof(tc_call_params_t) + 8 + sizeof(tc_call_table_t) + 32 <= 512, "sample key");

// head: the pileup and the coverage scan (grid: the pileup kernel's CTAs, 0 for one per SM)
static int sample_head(tc_ctx* ctx, tc_sample_slot& sl, int grid, cudaStream_t s) {
    // timing on: the events around the pileup kernel are this sample's own (two samples may be in flight)
    const cudaEvent_t e0 = ctx->ev0, e1 = ctx->ev1;
    sl.timed = ctx->timing;
    if (ctx->timing) { ctx->ev0 = sl.t0; ctx->ev1 = sl.t1; }
    const int rc = tc_pileup_enqueue(ctx, &sl.reads, sl.ref_len, &sl.pp, sl.counts, s, &sl.pend, 0, grid);
    ctx->ev0 = e0; ctx->ev1 = e1;
    return rc;
}

// tail: everything behind the count table, up to the results block's copy to the host
static int sample_tail(tc_ctx* ctx, tc_sample_slot& sl, cudaStream_t s) {
    int rc = tc_call(ctx, sl.counts, sl.ref_len, &sl.cp, &sl.table, (void*)s);       // device outputs only: enqueues and returns
    if (rc) return rc;
    int32_t *d_ncand, *d_cand;
    rc = tc_candidates_enqueue(ctx, sl.table.flags, sl.ref_len, TC_SAMPLE_MAX_CAND, &d_ncand, &d_cand, s);
    if (rc) return rc;
    return tc_inserts_enqueue_dev(ctx, &sl.reads, d_cand, d_ncand, TC_SAMPLE_MAX_CAND, &sl.ip, sl.pend.d_status, sl.host_block, s, &sl.ipend);
}

// Whether two samples' device outputs (count table, call-table columns) share a byte.  The tail of one and the head (or the
// fallback calls on the caller's stream) of the other then must not overlap.
static bool outputs_overlap(const tc_sample_slot& a, const int32_t* counts, const tc_call_table_t& t, int32_t L) {
    auto ranges = [](const int32_t* c, const tc_call_table_t& u, size_t n, const char** lo, size_t* len) {
        const void* p[7] = {c, u.call_char, u.flags, u.xrun, u.rank_letter, u.rank_count, u.ambig_char};
        const size_t b[7] = {4 * TC_NROWS * n, n, n, 4 * n, 4 * n, 16 * n, n};
        for (int i = 0; i < 7; ++i) { lo[i] = (const char*)p[i]; len[i] = p[i] ? b[i] : 0; }
    };
    const char *alo[7], *blo[7];
    size_t alen[7], blen[7];
    ranges(a.counts, a.table, (size_t)a.ref_len, alo, alen);
    ranges(counts, t, (size_t)L, blo, blen);
    for (int i = 0; i < 7; ++i)
        for (int j = 0; j < 7; ++j)
            if (alen[i] && blen[j] && alo[i] < blo[j] + blen[j] && blo[j] < alo[i] + alen[i]) return true;
    return false;
}

TC_API int tc_sample_enqueue(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* pp,
                             const tc_call_params_t* cp, const tc_pileup_params_t* ip, int32_t* counts, const tc_call_table_t* table,
                             void* stream, int32_t* ticket) {
    if (!ctx) return TC_ERR_ARG;
    if (!reads || !pp || !cp || !ip || !counts || !table || !ticket || ref_len <= 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    if (!tc_is_device_ptr(counts) || !table->flags || !tc_is_device_ptr(table->flags))
        return tc_fail(ctx, TC_ERR_ARG, "the chained sample calls need device pointers for counts and table->flags");
    cudaStream_t s = (cudaStream_t)stream;
    TC_CUDA(cudaSetDevice(ctx->device));
    int rc = sample_slots(ctx);
    if (rc) return rc;
    const int slot = ctx->sample_next;
    tc_sample_slot& sl = ctx->samples[slot];
    const tc_sample_slot& other = ctx->samples[slot ^ 1];
    if (sl.state != 0) return tc_fail(ctx, TC_ERR_ARG, "two samples are in flight on this context already: finish one first");
    // the other sample's tail may still be running beside this sample's work: with shared outputs, everything of this one waits for it
    const bool shares = other.state != 0 && outputs_overlap(other, counts, *table, ref_len);
    if (shares && other.state == 1) TC_CUDA(cudaStreamWaitEvent(s, other.done, 0));
    sl.reads = *reads; sl.ref_len = ref_len; sl.pp = *pp; sl.cp = *cp; sl.ip = *ip; sl.counts = counts; sl.table = *table; sl.stream = stream;
    const tc_call_table_t& t = *table;
    const bool table_dev = (!t.call_char || tc_is_device_ptr(t.call_char)) && (!t.xrun || tc_is_device_ptr(t.xrun)) &&
                           (!t.rank_letter || tc_is_device_ptr(t.rank_letter)) && (!t.rank_count || tc_is_device_ptr(t.rank_count)) &&
                           (!t.ambig_char || tc_is_device_ptr(t.ambig_char));
    if (!tc_reads_all_device(reads) || !table_dev || pp->min_base_quality > 0) {
        sl.state = 2;           // inputs the chained form does not take: the separate calls, at finish time
    } else {
        // The tail goes to the slot's own stream, where it can run under the next sample's pileup, unless the other sample
        // runs its separate calls at finish time (state 2) or shares outputs with this one: then it stays in stream order.
        // This head leaves k SMs to the other sample's tail when that one is on its own stream.
        const int k = overlap_sms();
        const bool side = k >= 0 && !shares && other.state != 2;
        const int grid = other.state == 1 && other.side && side && k > 0 && k < ctx->sm_count ? ctx->sm_count - k : 0;
        unsigned char key[512];
        ctx->bank = sl.bufs;
        int key_len = sample_key(ctx, reads, ref_len, pp, cp, ip, counts, table, grid, key);
        rc = tc_graph_run(ctx, sl.head, key, key_len, true, [&](cudaStream_t cs) { return sample_head(ctx, sl, grid, cs); }, s);
        cudaStream_t ts = s;
        if (rc == TC_OK && side) {
            ts = sl.tail_stream;
            cudaError_t e = cudaEventRecord(sl.head_done, s);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ts, sl.head_done, 0);
            if (e != cudaSuccess) rc = tc_cuda_fail(ctx, e, "tail stream");
        }
        if (rc == TC_OK) {
            key_len = sample_key(ctx, reads, ref_len, pp, cp, ip, counts, table, 0, key);
            rc = tc_graph_run(ctx, sl.tail, key, key_len, true, [&](cudaStream_t cs) { return sample_tail(ctx, sl, cs); }, ts);
        }
        ctx->bank = nullptr;
        if (rc) return rc;
        TC_CUDA(cudaEventRecord(sl.done, ts));
        sl.side = side ? 1 : 0;
        sl.state = 1;
    }
    ctx->sample_next = slot ^ 1;
    *ticket = slot;
    return TC_OK;
}

TC_API int tc_sample_finish(tc_ctx_t* ctx, int32_t ticket, tc_insert_call_t* calls, int32_t calls_cap, int32_t* n_calls,
                            uint8_t* bases, int64_t bases_cap) {
    if (!ctx) return TC_ERR_ARG;
    if (ticket < 0 || ticket > 1 || !ctx->samples || ctx->samples[ticket].state == 0 || !n_calls || (calls_cap > 0 && !calls) || calls_cap < 0)
        return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    TC_CUDA(cudaSetDevice(ctx->device));
    tc_sample_slot& sl = ctx->samples[ticket];
    const int state = sl.state;
    sl.state = 0;
    *n_calls = 0;
    const tc_reads_t* reads = &sl.reads;
    const int32_t ref_len = sl.ref_len;
    if (state == 2)
        return sample_unchained(ctx, reads, ref_len, &sl.pp, &sl.cp, &sl.ip, sl.counts, &sl.table, false, calls, calls_cap, n_calls, bases, bases_cap, sl.stream);
    TC_CUDA(cudaEventSynchronize(sl.done));                          // the one synchronisation of the sample
    ctx->finished_ms = -1.0f;
    if (sl.timed && sl.pend.n_reads > 0 && cudaEventElapsedTime(&ctx->finished_ms, sl.t0, sl.t1) != cudaSuccess) { cudaGetLastError(); ctx->finished_ms = -1.0f; }

    tc_status pst;
    int32_t cands[TC_SAMPLE_MAX_CAND];
    tc_insert_call_t tmp_calls[TC_SAMPLE_MAX_CAND];
    int32_t n = 0; int fit = 0;
    // the pileup's verdict first: its errors win, and a batch the bit-parallel kernel declined is redone from the start
    const int ins_rc = tc_inserts_finish_dev(ctx, &sl.ipend, sl.host_block, &pst, cands, &n, tmp_calls, bases, bases_cap, &fit);
    int redone = 0;
    int rc = tc_pileup_settle(ctx, pst, sl.pend, reads, ref_len, &sl.pp, sl.counts, (cudaStream_t)sl.stream, &redone);
    if (rc) return rc;
    if (redone) return sample_unchained(ctx, reads, ref_len, &sl.pp, &sl.cp, &sl.ip, sl.counts, &sl.table, true, calls, calls_cap, n_calls, bases, bases_cap, sl.stream);
    if (ins_rc) return ins_rc;
    *n_calls = n;
    if (n > calls_cap) return tc_fail(ctx, TC_ERR_CAPACITY, "%d insertion candidates, capacity %d", n, calls_cap);
    if (n == 0) return TC_OK;
    if (fit != 1) {
        // D did not hold it here: the separate call, with the candidate list that came back (or, beyond the chained form's
        // capacity, with a fresh one)
        if (n > TC_SAMPLE_MAX_CAND) {
            int32_t* cand = (int32_t*)malloc(4 * (size_t)n);
            if (!cand) return tc_fail(ctx, TC_ERR_NOMEM, "out of host memory");
            int32_t n2 = 0;
            rc = tc_list_insert_candidates(ctx, sl.table.flags, ref_len, cand, n, &n2, sl.stream);
            if (rc == TC_OK) rc = tc_extract_inserts(ctx, reads, ref_len, cand, n2, &sl.ip, calls, bases, bases_cap, sl.stream);
            free(cand);
            return rc;
        }
        return tc_extract_inserts(ctx, reads, ref_len, cands, n, &sl.ip, calls, bases, bases_cap, sl.stream);
    }
    memcpy(calls, tmp_calls, sizeof(tc_insert_call_t) * (size_t)n);
    return TC_OK;
}

TC_API int tc_pileup_call_inserts(tc_ctx_t* ctx, const tc_reads_t* reads, int32_t ref_len, const tc_pileup_params_t* pp,
                                  const tc_call_params_t* cp, const tc_pileup_params_t* ip, int32_t* counts, const tc_call_table_t* table,
                                  tc_insert_call_t* calls, int32_t calls_cap, int32_t* n_calls, uint8_t* bases, int64_t bases_cap, void* stream) {
    if (!ctx) return TC_ERR_ARG;
    if (!n_calls || (calls_cap > 0 && !calls) || calls_cap < 0) return tc_fail(ctx, TC_ERR_ARG, "bad argument");
    int32_t ticket = -1;
    int rc = tc_sample_enqueue(ctx, reads, ref_len, pp, cp, ip, counts, table, stream, &ticket);
    if (rc) return rc;
    return tc_sample_finish(ctx, ticket, calls, calls_cap, n_calls, bases, bases_cap);
}
