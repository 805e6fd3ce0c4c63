"""Two chained samples in flight on one context (tc_sample_enqueue / tc_sample_finish).  Each sample's tail (call table,
insertion candidates, ExtractInserts) runs on a stream of the context's own, beside the next sample's pileup, with scratch
of its own.  Whatever runs beside what, every sample's count table, call table and insertion calls must equal those of the
separate calls, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TABLE = ("call_char", "flags", "xrun", "rank_letter", "rank_count", "ambig_char")


@pytest.fixture(scope="module")
def lib():
    from trueconsense_b200 import build, gpu

    build.build_host()
    build.build_cuda()
    return gpu


class Sample:
    """A sample's reads in device memory (uploaded through a context of their own, so that they stay valid while other
    samples are uploaded) and the separate calls' results on it."""

    def __init__(self, gpu, batch, L, mincov):
        self.batch, self.L, self.mincov = batch, L, mincov
        self.up = gpu.Context(0)
        self.dev = self.up.upload(batch)
        ref = gpu.Context(0)
        self.counts = ref.pileup_counts(batch, L)
        res = ref.call(self.counts, L, mincov, True)
        self.table = {k: getattr(res, k) for k in TABLE}
        self.ins = ref.extract_inserts(batch, L, ref.list_insert_candidates(res.flags, L))
        ref.close()


class Outputs:
    """One set of device outputs: the count table and every column of the call table."""

    def __init__(self, gpu, L):
        import torch

        self.counts = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
        self.cols = {"call_char": torch.empty(L, dtype=torch.uint8, device="cuda"), "flags": torch.empty(L, dtype=torch.uint8, device="cuda"),
                     "xrun": torch.empty(L, dtype=torch.int32, device="cuda"), "rank_letter": torch.empty((4, L), dtype=torch.uint8, device="cuda"),
                     "rank_count": torch.empty((4, L), dtype=torch.int32, device="cuda"), "ambig_char": torch.empty(L, dtype=torch.uint8, device="cuda")}
        self.table = gpu.CallTable(*[self.cols[k].data_ptr() for k in TABLE])

    def shares(self, other):
        ptrs = lambda o: {o.counts.data_ptr(), *(c.data_ptr() for c in o.cols.values())}
        return bool(ptrs(self) & ptrs(other))

    def check(self, s):
        assert np.array_equal(self.counts.cpu().numpy(), s.counts)
        for k in TABLE:
            assert np.array_equal(self.cols[k].cpu().numpy(), s.table[k]), k


def _synth(gpu, scale, seed):
    from trueconsense_b200 import synth

    w = synth.config(1, scale=scale, seed=seed)
    return Sample(gpu, synth.generate_reads(w.params, w.ref), len(w.ref), w.mincov)


@pytest.fixture(scope="module")
def samples(lib):
    """Three shallow amplicon samples on different seeds, and one the bit-parallel kernel declines (pads: the scatter
    kernel redoes it at finish time)."""
    from oracle import fixtures

    out = {k: _synth(lib, 0.01, seed) for k, seed in (("a", 11), ("b", 12), ("c", 13))}
    out["q"] = Sample(lib, fixtures.quirk_batch(), fixtures.QUIRK_REF_LEN, 2)
    assert all(len(out[k].ins) > 0 for k in "abc")
    return out


@pytest.fixture(scope="module")
def deep(lib):
    """The benchmark's sample (2 M reads, ~25,000x): its candidate columns hold more entries than a new context's
    speculative ExtractInserts layout."""
    return _synth(lib, 1.0, None)


def _run(ctx, seq):
    """Enqueue sample i + 1 before finishing sample i: always two in flight.  seq: (sample, outputs) pairs.  A sample's
    tables are checked when it is finished, unless the next sample writes the same outputs.  Returns, per sample, the
    launches its finish made and tc_last_pileup_kernel_ms after it."""
    def enqueue(k):
        s, o = seq[k]
        return ctx.sample_enqueue(s.dev, s.L, s.mincov, True, o.counts, o.table)

    out = []
    ticket = enqueue(0)
    for i, (s, o) in enumerate(seq):
        nxt = enqueue(i + 1) if i + 1 < len(seq) else None
        l0 = ctx.launches
        assert ctx.sample_finish(ticket) == s.ins, i
        out.append((ctx.launches - l0, ctx.last_pileup_kernel_ms()))
        if nxt is None or not seq[i + 1][1].shares(o):
            o.check(s)
        ticket = nxt
    return out


def _alternating(lib, samples, order):
    """Each position its own outputs: neighbours never share a buffer."""
    sets = {}
    seq = []
    for i, k in enumerate(order):
        s = samples[k]
        key = (s.L, i % 2)
        if key not in sets:
            sets[key] = Outputs(lib, s.L)
        seq.append((s, sets[key]))
    return seq


@pytest.mark.parametrize("overlap", [None, "-1", "16"])
def test_alternating_outputs_equal_separate_calls(lib, samples, monkeypatch, overlap):
    """Different seeds, outputs alternating between two sets, a declined sample (scatter fallback) in flight next to
    accepted ones; with the library's SM reserve, with every tail in stream order, and with a larger reserve."""
    if overlap is not None:
        monkeypatch.setenv("TC_OVERLAP_SMS", overlap)
    ctx = lib.Context(0)
    _run(ctx, _alternating(lib, samples, "abqcaqbcab"))
    ctx.close()


def test_shared_outputs_do_not_overlap(lib, samples):
    """Both samples in flight given the same count table and call table: the second waits for the first, so each one's
    insertion calls are its own, and the last one's tables are what the buffers hold at the end."""
    ctx = lib.Context(0)
    o = Outputs(lib, samples["a"].L)
    _run(ctx, [(samples[k], o) for k in "abcab"])
    # the same count table with different call-table columns share bytes too
    o2 = Outputs(lib, samples["a"].L)
    o2.counts = o.counts
    _run(ctx, [(samples["c"], o), (samples["a"], o2), (samples["b"], o)])
    ctx.close()


def test_layout_grows_while_other_tail_runs(lib, samples, deep):
    """On a new context the deep sample overflows the speculative ExtractInserts layout: its finish reruns the separate call
    and grows the layout while the next sample is in flight, and the next deep sample's enqueue reallocates that slot's
    buffers while the other slot's tail may still be running."""
    ctx = lib.Context(0)
    samples = dict(samples, d=deep)
    launches = [n for n, _ in _run(ctx, _alternating(lib, samples, "adadbd"))]
    assert launches[1] > 0, "the first deep sample fit the initial layout: this test no longer grows it"
    assert launches[3] == 0 and launches[5] == 0
    ctx.close()


def test_timing_reports_each_samples_own_kernel(lib, samples, deep):
    """Timing on: after each finish, tc_last_pileup_kernel_ms is the pileup kernel of the sample just finished, not of the
    one in flight beside it."""
    ctx = lib.Context(0)
    ctx.set_timing(True)
    ms = [m for _, m in _run(ctx, _alternating(lib, dict(samples, d=deep), "adadad"))]
    assert all(m > 0 for m in ms), ms
    shallow, deep_ms = ms[0::2], ms[1::2]
    assert min(deep_ms) > 4 * max(shallow), ms
    ctx.close()


def test_no_graph(lib, samples, monkeypatch):
    """TC_NO_GRAPH=1: heads and tails enqueued eagerly every time, on the same streams."""
    monkeypatch.setenv("TC_NO_GRAPH", "1")
    ctx = lib.Context(0)
    _run(ctx, _alternating(lib, samples, "abqcab"))
    ctx.close()
