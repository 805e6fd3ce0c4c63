"""The pileup's kernel choice and its fallback ladder (tc_pileup_settle), reached through the public API.  Every case runs on
a fresh context, through host and device reads into host and device tables, and each table must equal the oracle's;
tc_depth must equal its coverage row; on the cases that fall back, the chained sample must equal the separate calls.
Each call's kernel launches and bytes copied each way are pinned to what the same calls took before the ladder became
one loop (measured on an NVIDIA B200): a route that runs one more kernel or one more copy fails."""
import copy

import numpy as np
import pytest

from test_gpu_parity import _chained

pytestmark = pytest.mark.gpu

# (launches, host->device bytes, device->host bytes) of every call of a case, in the order _run_case makes them
PINNED = {
    "explicit": [(6, 1387, 3904), (11, 34463627, 6310760), (0, 13223276, 0)],
    "long_bound": [(11, 34463623, 6310760), (11, 34463623, 72), (3, 9757359, 788900), (11, 0, 6310760), (11, 0, 72), (3, 0, 64)],
    "long_nobound": [(17, 68927246, 12621512), (17, 68927246, 136), (3, 9757359, 788900), (17, 0, 12621512), (17, 0, 136), (3, 0, 64), (41, 4, 28412)],
    "long_pad_bound": [(14, 68927254, 12621512), (14, 68927254, 136), (3, 9757363, 788900), (14, 0, 12621512), (14, 0, 136), (3, 0, 64), (36, 4, 28412)],
    "long_pad_nobound": [(20, 103390881, 18932264), (20, 103390881, 200), (3, 9757363, 788900), (20, 0, 18932264), (20, 0, 200), (3, 0, 64), (44, 4, 28476)],
    "quirk_bound": [(6, 2774, 7808), (6, 2774, 128), (3, 775, 544), (6, 0, 7808), (6, 0, 128), (3, 0, 64), (28, 4, 28404)],
    "quirk_nobound": [(9, 2774, 7808), (9, 2774, 128), (3, 775, 544), (9, 0, 7808), (9, 0, 128), (3, 0, 64), (33, 4, 28404)],
    "short_bound": [(3, 13223276, 956960), (3, 13223276, 64), (3, 4809252, 119676), (3, 0, 956960), (3, 0, 64), (3, 0, 64)],
    "short_min_bq": [(1, 29411316, 956960), (1, 29411316, 64), (3, 4809252, 119676), (1, 0, 956960), (1, 0, 64), (3, 0, 64)],
    "short_nobound": [(6, 13223276, 956960), (6, 13223276, 64), (3, 4809252, 119676), (6, 0, 956960), (6, 0, 64), (3, 0, 64)],
}


@pytest.fixture(scope="module")
def orc():
    from oracle import pileup

    pileup.build()
    return pileup


def _with_pad(b):
    """b with a 2-base pad in front of an insertion ("..M 2P nI..") of one read in the middle of the batch: legal, and
    declined by the bit-parallel kernels and the long-read split."""
    for k in range(b.n_reads // 2, b.n_reads):
        c0, c1 = int(b.cigar_off[k]), int(b.cigar_off[k + 1])
        ops = b.cigar[c0:c1] & 15
        at = [j for j in range(1, c1 - c0) if ops[j] == 1 and ops[j - 1] == 0]
        if at:
            break
    out = copy.copy(b)
    out.cigar = np.insert(b.cigar, c0 + at[0], np.uint32((2 << 4) | 6))
    out.cigar_off = b.cigar_off.copy()
    out.cigar_off[k + 1:] += 1
    out.validate()
    return out


def _synth(idx, scale):
    from trueconsense_b200 import synth

    w = synth.config(idx, scale=scale)
    b = synth.generate_reads(w.params, w.ref)
    assert b.max_ref_span > 0
    return b, len(w.ref), w.mincov


def _case(name):
    """(batch, ref_len, mincov, min_base_quality) of a case (CASES: the route the library takes)."""
    from oracle import fixtures

    if name.startswith("short"):
        b, L, mincov = _synth(1, 0.02)
    elif name.startswith("long"):
        b, L, mincov = _synth(4, 0.05)
        assert b.max_ref_span > 5000
    else:
        b, L, mincov = fixtures.quirk_batch(), fixtures.QUIRK_REF_LEN, 2
    if "pad" in name:
        b = _with_pad(b)
    if name.endswith("nobound"):
        b = copy.copy(b)
        b.max_ref_span = -1
    elif b.max_ref_span <= 0:           # the quirk batch comes without a bound
        b.max_ref_span = int(b.ref_spans().max())
    return b, L, mincov, 13 if name == "short_min_bq" else 0


CASES = {
    "short_bound": "3, no span pass",
    "short_nobound": "span pass + 3",
    "short_min_bq": "1",
    "long_bound": "span pass + 4",
    "long_nobound": "span pass + 3 -> 4",
    "quirk_nobound": "span pass + 3 -> 1",
    "quirk_bound": "3 -> 1",
    "long_pad_bound": "4 -> 1",
    "long_pad_nobound": "3 -> 4 -> 1",
}


def _counted(ctx, fn):
    l0, (h0, d0) = ctx.launches, ctx.transfer_bytes()
    out = fn()
    h1, d1 = ctx.transfer_bytes()
    return out, (ctx.launches - l0, h1 - h0, d1 - d0)


def _run_case(pileup, name):
    """Every route of one case on a fresh context; returns each call's counters."""
    import torch

    from trueconsense_b200 import gpu

    b, L, mincov, min_bq = _case(name)
    exp = pileup.pileup_counts(b, L, threads=8, min_base_quality=min_bq)
    cov = exp[0] if min_bq == 0 else pileup.pileup_counts(b, L, threads=8)[0]
    p = gpu.buildindex_params(0)
    p.min_base_quality = min_bq
    ctx = gpu.Context(0)
    counters = []
    for dev_reads in (False, True):
        reads = ctx.upload(b) if dev_reads else b
        for dev_out in (False, True):
            out = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda") if dev_out else None
            got, n = _counted(ctx, lambda: ctx.pileup_counts(reads, L, p, out=out))
            got = got.cpu().numpy() if dev_out else got
            assert np.array_equal(got, exp), (name, dev_reads, dev_out)
            counters.append(n)
        out = torch.empty(L, dtype=torch.int32, device="cuda") if dev_reads else None
        got, n = _counted(ctx, lambda: ctx.depth(reads, L, gpu.buildindex_params(0), out=out))
        assert np.array_equal(got.cpu().numpy() if dev_reads else got, cov), (name, "depth", dev_reads)
        counters.append(n)
    if "->" in CASES[name]:
        counts = ctx.pileup_counts(b, L)
        res = ctx.call(counts, L, mincov, True)
        sep = ctx.extract_inserts(b, L, ctx.list_insert_candidates(res.flags, L))
        dev = ctx.upload(b)
        (c2, f2, _, _, ins), n = _counted(ctx, lambda: _chained(ctx, b, L, mincov, dev))
        assert np.array_equal(c2, counts) and np.array_equal(f2, res.flags) and ins == sep, name
        counters.append(n)
    return counters


@pytest.mark.parametrize("name", sorted(CASES))
def test_pileup_route(orc, name):
    assert _run_case(orc, name) == PINNED[name]


def test_explicit_kernels_decline(orc):
    """An explicit kernel reports what it declines (TC_ERR_CAPACITY) instead of falling back; kernel 2 is no variant of
    tc_pileup_counts (TC_ERR_ARG)."""
    from trueconsense_b200 import gpu

    counters = []
    for name, kernel, code in (("quirk_nobound", 3, -8), ("long_pad_bound", 4, -8), ("short_bound", 2, -2)):
        b, L, _, _ = _case(name)
        ctx = gpu.Context(0)
        with pytest.raises(gpu.TcError) as e:
            ctx.pileup_counts(b, L, gpu.buildindex_params(kernel))
        assert e.value.code == code, (name, kernel)
        counters.append((ctx.launches,) + ctx.transfer_bytes())
    assert counters == PINNED["explicit"]
