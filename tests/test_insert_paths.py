"""ExtractInserts' retry and fallback branches, reached through the public API.  Every case runs on fresh contexts (the
grow-only capacities start small), through the separate call with host and device reads and in both forms, and through
the chained sample; every route must give the oracle's calls."""
import numpy as np
import pytest

from test_gpu_parity import _chained, _oracle_modal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def orc():
    from oracle import pileup

    pileup.build()
    return pileup


def _all_routes(pileup, b, L, positions, mincov=10):
    from trueconsense_b200 import gpu

    exp = [_oracle_modal(pileup, b, int(p)) for p in positions]
    for kernel, on_device in ((0, False), (0, True), (2, False), (2, True)):
        ctx = gpu.Context(0)
        p = gpu.extractinserts_params()
        p.kernel = kernel
        got = ctx._extract_inserts_raw(ctx.upload(b) if on_device else b, L, np.asarray(positions, np.int32), p)
        assert [(g["string"], g["n_entries"]) for g in got] == exp, (kernel, on_device)
    ctx = gpu.Context(0)
    ins = _chained(ctx, b, L, mincov, ctx.upload(b))[4]
    assert len(ins) > 0
    assert [(g["string"], g["n_entries"]) for g in ins] == [_oracle_modal(pileup, b, g["pos"]) for g in ins]
    return exp


def test_insertion_longer_than_the_fixed_bases(orc):
    """More than INS_BASES_FIXED (64) inserted characters: fetched by one more kernel after the calls."""
    rng = np.random.default_rng(11)
    long_a = "".join(rng.choice(list("ACGT"), 80))
    recs = [dict(pos=0, cigar="6M80I6M", seq="ACGTAC" + long_a + "GTACGT") for _ in range(30)]
    recs += [dict(pos=0, cigar="6M70I6M", seq="ACGTAC" + "".join(rng.choice(list("ACGT"), 70)) + "GTACGT") for _ in range(10)]
    from trueconsense_b200.reads import ReadBatch

    exp = _all_routes(orc, ReadBatch.from_records(recs), 40, np.arange(1, 13))
    assert exp[5] == ("C+80" + long_a, 40)


def test_column_deeper_than_the_initial_entry_slots(orc):
    """70,000 reads over one column: more entry slots than the first speculative layout holds (65,536)."""
    from trueconsense_b200.reads import ReadBatch

    recs = [dict(pos=0, cigar="10M3I10M", seq="ACGTACGTAC" + ("TTT" if i % 4 else "GGA") + "ACGTACGTAC") for i in range(70000)]
    exp = _all_routes(orc, ReadBatch.from_records(recs), 40, [5, 10, 15])
    assert exp[1] == ("C+3TTT", 8000)


def test_column_with_more_distinct_strings_than_the_hash_table(orc):
    """5,000 distinct inserted strings in one column: more keys than the count kernel's table holds (4,096)."""
    from trueconsense_b200.reads import ReadBatch

    rng = np.random.default_rng(12)
    codes = rng.choice(4 ** 7, 5000, replace=False)
    recs = []
    for k in codes:
        ins = "".join("ACGT"[(int(k) >> (2 * j)) & 3] for j in range(7))
        recs.append(dict(pos=0, cigar="10M7I10M", seq="ACGTACGTAC" + ins + "ACGTACGTAC"))
    exp = _all_routes(orc, ReadBatch.from_records(recs), 40, [10, 12])
    assert exp[0][1] == 5000


def test_more_candidates_than_a_64_kib_results_block(orc):
    """720 candidate columns: the results the separate call copies back (96 bytes per candidate) outgrow 64 KiB, and the
    chained sample's list outgrows its 256 candidates."""
    from trueconsense_b200.reads import ReadBatch

    rng = np.random.default_rng(14)
    n_sites = 720
    sites = [("".join(rng.choice(list("ACGT"), 2)), ["".join(rng.choice(list("ACGT"), 1 + k % 3)) for _ in range(2)])
             for k in range(n_sites)]
    recs = []
    for i in range(12):
        ins = [v[1] if i % 3 == 0 else v[0] for _, v in sites]
        recs.append(dict(pos=0, cigar="".join(f"2M{len(s)}I" for s in ins) + "2M",
                         seq="".join(m + s for (m, _), s in zip(sites, ins)) + "AC"))
    exp = _all_routes(orc, ReadBatch.from_records(recs), 2 * n_sites + 2, 2 * np.arange(n_sites) + 2)
    assert exp == [(m[1] + f"+{len(v[0])}" + v[0], 12) for m, v in sites]


def test_overlapping_mates_beyond_the_initial_pair_scratch(orc):
    """4,000 overlapping pairs of 1,000-base mates over one column: their rewritten qualities take 8 MB, more than the first
    pair scratch (4 MB)."""
    from trueconsense_b200.reads import ReadBatch

    rng = np.random.default_rng(13)
    tmpl = "".join(rng.choice(list("ACGT"), 1000))
    recs = []
    for i in range(4000):
        for first in (True, False):
            recs.append(dict(pos=0, cigar="500M2I498M", seq=tmpl, qname=f"p{i}", mpos=0, isize=998 if first else -998,
                             flag=(1 | 2 | 32 | 64) if first else (1 | 2 | 16 | 128)))
    _all_routes(orc, ReadBatch.from_records(recs), 1200, [500, 501])
