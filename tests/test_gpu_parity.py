"""GPU parity tests proper: the CUDA path (through the C-ABI, via ctypes) against the CPU oracle
on the same seeded inputs, against the committed golden vectors generated from the reference,
and through size-independent properties at larger sizes.  Bit-exact everywhere (integer / byte /
index work; the FP64 threshold tests of the call kernel must reproduce CPython's doubles).
"""
import json
import os
from collections import Counter

import numpy as np
import pytest

from conftest import GOLD, load_golden_counts, load_golden_json

pytestmark = pytest.mark.gpu

MINIS = ("quirk", "mini_illumina", "mini_ont", "mini_long", "mini_overlap")
KERNELS = [1, 3, 4]   # pileup kernel variants: 1 scatter (smem atomics), 3 bit-parallel warp streams, 4 pieces of long reads + 3


@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import build, gpu

    build.build_host()
    if not os.path.exists(build.CUDA_LIB):
        build.build_cuda()
    return gpu.Context(0)


@pytest.fixture(scope="module")
def orc():
    from oracle import call, pileup

    pileup.build()
    return pileup, call


def _pileup(ctx, b, L, kernel):
    """tc_pileup_counts with an explicit kernel variant.  The bit-parallel variants decline inputs they cannot
    stage (reads spanning more than their windows) with TC_ERR_CAPACITY; the library's own choice
    (kernel=0) must then transparently use the scatter kernel."""
    from trueconsense_b200 import gpu

    try:
        return ctx.pileup_counts(b, L, gpu.buildindex_params(kernel))
    except gpu.TcError as e:
        if kernel in (3, 4) and e.code == -8:
            return ctx.pileup_counts(b, L, gpu.buildindex_params(0))
        raise


def _mini_batch(name):
    from trueconsense_b200 import bamio

    return bamio.read_bam(f"{GOLD}/{name}.bam")


# ---------------------------------------------------------------------------- (1) pileup
@pytest.mark.parametrize("name", MINIS)
@pytest.mark.parametrize("kernel", KERNELS)
def test_pileup_golden_and_oracle(ctx, orc, name, kernel):
    from trueconsense_b200 import gpu

    pileup, _ = orc
    b = _mini_batch(name)
    exp = load_golden_counts(name)
    L = exp.shape[1]
    got = _pileup(ctx, b, L, kernel)
    assert np.array_equal(got[:7], exp), "GPU count table differs from the reference-generated golden table"
    assert np.array_equal(got, pileup.pileup_counts(b, L))
    assert not got[7].any()


@pytest.mark.parametrize("kernel", KERNELS)
def test_pileup_quirk_batch_direct(ctx, orc, kernel):
    from oracle import fixtures
    from trueconsense_b200 import gpu

    pileup, _ = orc
    b = fixtures.quirk_batch()
    got = _pileup(ctx, b, fixtures.QUIRK_REF_LEN, kernel)
    assert np.array_equal(got, pileup.pileup_counts(b, fixtures.QUIRK_REF_LEN))


@pytest.mark.parametrize("kernel", [3])
def test_pileup_warp_kernel_takes_plain_quirks_itself(ctx, orc, kernel):
    """Variant 3 declines only pads and zero-length ops (TC_ERR_CAPACITY -> scatter kernel).  Everything else of
    the quirk set — SEQ '*', IUPAC codes, leading deletions, D/N/I adjacencies, clips, flags — it must take itself
    (explicit kernel, no fallback), bit-exact with the oracle."""
    from oracle import fixtures
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    recs = [r for r in fixtures.quirk_records() if "P" not in r["cigar"]]
    assert any(r["seq"] == "*" for r in recs)
    b = ReadBatch.from_records(recs)
    got = ctx.pileup_counts(b, fixtures.QUIRK_REF_LEN, gpu.buildindex_params(kernel))
    assert np.array_equal(got, pileup.pileup_counts(b, fixtures.QUIRK_REF_LEN))
    # ... and with pads present it declines, while the library's own choice falls back transparently
    with pytest.raises(gpu.TcError) as e:
        ctx.pileup_counts(fixtures.quirk_batch(), fixtures.QUIRK_REF_LEN, gpu.buildindex_params(kernel))
    assert e.value.code == -8


def test_pileup_ops_longer_than_16_bits(ctx, orc):
    """Variant 3 stages CIGAR ops as 16 bits (length < 4096).  Longer hard clips count for nothing, a longer soft
    clip is fine at the end of a read; in front of aligned bases it is declined (explicit kernel=3) and the
    library's own choice (kernel=0) still answers bit-exactly."""
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    rng = np.random.default_rng(5)
    L = 400
    seq = lambda n: "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    ok = [dict(pos=5, cigar="5000H20M2I10M", seq=seq(32)), dict(pos=6, cigar="20M1D10M70000H", seq=seq(30)),
          dict(pos=7, cigar="30M4500S", seq=seq(4530)), dict(pos=7, cigar="4096H10M2D5M3S4096H", seq=seq(18), flag=16),
          dict(pos=9, cigar="40M", seq=seq(40))]
    b = ReadBatch.from_records(ok)
    exp = pileup.pileup_counts(b, L)
    assert np.array_equal(ctx.pileup_counts(b, L, gpu.buildindex_params(3)), exp)
    assert np.array_equal(ctx.pileup_counts(b, L, gpu.buildindex_params(0)), exp)
    lead = ok + [dict(pos=12, cigar="4200S30M", seq=seq(4230))]
    b2 = ReadBatch.from_records(lead)
    exp2 = pileup.pileup_counts(b2, L)
    with pytest.raises(gpu.TcError) as e:
        ctx.pileup_counts(b2, L, gpu.buildindex_params(3))
    assert e.value.code == -8
    assert np.array_equal(ctx.pileup_counts(b2, L, gpu.buildindex_params(0)), exp2)

@pytest.mark.parametrize("kernel", [3])
@pytest.mark.parametrize("span,seed", [(390, 1), (390, 2), (200, 3), (880, 4), (880, 5)])
def test_pileup_phase_boundaries_fuzz(ctx, orc, span, seed, kernel):
    """Variant 3 walks a window in phases of 256 columns.  Reads that all start within a few columns of each other
    (one window) with random CIGARs — match ops, deletions and reference skips that end on, start on or straddle
    the phase borders, insertions and clips anywhere — must give the oracle's table, without falling back."""
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    rng = np.random.default_rng(1000 + seed)
    L = 3000
    base = 1000                      # the window starts here: phase borders at base + 256, + 512, + 768
    recs = []
    for i in range(1500):
        pos = base + int(rng.integers(0, 24))
        x, ops, qlen = pos, [], 0
        if rng.random() < 0.2:
            l = int(rng.integers(1, 12)); ops.append(("S", l)); qlen += l
        target = pos + span + int(rng.integers(-20, 20))
        while x < target:
            # steer some ops to end exactly on (or one off) a phase border
            border = base + 256 * (1 + (x - base) // 256)
            l = int(rng.integers(1, 60))
            if rng.random() < 0.35 and border - x < 80:
                l = border - x + int(rng.integers(-1, 2))
            l = max(1, min(l, target - x + 2))
            ops.append(("M", l)); x += l; qlen += l
            u = rng.random()
            if u < 0.35:
                l = int(rng.integers(1, 4)); ops.append(("I", l)); qlen += l
            elif u < 0.7:
                l = int(rng.integers(1, 30)) if rng.random() < 0.2 and x + 30 < target else int(rng.integers(1, 3)); ops.append(("D", l)); x += l
            elif u < 0.75 and x + 40 < target:
                l = int(rng.integers(1, 40)); ops.append(("N", l)); x += l
            elif u < 0.8:
                li, ld = int(rng.integers(1, 3)), int(rng.integers(1, 3))
                ops += [("D", ld), ("I", li)] if rng.random() < 0.5 else [("I", li), ("D", ld)]
                x += ld; qlen += li
        if ops[-1][0] != "M":
            ops.append(("M", 3)); qlen += 3
        if rng.random() < 0.2:
            l = int(rng.integers(1, 12)); ops.append(("S", l)); qlen += l
        # merge equal neighbours (M M after a dropped op cannot happen here, but keep the CIGAR canonical)
        cig = "".join(f"{l}{o}" for o, l in ops)
        seq = "".join("ACGTN"[j] for j in rng.choice(5, qlen, p=[0.245, 0.245, 0.245, 0.245, 0.02]))
        recs.append(dict(pos=pos, cigar=cig, seq=seq, flag=16 if rng.random() < 0.5 else 0))
    recs.sort(key=lambda r: r["pos"])
    b = ReadBatch.from_records(recs)
    exp = pileup.pileup_counts(b, L, threads=4)
    got = ctx.pileup_counts(b, L, gpu.buildindex_params(kernel))
    assert np.array_equal(got, exp)
    b.max_ref_span = int(max(sum(int(l) for l, o in __import__("re").findall(r"(\d+)([MDN])", r["cigar"])) for r in recs))
    got2 = ctx.pileup_counts(b, L, gpu.buildindex_params(kernel))
    assert np.array_equal(got2, exp)


SYNTH_CASES = {
    "shotgun_indels": dict(n_reads=6000, read_len=120, read_len_jitter=30, indel_rate=0.03, indel_maxlen=3, softclip_rate=0.2,
                           softclip_max=12, n_rate=0.01, iupac_rate=0.01, refskip_rate=0.05, special_flag_rate=0.05, sub_rate=0.02),
    "paired": dict(n_reads=8000, read_len=150, paired=True, softclip_rate=0.05, softclip_max=10, special_flag_rate=0.05),
    "amplicon_deep": dict(n_reads=30000, read_len=400, read_len_jitter=20, n_amplicons=3, amplicon_jitter=2, indel_rate=1 / 30,
                          softclip_rate=0.05, softclip_max=20, n_rate=0.001),
    "long_reads": dict(n_reads=400, read_len=3000, read_len_jitter=800, indel_rate=1 / 40, indel_maxlen=2, softclip_rate=0.2,
                       softclip_max=60),
    "mid_reads": dict(n_reads=3000, read_len=700, read_len_jitter=100, indel_rate=1 / 40, indel_maxlen=3, softclip_rate=0.2,
                      softclip_max=30, n_rate=0.002),
    "tiny": dict(n_reads=3, read_len=50),
    "one_read": dict(n_reads=1, read_len=10),
}


def _synth(case, L=5000, seed=7):
    from trueconsense_b200 import synth

    ref, feats = synth.make_genome(L, seed, "sars2")
    a = feats[0]["start"] - 1
    V = synth.Variant
    vs = [V(a + 50, synth.VAR_INS, 3, 5, 0.9), V(a + 120, synth.VAR_INS, 7, 6, 0.7), V(a + 200, synth.VAR_DEL, 3, 0, 0.8),
          V(a + 260, synth.VAR_DEL, 1, 0, 0.2), V(a + 330, synth.VAR_INS, 1, 9, 0.56), V(a + 400, synth.VAR_SUB, 1, 4, 0.5)]
    p = synth.SynthParams(seed=seed, ref_len=L, variants=vs, **SYNTH_CASES[case])
    return ref, feats, synth.generate_reads(p, ref)


@pytest.mark.parametrize("case", list(SYNTH_CASES))
@pytest.mark.parametrize("kernel", KERNELS)
def test_pileup_synthetic_vs_oracle(ctx, orc, case, kernel):
    from trueconsense_b200 import gpu

    pileup, _ = orc
    ref, _, b = _synth(case)
    got = _pileup(ctx, b, len(ref), kernel)
    exp = pileup.pileup_counts(b, len(ref), threads=4)
    assert np.array_equal(got, exp)
    # size-independent properties
    assert got[0].sum() == b.count_aligned_bases(0x4)
    assert np.all(got[1:6].sum(axis=0) <= got[0])


def test_pileup_empty_and_device_io(ctx):
    import torch

    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    empty = ReadBatch.from_records([])
    got = ctx.pileup_counts(empty, 100)
    assert got.shape == (8, 100) and not got.any()
    ref, _, b = _synth("paired")
    host = ctx.pileup_counts(b, len(ref))
    dev_reads = ctx.upload(b)
    out = torch.empty((8, len(ref)), dtype=torch.int32, device="cuda")
    ctx.pileup_counts(dev_reads, len(ref), out=out)
    assert np.array_equal(out.cpu().numpy(), host)


def test_pileup_min_base_quality(ctx, orc):
    from trueconsense_b200 import gpu

    pileup, _ = orc
    ref, _, b = _synth("shotgun_indels")
    p = gpu.buildindex_params(1)
    p.min_base_quality = 13
    got = ctx.pileup_counts(b, len(ref), p)
    exp = pileup.pileup_counts(b, len(ref), min_base_quality=13)
    assert np.array_equal(got, exp)


def test_pileup_samtools_stepper_filters(ctx, orc):
    from trueconsense_b200 import gpu

    pileup, _ = orc
    ref, _, b = _synth("paired")
    p = gpu.PileupParams(flag_filter=0x704, min_mapq=10, min_base_quality=0, ignore_orphans=1, max_depth=10_000_000, kernel=0)
    got = ctx.pileup_counts(b, len(ref), p)
    exp = pileup.pileup_counts(b, len(ref), flag_filter=0x704, min_mapq=10, ignore_orphans=1)
    assert np.array_equal(got, exp)
    assert got[0].sum() < b.count_aligned_bases(0x4)


def test_pileup_errors(ctx):
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    unsorted = ReadBatch.from_records([dict(pos=50, cigar="10M", seq="A" * 10), dict(pos=10, cigar="10M", seq="A" * 10)])
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(unsorted, 100)
    assert ei.value.code == -3
    beyond = ReadBatch.from_records([dict(pos=95, cigar="10M", seq="A" * 10)])
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(beyond, 100)
    assert ei.value.code == -7
    ok = ReadBatch.from_records([dict(pos=90, cigar="10M", seq="A" * 10)])
    p = gpu.buildindex_params()
    p.max_depth = 2
    many = ReadBatch.from_records([dict(pos=5, cigar="10M", seq="A" * 10)] * 5)
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(many, 100, p)
    assert ei.value.code == -4
    assert ctx.pileup_counts(ok, 100)[0, 90:].tolist() == [1] * 10


# ---------------------------------------------------------------------------- (3) depth
@pytest.mark.parametrize("case", ["shotgun_indels", "paired", "amplicon_deep"])
def test_depth_equals_coverage_row(ctx, case):
    ref, _, b = _synth(case)
    counts = ctx.pileup_counts(b, len(ref))
    depth = ctx.depth(b, len(ref))
    assert np.array_equal(depth, counts[0])


# ---------------------------------------------------------------------------- (4) call
def test_call_vs_oracle_random_tables(ctx, orc):
    from oracle import fixtures

    _, call = orc
    rng = np.random.default_rng(11)
    for it in range(40):
        L = int(rng.integers(1, 400))
        depth = int(rng.choice([10, 40, 100, 1000]))
        counts = np.zeros((8, L), np.int64)
        counts[:] = fixtures.random_counts(rng, L, depth)
        mincov = int(rng.choice([0, 1, 5, 10, 30]))
        amb = bool(it & 1)
        exp = call.call_table(counts, mincov, amb)
        got = ctx.call(counts.astype(np.int32), L, mincov, amb)
        for k in ("call_char", "flags", "xrun", "rank_letter", "rank_count", "ambig_char"):
            assert np.array_equal(getattr(got, k), exp[k]), (k, it)


def test_call_long_xruns(ctx, orc):
    """X-runs crossing the per-thread chunks of the reverse scan, and runs reaching the end."""
    _, call = orc
    rng = np.random.default_rng(3)
    for L in (1, 2, 1023, 1024, 1025, 5000, 30011):
        counts = np.zeros((8, L), np.int64)
        counts[0] = 50
        counts[1] = 50
        x = rng.random(L) < 0.97
        if L > 10:
            x[L // 2] = False
        counts[1, x] = 0
        counts[5, x] = 50
        exp = call.call_table(counts, 10, True)
        got = ctx.call(counts.astype(np.int32), L, 10, True)
        assert np.array_equal(got.xrun, exp["xrun"]), L
        assert np.array_equal(got.flags, exp["flags"]), L


def test_is_ambiguous_kat(ctx):
    kat = load_golden_json("kat.json")["is_ambiguous"]
    cases = [c for c in kat if c["status"] == "ok"]
    letters = np.array([[ord(c["ranks"][k][0]) for c in cases] for k in range(4)], dtype=np.uint8)
    counts = np.array([[c["ranks"][k][1] for c in cases] for k in range(4)], dtype=np.int32)
    cov = np.array([c["cov"] for c in cases], dtype=np.int32)
    got = ctx.is_ambiguous(letters, counts, cov)
    for g, c in zip(got, cases):
        exp = c["result"]
        assert (bool(g), chr(g) if g else None) == (exp[0], exp[1]), c


def test_ieee_thresholds_on_device(ctx):
    """SURVEY.md §4.3: (55/100)*100 = 55.00000000000001; integer math gets these wrong."""
    c = np.zeros((8, 4), np.int32)
    c[0] = [100, 10, 100, 100]
    c[1] = [55, 6, 85, 100]          # A
    c[3] = [45, 5, 0, 0]             # C
    c[5] = [0, 0, 15, 0]             # X
    c[6] = [0, 0, 0, 55]             # I
    got = ctx.call(c, 4, 1, True)
    assert got.ambig_char[0] == 0 and chr(got.ambig_char[1]) == "M"
    assert got.flags[2] & 0x04          # 15 % deletions -> minority deletion
    assert got.flags[3] & 0x08          # (55/100)*100 > 55 -> insertion candidate


# ---------------------------------------------------------------------------- (2) insertions
def _oracle_modal(pileup, b, pos1):
    cols = pileup.pileup_columns(b, region=(pos1 - 1, pos1), **pileup.EXTRACTINSERTS)
    if not cols or cols[0][1] == "":
        return None, 0
    strings = [s.upper() for s in cols[0][1]]
    top = next(iter(dict(Counter(strings).most_common())))
    return top, len(strings)


@pytest.mark.parametrize("name", MINIS)
def test_extract_inserts_golden_batches(ctx, orc, name):
    pileup, call = orc
    b = _mini_batch(name)
    L = load_golden_counts(name).shape[1]
    rng = np.random.default_rng(1)
    cands = call.insert_candidates(np.vstack([load_golden_counts(name), np.zeros((1, L), np.int32)]).astype(np.int64), 1)
    positions = sorted(set(cands[:40]) | set(int(x) for x in rng.integers(1, L + 1, 25)) | {1, L})
    got = ctx.extract_inserts(b, L, positions)
    for g in got:
        exp, n = _oracle_modal(pileup, b, g["pos"])
        assert g["string"] == exp, g
        assert g["n_entries"] == n


def test_extract_inserts_depth_cap_binds(ctx, orc):
    """> 8000 reads over the candidate columns: the cap keeps the first 8000 fetched reads plus the
    first read of every later start coordinate (htslib bam_plp_push)."""
    pileup, _ = orc
    ref, _, b = _synth("amplicon_deep")
    L = len(ref)
    counts = ctx.pileup_counts(b, L)
    assert counts[0].max() > 9000
    table = ctx.call(counts, L, 30, True)
    cands = ctx.list_insert_candidates(table.flags, L)
    assert len(cands) >= 2
    deep = [int(p) for p in np.argsort(counts[0])[-5:] + 1]
    positions = sorted(set(int(c) for c in cands) | set(deep))
    got = ctx.extract_inserts(b, L, positions)
    for g in got:
        exp, n = _oracle_modal(pileup, b, g["pos"])
        assert (g["string"], g["n_entries"]) == (exp, n), g
    assert max(g["n_entries"] for g in got) <= 8000 + 400


def test_extract_inserts_ties_and_quality(ctx, orc):
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    S = "ACGTACGTACGTACGTACGT"
    recs = [
        dict(pos=0, cigar="5M1I5M", seq="ACGTA" + "T" + "CGTAC"),
        dict(pos=0, cigar="5M1I5M", seq="ACGTA" + "G" + "CGTAC"),
        dict(pos=0, cigar="5M1I5M", seq="ACGTA" + "G" + "CGTAC", flag=16),
        dict(pos=0, cigar="5M1I5M", seq="ACGTA" + "T" + "CGTAC"),
        dict(pos=0, cigar="5M2D5M", seq=S[:10]),
        dict(pos=0, cigar="10M", seq=S[:10], qual=5),                    # filtered by min_base_quality 13
        dict(pos=1, cigar="10M", seq=S[:10], flag=0x400),                # duplicate: dropped by the stepper
        dict(pos=1, cigar="10M", seq=S[:10], flag=1),                    # orphan
        dict(pos=2, cigar="3M4N3M", seq=S[:6]),
        dict(pos=12, cigar="4M", seq="AC=N"),
    ]
    b = ReadBatch.from_records(recs)
    got = ctx.extract_inserts(b, 40, list(range(1, 18)))
    for g in got:
        exp, n = _oracle_modal(pileup, b, g["pos"])
        assert (g["string"], g["n_entries"]) == (exp, n), g
    assert got[4]["string"] == "A+1T"      # tie between +1T and +1G: first encountered wins


# ---------------------------------------------------------------------------- public API vs golden
@pytest.mark.parametrize("name", MINIS)
def test_api_buildindex_listinserts_consensus_golden(ctx, name):
    from trueconsense_b200 import Coverage, Events, Sequences, indexing

    meta = load_golden_json(f"{name}.json")
    bam, fa, gff = (f"{GOLD}/{name}.{e}" for e in ("bam", "fasta", "gff"))
    df = indexing.BuildIndex(bam, fa)
    assert list(df.columns) == ["coverage", "A", "T", "C", "G", "X", "I"]
    assert df.index[0] == 1 and df.index.name is None and str(df.index.dtype) == "int64"
    assert all(str(t) == "int64" for t in df.dtypes)
    exp = load_golden_counts(name)
    assert np.array_equal(np.stack([df[c].to_numpy() for c in df.columns]), exp)
    index = df.to_dict("index")
    handle = indexing.Readbam(bam)
    has, pos = Events.ListInserts(index, meta["mincov"], handle)
    assert [has, None if pos is None else {str(k): v for k, v in pos.items()}] == meta["list_inserts"]
    assert np.array_equal(Coverage.DepthFromBam(handle), exp[0])
    gdf = indexing.Gffindex(gff).df
    gdf["seqid"] = name
    gdict = gdf.to_dict("index")
    for amb in (True, False):
        for inc in (True, False):
            e = meta[f"consensus_amb{int(amb)}_ins{int(inc)}"]
            if e["status"] == "raise":
                with pytest.raises(Exception) as ei:
                    Sequences.BuildConsensus(meta["mincov"], df.to_dict("index"), gdict, amb, handle, inc)
                assert type(ei.value).__name__ == e["exc"]
            else:
                cons, newgff = Sequences.BuildConsensus(meta["mincov"], df.to_dict("index"), gdict, amb, handle, inc)
                assert cons == e["consensus"]
                assert {str(k): [v["start"], v["end"]] for k, v in newgff.items()} == e["gff"]


def test_walk_cases_golden(ctx, orc):
    """The GPU call table + host walk against the reference's BuildConsensus on 600 random cases
    (consensus, corrected GFF, or the exception type)."""
    from trueconsense_b200 import Sequences

    _, call = orc
    cases = load_golden_json("walk_cases.json")
    for c in cases:
        counts = np.zeros((8, c["L"]), dtype=np.int64)
        counts[:7] = np.array(c["counts"], dtype=np.int64)
        gff = {int(k): v for k, v in c["gff"].items()}
        cols = {int(k): v for k, v in c["columns"].items()}
        inserts = call.list_inserts(counts, c["mincov"], lambda p: cols.get(p - 1))
        for inc in (True, False):
            exp = c[f"ins{int(inc)}"]
            if exp["status"] == "raise":
                with pytest.raises(Exception) as ei:
                    Sequences.consensus_from_inserts(c["mincov"], counts, gff, c["include_ambig"], inserts, inc)
                assert type(ei.value).__name__ == exp["exc"], c
            else:
                cons, newgff = Sequences.consensus_from_inserts(c["mincov"], counts, gff, c["include_ambig"], inserts, inc)
                assert cons == exp["consensus"]
                assert {str(k): [v["start"], v["end"]] for k, v in newgff.items()} == exp["gff"]


def test_scalar_api_kat(ctx):
    from trueconsense_b200 import Ambig, Events, Sequences

    kat = load_golden_json("kat.json")
    for case in kat["ranking"]:
        got = [list(Sequences.GetNucleotide({1: case["col"]}, 1, k)) for k in range(1, 6)]
        assert got == case["ranks"]
    for case in kat["minority_del"]:
        idx = {1: dict(coverage=case["cov"], A=0, T=0, C=0, G=0, X=case["X"], I=0)}
        if case["status"] == "raise":
            with pytest.raises(ZeroDivisionError):
                Events.MinorityDel(idx, 1)
        else:
            assert Events.MinorityDel(idx, 1) == case["result"]
    assert Ambig.IsAmbiguous(("A", 55), ("C", 45), ("T", 0), ("G", 0), 100) == (False, None)
    assert Ambig.IsAmbiguous(("A", 6), ("C", 5), ("T", 0), ("G", 0), 10) == (True, "M")
    assert Ambig.IsAmbiguous(("A", 33), ("C", 33), ("G", 33), ("T", 0), 99) == (True, "V")


# ---------------------------------------------------------------------------- larger sizes: properties
def test_config2_slice_properties(ctx, orc):
    """BASELINE configs[1] at 2 % (40k ONT reads, 16 M aligned bases): exact against the
    multi-threaded oracle, plus the invariants that hold at any size."""
    from trueconsense_b200 import gpu, synth

    pileup, _ = orc
    w = synth.config(1, scale=0.02)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    g1 = ctx.pileup_counts(b, L, gpu.buildindex_params(1))
    for k in KERNELS[1:]:
        assert np.array_equal(g1, ctx.pileup_counts(b, L, gpu.buildindex_params(k)))
    assert np.array_equal(g1, pileup.pileup_counts(b, L, threads=8))
    assert g1[0].sum() == b.count_aligned_bases(0x4) == b.aligned_bases
    assert np.array_equal(ctx.depth(b, L), g1[0])
    # read-range sharding is additive (what the multi-GPU allreduce relies on)
    half = b.n_reads // 2
    parts = ctx.pileup_counts(b.slice(0, half), L).astype(np.int64) + ctx.pileup_counts(b.slice(half, b.n_reads), L)
    assert np.array_equal(parts, g1)


def test_extract_inserts_partial_staging_equals_full_upload(ctx):
    """Host SEQ / QUAL / CIGAR are staged only over the candidate columns; same answers as with everything on
    the device, for host batches and for device reads that carry a host QUAL array."""
    ref, _, b = _synth("amplicon_deep")
    L = len(ref)
    counts = ctx.pileup_counts(b, L)
    cands = [int(c) for c in ctx.list_insert_candidates(ctx.call(counts, L, 30, True).flags, L)]
    positions = sorted(set(cands) | {1, 700, 701, 2500, L})
    full = ctx.extract_inserts(ctx.upload(b), L, positions)             # everything resident, QUAL included
    x0 = ctx.transfer_bytes()[0]
    host = ctx.extract_inserts(b, L, positions)                          # all host pointers
    x1 = ctx.transfer_bytes()[0]
    dev = ctx.upload(b, with_qual=False)
    x2 = ctx.transfer_bytes()[0]
    mixed = ctx.extract_inserts(dev.with_host_qual(), L, positions)      # device arrays + host QUAL
    x3 = ctx.transfer_bytes()[0]
    assert host == full and mixed == full
    assert x3 - x2 <= b.qual.nbytes + 4096            # nothing but QUAL stretches (and a few integers) travelled
    assert x1 - x0 < b.qual.nbytes + b.seq4.nbytes + b.cigar.nbytes + 64 * b.n_reads
    with pytest.raises(RuntimeError):
        ctx.pileup_counts(b, L)                 # stages host arrays through the context's buffers ...
        ctx.pileup_counts(dev, L)               # ... so the earlier upload is stale


# ---------------------------------------------------------------------------- CLI end to end
@pytest.mark.parametrize("name", ["quirk"] + list(MINIS))
def test_cli_outputs_equal_reference_cli(ctx, name, tmp_path, monkeypatch):
    """main() writes the files the reference's CLI wrote for the same BAM / FASTA / GFF
    (tests/golden/cli_*, generated by oracle/make_golden.py from the unmodified reference)."""
    import json

    from trueconsense_b200 import TrueConsense

    status = json.load(open(f"{GOLD}/cli_{name}.status.json"))
    meta = load_golden_json(f"{name}.json")
    out = str(tmp_path / f"cli_{name}")
    argv = ["--input", f"{GOLD}/{name}.bam", "--reference", f"{GOLD}/{name}.fasta", "--features", f"{GOLD}/{name}.gff",
            "--coverage-level", str(meta["mincov"]), "--samplename", name, "--output", out + ".fasta",
            "--variants", out + ".vcf", "--output-gff", out + ".gff", "--depth-of-coverage", out + ".cov.tsv", "--threads", "2"]
    monkeypatch.setattr("sys.argv", ["TrueConsense", "<golden>"])
    if status["status"] == "raise":
        with pytest.raises(Exception) as ei:
            TrueConsense.main(argv)
        assert type(ei.value).__name__ == status["exc"]
    else:
        TrueConsense.main(argv)
    for ext in ("fasta", "gff", "cov.tsv", "vcf"):
        gold = f"{GOLD}/cli_{name}.{ext}"
        if not os.path.exists(gold):
            assert not os.path.exists(f"{out}.{ext}"), ext
            continue
        got = open(f"{out}.{ext}").read()
        if ext == "vcf":
            got = "".join("##fileDate=<date>\n" if l.startswith("##fileDate=") else l for l in got.splitlines(keepends=True))
            got = got.replace(GOLD + os.sep, "")
        assert got == open(gold).read(), ext


def test_extract_inserts_sorted_form_equals_hash_form(ctx):
    """The shared-memory hash count and the radix sort + run-length form give the same calls."""
    from trueconsense_b200 import gpu

    ref, _, b = _synth("amplicon_deep")
    L = len(ref)
    counts = ctx.pileup_counts(b, L)
    cands = [int(c) for c in ctx.list_insert_candidates(ctx.call(counts, L, 30, True).flags, L)]
    positions = np.asarray(sorted(set(cands) | {1, 350, 700, 701, 1200, 2500, L}), np.int32)
    p_hash = gpu.extractinserts_params()
    p_sort = gpu.extractinserts_params()
    p_sort.kernel = 2
    a = ctx._extract_inserts_raw(b, L, positions, p_hash)
    s_ = ctx._extract_inserts_raw(b, L, positions, p_sort)
    assert a == s_
    assert any(x["n_entries"] > 0 for x in a)


def test_span_bound_hint(ctx, orc):
    """tc_reads_t.max_ref_span: with a bound the span pass is folded into the pileup kernel; same table, same
    errors; a bound that is too small is rejected."""
    import copy

    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    for case in ("amplicon_deep", "paired", "shotgun_indels", "mid_reads"):
        ref, _, b = _synth(case)
        assert b.max_ref_span > 0
        nb = copy.copy(b)
        nb.max_ref_span = -1
        with_hint = _pileup(ctx, b, len(ref), 3)
        without = _pileup(ctx, nb, len(ref), 3)
        assert np.array_equal(with_hint, without)
        assert np.array_equal(with_hint, pileup.pileup_counts(b, len(ref), threads=4))
        assert np.array_equal(ctx.depth(b, len(ref)), with_hint[0])
    ref, _, b = _synth("paired")
    small = copy.copy(b)
    small.max_ref_span = 20
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(small, len(ref))
    assert ei.value.code == -2
    # tc_extract_inserts does not trust a bound tc_pileup_counts has not verified for these arrays: a bound that is too small
    # would silently narrow the range of reads fetched for a column
    ref, _, amp = _synth("amplicon_deep")
    counts = ctx.pileup_counts(amp, len(ref))
    cands = ctx.list_insert_candidates(ctx.call(counts, len(ref), 10, True).flags, len(ref))
    assert len(cands) > 0
    good = ctx.extract_inserts(amp, len(ref), cands)
    lying = copy.copy(amp)
    lying.max_ref_span = 20
    assert ctx.extract_inserts(lying, len(ref), cands) == good
    # the checks the span pass used to make
    unsorted = ReadBatch.from_records([dict(pos=50, cigar="10M", seq="A" * 10), dict(pos=10, cigar="10M", seq="A" * 10)])
    unsorted.max_ref_span = 10
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(unsorted, 100)
    assert ei.value.code == -3
    beyond = ReadBatch.from_records([dict(pos=95, cigar="10M", seq="A" * 10)])
    beyond.max_ref_span = 10
    with pytest.raises(gpu.TcError) as ei:
        ctx.pileup_counts(beyond, 100)
    assert ei.value.code == -7
    zero = ReadBatch.from_records([dict(pos=5, cigar="4S", seq="ACGT"), dict(pos=7, cigar="10M", seq="A" * 10)])
    zero.max_ref_span = 10
    assert ctx.pileup_counts(zero, 100)[0, 7:17].tolist() == [1] * 10


def test_extract_inserts_long_insertions_both_forms(ctx, orc):
    """Insertions longer than 8 bases use hashed keys (verified entry by entry); '=' bases print strand marks."""
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    rng = np.random.default_rng(5)
    ins_a, ins_b = "ACGTACGTACGT", "ACGTACGTACGA"
    recs = []
    for i in range(60):
        ins = ins_a if i % 3 else ins_b
        recs.append(dict(pos=0, cigar="6M12I6M", seq="ACGTAC" + ins + "GTACGT", flag=16 if i % 5 == 0 else 0))
    for i in range(25):
        n = int(rng.integers(9, 20))
        recs.append(dict(pos=0, cigar=f"6M{n}I6M", seq="ACGTAC" + "".join(rng.choice(list("ACGT"), n)) + "GTACGT"))
    recs += [dict(pos=0, cigar="6M3I6M", seq="ACGTAC" + "A=A" + "GTACGT"), dict(pos=0, cigar="6M3I6M", seq="ACGTAC" + "A=A" + "GTACGT", flag=16),
             dict(pos=0, cigar="6M3I6M", seq="ACGTAC" + "A=A" + "GTACGT", flag=16), dict(pos=2, cigar="4M9D4M", seq="ACGTACGT")]
    b = ReadBatch.from_records(recs)
    positions = np.arange(1, 16, dtype=np.int32)
    for kernel in (0, 2):
        p = gpu.extractinserts_params()
        p.kernel = kernel
        got = ctx._extract_inserts_raw(b, 40, positions, p)
        for g in got:
            exp, n = _oracle_modal(pileup, b, g["pos"])
            assert (g["string"], g["n_entries"]) == (exp, n), (kernel, g)
    assert got[5]["string"] == "C+12" + ins_a


def test_compact_cigar_transport(ctx, orc):
    """tc_reads_t.cigar16: the CIGARs travel as 16-bit entries and are widened on the device — same tables, same insertion
    calls, half the CIGAR bytes over the link; a batch with an operation of 4096 or more keeps the 32-bit array."""
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    for case in ("amplicon_deep", "shotgun_indels", "tiny", "one_read"):
        ref, _, b = _synth(case)
        L = len(ref)
        c = b.with_cigar16()
        assert c.cigar16 is not None and c.cigar16.dtype == np.uint16 and np.array_equal(c.cigar16, b.cigar)
        exp = pileup.pileup_counts(b, L, threads=4)
        x0 = ctx.transfer_bytes()[0]
        assert np.array_equal(ctx.pileup_counts(c, L), exp)
        x1 = ctx.transfer_bytes()[0]
        assert np.array_equal(ctx.pileup_counts(b, L), exp)
        x2 = ctx.transfer_bytes()[0]
        assert (x2 - x1) - (x1 - x0) == 2 * b.cigar.size
        dev = ctx.upload(c)
        assert np.array_equal(ctx.download(dev.struct.cigar, b.cigar.size, np.uint32), b.cigar)
        assert np.array_equal(ctx.pileup_counts(dev, L), exp)
        cands = ctx.list_insert_candidates(ctx.call(exp, L, 10, True).flags, L)
        if len(cands):
            assert ctx.extract_inserts(c, L, cands) == ctx.extract_inserts(b, L, cands)
            assert ctx.extract_inserts(ctx.upload(c), L, cands) == ctx.extract_inserts(b, L, cands)
    long_op = ReadBatch.from_records([dict(pos=0, cigar="5000M", seq="A" * 5000)])
    assert long_op.with_cigar16() is long_op


def test_compact_seq_transport(ctx, orc):
    """tc_reads_t.seq2: SEQ travels at two bits per base plus the list of words that hold anything else than A C G T, and seq4
    is rebuilt on the device bit for bit (N / IUPAC / '=' codes, zero padding of every read's last word, reads without SEQ);
    same tables and insertion calls; half the SEQ bytes over the link."""
    from trueconsense_b200.reads import ReadBatch

    pileup, _ = orc
    for case in ("amplicon_deep", "shotgun_indels", "paired", "tiny", "one_read"):
        ref, _, b = _synth(case)
        L = len(ref)
        c = b.with_seq2(max_exception_fraction=1.0).with_cigar16()     # (shotgun_indels: N and IUPAC codes in a fifth of the words)
        assert c.seq2 is not None and c.seq2.dtype == np.uint16 and c.seq2.shape == b.seq4.shape
        dev = ctx.upload(c)
        assert np.array_equal(ctx.download(dev.struct.seq4, b.seq4.size, np.uint32), b.seq4), case
        exp = pileup.pileup_counts(b, L, threads=4)
        assert np.array_equal(ctx.pileup_counts(dev, L), exp)
        x0 = ctx.transfer_bytes()[0]
        assert np.array_equal(ctx.pileup_counts(b.with_seq2(max_exception_fraction=1.0), L), exp)
        x1 = ctx.transfer_bytes()[0]
        assert np.array_equal(ctx.pileup_counts(b, L), exp)
        x2 = ctx.transfer_bytes()[0]
        assert (x2 - x1) - (x1 - x0) == 2 * b.seq4.size - 8 * c.seq_exc_idx.size
        cands = ctx.list_insert_candidates(ctx.call(exp, L, 10, True).flags, L)
        if len(cands):
            assert ctx.extract_inserts(c, L, cands) == ctx.extract_inserts(b, L, cands)
            assert ctx.extract_inserts(ctx.upload(c), L, cands) == ctx.extract_inserts(b, L, cands)
    # every code, odd lengths, a read without SEQ, '=' bases
    recs = [dict(pos=3, cigar="16M", seq="=ACMGRSVTWYHKDBN"), dict(pos=4, cigar="5M", seq="ACGTN"), dict(pos=5, cigar="9M", seq="ACGTACGTA"),
            dict(pos=6, cigar="7M", seq="*"), dict(pos=7, cigar="1M", seq="T"), dict(pos=8, cigar="8M", seq="GGGGGGGG"),
            dict(pos=9, cigar="17M", seq="ACGTACGTACGTACGT=")]
    odd = ReadBatch.from_records(recs)
    c = odd.with_seq2(max_exception_fraction=1.0)
    assert c.seq2 is not None and c.seq_exc_idx.size >= 3
    assert np.array_equal(ctx.download(ctx.upload(c).struct.seq4, odd.seq4.size, np.uint32), odd.seq4)
    assert np.array_equal(ctx.pileup_counts(c, 40), pileup.pileup_counts(odd, 40))
    assert odd.with_seq2(max_exception_fraction=0.01) is odd          # too many exceptions: the 4-bit words travel


# ---------------------------------------------------------------------------- multi-GPU pieces on one device
def test_read_range_sharding_single_rank_and_emulated_ranks(ctx, orc):
    """tc_allreduce_counts through a real NCCL communicator (one rank: identity), and the per-rank slices of
    sharding.read_range summed on one device equal the full table."""
    import torch

    from trueconsense_b200 import sharding

    pileup, _ = orc
    ref, _, b = _synth("amplicon_deep")
    L = len(ref)
    exp = pileup.pileup_counts(b, L, threads=4)
    comm = sharding.NcclComm(0, 1, 0)
    try:
        out = sharding.pileup_counts_read_range(ctx, b, L, 0, 1, comm)
        ctx.allreduce_counts(out, comm)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), exp)
    finally:
        comm.close()
    # the shard's pileup and the sum in one enqueue (tc_pileup_counts_allreduce): eager, captured, replayed; a shard the
    # bit-parallel kernel declines sends every rank through the separate calls; a failing shard still makes its collective call
    import copy

    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    comm = sharding.NcclComm(0, 1, 0)
    try:
        p = gpu.buildindex_params()
        p.max_depth = 0
        dev = ctx.upload(b, with_qual=False)
        out = torch.empty((8, L), dtype=torch.int32, device="cuda")
        for i in range(4):
            out.fill_(-1)
            ctx.pileup_counts_allreduce(dev, L, p, out, comm)
            assert np.array_equal(out.cpu().numpy(), exp), i
        # two passes in flight, a table each, finished in order; a third is refused
        out_b = torch.empty_like(out)
        t0 = ctx.pileup_counts_allreduce_enqueue(dev, L, p, out, comm)
        for i in range(5):
            t1 = ctx.pileup_counts_allreduce_enqueue(dev, L, p, out if i % 2 else out_b, comm)
            ctx.pileup_counts_allreduce_finish(t0)
            assert np.array_equal((out_b if i % 2 else out).cpu().numpy(), exp), i
            t0 = t1
        t1 = ctx.pileup_counts_allreduce_enqueue(dev, L, p, out, comm)
        with pytest.raises(gpu.TcError):
            ctx.pileup_counts_allreduce_enqueue(dev, L, p, out, comm)
        ctx.pileup_counts_allreduce_finish(t0)
        ctx.pileup_counts_allreduce_finish(t1)
        assert np.array_equal(out.cpu().numpy(), exp) and np.array_equal(out_b.cpu().numpy(), exp)
        ctx.pileup_counts_allreduce(b, L, p, out, comm)                 # host arrays: staged, never captured
        assert np.array_equal(out.cpu().numpy(), exp)
        ref2, _, long_b = _synth("long_reads")
        unbounded = copy.copy(long_b)
        unbounded.max_ref_span = -1
        exp2 = pileup.pileup_counts(long_b, len(ref2), threads=4)
        out2 = torch.empty((8, len(ref2)), dtype=torch.int32, device="cuda")
        dev2 = ctx.upload(unbounded, with_qual=False)
        for i in range(3):
            ctx.pileup_counts_allreduce(dev2, len(ref2), p, out2, comm)
            assert np.array_equal(out2.cpu().numpy(), exp2), i
        unsorted = ReadBatch.from_records([dict(pos=50, cigar="10M", seq="A" * 10), dict(pos=10, cigar="10M", seq="A" * 10)])
        with pytest.raises(gpu.TcError) as ei:
            ctx.pileup_counts_allreduce(unsorted, L, p, out, comm)
        assert ei.value.code == -3
        ctx.pileup_counts_allreduce(ctx.upload(b, with_qual=False), L, p, out, comm)
        assert np.array_equal(out.cpu().numpy(), exp)
    finally:
        comm.close()
    total = torch.zeros((8, L), dtype=torch.int32, device="cuda")
    for rank in range(3):
        lo, hi = sharding.read_range(b.n_reads, rank, 3)
        part = torch.empty_like(total)
        ctx.pileup_counts(b.slice(lo, hi), L, out=part)
        total += part
    assert np.array_equal(total.cpu().numpy(), exp)


# ---------------------------------------------------------------------------- BASELINE.json's five configs
FIVE = [(0, 1.0), (1, 0.1), (2, 0.2), (3, 0.005), (4, 0.1)]


@pytest.mark.parametrize("idx,scale", FIVE)
def test_five_configs_hot_path_vs_oracle(ctx, orc, idx, scale):
    """Each of BASELINE.json's configs at a size the oracle finishes in seconds: count table, call table,
    insertion candidates and insertion calls bit for bit; then the host walk runs over the GPU's table."""
    from trueconsense_b200 import Sequences, synth

    pileup, call = orc
    w = synth.config(idx, scale=scale)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    exp = pileup.pileup_counts(b, L, threads=8)
    got = ctx.pileup_counts(b, L)
    assert np.array_equal(got, exp)
    assert got[0].sum() == b.count_aligned_bases(0x4)
    table = ctx.call(got, L, w.mincov, True)
    ref = call.call_table(exp.astype(np.int64), w.mincov, True)
    for k in ("call_char", "flags", "xrun", "ambig_char"):
        assert np.array_equal(getattr(table, k), ref[k]), k
    cands = [int(c) for c in ctx.list_insert_candidates(table.flags, L)]
    assert cands == call.insert_candidates(exp.astype(np.int64), w.mincov)
    positions = sorted(set(cands) | {1, L // 3, L // 2, L})
    calls = ctx.extract_inserts(b, L, positions)
    inserts = {}
    for g in calls:
        s_exp, n = _oracle_modal(pileup, b, g["pos"])
        assert (g["string"], g["n_entries"]) == (s_exp, n), g
        bases, size = call.extract_insert([s_exp] if s_exp else "")
        if g["pos"] in cands and bases is not None:
            inserts[g["pos"]] = {size: bases}
    gff = synth.gff_dict(w.feats)
    if idx == 4:
        return      # the walk over 197 kb x 114 features is the host's business (tests/test_host_cpu.py covers its logic)
    cons, newgff = Sequences.consensus_from_inserts(w.mincov, got, gff, True, (True, inserts) if inserts else (False, None), True)
    assert len(cons) >= L - 64 and set(cons) <= set("ACGTNacgtn-MRWSYKVHDB")
    assert set(newgff) == set(gff)


def test_long_reads_take_the_pieces_path(ctx, orc):
    """Reads spanning thousands of columns are cut into pieces and go through the SWAR kernel (variant 4) — no
    fallback to the scatter kernel — with and without a span bound; BASELINE config 5 shape."""
    import copy

    from trueconsense_b200 import gpu, synth

    pileup, _ = orc
    w = synth.config(4, scale=0.05)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    assert b.max_ref_span > 5000
    exp = pileup.pileup_counts(b, L, threads=8)
    assert np.array_equal(ctx.pileup_counts(b, L, gpu.buildindex_params(4)), exp)      # explicit: raises instead of falling back
    nb = copy.copy(b)
    nb.max_ref_span = -1
    l0 = ctx.launches
    assert np.array_equal(ctx.pileup_counts(nb, L), exp)                                # no bound: 3 declines, 4 takes over
    assert ctx.launches - l0 < 40
    ref, _, s = _synth("long_reads")
    assert np.array_equal(ctx.pileup_counts(s, len(ref), gpu.buildindex_params(4)), pileup.pileup_counts(s, len(ref), threads=4))


def _chained(ctx, b, L, mincov, dev_reads, pileup=None):
    import torch

    from trueconsense_b200 import gpu

    counts = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
    flags = torch.empty(L, dtype=torch.uint8, device="cuda")
    cc = torch.empty(L, dtype=torch.uint8, device="cuda")
    xrun = torch.empty(L, dtype=torch.int32, device="cuda")
    table = gpu.CallTable(cc.data_ptr(), flags.data_ptr(), xrun.data_ptr(), None, None, None)
    ins = ctx.pileup_call_inserts(dev_reads, L, mincov, True, counts, table, pileup=pileup)
    torch.cuda.synchronize()
    return counts.cpu().numpy(), flags.cpu().numpy(), cc.cpu().numpy(), xrun.cpu().numpy(), ins


@pytest.mark.parametrize("name", MINIS)
def test_chained_sample_equals_separate_calls(ctx, orc, name):
    """tc_pileup_call_inserts (one enqueue, one synchronisation per sample) == tc_pileup_counts -> tc_call ->
    tc_list_insert_candidates -> tc_extract_inserts, for device-resident reads and — through its internal fallback —
    for host arrays; both == the oracle's table."""
    pileup, _ = orc
    b = _mini_batch(name)
    exp = load_golden_counts(name)
    L = exp.shape[1]
    mincov = 10
    counts = ctx.pileup_counts(b, L)
    res = ctx.call(counts, L, mincov, True)
    cands = ctx.list_insert_candidates(res.flags, L)
    sep = ctx.extract_inserts(b, L, cands)
    for reads in (ctx.upload(b), b):
        c2, f2, cc2, x2, ins = _chained(ctx, b, L, mincov, reads)
        assert np.array_equal(c2, counts) and np.array_equal(c2[:7], exp)
        assert np.array_equal(f2, res.flags) and np.array_equal(cc2, res.call_char) and np.array_equal(x2, res.xrun)
        assert ins == sep
        assert [d["pos"] for d in ins] == list(cands)


def test_chained_sample_config2_slice_and_fallbacks(ctx, orc):
    """The chained form on a deep amplicon sample (insertion candidates present, the 8000-read depth cap binding), on a
    batch the bit-parallel kernel declines (pads -> scatter kernel), and its error reporting."""
    from oracle import fixtures
    from trueconsense_b200 import gpu, synth

    pileup, call = orc
    w = synth.config(1, scale=0.02)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    counts = ctx.pileup_counts(b, L)
    assert np.array_equal(counts, pileup.pileup_counts(b, L, threads=8))
    res = ctx.call(counts, L, w.mincov, True)
    cands = ctx.list_insert_candidates(res.flags, L)
    assert len(cands) > 0
    sep = ctx.extract_inserts(b, L, cands)
    l0 = ctx.launches
    c2, f2, _, _, ins = _chained(ctx, b, L, w.mincov, ctx.upload(b))
    assert ctx.launches - l0 <= 16              # nothing ran twice
    assert np.array_equal(c2, counts) and np.array_equal(f2, res.flags) and ins == sep
    # pads: variant 3 declines, the chained form redoes the sample through the separate calls
    q = fixtures.quirk_batch()
    Lq = fixtures.QUIRK_REF_LEN
    cq = ctx.pileup_counts(q, Lq)
    rq = ctx.call(cq, Lq, 2, True)
    sq = ctx.extract_inserts(q, Lq, ctx.list_insert_candidates(rq.flags, Lq))
    c3, f3, _, _, ins3 = _chained(ctx, q, Lq, 2, ctx.upload(q))
    assert np.array_equal(c3, cq) and np.array_equal(f3, rq.flags) and ins3 == sq
    # errors of the pileup surface from the chained call as they do from tc_pileup_counts
    from trueconsense_b200.reads import ReadBatch

    unsorted = ReadBatch.from_records([dict(pos=50, cigar="10M", seq="A" * 10), dict(pos=10, cigar="10M", seq="A" * 10)])
    with pytest.raises(gpu.TcError) as ei:
        _chained(ctx, unsorted, 100, 2, ctx.upload(unsorted))
    assert ei.value.code == -3


def test_two_samples_in_flight(ctx, orc):
    """tc_sample_enqueue / tc_sample_finish: two samples in flight on one stream give what they give one at a time; a third
    enqueue is refused."""
    import torch

    from trueconsense_b200 import gpu, synth

    w = synth.config(1, scale=0.01)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    dev = ctx.upload(b)
    ref_counts, ref_flags, _, _, ref_ins = _chained(ctx, b, L, w.mincov, dev)
    bufs = []
    for _ in range(2):
        counts = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
        flags = torch.empty(L, dtype=torch.uint8, device="cuda")
        xrun = torch.empty(L, dtype=torch.int32, device="cuda")
        bufs.append((counts, flags, gpu.CallTable(None, flags.data_ptr(), xrun.data_ptr(), None, None, None), xrun))
    t0 = ctx.sample_enqueue(dev, L, w.mincov, True, bufs[0][0], bufs[0][2])
    t1 = ctx.sample_enqueue(dev, L, w.mincov, True, bufs[1][0], bufs[1][2])
    with pytest.raises(gpu.TcError):
        ctx.sample_enqueue(dev, L, w.mincov, True, bufs[0][0], bufs[0][2])
    for t, (counts, flags, _, _) in zip((t0, t1), bufs):
        assert ctx.sample_finish(t) == ref_ins
        assert np.array_equal(counts.cpu().numpy(), ref_counts) and np.array_equal(flags.cpu().numpy(), ref_flags)
    for i in range(5):          # steady state: enqueue i + 1, finish i
        t = ctx.sample_enqueue(dev, L, w.mincov, True, bufs[i % 2][0], bufs[i % 2][2])
        assert ctx.sample_finish(t) == ref_ins


# ---------------------------------------------------------------------------- mate overlaps (htslib tweak_overlap_quality)
def _column_strings(g):
    return g["string"], g["n_entries"], g["mode_count"]


def _expected_call(pileup, call, b, pos1, **params):
    kw = dict(pileup.EXTRACTINSERTS)
    kw.update(params)
    cols = pileup.pileup_columns(b, region=(pos1 - 1, pos1), **kw)
    strings = cols[0][1] if cols else ""
    up = [s.upper() for s in strings] if strings else []
    if not up:
        return None, 0, 0
    cnt = Counter(up)
    best = max(cnt.values())
    first = next(s for s in up if cnt[s] == best)
    return first, len(up), best


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_mate_overlap_rewrite_kat(ctx, orc, mode):
    """The hand-derived cases of oracle/fixtures.overlap_kat_records through tc_extract_inserts: the column holds exactly the
    entries htslib's mate-overlap quality rewriting leaves (count and mode), in all three modes of the rewrite, for host
    arrays (ranges staged) and device-resident reads."""
    from oracle import fixtures
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, call = orc
    recs, exp = fixtures.overlap_kat_records()
    b = ReadBatch.from_records(recs)
    L = fixtures.OVERLAP_REF_LEN
    pos1 = fixtures.OVERLAP_COL + 1
    p = gpu.extractinserts_params()
    p.reserved = mode << 8
    want = _expected_call(pileup, call, b, pos1, reserved=mode << 8)
    if mode == 0:
        assert want[1] == len(exp)          # ... which the CPU suite has checked against the hand-derived list
    for make in (lambda: b, lambda: ctx.upload(b)):
        got = ctx.extract_inserts(make(), L, [pos1], p)[0]
        assert (got["string"], got["n_entries"], got["mode_count"]) == want


def _paired_fuzz_records(rng, n_pairs, L, col):
    """Proper pairs (and a few triples: a supplementary alignment shares the QNAME) whose mates mostly both cover `col`, with
    random indels / clips / reference skips around it, random qualities near the threshold of 13 and a good share of
    disagreeing bases."""
    recs = []

    def alignment(pos, span_target):
        ops, x, q = [], pos, 0
        if rng.random() < 0.2:
            l = int(rng.integers(1, 6)); ops.append(("S", l)); q += l
        while x < pos + span_target:
            l = int(rng.integers(1, 25)); ops.append(("M", l)); x += l; q += l
            u = rng.random()
            if u < 0.25:
                l = int(rng.integers(1, 4)); ops.append(("I", l)); q += l
            elif u < 0.5:
                l = int(rng.integers(1, 6)); ops.append(("D", l)); x += l
            elif u < 0.55:
                l = int(rng.integers(1, 8)); ops.append(("N", l)); x += l
            elif u < 0.6:
                ops += [("D", 1), ("I", 1)]; x += 1; q += 1
        if ops[-1][0] != "M":
            ops.append(("M", 2)); x += 2; q += 2
        return "".join(f"{l}{o}" for o, l in ops), q, x

    for i in range(n_pairs):
        pa = col - int(rng.integers(5, 60))
        pb = pa + int(rng.integers(0, 40))
        ca, qa, ea = alignment(pa, int(rng.integers(40, 90)))
        cb, qb, eb = alignment(pb, int(rng.integers(40, 90)))
        name = f"p{i}"
        proper = rng.random() < 0.9
        fa = 1 | (2 if proper else 0) | 0x40 | (0x20 if rng.random() < 0.5 else 0)
        fb = 1 | (2 if proper else 0) | 0x80 | (0x10 if rng.random() < 0.5 else 0)
        mk = lambda n: "".join("ACGT"[j] for j in rng.choice(4, n, p=[0.7, 0.1, 0.1, 0.1]))
        mq = lambda n: [int(v) for v in rng.choice([2, 7, 8, 12, 13, 14, 16, 17, 20, 30, 40], n)]
        isz = eb - pa
        if rng.random() < 0.1:
            isz = 1000                              # "no overlap possible, unless some wild cigar"
        mpa, mpb = pb, pa
        if rng.random() < 0.05:
            mpa = -1
        recs.append(dict(pos=pa, cigar=ca, seq=mk(qa), qual=mq(qa), flag=fa, qname=name, mpos=mpa, isize=isz))
        recs.append(dict(pos=pb, cigar=cb, seq=mk(qb), qual=mq(qb), flag=fb, qname=name, mpos=mpb, isize=-isz))
        if rng.random() < 0.08:                     # a supplementary alignment of mate a (same name, passes the stepper's filter)
            pc = pa + int(rng.integers(0, 30))
            cc, qc, _ = alignment(pc, 50)
            recs.append(dict(pos=pc, cigar=cc, seq=mk(qc), qual=mq(qc), flag=fa | 0x800, qname=name, mpos=mpa, isize=isz))
    recs.sort(key=lambda r: r["pos"])
    return recs


@pytest.mark.parametrize("seed,max_depth", [(1, 8000), (2, 8000), (3, 60), (4, 25)])
def test_mate_overlap_rewrite_fuzz(ctx, orc, seed, max_depth):
    """Random overlapping pairs around several columns, with the depth cap binding in two of the cases (a capped mate makes
    htslib forget the stored one): tc_extract_inserts == the oracle's column (entries, modal string, its count) in every mode."""
    from trueconsense_b200 import gpu
    from trueconsense_b200.reads import ReadBatch

    pileup, call = orc
    rng = np.random.default_rng(300 + seed)
    L = 400
    col = 200
    b = ReadBatch.from_records(_paired_fuzz_records(rng, 150, L, col))
    positions = [col - 3, col, col + 1, col + 2, col + 9, col + 17]
    for mode in (0, 1, 2):
        p = gpu.extractinserts_params()
        p.reserved = mode << 8
        p.max_depth = max_depth
        got = ctx.extract_inserts(b, L, positions, p)
        for g in got:
            want = _expected_call(pileup, call, b, g["pos"], reserved=mode << 8, max_depth=max_depth)
            assert (g["string"], g["n_entries"], g["mode_count"]) == want, (mode, g["pos"])
        p.kernel = 2            # the sorted form counts the same keys
        assert [(_column_strings(g)) for g in ctx.extract_inserts(b, L, positions, p)] == [(_column_strings(g)) for g in got]


def test_config1_full_size_insertion_inside_mate_overlap(ctx, orc):
    """BASELINE configs[0] at full size (25 k overlapping 2x150 pairs): count table == oracle, and every insertion candidate's
    ExtractInserts call == the oracle's column under the mate-overlap rewrite — including an insertion placed where most
    pairs overlap."""
    from trueconsense_b200 import gpu, synth

    pileup, call = orc
    w = synth.config(0, scale=1.0)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    counts = ctx.pileup_counts(b, L)
    assert np.array_equal(counts, pileup.pileup_counts(b, L, threads=8))
    res = ctx.call(counts, L, w.mincov, True)
    cands = ctx.list_insert_candidates(res.flags, L)
    assert list(cands) == call.insert_candidates(counts.astype(np.int64), w.mincov) and len(cands) > 0
    got = ctx.extract_inserts(b, L, cands)
    n_diff = 0
    for g in got:
        want = _expected_call(pileup, call, b, g["pos"])
        assert (g["string"], g["n_entries"], g["mode_count"]) == want, g["pos"]
        n_diff += want[1] != _expected_call(pileup, call, b, g["pos"], reserved=1 << 8)[1]
    assert n_diff > 0           # the rewrite does change these columns


# ---------------------------------------------------------------------------- benchmark sizes
@pytest.mark.parametrize("idx,scale", [(1, 1.0), (3, 0.1), (4, 1.0)])
def test_full_size_configs_vs_oracle(ctx, orc, idx, scale):
    """BASELINE configs[1] (2 M ONT-like reads: the benchmarked sample), configs[3] at 5 M reads and configs[4] (98.5 k reads
    of 10 kb) at FULL size: the count table equals the multi-threaded oracle's bit for bit; for configs[1] also the chained
    sample call — every insertion candidate (depth 25,000: the 8000-read cap drops two thirds of each column) against the
    oracle's column."""
    import os

    from trueconsense_b200 import synth

    pileup, call = orc
    w = synth.config(idx, scale=scale)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    exp = pileup.pileup_counts(b, L, threads=os.cpu_count() or 8)
    if idx != 1:
        assert np.array_equal(ctx.pileup_counts(b, L), exp)
        return
    counts, flags, _, _, ins = _chained(ctx, b, L, w.mincov, ctx.upload(b))
    assert np.array_equal(counts, exp)
    cands = call.insert_candidates(exp.astype(np.int64), w.mincov)
    assert [g["pos"] for g in ins] == cands and len(cands) >= 3
    for g in ins:
        assert (g["string"], g["n_entries"], g["mode_count"]) == _expected_call(pileup, call, b, g["pos"]), g["pos"]


# ---------------------------------------------------------------------------- BAM records parsed on the device
@pytest.mark.parametrize("name", MINIS)
def test_bam_records_parsed_on_device_equal_host_decode(ctx, name):
    """tc_bam_records_to_reads (inflate + record hop on the host, everything else on the GPU) fills exactly the arrays
    csrc/host/bamio.c's reader fills: every array byte for byte, the statistics, and the count table / insertion calls on top."""
    from trueconsense_b200 import bamio

    path = f"{GOLD}/{name}.bam"
    host = bamio.read_bam(path)
    payload = bamio.read_bam_payload(path)
    assert payload.n_reads == host.n_reads and payload.ref_lens == host.ref_lens and payload.ref_names == host.ref_names
    dev = ctx.bam_to_device(payload)
    st = dev.stats
    assert (st.n_seq_words, st.n_cigar_ops) == (host.seq4.shape[0], host.cigar.shape[0])
    assert st.max_ref_span == host.max_ref_span and bool(st.sorted) == host.sorted and not st.multi_contig
    assert st.aligned_bases == host.count_aligned_bases(0)
    s = dev.struct
    for field, arr in (("pos", host.pos), ("flag", host.flag), ("mapq", host.mapq), ("l_seq", host.l_seq), ("seq_off", host.seq_off),
                       ("cigar_off", host.cigar_off), ("seq4", host.seq4), ("qual", host.qual), ("cigar", host.cigar),
                       ("qname_hash", host.qname_hash), ("mpos", host._mpos_for_abi()), ("isize", host.isize)):
        got = ctx.download(getattr(s, field), arr.size, arr.dtype)
        assert np.array_equal(got, arr.reshape(-1)), field
    L = host.ref_lens[0]
    assert np.array_equal(ctx.pileup_counts(dev, L), ctx.pileup_counts(host, L))


# ---------------------------------------------------------------------------- BAM files inflated and indexed on the device
def _assert_device_reads_equal_host(ctx, dev, host):
    st = dev.stats
    assert dev.n_reads == host.n_reads
    assert (st.n_seq_words, st.n_cigar_ops) == (host.seq4.shape[0], host.cigar.shape[0])
    if host.n_reads:
        assert st.max_ref_span == host.max_ref_span and bool(st.sorted) == host.sorted
        assert st.aligned_bases == host.count_aligned_bases(0)
    s = dev.struct
    for field, arr in (("pos", host.pos), ("flag", host.flag), ("mapq", host.mapq), ("l_seq", host.l_seq), ("seq_off", host.seq_off),
                       ("cigar_off", host.cigar_off), ("seq4", host.seq4), ("qual", host.qual), ("cigar", host.cigar),
                       ("qname_hash", host.qname_hash), ("mpos", host._mpos_for_abi()), ("isize", host.isize)):
        if host.n_reads == 0 and field in ("seq_off", "cigar_off"):
            continue
        got = ctx.download(getattr(s, field), arr.size, arr.dtype)
        assert np.array_equal(got, arr.reshape(-1)), field


def _rebgzf(src: str, dst: str, member_bytes, level=6, strategy=0, empty_every=0):
    """Re-block a BAM's payload into BGZF members of the given payload sizes (cycled), compression level and strategy."""
    import gzip
    import struct
    import zlib

    with gzip.open(src, "rb") as fh:
        payload = fh.read()
    out, p, k = [], 0, 0

    def member(chunk):
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        data = c.compress(chunk) + c.flush()
        bsize = 18 + len(data) + 8
        assert bsize <= 65536
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + data +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    while p < len(payload):
        n = member_bytes[k % len(member_bytes)]
        out.append(member(payload[p:p + n]))
        p += n
        k += 1
        if empty_every and k % empty_every == 0:
            out.append(member(b""))
    out.append(member(b""))
    with open(dst, "wb") as fh:
        fh.write(b"".join(out))
    return payload


@pytest.mark.parametrize("name", MINIS)
def test_bam_file_inflated_and_indexed_on_device(ctx, name, tmp_path):
    """tc_bgzf_inflate + tc_bam_index_records + tc_bam_records_to_reads (the host only maps the file and walks the member
    headers) give exactly the arrays of csrc/host/bamio.c's reader — for the golden BAMs as they are and re-blocked into
    members of odd sizes (records split across members at every possible place), at compression levels 0 (stored blocks),
    1, 9, with fixed Huffman codes, and with empty members in between."""
    import zlib

    from trueconsense_b200 import bamio

    path = f"{GOLD}/{name}.bam"
    host = bamio.read_bam(path)
    dev = ctx.bam_file_to_device(path)
    assert (dev.ref_names, dev.ref_lens) == (host.ref_names, host.ref_lens)
    assert dev.info["n_records"] == host.info["n_records"] and dev.info["n_dropped_unplaced"] == host.info["n_dropped_unplaced"]
    _assert_device_reads_equal_host(ctx, dev, host)
    assert bamio.read_bam_header(path) == (host.ref_names, host.ref_lens)
    L = host.ref_lens[0]
    assert np.array_equal(ctx.pileup_counts(dev, L), ctx.pileup_counts(host, L))
    for k, (sizes, level, strategy, empty) in enumerate((([65280], 0, 0, 0), ([1, 7, 300, 4000], 1, 0, 3), ([60000, 13], 9, zlib.Z_FIXED, 0),
                                                          ([997], 6, zlib.Z_HUFFMAN_ONLY, 5))):
        p2 = str(tmp_path / f"re{k}.bam")
        _rebgzf(path, p2, sizes, level, strategy, empty)
        host2 = bamio.read_bam(p2)
        assert host2.n_reads == host.n_reads
        _assert_device_reads_equal_host(ctx, ctx.bam_file_to_device(p2), host)


def test_bam_file_on_device_synthetic_sizes(ctx, tmp_path):
    """Thousands of members and records; reads longer than a 64 KiB chunk of the payload (the chain of records jumps over
    chunks: the resolver's walk); a BAM with a header and no record; unplaced records in between."""
    from trueconsense_b200 import bamio, synth
    from trueconsense_b200.reads import ReadBatch

    for case in ("amplicon_deep", "shotgun_indels", "long_reads", "paired"):
        ref, _, b = _synth(case)
        p = str(tmp_path / f"{case}.bam")
        bamio.write_bam(p, b, "ref", len(ref), level=1)
        host = bamio.read_bam(p)
        dev = ctx.bam_file_to_device(p)
        _assert_device_reads_equal_host(ctx, dev, host)
        assert np.array_equal(ctx.pileup_counts(dev, len(ref)), ctx.pileup_counts(b, len(ref)))
    rng = np.random.default_rng(2)
    recs = []
    for i, n in enumerate((50, 70000, 30, 120000, 65536, 10, 200000, 40)):      # records of up to 300 KB between short ones
        recs.append(dict(pos=5 + i, cigar=f"{n}M", seq="".join("ACGT"[x] for x in rng.integers(0, 4, n)), qual=[int(x) for x in rng.integers(0, 40, n)]))
    big = ReadBatch.from_records(recs)
    p = str(tmp_path / "big.bam")
    bamio.write_bam(p, big, "ref", 300000, level=1)
    _assert_device_reads_equal_host(ctx, ctx.bam_file_to_device(p), bamio.read_bam(p))
    empty = ReadBatch.from_records([])
    p = str(tmp_path / "empty.bam")
    bamio.write_bam(p, empty, "ref", 1000, level=1)
    dev = ctx.bam_file_to_device(p)
    assert dev.n_reads == 0 and dev.ref_lens == [1000]


def test_bam_file_on_device_rejects_damaged_files(ctx, tmp_path):
    """A flipped payload bit is a CRC-32 mismatch (htslib fails there too), a damaged DEFLATE stream does not inflate, a
    record whose sizes do not add up is refused — errors, not crashes; BamHandle then lets the host reader name the spot."""
    from trueconsense_b200 import bamio, gpu
    from trueconsense_b200.indexing import BamHandle

    ref, _, b = _synth("shotgun_indels")
    good = str(tmp_path / "good.bam")
    bamio.write_bam(good, b, "ref", len(ref), level=1)
    raw = bytearray(open(good, "rb").read())
    m = bamio.map_bgzf(good)
    blocks = m.blocks()
    m.release()
    assert len(blocks) > 5
    rng = np.random.default_rng(9)
    refused = 0
    for trial in range(24):
        bad = bytearray(raw)
        blk = blocks[int(rng.integers(0, len(blocks) - 1))]
        if trial % 3 == 0:          # the stored CRC
            bad[int(blk["coff"]) + int(blk["csize"]) + int(rng.integers(0, 4))] ^= 1 << int(rng.integers(0, 8))
        else:                       # the DEFLATE stream
            bad[int(blk["coff"]) + int(rng.integers(0, blk["csize"]))] ^= 1 << int(rng.integers(0, 8))
        p = str(tmp_path / f"bad{trial}.bam")
        open(p, "wb").write(bytes(bad))
        with pytest.raises(gpu.TcError) as ei:
            ctx.bam_file_to_device(p)
        assert "BGZF member" in str(ei.value)
        refused += 1
        if trial < 3:
            with pytest.raises(OSError):
                BamHandle(p).device_reads()
    assert refused == 24
    # a record that lies about its sizes, inside intact members
    import struct

    payload = bytearray(_rebgzf(good, str(tmp_path / "tmp.bam"), [65280]))
    hdr = bamio.parse_bam_header(bytes(payload[:4096]), len(payload))
    q = hdr[2]
    for _ in range(40):
        q += 4 + struct.unpack_from("<i", payload, q)[0]
    struct.pack_into("<I", payload, q + 4 + 16, 1 << 20)            # l_seq far beyond block_size
    src = str(tmp_path / "lying_payload.bin.gz")
    import gzip

    with gzip.open(src, "wb") as fh:
        fh.write(bytes(payload))
    lying = str(tmp_path / "lying.bam")
    _rebgzf(src, lying, [65280])
    with pytest.raises(gpu.TcError):
        ctx.bam_file_to_device(lying)
    with pytest.raises(OSError) as ei:
        BamHandle(lying).device_reads()
    assert "shorter than its fields" in str(ei.value)
    # and the context still works
    _assert_device_reads_equal_host(ctx, ctx.bam_file_to_device(good), bamio.read_bam(good))


def test_bam_file_on_device_long_header_and_unplaced_records(ctx, tmp_path):
    """A header of 6000 references (longer than two 64 KiB chunks of the payload: the chain's anchor is not chunk 0) and
    unplaced records (refID -1) between and behind the placed ones: same arrays, same counts as the host reader."""
    import gzip
    import struct

    from trueconsense_b200 import bamio

    src = f"{GOLD}/mini_illumina.bam"
    with gzip.open(src, "rb") as fh:
        payload = fh.read()
    names, lens, first = bamio.parse_bam_header(payload[:65536], len(payload))
    refs = [(names[0], lens[0])] + [(f"decoy_{i:05d}_with_a_long_name", 1000 + i) for i in range(6000)]
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    hdr = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for n, l in refs:
        nb = n.encode() + b"\0"
        hdr += struct.pack("<i", len(nb)) + nb + struct.pack("<i", l)
    assert len(hdr) > 2 * 65536
    # the records, with an unplaced one (refID -1, pos -1) spliced in after every 50th and three at the end
    recs, q = [], first
    while q + 4 <= len(payload):
        bs = struct.unpack_from("<i", payload, q)[0]
        recs.append(payload[q:q + 4 + bs])
        q += 4 + bs

    def unplaced(k):
        name = b"unplaced%04d\0" % k
        body = struct.pack("<iiBBHHHIiii", -1, -1, len(name), 0, 4680, 0, 4, 6, -1, -1, 0) + name + bytes([0x12, 0x48, 0x21]) + bytes([30] * 6)
        return struct.pack("<i", len(body)) + body

    out = []
    for i, r in enumerate(recs):
        out.append(r)
        if i % 50 == 49:
            out.append(unplaced(i))
    out += [unplaced(9000 + k) for k in range(3)]
    body = hdr + b"".join(out)
    raw = str(tmp_path / "payload.gz")
    with gzip.open(raw, "wb") as fh:
        fh.write(body)
    path = str(tmp_path / "long_header.bam")
    _rebgzf(raw, path, [65280, 40000, 777])
    host = bamio.read_bam(path)
    assert host.n_reads == len(recs) and host.info["n_dropped_unplaced"] == len(out) - len(recs) and len(host.ref_names) == 6001
    dev = ctx.bam_file_to_device(path)
    assert dev.ref_names == host.ref_names and dev.ref_lens == host.ref_lens
    assert dev.info["n_records"] == len(out) and dev.info["n_dropped_unplaced"] == len(out) - len(recs)
    _assert_device_reads_equal_host(ctx, dev, host)
    assert bamio.read_bam_header(path) == (host.ref_names, host.ref_lens)


# ---------------------------------------------------------------------------- (7) bench.py --dump-outputs
def test_bench_dump_outputs_are_the_last_steps_results(orc, tmp_path):
    """`bench.py --dump-outputs DIR`: the last timed step's count table, call table and insertion calls as float64 arrays —
    the same from run to run (an odd and an even number of steps read back the two different sets of tables the chained
    loop alternates between) and equal to the oracle's on the benchmarked sample."""
    import importlib.util
    import re
    import subprocess
    import sys

    from conftest import ROOT

    pileup, call = orc
    dumps = []
    for steps in (1, 2):
        d = tmp_path / f"steps{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                              "--scale", "0.01", "--spinup", "0", "--no-read-range", "--no-configs", "--cpu-reads", "2000",
                              "--e2e-lanes", "1", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a, b = dumps
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20

    spec = importlib.util.spec_from_file_location("tc_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    w, batch = bench.make_sample(0.01, 0)
    L = len(w.ref)
    exp = pileup.pileup_counts(batch, L).astype(np.int64)
    assert np.array_equal(a["counts"], exp)
    ref = call.call_table(exp, w.mincov, True)
    for k in ("call_char", "flags", "xrun", "ambig_char"):
        assert np.array_equal(a[k], ref[k]), k
    cands = call.insert_candidates(exp, w.mincov)
    assert len(cands) > 0 and a["insert_pos"].tolist() == cands
    for i, p in enumerate(cands):
        cols = pileup.pileup_columns(batch, region=(p - 1, p), **pileup.EXTRACTINSERTS)
        exp_bases = call.extract_insert(cols[0][1] if cols else "")
        s = "".join(chr(int(c)) for c in a["insert_string"][i] if c)
        m = re.search(r"(\d)([a-zA-Z]+)", s)
        assert ((m.group(2), m.group(1)) if m else (None, None)) == exp_bases, (p, s)
