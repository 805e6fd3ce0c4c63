"""BAM files that are not coordinate-sorted, accepted with ``sort=True`` / ``--sort-input``: the records are put in samtools'
default coordinate order on the GPU (``tc_bam_sort_records``) and every pass then computes what it computes on the file
``samtools sort`` would have written.  The order oracle here restates that order on the host (refID, pos + 1, forward
before reverse, file order; a file already sorted by (refID, pos) is used as written) and writes the same record bytes in
that order, so each device result is compared with the existing path over the oracle-ordered file."""
import json
import os
import struct

import numpy as np
import pytest

from bamfiles import assert_same_arrays, dev_arrays, mini_argv, multi_ref_files, run_cli, split, write
from conftest import GOLD, load_golden_counts

MINIS = ("quirk", "mini_illumina", "mini_ont", "mini_long", "mini_overlap")


# ---------------------------------------------------------------------------- fixture helpers (host only)
def _rec_keys(recs):
    """refID, pos, FLAG of raw records."""
    tid = np.array([struct.unpack_from("<i", r, 4)[0] for r in recs], np.int64)
    pos = np.array([struct.unpack_from("<i", r, 8)[0] for r in recs], np.int64)
    flag = np.array([struct.unpack_from("<H", r, 18)[0] for r in recs], np.int64)
    return tid, pos, flag


def _shuffle(src, dst, seed, order=None):
    """The records of ``src`` in a seeded random order (or ``order``), re-blocked into members of varying size."""
    head, recs = split(src)
    rng = np.random.default_rng(seed)
    perm = rng.permutation(len(recs)) if order is None else order
    sizes = tuple(int(x) for x in rng.integers(200, 65280, 7))
    return write(dst, head, [recs[i] for i in perm], sizes)


def oracle_order(tid, pos, flag, strand=True):
    """samtools' default coordinate order (bam_sort.c bam1_cmp_core + its stable merge) of placed records: refID, pos + 1,
    forward before reverse, file order.  Records already sorted by (refID, pos) keep their order."""
    tid, pos, flag = (np.asarray(x, np.int64) for x in (tid, pos, flag))
    n = tid.shape[0]
    if n < 2 or np.all((np.diff(tid) > 0) | ((np.diff(tid) == 0) & (np.diff(pos) >= 0))):
        return np.arange(n)
    rev = (flag >> 4) & 1 if strand else np.zeros(n, np.int64)
    return np.lexsort((np.arange(n), rev, pos + 1, tid))


def _oracle_bam(src, dst, strand=True):
    """The placed records of ``src`` in the oracle's order, keys from the host decode (bamio.read_bam, file order)."""
    from trueconsense_b200 import bamio

    head, recs = split(src)
    recs = [r for r in recs if struct.unpack_from("<i", r, 4)[0] >= 0]
    b = bamio.read_bam(src)
    assert b.n_reads == len(recs) and np.array_equal(b.pos, _rec_keys(recs)[1])
    tid = np.zeros(b.n_reads, np.int64) if b.tid is None else b.tid
    order = oracle_order(tid, b.pos, b.flag, strand)
    write(dst, head, [recs[i] for i in order])
    return dst, order


def _all_columns(ctx, d, L, params=None):
    return ctx.extract_inserts(d, L, np.arange(1, L + 1, dtype=np.int32), params)


def _golden(name):
    """The reference CLI's files for a golden BAM (tests/golden/cli_*)."""
    return {e: open(f"{GOLD}/cli_{name}.{'cov.tsv' if e == 'tsv' else e}").read() for e in ("fasta", "vcf", "gff", "tsv")}


def _as_golden(got):
    """CLI outputs with the VCF header's date, reference directory and command line as the golden files hold them."""
    assert isinstance(got, dict), got
    vcf = "".join("##fileDate=<date>\n" if l.startswith("##fileDate=") else l for l in got["vcf"].splitlines(keepends=True))
    return dict(got, vcf=vcf.replace(GOLD + os.sep, "").replace("<sorted>", "<golden>"))


# ---------------------------------------------------------------------------- CPU tests
def test_order_oracle_hand_cases():
    # sorted by (refID, pos): as written, ties and strands included
    assert oracle_order([0, 0, 0, 1], [5, 5, 5, 0], [16, 0, 16, 0]).tolist() == [0, 1, 2, 3]
    # refID first, then pos, then forward before reverse, then file order
    tid = [1, 0, 0, 0, 0, 0]
    pos = [0, 9, 3, 3, 3, 3]
    flag = [0, 0, 16, 0, 16, 0x40]
    assert oracle_order(tid, pos, flag).tolist() == [3, 5, 2, 4, 1, 0]
    assert oracle_order(tid, pos, flag, strand=False).tolist() == [2, 3, 4, 5, 1, 0]
    # pos -1 (a placed record without a position) sorts before pos 0
    assert oracle_order([0, 0], [0, -1], [0, 0]).tolist() == [1, 0]
    assert oracle_order([], [], []).tolist() == [] and oracle_order([3], [7], [16]).tolist() == [0]


def test_sort_input_flag(tmp_path):
    from trueconsense_b200 import TrueConsense, indexing

    bam = tmp_path / "a.bam"; fa = tmp_path / "r.fasta"; gff = tmp_path / "f.gff"; ov = tmp_path / "o.csv.gz"
    for p in (bam, fa, gff, ov):
        p.write_text("x")
    base = ["-i", str(bam), "-ref", str(fa), "-gff", str(gff), "-cov", "30", "-name", "s", "-o", str(tmp_path / "c.fa")]
    assert TrueConsense.GetArgs(base).sort_input is False
    assert TrueConsense.GetArgs(base + ["--sort-input"]).sort_input is True
    o = TrueConsense.GetArgs(base + ["--sort-input", "--all-contigs"])
    assert o.sort_input and o.all_contigs
    o = TrueConsense.GetArgs(base + ["--sort-input", "--index-override", str(ov)])
    assert o.sort_input and o.index_override == str(ov)
    assert indexing.Readbam(str(bam), sort=True).sort is True
    assert indexing.Readbam(str(bam)).sort is False
    h = indexing.BamHandle(str(bam), sort=True)
    assert indexing.Readbam(h) is h


def test_shuffle_helpers_keep_the_records(tmp_path):
    """The fixture helpers themselves: a shuffle keeps every record's bytes, the oracle file holds them in the oracle's order."""
    from trueconsense_b200 import build

    build.build_host()
    src = f"{GOLD}/mini_illumina.bam"
    shuf = _shuffle(src, str(tmp_path / "s.bam"), 3)
    h0, r0 = split(src)
    h1, r1 = split(shuf)
    assert h0 == h1 and sorted(r0) == sorted(r1) and r0 != r1
    dst, order = _oracle_bam(shuf, str(tmp_path / "o.bam"))
    _, r2 = split(dst)
    assert r2 == [r1[i] for i in order]
    tid, pos, flag = _rec_keys(r2)
    key = (tid << 33) | ((pos + 1) << 1) | ((flag >> 4) & 1)
    assert np.all(np.diff(key) >= 0)


# ---------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import build, gpu

    build.build_host()
    if not os.path.exists(build.CUDA_LIB):
        build.build_cuda()
    return gpu.default_context()


@pytest.mark.gpu
@pytest.mark.parametrize("name", MINIS)
def test_sorted_files_are_untouched(ctx, name, tmp_path, monkeypatch):
    """A coordinate-sorted file with sort=True: the same device arrays as without, nothing reordered, and --sort-input writes
    the reference CLI's golden files."""
    path = f"{GOLD}/{name}.bam"
    plain = dev_arrays(ctx, ctx.bam_file_to_device(path))
    d = ctx.bam_file_to_device(path, sort=True)
    assert d.info["reordered"] is False and not d.stats.unsorted
    assert_same_arrays(dev_arrays(ctx, d), plain, name)
    got = run_cli(["--sort-input"] + mini_argv(name, path), str(tmp_path / name), monkeypatch, argv0="<sorted>")
    assert _as_golden(got) == _golden(name)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("name", MINIS)
def test_shuffled_goldens(ctx, name, seed, tmp_path, monkeypatch):
    """A golden BAM shuffled: device arrays == the plain decode of the oracle-ordered file, BuildIndex == the golden table,
    ListInserts and ExtractInserts (every column) == the path over the oracle-ordered file, and so are the CLI's outputs.
    Where the oracle's order is the golden file's own, the CLI writes the golden files."""
    from trueconsense_b200 import Events, indexing

    src = f"{GOLD}/{name}.bam"
    shuf = _shuffle(src, str(tmp_path / "shuf.bam"), seed)
    ordered, _ = _oracle_bam(shuf, str(tmp_path / "ordered.bam"))
    L = load_golden_counts(name).shape[1]
    want = dev_arrays(ctx, ctx.bam_file_to_device(ordered))
    d = ctx.bam_file_to_device(shuf, sort=True)
    assert d.info["reordered"] is True and not d.stats.unsorted and not d.stats.multi_contig
    assert_same_arrays(dev_arrays(ctx, d), want, name)
    cols = _all_columns(ctx, d, L)
    assert cols == _all_columns(ctx, ctx.bam_file_to_device(ordered), L)
    with pytest.raises(ValueError, match="Unsorted input. Pileup aborts"):
        indexing.BuildIndex(shuf, f"{GOLD}/{name}.fasta")
    h = indexing.Readbam(shuf, sort=True)
    frame = indexing.BuildIndex(h, f"{GOLD}/{name}.fasta")
    assert np.array_equal(np.stack([frame[c].to_numpy() for c in indexing.COLUMNS]), load_golden_counts(name))
    index = frame.to_dict("index")
    mincov = json.load(open(f"{GOLD}/{name}.json"))["mincov"]
    assert Events.ListInserts(index, mincov, h) == Events.ListInserts(index, mincov, indexing.Readbam(ordered))
    got = run_cli(["--sort-input"] + mini_argv(name, shuf), str(tmp_path / "s"), monkeypatch, argv0="<sorted>")
    exp = run_cli(mini_argv(name, ordered), str(tmp_path / "o"), monkeypatch, argv0="<sorted>")
    assert got == exp
    _, golden_recs = split(src)
    _, ordered_recs = split(ordered)
    if ordered_recs == [r for r in golden_recs if struct.unpack_from("<i", r, 4)[0] >= 0]:
        # the oracle restores the golden file's own order: the reference CLI's files apply as they are
        assert _as_golden(got) == _golden(name), f"{name}: the oracle order is the golden file's own order"


def _tie_batch():
    """9000 single-end reads over one column, all starting at 100: 4500 forward reads with insertion AC, 4500 reverse ones
    with GT (quality 30)."""
    from trueconsense_b200.reads import ReadBatch

    recs = [dict(pos=100, cigar="10M2I40M", seq="A" * 10 + ("AC" if j < 4500 else "GT") + "A" * 40, flag=0 if j < 4500 else 16,
                 qname=f"t{j}") for j in range(9000)]
    return ReadBatch.from_records(recs)


@pytest.mark.gpu
def test_ties_decide_the_result(ctx, tmp_path):
    """The 8000-read cap admits reads in the order they arrive, so the tie rule decides the call: samtools' order puts the
    forward reads (AC) first.  The same shuffled file ordered without the strand key admits more GT reads and calls GT."""
    from trueconsense_b200 import Events, bamio, indexing
    from trueconsense_b200.reads import ReadBatch

    sorted_bam = str(tmp_path / "col.bam")
    bamio.write_bam(sorted_bam, _tie_batch(), "ref", 1000)
    later = str(tmp_path / "later.bam")
    bamio.write_bam(later, ReadBatch.from_records([dict(pos=300, cigar="50M", seq="C" * 50, qname=f"l{j}") for j in range(3)]),
                    "ref", 1000)
    head, recs = split(sorted_bam)
    perm = np.random.default_rng(8).permutation(len(recs))
    shuffled = split(later)[1] + [recs[i] for i in perm]          # a few later reads ahead: not sorted by (refID, pos)
    path = write(str(tmp_path / "shuf.bam"), head, shuffled, (40000, 9000, 65280))
    assert np.sum(perm[:8000] < 4500) < 4000                        # the file's own order admits more GT than AC
    col = 110                       # 1-based: the last M column before the insertion
    assert Events.ExtractInserts(indexing.Readbam(path, sort=True), col) == ("AC", "2")
    d = ctx.bam_file_to_device(path, sort=True)
    got = ctx.extract_inserts(d, 1000, [col])[0]
    assert got["n_entries"] == 8000 and got["string"] == "A+2AC" and got["mode_count"] == 4500
    strandless, _ = _oracle_bam(path, str(tmp_path / "nostrand.bam"), strand=False)
    assert Events.ExtractInserts(indexing.Readbam(strandless), col) == ("GT", "2")
    ordered, _ = _oracle_bam(path, str(tmp_path / "ordered.bam"))
    assert Events.ExtractInserts(indexing.Readbam(ordered), col) == ("AC", "2")


@pytest.mark.gpu
def test_mates_far_apart(ctx, tmp_path):
    """Overlapping mates placed far apart in the file (every first mate, then every second mate in the reverse order):
    ExtractInserts on every column == the oracle-ordered path, under htslib >= 1.13's and <= 1.12's overlap rewrite."""
    from trueconsense_b200 import gpu

    src = f"{GOLD}/mini_overlap.bam"
    _, recs = split(src)
    _, _, flag = _rec_keys(recs)
    rng = np.random.default_rng(4)
    first = rng.permutation(np.flatnonzero(flag & 0x40))
    second = np.flatnonzero((flag & 0x40) == 0)
    second = second[np.argsort(rng.random(second.size))][::-1]
    order = np.concatenate([first, second])
    assert sorted(order.tolist()) == list(range(len(recs)))
    shuf = _shuffle(src, str(tmp_path / "far.bam"), 4, order=order)
    ordered, _ = _oracle_bam(shuf, str(tmp_path / "ordered.bam"))
    L = load_golden_counts("mini_overlap").shape[1]
    for mode in (0, 2):
        p = gpu.extractinserts_params()
        p.reserved = mode << 8
        got = _all_columns(ctx, ctx.bam_file_to_device(shuf, sort=True), L, p)
        exp = _all_columns(ctx, ctx.bam_file_to_device(ordered), L, p)
        assert got == exp, mode
        assert any(c["n_entries"] for c in got)


@pytest.mark.gpu
def test_multi_reference_interleaved_long_header(ctx, tmp_path, monkeypatch):
    """References' records interleaved (refIDs decreasing, shuffled inside each reference) under a header of 6003
    references (13 key bits of refID): --all-contigs --sort-input == --all-contigs over the oracle-ordered file —
    first_read, counts, insertion calls and the four output files.  Without the flag: the unsorted refusal."""
    from trueconsense_b200 import Events, indexing

    tmp = str(tmp_path)
    head, real, slots, fasta, gff = multi_ref_files(tmp)
    rng = np.random.default_rng(9)
    body = []
    for i in reversed(slots):
        recs = real[i]["recs"]
        body += [recs[j] for j in rng.permutation(len(recs))]
    shuf = write(os.path.join(tmp, "shuf.bam"), head, body, (65280, 3000, 20000))
    ordered, _ = _oracle_bam(shuf, os.path.join(tmp, "ordered.bam"))
    hs, ho = indexing.Readbam(shuf, sort=True), indexing.Readbam(ordered)
    fs, fo = indexing.BuildIndexContigs(hs, fasta), indexing.BuildIndexContigs(ho, fasta)
    assert list(fs) == list(fo) and len(fs) == 6003
    for n in fs:
        assert fs[n].equals(fo[n]), n
    names = list(fs)
    lens = [len(fs[n]) for n in names]
    _, lay_s = hs.device_reads_contigs(names, lens)
    _, lay_o = ho.device_reads_contigs(names, lens)
    assert np.array_equal(lay_s.first_read, lay_o.first_read)
    assert [int(lay_s.first_read[i + 1] - lay_s.first_read[i]) for i in slots] == [len(real[i]["recs"]) for i in slots]
    idx = {n: f.to_dict("index") for n, f in fs.items()}
    ins_s, ins_o = Events.ListInsertsContigs(idx, 30, hs), Events.ListInsertsContigs(idx, 30, ho)
    assert ins_s == ins_o and ins_s["c0"][0] and ins_s["c2"][0]
    base = ["-ref", fasta, "-gff", gff, "-cov", "30", "-name", "S", "--all-contigs"]
    got = run_cli(["--sort-input", "-i", shuf] + base, os.path.join(tmp, "s"), monkeypatch, argv0="<sorted>")
    exp = run_cli(["-i", ordered] + base, os.path.join(tmp, "o"), monkeypatch, argv0="<sorted>")
    assert isinstance(got, dict) and got == exp
    assert got["fasta"].count(">") == 6003
    with pytest.raises(ValueError, match="Unsorted input. Pileup aborts"):
        indexing.BuildIndexContigs(indexing.Readbam(shuf), fasta)


@pytest.mark.gpu
def test_host_inflate_route(ctx, tmp_path):
    """bam_to_device(read_bam_payload(path), sort=True) == the device route, with the payload uploaded once."""
    from trueconsense_b200 import bamio

    shuf = _shuffle(f"{GOLD}/mini_illumina.bam", str(tmp_path / "shuf.bam"), 5)
    d = ctx.bam_file_to_device(shuf, sort=True)
    assert d.info["reordered"] is True
    want = dev_arrays(ctx, d)
    payload = bamio.read_bam_payload(shuf)
    x0 = ctx.transfer_bytes()[0]
    h = ctx.bam_to_device(payload, sort=True)
    x1 = ctx.transfer_bytes()[0]
    assert h.info["reordered"] is True and not h.stats.unsorted
    assert x1 - x0 <= payload.n_bytes + 8 * payload.n_reads + 4096, (x1 - x0, payload.n_bytes)
    assert_same_arrays(dev_arrays(ctx, h), want)
    # and first_read from the sorted offsets
    h = ctx.bam_to_device(payload, sort=True, contig_ranges=True)
    assert h.first_read.tolist() == [0, payload.n_reads]
    payload.release()


@pytest.mark.gpu
def test_size_200k_config2_slice(ctx, tmp_path):
    """A 200 k-read config-2 slice, shuffled: arrays == the oracle-ordered decode, counts == the synthetic batch's, and the
    chained sample (tc_sample_enqueue / finish) over the reads sorted on the device == the separate calls."""
    import torch

    from trueconsense_b200 import bamio, gpu, synth

    w = synth.config(1, scale=0.1)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    assert b.n_reads == 200_000
    src = str(tmp_path / "cfg2.bam")
    bamio.write_bam(src, b, "ref", L)
    shuf = _shuffle(src, str(tmp_path / "shuf.bam"), 6)
    ordered, _ = _oracle_bam(shuf, str(tmp_path / "ordered.bam"))
    want = dev_arrays(ctx, ctx.bam_file_to_device(ordered))
    exp_counts = ctx.pileup_counts(b, L)
    d = ctx.bam_file_to_device(shuf, sort=True)
    assert d.info["reordered"] is True and d.n_reads == b.n_reads
    assert_same_arrays(dev_arrays(ctx, d), want)
    assert np.array_equal(ctx.pileup_counts(d, L), exp_counts)
    res = ctx.call(exp_counts, L, w.mincov, True)
    cands = ctx.list_insert_candidates(res.flags, L)
    assert len(cands) > 0
    sep = ctx.extract_inserts(d, L, cands)
    counts = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
    flags = torch.empty(L, dtype=torch.uint8, device="cuda")
    xrun = torch.empty(L, dtype=torch.int32, device="cuda")
    t = ctx.sample_enqueue(d, L, w.mincov, True, counts, gpu.CallTable(None, flags.data_ptr(), xrun.data_ptr(), None, None, None))
    assert ctx.sample_finish(t) == sep
    assert np.array_equal(counts.cpu().numpy(), exp_counts) and np.array_equal(flags.cpu().numpy(), res.flags)


@pytest.mark.gpu
def test_edge_cases(ctx, tmp_path):
    """No record, one record, every record at one position; records a placed read may not hold -> TC_ERR_RANGE naming
    the record."""
    from trueconsense_b200 import bamio, gpu
    from trueconsense_b200.reads import ReadBatch

    empty = str(tmp_path / "empty.bam")
    bamio.write_bam(empty, ReadBatch.from_records([]), "ref", 100)
    d = ctx.bam_file_to_device(empty, sort=True)
    assert d.n_reads == 0 and d.info["reordered"] is False
    p = bamio.read_bam_payload(empty)
    assert ctx.bam_to_device(p, sort=True).n_reads == 0
    p.release()

    one = str(tmp_path / "one.bam")
    bamio.write_bam(one, ReadBatch.from_records([dict(pos=7, cigar="5M", seq="ACGTA", flag=16)]), "ref", 100)
    want = dev_arrays(ctx, ctx.bam_file_to_device(one))
    d = ctx.bam_file_to_device(one, sort=True)
    assert d.info["reordered"] is False
    assert_same_arrays(dev_arrays(ctx, d), want)

    rng = np.random.default_rng(2)
    recs = [dict(pos=20, cigar="30M", seq="".join(rng.choice(list("ACGT"), 30)), flag=int(16 * (j % 3 == 0)), qname=f"s{j}")
            for j in range(3000)]
    same = str(tmp_path / "same.bam")
    bamio.write_bam(same, ReadBatch.from_records(recs), "ref", 100)
    # one position only: every order is sorted by (refID, pos), so the records stay as written ...
    shuf = _shuffle(same, str(tmp_path / "same_shuf.bam"), 2)
    d = ctx.bam_file_to_device(shuf, sort=True)
    assert d.info["reordered"] is False
    assert_same_arrays(dev_arrays(ctx, d), dev_arrays(ctx, ctx.bam_file_to_device(shuf)))
    # ... unless one record at another position makes the file unsorted: then forward before reverse, file order in each
    head, rr = split(shuf)
    before = bytearray(rr[-1])
    struct.pack_into("<i", before, 8, 25)
    mixed = write(str(tmp_path / "mixed.bam"), head, [bytes(before)] + rr[:-1])
    ordered, order = _oracle_bam(mixed, str(tmp_path / "mixed_ordered.bam"))
    assert order[-1] == 0
    d = ctx.bam_file_to_device(mixed, sort=True)
    assert d.info["reordered"] is True
    assert_same_arrays(dev_arrays(ctx, d), dev_arrays(ctx, ctx.bam_file_to_device(ordered)))

    # refID >= n_ref / pos < -1: the host reader passes them on, the sort refuses them and names the record
    head, rr = split(same)
    for off, value in ((4, 1), (8, -2)):
        bad = bytearray(rr[5])
        struct.pack_into("<i", bad, off, value)
        path = write(str(tmp_path / f"bad{off}.bam"), head, rr[:5] + [bytes(bad)] + rr[6:])
        p = bamio.read_bam_payload(path)
        with pytest.raises(gpu.TcError) as ei:
            ctx.bam_to_device(p, sort=True)
        p.release()
        assert ei.value.code == -7 and "record 5 " in str(ei.value), str(ei.value)
