"""Every reference of a multi-reference BAM in one device pass (--all-contigs, BuildIndexContigs, ListInsertsContigs,
WriteOutputsContigs, tc_call_contigs): each reference's results equal what the single-reference path computes for a BAM
holding only that reference's records (mates elsewhere still "on another reference"), the FASTA record of its name, its
GFF rows and the sample name {sample}_{reference}.  The fixtures are built here from seeded synthetic reads."""
import gzip
import os
import struct
import zlib

import numpy as np
import pytest

from conftest import GOLD


# ---------------------------------------------------------------------------- fixture helpers (host only)
def _bgzf(path: str, payload: bytes, member_bytes: int = 65280) -> None:
    """Write a BAM payload as BGZF members (and the EOF member)."""
    def member(chunk):
        c = zlib.compressobj(1, zlib.DEFLATED, -15, 8, 0)
        data = c.compress(chunk) + c.flush()
        bsize = 18 + len(data) + 8
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + data +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    out = [member(payload[p:p + member_bytes]) for p in range(0, len(payload), member_bytes)]
    out.append(member(b""))
    with open(path, "wb") as fh:
        fh.write(b"".join(out))


def _records(path: str) -> list[bytes]:
    """The records of a BAM file, each with its block_size."""
    from trueconsense_b200 import bamio

    with gzip.open(path, "rb") as fh:
        payload = fh.read()
    _, _, q = bamio.parse_bam_header(payload, len(payload))
    recs = []
    while q + 4 <= len(payload):
        bs = struct.unpack_from("<i", payload, q)[0]
        recs.append(payload[q:q + 4 + bs])
        q += 4 + bs
    return recs


def _unplaced(k: int) -> bytes:
    name = b"unplaced%04d\0" % k
    body = struct.pack("<iiBBHHHIiii", -1, -1, len(name), 0, 4680, 0, 4, 6, -1, -1, 0) + name + bytes([0x12, 0x48, 0x21]) + bytes([30] * 6)
    return struct.pack("<i", len(body)) + body


def _header(refs) -> bytes:
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    h = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for n, l in refs:
        nb = n.encode() + b"\0"
        h += struct.pack("<i", len(nb)) + nb + struct.pack("<i", l)
    return h


def _multi_bam(path, contigs, extra_refs=(), unplaced_every=0, order=None):
    """One BAM of all contigs from their single-contig BAMs: refID -> the contig's index, next refID 0 (same reference)
    -> the same, 1 (another reference) -> the next contig; ``extra_refs`` (name, length) follow in the header without
    records; unplaced records (refID -1) spliced in after every ``unplaced_every``-th record and three at the end."""
    n = len(contigs)
    body = []
    for k in (order or range(n)):
        for r in _records(contigs[k]["bam"]):
            r = bytearray(r)
            mtid = struct.unpack_from("<i", r, 24)[0]
            struct.pack_into("<i", r, 4, k)
            if mtid >= 0:
                struct.pack_into("<i", r, 24, k if mtid == 0 else (k + 1) % n)
            body.append(bytes(r))
            if unplaced_every and len(body) % unplaced_every == 0:
                body.append(_unplaced(len(body)))
    if unplaced_every:
        body += [_unplaced(90000 + j) for j in range(3)]
    refs = [(c["name"], c["bam_len"]) for c in contigs] + list(extra_refs)
    _bgzf(path, _header(refs) + b"".join(body))


def _with_mates(b, rng, frac_other):
    """tid 0; mtid 0 for paired reads (1 = mate on another reference for a share of them), -1 otherwise."""
    paired = (b.flag & 1) != 0
    mtid = np.where(paired, 0, -1).astype(np.int32)
    mtid[paired & (rng.random(b.n_reads) < frac_other)] = 1
    b.tid = np.zeros(b.n_reads, np.int32)
    b.mtid = mtid
    return b


def _hand_batch(recs):
    from trueconsense_b200.reads import ReadBatch

    b = ReadBatch.from_records(recs)
    b.mtid = np.full(b.n_reads, -1, np.int32)
    return b


def _write_contig(tmp, c, b):
    from trueconsense_b200 import bamio, synth

    c["bam"] = os.path.join(tmp, f"{c['name']}.bam")
    c["fasta"] = os.path.join(tmp, f"{c['name']}.fasta")
    c["gff"] = os.path.join(tmp, f"{c['name']}.gff")
    c.setdefault("bam_len", len(c["seq"]))
    bamio.write_bam(c["bam"], b, c["name"], c["bam_len"], level=1)
    synth.write_fasta(c["fasta"], c["name"], c["seq"])
    _write_gff_rows(c["gff"], [c])


def _write_gff_rows(path, contigs):
    with open(path, "w") as fh:
        fh.write("##gff-version 3\n")
        for c in contigs:
            for f in c["feats"]:
                attrs = f"ID=cds-{c['name']}-{f['name']};Name={f['name']};gbkey=CDS"
                fh.write("\t".join([c["name"], "synthetic", "CDS", str(f["start"]), str(f["end"]), ".", f["strand"], "0", attrs]) + "\n")


def _write_multi(tmp, contigs, stem="flu", **kw):
    from trueconsense_b200 import synth

    paths = {e: os.path.join(tmp, f"{stem}.{e}") for e in ("bam", "fasta", "gff")}
    _multi_bam(paths["bam"], contigs, **kw)
    with open(paths["fasta"], "w") as fh:
        for c in contigs:
            fh.write(f">{c['name']} segment\n")
            for i in range(0, len(c["seq"]), 60):
                fh.write(c["seq"][i:i + 60] + "\n")
    _write_gff_rows(paths["gff"], contigs)
    return paths


FLU_LENGTHS = [2341, 2341, 2233, 1778, 1565, 1413, 1027, 890]


def _flu_contigs(tmp, with_tiny=True):
    """Eight segments of 890-2341 bp with stop-free '+' ORFs, a reference without reads and one of length 1:
    * seg2: 9000 reads ending at its last column, 60 % of them with a 2-bp insertion — the 8000 cap binds at that column;
    * seg3, right behind seg2: a 3-bp insertion (60 %) at its first column, its plain reads first in file order;
    * seg4: a 3-bp deletion inside an ORF; seg6: a 3-bp insertion inside an ORF;
    * paired reads, some with mates on another reference."""
    from trueconsense_b200 import synth

    rng = np.random.default_rng(11)
    contigs = []
    for i, L in enumerate(FLU_LENGTHS):
        name = f"seg{i + 1}"
        seq, feats = synth.make_genome(L, 100 + i, "sars2")
        c = {"name": name, "seq": seq, "feats": feats}
        if name == "seg2":
            ins = seq[L - 100:L - 50] + "GT" + seq[L - 50:]
            recs = [dict(pos=L - 100, cigar="50M2I50M" if j % 5 < 3 else "100M", seq=ins if j % 5 < 3 else seq[L - 100:], qname=f"d{j}")
                    for j in range(9000)]
            b = _hand_batch(recs)
        elif name == "seg3":
            recs = [dict(pos=0, cigar="100M", seq=seq[:100], qname=f"p{j}") for j in range(200)]
            recs += [dict(pos=0, cigar="1M3I99M", seq=seq[0] + "TTG" + seq[1:100], qname=f"i{j}") for j in range(300)]
            b = _hand_batch(recs)
        else:
            a = feats[0]["start"] - 1
            vs = []
            if name == "seg4":
                vs.append(synth.Variant(a + 60, synth.VAR_DEL, 3, 0, 0.85))
            if name == "seg6":
                vs.append(synth.Variant(a + 90, synth.VAR_INS, 3, 7, 0.9))
            p = synth.SynthParams(seed=200 + i, n_reads=L * 60 // 150, ref_len=L, read_len=150, paired=(i % 2 == 0),
                                  insert_mean=300, insert_sd=40, sub_rate=0.01, softclip_rate=0.05, softclip_max=8, variants=vs)
            b = _with_mates(synth.generate_reads(p, seq), rng, 0.2)
        _write_contig(tmp, c, b)
        contigs.append(c)
    extra = [{"name": "noreads", "seq": synth.make_genome(901, 7, "sars2")[0], "feats": []}]
    if with_tiny:
        extra.append({"name": "one", "seq": "A", "feats": []})
    for c in extra:
        _write_contig(tmp, c, _hand_batch([]))
    # header order: seg1 seg2 seg3 noreads seg4 [one] seg5 .. seg8
    out = contigs[:3] + [extra[0]] + [contigs[3]] + extra[1:] + contigs[4:]
    return out


# ---------------------------------------------------------------------------- CPU tests
def test_gff_rows_partitioned_by_seqid(tmp_path):
    import pandas as pd

    from trueconsense_b200 import indexing

    df = pd.DataFrame({"seqid": ["b", "a", "b", "a"], "start": [1, 2, 3, 4], "end": [9, 9, 9, 9]})
    parts = indexing.gff_by_contig(df, ["a", "b", "c"])
    assert list(parts) == ["a", "b", "c"]
    assert parts["a"]["start"].tolist() == [2, 4] and parts["b"]["start"].tolist() == [1, 3] and len(parts["c"]) == 0
    assert list(parts["b"].index) == [0, 1]           # indexed like a GFF file of that reference's rows alone
    with pytest.raises(ValueError, match="'z'"):
        indexing.gff_by_contig(pd.DataFrame({"seqid": ["a", "z"], "start": [1, 2], "end": [3, 4]}), ["a", "b"])


def test_fasta_lengths_by_name(tmp_path):
    from trueconsense_b200 import Outputs, indexing

    fa = tmp_path / "r.fasta"
    fa.write_text(">b desc\nACGT\nAC\n>a\nTTT\n>b\nA\n")
    assert indexing.fasta_lengths_by_name(["a", "b"], str(fa)) == [3, 6]
    with pytest.raises(ValueError, match="'c'"):
        indexing.fasta_lengths_by_name(["a", "c"], str(fa))
    assert Outputs._fasta_records(str(fa)) == {"b": list("ACGTAC"), "a": list("TTT")}


def test_all_contigs_flag(tmp_path, capsys):
    from trueconsense_b200 import TrueConsense

    bam = tmp_path / "a.bam"; fa = tmp_path / "r.fasta"; gff = tmp_path / "f.gff"; ov = tmp_path / "o.csv.gz"
    for p in (bam, fa, gff, ov):
        p.write_text("x")
    base = ["-i", str(bam), "-ref", str(fa), "-gff", str(gff), "-cov", "30", "-name", "s", "-o", str(tmp_path / "c.fa")]
    assert TrueConsense.GetArgs(base).all_contigs is False
    assert TrueConsense.GetArgs(base + ["--all-contigs"]).all_contigs is True
    assert TrueConsense.GetArgs(base + ["--index-override", str(ov)]).index_override == str(ov)
    with pytest.raises(SystemExit) as e:
        TrueConsense.GetArgs(base + ["--all-contigs", "--index-override", str(ov)])
    assert e.value.code == 2
    assert "--index-override" in capsys.readouterr().err


def test_coverage_tsv_and_vcf_header(tmp_path, monkeypatch):
    from trueconsense_b200 import Coverage, Outputs

    idx = {"a": {1: {"coverage": 5}, 2: {"coverage": 0}}, "b": {1: {"coverage": 7}}}
    out = tmp_path / "d.tsv"
    Coverage.BuildCoverageContigs(idx, str(out))
    assert out.read_text() == "a\t1\t5\na\t2\t0\nb\t1\t7\n"
    monkeypatch.setattr("sys.argv", ["TrueConsense", "--all-contigs"])
    h = Outputs.vcf_header("r.fasta", ["a", "b"])
    one = Outputs.VCF_HEADER.format(today="D", argv="--all-contigs", ref="r.fasta", contig="a")
    lines = h.splitlines()
    assert [l for l in lines if l.startswith("##contig")] == ["##contig=<ID=a>", "##contig=<ID=b>"]
    assert [l for l in lines if not l.startswith(("##contig", "##fileDate"))] == \
           [l for l in one.splitlines() if not l.startswith(("##contig", "##fileDate"))]


def test_first_read_from_tid():
    from trueconsense_b200 import indexing

    fr = indexing.contig_ranges_from_tid(np.array([0, 0, 2, 2, 2, 4], np.int32), 6, 6)
    assert fr.tolist() == [0, 2, 2, 5, 5, 6, 6]
    assert indexing.contig_ranges_from_tid(None, 2, 3).tolist() == [0, 3, 3]
    with pytest.raises(ValueError, match="Unsorted"):
        indexing.contig_ranges_from_tid(np.array([1, 0], np.int32), 2, 2)
    with pytest.raises(ValueError):
        indexing.contig_ranges_from_tid(np.array([0, 3], np.int32), 2, 2)
    lay = indexing.ContigLayout(["a", "b", "c"], [3, 0, 4], np.array([0, 3, 3, 7]), fr[:4])
    k, p = lay.locate([1, 3, 4, 7])
    assert k.tolist() == [0, 0, 2, 2] and p.tolist() == [1, 3, 1, 4] and lay.total == 7


# ---------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def flu(tmp_path_factory):
    from trueconsense_b200 import build

    build.build_host()
    if not os.path.exists(build.CUDA_LIB):
        build.build_cuda()
    tmp = str(tmp_path_factory.mktemp("flu"))
    contigs = _flu_contigs(tmp)
    return {"tmp": tmp, "contigs": contigs, **_write_multi(tmp, contigs, unplaced_every=97)}


def _fresh(path_or_batch):
    from trueconsense_b200 import indexing

    return indexing.BamHandle(path_or_batch) if isinstance(path_or_batch, str) else indexing.BamHandle("<batch>", path_or_batch)


@pytest.mark.gpu
def test_counts_equal_single_contig_runs(flu):
    """BuildIndexContigs == BuildIndex on every reference alone == the CPU oracle, for the file decoded on the device and
    for a host-decoded batch; the device's first_read equals the host's np.searchsorted over ReadBatch.tid."""
    from oracle import pileup

    from trueconsense_b200 import bamio, gpu, indexing

    pileup.build()
    host = bamio.read_bam(flu["bam"])
    assert host.info["n_dropped_unplaced"] > 3 and len(host.ref_names) == len(flu["contigs"])
    frames = indexing.BuildIndexContigs(flu["bam"], flu["fasta"])
    frames_host = indexing.BuildIndexContigs(_fresh(host), flu["fasta"])
    assert list(frames) == [c["name"] for c in flu["contigs"]] == list(frames_host)
    for c in flu["contigs"]:
        single = indexing.BuildIndex(c["bam"], c["fasta"])
        assert frames[c["name"]].equals(single), c["name"]
        assert frames_host[c["name"]].equals(single), c["name"]
        b = bamio.read_bam(c["bam"])
        exp = pileup.pileup_counts(b, len(c["seq"]))
        assert np.array_equal(np.stack([single[k].to_numpy() for k in indexing.COLUMNS]), exp[:7]), c["name"]
    ctx = gpu.default_context()
    d = ctx.bam_file_to_device(flu["bam"], contig_ranges=True)
    assert np.array_equal(d.first_read, indexing.contig_ranges_from_tid(host.tid, len(host.ref_names), host.n_reads))
    # the moved reads cannot be moved a second time
    h = _fresh(flu["bam"])
    names = [c["name"] for c in flu["contigs"]]
    dd, lay = h.device_reads_contigs(names, [len(c["seq"]) for c in flu["contigs"]])
    with pytest.raises(RuntimeError, match="already"):
        ctx.reads_to_contig_coords(dd, lay.lens, lay.first_read)
    assert h.device_reads_contigs(names, lay.lens)[0] is dd          # cached while the context stages nothing else


def _random_tables(rng, lens):
    parts = []
    for L in lens:
        c = np.zeros((8, L), np.int32)
        c[1:6] = rng.integers(0, 40, (5, L))
        c[5, rng.random(L) < 0.5] += 60                   # many X-primary columns: runs of every length
        c[6] = rng.integers(0, 30, L)
        c[0] = c[1:6].sum(axis=0)
        parts.append(c)
    return parts


@pytest.mark.gpu
def test_segmented_call_equals_per_reference_call(flu):
    """tc_call_contigs == tc_call on every reference's slice, all six outputs: random tables with X-runs that reach a
    reference's end, boundaries off the 256-column blocks, empty references, a run across a block inside a reference, and
    the fixture's own table."""
    from trueconsense_b200 import gpu, indexing

    ctx = gpu.default_context()
    rng = np.random.default_rng(5)
    cases = [[300, 1, 0, 777, 256, 513, 5], [1000], [3, 700, 900]]
    for lens in cases:
        parts = _random_tables(rng, lens)
        # all-X stretches: the tail of the first reference, and across a 256 block inside the last long one
        parts[0][5, -40:] = 500
        big = max(range(len(lens)), key=lambda i: lens[i])
        if lens[big] > 600:
            parts[big][5, 200:520] = 500
        parts = [np.ascontiguousarray(p) for p in parts]
        for p in parts:
            p[0] = p[1:6].sum(axis=0)
        start = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
        for mincov, amb in ((30, True), (1, False)):
            whole = ctx.call_contigs(np.concatenate(parts, axis=1), start, mincov, amb)
            for k, L in enumerate(lens):
                if L == 0:
                    continue
                one = ctx.call(parts[k], L, mincov, amb)
                got = whole.slice(int(start[k]), int(start[k + 1]))
                for f in ("call_char", "flags", "xrun", "rank_letter", "rank_count", "ambig_char"):
                    assert np.array_equal(getattr(got, f), getattr(one, f)), (lens, k, f)
                assert got.flags[-1] & gpu.CF_XRUN_OFF_END
    frames = indexing.BuildIndexContigs(flu["bam"], flu["fasta"])
    parts = [np.vstack([f[c].to_numpy() for c in indexing.COLUMNS] + [np.zeros(len(f), np.int64)]).astype(np.int32) for f in frames.values()]
    start = np.concatenate(([0], np.cumsum([p.shape[1] for p in parts]))).astype(np.int32)
    whole = ctx.call_contigs(np.concatenate(parts, axis=1), start, 30, True)
    for k, p in enumerate(parts):
        one = ctx.call(p, p.shape[1], 30, True)
        got = whole.slice(int(start[k]), int(start[k + 1]))
        for f in ("call_char", "flags", "xrun", "rank_letter", "rank_count", "ambig_char"):
            assert np.array_equal(getattr(got, f), getattr(one, f)), (k, f)
    bad = start.copy()
    bad[1], bad[2] = bad[2], bad[1]
    with pytest.raises(gpu.TcError) as ei:
        ctx.call_contigs(np.concatenate(parts, axis=1), bad, 30, True)
    assert ei.value.code == -2


@pytest.mark.gpu
def test_list_inserts_equal_single_contig_runs(flu):
    """ListInsertsContigs == ListInserts on every reference alone; the raw ExtractInserts columns too — in particular the
    insertion at seg3's first column, right behind seg2's 9000 reads: they sit in its fetch range but never count towards
    its 8000-read cap (else only seg3's first read, a plain one, would be admitted)."""
    from trueconsense_b200 import Events, gpu, indexing

    frames = indexing.BuildIndexContigs(flu["bam"], flu["fasta"])
    indexes = {n: f.to_dict("index") for n, f in frames.items()}
    got = Events.ListInsertsContigs(indexes, 30, indexing.Readbam(flu["bam"]))
    assert list(got) == list(frames)
    for c in flu["contigs"]:
        single = indexing.BuildIndex(c["bam"], c["fasta"]).to_dict("index")
        assert got[c["name"]] == Events.ListInserts(single, 30, indexing.Readbam(c["bam"])), c["name"]
    assert got["seg3"][0] and 1 in got["seg3"][1]
    assert got["seg2"][0] and got["seg6"][0]
    # raw columns: n_entries (the cap binds at seg2's column), strings, counts; first_read relative to the reference
    ctx = gpu.default_context()
    h = indexing.Readbam(flu["bam"])
    names = [c["name"] for c in flu["contigs"]]
    d, lay = h.device_reads_contigs(names, [len(c["seq"]) for c in flu["contigs"]])
    by_name = {c["name"]: c for c in flu["contigs"]}
    for name, col in (("seg2", len(by_name["seg2"]["seq"]) - 50), ("seg3", 1), ("seg6", None)):
        k = names.index(name)
        if col is None:
            col = next(iter(got[name][1]))
        multi = ctx.extract_inserts(d, lay.total, [int(lay.start[k]) + col])[0]
        one = ctx.extract_inserts(indexing.Readbam(by_name[name]["bam"]).device_reads(), len(by_name[name]["seq"]), [col])[0]
        multi["pos"] -= int(lay.start[k])
        multi["first_read"] -= int(lay.first_read[k])
        assert multi == one, name
        d, lay = h.device_reads_contigs(names, lay.lens)
    seg2 = ctx.extract_inserts(d, lay.total, [int(lay.start[1]) + len(by_name["seg2"]["seq"]) - 50])[0]
    assert seg2["n_entries"] == 8000


def _cli(argv, monkeypatch):
    from trueconsense_b200 import TrueConsense

    monkeypatch.setattr("sys.argv", ["TrueConsense"] + argv)
    TrueConsense.main(argv)


def _vcf_records(text):
    return [l for l in text.splitlines(keepends=True) if not l.startswith("#")]


def _norm_vcf_header(text):
    return [l for l in text.splitlines() if l.startswith("#") and not l.startswith(("##fileDate", "##source", "##reference", "##contig"))]


def _single_runs(contigs, out_dir, sample, monkeypatch, mincov=30):
    res = {}
    for c in contigs:
        out = os.path.join(out_dir, f"single_{c['name']}")
        _cli(["-i", c["bam"], "-ref", c["fasta"], "-gff", c["gff"], "-cov", str(mincov), "-name", f"{sample}_{c['name']}",
              "-o", out + ".fasta", "-vcf", out + ".vcf", "-ogff", out + ".gff", "-doc", out + ".tsv", "-t", "2"], monkeypatch)
        res[c["name"]] = {e: open(f"{out}.{e}").read() for e in ("fasta", "vcf", "gff", "tsv")}
    return res


@pytest.mark.gpu
def test_cli_all_contigs_equals_per_contig_runs(tmp_path, monkeypatch):
    """--all-contigs writes one FASTA record per reference, the GFF header once plus every reference's corrected
    features, one VCF header with a ##contig line per reference plus every reference's records, and the three-column
    depth file — all assembled from runs of the plain CLI on every reference alone.  Without the flag the same command
    still stops at the multi-contig ValueError."""
    tmp = str(tmp_path)
    contigs = _flu_contigs(tmp, with_tiny=False)
    paths = _write_multi(tmp, contigs, unplaced_every=50)
    out = os.path.join(tmp, "S")
    argv = ["-i", paths["bam"], "-ref", paths["fasta"], "-gff", paths["gff"], "-cov", "30", "-name", "S", "-o", out + ".fasta",
            "-vcf", out + ".vcf", "-ogff", out + ".gff", "-doc", out + ".tsv", "-t", "2"]
    _cli(["--all-contigs"] + argv, monkeypatch)
    single = _single_runs(contigs, tmp, "S", monkeypatch)
    names = [c["name"] for c in contigs]
    got = {e: open(f"{out}.{e}").read() for e in ("fasta", "vcf", "gff", "tsv")}
    assert got["fasta"] == "".join(single[n]["fasta"] for n in names)
    assert got["fasta"].count(">") == len(names)
    assert got["gff"] == "##gff-version 3\n" + "".join(single[n]["gff"].split("\n", 1)[1] for n in names)
    assert got["tsv"] == "".join(f"{n}\t{l}\n" for n in names for l in single[n]["tsv"].splitlines())
    assert _vcf_records(got["vcf"]) == [l for n in names for l in _vcf_records(single[n]["vcf"])]
    assert [l for l in got["vcf"].splitlines() if l.startswith("##contig")] == [f"##contig=<ID={n}>" for n in names]
    assert _norm_vcf_header(got["vcf"]) == _norm_vcf_header(single[names[0]]["vcf"])
    assert any(l.rstrip().endswith(";INDEL") for l in _vcf_records(got["vcf"]))   # insertions and the deletion reach the VCF
    with pytest.raises(ValueError, match="multi-contig"):
        _cli(argv, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["quirk", "mini_illumina", "mini_ont", "mini_long", "mini_overlap"])
def test_cli_all_contigs_on_single_reference_goldens(name, tmp_path, monkeypatch):
    """A BAM with one reference ('ref'): --all-contigs writes what the plain CLI writes with -name {name}_ref (the depth
    file with the reference's name in front)."""
    import json

    mincov = json.load(open(f"{GOLD}/{name}.json"))["mincov"]
    runs = {}
    for mode in ("multi", "single"):
        out = str(tmp_path / mode)
        argv = ["-i", f"{GOLD}/{name}.bam", "-ref", f"{GOLD}/{name}.fasta", "-gff", f"{GOLD}/{name}.gff", "-cov", str(mincov),
                "-name", name if mode == "multi" else f"{name}_ref", "-o", out + ".fasta", "-vcf", out + ".vcf", "-ogff", out + ".gff",
                "-doc", out + ".tsv", "-t", "2"]
        _cli((["--all-contigs"] if mode == "multi" else []) + argv, monkeypatch)
        runs[mode] = {e: open(f"{out}.{e}").read() for e in ("fasta", "vcf", "gff", "tsv")}
    m, s = runs["multi"], runs["single"]
    assert m["fasta"] == s["fasta"] and m["gff"] == s["gff"]
    assert m["tsv"] == "".join(f"ref\t{l}\n" for l in s["tsv"].splitlines())
    strip = lambda t: [l for l in t.splitlines() if not l.startswith(("##fileDate", "##source"))]     # noqa: E731
    assert strip(m["vcf"]) == strip(s["vcf"])


@pytest.mark.gpu
def test_long_header_same_results_and_launches(flu, tmp_path):
    """The same records under a header of 6000 more references (every one in the FASTA): same frames and insertion
    calls, and BuildIndexContigs + ListInsertsContigs launch as many kernels as under the fixture's header."""
    from trueconsense_b200 import Events, gpu, indexing

    tmp = str(tmp_path)
    decoys = [(f"decoy_{i:05d}_with_a_long_name", 10 + i % 23) for i in range(6000)]
    bam = os.path.join(tmp, "long.bam")
    _multi_bam(bam, flu["contigs"], extra_refs=decoys, unplaced_every=97)
    fasta = os.path.join(tmp, "long.fasta")
    with open(fasta, "w") as fh:
        fh.write(open(flu["fasta"]).read())
        for n, l in decoys:
            fh.write(f">{n}\n{'ACGT' * (l // 4)}{'A' * (l % 4)}\n")
    ctx = gpu.default_context()

    def run(b, f):
        h = indexing.Readbam(b)
        frames = indexing.BuildIndexContigs(h, f)
        indexes = {n: fr.to_dict("index") for n, fr in frames.items()}
        h = indexing.Readbam(b)
        l0 = ctx.launches
        frames = indexing.BuildIndexContigs(h, f)
        ins = Events.ListInsertsContigs(indexes, 30, h)
        return frames, ins, ctx.launches - l0

    run(flu["bam"], flu["fasta"]), run(bam, fasta)         # warm-up: buffers sized, nothing grows below
    f8, i8, n8 = run(flu["bam"], flu["fasta"])
    fl, il, nl = run(bam, fasta)
    assert len(fl) == len(f8) + 6000
    for n in f8:
        assert fl[n].equals(f8[n]) and il[n] == i8[n], n
    assert all(not il[n][0] and int(fl[n]["coverage"].sum()) == 0 for n, _ in decoys[:50])
    assert nl == n8, (nl, n8)


def _two_refs(tmp, a_recs, a_len, b_len=600, a_bam_len=None):
    from trueconsense_b200 import synth

    seq_b, feats_b = synth.make_genome(b_len, 3, "sars2")
    b = synth.generate_reads(synth.SynthParams(seed=3, n_reads=300, ref_len=b_len, read_len=100), seq_b)
    seq_a = synth.make_genome(a_len, 4, "none")[0]
    ca = {"name": "a", "seq": seq_a, "feats": [], "bam_len": a_bam_len or a_len}
    cb = {"name": "b", "seq": seq_b, "feats": feats_b}
    _write_contig(tmp, ca, _hand_batch(a_recs(seq_a)))
    _write_contig(tmp, cb, _with_mates(b, np.random.default_rng(1), 0.0))
    return [ca, cb]


@pytest.mark.gpu
def test_errors(tmp_path, monkeypatch):
    from trueconsense_b200 import gpu, indexing
    from trueconsense_b200.reads import ReadBatch

    tmp = str(tmp_path)
    # a read running past its reference's end (the FASTA's length): TC_ERR_RANGE naming the reference, as BuildIndex says
    cs = _two_refs(tmp, lambda s: [dict(pos=0, cigar="100M", seq=s[:100]), dict(pos=450, cigar="60M", seq=s[:60])], 500, a_bam_len=600)
    with open(cs[0]["fasta"], "w") as fh:
        fh.write(">a\n" + cs[0]["seq"][:480] + "\n")
    cs[0]["seq"] = cs[0]["seq"][:480]
    p = _write_multi(tmp, cs, stem="past")
    with pytest.raises(gpu.TcError) as ei:
        indexing.BuildIndexContigs(p["bam"], p["fasta"])
    assert ei.value.code == -7 and "'a'" in str(ei.value)
    with pytest.raises(gpu.TcError) as ei:
        indexing.BuildIndex(cs[0]["bam"], cs[0]["fasta"])
    assert ei.value.code == -7
    # unsorted: the second reference's records first
    p = _write_multi(tmp, cs, stem="unsorted", order=[1, 0])
    with pytest.raises(ValueError, match="Unsorted input. Pileup aborts"):
        indexing.BuildIndexContigs(p["bam"], p["fasta"])
    # lengths adding up to more than INT32_MAX, straight to the binding
    ctx = gpu.default_context()
    d = ctx.upload(ReadBatch.from_records([dict(pos=0, cigar="4M", seq="ACGT")]))
    with pytest.raises(gpu.TcError) as ei:
        ctx.reads_to_contig_coords(d, [2**31 - 1, 5], [0, 1, 1])
    assert ei.value.code == -2 and d.contig_start is None
    # a header reference missing from the FASTA
    cs = _two_refs(tmp, lambda s: [dict(pos=0, cigar="100M", seq=s[:100])], 500)
    p = _write_multi(tmp, cs, stem="nofasta")
    with open(p["fasta"], "w") as fh:
        fh.write(">b\n" + cs[1]["seq"] + "\n")
    with pytest.raises(ValueError, match="'a'"):
        indexing.BuildIndexContigs(p["bam"], p["fasta"])
    # BuildIndex on the multi-reference BAM: the old refusal
    p = _write_multi(tmp, cs, stem="multi")
    with pytest.raises(ValueError, match="multi-contig"):
        indexing.BuildIndex(p["bam"], p["fasta"])
    # >= 15 % deletions on a reference's last column under a non-X primary: KeyError, as on that reference alone
    L = 400

    def tail_del(s):
        recs = [dict(pos=L - 51, cigar="50M1D", seq=s[L - 51:L - 1], qname=f"d{j}") for j in range(20)]
        return recs + [dict(pos=L - 51, cigar="51M", seq=s[L - 51:], qname=f"m{j}") for j in range(80)]

    cs = _two_refs(tmp, tail_del, L)
    p = _write_multi(tmp, cs, stem="taildel")
    out = os.path.join(tmp, "T")
    with pytest.raises(KeyError):
        _cli(["--all-contigs", "-i", p["bam"], "-ref", p["fasta"], "-gff", p["gff"], "-cov", "30", "-name", "T", "-o", out + ".fasta"],
             monkeypatch)
    assert not os.path.exists(out + ".fasta")
    with pytest.raises(KeyError):
        _cli(["-i", cs[0]["bam"], "-ref", cs[0]["fasta"], "-gff", cs[0]["gff"], "-cov", "30", "-name", "T_a", "-o", out + "_a.fasta"],
             monkeypatch)
