"""SAM text straight from the aligner, read with ``Context.sam_file_to_device`` / a ``.sam`` path: the GPU turns every line
into the BAM record ``samtools view -b`` would write and the BAM route's steps follow, so every result must equal what the
BAM route computes for the same records.  The SAM inputs are written here at test time: from a BAM's records as
``samtools view -h`` prints them (``sam_line``), or by hand; a small SAM -> BAM encoder (``sam_record``) restates the
conversion rules for hand-written lines, so each device result is compared with the BAM route over the encoded file."""
import json
import os
import re
import struct

import numpy as np
import pytest

from bamfiles import (MM2_AUX, assert_same_arrays, bam_header, bam_to_sam, bgzf, dev_arrays, mini_argv, refs_of, run_cli, sam_header,
                      sam_line, sam_record, split)
from conftest import GOLD, load_golden_counts

MINIS = ("quirk", "mini_illumina", "mini_ont", "mini_long", "mini_overlap")
STATS = ("aligned_bases", "max_ref_span", "unsorted", "multi_contig", "sorted", "n_seq_words", "n_cigar_ops")


# ---------------------------------------------------------------------------- fixture helpers (host only)
def write_pair(tmp, stem, refs, lines, newline_at_end=True):
    """Hand-written SAM lines as a .sam file and, encoded by ``sam_record``, as a .bam file (RNAME '*' lines left out)."""
    names = [n for n, _ in refs]
    sam, bam = os.path.join(tmp, stem + ".sam"), os.path.join(tmp, stem + ".bam")
    body = b"".join(lines)
    with open(sam, "wb") as fh:
        fh.write(sam_header(refs) + (body if newline_at_end else body[:-1]))
    recs = [r for r in (sam_record(l, names) for l in lines) if r is not None]
    bgzf(bam, bam_header(refs) + b"".join(recs))
    return sam, bam


def _snapshot(ctx, d):
    return (dev_arrays(ctx, d), {k: getattr(d.stats, k) for k in STATS}, d.ref_names, d.ref_lens,
            d.info["n_records"], d.info["n_dropped_unplaced"], None if d.first_read is None else d.first_read.tolist())


def _assert_same(a, b, what=""):
    assert_same_arrays(a[0], b[0], what)
    assert a[1:] == b[1:], what


REFS = [(b"chr1", 5000), (b"chr2", 3000)]


def _good_lines(n, rname=b"chr1", start=100, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for j in range(n):
        seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), 40).tobytes()
        out.append(b"g%d\t0\t%s\t%d\t60\t40M\t*\t0\t0\t%s\t%s\n" % (j, rname, start + 3 * j, seq, b"I" * 40))
    return out


# ---------------------------------------------------------------------------- CPU tests
def test_read_sam_header(tmp_path):
    from trueconsense_b200 import bamio

    p = tmp_path / "h.sam"
    p.write_bytes(b"@HD\tVN:1.6\n@SQ\tSN:b\tLN:7\tM5:x\n@RG\tID:r\n@SQ\tLN:9\tSN:a\n@PG\tID:p\n@CO\tfree text\n"
                  b"r\t4\t*\t0\t0\t*\t*\t0\t0\tA\t*\n")
    names, lens, off, no = bamio.read_sam_header(str(p))
    assert (names, lens, no) == (["b", "a"], [7, 9], 7)
    assert p.read_bytes()[off:].startswith(b"r\t4")
    # header only, and an empty file
    p.write_bytes(b"@SQ\tSN:x\tLN:2147483647\n")
    assert bamio.read_sam_header(str(p)) == (["x"], [2147483647], p.stat().st_size, 2)
    p.write_bytes(b"")
    assert bamio.read_sam_header(str(p)) == ([], [], 0, 1)
    for bad, what in ((b"@SQ\tSN:a\tLN:5\n@SQ\tSN:a\tLN:6\n", "line 2: reference 'a' is listed twice"),
                      (b"@HD\tVN:1.6\n@SQ\tSN:a\n", "line 2: reference 'a' needs a length"),
                      (b"@SQ\tSN:a\tLN:0\n", "line 1: reference 'a' needs a length"),
                      (b"@SQ\tSN:a\tLN:2147483648\n", "needs a length"),
                      (b"@SQ\tSN:a\tLN:12x\n", "needs a length"),
                      (b"@SQ\tLN:5\n", "line 1: @SQ line without a reference name")):
        p.write_bytes(bad)
        with pytest.raises(OSError, match=re.escape(what)):
            bamio.read_sam_header(str(p))


def test_read_sam_header_6000_references(tmp_path):
    from trueconsense_b200 import bamio

    refs = [(b"decoy_%05d_with_a_long_name" % i, 10 + i % 23) for i in range(6000)]
    p = tmp_path / "many.sam"
    p.write_bytes(sam_header(refs) + b"".join(_good_lines(3, rname=refs[4321][0])))
    names, lens, off, no = bamio.read_sam_header(str(p))
    assert names == [n.decode() for n, _ in refs] and lens == [l for _, l in refs]
    assert no == 6003 and p.read_bytes()[off:].startswith(b"g0\t")


def test_cli_accepts_sam(tmp_path):
    from trueconsense_b200 import TrueConsense, indexing

    sam = tmp_path / "a.sam"; fa = tmp_path / "r.fasta"; gff = tmp_path / "f.gff"; txt = tmp_path / "a.txt"
    for p in (sam, fa, gff, txt):
        p.write_text("x")
    base = ["-i", str(sam), "-ref", str(fa), "-gff", str(gff), "-cov", "30", "-name", "s", "-o", str(tmp_path / "c.fa")]
    assert TrueConsense.GetArgs(base).input == str(sam)
    o = TrueConsense.GetArgs(base + ["--sort-input", "--all-contigs"])
    assert o.sort_input and o.all_contigs
    with pytest.raises(SystemExit) as e:
        TrueConsense.GetArgs(["-i", str(txt)] + base[2:])
    assert e.value.code == 2
    assert indexing.Readbam(str(sam), sort=True).is_sam
    assert not indexing.Readbam(str(tmp_path / "a.bam")).is_sam


def test_sam_handle_header_without_a_device(tmp_path):
    from trueconsense_b200 import indexing

    p = tmp_path / "x.sam"
    p.write_bytes(sam_header(REFS) + b"".join(_good_lines(2)))
    h = indexing.Readbam(str(p))
    assert h.references == ("chr1", "chr2") and h.lengths == (5000, 3000) and h.ref_len == 5000
    with pytest.raises(NotImplementedError, match="SAM"):
        h.reads


def test_sam_helpers_round_trip(tmp_path):
    """The fixture helpers themselves: every golden record printed as SAM and encoded back is the record (bin aside)."""
    from trueconsense_b200 import build

    build.build_host()
    for name in MINIS:
        head, recs = split(f"{GOLD}/{name}.bam")
        names = [n for n, _ in refs_of(head)]
        for r in recs:
            line = sam_line(r, names, MM2_AUX % 3)
            assert line.count(b"\t") == 20 and line.endswith(b"\n")
            assert sam_record(line, names) == r[:14] + b"\0\0" + r[16:], name
    line = b"q\t0\tchr1\t1\t0\t3M\t*\t0\t0\t=aU\t*\n"
    assert sam_record(line, [b"chr1"])[-5:] == bytes([0x01, 0xF0, 0xFF, 0xFF, 0xFF])


# ---------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import build, gpu

    build.build_host()
    if not os.path.exists(build.CUDA_LIB):
        build.build_cuda()
    return gpu.default_context()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "mm2_fields", "lower_case"])
@pytest.mark.parametrize("name", MINIS)
def test_goldens_equal_bam_route(ctx, name, variant, tmp_path):
    """The SAM of a golden BAM: every read array, the stats and the header equal the BAM route's; BuildIndex over it gives
    the golden count table."""
    from trueconsense_b200 import indexing

    bam = f"{GOLD}/{name}.bam"
    sam = bam_to_sam(bam, str(tmp_path / f"{name}.sam"), aux=variant == "mm2_fields", lower=variant == "lower_case")
    want = _snapshot(ctx, ctx.bam_file_to_device(bam, contig_ranges=True))
    d = ctx.sam_file_to_device(sam, contig_ranges=True)
    assert d.info["n_lines"] == want[4] and d.info["sam_bytes"] == os.path.getsize(sam) and d.info["reordered"] is False
    _assert_same(_snapshot(ctx, d), want, name)
    frame = indexing.BuildIndex(sam, f"{GOLD}/{name}.fasta")
    assert np.array_equal(np.stack([frame[c].to_numpy() for c in indexing.COLUMNS]), load_golden_counts(name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", MINIS)
def test_cli_parity(ctx, name, tmp_path, monkeypatch):
    """main() over the golden's SAM writes the reference CLI's golden files (the raising case raises the same type)."""
    from trueconsense_b200 import TrueConsense

    sam = bam_to_sam(f"{GOLD}/{name}.bam", str(tmp_path / f"{name}.sam"), aux=True)
    status = json.load(open(f"{GOLD}/cli_{name}.status.json"))
    out = str(tmp_path / f"cli_{name}")
    argv = mini_argv(name, sam) + ["-o", out + ".fasta", "-vcf", out + ".vcf", "-ogff", out + ".gff",
                                    "-doc", out + ".cov.tsv", "-t", "2"]
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


@pytest.mark.gpu
@pytest.mark.parametrize("name", MINIS)
def test_shuffled_sam_sorted_on_device(ctx, name, tmp_path, monkeypatch):
    """A shuffled SAM with sort=True / --sort-input == the same shuffle as a BAM with sort=True: arrays, insertion calls on
    every column and the CLI's files.  Without sort: the unsorted refusal."""
    from trueconsense_b200 import indexing

    bam = f"{GOLD}/{name}.bam"
    head, recs = split(bam)
    order = np.random.default_rng(11).permutation(len(recs))
    sam = bam_to_sam(bam, str(tmp_path / "shuf.sam"), aux=True, order=order)
    shuf_bam = str(tmp_path / "shuf.bam")
    bgzf(shuf_bam, head + b"".join(recs[i] for i in order), (3000, 65280))
    L = load_golden_counts(name).shape[1]
    b = ctx.bam_file_to_device(shuf_bam, sort=True)
    want = _snapshot(ctx, b)
    want_cols = ctx.extract_inserts(b, L, np.arange(1, L + 1, dtype=np.int32))
    d = ctx.sam_file_to_device(sam, sort=True)
    assert d.info["reordered"] is True
    _assert_same(_snapshot(ctx, d), want, name)
    assert ctx.extract_inserts(d, L, np.arange(1, L + 1, dtype=np.int32)) == want_cols
    with pytest.raises(ValueError, match="Unsorted input. Pileup aborts"):
        indexing.BuildIndex(sam, f"{GOLD}/{name}.fasta")
    got = run_cli(["--sort-input"] + mini_argv(name, sam), str(tmp_path / "s"), monkeypatch)
    exp = run_cli(["--sort-input"] + mini_argv(name, shuf_bam), str(tmp_path / "b"), monkeypatch)
    assert got == exp


def _multi_ref(tmp, n_decoys=40):
    """Three references with reads (an insertion, a deletion, paired reads) among n_decoys + 3 references, the FASTA and the
    GFF rows of the three: (BAM header, refs, {slot: records}, fasta, gff)."""
    from trueconsense_b200 import bamio, synth

    real = {}
    slots = [0, n_decoys // 2 + 1, n_decoys + 2]
    for k, (L, seed) in enumerate(((2341, 1), (1565, 2), (890, 3))):
        seq, feats = synth.make_genome(L, 300 + seed, "sars2")
        a = feats[0]["start"] - 1
        vs = [synth.Variant(a + 400, synth.VAR_INS, 3, 7, 0.9)] if k != 1 else [synth.Variant(a + 60, synth.VAR_DEL, 3, 0, 0.85)]
        p = synth.SynthParams(seed=400 + seed, n_reads=L * 60 // 150, ref_len=L, read_len=150, paired=(k != 2), insert_mean=300,
                              insert_sd=40, sub_rate=0.01, softclip_rate=0.05, softclip_max=8, variants=vs)
        one = os.path.join(tmp, f"c{k}.bam")
        bamio.write_bam(one, synth.generate_reads(p, seq), f"c{k}", L)
        recs = []
        for r in split(one)[1]:
            r = bytearray(r)
            struct.pack_into("<i", r, 4, slots[k])
            if struct.unpack_from("<i", r, 24)[0] >= 0:
                struct.pack_into("<i", r, 24, slots[k])
            recs.append(bytes(r))
        real[slots[k]] = {"name": f"c{k}", "seq": seq, "feats": feats, "recs": recs}
    refs = [(real[i]["name"].encode(), len(real[i]["seq"])) if i in real else (b"decoy_%05d" % i, 10 + i % 23)
            for i in range(n_decoys + 3)]
    fasta = os.path.join(tmp, "multi.fasta")
    with open(fasta, "w") as fh:
        for i, (n, l) in enumerate(refs):
            s = real[i]["seq"] if i in real else "ACGT" * (l // 4) + "A" * (l % 4)
            fh.write(f">{n.decode()}\n" + "".join(s[j:j + 60] + "\n" for j in range(0, len(s), 60)))
    gff = os.path.join(tmp, "multi.gff")
    with open(gff, "w") as fh:
        fh.write("##gff-version 3\n")
        for i in slots:
            c = real[i]
            for f in c["feats"]:
                attrs = f"ID=cds-{c['name']}-{f['name']};Name={f['name']};gbkey=CDS"
                fh.write("\t".join([c["name"], "synthetic", "CDS", str(f["start"]), str(f["end"]), ".", f["strand"], "0", attrs]) + "\n")
    return bam_header(refs, b"@HD\tVN:1.6\tSO:unsorted\n"), refs, real, slots, fasta, gff


@pytest.mark.gpu
def test_multi_reference_interleaved(ctx, tmp_path, monkeypatch):
    """An interleaved multi-reference SAM with --all-contigs --sort-input == its BAM counterpart: frames, layout, insertion
    calls and the four files; a plain sorted one with --all-contigs alone too.  Outside --all-contigs: the multi-contig
    refusal."""
    from trueconsense_b200 import Events, indexing

    tmp = str(tmp_path)
    head, refs, real, slots, fasta, gff = _multi_ref(tmp)
    rng = np.random.default_rng(9)
    body = []
    for i in reversed(slots):
        recs = real[i]["recs"]
        body += [recs[j] for j in rng.permutation(len(recs))]
    names = [n for n, _ in refs]
    for stem, rs, flags in (("shuf", body, ["--sort-input"]), ("sorted", [r for i in slots for r in real[i]["recs"]], [])):
        bam, sam = os.path.join(tmp, stem + ".bam"), os.path.join(tmp, stem + ".sam")
        bgzf(bam, head + b"".join(rs), (65280, 3000))
        with open(sam, "wb") as fh:
            fh.write(sam_header(refs, b"@HD\tVN:1.6\tSO:unsorted\n") + b"".join(sam_line(r, names, MM2_AUX % 1) for r in rs))
        sort = bool(flags)
        hs, hb = indexing.Readbam(sam, sort=sort), indexing.Readbam(bam, sort=sort)
        fs, fb = indexing.BuildIndexContigs(hs, fasta), indexing.BuildIndexContigs(hb, fasta)
        assert list(fs) == list(fb) and len(fs) == len(refs)
        for n in fs:
            assert fs[n].equals(fb[n]), n
        lens = [len(fs[n]) for n in fs]
        _, lay_s = hs.device_reads_contigs(list(fs), lens)
        _, lay_b = hb.device_reads_contigs(list(fs), lens)
        assert np.array_equal(lay_s.first_read, lay_b.first_read) and np.array_equal(lay_s.start, lay_b.start)
        idx = {n: f.to_dict("index") for n, f in fs.items()}
        ins = Events.ListInsertsContigs(idx, 30, hs)
        assert ins == Events.ListInsertsContigs(idx, 30, hb) and ins["c0"][0]
        base = ["-ref", fasta, "-gff", gff, "-cov", "30", "-name", "S", "--all-contigs"] + flags
        got = run_cli(["-i", sam] + base, os.path.join(tmp, stem + "_s"), monkeypatch)
        exp = run_cli(["-i", bam] + base, os.path.join(tmp, stem + "_b"), monkeypatch)
        assert isinstance(got, dict) and got == exp
        assert got["fasta"].count(">") == len(refs)
        with pytest.raises(ValueError, match="multi-contig"):
            indexing.BuildIndex(indexing.Readbam(sam, sort=True), fasta)


@pytest.mark.gpu
def test_dialect(ctx, tmp_path):
    """Hand-written lines over the corners of the format == the encoder's BAM through the BAM route."""
    ctxt = str(tmp_path)
    lines = [
        b"a1\t0\tchr1\t10\t60\t4M\t*\t0\t0\tAC=T\tIIII\n",                              # '=' in SEQ
        b"a2\t16\tchr1\t11\t0\t16M\t=\t300\t-305\t=ACMGRSVTWYHKDBN\t!!!!!!!!!!!!!!!~\n",  # every IUPAC code, RNEXT '=', QUAL edges
        b"a3\t1\tchr1\t12\t30\t6M\tchr2\t55\t0\tXUZ.-*\t*\n",                            # non-IUPAC letters -> N; QUAL '*'; RNEXT a name
        b"a4\t0\tchr1\t12\t30\t3S4M1I2M1D3M2H\t*\t0\t0\tacgtacgtacgta\tABCDEFGHIJKLM\n",  # lower case, every op
        b"a5\t0\tchr1\t13\t255\t5M\t*\t0\t0\t*\t*\n",                                   # SEQ '*' with a CIGAR
        b"*\t0\tchr1\t14\t60\t*\t*\t0\t2147483647\tACGT\tIIII\n",                         # QNAME '*', CIGAR '*', TLEN max
        b"a7\t4\tchr1\t15\t0\t*\t=\t15\t0\tACGTN\t#####\n",                              # unmapped with an RNAME: kept
        b"a8\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\tIIII\n",                                    # RNAME '*': dropped
        b"a9\t65535\tchr1\t20\t0\t2=1X1=\tchr1\t0\t-2147483648\tACGT\tIIII\tNM:i:1\tCG:B:I,64\n",   # PNEXT 0; CG:B with a real CIGAR
        b"%s\t0\tchr2\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n" % (b"q" * 254),                 # longest QNAME, another reference
        b"a11\t0\tchr2\t0\t60\t4M\t*\t0\t0\tACGT\tIIII\tXP:Z:tab-free text\n",            # POS 0 with an RNAME
        b"a12\t8\t*\t0\t0\t*\tchr1\t5\t0\t*\t*\n",                                      # RNAME '*' with an RNEXT: dropped
        b"a13\t0\tchr2\t40\t007\t4M\t*\t0\t+12\tACGT\tIIII\n",                     # leading zeros, '+' in TLEN
    ]
    for newline_at_end in (True, False):
        sam, bam = write_pair(ctxt, f"d{int(newline_at_end)}", REFS, lines, newline_at_end)
        want = _snapshot(ctx, ctx.bam_file_to_device(bam))
        d = ctx.sam_file_to_device(sam)
        _assert_same(_snapshot(ctx, d), (want[0], want[1], want[2], want[3], len(lines), 2, None))
        assert d.info["n_lines"] == len(lines) and d.n_reads == len(lines) - 2
    # an empty body, a header-only file without its last newline, a file without anything
    for text in (sam_header(REFS), sam_header(REFS)[:-1], b""):
        p = os.path.join(ctxt, "empty.sam")
        open(p, "wb").write(text)
        d = ctx.sam_file_to_device(p, contig_ranges=True, sort=True)
        assert d.n_reads == 0 and d.info["n_records"] == 0
        assert d.ref_names == ([] if not text else ["chr1", "chr2"])
    # one line of more than 300 KB, between two short ones, with and without a newline behind it
    rng = np.random.default_rng(5)
    seq = rng.choice(np.frombuffer(b"ACGTN", np.uint8), 160_000).tobytes()
    qual = bytes(rng.integers(33, 75, 160_000, dtype=np.uint8))
    long = b"long\t0\tchr1\t1\t60\t100S159800M10I90S\t*\t0\t0\t%s\t%s\tNM:i:10\n" % (seq, qual)
    short = _good_lines(2, start=50)
    for newline_at_end in (True, False):
        sam, bam = write_pair(ctxt, "long", [(b"chr1", 170_000)], [short[0], long, short[1]][: 3 if newline_at_end else 2],
                              newline_at_end)
        _assert_same(_snapshot(ctx, ctx.sam_file_to_device(sam)), _snapshot(ctx, ctx.bam_file_to_device(bam)))


@pytest.mark.gpu
def test_lines_across_tile_edges(ctx, tmp_path):
    """Newlines at every offset around the line index's 4 KiB tiles and 16-byte loads: a padding field grows one byte a line
    over a whole tile, and lines are placed so that their newline lands just before, on and just behind tile edges."""
    rng = np.random.default_rng(3)
    lines = []

    def make(pad):
        k = len(lines)
        return b"t%05d\t%d\tchr1\t%d\t60\t8M\t*\t0\t0\t%s\tIIIIIIII\tXP:Z:%s\n" % (
            k, 16 * (k % 2), 1 + k // 3, rng.choice(np.frombuffer(b"ACGT", np.uint8), 8).tobytes(), b"p" * pad)

    for pad in range(300):              # one byte longer each line: newlines at every offset modulo a 16-byte load
        lines.append(make(pad))
    body_len = sum(map(len, lines))
    for t in range(body_len // 4096 + 1, body_len // 4096 + 40):
        for d in (-17, -16, -2, -1, 0, 1, 15, 16):
            end = 4096 * t + d + 1          # the byte behind a newline at offset 4096 t + d
            if end - body_len < len(make(0)):
                continue
            while end - body_len > len(make(0)) + 4000:
                lines.append(make(3000))
                body_len += len(lines[-1])
            lines.append(make(end - body_len - len(make(0))))
            body_len += len(lines[-1])
            assert body_len == end
    sam, bam = write_pair(str(tmp_path), "tiles", REFS, lines)
    d = ctx.sam_file_to_device(sam)
    assert d.n_reads == len(lines) and d.info["n_lines"] == len(lines)
    _assert_same(_snapshot(ctx, d), _snapshot(ctx, ctx.bam_file_to_device(bam)))


@pytest.mark.gpu
def test_size_200k_config2_slice(ctx, tmp_path):
    """A 200 k-read config-2 slice as SAM (minimap2-like fields) == its BAM: arrays, stats, count table."""
    from trueconsense_b200 import bamio, synth

    w = synth.config(1, scale=0.1)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    assert b.n_reads == 200_000
    bam = str(tmp_path / "cfg2.bam")
    bamio.write_bam(bam, b, "ref", L)
    sam = bam_to_sam(bam, str(tmp_path / "cfg2.sam"), aux=True)
    want = _snapshot(ctx, ctx.bam_file_to_device(bam))
    exp_counts = ctx.pileup_counts(b, L)
    d = ctx.sam_file_to_device(sam)
    assert d.n_reads == b.n_reads
    _assert_same(_snapshot(ctx, d), want)
    assert np.array_equal(ctx.pileup_counts(d, L), exp_counts)


BAD = {
    "fields": (b"b\t0\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\n", "fewer than 11 tab-separated fields"),
    "flag_text": (b"b\t0x10\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "FLAG is not a number"),
    "flag_range": (b"b\t65536\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "FLAG is not a number"),
    "pos_negative": (b"b\t0\tchr1\t-1\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "POS is not a number"),
    "pos_range": (b"b\t0\tchr1\t2147483648\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "POS is not a number"),
    "mapq_range": (b"b\t0\tchr1\t1\t256\t4M\t*\t0\t0\tACGT\tIIII\n", "MAPQ is not a number"),
    "pnext_text": (b"b\t0\tchr1\t1\t60\t4M\t*\tx\t0\tACGT\tIIII\n", "PNEXT is not a number"),
    "tlen_range": (b"b\t0\tchr1\t1\t60\t4M\t*\t0\t2147483648\tACGT\tIIII\n", "TLEN is not a number"),
    "rname_unknown": (b"b\t0\tchr3\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "RNAME names no reference"),
    "rname_prefix": (b"b\t0\tchr\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n", "RNAME names no reference"),
    "rnext_unknown": (b"b\t0\tchr1\t1\t60\t4M\tchr11\t5\t0\tACGT\tIIII\n", "RNEXT is not"),
    "cigar_op": (b"b\t0\tchr1\t1\t60\t2M2Q\t*\t0\t0\tACGT\tIIII\n", "bad CIGAR"),
    "cigar_no_length": (b"b\t0\tchr1\t1\t60\tM4M\t*\t0\t0\tACGT\tIIII\n", "bad CIGAR"),
    "cigar_zero": (b"b\t0\tchr1\t1\t60\t0M4M\t*\t0\t0\tACGT\tIIII\n", "bad CIGAR"),
    "cigar_too_long": (b"b\t0\tchr1\t1\t60\t268435456M\t*\t0\t0\t*\t*\n", "bad CIGAR"),
    "cigar_trailing": (b"b\t0\tchr1\t1\t60\t4M4\t*\t0\t0\tACGT\tIIII\n", "bad CIGAR"),
    "cigar_ops": (b"b\t0\tchr1\t1\t60\t%s\t*\t0\t0\t*\t*\n" % (b"1M1I" * 32768), "more than 65535 CIGAR operations"),
    "cigar_seq": (b"b\t0\tchr1\t1\t60\t5M\t*\t0\t0\tACGT\tIIII\n", "CIGAR and SEQ lengths differ"),
    "qual_seq": (b"b\t0\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\tIII\n", "QUAL and SEQ lengths differ"),
    "qual_without_seq": (b"b\t0\tchr1\t1\t60\t4M\t*\t0\t0\t*\tIIII\n", "QUAL and SEQ lengths differ"),
    "qual_char": (b"b\t0\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\tII I\n", "QUAL character below '!'"),
    "qname_long": (b"%s\t0\tchr1\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n" % (b"q" * 255), "QNAME must hold 1 to 254"),
    "empty_line": (b"\n", "empty line"),
    "header_late": (b"@CO\tlate\n", "header line after the first record"),
    "cg_placeholder": (b"b\t0\tchr1\t1\t60\t4S9N\t*\t0\t0\tACGT\tIIII\tCG:B:I,144\n", "CG:B"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(BAD))
def test_malformed_line(ctx, case, tmp_path):
    """A bad line among good ones: OSError naming the file, the line (1-based in the file) and the reason; the context then
    converts the next file as before."""
    bad, reason = BAD[case]
    good = _good_lines(300)
    k = 137
    path = str(tmp_path / "bad.sam")
    header = sam_header(REFS)
    with open(path, "wb") as fh:
        fh.write(header + b"".join(good[:k] + [bad] + good[k:]))
    line_no = header.count(b"\n") + k + 1
    with pytest.raises(OSError) as ei:
        ctx.sam_file_to_device(path)
    assert str(ei.value).startswith(f"{path}: line {line_no}: ") and reason in str(ei.value), str(ei.value)
    sam, bam = write_pair(str(tmp_path), "ok", REFS, good)
    _assert_same(_snapshot(ctx, ctx.sam_file_to_device(sam)), _snapshot(ctx, ctx.bam_file_to_device(bam)))


@pytest.mark.gpu
def test_first_bad_line_is_named(ctx, tmp_path):
    """Of several bad lines the first is named, whatever its reason; through Readbam the error is the same OSError."""
    from trueconsense_b200 import indexing

    good = _good_lines(2000)
    lines = good[:1500] + [BAD["qual_char"][0]] + good[1500:1700] + [BAD["fields"][0]] + good[1700:]
    lines[900] = BAD["cigar_op"][0]
    path = str(tmp_path / "two.sam")
    header = sam_header(REFS)
    open(path, "wb").write(header + b"".join(lines))
    line_no = header.count(b"\n") + 901
    with pytest.raises(OSError, match=f"line {line_no}: bad CIGAR"):
        ctx.sam_file_to_device(path)
    with pytest.raises(OSError, match=f"line {line_no}: bad CIGAR"):
        indexing.Readbam(path).device_reads()
