"""Amplicon primers clipped off the aligned reads on the GPU (``--primers``, ``tc_bam_clip_primers``).

The CPU tests pin the rule (DESIGN §4) through ``oracle/primer_clip.py`` with hand-derived cases and invariants over random
CIGARs, and check the BED reader and the flags.  The GPU tests compare the clip's record bytes with the oracle's, and every
decode route with primers against the plain decode of a BAM this file writes from the oracle's clipped and sorted records —
down to the CLI's four output files."""
import json
import os
import struct

import numpy as np
import pytest

from conftest import GOLD
from oracle import primer_clip as pc
from test_sam_input import _sam_header, sam_line
from test_sort_input import _multi_ref_files, _split, _write

MINIS = ("quirk", "mini_illumina", "mini_ont", "mini_long", "mini_overlap")
FIELDS = (("pos", np.int32), ("flag", np.uint16), ("mapq", np.uint8), ("l_seq", np.int32), ("seq_off", np.uint32),
          ("cigar_off", np.uint32), ("seq4", np.uint32), ("qual", np.uint8), ("cigar", np.uint32), ("qname_hash", np.uint64),
          ("mpos", np.int32), ("isize", np.int32))
OPS = "MIDNSHP=X"


# ---------------------------------------------------------------------------- helpers (host only)
def _ops(cigar):
    import re

    return [(OPS.index(o), int(n)) for n, o in re.findall(r"(\d+)([MIDNSHP=X])", cigar)]


def _str(ops):
    return "".join(f"{n}{OPS[o]}" for o, n in ops)


def make_rec(pos, cigar, flag=0, tid=0, name=b"r", mtid=-1, mpos=-1, tlen=0, aux=b"", seed=0, bin_=4680):
    """A BAM record (block_size included) with random SEQ / QUAL of the CIGAR's query length."""
    ops = _ops(cigar) if isinstance(cigar, str) else cigar
    l_seq = sum(n for o, n in ops if o in pc.QUERY)
    rng = np.random.default_rng(seed)
    seq = rng.integers(0, 256, (l_seq + 1) // 2, dtype=np.uint8).tobytes()
    qual = rng.integers(0, 42, l_seq, dtype=np.uint8).tobytes()
    body = (struct.pack("<iiBBHHHiiii", tid, pos, len(name) + 1, 60, bin_, len(ops), flag, l_seq, mtid, mpos, tlen) + name + b"\0" +
            struct.pack(f"<{len(ops)}I", *[n << 4 | o for o, n in ops]) + seq + qual + aux)
    return struct.pack("<i", len(body)) + body


def kat(cigar, pos, primers, flag=0, t=5, both=False):
    """(CIGAR, pos, what happened) of one record after the oracle's clip; primers: (start, end) on reference 0."""
    rec = make_rec(pos, cigar, flag)
    out, kind, *_ = pc.clip_record(rec, [(0, s, e) for s, e in primers], t, both)
    f = pc.parse(out)
    assert f["tail"] == pc.parse(rec)["tail"]
    if kind == "unmapped":
        assert f["flag"] == flag | 4 and out[:18] == rec[:18] and out[20:] == rec[20:]
    return _str(f["cigar"]), f["pos"], kind


def _bam_header(refs):
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    head = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for n, l in refs:
        head += struct.pack("<i", len(n) + 1) + n + b"\0" + struct.pack("<i", l)
    return head


def _write_bed(path, rows, extra=""):
    with open(path, "w") as fh:
        fh.write("".join(f"{c}\t{s}\t{e}{extra}\n" for c, s, e in rows))
    return str(path)


def _placed(recs):
    return [r for r in recs if struct.unpack_from("<i", r, 4)[0] >= 0]


def _oracle_file(src_recs, head, rows, dst, tol=5, both=False):
    """The oracle's clipped and sorted records written as a BAM; returns (path, stats)."""
    out, st = pc.clip_and_sort(_placed(src_recs), rows, tol, both)
    _write(dst, head, out)
    return dst, st


def _stats(info):
    return dict(n_left=info["n_clipped_left"], n_right=info["n_clipped_right"], n_unmapped=info["n_fully_clipped"],
                n_columns=info["clipped_columns"])


def random_cigar(rng, body_ops=(0, 1, 2, 3, 6, 7, 8), n_body=None):
    """A CIGAR with optional leading H / S, a body drawn from ``body_ops`` that holds a match op and starts and ends with
    one (as an aligner writes), and optional trailing S / H."""
    ops = []
    if rng.random() < 0.2:
        ops.append((pc.H, int(rng.integers(1, 30))))
    if rng.random() < 0.4:
        ops.append((pc.S, int(rng.integers(1, 30))))
    n_body = int(rng.integers(1, 40)) if n_body is None else n_body
    ops.append((int(rng.choice([0, 7, 8])), int(rng.integers(1, 12))))
    for _ in range(n_body):
        ops.append((int(rng.choice(body_ops)), int(rng.integers(1, 12))))
    ops.append((int(rng.choice([0, 7, 8])), int(rng.integers(1, 12))))
    if rng.random() < 0.4:
        ops.append((pc.S, int(rng.integers(1, 30))))
    if rng.random() < 0.2:
        ops.append((pc.H, int(rng.integers(1, 30))))
    return ops


FLAGS = (0, 16, 0x1 | 0x2 | 0x20 | 0x40, 0x1 | 0x2 | 0x10 | 0x80, 0x1 | 0x40, 0x100, 0x110, 0x800, 0x810, 0x400, 0x200, 0x4,
         0x1 | 0x8 | 0x40)


def scheme_rows(L, width=300, step=250, plen=22, alt_every=3):
    """An ARTIC-like tiling over [0, L): left primer [a, a + plen), right primer [a + width - plen, a + width) per amplicon,
    every ``alt_every``-th amplicon with an alt primer shifted by 4 bases."""
    rows = []
    for k, a in enumerate(range(0, L - width, step)):
        rows += [(a, a + plen), (a + width - plen, a + width)]
        if k % alt_every == 0:
            rows += [(a + 4, a + 4 + plen), (a + width - plen - 4, a + width - 4)]
    return rows


def random_records(seed, L=3000, n=3000, n_ref=2):
    """Records near the primers of scheme_rows(L) on references 0..n_ref-1: every flag kind, random CIGARs of every op code,
    read ends steered to 0..60 bases around a primer so that every tolerance matters, a few records without a match op."""
    rng = np.random.default_rng(seed)
    rows = scheme_rows(L)
    recs = []
    for j in range(n):
        ops = random_cigar(rng)
        span = sum(x for o, x in ops if o in pc.REF)
        s, e = rows[int(rng.integers(len(rows)))]
        if rng.random() < 0.5:
            pos = s + int(rng.integers(-60, 30))
        else:
            pos = e - span + int(rng.integers(-30, 60))
        pos = min(max(pos, 0), L - span - 1)
        if rng.random() < 0.02:
            ops = [(pc.S, 10), (pc.I, 5)]
        flag = int(FLAGS[int(rng.integers(len(FLAGS)))])
        tid = int(rng.integers(n_ref))
        recs.append(make_rec(pos, ops, flag, tid, name=b"q%d" % (j // 2), mtid=tid, mpos=pos + 100, tlen=300, aux=b"NMC\x03" * (j % 3),
                             seed=seed * 100000 + j))
    order = np.argsort([struct.unpack_from("<i", r, 8)[0] + (struct.unpack_from("<i", r, 4)[0] << 20) for r in recs], kind="stable")
    recs = [recs[i] for i in order]
    refs = [(b"chr%d" % k, L) for k in range(n_ref)]
    primers = [(k, s, e) for k in range(n_ref) for s, e in rows if (k + s) % 7]        # each reference its own subset
    return refs, recs, primers


# ---------------------------------------------------------------------------- CPU tests: the rule
def test_kat_split_match_keeps_op_code():
    assert kat("50M", 100, [(95, 110)]) == ("10S40M", 110, "clipped")
    assert kat("5=45X", 100, [(100, 108)]) == ("8S42X", 108, "clipped")
    assert kat("20=30X", 100, [(100, 108)]) == ("8S12=30X", 108, "clipped")


def test_kat_insertion_after_the_cut_is_absorbed():
    assert kat("10M3I40M", 100, [(100, 110)]) == ("13S40M", 110, "clipped")


def test_kat_deletion_crossing_the_boundary():
    assert kat("8M4D40M", 100, [(100, 110)]) == ("8S40M", 112, "clipped")
    out, kind, left, right, cols = pc.clip_record(make_rec(100, "8M4D40M"), [(0, 100, 110)])
    assert (left, right, cols) == (True, False, 12)


def test_kat_skip_and_pad():
    assert kat("5M2P3N40M", 100, [(100, 106)]) == ("5S40M", 108, "clipped")
    assert kat("6M1P2I40M", 100, [(100, 106)]) == ("8S40M", 106, "clipped")


def test_kat_leading_hard_and_soft_clips():
    assert kat("3H4S30M", 100, [(100, 110)]) == ("3H14S20M", 110, "clipped")


def test_kat_reverse_read_clipped_on_the_right():
    assert kat("50M", 100, [(140, 160)], flag=16) == ("40M10S", 100, "clipped")
    assert kat("40M5S2H", 100, [(130, 150)], flag=16) == ("30M15S2H", 100, "clipped")
    # the 5' end only: a reverse read keeps its left end, a forward read its right end
    assert kat("50M", 100, [(95, 110)], flag=16) == ("50M", 100, None)
    assert kat("50M", 100, [(140, 160)]) == ("50M", 100, None)


def test_kat_both_ends():
    primers = [(95, 110), (190, 215)]
    assert kat("100M", 100, primers, both=True) == ("10S80M10S", 110, "clipped")
    assert kat("100M", 100, primers, flag=16, both=True) == ("10S80M10S", 110, "clipped")
    assert kat("100M", 100, primers) == ("10S90M", 110, "clipped")
    assert kat("100M", 100, primers, flag=16) == ("90M10S", 100, "clipped")
    # one op cut from both sides
    out, kind, left, right, cols = pc.clip_record(make_rec(100, "100M"), [(0, *p) for p in primers], 5, True)
    assert (left, right, cols) == (True, True, 20)


@pytest.mark.parametrize("t", [0, 5, 50])
def test_kat_tolerance_bounds(t):
    # left: s - p = t - 1 and t match, t + 1 does not (primer [110, 130))
    s, e = 110, 130
    for d, match in ((t - 1, True), (t, True), (t + 1, False)):
        p = s - d
        got = kat("200M", p, [(s, e)], t=t)
        assert got == ((f"{e - p}S{200 - (e - p)}M", e, "clipped") if match else ("200M", p, None)), (t, d)
    # right: s <= q < e + t: a read end t - 1 and t columns behind the primer's last column (e - 1) matches, t + 1 not
    s, e = 150, 170
    for d, match in ((t - 1, True), (t, True), (t + 1, False)):
        q = e - 1 + d
        p = q - 199
        got = kat("200M", p, [(s, e)], flag=16, t=t)
        assert got == ((f"{s - p}M{q - s + 1}S", p, "clipped") if match else ("200M", p, None)), (t, d)


def test_kat_overlapping_and_alt_primers():
    # left: the largest end over the matching primers
    assert kat("50M", 103, [(100, 120), (105, 125), (110, 130)]) == ("22S28M", 125, "clipped")
    # right: the smallest start
    assert kat("50M", 100, [(140, 160), (135, 158), (150, 170)], flag=16) == ("35M15S", 100, "clipped")


def test_kat_fully_clipped():
    # a read inside one primer
    assert kat("20M", 100, [(95, 130)]) == ("20M", 100, "unmapped")
    # both clips meet
    assert kat("40M", 100, [(98, 125), (115, 150)], both=True) == ("40M", 100, "unmapped")
    _, st = pc.clip_records([make_rec(100, "40M")], [(0, 98, 125), (0, 115, 150)], 5, True)
    assert st == dict(n_left=0, n_right=0, n_unmapped=1, n_columns=0)


def test_kat_untouched_records():
    primers = [(0, 95, 110)]
    for rec in (make_rec(100, "50M", flag=4), make_rec(100, "50M", tid=-1), make_rec(100, "20S"), make_rec(100, "10S5I"),
                make_rec(300, "50M"), make_rec(100, "50M", tid=1)):
        out, kind, left, right, cols = pc.clip_record(rec, primers)
        assert out == rec and kind is None and not left and not right and cols == 0


def test_kat_cigars_the_rule_does_not_cover():
    """An op of length 0, or an H / S op between other ops, in an eligible record: refused (the SAM spec allows neither)."""
    for cigar in ("10M5S40M", "10M2H40M", ((0, 10), (0, 0), (0, 40)), ((0, 10), (1, 0), (0, 40))):
        with pytest.raises(ValueError, match="length 0, or an H / S op between"):
            pc.clip_record(make_rec(100, _ops(cigar) if isinstance(cigar, str) else list(cigar)), [(0, 95, 110)])
    # not eligible: left as they are
    rec = make_rec(100, "10M5S40M", flag=4)
    assert pc.clip_record(rec, [(0, 95, 110)])[0] == rec


def test_reg2bin():
    assert pc.reg2bin(0, 1) == 4681 and pc.reg2bin(16384, 16385) == 4682
    assert pc.reg2bin(16380, 16390) == 585 and pc.reg2bin(0, 1 << 29) == 0


@pytest.mark.parametrize("seed", range(6))
def test_invariants_over_random_cigars(seed):
    """Query length kept, new span = old span - removed columns, a match op next to the clips of every clipped end, bin."""
    rng = np.random.default_rng(seed)
    for j in range(1500):
        ops = random_cigar(rng)
        span = sum(n for o, n in ops if o in pc.REF)
        pos = int(rng.integers(0, 200))
        flag = int(rng.choice([0, 16]))
        primers = [(0, int(a), int(a) + int(rng.integers(1, 40))) for a in rng.integers(0, 200 + span, 4)]
        both = bool(rng.random() < 0.5)
        t = int(rng.choice([0, 5, 50]))
        rec = make_rec(pos, ops, flag)
        out, kind, left, right, cols = pc.clip_record(rec, primers, t, both)
        f = pc.parse(out)
        new = f["cigar"]
        assert sum(n for o, n in new if o in pc.QUERY) == sum(n for o, n in ops if o in pc.QUERY)
        if kind != "clipped":
            assert new == ops and f["pos"] == pos
            continue
        new_span = sum(n for o, n in new if o in pc.REF)
        assert new_span == span - cols and f["pos"] + new_span <= pos + span and f["pos"] >= pos
        assert f["bin"] == pc.reg2bin(f["pos"], f["pos"] + new_span)
        if left:
            first = next(o for o, _ in new if o not in (pc.H, pc.S))
            assert first in pc.MATCH
        if right:
            last = next(o for o, _ in reversed(new) if o not in (pc.H, pc.S))
            assert last in pc.MATCH
        assert sum(1 for o, _ in new if o == pc.S) <= 2


# ---------------------------------------------------------------------------- CPU tests: BED reader and flags
def test_read_bed(tmp_path):
    from trueconsense_b200 import primers

    p = tmp_path / "s.bed"
    p.write_bytes(b"# scheme\r\ntrack name=x\r\nbrowser position chr1\r\ntrack\r\n\r\n"
                  b"MN908947.3\t30\t54\tnCoV-2019_1_LEFT\t1\t+\tACCAACCAACTTTCGATCTCTTGT\r\n"
                  b"MN908947.3\t385\t410\tnCoV-2019_1_RIGHT\t1\t-\r\nchr2\t0\t1\r\n")
    s = primers.read_bed(str(p))
    assert s.chrom == ("MN908947.3", "MN908947.3", "chr2")
    assert s.start.tolist() == [30, 385, 0] and s.end.tolist() == [54, 410, 1]
    assert (s.tolerance, s.both_ends, len(s)) == (5, False, 3)
    ref, st, en = s.rows(["chr2", "MN908947.3"])
    assert ref.tolist() == [1, 1, 0] and st.dtype == np.int32 and en.tolist() == [54, 410, 1]
    with pytest.raises(ValueError, match=r"primer chrom 'chr2' names no reference"):
        s.rows(["MN908947.3"])
    t = tmp_path / "t.bed"
    t.write_text("track\tname=x\ntrack1\t3\t9\nbrowser_chr\t1\t2\n")
    assert primers.read_bed(str(t)).chrom == ("track1", "browser_chr")
    e = tmp_path / "e.bed"
    e.write_text("# nothing\n\n")
    assert len(primers.read_bed(str(e))) == 0
    assert primers.read_bed(str(e)).rows(["a"])[0].shape == (0,)
    s2 = primers.read_bed(str(p), tolerance=0, both_ends=True)
    assert (s2.tolerance, s2.both_ends) == (0, True)
    with pytest.raises(ValueError, match="tolerance"):
        primers.read_bed(str(p), tolerance=-1)


@pytest.mark.parametrize("line,reason", [
    ("chr1\t5", "fewer than 3 tab-separated fields"),
    ("chr1 5 9", "fewer than 3 tab-separated fields"),
    ("chr1\tx\t9", "start 'x' is not an integer"),
    ("chr1\t5\t9.5", "end '9.5' is not an integer"),
    ("chr1\t1_0\t20", "start '1_0' is not an integer"),
    ("chr1\t-1\t9", "start -1 is negative"),
    ("chr1\t9\t9", "start 9 is not below end 9"),
    ("chr1\t9\t4", "start 9 is not below end 4"),
    ("chr1\t1\t2147483648", "end 2147483648 is above 2"),
])
def test_read_bed_errors(tmp_path, line, reason):
    from trueconsense_b200 import primers

    p = tmp_path / "bad.bed"
    p.write_text("# h\nchr1\t1\t4\n" + line + "\nchr1\t7\t8\n")
    with pytest.raises(ValueError) as ei:
        primers.read_bed(str(p))
    assert str(ei.value).startswith(f"{p}: line 3: ") and reason in str(ei.value), str(ei.value)


def test_cli_flags(tmp_path, capsys):
    from trueconsense_b200 import TrueConsense, indexing

    bam = tmp_path / "a.bam"; fa = tmp_path / "r.fasta"; gff = tmp_path / "f.gff"; bed = tmp_path / "s.bed"
    for p in (bam, fa, gff, bed):
        p.write_text("x")
    base = ["-i", str(bam), "-ref", str(fa), "-gff", str(gff), "-cov", "30", "-name", "s", "-o", str(tmp_path / "c.fa")]
    o = TrueConsense.GetArgs(base)
    assert (o.primers, o.primer_tolerance, o.primer_both_ends) == (None, 5, False)
    o = TrueConsense.GetArgs(base + ["--primers", str(bed)])
    assert (o.primers, o.primer_tolerance, o.primer_both_ends) == (str(bed), 5, False)
    o = TrueConsense.GetArgs(base + ["--primers", str(bed), "--primer-tolerance", "0", "--primer-both-ends", "--all-contigs",
                                     "--sort-input"])
    assert (o.primer_tolerance, o.primer_both_ends, o.all_contigs, o.sort_input) == (0, True, True, True)
    ov = tmp_path / "o.csv.gz"
    ov.write_text("x")
    assert TrueConsense.GetArgs(base + ["--primers", str(bed), "--index-override", str(ov)]).index_override == str(ov)
    for extra in (["--primer-tolerance", "3"], ["--primer-both-ends"], ["--primers", str(bed), "--primer-tolerance", "-1"],
                  ["--primers", str(fa)]):
        with pytest.raises(SystemExit) as ei:
            TrueConsense.GetArgs(base + extra)
        assert ei.value.code == 2, extra
    with pytest.raises(SystemExit) as ei:
        TrueConsense.GetArgs(base + ["--primers", str(tmp_path / "missing.bed")])
    assert ei.value.code == 1 and "is not a file" in capsys.readouterr().out
    # the handle: primers imply the sort, no host decode, no host batch
    from trueconsense_b200 import primers
    from trueconsense_b200.reads import ReadBatch

    bed.write_text("chr1\t1\t5\n")
    sch = primers.read_bed(str(bed))
    h = indexing.Readbam(str(bam), primers=sch)
    assert h.sort is True and h.primers is sch and indexing.Readbam(h) is h
    with pytest.raises(NotImplementedError, match="primers are clipped on the GPU only"):
        h.reads
    with pytest.raises(ValueError, match="host ReadBatch"):
        indexing.BamHandle(str(bam), reads=ReadBatch.from_records([]), primers=sch)
    assert indexing.Readbam(str(bam)).primers is None


# ---------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import build, gpu

    build.build_host()
    if not os.path.exists(build.CUDA_LIB):
        build.build_cuda()
    return gpu.default_context()


def _dev_arrays(ctx, d):
    s, n = d.struct, d.n_reads
    if n == 0:
        return {}
    sizes = {"seq_off": n + 1, "cigar_off": n + 1, "seq4": d.stats.n_seq_words, "qual": 8 * d.stats.n_seq_words,
             "cigar": d.stats.n_cigar_ops}
    return {f: ctx.download(getattr(s, f), sizes.get(f, n), t) for f, t in FIELDS}


def _assert_same(a, b, what=""):
    assert a.keys() == b.keys(), what
    for f in a:
        assert np.array_equal(a[f], b[f]), (what, f)


def _scheme(path, rows, names, tol=5, both=False):
    from trueconsense_b200 import primers

    return primers.read_bed(_write_bed(path, [(names[r], s, e) for r, s, e in rows]), tol, both)


def _clip_host(ctx, head, recs, names, scheme):
    """tc_bam_clip_primers over a host payload: (the output records, stats)."""
    payload = np.frombuffer(head + b"".join(recs), np.uint8).copy()
    off = np.cumsum([len(head)] + [len(r) for r in recs])[:-1] + 4
    rec = np.ascontiguousarray(off, np.int64)
    p, nb, r, st = ctx.clip_primers(payload.ctypes.data, payload.nbytes, rec.ctypes.data, len(recs), names, scheme)
    out = ctx.download(p, nb, np.uint8).tobytes()
    offs = ctx.download(r, len(recs), np.int64)
    got = [out[o - 4:o + struct.unpack_from("<i", out, o - 4)[0]] for o in offs]
    return got, dict(n_left=st.n_left, n_right=st.n_right, n_unmapped=st.n_unmapped, n_columns=st.n_columns)


@pytest.mark.gpu
@pytest.mark.parametrize("tol", [0, 5, 50])
@pytest.mark.parametrize("both", [False, True])
@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_record_bytes(ctx, seed, both, tol, tmp_path):
    """tc_bam_clip_primers' records == the oracle's, byte for byte, with its stats; then the BAM, SAM and host-payload routes
    give the arrays of the oracle's clipped and sorted records, and the oracle's stats."""
    refs, recs, rows = random_records(seed)
    names = [n.decode() for n, _ in refs]
    head = _bam_header(refs)
    sch = _scheme(tmp_path / "s.bed", rows, names, tol, both)
    want, want_st = pc.clip_records(recs, rows, tol, both)
    got, st = _clip_host(ctx, head, recs, names, sch)
    assert st == want_st and want_st["n_left"] + want_st["n_right"] > 100
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, (i, pc.parse(recs[i])["cigar"], pc.parse(g)["cigar"], pc.parse(w)["cigar"])
    src = _write(str(tmp_path / "in.bam"), head, recs, (65280, 3000))
    exp_bam, st2 = _oracle_file(recs, head, rows, str(tmp_path / "oracle.bam"), tol, both)
    assert st2 == want_st
    want_arr = _dev_arrays(ctx, ctx.bam_file_to_device(exp_bam))
    d = ctx.bam_file_to_device(src, primers=sch)
    assert _stats(d.info) == want_st and d.info["t_clip_s"] > 0
    _assert_same(_dev_arrays(ctx, d), want_arr, "bam")
    from trueconsense_b200 import bamio

    payload = bamio.read_bam_payload(src)
    h = ctx.bam_to_device(payload, primers=sch)
    payload.release()
    assert _stats(h.info) == want_st
    _assert_same(_dev_arrays(ctx, h), want_arr, "host payload")
    # SAM: the records the SAM route builds (bin 0, no optional fields), clipped by the oracle
    from test_sam_input import sam_record

    lines = [sam_line(r, [n for n, _ in refs]) for r in recs]
    sam = str(tmp_path / "in.sam")
    with open(sam, "wb") as fh:
        fh.write(_sam_header(refs) + b"".join(lines))
    sam_recs = [sam_record(l, [n for n, _ in refs]) for l in lines]
    exp_sam, st3 = _oracle_file(sam_recs, head, rows, str(tmp_path / "oracle_sam.bam"), tol, both)
    want_sam = _dev_arrays(ctx, ctx.bam_file_to_device(exp_sam))
    s = ctx.sam_file_to_device(sam, primers=sch)
    assert _stats(s.info) == st3 == want_st
    _assert_same(_dev_arrays(ctx, s), want_sam, "sam")


def _mini_scheme(name, tmp):
    """A synthetic scheme over a golden mini's reference: 20-base primers at both ends of 50-base tiles."""
    from trueconsense_b200 import bamio

    names, lens = bamio.read_bam_header(f"{GOLD}/{name}.bam")
    L = lens[0]
    rows = [(0, a, a + 20) for a in range(0, L - 20, 50)] + [(0, a - 20, a) for a in range(50, L, 50)]
    return names, rows, _write_bed(os.path.join(tmp, f"{name}.bed"), [(names[r], s, e) for r, s, e in rows])


def _cli(argv, out, monkeypatch):
    from trueconsense_b200 import TrueConsense

    monkeypatch.setattr("sys.argv", ["TrueConsense", "<cli>"])
    try:
        TrueConsense.main(argv + ["-o", out + ".fasta", "-vcf", out + ".vcf", "-ogff", out + ".gff", "-doc", out + ".tsv", "-t", "2"])
    except Exception as e:          # the reference's own exceptions (e.g. KeyError) must match too
        return type(e).__name__
    return {e: open(f"{out}.{e}").read() if os.path.exists(f"{out}.{e}") else None for e in ("fasta", "vcf", "gff", "tsv")}


def _mini_argv(name, path):
    mincov = json.load(open(f"{GOLD}/{name}.json"))["mincov"]
    return ["-i", path, "-ref", f"{GOLD}/{name}.fasta", "-gff", f"{GOLD}/{name}.gff", "-cov", str(mincov), "-name", name]


@pytest.mark.gpu
@pytest.mark.parametrize("both", [False, True])
@pytest.mark.parametrize("name", MINIS)
def test_goldens_with_a_scheme(ctx, name, both, tmp_path, monkeypatch):
    """A golden mini with a synthetic scheme: the arrays and the CLI's four files equal the plain path over the oracle's file."""
    from trueconsense_b200 import primers

    tmp = str(tmp_path)
    names, rows, bed = _mini_scheme(name, tmp)
    src = f"{GOLD}/{name}.bam"
    head, recs = _split(src)
    exp, st = _oracle_file(recs, head, rows, os.path.join(tmp, "oracle.bam"), 5, both)
    d = ctx.bam_file_to_device(src, primers=primers.read_bed(bed, 5, both))
    assert _stats(d.info) == st and st["n_left"] + st["n_right"] > 0
    _assert_same(_dev_arrays(ctx, d), _dev_arrays(ctx, ctx.bam_file_to_device(exp)), name)
    flags = ["--primers", bed] + (["--primer-both-ends"] if both else [])
    got = _cli(flags + _mini_argv(name, src), os.path.join(tmp, "p"), monkeypatch)
    want = _cli(_mini_argv(name, exp), os.path.join(tmp, "o"), monkeypatch)
    assert got == want
    # the same records as a shuffled SAM; the oracle clips them in that order (ties of the sort keep it)
    from test_sam_input import bam_to_sam

    perm = np.random.default_rng(7).permutation(len(recs))
    sam = bam_to_sam(src, os.path.join(tmp, "shuf.sam"), aux=True, order=perm)
    exp_sam, st_sam = _oracle_file([recs[i] for i in perm], head, rows, os.path.join(tmp, "oracle_sam.bam"), 5, both)
    assert st_sam == st
    got = _cli(flags + _mini_argv(name, sam), os.path.join(tmp, "s"), monkeypatch)
    assert got == _cli(_mini_argv(name, exp_sam), os.path.join(tmp, "os"), monkeypatch)


def _amplicon_pairs(tmp, L=1500, width=320, step=280, read_len=190, ins_at=None):
    """An amplicon-shaped paired sample: per amplicon, mates reading inwards from its two primers (jittered by up to 3
    bases), overlapping in the middle, where most pairs carry a 3-base insertion; the reference, GFF and scheme."""
    from trueconsense_b200 import bamio, synth
    from trueconsense_b200.reads import ReadBatch

    seq, feats = synth.make_genome(L, 77, "sars2")
    rng = np.random.default_rng(5)
    recs, rows = [], []
    amps = list(range(0, L - width, step))
    for k, a in enumerate(amps):
        rows += [(0, a, a + 24), (0, a + width - 24, a + width)]
        mid = a + width // 2
        for j in range(60):
            ins = rng.random() < 0.8
            s1 = a + int(rng.integers(-3, 4)); s1 = max(s1, 0)
            e2 = min(a + width + int(rng.integers(-3, 4)), L)
            s2 = e2 - read_len
            def read(s, rev, first):
                e = s + read_len
                if ins and s < mid <= e - 1:
                    c = f"{mid - s}M3I{e - mid}M"
                    q = seq[s:mid] + "GTA" + seq[mid:e]
                else:
                    c = f"{read_len}M"
                    q = seq[s:e]
                flag = 0x1 | 0x2 | (0x10 if rev else 0x20) | (0x40 if first else 0x80)
                return dict(pos=s, cigar=c, seq=q, qual=[int(x) for x in rng.integers(10, 40, len(q))], flag=flag,
                            qname=f"a{k}_{j}", mpos=s2 if first else s1, isize=(e2 - s1) * (1 if first else -1))
            recs += [read(s1, False, True), read(s2, True, False)]
    recs.sort(key=lambda r: r["pos"])
    src = os.path.join(tmp, "amp.bam")
    bamio.write_bam(src, ReadBatch.from_records(recs), "ref", L)
    synth.write_fasta(os.path.join(tmp, "amp.fasta"), "ref", seq)
    synth.write_gff(os.path.join(tmp, "amp.gff"), "ref", L, feats)
    return src, rows


@pytest.mark.gpu
def test_amplicon_pairs_with_insertions_in_mate_overlaps(ctx, tmp_path, monkeypatch):
    from trueconsense_b200 import primers

    tmp = str(tmp_path)
    src, rows = _amplicon_pairs(tmp)
    bed = _write_bed(os.path.join(tmp, "amp.bed"), [("ref", s, e) for _, s, e in rows], "\tamp\t1\t+")
    head, recs = _split(src)
    for both in (False, True):
        exp, st = _oracle_file(recs, head, rows, os.path.join(tmp, f"oracle{both}.bam"), 5, both)
        assert st["n_left"] > 0 and st["n_right"] > 0
        d = ctx.bam_file_to_device(src, primers=primers.read_bed(bed, 5, both))
        assert _stats(d.info) == st
        _assert_same(_dev_arrays(ctx, d), _dev_arrays(ctx, ctx.bam_file_to_device(exp)))
        argv = ["-ref", os.path.join(tmp, "amp.fasta"), "-gff", os.path.join(tmp, "amp.gff"), "-cov", "10", "-name", "A"]
        flags = ["--primers", bed] + (["--primer-both-ends"] if both else [])
        got = _cli(flags + ["-i", src] + argv, os.path.join(tmp, f"p{both}"), monkeypatch)
        want = _cli(["-i", exp] + argv, os.path.join(tmp, f"o{both}"), monkeypatch)
        assert isinstance(got, dict) and got == want
        assert sum(1 for l in got["vcf"].splitlines() if l and not l.startswith("#") and len(l.split("\t")[4]) > 1) >= 1


@pytest.mark.gpu
def test_all_contigs_each_reference_its_scheme(ctx, tmp_path, monkeypatch):
    from trueconsense_b200 import primers

    tmp = str(tmp_path)
    head, real, slots, fasta, gff = _multi_ref_files(tmp, n_decoys=4)
    rows, bed_rows = [], []
    for i in slots:
        L = len(real[i]["seq"])
        for a in range(0, L - 200, 150 + 10 * i):
            rows += [(i, a, a + 20), (i, a + 180, a + 200)]
            bed_rows += [(real[i]["name"], a, a + 20), (real[i]["name"], a + 180, a + 200)]
    bed = _write_bed(os.path.join(tmp, "multi.bed"), bed_rows)
    body = [r for i in slots for r in real[i]["recs"]]
    src = _write(os.path.join(tmp, "multi.bam"), head, body)
    exp, st = _oracle_file(body, head, rows, os.path.join(tmp, "oracle.bam"), 5, True)
    d = ctx.bam_file_to_device(src, primers=primers.read_bed(bed, 5, True), contig_ranges=True)
    assert _stats(d.info) == st
    want = ctx.bam_file_to_device(exp, contig_ranges=True)
    assert d.first_read.tolist() == want.first_read.tolist()
    base = ["-ref", fasta, "-gff", gff, "-cov", "30", "-name", "S", "--all-contigs"]
    got = _cli(["--primers", bed, "--primer-both-ends", "-i", src] + base, os.path.join(tmp, "p"), monkeypatch)
    exp_out = _cli(["-i", exp] + base, os.path.join(tmp, "o"), monkeypatch)
    assert isinstance(got, dict) and got == exp_out
    # a primer row on a chrom the header does not list
    bad = _write_bed(os.path.join(tmp, "bad.bed"), bed_rows + [("nowhere", 1, 5)])
    with pytest.raises(ValueError, match="'nowhere' names no reference"):
        ctx.bam_file_to_device(src, primers=primers.read_bed(bad))


@pytest.mark.gpu
def test_no_op_scheme_and_empty_scheme(ctx, tmp_path):
    from trueconsense_b200 import bamio, primers

    src = f"{GOLD}/mini_illumina.bam"
    names, lens = bamio.read_bam_header(src)
    plain = _dev_arrays(ctx, ctx.bam_file_to_device(src))
    far = primers.read_bed(_write_bed(tmp_path / "far.bed", [(names[0], lens[0] + 100, lens[0] + 120)]), 5, True)
    d = ctx.bam_file_to_device(src, primers=far)
    assert _stats(d.info) == dict(n_left=0, n_right=0, n_unmapped=0, n_columns=0) and d.info["reordered"] is False
    _assert_same(_dev_arrays(ctx, d), plain)
    (tmp_path / "empty.bed").write_text("")
    d = ctx.bam_file_to_device(src, primers=primers.read_bed(str(tmp_path / "empty.bed")))
    _assert_same(_dev_arrays(ctx, d), plain)


@pytest.mark.gpu
def test_size_200k_config2_amplicons(ctx, tmp_path):
    """200 k config-2-like ONT amplicon reads on a scheme at the generator's amplicon starts, both ends: arrays == the
    oracle's."""
    from trueconsense_b200 import bamio, primers, synth

    w = synth.config(1, scale=0.1)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    src = str(tmp_path / "cfg2.bam")
    bamio.write_bam(src, b, "ref", L)
    p = w.params
    room = L - p.read_len - p.read_len_jitter
    rows = []
    for a in range(p.n_amplicons):
        st = room * a // (p.n_amplicons - 1)
        rows += [(0, st, st + 24), (0, st + p.read_len - 24, st + p.read_len)]
    bed = _write_bed(tmp_path / "cfg2.bed", [("ref", s, e) for _, s, e in rows])
    head, recs = _split(src)
    exp, st = _oracle_file(recs, head, rows, str(tmp_path / "oracle.bam"), 5, True)
    d = ctx.bam_file_to_device(src, primers=primers.read_bed(bed, 5, True))
    assert d.n_reads == 200_000 and _stats(d.info) == st and st["n_left"] > 100_000
    _assert_same(_dev_arrays(ctx, d), _dev_arrays(ctx, ctx.bam_file_to_device(exp)))


@pytest.mark.gpu
def test_too_many_ops_after_the_clip(ctx, tmp_path):
    """A CIGAR of 65535 ops that gains a soft clip: TC_ERR_ARG naming the record."""
    from trueconsense_b200 import gpu, primers

    ops = [(0, 20)] + [(1, 1), (0, 1)] * 32767
    recs = [make_rec(100, "50M", name=b"a"), make_rec(100, ops, name=b"b")]
    sch = primers.read_bed(_write_bed(tmp_path / "s.bed", [("chr1", 95, 110)]))
    with pytest.raises(gpu.TcError) as ei:
        _clip_host(ctx, _bam_header([(b"chr1", 200000)]), recs, ["chr1"], sch)
    assert ei.value.code == -2 and "record 1 " in str(ei.value)


@pytest.mark.gpu
def test_cigars_the_rule_does_not_cover(ctx, tmp_path):
    """A mapped record whose CIGAR has an op of length 0 or an H / S op between other ops: TC_ERR_ARG naming the record,
    whether or not a primer touches it; unmapped, such a record is copied.  No records: the inputs come back."""
    from trueconsense_b200 import gpu, primers

    sch = primers.read_bed(_write_bed(tmp_path / "s.bed", [("chr1", 95, 110)]))
    head = _bam_header([(b"chr1", 5000)])
    for bad in ("10M5S40M", "10M2H40M", [(0, 10), (2, 0), (0, 40)]):
        recs = [make_rec(100, "50M", name=b"a"), make_rec(100, "50M", name=b"b"), make_rec(3000, bad, name=b"c")]
        with pytest.raises(gpu.TcError) as ei:
            _clip_host(ctx, head, recs, ["chr1"], sch)
        assert ei.value.code == -2 and "record 2 " in str(ei.value) and "length 0" in str(ei.value), str(ei.value)
        recs[2] = make_rec(3000, bad, flag=4, name=b"c")
        got, st = _clip_host(ctx, head, recs, ["chr1"], sch)
        assert got == pc.clip_records(recs, [(0, 95, 110)])[0] and got[2] == recs[2] and st["n_left"] == 2
    payload = np.frombuffer(head, np.uint8).copy()
    p, nb, r, st = ctx.clip_primers(payload.ctypes.data, payload.nbytes, None, 0, ["chr1"], sch)
    assert (p, nb, r) == (payload.ctypes.data, payload.nbytes, None) and st.n_left == 0
