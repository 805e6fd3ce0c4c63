"""The decoded records written back as a BAM, BGZF members compressed on the GPU (``gpu.Context.write_bam``,
``--output-bam``).  Every written file is taken apart on the host: its members inflate with zlib, their CRC-32 / ISIZE /
BSIZE fields hold, it ends with the EOF member, the payload equals the rewritten header plus the independent oracles'
records with ``bin`` recomputed, and every member's compressed bytes equal the CPU harness's for the same input."""
import os
import struct
import zlib

import numpy as np
import pytest

from bamfiles import (assert_same_arrays, bam_header, bam_to_sam, dev_arrays, mini_argv, multi_ref_files, refs_of, run_cli,
                      sam_line, sam_record, split, write)
from conftest import GOLD
from test_deflate_core import deflate, h  # noqa: F401  (the harness fixture)

MEMBER = 0xFF00
EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
REF_OPS = (0, 2, 3, 7, 8)


@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import gpu

    return gpu.Context(0)


# ---------------------------------------------------------------------------- the file taken apart
def members(path):
    """[(raw DEFLATE stream, uncompressed bytes)] of every member before the EOF member, every framing field checked."""
    data = open(path, "rb").read()
    assert data.endswith(EOF)
    out, p = [], 0
    while p < len(data) - len(EOF):
        assert data[p:p + 4] == b"\x1f\x8b\x08\x04" and data[p + 10:p + 16] == b"\x06\x00BC\x02\x00"
        size = struct.unpack_from("<H", data, p + 16)[0] + 1
        assert size <= 65536
        comp = data[p + 18:p + size - 8]
        crc, isize = struct.unpack_from("<II", data, p + size - 8)
        raw = zlib.decompressobj(-15).decompress(comp)
        assert len(raw) == isize <= MEMBER and zlib.crc32(raw) == crc
        out.append((comp, raw))
        p += size
    assert p == len(data) - len(EOF)
    return out


def with_bin(r: bytes) -> bytes:
    """A record (block_size included) with bin = reg2bin(pos, end), end = pos + the CIGAR's reference length or pos + 1."""
    from oracle.primer_clip import reg2bin

    pos, l_name, n_cig = struct.unpack_from("<i", r, 8)[0], r[12], struct.unpack_from("<H", r, 16)[0]
    cig = struct.unpack_from(f"<{n_cig}I", r, 36 + l_name)
    span = sum(c >> 4 for c in cig if (c & 15) in REF_OPS)
    return r[:14] + struct.pack("<H", reg2bin(pos, pos + (span if span else 1))) + r[16:]


def check_file(path, header, recs, harness=None):
    """The written file == the header (``@HD ... SO:coordinate``) and ``recs`` with bin recomputed, in members as htslib cuts
    them; with ``harness`` every member's stream equals the CPU compressor's."""
    from trueconsense_b200 import bamio

    ms = members(path)
    head = bamio.coordinate_header(header)
    body = b"".join(with_bin(r) for r in recs)
    assert b"".join(raw for _, raw in ms) == head + body
    cut = [len(head[o:o + MEMBER]) for o in range(0, len(head), MEMBER)] + [len(body[o:o + MEMBER]) for o in range(0, len(body), MEMBER)]
    assert [len(raw) for _, raw in ms] == cut
    if harness is not None:
        for comp, raw in ms:
            assert deflate(harness, raw)[0] == comp
    return ms


def _placed(recs):
    return [r for r in recs if struct.unpack_from("<i", r, 4)[0] >= 0]


def _scheme(tmp, name, L, both):
    from trueconsense_b200 import primers

    rows = [(s, s + 22) for s in range(0, L - 300, 250)] + [(s + 278, s + 300) for s in range(0, L - 300, 250)]
    bed = tmp / "s.bed"
    bed.write_text("".join(f"{name}\t{s}\t{e}\n" for s, e in rows))
    return primers.read_bed(str(bed), 5, both), [(0, s, e) for s, e in rows]


# ---------------------------------------------------------------------------- every route, every mode
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "sort", "primers_both", "primers_5"])
@pytest.mark.parametrize("route", ["bam", "sam", "payload"])
@pytest.mark.parametrize("name", ["mini_illumina", "mini_ont", "mini_long"])
def test_written_file_equals_the_oracle(ctx, h, name, route, mode, tmp_path):  # noqa: F811
    from oracle import primer_clip as pc
    from trueconsense_b200 import bamio

    head, recs = split(f"{GOLD}/{name}.bam")
    names = [n for n, _ in refs_of(head)]
    src = f"{GOLD}/{name}.bam"
    kw = {}
    if mode == "sort":
        perm = np.random.default_rng(5).permutation(len(recs))
        recs = [recs[i] for i in perm]
        src = write(str(tmp_path / "shuf.bam"), head, recs, (1000, 65280, 30000))
        kw["sort"] = True
    placed = _placed(recs)
    if mode.startswith("primers"):
        kw["primers"], rows = _scheme(tmp_path, names[0].decode(), refs_of(head)[0][1], mode == "primers_both")
        want, _ = pc.clip_and_sort(placed, rows, 5, mode == "primers_both")
    else:
        want = [placed[i] for i in pc.sort_order(placed)] if mode == "sort" else placed
    if route == "sam":
        src = bam_to_sam(src, str(tmp_path / "in.sam"))
        want = [sam_record(sam_line(r, names), names) for r in want]
        header = bamio.sam_bam_header(src, *bamio.read_sam_header(src)[:2], bamio.read_sam_header(src)[2])
        d = ctx.sam_file_to_device(src, **kw)
    elif route == "payload":
        header = head
        payload = bamio.read_bam_payload(src)
        d = ctx.bam_to_device(payload, **kw)
    else:
        header = head
        d = ctx.bam_file_to_device(src, **kw)
    before = dev_arrays(ctx, d)
    out = str(tmp_path / "out.bam")
    info = ctx.write_bam(d, out)
    assert info["n_written"] == len(want) == d.n_reads and info["bam_out_bytes"] == os.path.getsize(out)
    assert d.info["n_out_members"] == info["n_out_members"] and d.info["t_write_s"] > 0
    check_file(out, header, want, h)
    assert_same_arrays(dev_arrays(ctx, d), before)          # writing leaves the decoded reads as they were
    # read back: the device route and the host reader give the arrays of the decode that wrote the file
    assert_same_arrays(dev_arrays(ctx, ctx.bam_file_to_device(out)), before)
    b = bamio.read_bam(out)
    assert np.array_equal(b.pos, before["pos"]) and np.array_equal(b.flag, before["flag"])
    if route == "payload":
        payload.release()


@pytest.mark.gpu
def test_pileup_after_the_write(ctx, tmp_path):
    from trueconsense_b200 import bamio

    L = bamio.read_fasta_lengths(f"{GOLD}/mini_ont.fasta")[1][0]
    d = ctx.bam_file_to_device(f"{GOLD}/mini_ont.bam")
    first = ctx.pileup_counts(d, L)
    ctx.write_bam(d, str(tmp_path / "o.bam"))
    assert np.array_equal(ctx.pileup_counts(d, L), first)


# ---------------------------------------------------------------------------- edges
@pytest.mark.gpu
def test_no_placed_records(ctx, h, tmp_path):  # noqa: F811
    head, recs = split(f"{GOLD}/mini_illumina.bam")
    unplaced = bytearray(recs[0])
    struct.pack_into("<i", unplaced, 4, -1)
    for rs in ([], [bytes(unplaced)]):
        src = write(str(tmp_path / "e.bam"), head, rs)
        d = ctx.bam_file_to_device(src)
        out = str(tmp_path / "e_out.bam")
        assert ctx.write_bam(d, out)["n_written"] == 0
        ms = check_file(out, head, [], h)
        assert len(ms) == 1


@pytest.mark.gpu
def test_long_header_and_all_contigs_cli(ctx, h, tmp_path, monkeypatch):  # noqa: F811
    """The 6003-reference header spans several members; the CLI over --all-contigs writes a BAM on which a second run gives
    the same outputs."""
    head, real, slots, fasta, gff = multi_ref_files(str(tmp_path))
    recs = [r for k in slots for r in real[k]["recs"]]
    src = write(str(tmp_path / "multi.bam"), head, recs)
    assert len(head) > 3 * MEMBER
    d = ctx.bam_file_to_device(src, contig_ranges=True)
    out = str(tmp_path / "w.bam")
    ctx.write_bam(d, out)
    check_file(out, head, recs, h)
    argv = ["-ref", fasta, "-gff", gff, "-cov", "5", "-name", "M", "--all-contigs"]
    obam = str(tmp_path / "cli.bam")
    first = run_cli(["-i", src, "--output-bam", obam] + argv, str(tmp_path / "a"), monkeypatch)
    assert isinstance(first, dict) and first["fasta"]
    check_file(obam, head, recs)
    assert run_cli(["-i", obam] + argv, str(tmp_path / "b"), monkeypatch) == first


def _z_tag(k):
    return b"XZZ" + b"a" * k + b"\0"


@pytest.mark.gpu
def test_records_spanning_members_and_exact_multiples(ctx, h, tmp_path):  # noqa: F811
    """Records of 300 KB span several members; a record stream of exactly 3 x 0xff00 bytes ends on a member's end."""
    from test_primer_clip import make_rec

    head = bam_header([(b"chr1", 500_000)])
    big = [make_rec(1000 + 7 * i, "200000M", name=b"big%d" % i, seed=i) for i in range(3)]
    assert all(len(r) > 300_000 for r in big)
    small = [make_rec(5000 + i, "150M", name=b"s%d" % i, seed=10 + i) for i in range(200)]
    for recs in (big + small, small[:100] + big[:1] + small[100:]):
        recs = sorted(recs, key=lambda r: struct.unpack_from("<i", r, 8)[0])
        src = write(str(tmp_path / "big.bam"), head, recs)
        out = str(tmp_path / "big_out.bam")
        ctx.write_bam(ctx.bam_file_to_device(src), out)
        check_file(out, head, recs, h)
    recs = [make_rec(100 + i, "150M", name=b"e%d" % i, seed=30 + i) for i in range(300)]
    short = 3 * MEMBER - sum(len(r) for r in recs)
    last = make_rec(500, "150M", name=b"last", seed=99, aux=_z_tag(0))
    recs.append(make_rec(500, "150M", name=b"last", seed=99, aux=_z_tag(short - len(last))))
    assert sum(len(r) for r in recs) == 3 * MEMBER
    src = write(str(tmp_path / "exact.bam"), head, recs)
    out = str(tmp_path / "exact_out.bam")
    assert ctx.write_bam(ctx.bam_file_to_device(src), out)["n_out_members"] == 1 + 3
    check_file(out, head, recs, h)


@pytest.mark.gpu
def test_handle_writes_once_and_refusals_leave_no_file(ctx, tmp_path):
    from trueconsense_b200 import indexing

    head, recs = split(f"{GOLD}/mini_illumina.bam")
    shuf = write(str(tmp_path / "shuf.bam"), head, [recs[i] for i in np.random.default_rng(1).permutation(len(recs))])
    out = tmp_path / "o.bam"
    with pytest.raises(ValueError, match="Unsorted"):
        indexing.BamHandle(shuf, output_bam=str(out)).device_reads()
    assert not out.exists()
    mhead, real, slots, _, _ = multi_ref_files(str(tmp_path), n_decoys=3)
    multi = write(str(tmp_path / "multi.bam"), mhead, [r for k in slots for r in real[k]["recs"]])
    with pytest.raises(ValueError, match="multi-contig"):
        indexing.BamHandle(multi, output_bam=str(out)).device_reads()
    assert not out.exists() and not [p for p in os.listdir(tmp_path) if p.endswith(".tmp")]
    hd = indexing.BamHandle(shuf, sort=True, output_bam=str(out))
    d = hd.device_reads()
    assert out.exists() and d.info["n_written"] == len(recs)
    out.unlink()
    hd.device_reads()
    names, lens = list(hd.references), list(hd.lengths)
    hd.device_reads_contigs(names, lens)
    hd.device_reads()
    assert not out.exists()
    # the host-payload route keeps the payload until the write
    from trueconsense_b200 import bamio

    p = bamio.read_bam_payload(shuf)
    d = ctx.bam_to_device(p)
    assert d.records[1] == p.payload_ptr
    ctx.write_bam(ctx.bam_to_device(p, sort=True), str(out))
    from oracle import primer_clip as pc

    shuffled = split(shuf)[1]
    check_file(str(out), head, [shuffled[i] for i in pc.sort_order(shuffled)])
    p.release()
    ctx.bam_file_to_device(shuf, sort=True)
    with pytest.raises(RuntimeError, match="stale"):
        ctx.write_bam(d, str(tmp_path / "stale.bam"))
    with pytest.raises(ValueError, match="host ReadBatch"):
        ctx.write_bam(ctx.upload(bamio.read_bam(f"{GOLD}/mini_illumina.bam")), str(tmp_path / "up.bam"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mini_illumina", "mini_ont"])
def test_cli_round_trip(ctx, name, tmp_path, monkeypatch):
    """The CLI with --output-bam on a shuffled SAM with primers; the CLI on the written BAM gives the same files."""
    head, recs = split(f"{GOLD}/{name}.bam")
    shuf = write(str(tmp_path / "shuf.bam"), head, [recs[i] for i in np.random.default_rng(2).permutation(len(recs))])
    sam = bam_to_sam(shuf, str(tmp_path / "shuf.sam"))
    names = [n for n, _ in refs_of(head)]
    bed = tmp_path / "s.bed"
    L = refs_of(head)[0][1]
    bed.write_text("".join(f"{names[0].decode()}\t{s}\t{s + 22}\n" for s in range(0, L - 300, 250)))
    obam = str(tmp_path / "o.bam")
    first = run_cli(mini_argv(name, sam) + ["--primers", str(bed), "--primer-both-ends", "-obam", obam], str(tmp_path / "a"),
                    monkeypatch)
    assert isinstance(first, dict) and first["fasta"] and os.path.exists(obam)
    assert run_cli(mini_argv(name, obam), str(tmp_path / "b"), monkeypatch) == first


@pytest.mark.gpu
def test_size_200k_config2_amplicons(ctx, h, tmp_path):  # noqa: F811
    """200 k config-2-like amplicon reads with primers clipped: the written BAM decodes to the arrays that wrote it."""
    from trueconsense_b200 import bamio, primers, synth

    w = synth.config(1, scale=0.1)
    b = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    src = str(tmp_path / "cfg2.bam")
    bamio.write_bam(src, b, "ref", L)
    p = w.params
    room = L - p.read_len - p.read_len_jitter
    bed = tmp_path / "cfg2.bed"
    rows = []
    for a in range(p.n_amplicons):
        st = room * a // (p.n_amplicons - 1)
        rows += [(st, st + 24), (st + p.read_len - 24, st + p.read_len)]
    bed.write_text("".join(f"ref\t{s}\t{e}\n" for s, e in rows))
    d = ctx.bam_file_to_device(src, primers=primers.read_bed(str(bed), 5, True))
    assert d.n_reads == 200_000 and d.info["n_clipped_left"] > 100_000
    want = dev_arrays(ctx, d)
    out = str(tmp_path / "out.bam")
    info = ctx.write_bam(d, out)
    assert info["n_written"] == 200_000
    ms = members(out)
    for comp, raw in ms[:: max(1, len(ms) // 8)]:
        assert deflate(h, raw)[0] == comp
    assert_same_arrays(dev_arrays(ctx, ctx.bam_file_to_device(out)), want)
