"""BAM and SAM files written and taken apart on the host for the decode tests (sort, SAM input, primer clip, contigs), and
the comparisons those tests share: the device read arrays and the CLI's output files."""
import gzip
import json
import os
import re
import struct
import zlib

import numpy as np

from conftest import GOLD

FIELDS = (("pos", np.int32), ("flag", np.uint16), ("mapq", np.uint8), ("l_seq", np.int32), ("seq_off", np.uint32),
          ("cigar_off", np.uint32), ("seq4", np.uint32), ("qual", np.uint8), ("cigar", np.uint32), ("qname_hash", np.uint64),
          ("mpos", np.int32), ("isize", np.int32))
OPS = b"MIDNSHP=X"
NT16 = b"=ACMGRSVTWYHKDBN"
_HI = bytes(NT16[b >> 4] for b in range(256))
_LO = bytes(NT16[b & 15] for b in range(256))
_Q33 = bytes((b + 33) & 0xFF for b in range(256))
COORDINATE = b"@HD\tVN:1.6\tSO:coordinate\n"
MM2_AUX = b"\tNM:i:%d\tms:i:372\tAS:i:372\tnn:i:0\ttp:A:P\tcm:i:41\ts1:i:355\ts2:i:0\tde:f:0.0123\trl:i:0"


# ---------------------------------------------------------------------------- BAM files
def bgzf(path, payload: bytes, member_bytes=(65280,)) -> None:
    """Write a BAM payload as BGZF members of the given payload size (an int, or a tuple of sizes cycled), and the EOF
    member."""
    def member(chunk):
        c = zlib.compressobj(1, zlib.DEFLATED, -15, 8, 0)
        data = c.compress(chunk) + c.flush()
        bsize = 18 + len(data) + 8
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + data +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    sizes = (member_bytes,) if isinstance(member_bytes, int) else member_bytes
    out, p, k = [], 0, 0
    while p < len(payload):
        n = sizes[k % len(sizes)]
        out.append(member(payload[p:p + n]))
        p, k = p + n, k + 1
    out.append(member(b""))
    with open(path, "wb") as fh:
        fh.write(b"".join(out))


def split(path):
    """(header bytes, [records with their block_size]) of a BAM file."""
    from trueconsense_b200 import bamio

    with gzip.open(path, "rb") as fh:
        payload = fh.read()
    _, _, q = bamio.parse_bam_header(payload, len(payload))
    head, recs = payload[:q], []
    while q + 4 <= len(payload):
        bs = struct.unpack_from("<i", payload, q)[0]
        recs.append(payload[q:q + 4 + bs])
        q += 4 + bs
    return head, recs


def write(path, head, recs, member_bytes=(65280,)):
    bgzf(path, head + b"".join(recs), member_bytes)
    return path


def bam_header(refs, text=COORDINATE) -> bytes:
    """A BAM header (payload bytes up to the first record) of ``refs``: (name as bytes, length)."""
    head = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for n, l in refs:
        head += struct.pack("<i", len(n) + 1) + n + b"\0" + struct.pack("<i", l)
    return head


def refs_of(head):
    """The (name as bytes, length) of every reference of a BAM header."""
    from trueconsense_b200 import bamio

    names, lens, _ = bamio.parse_bam_header(head, len(head))
    return [(n.encode(), l) for n, l in zip(names, lens)]


def multi_ref_files(tmp, n_decoys=6000):
    """Three references with reads (insertions and a deletion inside ORFs, paired reads) spread over a header of
    n_decoys + 3 references (refIDs 0, n_decoys // 2 + 1, n_decoys + 2), the FASTA of all of them and the GFF rows of the
    three.  Returns the paths and the records of each reference (refID patched)."""
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
    refs = []
    for i in range(n_decoys + 3):
        refs.append((real[i]["name"], len(real[i]["seq"])) if i in real else (f"decoy_{i:05d}_with_a_long_name", 10 + i % 23))
    head = bam_header([(n.encode(), l) for n, l in refs], b"@HD\tVN:1.6\tSO:unsorted\n")
    fasta = os.path.join(tmp, "multi.fasta")
    with open(fasta, "w") as fh:
        for i, (n, l) in enumerate(refs):
            s = real[i]["seq"] if i in real else "ACGT" * (l // 4) + "A" * (l % 4)
            fh.write(f">{n}\n" + "".join(s[j:j + 60] + "\n" for j in range(0, len(s), 60)))
    gff = os.path.join(tmp, "multi.gff")
    with open(gff, "w") as fh:
        fh.write("##gff-version 3\n")
        for i in slots:
            c = real[i]
            for f in c["feats"]:
                attrs = f"ID=cds-{c['name']}-{f['name']};Name={f['name']};gbkey=CDS"
                fh.write("\t".join([c["name"], "synthetic", "CDS", str(f["start"]), str(f["end"]), ".", f["strand"], "0", attrs]) + "\n")
    return head, real, slots, fasta, gff


# ---------------------------------------------------------------------------- SAM text
def sam_header(refs, text=COORDINATE) -> bytes:
    return text + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n, l) for n, l in refs) + b"@PG\tID:minimap2\tPN:minimap2\tVN:2.28\n"


def sam_line(r: bytes, names, aux=b"", lower=False) -> bytes:
    """A BAM record (block_size included) as ``samtools view`` prints it (its optional fields replaced by ``aux``)."""
    tid, pos, l_name, mapq, _, n_cig, flag, l_seq, mtid, mpos, tlen = struct.unpack_from("<iiBBHHHiiii", r, 4)
    p = 36
    qname = r[p:p + l_name - 1]
    p += l_name
    cig = struct.unpack_from(f"<{n_cig}I", r, p)
    p += 4 * n_cig
    sb = (l_seq + 1) // 2
    packed = r[p:p + sb]
    qual = r[p + sb:p + sb + l_seq]
    seq = bytearray(2 * sb)
    seq[0::2] = packed.translate(_HI)
    seq[1::2] = packed.translate(_LO)
    seq = bytes(seq[:l_seq]) or b"*"
    if lower:
        seq = seq.lower()
    q = b"*" if not l_seq or qual[0] == 0xFF else qual.translate(_Q33)
    cigar = b"".join(b"%d%c" % (c >> 4, OPS[c & 15]) for c in cig) or b"*"
    rnext = b"*" if mtid < 0 else b"=" if mtid == tid else names[mtid]
    return b"\t".join([qname, b"%d" % flag, names[tid] if tid >= 0 else b"*", b"%d" % (pos + 1), b"%d" % mapq, cigar, rnext,
                       b"%d" % (mpos + 1), b"%d" % tlen, seq, q]) + aux + b"\n"


def sam_record(line: bytes, names):
    """The BAM record (block_size included, ``bin`` 0, no optional fields) of a valid SAM line; None for RNAME '*'."""
    f = line.rstrip(b"\n").split(b"\t")
    qname, flag, rname, pos, mapq, cigar, rnext, pnext, tlen, seq, qual = f[:11]
    index = {n: i for i, n in enumerate(names)}
    if rname == b"*":
        return None
    tid = index[rname]
    mtid = tid if rnext == b"=" else -1 if rnext == b"*" else index[rnext]
    ops = [] if cigar == b"*" else [int(n) << 4 | OPS.index(o) for n, o in re.findall(rb"(\d+)([MIDNSHP=X])", cigar)]
    seq = b"" if seq == b"*" else seq
    codes = [NT16.find(bytes([c]).upper()) % 16 if bytes([c]).upper() in NT16 else 15 for c in seq] + [0]
    packed = bytes(codes[i] << 4 | codes[i + 1] for i in range(0, len(seq), 2))
    q = b"\xff" * len(seq) if qual == b"*" else bytes(c - 33 for c in qual)
    body = (struct.pack("<iiBBHHHiiii", tid, int(pos) - 1, len(qname) + 1, int(mapq), 0, len(ops), int(flag), len(seq), mtid,
                        int(pnext) - 1, int(tlen)) + qname + b"\0" + struct.pack(f"<{len(ops)}I", *ops) + packed + q)
    return struct.pack("<i", len(body)) + body


def bam_to_sam(bam, sam, aux=False, lower=False, order=None, newline_at_end=True):
    """A BAM file written as SAM (header with @SQ lines, every record; ``order``: the records in that order), each line with
    minimap2-like optional fields (``aux``) and lower-case SEQ (``lower``) when asked."""
    head, recs = split(bam)
    names = [n for n, _ in refs_of(head)]
    lines = [sam_line(r, names, MM2_AUX % (i % 7) if aux else b"", lower) for i, r in enumerate(recs)]
    if order is not None:
        lines = [lines[i] for i in order]
    body = b"".join(lines)
    if not newline_at_end:
        body = body[:-1]
    with open(sam, "wb") as fh:
        fh.write(sam_header(refs_of(head)) + body)
    return sam



# ---------------------------------------------------------------------------- comparisons
def dev_arrays(ctx, d):
    """Every array of device reads, on the host (taken before the context stages anything else)."""
    s, n = d.struct, d.n_reads
    if n == 0:
        return {}
    sizes = {"seq_off": n + 1, "cigar_off": n + 1, "seq4": d.stats.n_seq_words, "qual": 8 * d.stats.n_seq_words,
             "cigar": d.stats.n_cigar_ops}
    return {f: ctx.download(getattr(s, f), sizes.get(f, n), t) for f, t in FIELDS}


def assert_same_arrays(a, b, what=""):
    assert a.keys() == b.keys(), what
    for f in a:
        assert np.array_equal(a[f], b[f]), (what, f)


def run_cli(argv, out, monkeypatch, argv0="<cli>"):
    """main(argv) writing {out}.{ext}: the files' text, or the exception type's name.  ``argv0``: the command line's
    placeholder in sys.argv (the VCF header records it)."""
    from trueconsense_b200 import TrueConsense

    monkeypatch.setattr("sys.argv", ["TrueConsense", argv0])
    try:
        TrueConsense.main(argv + ["-o", out + ".fasta", "-vcf", out + ".vcf", "-ogff", out + ".gff", "-doc", out + ".tsv", "-t", "2"])
    except Exception as e:          # the reference's own exceptions (e.g. KeyError) must match too
        return type(e).__name__
    return {e: open(f"{out}.{e}").read() if os.path.exists(f"{out}.{e}") else None for e in ("fasta", "vcf", "gff", "tsv")}


def mini_argv(name, path):
    """The CLI arguments of a golden mini sample (tests/golden/{name}.*) with ``path`` as its input."""
    mincov = json.load(open(f"{GOLD}/{name}.json"))["mincov"]
    return ["-i", path, "-ref", f"{GOLD}/{name}.fasta", "-gff", f"{GOLD}/{name}.gff", "-cov", str(mincov), "-name", name]
