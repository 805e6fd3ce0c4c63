"""What reading the aligner's SAM text costs against a BAM of the same records, on one GPU.

    python scripts/sam_rate.py [--reads 200000 1000000] [--reps 5] [--out profiles/sam_rate.json]

For each read count: a seeded config-2-like read set (ONT amplicons of ~400 bp, synth.config(1)) written as
  * a sorted BAM;
  * a sorted SAM whose lines carry minimap2-like optional fields (NM, ms, AS, nn, tp, cm, s1, s2, de, rl);
  * a shuffled SAM (the same lines in a seeded random order), and the same shuffle as a BAM.
Timed (host clock around each call, which ends in a device synchronise; one warm-up, median of --reps):
  * bam_sorted:   gpu.Context.bam_file_to_device(sorted BAM)             (the BAM route)
  * sam_sorted:   gpu.Context.sam_file_to_device(sorted SAM)
  * sam_shuffled: gpu.Context.sam_file_to_device(shuffled SAM, sort=True)
with the ``.info`` breakdown of the last call of each (upload, line index, convert, sort, parse; the BAM route's map, inflate,
index, sort, parse).  Checks: the sorted SAM's read arrays equal the sorted BAM's, and the shuffled SAM's equal the shuffled
BAM's with sort=True (ties may order differently from the sorted file, so those two are not compared with each other).
Prints the card's name, power limit and max SM clock, then one JSON line per read count; --out also writes them as one JSON
document.  The files go to a temporary directory."""
import argparse
import gzip
import json
import os
import struct
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from trueconsense_b200 import bamio, gpu, synth  # noqa: E402

FIELDS = (("pos", np.int32), ("flag", np.uint16), ("mapq", np.uint8), ("l_seq", np.int32), ("seq_off", np.uint32),
          ("cigar_off", np.uint32), ("seq4", np.uint32), ("qual", np.uint8), ("cigar", np.uint32), ("qname_hash", np.uint64),
          ("mpos", np.int32), ("isize", np.int32))
OPS = b"MIDNSHP=X"
NT16 = b"=ACMGRSVTWYHKDBN"
_HI = bytes(NT16[b >> 4] for b in range(256))
_LO = bytes(NT16[b & 15] for b in range(256))
_Q33 = bytes((b + 33) & 0xFF for b in range(256))
MM2_AUX = b"\tNM:i:%d\tms:i:372\tAS:i:372\tnn:i:0\ttp:A:P\tcm:i:41\ts1:i:355\ts2:i:0\tde:f:0.0123\trl:i:0"


def card() -> dict:
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("sam_rate.py measures on a CUDA device; none is available")
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:          # the query is informative only
        out["power_limit"] = f"unknown ({e})"
    return out


def records(path):
    """(payload header bytes, reference names, [records with their block_size]) of a BAM."""
    with gzip.open(path, "rb") as fh:
        payload = fh.read()
    names, lens, q = bamio.parse_bam_header(payload, len(payload))
    head, recs = payload[:q], []
    while q + 4 <= len(payload):
        bs = struct.unpack_from("<i", payload, q)[0]
        recs.append(payload[q:q + 4 + bs])
        q += 4 + bs
    return head, names, lens, recs


def sam_line(r: bytes, names, aux: bytes) -> bytes:
    """A BAM record as ``samtools view`` prints it, with ``aux`` as its optional fields."""
    tid, pos, l_name, mapq, _, n_cig, flag, l_seq, mtid, mpos, tlen = struct.unpack_from("<iiBBHHHiiii", r, 4)
    p = 36 + l_name
    cig = struct.unpack_from(f"<{n_cig}I", r, p)
    p += 4 * n_cig
    sb = (l_seq + 1) // 2
    packed, qual = r[p:p + sb], r[p + sb:p + sb + l_seq]
    seq = bytearray(2 * sb)
    seq[0::2] = packed.translate(_HI)
    seq[1::2] = packed.translate(_LO)
    q = b"*" if not l_seq or qual[0] == 0xFF else qual.translate(_Q33)
    rnext = b"*" if mtid < 0 else b"=" if mtid == tid else names[mtid]
    return b"\t".join([r[36:36 + l_name - 1], b"%d" % flag, names[tid] if tid >= 0 else b"*", b"%d" % (pos + 1), b"%d" % mapq,
                       b"".join(b"%d%c" % (c >> 4, OPS[c & 15]) for c in cig) or b"*", rnext, b"%d" % (mpos + 1), b"%d" % tlen,
                       bytes(seq[:l_seq]) or b"*", q]) + aux + b"\n"


def bgzf(path: str, data: bytes) -> None:
    def member(chunk: bytes) -> bytes:
        c = zlib.compressobj(1, zlib.DEFLATED, -15, 8, 0)
        z = c.compress(chunk) + c.flush()
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<HHHH", 6, 0x4342, 2, 18 + len(z) + 8 - 1) + z +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    with open(path, "wb") as fh:
        for p in range(0, len(data), 65280):
            fh.write(member(data[p:p + 65280]))
        fh.write(member(b""))


def timed(fn, reps: int):
    fn()                                    # warm-up: modules loaded, buffers sized
    ms, res = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return res, float(np.median(ms)), sorted(round(x, 2) for x in ms)


def arrays(ctx, d) -> dict:
    s, n = d.struct, d.n_reads
    sizes = {"seq_off": n + 1, "cigar_off": n + 1, "seq4": d.stats.n_seq_words, "qual": 8 * d.stats.n_seq_words,
             "cigar": d.stats.n_cigar_ops}
    return {f: ctx.download(getattr(s, f), sizes.get(f, n), t) for f, t in FIELDS}


def same(a: dict, b: dict) -> bool:
    return a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)


def steps(info: dict) -> dict:
    return {k: round(v * 1e3, 3) for k, v in info.items() if k.startswith("t_")}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, nargs="+", default=[200_000, 1_000_000])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results here as one JSON document")
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    ctx = gpu.default_context()
    rows = []
    for n in args.reads:
        w = synth.config(1, scale=n / 2_000_000)
        b = synth.generate_reads(w.params, w.ref)
        with tempfile.TemporaryDirectory() as tmp:
            p = {k: os.path.join(tmp, k) for k in ("sorted.bam", "sorted.sam", "shuffled.sam", "shuffled.bam")}
            bamio.write_bam(p["sorted.bam"], b, "ref", len(w.ref), level=1)
            head, names, lens, recs = records(p["sorted.bam"])
            bnames = [x.encode() for x in names]
            sam_head = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (x, l) for x, l in zip(bnames, lens))
            sam_head += b"@PG\tID:minimap2\tPN:minimap2\tVN:2.28\n"
            lines = [sam_line(r, bnames, MM2_AUX % (i % 7)) for i, r in enumerate(recs)]
            order = np.random.default_rng(17).permutation(len(recs))
            with open(p["sorted.sam"], "wb") as fh:
                fh.write(sam_head + b"".join(lines))
            with open(p["shuffled.sam"], "wb") as fh:
                fh.write(sam_head + b"".join(lines[i] for i in order))
            bgzf(p["shuffled.bam"], head + b"".join(recs[i] for i in order))
            del lines, recs
            row = {"reads": b.n_reads, "bytes": {k: os.path.getsize(v) for k, v in p.items()}}
            d, row["bam_sorted_ms"], row["bam_sorted_ms_all"] = timed(lambda: ctx.bam_file_to_device(p["sorted.bam"]), args.reps)
            row["bam_sorted_steps_ms"] = steps(d.info)
            want = arrays(ctx, d)
            d, row["sam_sorted_ms"], row["sam_sorted_ms_all"] = timed(lambda: ctx.sam_file_to_device(p["sorted.sam"]), args.reps)
            row["sam_sorted_steps_ms"] = steps(d.info)
            row["sam_sorted_equals_bam_sorted"] = same(arrays(ctx, d), want)
            want = arrays(ctx, ctx.bam_file_to_device(p["shuffled.bam"], sort=True))
            d, row["sam_shuffled_sort_ms"], row["sam_shuffled_sort_ms_all"] = timed(
                lambda: ctx.sam_file_to_device(p["shuffled.sam"], sort=True), args.reps)
            row["sam_shuffled_sort_steps_ms"] = steps(d.info)
            row["sam_shuffled_reordered"] = d.info["reordered"]
            row["sam_shuffled_equals_bam_shuffled_sort"] = same(arrays(ctx, d), want)
            row.update(info)
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": info, "results": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
