"""What writing the decoded records as a BAM (``--output-bam``, ``gpu.Context.write_bam``) costs on one GPU, against host zlib.

    python scripts/bamwrite_rate.py [--reads 200000 1000000] [--reps 5] [--out profiles/bamwrite_rate.json]

For each read count: a seeded config-2-like read set (ONT amplicon reads of ~400 bp, synth.config(1)) written as a sorted BAM,
decoded once plain and once with an ARTIC-like scheme clipped at both ends (clip_rate.py's), then written back.  Reported per
decode (one warm-up, median of --reps):
  * device_ms:   CUDA-event time of the gather, the member compression and the compaction (tc_bam_write_records' t_ms)
  * write_ms:    host clock around write_bam: the above plus the size read-back, the download and the file write
  * out_bytes / zlib1_bytes:  the written file against zlib level 1 over the same 0xff00-byte members (26 bytes of framing each,
                 the EOF member on both sides)
  * zlib1_all_threads_ms:  host clock of zlib level 1 over those members on every host thread (Python zlib in a thread pool)
Prints the card's name, power limit and max SM clock, then one JSON line per read count and decode; --out also writes them as
one JSON document.  The files go to a temporary directory."""
import argparse
import concurrent.futures as cf
import dataclasses
import json
import os
import struct
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from clip_rate import scheme_rows  # noqa: E402
from sam_rate import card  # noqa: E402
from trueconsense_b200 import bamio, gpu, primers, synth  # noqa: E402


def member_payloads(path):
    """The uncompressed bytes of every member of a BGZF file but the EOF member."""
    data = open(path, "rb").read()
    out, p = [], 0
    while p < len(data):
        size = struct.unpack_from("<H", data, p + 16)[0] + 1
        raw = zlib.decompressobj(-15).decompress(data[p + 18:p + size - 8])
        if raw:
            out.append(raw)
        p += size
    return out


def zlib1(chunk: bytes) -> int:
    c = zlib.compressobj(1, zlib.DEFLATED, -15)
    return len(c.compress(chunk) + c.flush()) + 26


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, nargs="+", default=[200_000, 1_000_000])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results here as one JSON document")
    args = ap.parse_args()
    info = card()
    info["host_threads"] = os.cpu_count()
    print(json.dumps(info), flush=True)
    ctx = gpu.default_context()
    out = []
    for n in args.reads:
        w = synth.config(1, scale=n / 2_000_000)
        prm = dataclasses.replace(w.params, read_len_jitter=3)
        b = synth.generate_reads(prm, w.ref)
        L = len(w.ref)
        rows = scheme_rows(prm, L)
        with tempfile.TemporaryDirectory() as tmp:
            src, bed, dst = (os.path.join(tmp, k) for k in ("sorted.bam", "scheme.bed", "out.bam"))
            bamio.write_bam(src, b, "ref", L, level=1)
            with open(bed, "w") as fh:
                fh.write("".join(f"ref\t{s}\t{e}\n" for _, s, e in rows))
            for tag, kw in (("plain", {}), ("primers", {"primers": primers.read_bed(bed, 5, True)})):
                d = ctx.bam_file_to_device(src, **kw)
                ctx.write_bam(d, dst)                       # warm-up: buffers sized, modules loaded
                host, dev = [], []
                for _ in range(args.reps):
                    r = ctx.write_bam(d, dst)
                    host.append(r["t_write_s"] * 1e3)
                    dev.append(r["t_device_ms"])
                chunks = member_payloads(dst)
                z = sum(zlib1(c) for c in chunks) + 28
                with cf.ThreadPoolExecutor(max_workers=os.cpu_count()) as pool:
                    list(pool.map(zlib1, chunks))           # warm-up
                    zt = []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        list(pool.map(zlib1, chunks))
                        zt.append((time.perf_counter() - t0) * 1e3)
                row = {"reads": b.n_reads, "decode": tag, "n_written": r["n_written"], "payload_bytes": sum(len(c) for c in chunks),
                       "members": r["n_out_members"], "out_bytes": r["bam_out_bytes"], "zlib1_bytes": z,
                       "out_over_zlib1": round(r["bam_out_bytes"] / z, 4),
                       "device_ms": float(np.median(dev)), "device_ms_all": sorted(round(x, 3) for x in dev),
                       "write_ms": float(np.median(host)), "write_ms_all": sorted(round(x, 2) for x in host),
                       "zlib1_all_threads_ms": float(np.median(zt)), "zlib1_all_threads_ms_all": sorted(round(x, 2) for x in zt)}
                row.update(info)
                print(json.dumps(row), flush=True)
                out.append(row)
                del d, chunks
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": info, "results": out}, fh, indent=1)


if __name__ == "__main__":
    main()
