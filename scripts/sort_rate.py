"""What accepting an unsorted BAM costs: the device decode of a coordinate-sorted file against the same records shuffled and
put back in coordinate order on the GPU (tc_bam_sort_records), on one GPU.

    python scripts/sort_rate.py [--reads 200000 1000000] [--reps 5] [--out sort_rate.json]

For each read count: a seeded config-2-like read set (ONT amplicons, synth.config(1)) written as a sorted BAM, and a copy
whose records are permuted by a seeded shuffle and re-blocked.  Timed (host clock around gpu.Context.bam_file_to_device,
which ends in a device synchronise; one warm-up, median of --reps):
  * sorted:          the sorted file, sort=False (today's path);
  * sorted_check:    the sorted file, sort=True (the key kernel finds it sorted: the check alone);
  * shuffled_sort:   the shuffled file, sort=True (keys, check and the radix sort over the record offsets);
  * t_sort:          the sort step of the last (shuffled_sort's ``.info["t_sort_s"]``).
Also checks that the shuffled file sorted on the device gives the sorted file's count table.  Prints the card's name and
power limit, then one JSON line per read count; --out also writes them as one JSON document.  The BAM files go to a
temporary directory."""
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


def card() -> dict:
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("sort_rate.py measures on a CUDA device; none is available")
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:          # the query is informative only
        out["power_limit"] = f"unknown ({e})"
    return out


def shuffled_copy(src: str, dst: str, seed: int) -> None:
    """The records of src in a seeded random order, re-blocked into BGZF members of varying payload size."""
    with gzip.open(src, "rb") as fh:
        payload = fh.read()
    q = bamio.parse_bam_header(payload, len(payload))[2]
    head, starts = payload[:q], []
    while q + 4 <= len(payload):
        starts.append(q)
        q += 4 + struct.unpack_from("<i", payload, q)[0]
    starts.append(q)
    rng = np.random.default_rng(seed)
    body = b"".join(payload[starts[i]:starts[i + 1]] for i in rng.permutation(len(starts) - 1))
    data = head + body
    sizes = [int(x) for x in rng.integers(16000, 65280, 64)]

    def member(chunk: bytes) -> bytes:
        c = zlib.compressobj(1, zlib.DEFLATED, -15, 8, 0)
        z = c.compress(chunk) + c.flush()
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<HHHH", 6, 0x4342, 2, 18 + len(z) + 8 - 1) + z +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    with open(dst, "wb") as fh:
        p, k = 0, 0
        while p < len(data):
            n = sizes[k % len(sizes)]
            fh.write(member(data[p:p + n]))
            p, k = p + n, k + 1
        fh.write(member(b""))


def timed(fn, reps: int):
    fn()                                    # warm-up: modules loaded, buffers sized, cub's sort instantiated
    ms, res = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return res, float(np.median(ms)), sorted(round(x, 2) for x in ms)


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
        L = len(w.ref)
        with tempfile.TemporaryDirectory() as tmp:
            srt, shuf = os.path.join(tmp, "sorted.bam"), os.path.join(tmp, "shuffled.bam")
            bamio.write_bam(srt, b, "ref", L, level=1)
            shuffled_copy(srt, shuf, 17)
            row = {"reads": b.n_reads, "sorted_bam_bytes": os.path.getsize(srt), "shuffled_bam_bytes": os.path.getsize(shuf)}
            _, row["sorted_ms"], row["sorted_ms_all"] = timed(lambda: ctx.bam_file_to_device(srt), args.reps)
            d, row["sorted_check_ms"], row["sorted_check_ms_all"] = timed(lambda: ctx.bam_file_to_device(srt, sort=True), args.reps)
            row["sorted_check_reordered"] = d.info["reordered"]
            row["payload_bytes"] = d.info["payload_bytes"]
            want = ctx.pileup_counts(d, L)
            sorts = []

            def shuffled():
                d = ctx.bam_file_to_device(shuf, sort=True)
                sorts.append(d.info["t_sort_s"] * 1e3)
                return d

            d, row["shuffled_sort_ms"], row["shuffled_sort_ms_all"] = timed(shuffled, args.reps)
            row["shuffled_reordered"] = d.info["reordered"]
            row["t_sort_ms"] = round(float(np.median(sorts[1:])), 3)
            row["t_sort_ms_all"] = sorted(round(x, 3) for x in sorts[1:])
            row["counts_equal"] = bool(np.array_equal(ctx.pileup_counts(d, L), want))
            row.update(info)
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": info, "results": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
