"""What clipping amplicon primers off the reads (``--primers --primer-both-ends``) adds to a decode, on one GPU.

    python scripts/clip_rate.py [--reads 200000 1000000] [--reps 5] [--check-max 200000] [--out profiles/clip_rate.json]

For each read count: a seeded config-2-like read set (ONT amplicon reads of ~400 bp, synth.config(1): 98 overlapping amplicons
tiled over 29,903 bp) whose reads start and end within 3 bases of their amplicon's ends (read_len_jitter 3), and an
ARTIC-like scheme with a 24-base primer at both ends of every amplicon.  The reads are written as a sorted BAM and as a
sorted SAM.  Timed (host clock around each call, which ends in a device synchronise; one warm-up, median of --reps):
  * bam / bam_primers:  gpu.Context.bam_file_to_device(path[, primers=scheme])
  * sam / sam_primers:  gpu.Context.sam_file_to_device(path[, primers=scheme])
with ``.info``'s steps of the last call (``t_clip_s`` among them), and the clip kernels alone: CUDA events around
``Context.clip_primers`` on device-resident records (primer tables up, plan, scan, pack, stats back; median of --reps).
Checks: up to --check-max reads, the arrays of both routes with primers equal the plain decode of a BAM holding
oracle/primer_clip.py's clipped and sorted records; above it, the two routes' arrays equal each other.
Prints the card's name, power limit and max SM clock, then one JSON line per read count; --out also writes them as one JSON
document.  The files go to a temporary directory."""
import argparse
import dataclasses
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from oracle import primer_clip  # noqa: E402
from sam_rate import MM2_AUX, arrays, bgzf, card, records, same, sam_line, steps, timed  # noqa: E402
from trueconsense_b200 import bamio, gpu, primers, synth  # noqa: E402


def scheme_rows(p: synth.SynthParams, L: int):
    """A 24-base primer at both ends of each of the generator's amplicons (synth.c: start = room * a / (n - 1))."""
    room = L - p.read_len - p.read_len_jitter
    rows = []
    for a in range(p.n_amplicons):
        s = room * a // (p.n_amplicons - 1)
        rows += [(0, s, s + 24), (0, s + p.read_len - 24, s + p.read_len)]
    return rows


def clip_event_ms(ctx, payload, scheme, reps: int):
    """CUDA events around Context.clip_primers on device-resident records."""
    import torch

    pay = torch.from_numpy(np.ctypeslib.as_array((np.ctypeslib.ctypes.c_uint8 * payload.n_bytes).from_address(payload.payload_ptr))).cuda()
    rec = torch.from_numpy(np.ctypeslib.as_array((np.ctypeslib.ctypes.c_int64 * payload.n_reads).from_address(payload.rec_off_ptr))).cuda()
    torch.cuda.synchronize()
    ms = []
    for k in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.clip_primers(pay.data_ptr(), payload.n_bytes, rec.data_ptr(), payload.n_reads, payload.ref_names, scheme)
        e1.record()
        torch.cuda.synchronize()
        if k:
            ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), sorted(round(x, 3) for x in ms)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, nargs="+", default=[200_000, 1_000_000])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--check-max", type=int, default=200_000, help="largest read count checked against the Python oracle")
    ap.add_argument("--out", default=None, help="also write the results here as one JSON document")
    args = ap.parse_args()
    info = card()
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
            p = {k: os.path.join(tmp, k) for k in ("sorted.bam", "sorted.sam", "scheme.bed")}
            bamio.write_bam(p["sorted.bam"], b, "ref", L, level=1)
            head, names, lens, recs = records(p["sorted.bam"])
            with open(p["scheme.bed"], "w") as fh:
                fh.write("".join(f"ref\t{s}\t{e}\tamp\t1\n" for _, s, e in rows))
            scheme = primers.read_bed(p["scheme.bed"], 5, True)
            bnames = [x.encode() for x in names]
            sam_head = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (x, l) for x, l in zip(bnames, lens))
            with open(p["sorted.sam"], "wb") as fh:
                fh.write(sam_head + b"".join(sam_line(r, bnames, MM2_AUX % (i % 7)) for i, r in enumerate(recs)))
            row = {"reads": b.n_reads, "primers": len(rows), "tolerance": 5, "both_ends": True,
                   "bytes": {k: os.path.getsize(v) for k, v in p.items()}}
            got = {}
            for route, fn in (("bam", ctx.bam_file_to_device), ("sam", ctx.sam_file_to_device)):
                for tag, kw in (("", {}), ("_primers", {"primers": scheme})):
                    d, row[f"{route}{tag}_ms"], row[f"{route}{tag}_ms_all"] = timed(lambda: fn(p[f"sorted.{route}"], **kw), args.reps)
                    row[f"{route}{tag}_steps_ms"] = steps(d.info)
                    if tag:
                        row[f"{route}_clip_stats"] = {k: d.info[k] for k in ("n_clipped_left", "n_clipped_right", "n_fully_clipped",
                                                                              "clipped_columns")}
                        got[route] = arrays(ctx, d)
            row["bam_primers_equals_sam_primers"] = same(got["bam"], got["sam"])
            if b.n_reads <= args.check_max:
                clipped, st = primer_clip.clip_and_sort(recs, rows, 5, True)
                bgzf(os.path.join(tmp, "oracle.bam"), head + b"".join(clipped))
                want = arrays(ctx, ctx.bam_file_to_device(os.path.join(tmp, "oracle.bam")))
                row["oracle_stats"] = st
                row["bam_primers_equals_oracle"] = same(got["bam"], want)
                row["sam_primers_equals_oracle"] = same(got["sam"], want)
                del clipped, want
            del recs, got
            payload = bamio.read_bam_payload(p["sorted.bam"])
            row["clip_event_ms"], row["clip_event_ms_all"] = clip_event_ms(ctx, payload, scheme, args.reps)
            payload.release()
            row.update(info)
            print(json.dumps(row), flush=True)
            out.append(row)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": info, "results": out}, fh, indent=1)


if __name__ == "__main__":
    main()
