"""Time the multi-reference device pass against one single-reference pass per reference, on one GPU.

    python scripts/contigs_rate.py [--reads 1500000] [--refs1000-reads 1000000] [--reps 5]

Two seeded samples: 8 influenza-like segments (890-2341 bp, 150-bp pairs), and 1000 references of 1-3 kb.  For each:
  * contigs: one BamHandle over the multi-reference BAM: decode on the device, tc_bam_contig_ranges, tc_reads_to_contig_coords,
    one tc_pileup_counts, tc_call_contigs, the candidate list and one tc_extract_inserts;
  * single:  the same work per reference over a BAM of that reference alone (decode, pileup, tc_call, candidates, inserts).
Prints the card's name and power limit, then one JSON line per sample: ms per sample (median of --reps, host clock around
work that ends with results on the host), kernel launches per sample, and whether both ways computed the same counts and
insertion calls.  Everything it writes goes to a temporary directory."""
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
from trueconsense_b200 import bamio, gpu, indexing, synth  # noqa: E402

FLU_LENGTHS = [2341, 2341, 2233, 1778, 1565, 1413, 1027, 890]


def card() -> dict:
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("contigs_rate.py measures on a CUDA device; none is available")
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:          # the query is informative only
        out["power_limit"] = f"unknown ({e})"
    return out


def bgzf(path: str, payload: bytes) -> None:
    def member(chunk: bytes) -> bytes:
        c = zlib.compressobj(1, zlib.DEFLATED, -15, 8, 0)
        data = c.compress(chunk) + c.flush()
        return (bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<HHHH", 6, 0x4342, 2, 18 + len(data) + 8 - 1) + data +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    with open(path, "wb") as fh:
        fh.write(b"".join([member(payload[p:p + 65280]) for p in range(0, len(payload), 65280)] + [member(b"")]))


def make_sample(tmp: str, lens: list[int], n_reads: int, seed: int):
    """Per-reference BAM + FASTA files and the multi-reference BAM + FASTA built from them (records spliced, refIDs set)."""
    refs, body, n_total = [], [], 0
    total = sum(lens)
    fasta = os.path.join(tmp, "all.fasta")
    with open(fasta, "w") as fa:
        for k, L in enumerate(lens):
            name = f"r{k:04d}"
            seq, feats = synth.make_genome(L, seed + k, "sars2")
            a = feats[0]["start"] - 1 if feats else 10
            vs = [synth.Variant(a + 30, synth.VAR_INS, 3, 5 + k, 0.9), synth.Variant(a + 90, synth.VAR_DEL, 3, 0, 0.8)]
            p = synth.SynthParams(seed=seed * 7 + k, n_reads=max(1, n_reads * L // total), ref_len=L, read_len=150, paired=True,
                                  sub_rate=0.005, softclip_rate=0.02, softclip_max=8, variants=vs)
            b = synth.generate_reads(p, seq)
            n_total += b.n_reads
            path = os.path.join(tmp, f"{name}.bam")
            bamio.write_bam(path, b, name, L, level=1)
            with open(os.path.join(tmp, f"{name}.fasta"), "w") as fh:
                fh.write(f">{name}\n{seq}\n")
            fa.write(f">{name}\n{seq}\n")
            refs.append((name, L, path))
            with gzip.open(path, "rb") as fh:
                payload = fh.read()
            q = bamio.parse_bam_header(payload, len(payload))[2]
            raw = bytearray(payload[q:])
            o = 0
            while o + 4 <= len(raw):            # refID and next refID of every record -> k
                bs = struct.unpack_from("<i", raw, o)[0]
                struct.pack_into("<i", raw, o + 4, k)
                if struct.unpack_from("<i", raw, o + 24)[0] >= 0:
                    struct.pack_into("<i", raw, o + 24, k)
                o += 4 + bs
            body.append(bytes(raw))
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    hdr = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for name, L, _ in refs:
        hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", L)
    multi = os.path.join(tmp, "all.bam")
    bgzf(multi, hdr + b"".join(body))
    return refs, multi, n_total


def contigs_pass(ctx, bam: str, names, lens):
    h = indexing.BamHandle(bam)
    d, lay = h.device_reads_contigs(names, lens)
    counts = ctx.pileup_counts(d, lay.total)
    table = ctx.call_contigs(counts, lay.start, 30, True)
    cands = ctx.list_insert_candidates(table.flags, lay.total)
    ins = ctx.extract_inserts(d, lay.total, cands) if len(cands) else []
    k, local = lay.locate(cands)
    calls = [(int(kk), int(p), r["string"], r["n_entries"]) for kk, p, r in zip(k, local, ins)]
    return counts, lay.start, calls


def single_passes(ctx, refs):
    out_counts, calls = [], []
    for k, (_, L, path) in enumerate(refs):
        d = indexing.BamHandle(path).device_reads()
        counts = ctx.pileup_counts(d, L)
        table = ctx.call(counts, L, 30, True)
        cands = ctx.list_insert_candidates(table.flags, L)
        ins = ctx.extract_inserts(d, L, cands) if len(cands) else []
        out_counts.append(counts)
        calls += [(k, int(p), r["string"], r["n_entries"]) for p, r in zip(cands, ins)]
    return out_counts, calls


def timed(fn, reps: int, ctx):
    fn()                                    # warm-up: modules loaded, buffers sized
    ms, launches = [], []
    for _ in range(reps):
        l0 = ctx.launches
        t0 = time.perf_counter()
        res = fn()
        ms.append((time.perf_counter() - t0) * 1e3)
        launches.append(ctx.launches - l0)
    return res, float(np.median(ms)), sorted(ms), launches[-1]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, default=1_500_000, help="reads of the 8-segment sample")
    ap.add_argument("--refs1000-reads", type=int, default=1_000_000, help="reads of the 1000-reference sample")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    ctx = gpu.default_context()
    rng = np.random.default_rng(3)
    cases = [("8_segments", FLU_LENGTHS, args.reads), ("1000_references", [int(x) for x in rng.integers(1000, 3000, 1000)],
                                                        args.refs1000_reads)]
    for label, lens, n_reads in cases:
        with tempfile.TemporaryDirectory() as tmp:
            refs, multi, n_total = make_sample(tmp, lens, n_reads, 1000 + len(lens))
            names = [r[0] for r in refs]
            (counts, start, calls_m), ms_m, all_m, l_m = timed(lambda: contigs_pass(ctx, multi, names, lens), args.reps, ctx)
            (counts_s, calls_s), ms_s, all_s, l_s = timed(lambda: single_passes(ctx, refs), args.reps, ctx)
            equal = all(np.array_equal(counts[:, start[k]:start[k + 1]], counts_s[k]) for k in range(len(refs))) and calls_m == calls_s
            print(json.dumps({"sample": label, "references": len(lens), "reads": n_total,
                              "columns": int(start[-1]), "insertion_calls": len(calls_m),
                              "contigs_ms": round(ms_m, 2), "contigs_ms_all": [round(x, 2) for x in all_m], "contigs_launches": l_m,
                              "single_ms": round(ms_s, 2), "single_ms_all": [round(x, 2) for x in all_s], "single_launches": l_s,
                              "equal": bool(equal), **info}), flush=True)


if __name__ == "__main__":
    main()
