#!/usr/bin/env python
"""Benchmark of the pileup-and-call hot path (BASELINE.json: aligned bases/sec pileup+consensus).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scale S]

One *step* is one pass of the hot path over one synthetic sample of BASELINE.json configs[1]
(29,903-bp genome, 2 M ONT-like 400-bp amplicon reads, ~25,000x):
    pileup kernel + coverage scan -> call kernel + X-run scan -> insertion candidates -> ExtractInserts
    (select, depth cap, mate-overlap rewrite, count), chained on the device by tc_sample_enqueue / tc_sample_finish:
    one enqueue and one synchronisation per sample, step i + 1 enqueued before step i is finished.
`value`  : aligned bases/s with the reads already resident in HBM, CUDA-event timed.
`e2e`    : the same pass through the C-ABI with HOST (pinned) buffers: the H2D copy of every read
           array and the D2H copy of the count and call tables are inside the timed region.  Two samples travel at a
           time (two host threads, a context and a stream each): one's upload overlaps the other's kernels.
N > 1    : one process per GPU (torchrun), each rank piles up its own sample (the 96-sample plate
           of configs[2] sharded by sample): no data-path collective, weak scaling.
`read_range` (every N): configs[3], ONE ultra-deep sample sharded by read range, the per-rank tables summed
           with the pileup in one enqueue (tc_pileup_counts_allreduce, NCCL) inside the timed region — strong scaling, checked bit for bit
           against the single-GPU table.  `configs` (N = 1): tc_pileup_counts on the other configs.
           `parity_checked`: the GPU table over the cpu_baseline prefix equals the oracle's.
`--dump-outputs DIR`: after the timed steps, the last step's count table, call table and insertion calls go to DIR/<name>.npy
           (float64).  The sample is generated from a fixed seed, so two builds run with the same arguments can be compared
           output for output.
`--impl reference` times the CPU oracle port of the reference path (oracle/, all host threads) on a
bounded sample of the same workload; the reference itself is pure Python on pysam, which is not
installable here (DESIGN.md), so oracle/_ref does not exist.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "aligned_bases_per_sec_pileup_consensus"
UNIT = "aligned bases/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("pileup_kernel_dram_bytes_per_launch")
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi polled in the background.  It is started (and its first sample awaited) BEFORE the timed regions:
    the start-up of one nvidia-smi per rank (NVML initialisation) inside a timed region of a few milliseconds
    disturbed the launches of every rank.  Only samples taken inside the marked windows are reported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.rows = []          # (time, fields)
        self.windows = []       # [t0, t1]
        self.thread = None

    def start(self):
        import threading

        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()
        t_end = time.time() + 10.0
        while not self.rows and time.time() < t_end:        # NVML is up once the first sample is out
            time.sleep(0.01)

    def open_window(self):
        self.windows.append([time.time(), None])

    def close_window(self):
        if self.windows and self.windows[-1][1] is None:
            self.windows[-1][1] = time.time()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        # a window shorter than the polling interval may hold no sample: widen it by one interval on both sides
        wins = [(a - 0.06, (b if b is not None else time.time()) + 0.06) for a, b in self.windows]
        sm, mx, reasons = [], [], set()
        for t, f in self.rows:
            if wins and not any(a <= t <= b for a, b in wins):
                continue
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_sample(scale: float, sample: int):
    from trueconsense_b200 import synth

    w = synth.config(1, scale=scale)
    w.params.seed = w.params.seed * 1000 + sample
    batch = synth.generate_reads(w.params, w.ref)
    return w, batch


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(counts, table, calls) -> dict:
    """What a caller of the hot path receives from one step, as float64 host arrays (exact for every value here): the count
    table, the call table's columns and the insertion calls (strings as character codes, zero-padded; a call without
    entries is a row of zeros)."""
    names = ("call_char", "flags", "xrun", "rank_letter", "rank_count", "ambig_char")
    out = {"counts": counts.cpu().numpy()}
    out.update({n: t.cpu().numpy() for n, t in zip(names, table)})
    width = max([len(c["string"] or "") for c in calls], default=0)
    strings = np.zeros((len(calls), width))
    for i, c in enumerate(calls):
        strings[i, :len(c["string"] or "")] = [ord(ch) for ch in c["string"] or ""]
    for k in ("pos", "n_entries", "mode_count", "first_read"):
        out[f"insert_{k}"] = np.array([c[k] for c in calls])
    out["insert_string"] = strings
    return {k: v.astype(np.float64) for k, v in out.items()}


def dump_outputs(directory: str, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def hot_path(ctx, reads, L, mincov, counts_dev, table, flags_dev, stream, params=None, chained=True):
    """One pass: pileup -> call -> insertion candidates -> insertion calls.  Returns the calls.
    chained: tc_pileup_call_inserts (one enqueue, one synchronisation per sample); otherwise the four separate calls."""
    if chained:
        return ctx.pileup_call_inserts(reads, L, mincov, True, counts_dev, table, pileup=params, stream=stream)
    ctx.pileup_counts(reads, L, params, out=counts_dev, stream=stream)
    ctx.call_device(counts_dev, L, mincov, True, table, stream=stream)
    cands = ctx.list_insert_candidates(flags_dev, L)
    return ctx.extract_inserts(reads, L, cands)


def cpu_port(batch, L, mincov, threads, max_reads):
    """The oracle port of the reference path on the first max_reads reads (start-sorted prefix).
    Returns (aligned bases, seconds, sample description)."""
    from oracle import call, pileup

    sub = batch.slice(0, min(batch.n_reads, max_reads))
    bases = sub.count_aligned_bases(0x4)
    t0 = time.perf_counter()
    counts = pileup.pileup_counts(sub, L, threads=threads)
    t1 = time.perf_counter()
    call.call_table(counts.astype(np.int64), mincov, True)
    cands = call.insert_candidates(counts.astype(np.int64), mincov)
    for p in cands[:64]:
        cols = pileup.pileup_columns(sub, region=(p - 1, p), **pileup.EXTRACTINSERTS)
        call.extract_insert(cols[0][1] if cols else "")
    t2 = time.perf_counter()
    cpu_port.last = (sub, counts, cands)        # the oracle's table over the prefix: bench.py's parity check of the GPU path
    return bases, t2 - t0, f"first {sub.n_reads} start-sorted reads of the sample ({bases} aligned bases); pileup {t1 - t0:.2f}s + call/inserts {t2 - t1:.2f}s"


def host_decode_rate(batch, L, ctx=None, max_reads=200_000):
    """BAM decode, reported separately from the kernels (north_star): a bounded slice of the sample is written as a
    BGZF-compressed BAM and decoded back with all host threads.  Two ways: `cpu_parse` — inflate and record parsing on the
    host (csrc/host/bamio.c tc_bam_read), the arrays then still have to travel; `gpu_parse` — the product path: inflate + one
    hop over the records on the host (tc_bam_payload), the payload to the device once, record parsing and repacking there
    (tc_bam_records_to_reads), arrays resident in HBM when it returns; `gpu_inflate` — what indexing.BamHandle does: the
    file's bytes to the device as they are, BGZF members inflated and CRC-checked, records indexed and parsed there
    (gpu.Context.bam_file_to_device).  Returns a dict for the JSON line; its top-level rate is the last one's."""
    import tempfile

    from trueconsense_b200 import bamio

    sub = batch.slice(0, min(batch.n_reads, max_reads))
    bases = sub.count_aligned_bases(0)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "decode.bam")
        bamio.write_bam(path, sub, "ref", L, level=1)
        size = os.path.getsize(path)
        bamio.read_bam(path)                    # page cache and allocator warm for both ways
        t0 = time.perf_counter()
        back = bamio.read_bam(path)
        dt = time.perf_counter() - t0
        out = {"reads": int(back.n_reads), "bam_bytes": int(size), "threads": os.cpu_count() or 1,
               "cpu_parse": {"seconds": dt, "aligned_bases_per_s": bases / dt, "t_inflate_s": float(back.info.get("t_inflate_s", 0.0)),
                             "t_parse_s": float(back.info.get("t_parse_s", 0.0))}}
        if ctx is not None:
            import torch

            ctx.bam_to_device(bamio.read_bam_payload(path))        # buffers allocated
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            payload = bamio.read_bam_payload(path)
            t1 = time.perf_counter()
            dev = ctx.bam_to_device(payload)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            out["gpu_parse"] = {"seconds": t2 - t0, "aligned_bases_per_s": bases / (t2 - t0), "t_inflate_s": payload.info["t_inflate_s"],
                                "t_record_hop_s": payload.info["t_index_s"], "t_host_s": t1 - t0, "t_device_s": t2 - t1,
                                "payload_bytes": int(payload.n_bytes), "reads": int(dev.n_reads)}
            # the product path (indexing.BamHandle): the file's bytes travel as they are; inflate, CRC-32, record index and
            # parsing on the device — the host maps the file and reads one header per BGZF member
            ctx.bam_file_to_device(path)                           # buffers allocated
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev = ctx.bam_file_to_device(path)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            out["gpu_inflate"] = {"seconds": t3 - t0, "aligned_bases_per_s": bases / (t3 - t0), "reads": int(dev.n_reads),
                                  **{k: v for k, v in dev.info.items() if k.startswith("t_") or k in ("n_members", "payload_bytes")}}
            out["seconds"] = t3 - t0
            out["aligned_bases_per_s"] = bases / (t3 - t0)
            out["path"] = "gpu_inflate"
        else:
            out["seconds"] = dt
            out["aligned_bases_per_s"] = bases / dt
    return out


def time_pileup(ctx, dev, L, params, out, steps, warmup, torch):
    """Mean CUDA-event ms of tc_pileup_counts (device-resident reads, device output) and of its pileup kernel alone."""
    for _ in range(warmup):
        ctx.pileup_counts(dev, L, params, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = []
    e0.record()
    for _ in range(steps):
        ctx.pileup_counts(dev, L, params, out=out)
        k.append(ctx.last_pileup_kernel_ms())
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, statistics.mean(k)


def configs_block(ctx, gpu, torch, peak, steps, deep):
    """The other BASELINE configs on one GPU, device-resident, with a clock record of their own (the driver-run line carries
    them): tc_pileup_counts per sample — config 1 at full size, one sample of config 3's plate, config 4 at `deep_scale` of
    its 50 M reads (the read_range block's single-GPU pass: `deep`), config 5 at half its reads (the long-read path: span
    pass, split into pieces, sort, pileup)."""
    from trueconsense_b200 import synth

    out = {}
    if deep is not None:
        out[deep["workload"]] = {"reads": deep["reads"], "aligned_bases": deep["aligned_bases"], "pileup_counts_ms": deep["single_gpu_ms_per_pass"],
                                 "aligned_bases_per_s": deep["aligned_bases"] / (deep["single_gpu_ms_per_pass"] * 1e-3),
                                 "roofline_frac_call": deep["roofline_frac"], "note": "the read_range block's pass on one GPU"}
    for idx, scale in ((0, 1.0), (2, 1.0), (4, 0.5)):
        w = synth.config(idx, scale=scale)
        b = synth.generate_reads(w.params, w.ref)
        L = len(w.ref)
        dev = ctx.upload(b, with_qual=False)
        table = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
        bases = b.count_aligned_bases(0x4)
        alg = b.algorithmic_bytes(L)
        ms, k_ms = time_pileup(ctx, dev, L, gpu.buildindex_params(), table, steps, 3, torch)
        out[w.name] = {"scale": scale, "reads": int(b.n_reads), "ref_len": L, "aligned_bases": int(bases), "algorithmic_bytes": int(alg),
                       "pileup_counts_ms": ms, "pileup_kernel_ms": k_ms, "aligned_bases_per_s": bases / (ms * 1e-3),
                       "roofline_frac_kernel": alg / (k_ms * 1e-3) / 1e9 / peak, "roofline_frac_call": alg / (ms * 1e-3) / 1e9 / peak}
        del dev, table, b
    return out


def read_range_block(ctx, gpu, torch, dist, rank, world, local, steps, warmup, deep_scale, peak):
    """BASELINE configs[3]: ONE ultra-deep sample sharded by read range — every rank piles up a contiguous slice of the
    start-sorted reads into a full-length table, the tables are summed with tc_allreduce_counts (NCCL int32 sum over NVLink)
    inside the timed region.  Strong scaling: the sample is fixed, the ranks share it.  Rank 0 also piles up the whole sample
    alone: the summed table must equal that table bit for bit, and its time is the 1-GPU reference of the efficiency."""
    from trueconsense_b200 import sharding, synth

    w = synth.config(3, scale=deep_scale)
    n_reads = int(w.params.n_reads)
    L = len(w.ref)
    lo, hi = sharding.read_range(n_reads, rank, world)
    shard = synth.generate_reads(w.params, w.ref, read_range=(lo, hi))
    dev = ctx.upload(shard, with_qual=False)
    out = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
    p = gpu.buildindex_params()
    p.max_depth = 0                 # the depth cap is a property of the SUMMED coverage (checked below), not of a shard
    comm = sharding.NcclComm(rank, world, local) if world > 1 else None
    stream = torch.cuda.current_stream().cuda_stream

    out_b = torch.empty_like(out)      # two passes in flight, a table each

    def run_passes(n):
        """n passes of the shard (+ sum): pass i + 1 is enqueued before pass i is finished, like the samples of the main loop"""
        if comm is None:
            for _ in range(n):
                ctx.pileup_counts(dev, L, p, out=out, stream=stream)
            return
        ticket = ctx.pileup_counts_allreduce_enqueue(dev, L, p, out, comm, stream=stream)
        for i in range(n):
            nxt = None
            if i + 1 < n:
                nxt = ctx.pileup_counts_allreduce_enqueue(dev, L, p, out if i % 2 else out_b, comm, stream=stream)
            ctx.pileup_counts_allreduce_finish(ticket)
            ticket = nxt

    def one_pass():
        if comm is not None:
            ctx.pileup_counts_allreduce(dev, L, p, out, comm, stream=stream)
        else:
            ctx.pileup_counts(dev, L, p, out=out, stream=stream)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run_passes(2 * max(warmup, 3))
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_passes(steps)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1) / steps
    ar_ms = 0.0
    ar_iso_ms = 0.0
    if comm is not None:            # the collective alone (the table is summed in place over and over: timing only)
        scratch = out.clone()
        for _ in range(3):
            ctx.allreduce_counts(scratch, comm, stream=stream)
        sync()
        e0.record()
        for _ in range(steps):
            ctx.allreduce_counts(scratch, comm, stream=stream)
        e1.record()
        sync()
        ar_ms = e0.elapsed_time(e1) / steps
        ar_iso = []                 # ... and one at a time, every rank idle before it: the latency a pass pays
        for _ in range(min(steps, 20)):
            sync()
            e0.record()
            ctx.allreduce_counts(scratch, comm, stream=stream)
            e1.record()
            torch.cuda.synchronize()
            ar_iso.append(e0.elapsed_time(e1))
        ar_iso_ms = statistics.median(ar_iso)
        one_pass()                  # `out` again holds the sum of the shards' tables
    t = torch.tensor([ms, ar_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ar_ms = float(t[0]), float(t[1])
    # ---- the single-GPU table and time (rank 0), and the comparison on every rank
    single = torch.empty_like(out)
    single_ms = ms
    if world > 1:
        if rank == 0:
            whole = synth.generate_reads(w.params, w.ref)
            ctx2 = gpu.Context(local)
            dev2 = ctx2.upload(whole, with_qual=False)
            single_ms, _ = time_pileup(ctx2, dev2, L, gpu.buildindex_params(), single, steps, 3, torch)
            bases = whole.count_aligned_bases(0x4)
            alg = whole.algorithmic_bytes(L)
            meta = torch.tensor([single_ms, float(bases), float(alg)], dtype=torch.float64, device="cuda")
            del dev2, ctx2, whole
        else:
            meta = torch.zeros(3, dtype=torch.float64, device="cuda")
        dist.broadcast(single, src=0)
        dist.broadcast(meta, src=0)
        single_ms, bases, alg = float(meta[0]), float(meta[1]), float(meta[2])
        equal = torch.tensor([int(torch.equal(out, single))], device="cuda")
        dist.all_reduce(equal, op=dist.ReduceOp.MIN)
        equal = bool(equal.item())
    else:
        bases = float(shard.count_aligned_bases(0x4))
        alg = float(shard.algorithmic_bytes(L))
        ctx.pileup_counts(dev, L, gpu.buildindex_params(), out=single)      # with the depth cap proven non-binding
        equal = bool(torch.equal(out, single))
    sharding.check_depth_cap(int(out[0].max().item()), 0, 10_000_000)
    if comm is not None:
        comm.close()
    block = {
        "workload": w.name, "sharding": "by read range, tc_pileup_counts_allreduce_enqueue / _finish per pass (shard pileup + ncclAllReduce int32 sum in one enqueue, replayed as a CUDA graph, pass i + 1 enqueued before pass i is finished)",
        "scaling": "strong", "n_gpus": world, "reads": n_reads, "reads_per_rank": int(hi - lo), "aligned_bases": bases,
        "ms_per_pass": ms, "aligned_bases_per_s": bases / (ms * 1e-3), "allreduce_ms": ar_ms, "allreduce_isolated_ms": ar_iso_ms, "allreduce_bytes": int(out.numel() * 4),
        "single_gpu_ms_per_pass": single_ms, "strong_scaling_efficiency": single_ms / (world * ms),
        "roofline_frac": alg / (ms * 1e-3) / 1e9 / (peak * world), "table_equals_single_gpu": equal,
        "limiter": ("pileup of the shard (%.3f ms) + allreduce of %.2f MB (%.3f ms: latency-bound on NVLink)" %
                    (ms - ar_ms, out.numel() * 4 / 1e6, ar_ms)) if world > 1 else "one GPU: no collective",
    }
    del dev, out, single, shard
    import gc

    gc.collect()
    return block


def h2d_ceiling(torch, dist, world, nbytes, steps=5):
    """What the box gives all ranks at once for pinned host -> device copies of one sample's size: the end-to-end number is
    PCIe / host-memory bound, and the ranks share the host's memory path."""
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    devb = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        devb.copy_(host, non_blocking=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        devb.copy_(host, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return {"bytes_per_rank": int(nbytes), "ms": float(ms[0]), "gb_per_s_per_rank": nbytes / (float(ms[0]) * 1e-3) / 1e9,
            "gb_per_s_all_ranks": world * nbytes / (float(ms[0]) * 1e-3) / 1e9}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pileup

    pileup.build()
    threads = os.cpu_count() or 1
    w, batch = make_sample(args.scale, 0)
    L = len(w.ref)
    max_reads = int(args.ref_reads)
    times, bases = [], 0
    desc = ""
    for i in range(args.warmup + args.steps):
        b, t, desc = cpu_port(batch, L, w.mincov, threads, max_reads)
        if i >= args.warmup:
            times.append(t); bases = b
    v = bases * len(times) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": w.name, "ref_len": L, "reads_per_sample": batch.n_reads, "mincov": w.mincov,
                   "note": "CPU oracle port of the reference path (C pileup engine + classifier, OpenMP over read ranges); "
                           "the reference's own path is pure Python on pysam/htslib, not installable in this image"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # stdout carries the one JSON line and nothing else
    import torch
    import torch.distributed as dist

    from trueconsense_b200 import gpu

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU implementation")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = gpu.Context(local)
    if args.read_range_only:        # diagnostics: the read-range block alone (not a bench line)
        rr = read_range_block(ctx, gpu, torch, dist, rank, world, local, args.steps, args.warmup, args.deep_scale, peaks()[0])
        if rank == 0:
            print(json.dumps({"read_range": rr}))
        if world > 1:
            dist.destroy_process_group()
        return
    w, batch = make_sample(args.scale, rank)
    L = len(w.ref)
    bases = batch.count_aligned_bases(0x4)
    alg_bytes = batch.algorithmic_bytes(L)
    # the host batch in its compact transport forms: 16-bit CIGARs (when every operation is shorter than 4096), two bits per base
    # plus the words that hold anything else than A C G T (what a decoder emits next to the 4-bit words: tc_seq2_pack)
    pinned = batch.with_cigar16().with_seq2().pin()
    stream = torch.cuda.current_stream().cuda_stream

    counts_dev = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
    call_char = torch.empty(L, dtype=torch.uint8, device="cuda")
    flags_dev = torch.empty(L, dtype=torch.uint8, device="cuda")
    xrun = torch.empty(L, dtype=torch.int32, device="cuda")
    rank_letter = torch.empty((4, L), dtype=torch.uint8, device="cuda")
    rank_count = torch.empty((4, L), dtype=torch.int32, device="cuda")
    ambig = torch.empty(L, dtype=torch.uint8, device="cuda")
    table = gpu.CallTable(call_char.data_ptr(), flags_dev.data_ptr(), xrun.data_ptr(), rank_letter.data_ptr(),
                          rank_count.data_ptr(), ambig.data_ptr())
    # a second set of outputs: two samples are in flight at a time
    counts_dev2 = torch.empty_like(counts_dev)
    out2 = [torch.empty_like(x) for x in (call_char, flags_dev, xrun, rank_letter, rank_count, ambig)]
    table2 = gpu.CallTable(*[x.data_ptr() for x in out2])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident: `value`
    dev = ctx.upload(pinned, stream)
    torch.cuda.synchronize()
    ctx.set_timing(True)
    params = gpu.buildindex_params(args.kernel)
    sampler = ClockSampler(local)
    sampler.start()
    # spin-up (not steps): W warm-up passes are 2-3 ms of GPU work, far less than a cold GPU needs to reach its clocks and
    # the driver to settle — the first run on a fresh box measured 0.93 ms per step where every later run measured 0.74
    t_spin = time.time() + args.spinup
    while time.time() < t_spin:
        hot_path(ctx, dev, L, w.mincov, counts_dev, table, flags_dev, stream, params)
    for _ in range(args.warmup):
        calls = hot_path(ctx, dev, L, w.mincov, counts_dev, table, flags_dev, stream, params)
    barrier()
    sampler.open_window()
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    ev0.record()
    if args.unchained:
        for _ in range(args.steps):
            calls = hot_path(ctx, dev, L, w.mincov, counts_dev, table, flags_dev, stream, params, chained=False)
            kernel_ms.append(ctx.last_pileup_kernel_ms())
    else:
        # one enqueue per sample, and the host's share of a step (unpacking the calls, the next enqueue) behind the device's
        # work on the next step: step i + 1 is enqueued (same stream, its own count / call tables) before step i is finished
        ticket = ctx.sample_enqueue(dev, L, w.mincov, True, counts_dev, table, pileup=params, stream=stream)
        for i in range(1, args.steps + 1):
            nxt = None
            if i < args.steps:
                c2, t2 = (counts_dev2, table2) if i % 2 else (counts_dev, table)
                nxt = ctx.sample_enqueue(dev, L, w.mincov, True, c2, t2, pileup=params, stream=stream)
            calls = ctx.sample_finish(ticket)
            kernel_ms.append(ctx.last_pileup_kernel_ms())
            ticket = nxt
    ev1.record()
    barrier()
    sampler.close_window()
    launches = ctx.launches - launches0
    ms_total = ev0.elapsed_time(ev1)
    dumped = None
    if args.dump_outputs and rank == 0:
        # the chained loop alternates two sets of tables: step s wrote the second set when s is even; the end-to-end loop
        # below writes into both count tables, so the last step's outputs are read back here
        last = (counts_dev2, out2) if args.steps % 2 == 0 and not args.unchained else \
            (counts_dev, (call_char, flags_dev, xrun, rank_letter, rank_count, ambig))
        dumped = step_outputs(*last, calls)
    # ---------------- end to end through the C-ABI with host buffers: `e2e`
    # Two samples travel at a time: two host threads, each with a context, a stream and output buffers of its own, so one
    # sample's upload overlaps the other's kernels and read-backs (every call below blocks its own thread only; the C-ABI
    # releases the interpreter lock).  The copies share the one PCIe link: the step time is the upload time.
    import threading

    n_lanes = max(1, min(2, args.e2e_lanes))
    lanes = [(ctx, torch.cuda.Stream(), counts_dev)]
    if n_lanes == 2:
        lanes.append((gpu.Context(local), torch.cuda.Stream(), counts_dev2))

    def e2e_step(lane):
        c, ts, cdev = lanes[lane]
        st = ts.cuda_stream
        d = c.upload(pinned, st, with_qual=False)            # H2D of every read array the pileup needs (pinned memory)
        c.pileup_counts(d, L, params, out=cdev, stream=st)
        res = c.call(cdev, L, w.mincov, True, stream=st)     # D2H of the call table
        cands = c.list_insert_candidates(res.flags, L, stream=st)
        ins = c.extract_inserts(d.with_host_qual(), L, cands, stream=st)     # H2D of QUAL over the candidate columns only
        h = c.download(cdev.data_ptr(), cdev.numel(), np.int32, stream=st)   # D2H of the count table
        return h, res, ins

    def e2e_run(n_steps):
        last, errs = [None] * n_lanes, []

        def lane_loop(lane, n):
            try:
                torch.cuda.set_device(local)
                for _ in range(n):
                    last[lane] = e2e_step(lane)
            except BaseException as e:      # noqa: BLE001 — re-raised on the main thread
                errs.append(e)

        ths = [threading.Thread(target=lane_loop, args=(k, (n_steps + n_lanes - 1 - k) // n_lanes)) for k in range(n_lanes)]
        for t_ in ths:
            t_.start()
        for t_ in ths:
            t_.join()
        if errs:
            raise errs[0]
        return last[0]

    e2e_run(n_lanes * min(args.warmup, 2))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    xfer0 = [c.transfer_bytes() for c, _, _ in lanes]
    sampler.open_window()
    e0.record()
    h, res, ins = e2e_run(args.steps)
    torch.cuda.synchronize()        # both lanes' streams: e1 is stamped behind everything
    e1.record()
    barrier()
    sampler.close_window()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()          # sampled over both timed regions (device-resident steps, then end-to-end steps)
    h2d = sum(c.transfer_bytes()[0] - x[0] for (c, _, _), x in zip(lanes, xfer0)) // args.steps
    d2h = sum(c.transfer_bytes()[1] - x[1] for (c, _, _), x in zip(lanes, xfer0)) // args.steps
    for c, _, _ in lanes[1:]:
        c.close()
    # ---------------- max over ranks
    t = torch.tensor([ms_total, e2e_ms, float(bases), float(launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, e2e_ms = float(tmax[0]), float(tmax[1])
        total_bases, launches = float(tsum[2]), int(tsum[3])
    else:
        total_bases = float(bases)
    peak, peak_src = peaks()
    ceiling = h2d_ceiling(torch, dist, world, int(h2d)) if world > 1 or args.h2d_ceiling else None
    rr = None
    if not args.no_read_range:
        rr = read_range_block(ctx, gpu, torch, dist, rank, world, local, args.steps, args.warmup, args.deep_scale, peak)
    cfgs = None
    if world == 1 and not args.no_configs:
        cfgs = configs_block(ctx, gpu, torch, peak, args.steps, rr)
    parity = None
    if rank == 0:
        k_ms = statistics.mean(kernel_ms)
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        value = total_bases * args.steps / (ms_total * 1e-3)
        e2e_v = total_bases * args.steps / (e2e_ms * 1e-3)
        cpu = None
        if world == 1:          # the CPU baseline is reported by the single-GPU run only (scaling runs stay short)
            from oracle import pileup as opile

            opile.build()
            cb, ct, desc = cpu_port(batch, L, w.mincov, 1, int(args.cpu_reads))
            cpu = {"value": cb / ct, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc}
            # parity at benchmark size, outside every timed region: the GPU's table, call flags and insertion candidates over
            # the same prefix of the benchmarked sample must equal the oracle's
            sub, o_counts, o_cands = cpu_port.last
            g_counts = ctx.pileup_counts(sub, L, params)
            g_res = ctx.call(g_counts, L, w.mincov, True)
            g_cands = ctx.list_insert_candidates(g_res.flags, L)
            parity = bool(np.array_equal(g_counts, o_counts)) and list(g_cands) == list(o_cands)
            if not parity:
                raise SystemExit("bench.py: the GPU count table / candidates differ from the oracle's on the benchmarked sample")
        try:
            decode = host_decode_rate(batch, L, ctx)
        except Exception as e:      # reporting aid only
            decode = {"error": str(e)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": w.name, "ref_len": L, "reads_per_sample": batch.n_reads, "samples": world,
                       "aligned_bases_per_sample": bases, "mincov": w.mincov, "sharding": "by sample, no collective",
                       "l2": f"inputs {alg_bytes / 1e6:.0f} MB per pass exceed the 126 MB L2 (no flush needed)",
                       "insert_candidates": len(calls),
                       "step": "tc_sample_enqueue + tc_sample_finish (chained, step i + 1 enqueued before step i is finished)"
                               if not args.unchained else "four separate calls, three synchronisations"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(), "kernel": "pileup kernel (tc_pileup_counts)", "kernel_ms": k_ms,
                         "algorithmic_bytes": alg_bytes, "peak_source": peak_src},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "host_decode": decode,
            "parity_checked": parity,
            "read_range": rr,
            "configs": cfgs,
        }
        if ceiling is not None:
            line["e2e"]["h2d_ceiling"] = ceiling
            line["e2e"]["h2d_frac_of_ceiling"] = (h2d / (e2e_ms / args.steps * 1e-3) / 1e9) / ceiling["gb_per_s_per_rank"]
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", type=int, default=0, help="pileup kernel variant (0 = library's choice; A/B measurements only)")
    ap.add_argument("--unchained", action="store_true", help="the four separate calls per step (three synchronisations) instead of tc_sample_enqueue / tc_sample_finish")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the 2 M reads of configs[1] (tests only)")
    ap.add_argument("--spinup", type=float, default=0.5, help="seconds of untimed passes before the warm-up steps (clock / driver spin-up of a cold GPU)")
    ap.add_argument("--deep-scale", type=float, default=1.0, help="fraction of configs[3]'s 50 M reads in the read-range block (1.0: the whole sample, 4.8 GB of read arrays on one GPU)")
    ap.add_argument("--no-read-range", action="store_true", help="skip the read-range sharded block (configs[3])")
    ap.add_argument("--read-range-only", action="store_true", help="diagnostics: only the read-range block, printed on its own")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block (N = 1 only)")
    ap.add_argument("--e2e-lanes", type=int, default=2, help="samples travelling at a time in the end-to-end loop (1 or 2)")
    ap.add_argument("--h2d-ceiling", action="store_true", help="also measure the concurrent pinned H2D ceiling at N = 1")
    ap.add_argument("--cpu-reads", type=float, default=1_000_000, help="reads in the cpu_baseline sample (1 M reads = 400 M aligned bases, 10-15 s on one core)")
    ap.add_argument("--ref-reads", type=float, default=400_000, help="reads per step of the --impl reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's sample) to DIR/<name>.npy "
                                                         "as float64: count table, call table, insertion calls")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
