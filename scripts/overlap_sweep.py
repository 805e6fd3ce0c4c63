"""How many SMs the pileup kernel should leave to the previous sample's tail (TC_OVERLAP_SMS, sample.cu).

    python scripts/overlap_sweep.py [--steps 200] [--rounds 5] [--out profiles/overlap_sweep.json] [--trace-dir DIR]

bench.py's chained loop over its sample (configs[1]: 2 M ONT amplicon reads, 29,903 columns, device-resident; two sets of
outputs, sample i + 1 enqueued before sample i is finished), timed with CUDA events around a window that starts and ends
host-synchronised, for each setting:
  * "off" (TC_OVERLAP_SMS=-1): every tail behind its head on the caller's stream, as one stream serialises them;
  * k = 0, 2, 4, 6, 8, 12, 16: tails on the context's own stream, the pileup kernel launched on sm_count - k CTAs while the other
    sample's tail can still be running (k = 0: the full grid).
The settings take turns, --rounds times; reported per setting: median / min / max ms per step and the mean pileup-kernel time
(CUDA events around the kernel, tc_last_pileup_kernel_ms).  Then, with --trace-dir, one torch.profiler run (CUDA activities)
of a few steps at the library's default k: its Chrome trace goes to DIR, and the JSON counts how many of step i's tail
kernels ran inside step i + 1's warp_pileup_kernel.  Prints the card's name, power limit and max SM clock with the results."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from sam_rate import card  # noqa: E402

SETTINGS = ("off", "0", "2", "4", "6", "8", "12", "16")
TAIL = ("call_kernel", "xrun_", "list_candidates", "rank_sort", "cand_range", "ins_")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "overlap_sweep.json"))
    ap.add_argument("--trace-dir", help="also write a torch.profiler trace of a few steps here")
    args = ap.parse_args()
    info = card()
    import torch

    from trueconsense_b200 import gpu, synth

    w = synth.config(1)
    batch = synth.generate_reads(w.params, w.ref)
    L = len(w.ref)
    ctx = gpu.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    dev = ctx.upload(batch.with_cigar16().with_seq2().pin(), stream)
    outs = []
    for _ in range(2):
        counts = torch.empty((gpu.TC_NROWS, L), dtype=torch.int32, device="cuda")
        cols = [torch.empty(L, dtype=torch.uint8, device="cuda"), torch.empty(L, dtype=torch.uint8, device="cuda"),
                torch.empty(L, dtype=torch.int32, device="cuda"), torch.empty((4, L), dtype=torch.uint8, device="cuda"),
                torch.empty((4, L), dtype=torch.int32, device="cuda"), torch.empty(L, dtype=torch.uint8, device="cuda")]
        outs.append((counts, cols, gpu.CallTable(*[c.data_ptr() for c in cols])))
    params = gpu.buildindex_params()
    ctx.set_timing(True)

    def chained(n):
        """n samples, two in flight; returns the pileup-kernel ms of each"""
        ms = []
        t = ctx.sample_enqueue(dev, L, w.mincov, True, outs[0][0], outs[0][2], pileup=params, stream=stream)
        for i in range(1, n + 1):
            nxt = None
            if i < n:
                c, _, tb = outs[i % 2]
                nxt = ctx.sample_enqueue(dev, L, w.mincov, True, c, tb, pileup=params, stream=stream)
            ctx.sample_finish(t)
            ms.append(ctx.last_pileup_kernel_ms())
            t = nxt
        return ms

    def setting(k):
        os.environ["TC_OVERLAP_SMS"] = "-1" if k == "off" else k

    res = {k: {"ms_per_step": [], "kernel_ms": []} for k in SETTINGS}
    for _ in range(args.rounds):
        for k in SETTINGS:
            setting(k)
            chained(args.warmup)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            kms = chained(args.steps)
            e1.record()
            torch.cuda.synchronize()
            res[k]["ms_per_step"].append(e0.elapsed_time(e1) / args.steps)
            res[k]["kernel_ms"].append(statistics.mean(kms))
    rows = {}
    for k in SETTINGS:
        v = res[k]["ms_per_step"]
        rows[k] = {"ms_per_step_median": statistics.median(v), "ms_per_step_min": min(v), "ms_per_step_max": max(v),
                   "pileup_kernel_ms_mean": statistics.mean(res[k]["kernel_ms"]), "ms_per_step_rounds": v}
        print(f"k={k:>3s}  ms/step median {rows[k]['ms_per_step_median']:.4f} [{min(v):.4f}, {max(v):.4f}]  "
              f"pileup kernel {rows[k]['pileup_kernel_ms_mean']:.4f} ms", flush=True)
    doc = {"card": info, "workload": w.name, "reads": int(batch.n_reads), "ref_len": L, "steps": args.steps, "rounds": args.rounds,
           "sm_count": torch.cuda.get_device_properties(0).multi_processor_count, "settings": rows}
    os.environ.pop("TC_OVERLAP_SMS", None)
    if args.trace_dir:
        doc["trace"] = trace(chained, args.trace_dir, torch)
        print(json.dumps(doc["trace"]))
    print(json.dumps(info))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)


def trace(chained, directory, torch):
    """A few chained steps under torch.profiler: for every pileup kernel but the first, whether the tail kernels of the
    step before it ran inside its time span."""
    from torch.profiler import ProfilerActivity, profile

    chained(10)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        chained(8)
        torch.cuda.synchronize()
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, "overlap_trace.json")
    prof.export_chrome_trace(path)
    with open(path) as fh:
        ev = json.load(fh)
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    pile = [e for e in kern if "warp_pileup_kernel" in e["name"]]
    inside = total = 0
    for prev, cur in zip(pile, pile[1:]):
        # step i's tail: its kernels between the end of its pileup and the end of the next pileup
        tail = [e for e in kern if any(t in e["name"] for t in TAIL) and prev["ts"] + prev["dur"] <= e["ts"] < cur["ts"] + cur["dur"]]
        total += len(tail)
        inside += sum(1 for e in tail if cur["ts"] <= e["ts"] and e["ts"] + e["dur"] <= cur["ts"] + cur["dur"])
    return {"file": os.path.basename(path), "pileup_kernels": len(pile), "tail_kernels": total, "tail_kernels_inside_next_pileup": inside,
            "pileup_us": [round(e["dur"], 1) for e in pile]}


if __name__ == "__main__":
    main()
