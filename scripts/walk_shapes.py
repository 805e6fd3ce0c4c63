"""What stands in front of each match op of the pileup kernel's walk (no GPU): the run of ops that are not M / = / X
between a match op and the match op before it in the same read, counted by shape: what a short path for common op groups
in the walk of pileup_warp.cu could cover (DESIGN.md §3.1, profiles/walk_steps_experiment.md).

    python scripts/walk_shapes.py [--out profiles/walk_shapes.json]

Samples: bench.py's (configs[1], seed as in bench.py's make_sample, all 2 M reads), configs[0] (all 50 k reads), one
sample of configs[2]'s plate (all 1 M reads) and 1 M reads of configs[3].  Shapes:
  none        the match op follows a match op directly
  D1, I1      one 1-base deletion / insertion between two match ops (the insertion's anchor is the match op before it)
  D1I1, I1D1  the two in a row
  S_start     a soft clip in front of the read's first match op
  first       the read's first match op with nothing in front of it
  other       anything else (longer indels, three or more ops, N, H, P, a run at the read's start that is not one S)"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from trueconsense_b200 import synth  # noqa: E402

OP_M, OP_I, OP_D, OP_S, OP_EQ, OP_X = 0, 1, 2, 4, 7, 8
SHAPES = ("none", "D1", "I1", "D1I1", "I1D1", "S_start", "first", "other")


def shapes(batch) -> dict:
    c = batch.cigar.astype(np.int64)
    op, ln = c & 15, c >> 4
    off = batch.cigar_off.astype(np.int64)
    read = np.repeat(np.arange(batch.n_reads), np.diff(off))
    idx = np.arange(c.size)
    match = (op == OP_M) | (op == OP_EQ) | (op == OP_X)
    # index of the last match op at or before each op, then the one strictly before each match op
    last = np.maximum.accumulate(np.where(match, idx, -1))
    m = idx[match]
    pm = np.concatenate(([-1], last[:-1]))[m]
    start = off[read[m]]
    inside = pm >= start                   # a match op before it in the same read
    run = np.where(inside, m - pm - 1, m - start)
    one = (op == OP_D) * 1 + (op == OP_I) * 2       # per op: 1 = D1 candidate, 2 = I1 candidate (when ln == 1)
    one = np.where(ln == 1, one, 0)
    a = np.where(run >= 1, one[np.minimum(m - run, c.size - 1)], 0)      # first op of the run
    b = np.where(run >= 2, one[np.minimum(m - run + 1, c.size - 1)], 0)  # second op of the run
    out = {
        "none": int(np.sum(inside & (run == 0))),
        "D1": int(np.sum(inside & (run == 1) & (a == 1))),
        "I1": int(np.sum(inside & (run == 1) & (a == 2))),
        "D1I1": int(np.sum(inside & (run == 2) & (a == 1) & (b == 2))),
        "I1D1": int(np.sum(inside & (run == 2) & (a == 2) & (b == 1))),
        "S_start": int(np.sum(~inside & (run == 1) & (op[np.maximum(m - 1, 0)] == OP_S))),
        "first": int(np.sum(~inside & (run == 0))),
    }
    out["other"] = int(m.size) - sum(out.values())
    total = int(m.size)
    return {"reads": int(batch.n_reads), "ops": int(c.size), "match_ops": total,
            "ops_per_read": c.size / max(batch.n_reads, 1),
            "counts": out, "fraction": {k: v / max(total, 1) for k, v in out.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "walk_shapes.json"))
    args = ap.parse_args()
    res = {}
    for idx, scale in ((1, 1.0), (0, 1.0), (2, 1.0), (3, 0.02)):
        w = synth.config(idx, scale=scale)
        if idx == 1:                        # bench.py's sample 0 (make_sample)
            w.params.seed = w.params.seed * 1000
        b = synth.generate_reads(w.params, w.ref)
        r = shapes(b)
        r["scale"] = scale
        res[w.name] = r
        f = r["fraction"]
        print(f"{w.name:34s} {r['reads']:>8d} reads {r['ops_per_read']:5.1f} ops/read  " +
              "  ".join(f"{k} {100 * f[k]:.2f}%" for k in SHAPES))
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main()
