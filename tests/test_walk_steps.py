"""The short path of the pileup kernel's walk (pileup_warp.cu), against the oracle (bit for bit, all 8 rows).

A 1-base D or I right behind a match op of the same read skips the walk's generic op branch.  The reads below are dense
with such ops (one every few columns, so that every window has some on its phase borders, the 256-column multiples, and
one column before them), start on the slack's last column and run to the reference's last column, and mix them with
everything that must stay on the generic path: an op at a read's start, an I as a read's first op (no anchor), D1 I1 and
I1 D1 (also next to a clip), 2-base deletions and insertions, reference skips, a read ending in D in front of a read
starting with M.  Then sub-tiles that hold a read without SEQ (its match ops become reference skips, so nothing behind
them is a match op) or a soft clip of 4096+ bases.  Every batch runs through variant 3 explicitly and through the
library's choice, in the 256-, 512- and 1024-column geometries."""
import numpy as np
import pytest

from test_pileup_edges import _batch, _check, geometry
from test_piece_rule_cpu import record

pytestmark = pytest.mark.gpu

SPANS = (150, 400, 900)         # the 256-, 512- and 1024-column windows


@pytest.fixture(scope="module")
def orc():
    from oracle import pileup

    pileup.build()
    return pileup


@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import gpu

    return gpu.Context(0)


def _step_ops(rng, span: int):
    """Ops covering `span` columns (give or take the tail): match ops of 1-6 columns, mostly separated by D1 or I1, now
    and then by D1 I1, I1 D1, D2, I2 or N; a leading clip, I1 or nothing, and a tail of a clip, D1, I1 or nothing."""
    ops, x = [], 0
    u = rng.random()
    if u < 0.15:
        ops.append(("S", int(rng.integers(1, 9))))
        if rng.random() < 0.3:
            ops += [("I", 1), ("D", 1)] if rng.random() < 0.5 else [("D", 1), ("I", 1)]     # next to a clip
            x += 1
    elif u < 0.2:
        ops.append(("H", 3))
    elif u < 0.3:
        ops.append(("I", 1))                    # a read's first op: no anchor
    while True:
        l = max(1, min(int(rng.integers(1, 7)), span - x))
        ops.append(("M" if rng.random() < 0.9 else "=", l))
        x += l
        if x >= span - 1:
            break
        u = rng.random()
        if u < 0.42:
            ops.append(("D", 1)); x += 1
        elif u < 0.84:
            ops.append(("I", 1))
        elif u < 0.88:
            ops += [("D", 1), ("I", 1)]; x += 1
        elif u < 0.92:
            ops += [("I", 1), ("D", 1)]; x += 1
        elif u < 0.95:
            ops.append(("D", 2)); x += 2
        elif u < 0.98:
            ops.append(("I", 2))
        else:
            ops.append(("N", 3)); x += 3
    u = rng.random()
    if u < 0.1:
        ops.append(("D", 1))                    # a read ending in D (the next read may start with M)
    elif u < 0.2:
        ops.append(("I", 1))
    elif u < 0.3:
        ops += [("I", 1), ("S", 4)] if rng.random() < 0.5 else [("D", 1), ("I", 1), ("S", 4)]
    elif u < 0.4:
        ops.append(("S", int(rng.integers(1, 9))))
    return ops


def _reads(rng, span: int, n: int, special=None):
    """n reads of at most `span` columns, their starts steered like test_pileup_edges.test_geometry_edge's (the same
    start, a few columns on, a multiple of 8, the slack's last start column or one or two past it).  special(rng, pos):
    every eighth read, or None.  Returns the records and the reference length: the last column is some read's last."""
    ops = [_step_ops(rng, span - 2) for _ in range(n)]
    slack = geometry(max(_span({"cigar": o}) for o in ops))[1]
    recs, p = [], 40
    for i in range(n):
        u = rng.random()
        if u < 0.3:
            pass
        elif u < 0.55:
            p += int(rng.integers(1, 9))
        elif u < 0.65:
            p = (p | 7) + 1
        else:
            p = (p & ~7) + slack + int(rng.integers(-1, 2))
        recs.append(special(rng, p) if special is not None and i % 8 == 7 else record(rng, p, ops[i]))
    # the reference's last columns: a step group right in front of the last column, and an insertion anchored on it
    end = max(r["pos"] + _span(r) for r in recs)
    recs.append(record(rng, end - 8, [("M", 5), ("D", 1), ("M", 2)]))
    recs.append(record(rng, end - 8, [("M", 6), ("I", 1), ("M", 1), ("D", 1)]))
    recs.append(record(rng, end - 6, [("M", 4), ("I", 1), ("M", 2), ("I", 1)]))
    return recs, end


def _span(rec) -> int:
    import re

    c = rec["cigar"]
    if not isinstance(c, str):
        return sum(int(l) for o, l in c if o in ("M", "D", "N", "=", "X"))
    return sum(int(l) for l, o in re.findall(r"(\d+)([MIDNSHP=X])", c) if o in "MDN=X")


@pytest.mark.parametrize("span", SPANS)
def test_step_groups(ctx, orc, span):
    """Reads full of short-path ops, and every generic neighbour of one, in each window geometry."""
    rng = np.random.default_rng(span)
    recs, L = _reads(rng, span, 30000)
    b = _batch(recs)
    assert geometry(int(b.ref_spans().max()))[0] == geometry(span + 8)[0]
    _check(ctx, orc, b, L, 3)


def _no_seq(rng, pos):
    r = record(rng, pos, [("M", 12), ("D", 1), ("M", 9), ("I", 1), ("M", 14)])
    r["seq"] = "*"
    return r


def _long_clip(rng, pos):
    """A soft clip of 4096+ bases behind the read's last match op (it saturates: nothing follows it)."""
    return record(rng, pos, [("M", 10), ("I", 1), ("M", 7), ("D", 1), ("M", 12), ("S", 4100)])


@pytest.mark.parametrize("what", ["no_seq", "long_clip"])
@pytest.mark.parametrize("span", (150, 400))
def test_generic_subtiles(ctx, orc, span, what):
    """Every eighth read is one without SEQ or with a long clip, among reads dense with short-path ops."""
    rng = np.random.default_rng(1000 * span + len(what))
    special = {"no_seq": _no_seq, "long_clip": _long_clip}[what]
    recs, L = _reads(rng, span, 20000, special)
    _check(ctx, orc, _batch(recs), L, 3)
