"""The rule variant 4 of the pileup cuts long reads by (pileup_long.cu, header comment), restated in Python and checked on
the oracle alone: the reference is divided into cells of PIECE_COLS columns, the part of an alignment inside one cell
becomes a piece that looks like a short read, an op crossing a border is split in two, I / S / H ops stay with the piece
of the reference-consuming op in front of them, and the clips in front of the first aligned base are dropped.  Piled up
by the oracle, the pieces of a batch must give the same rows (coverage, A, T, C, G, X, I) as the reads themselves.

When a variant-4 case of test_pileup_edges.py fails, this test tells whether the rule is wrong (it fails too) or the
kernels apply it wrongly (it passes).  The generator of long reads below is shared with that file."""
import re

import numpy as np
import pytest

PIECE_COLS = 400            # TC_PIECE_COLS (pileup.cuh)
REF_OPS = set("MDN=X")
_BASES = np.frombuffer(b"ACGTNRYKM", np.uint8)
_BASE_P = [0.245] * 4 + [0.012] + [0.002] * 4


def rand_seq(rng, n: int) -> str:
    """n bases, mostly A/C/G/T, with N and IUPAC codes (they count towards coverage only)."""
    return _BASES[rng.choice(len(_BASES), n, p=_BASE_P)].tobytes().decode() if n else ""


def ops_str(ops) -> str:
    return "".join(f"{int(l)}{o}" for o, l in ops)


def record(rng, pos: int, ops, **kw) -> dict:
    """A read of `ops` at `pos` with random bases, on either strand."""
    q = sum(int(l) for o, l in ops if o in "MIS=X")
    return dict(pos=int(pos), cigar=ops_str(ops), seq=rand_seq(rng, q), flag=16 if rng.random() < 0.5 else 0, **kw)


def ref_span(rec) -> int:
    return sum(int(l) for l, o in re.findall(r"(\d+)([MIDNSHP=X])", rec["cigar"]) if o in REF_OPS)


def long_read_ops(rng, pos: int, span: int, dense_ops: int = 0):
    """The ops of a long read at `pos` covering about `span` columns, steered onto the cell borders (absolute multiples
    of PIECE_COLS) and one column off them: match ops ending on a border followed by I, D, N, "I D" or "D I"; D / N of
    400-5000 columns covering whole cells; D->I, I->D and N->I pairs; a first op after the clips that is an I; leading
    and trailing soft clips of 4096+ bases.  dense_ops: a stretch of that many ops of "1I1M1D1M" in the middle."""
    ops, x = [], pos
    u = rng.random()
    if u < 0.1:
        ops.append(("H", int(rng.integers(1, 60))))
    if u < 0.25:
        ops.append(("S", int(rng.integers(1, 40))))
    elif u < 0.3:
        ops.append(("S", int(rng.integers(4096, 6000))))
    if rng.random() < 0.08:
        ops.append(("I", int(rng.integers(1, 4))))
    end = pos + span
    dense_at = pos + span // 3 if dense_ops else None
    while x < end:
        border = PIECE_COLS * (x // PIECE_COLS + 1)
        l = int(rng.integers(1, 120))
        if rng.random() < 0.5 and border - x < 150:
            l = border - x + int(rng.integers(-1, 2))
        l = max(1, l)
        ops.append(("M" if rng.random() < 0.9 else "=X"[int(rng.integers(0, 2))], l))
        x += l
        if x >= end:
            break
        if dense_at is not None and x >= dense_at:
            ops += ([("I", 1), ("M", 1), ("D", 1), ("M", 1)] * (dense_ops // 4))[:-1]       # ends on a D: an M follows
            x += 3 * (dense_ops // 4) - 1
            dense_at = None
            continue
        u = rng.random()
        if u < 0.15:
            ops.append(("I", int(rng.integers(1, 4))))
        elif u < 0.3:
            l = int(rng.integers(1, 5)); ops.append(("D", l)); x += l
        elif u < 0.36:
            l = int(rng.integers(400, 5001)); ops.append(("DN"[int(rng.integers(0, 2))], l)); x += l
        elif u < 0.46:
            a, c = int(rng.integers(1, 4)), int(rng.integers(1, 3))
            d = "D" if rng.random() < 0.7 else "N"
            ops += [(d, a), ("I", c)] if rng.random() < 0.6 else [("I", c), (d, a)]
            x += a
    if ops[-1][0] not in "M=X":
        ops.append(("M", 5))
    u = rng.random()
    if u < 0.2:
        ops.append(("S", int(rng.integers(1, 40))))
    elif u < 0.24:
        ops.append(("S", int(rng.integers(4096, 8000))))
    if rng.random() < 0.05:
        ops.append(("H", int(rng.integers(1, 5000))))
    return ops


def long_read_records(rng, n: int, lo: int = 1000, hi: int = 12000, first: int = 0, dense: int = 0) -> list[dict]:
    """n long reads of lo..hi columns starting from column `first`, sorted by position.  A quarter start on a cell
    border or one off it, a fifth end on one; `dense` reads carry 2049-6000 ops (the split works in rounds of 2048)."""
    recs = []
    for i in range(n):
        cell = int(rng.integers(0, 8))
        u = rng.random()
        pos = first + PIECE_COLS * cell + (int(rng.integers(-1, 2)) if u < 0.25 else int(rng.integers(0, PIECE_COLS)))
        pos = max(pos, first)
        span = int(rng.integers(lo, hi))
        if rng.random() < 0.2:
            span = PIECE_COLS * ((pos + span) // PIECE_COLS) - pos       # ends on a border (unless an op overshoots)
        dense_ops = int(rng.integers(2049, 6001)) // 4 * 4 + 4 if i < dense else 0
        recs.append(record(rng, pos, long_read_ops(rng, pos, span, dense_ops)))
    recs.sort(key=lambda r: r["pos"])
    return recs


def cut_into_pieces(rec) -> list[dict]:
    """The pieces of one read, as reads of their own: each piece's SEQ runs from its first query base to the end of
    the read, the bases behind the piece become a soft clip."""
    ops = [(o, int(l)) for l, o in re.findall(r"(\d+)([MIDNSHP=X])", rec["cigar"])]
    k = y = 0
    while k < len(ops) and ops[k][0] in "HS":               # leading clips: dropped (a soft clip moves the query index)
        y += ops[k][1] if ops[k][0] == "S" else 0
        k += 1
    x = rec["pos"]
    cell_end = (x // PIECE_COLS + 1) * PIECE_COLS
    pieces, cur, has_ref = [], None, False
    for o, l in ops[k:]:
        if o not in REF_OPS:                                # I / S / H: with the piece in front (a leading I opens one)
            if cur is None:
                cur = dict(pos=x, y=y, ops=[])
            cur["ops"].append((o, l))
            y += l if o in "IS" else 0
            continue
        while l > 0:
            if x == cell_end:
                if cur is not None and has_ref:
                    pieces.append(cur)
                    cur, has_ref = None, False
                cell_end += PIECE_COLS
            if cur is None:
                cur = dict(pos=x, y=y, ops=[])
            t = min(l, cell_end - x)
            cur["ops"].append((o, t))
            has_ref = True
            x += t; l -= t
            y += t if o in "M=X" else 0
    if cur is not None:
        pieces.append(cur)
    out = []
    for p in pieces:
        q = sum(l for o, l in p["ops"] if o in "MIS=X")
        rest = len(rec["seq"]) - p["y"] - q
        out.append(dict(pos=p["pos"], cigar=ops_str(p["ops"] + ([("S", rest)] if rest > 0 else [])), seq=rec["seq"][p["y"]:],
                        flag=rec["flag"]))
    return out


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_pieces_pile_up_like_their_reads(seed):
    from oracle import pileup
    from trueconsense_b200.reads import ReadBatch

    rng = np.random.default_rng(seed)
    recs = long_read_records(rng, 300, lo=500, hi=4000, dense=4)
    pieces = sorted((p for r in recs for p in cut_into_pieces(r)), key=lambda p: p["pos"])
    for r in recs:                                          # every cell a read touches holds exactly one of its pieces
        ps = cut_into_pieces(r)
        assert [p["pos"] // PIECE_COLS for p in ps] == list(range(r["pos"] // PIECE_COLS, (r["pos"] + ref_span(r) - 1) // PIECE_COLS + 1))
        assert all(ref_span(p) <= PIECE_COLS for p in ps)
    assert max(len(re.findall(r"\d+[A-Z=]", r["cigar"])) for r in recs) > 2048
    assert any(re.fullmatch(rf"{PIECE_COLS}[DN](\d+S)?", p["cigar"]) for p in pieces)         # pieces of one D / N op
    L = max(r["pos"] + ref_span(r) for r in recs) + 7
    a = pileup.pileup_counts(ReadBatch.from_records(recs), L, threads=8)
    b = pileup.pileup_counts(ReadBatch.from_records(pieces), L, threads=8)
    assert a[:7].any(axis=1).all()
    assert np.array_equal(a, b)
