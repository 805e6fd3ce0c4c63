"""Consensus building with the reference's API (TrueConsense/Sequences.py).

``BuildConsensus(mincov, iDict, GFFdict, IncludeAmbig, bam, includeINS) -> (consensus, gffdict)``
has the reference's signature, return value, exceptions and side effects.  Everything that is
independent per position (ranking, IUPAC ambiguity, minority-deletion flag, X-run lengths,
insertion candidates) is computed for all positions at once by the GPU call kernel
(csrc/cuda/call.cu, ``tc_call``); the walk below only consumes that candidate table and carries
the sequential state (deletion skips, ORF bookkeeping) on the host — SURVEY.md Appendix B.
"""
from __future__ import annotations

import copy

import numpy as np

from . import gpu
from .Events import ListInserts, _counts_from_index
from .ORFs import GffTracker

_ROWS = ("coverage", "A", "T", "C", "G", "X", "I")


def GetDistribution(iDict, position):
    """Sequences.py:143-165."""
    row = iDict[position]
    return {k: row.get(k) for k in ("A", "T", "C", "G", "X")}


def _ranked_column(iDict, position):
    row = iDict[position]                     # KeyError for a missing position, like the reference
    counts = np.zeros((gpu.TC_NROWS, 1), dtype=np.int32)
    for r, k in enumerate(_ROWS):
        counts[r, 0] = row.get(k)
    return gpu.default_context().call(counts, 1, 0, False)


def GetNucleotide(iDict, position, count):
    """(letter, count) of rank ``count`` (1 = most frequent) at ``position`` — Sequences.py:119-140.
    Ties go to the larger letter (X > T > G > C > A).  Ranked on the GPU (call kernel) so it cannot
    drift from what BuildConsensus uses."""
    res = _ranked_column(iDict, position)
    if count == 5:
        dist = GetDistribution(iDict, position)
        top4 = {chr(res.rank_letter[k, 0]) for k in range(4)}
        (last,) = [l for l in dist if l not in top4]
        return last, dist[last]
    if not 1 <= count <= 4:
        raise IndexError("list index out of range")
    return chr(res.rank_letter[count - 1, 0]), int(res.rank_count[count - 1, 0])


def WalkForward(index, p, fixedpositions="expand"):
    """Positions after ``p`` whose most frequent letter is X (Sequences.py:9-53, "expand" mode)."""
    if fixedpositions != "expand":
        lastposition = list(index)[-1]
        p = p + 1
        target = p + fixedpositions
        if target >= lastposition:
            target = lastposition
        track = {}
        while p != target:
            track[p] = GetNucleotide(index, p, 1)[0]
            p += 1
        return track
    counts = _counts_from_index(index)
    L = counts.shape[1]
    res = gpu.default_context().call(counts, L, 0, False)
    if p + 1 > L or p < 0:
        raise KeyError(p + 1)
    if p >= 1:
        if res.flags[p - 1] & gpu.CF_XRUN_OFF_END:
            raise KeyError(L + 1)
        n = int(res.xrun[p - 1])
    else:
        n = 0
        while p + 1 + n <= L and res.flags[p + n] & gpu.CF_PRIMARY_X:
            n += 1
        if p + 1 + n > L:
            raise KeyError(L + 1)
    return list(range(p + 1, p + 1 + n))


def _orf_codonposition(gffdict, p):
    """Sequences.py:85-116."""
    a = []
    for g in gffdict.values():
        start = g.get("start")
        end = g.get("end") + 1
        if start <= p < end:
            attr = g.get("attributes", "")
            if not attr:
                continue
            split_attr = attr.split(";")
            if len(split_attr) < 2:
                a.extend((str(split_attr[0].split("=")[-1]), (p - start) % 3))
                continue
            a.extend((str(split_attr[1].split("=")[-1]), (p - start) % 3))
    if a:
        return tuple(a)
    return None, None


def complement_index(index, gffdict, skips):
    """Adds the (unused downstream) "ORF" annotation to every position — Sequences.py:56-82.
    Same values as the reference; built feature by feature instead of position by position."""
    per_pos: dict[int, list] = {}
    for g in gffdict.values():
        start = g.get("start")
        end = g.get("end") + 1
        attr = g.get("attributes", "")
        if not attr:
            continue
        split_attr = attr.split(";")
        name = str(split_attr[0].split("=")[-1]) if len(split_attr) < 2 else str(split_attr[1].split("=")[-1])
        for p in range(max(start, 1), end):
            if p in index:
                per_pos.setdefault(p, []).extend((name, (p - start) % 3))
    for p in index:
        if p in skips:
            continue
        a = per_pos.get(p)
        index[p]["ORF"] = tuple(a) if a else (None, None)
    return index


def BuildConsensus(mincov, iDict, GFFdict, IncludeAmbig, bam, includeINS):
    """Sequences.py:168-322: the consensus string and the corrected GFF dict."""
    p_index = complement_index(iDict, GFFdict, [])
    inserts = ListInserts(p_index, mincov, bam)
    return consensus_from_inserts(mincov, _counts_from_index(p_index), GFFdict, IncludeAmbig, inserts, includeINS)


_last_call: tuple | None = None      # (key, columns): WriteOutputs walks the same table twice (Outputs.py:95-98), with and without insertions


def _call_table(counts: np.ndarray, L: int, mincov: int, include_ambig: bool):
    """The call kernel's columns for this count table as Python lists; the table of the previous call is kept, so the second
    BuildConsensus of a run (same index, same thresholds) costs no second tc_call and no second conversion."""
    global _last_call
    import hashlib

    key = (L, int(mincov), include_ambig, hashlib.blake2b(counts.tobytes(), digest_size=16).digest())
    if _last_call is not None and _last_call[0] == key:
        return _last_call[1]
    table = gpu.default_context().call(counts, L, mincov, include_ambig)
    cols = (counts[0].tolist(), table.flags.tolist(), table.xrun.tolist(), table.call_char.tobytes().decode("ascii"))
    _last_call = (key, cols)
    return cols


def consensus_from_inserts(mincov, counts, GFFdict, IncludeAmbig, inserts, includeINS, table=None):
    """The walk of Sequences.py:175-322 over a count table [8][L] given ListInserts' result.  ``table``: the call table of
    exactly these columns computed with the same mincov and IncludeAmbig (a ``gpu.CallResult``, e.g. one reference's
    slice of a ``tc_call_contigs`` table); None: ``tc_call`` here."""
    hasinserts, insertpositions = inserts
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    L = counts.shape[1]
    if table is None:
        cov_l, flags, xrun, chars = _call_table(counts, L, mincov, bool(IncludeAmbig is True))
    else:
        if table.flags.shape[0] != L:
            raise ValueError(f"the call table holds {table.flags.shape[0]} columns, the count table {L}")
        cov_l, flags, xrun, chars = (counts[0].tolist(), table.flags.tolist(), table.xrun.tolist(),
                                     table.call_char.tobytes().decode("ascii"))

    LOWCOV, PRIMX, MDEL, OFFEND, ZEROCOV = gpu.CF_LOWCOV, gpu.CF_PRIMARY_X, gpu.CF_MINORITY_DEL, gpu.CF_XRUN_OFF_END, gpu.CF_ZERO_COV

    def walk(b):                    # len(WalkForward(b)); raises what the reference raises
        if b > L:
            raise KeyError(b + 1)
        if flags[b - 1] & OFFEND:
            raise KeyError(L + 1)
        return xrun[b - 1]

    def minority_del(b):
        if b > L:
            raise KeyError(b)
        f = flags[b - 1]
        if f & ZEROCOV:
            raise ZeroDivisionError("division by zero")
        return bool(f & MDEL)

    newGffdict = copy.deepcopy(GFFdict)
    tracker = GffTracker(GFFdict, newGffdict)
    cons: list[str] = []
    skip_until = 0          # positions <= skip_until already belong to a deletion (the reference's dskips)
    ins = insertpositions if hasinserts is True else None

    for b in range(1, L + 1):
        cov = cov_l[b - 1]
        within_orf = tracker.in_orf(b)
        f = flags[b - 1]
        if b <= skip_until:
            out = "-"
            cons.append(out); tracker.append(out)
            tracker.correct(b, out, insertpositions, mincov, cov)
            continue
        if f & LOWCOV:
            out = "N"
            cons.append(out); tracker.append(out)
            tracker.correct(b, out, insertpositions, mincov, cov)
            continue
        if not f & PRIMX:
            out = chars[b - 1]
            if minority_del(b):
                run = walk(b)
                if run:
                    # SolveTripletLength(run, [b]): (1 + run) % 3 == 0 unless run % 3 == 0 (then never)
                    if run % 3 != 0 and (1 + run) % 3 == 0:
                        out = "-"
                        skip_until = b + run
                elif minority_del(b + 1):
                    run2 = walk(b + 1)
                    if run2 and run2 % 3 != 0 and (2 + run2) % 3 == 0:
                        out = "-"
                        skip_until = b + 1 + run2
        else:
            if within_orf:
                run = walk(b)
                if run >= 2:
                    out = "-"
                    skip_until = b + run
                else:
                    out = chars[b - 1]
            else:
                out = "-"
        cons.append(out); tracker.append(out)
        last = out
        if includeINS is True and cov > mincov and ins is not None and b in ins:
            for size in ins[b]:
                s = str(ins[b][size])
                cons.append(s); tracker.append(s)
                last = s
        tracker.correct(b, last, insertpositions, mincov, cov)

    return "".join(cons), newGffdict
