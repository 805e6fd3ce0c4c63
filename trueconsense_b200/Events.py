"""Insertion calling and the minority-deletion test with the reference's API
(TrueConsense/Events.py), computed by the GPU kernels behind ``tc_call`` and
``tc_extract_inserts``.
"""
from __future__ import annotations

import re

import numpy as np

from . import gpu

_ROWS = ("coverage", "A", "T", "C", "G", "X", "I")
_INSERT_RE = re.compile(r"(\d)([a-zA-Z]+)")      # Events.py:75


def _counts_from_index(iDict) -> np.ndarray:
    """{pos: {"coverage","A","T","C","G","X","I"}} (the reference's ``IndexDF.to_dict("index")``,
    TrueConsense.py:237) -> int32[8][L].  Positions must be 1..L, the shape BuildIndex produces."""
    L = len(iDict)
    counts = np.zeros((gpu.TC_NROWS, L), dtype=np.int32)
    try:
        for p in range(1, L + 1):
            row = iDict[p]
            c = counts[:, p - 1]
            c[0] = row["coverage"]; c[1] = row["A"]; c[2] = row["T"]; c[3] = row["C"]; c[4] = row["G"]
            c[5] = row["X"]; c[6] = row["I"]
    except KeyError as e:
        raise ValueError(f"the index must hold positions 1..{L} with the seven count columns (missing {e})") from None
    return counts


def _bam_handle(bam):
    from .indexing import BamHandle, Readbam

    if isinstance(bam, BamHandle):
        return bam
    name = getattr(bam, "filename", None)
    if name is not None:
        return Readbam(name.decode() if isinstance(name, bytes) else name)
    raise TypeError("bam must come from trueconsense_b200.indexing.Readbam (or expose .filename)")


def _parse_modal(string):
    """Events.py:75-81 on the modal string: (letters, last digit before them) or (None, None)."""
    if string is None:
        return None, None
    m = _INSERT_RE.search(string)
    if m:
        return m.group(2), m.group(1)
    return None, None


def ExtractInserts(bam, position):
    """Most common upper-cased pileup string at ``position`` (1-based) under pysam's default
    pileup filters, reduced to (inserted letters, size digit) — Events.py:47-82."""
    h = _bam_handle(bam)
    if not 1 <= position <= h.ref_len:
        return None, None
    res = gpu.default_context().extract_inserts(h.device_reads(with_host_qual=True), h.ref_len, [position])
    return _parse_modal(res[0]["string"])


def ListInserts(iDict, mincov, bam):
    """(True, {pos: {size: bases}}) or (False, None) — Events.py:5-44.  The candidate test
    ``(I / cov) * 100 > 55`` runs in the call kernel (IEEE double, like the reference); the
    candidate columns are piled up, keyed, radix-sorted and run-length encoded on the GPU."""
    counts = _counts_from_index(iDict)
    L = counts.shape[1]
    if L == 0:
        return False, None
    ctx = gpu.default_context()
    h = None
    key = None
    if bam is not None:
        try:
            h = _bam_handle(bam)
            key = (int(mincov), counts[0].tobytes(), counts[6].tobytes())
            if key in h._insert_cache:
                has, pos = h._insert_cache[key]
                return has, (None if pos is None else {k: dict(v) for k, v in pos.items()})
        except TypeError:
            h = None
    table = ctx.call(counts, L, mincov, False)
    cands = ctx.list_insert_candidates(table.flags, L)
    positions = {}
    if len(cands):
        if h is None:
            raise TypeError("bam must come from trueconsense_b200.indexing.Readbam (or expose .filename)")
        cols = [int(c) for c in cands if c <= h.ref_len]
        res = ctx.extract_inserts(h.device_reads(with_host_qual=True), h.ref_len, cols) if cols else []
        for r in res:
            bases, size = _parse_modal(r["string"])
            if bases is None or size is None:
                continue
            positions[int(r["pos"])] = {size: bases}
    out = (True, positions) if positions else (False, None)
    if h is not None and key is not None:
        h._insert_cache[key] = (out[0], None if out[1] is None else {k: dict(v) for k, v in out[1].items()})
    return out


def ListInsertsContigs(indexes, mincov, bam):
    """``ListInserts`` for every reference of the BAM in one pass: ``{reference: (True, {pos: {size: bases}}) | (False, None)}``
    in header order, each equal to ``ListInserts`` over that reference alone.  ``indexes``: ``{reference: index dict}``
    (``BuildIndexContigs``' frames as dicts).  One segmented call (``tc_call_contigs``), one candidate list and one
    ExtractInserts call cover all references; positions come back per reference, 1-based."""
    h = _bam_handle(bam)
    names = list(h.references)
    missing = [n for n in names if n not in indexes]
    if missing:
        raise ValueError(f"no index for reference {missing[0]!r}")
    parts = [_counts_from_index(indexes[n]) for n in names]
    out = {n: (False, None) for n in names}
    lens = [c.shape[1] for c in parts]
    if sum(lens) == 0:
        return out
    d, lay = h.device_reads_contigs(names, lens)
    ctx = gpu.default_context()
    table = ctx.call_contigs(np.concatenate(parts, axis=1), lay.start, mincov, False)
    cands = ctx.list_insert_candidates(table.flags, lay.total)
    if not len(cands):
        return out
    k, local = lay.locate(cands)
    bam_lens = np.asarray(h.lengths, dtype=np.int64)
    keep = local <= bam_lens[k]                 # as ListInserts keeps the columns inside the BAM's reference
    res = ctx.extract_inserts(d, lay.total, cands[keep]) if keep.any() else []
    found: dict[str, dict] = {}
    for r, kk, pos in zip(res, k[keep].tolist(), local[keep].tolist()):
        bases, size = _parse_modal(r["string"])
        if bases is None or size is None:
            continue
        found.setdefault(names[kk], {})[int(pos)] = {size: bases}
    for n, positions in found.items():
        out[n] = (True, positions)
    return out


def MinorityDel(index, p):
    """``(X / cov) * 100 >= 15`` — Events.py:85-106 (ZeroDivisionError when cov == 0)."""
    row = index[p]
    cov = row.get("coverage")
    if cov == 0:
        raise ZeroDivisionError("division by zero")
    counts = np.zeros((gpu.TC_NROWS, 1), dtype=np.int32)
    counts[0, 0] = cov
    counts[5, 0] = row.get("X")
    res = gpu.default_context().call(counts, 1, 0, False)
    return bool(res.flags[0] & gpu.CF_MINORITY_DEL)
