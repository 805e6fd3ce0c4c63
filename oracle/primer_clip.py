"""Primer clipping restated in plain Python over raw BAM record bytes (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

The rule is DESIGN §4's, written out op by op as it reads there (no search tables, no warp scans), so that
``tc_bam_clip_primers`` (csrc/cuda/primerclip.cu) can be checked against it byte for byte:

* A record is eligible if refID >= 0, FLAG & 0x4 == 0 and its CIGAR has an M, = or X op.  Its aligned span is [p, q],
  p = pos, q = pos + refspan - 1 (refspan: the M, D, N, =, X lengths).  Only primers of its own reference count.
* Checked ends: the 5' end (left for forward reads, right for FLAG & 0x10), or both with ``both_ends``.
* Left: primers with s - t <= p < e match; E = max e; the columns [p, E) go.  Right: primers with s <= q < e + t match;
  S = min s; the columns [S, q] go.
* The walk (left; the right one is its mirror image): leading H / S ops are skipped; with r = p, c = 0 an M / = / X op of
  length L goes whole when r + L <= E (c += L, r += L), else it is split (c += E - r, its length L - (E - r), r = E) and the
  walk stops; I goes (c += L); D / N go (r += L), whole even when they cross E; P goes.  Once r >= E the I / D / N / P ops up
  to the next M / = / X op go too.  pos = r; the CIGAR: the leading H ops, one S op of old S + c when > 0, the rest.
* An eligible record whose CIGAR has an op of length 0 or an H / S op between other ops (the SAM spec allows neither) is
  refused: ValueError here, TC_ERR_ARG naming the record in tc_bam_clip_primers.
* No M / = / X op left: the record is fully clipped (FLAG |= 0x4, pos and CIGAR as they were).
* pos, CIGAR, n_cigar_op, block_size and FLAG change; bin is recomputed (reg2bin(pos, end, 14, 5)) when pos or the CIGAR
  changed; every other byte is copied.

``clip_records`` also returns the stats of ``tc_clip_stats_t``; ``sort_order`` is the order ``tc_bam_sort_records`` then gives
(samtools' coordinate order unless the records are sorted by (refID, pos) already), as tests/test_sort_input.py restates it.
"""
from __future__ import annotations

import struct

import numpy as np

M, I, D, N, S, H, P, EQ, X = range(9)
MATCH = (M, EQ, X)
REF = (M, D, N, EQ, X)
QUERY = (M, I, S, EQ, X)


def reg2bin(beg: int, end: int) -> int:
    """htslib's hts_reg2bin(beg, end, 14, 5)."""
    end -= 1
    for shift, t in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return t + (beg >> shift)
    return 0


def _walk_left(ops, p, E):
    """The left walk over [(op, len)]: (new ops, new pos), or None when no M / = / X op is left."""
    i = 0
    heads, old_s = [], 0
    while i < len(ops) and ops[i][0] in (H, S):
        if ops[i][0] == H:
            heads.append(ops[i])
        else:
            old_s += ops[i][1]
        i += 1
    r, c = p, 0
    rest = list(ops[i:])
    j = 0
    while j < len(rest) and r < E:
        op, L = rest[j]
        if op in MATCH:
            if r + L <= E:
                c += L
                r += L
                j += 1
            else:
                cut = E - r
                c += cut
                rest[j] = (op, L - cut)
                r = E
                break
        elif op == I:
            c += L
            j += 1
        elif op in (D, N):
            r += L
            j += 1
        elif op == P:
            j += 1
        else:                       # the trailing clips: nothing is left to keep
            return None
    while j < len(rest) and rest[j][0] in (I, D, N, P):
        op, L = rest[j]
        if op == I:
            c += L
        elif op != P:
            r += L
        j += 1
    rest = rest[j:]
    if not any(op in MATCH for op, _ in rest):
        return None
    new = heads + ([(S, old_s + c)] if old_s + c > 0 else []) + rest
    return new, r


def _walk_right(ops, q, S_):
    """The mirror image: the columns [S_, q] go.  (new ops) or None."""
    rev = list(reversed(ops))
    # walking the reversed CIGAR from the right end is the left walk over mirrored coordinates: column x -> -x
    res = _walk_left(rev, -q, -S_ + 1)
    if res is None:
        return None
    return list(reversed(res[0]))


def _span(ops) -> int:
    return sum(L for op, L in ops if op in REF)


def _qlen(ops) -> int:
    return sum(L for op, L in ops if op in QUERY)


def parse(rec: bytes) -> dict:
    """The fields of a record (block_size included) the clip reads."""
    tid, pos, l_name, mapq, bin_, n_cig, flag = struct.unpack_from("<iiBBHHH", rec, 4)
    c0 = 36 + l_name
    cig = struct.unpack_from(f"<{n_cig}I", rec, c0)
    return dict(tid=tid, pos=pos, l_name=l_name, bin=bin_, n_cig=n_cig, flag=flag, cigar=[(c & 15, c >> 4) for c in cig],
                tail=rec[c0 + 4 * n_cig:])


def _by_ref(primers):
    """{refID: (starts, ends)} as int64 arrays."""
    out = {}
    for r, s, e in primers:
        out.setdefault(int(r), ([], []))
        out[int(r)][0].append(int(s))
        out[int(r)][1].append(int(e))
    return {r: (np.array(s, np.int64), np.array(e, np.int64)) for r, (s, e) in out.items()}


def _matches(by_ref, tid, p, q, tol):
    """(E or None, S or None): the largest end of the primers matching the left end, the smallest start of those matching
    the right end."""
    if tid not in by_ref:
        return None, None
    s, e = by_ref[tid]
    left = e[(s - tol <= p) & (p < e)]
    right = s[(s <= q) & (q < e + tol)]
    return (int(left.max()) if left.size else None), (int(right.min()) if right.size else None)


def clip_record(rec: bytes, primers, tolerance: int = 5, both_ends: bool = False):
    """(the record after the clip, what happened: None / "clipped" / "unmapped", left clipped, right clipped, columns removed).
    ``primers``: (refID, start, end) rows, or what ``_by_ref`` makes of them."""
    if not isinstance(primers, dict):
        primers = _by_ref(primers)
    f = parse(rec)
    ops = f["cigar"]
    if f["tid"] < 0 or f["flag"] & 4 or not any(op in MATCH for op, _ in ops):
        return rec, None, False, False, 0
    body = [i for i, (op, _) in enumerate(ops) if op not in (H, S)]
    if any(L == 0 for _, L in ops) or any(ops[i][0] in (H, S) for i in range(body[0], body[-1] + 1)):
        raise ValueError("the CIGAR has an op of length 0, or an H / S op between other ops")
    p = f["pos"]
    q = p + _span(ops) - 1
    E, S_ = _matches(primers, f["tid"], p, q, tolerance)
    rev = bool(f["flag"] & 16)
    if not (both_ends or not rev):
        E = None
    if not (both_ends or rev):
        S_ = None
    if E is None and S_ is None:
        return rec, None, False, False, 0
    new, pos = ops, p
    full = False
    if E is not None:
        res = _walk_left(new, pos, E)
        if res is None:
            full = True
        else:
            new, pos = res
    if not full and S_ is not None:
        res = _walk_right(new, q, S_)
        if res is None:
            full = True
        else:
            new = res
    if full:
        out = bytearray(rec)
        struct.pack_into("<H", out, 18, f["flag"] | 4)
        return bytes(out), "unmapped", False, False, 0
    assert _qlen(new) == _qlen(ops)
    removed = _span(ops) - _span(new)
    end = pos + _span(new)
    body = bytearray(rec[4:36 + f["l_name"]])
    struct.pack_into("<i", body, 4, pos)
    struct.pack_into("<H", body, 10, reg2bin(pos, end))
    struct.pack_into("<H", body, 12, len(new))
    if len(new) > 65535:
        raise ValueError("the clipped CIGAR has more than 65535 operations")
    body += struct.pack(f"<{len(new)}I", *[L << 4 | op for op, L in new]) + f["tail"]
    return struct.pack("<i", len(body)) + bytes(body), "clipped", E is not None, S_ is not None, removed


def clip_records(recs, primers, tolerance: int = 5, both_ends: bool = False):
    """Every record clipped (input order) and the stats {n_left, n_right, n_unmapped, n_columns}.  ``primers``: (refID, start,
    end) rows."""
    primers = _by_ref(primers)
    out, st = [], dict(n_left=0, n_right=0, n_unmapped=0, n_columns=0)
    for r in recs:
        new, kind, left, right, removed = clip_record(r, primers, tolerance, both_ends)
        out.append(new)
        st["n_unmapped"] += kind == "unmapped"
        st["n_left"] += left
        st["n_right"] += right
        st["n_columns"] += removed
    return out, st


def sort_order(recs):
    """The order tc_bam_sort_records gives placed records: as they are when sorted by (refID, pos), else samtools' coordinate
    order (refID, pos + 1, forward before reverse, input order)."""
    keys = [struct.unpack_from("<iiBBHHH", r, 4) for r in recs]
    tp = [(k[0], k[1]) for k in keys]
    if all(tp[i] <= tp[i + 1] for i in range(len(tp) - 1)):
        return list(range(len(recs)))
    return sorted(range(len(recs)), key=lambda i: (keys[i][0], keys[i][1] + 1, (keys[i][6] >> 4) & 1, i))


def clip_and_sort(recs, primers, tolerance: int = 5, both_ends: bool = False):
    """What a decode with primers parses: the clipped records in tc_bam_sort_records' order, and the clip's stats."""
    out, st = clip_records(recs, primers, tolerance, both_ends)
    return [out[i] for i in sort_order(out)], st
