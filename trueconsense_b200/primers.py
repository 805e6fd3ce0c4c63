"""Amplicon primer schemes (BED) for the clip that ``gpu.Context`` runs on the decoded records (``tc_bam_clip_primers``).

``read_bed(path)`` reads ``chrom start end [...]`` rows, 0-based half-open, as ARTIC-style schemes ship them
(``*.primer.bed``); ``PrimerScheme.rows(names)`` maps the chrom names to the reference indices of a BAM / SAM header.
"""
from __future__ import annotations

import re
from dataclasses import dataclass

import numpy as np

INT32_MAX = 2**31 - 1


@dataclass(frozen=True)
class PrimerScheme:
    """The primers of a BED file and how they are clipped: ``tolerance`` (bases a read end may start in front of a primer's
    start, or end behind a primer's end, and still match it) and ``both_ends`` (check both ends of every read, as nanopore
    reads spanning the whole amplicon need; else only the 5' end)."""

    path: str
    chrom: tuple
    start: np.ndarray
    end: np.ndarray
    tolerance: int = 5
    both_ends: bool = False

    def __post_init__(self):
        if isinstance(self.tolerance, bool) or not isinstance(self.tolerance, (int, np.integer)) or self.tolerance < 0:
            raise ValueError(f"primer tolerance must be an integer >= 0, not {self.tolerance!r}")

    def __len__(self) -> int:
        return len(self.chrom)

    def rows(self, names) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(reference index, start, end) int32 arrays for a header whose references are ``names``.  A chrom that names no
        reference of the header is a ValueError naming it: dropping its rows would leave those primers in the reads."""
        index = {n: i for i, n in enumerate(names)}
        unknown = sorted(set(self.chrom) - set(index))
        if unknown:
            raise ValueError(f"{self.path}: primer chrom {unknown[0]!r} names no reference of the BAM ({len(index)} references)")
        ref = np.array([index[c] for c in self.chrom], np.int32)
        return ref, np.ascontiguousarray(self.start, np.int32), np.ascontiguousarray(self.end, np.int32)


def read_bed(path: str, tolerance: int = 5, both_ends: bool = False) -> PrimerScheme:
    """The primers of a BED file.  Blank lines, ``#`` lines and ``track`` / ``browser`` lines (the word, then a space, a tab
    or the line's end: a chrom such as ``track1`` is data) are skipped; fields are split on
    tabs (CRLF line ends are fine); columns after the third are ignored.  A row with fewer than 3 fields, a start or end
    that is not an integer, is negative or above 2^31 - 1, or start >= end is ``ValueError("<path>: line <k>: <reason>")``.
    An empty scheme is allowed."""
    chrom, start, end = [], [], []
    with open(path, "rb") as fh:
        for k, raw in enumerate(fh, 1):
            line = raw.decode(errors="surrogateescape").rstrip("\r\n")
            if not line.strip() or line.startswith("#") or re.match(r"(track|browser)([ \t]|$)", line):
                continue
            f = line.split("\t")
            if len(f) < 3:
                raise ValueError(f"{path}: line {k}: fewer than 3 tab-separated fields")
            vals = []
            for what, v in (("start", f[1]), ("end", f[2])):
                if not re.fullmatch(r"[+-]?[0-9]+", v.strip()):
                    raise ValueError(f"{path}: line {k}: {what} {v!r} is not an integer")
                x = int(v)
                if x < 0:
                    raise ValueError(f"{path}: line {k}: {what} {x} is negative")
                if x > INT32_MAX:
                    raise ValueError(f"{path}: line {k}: {what} {x} is above 2^31 - 1")
                vals.append(x)
            if vals[0] >= vals[1]:
                raise ValueError(f"{path}: line {k}: start {vals[0]} is not below end {vals[1]}")
            chrom.append(f[0])
            start.append(vals[0])
            end.append(vals[1])
    return PrimerScheme(str(path), tuple(chrom), np.array(start, np.int32), np.array(end, np.int32), tolerance, both_ends)
