"""Coverage with the reference's API (TrueConsense/Coverage.py) plus the depth kernel entry.

``GetCoverage`` / ``BuildCoverage`` read the ``coverage`` column of the index dict exactly like
the reference.  ``DepthFromBam`` is the direct route: kernel (3) computes the same column from the
reads alone (difference array over read spans + scan, ``tc_depth``) without the full pileup.
"""
from __future__ import annotations

import numpy as np

from . import gpu


def BuildCoverage(iDict, output):
    """Write ``pos<TAB>coverage`` for positions 1..len(iDict) — Coverage.py:1-16."""
    with open(output, "w") as outfile:
        for i in range(len(iDict)):
            cov = iDict[i + 1].get("coverage")
            outfile.write(str(i + 1) + "\t" + str(cov) + "\n")


def BuildCoverageContigs(indexes, output):
    """``reference<TAB>pos<TAB>coverage`` (the usual three-column depth format), positions 1-based per reference, for
    ``{reference: index dict}`` in its order."""
    with open(output, "w") as outfile:
        for name, iDict in indexes.items():
            outfile.write("".join(f"{name}\t{i + 1}\t{iDict[i + 1].get('coverage')}\n" for i in range(len(iDict))))


def GetCoverage(iDict, position):
    """Coverage.py:19-34."""
    return iDict[position].get("coverage")


def DepthFromBam(bam, ref_len: int | None = None) -> np.ndarray:
    """int32[ref_len] depth of a ``Readbam`` handle through the GPU depth kernel; equals the
    ``coverage`` column BuildIndex produces."""
    from .Events import _bam_handle

    h = _bam_handle(bam)
    L = h.ref_len if ref_len is None else int(ref_len)
    return gpu.default_context().depth(h.device_reads(), L)


def WriteCoverage(depth: np.ndarray, output: str) -> None:
    """Coverage.py:13-16's TSV straight from a depth array."""
    pos = np.arange(1, depth.shape[0] + 1)
    with open(output, "w") as fh:
        fh.write("".join(f"{p}\t{c}\n" for p, c in zip(pos.tolist(), depth.tolist())))
