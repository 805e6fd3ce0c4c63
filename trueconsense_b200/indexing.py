"""Pileup index building with the reference's API (TrueConsense/indexing.py).

``BuildIndex(bamfile, ref)`` returns the same DataFrame (seven int64 columns
``coverage,A,T,C,G,X,I``, int64 index 1..len(ref[0]), ``index.name is None``) the reference
builds from a pysam pileup plus a per-string Python classifier (indexing.py:75-154).  Here the
BAM is inflated on the host (csrc/host/bamio.c), its records are parsed on the GPU into flat arrays
(``tc_bam_records_to_reads``) and the whole pileup is one pass of the CUDA kernels behind ``tc_pileup_counts``.
"""
from __future__ import annotations

import pathlib
import threading
from dataclasses import dataclass

import numpy as np
import pandas as pd

from . import bamio, gpu
from .reads import ReadBatch

COLUMNS = ["coverage", "A", "T", "C", "G", "X", "I"]

# the refusals of a pass over one reference: pysam's pileup message for reads out of order, and ours for a second reference
UNSORTED = "Unsorted input. Pileup aborts"
MULTI_CONTIG = ("multi-contig BAM: TrueConsense indexes positions of a single reference "
                "(its DataFrame index would hold duplicate positions)")


def _refuse(multi_contig: bool, unsorted: bool) -> None:
    if multi_contig:
        raise ValueError(MULTI_CONTIG)
    if unsorted:
        raise ValueError(UNSORTED)


def _fresh(d, ctx) -> bool:
    """Whether device reads made earlier still sit in ``ctx``'s buffers (the context has staged nothing since)."""
    return d is not None and d.ctx is ctx and d.generation == ctx._generation


class BamHandle:
    """What ``Readbam`` returns: a BAM on its way to the device plus the attributes of ``pysam.AlignmentFile`` the reference
    touches (``references``; Events.py:63).  The file travels to the device as it is: BGZF members inflated, record offsets
    found and records parsed on the GPU (``gpu.Context.bam_file_to_device``) straight into the context's read buffers; ``reads`` (a host-side decode into numpy arrays) is
    only made when somebody asks for it.

    ``sort``: a file whose records are not sorted by (refID, pos) (aligner output, a queryname-sorted BAM) is accepted and its
    records are put in samtools' coordinate order on the GPU (``tc_bam_sort_records``), so every pass computes what it
    computes after ``samtools sort``; a sorted file is used as written.  Only the device reads are reordered: ``reads``, the
    host decode, stays in file order, and a handle made from a host ``ReadBatch`` (``reads=``) that is not sorted still
    raises ``ValueError`` (host batches are not sorted here).

    A path ending in ``.sam`` is an aligner's text output: its lines become BAM records on the GPU
    (``gpu.Context.sam_file_to_device``) and take the BAM route from there, ``sort`` included.  There is no host decode of
    SAM: ``reads`` raises ``NotImplementedError``, the device arrays are the product.

    ``primers`` (a ``primers.PrimerScheme``, ``primers.read_bed``): the amplicon primers are soft-clipped off the records on
    the GPU before the sort (``tc_bam_clip_primers``), so every pass computes what it computes after ``samtools ampliconclip``
    and ``samtools sort``; ``sort`` is then always on.  There is no host-side clip: ``reads`` raises
    ``NotImplementedError``, and a handle made from a host ``ReadBatch`` cannot take primers (``ValueError``).

    ``output_bam`` (a path): the records the device reads were parsed from (clipped and sorted when asked) are written there
    as a BAM (``gpu.Context.write_bam``), once, at the first device decode and after its checks pass: an input the decode
    refuses leaves no file.  A handle made from a host ``ReadBatch`` cannot take it (``ValueError``)."""

    def __init__(self, filename: str, reads: ReadBatch | None = None, sort: bool = False, primers=None, output_bam=None):
        if primers is not None and reads is not None:
            raise ValueError("primers are clipped on the GPU during the decode of a file; a host ReadBatch cannot take them")
        if output_bam is not None and reads is not None:
            raise ValueError("output_bam writes the records of a file decoded on the GPU; a host ReadBatch holds none")
        self.output_bam = output_bam
        self._written = output_bam is None
        self._payload = None            # the host payload of the fallback route, kept until the BAM is written
        self.filename = filename
        self.sort = sort or primers is not None
        self.primers = primers
        self.is_sam = reads is None and pathlib.Path(filename).suffix == ".sam"
        self._reads = reads
        self._hdr = None
        self._dev = None
        self._dev_contigs = None        # (key, DeviceReads, ContigLayout): the reads moved to a multi-reference layout
        self._lock = threading.Lock()
        self._insert_cache: dict = {}

    @property
    def reads(self) -> ReadBatch:
        with self._lock:
            if self._reads is None:
                if self.is_sam:
                    raise NotImplementedError(f"{self.filename}: a SAM file is decoded on the GPU only (device_reads); "
                                              "there are no host-side read arrays of it")
                if self.primers is not None:
                    raise NotImplementedError(f"{self.filename}: primers are clipped on the GPU only (device_reads); "
                                              "there are no host-side read arrays of the clipped reads")
                self._reads = bamio.read_bam(self.filename)
            return self._reads

    def _header(self):
        """(reference names, reference lengths) from whichever decode exists."""
        with self._lock:
            if self._reads is not None:
                return self._reads.ref_names, self._reads.ref_lens
            if self._hdr is None and self.is_sam:
                self._hdr = bamio.read_sam_header(self.filename)[:2]    # the '@' lines only
            if self._hdr is None:
                self._hdr = bamio.read_bam_header(self.filename)       # only the members holding the header are inflated
            return self._hdr

    @property
    def references(self):
        return tuple(self._header()[0])

    @property
    def lengths(self):
        return tuple(self._header()[1])

    @property
    def ref_len(self) -> int:
        return int(self._header()[1][0])

    def contig0(self) -> ReadBatch:
        """Host-side reads placed on the first reference (the only one the reference implementation is
        meaningful for: indexing.py:98,139 and Events.py:63 use lengths[0] / references[0])."""
        b = self.reads
        _refuse(b.tid is not None and b.n_reads and np.any(b.tid != 0), False)
        return b

    def device_reads(self, with_host_qual: bool = False):
        """The reads in device memory, made once per handle and reused by later passes while the context has not staged
        anything else.  From a file: inflated on the host, parsed on the GPU (QUAL and the mate fields included).  From a
        host batch handed to the constructor: uploaded without QUAL / mate fields, which ExtractInserts then stages for the
        reads over its candidate columns only."""
        ctx = gpu.default_context()
        with self._lock:
            d = self._dev
            if not _fresh(d, ctx):
                b = self._reads
                if b is not None:       # refused before anything is staged
                    _refuse(b.tid is not None and b.n_reads and np.any(b.tid != 0), not b.sorted)
                d = self._to_device(ctx)
                if b is None:
                    _refuse(d.stats.multi_contig, d.stats.unsorted)
                self._write_once(ctx, d)
                self._dev = d
            return d.with_host_qual() if with_host_qual else d

    def device_reads_contigs(self, names, lens):
        """The reads in device memory moved to the global columns of a multi-reference pass, and that layout
        (``ContigLayout``): every reference of the header (``names``, in header order) side by side with the lengths
        ``lens`` (from the FASTA).  Kept apart from :meth:`device_reads` — the two share the context's buffers, so making one
        makes the other stale, and each is made again when asked for."""
        ctx = gpu.default_context()
        key = (tuple(names), tuple(int(x) for x in lens))
        with self._lock:
            c = self._dev_contigs
            if c is not None and c[0] == key and _fresh(c[1], ctx):
                return c[1], c[2]
            self._dev_contigs = None
            b = self._reads
            if b is not None:           # refused before anything is staged
                _refuse(False, not b.sorted)
                first_read = contig_ranges_from_tid(b.tid, len(names), b.n_reads)
            d = self._to_device(ctx, contig_ranges=True)
            if b is None:
                _refuse(False, d.stats.unsorted)
                first_read = d.first_read
            if len(first_read) != len(names) + 1:
                raise ValueError(f"the BAM header holds {len(first_read) - 1} references, {len(names)} were given")
            self._write_once(ctx, d)
            start = ctx.reads_to_contig_coords(d, key[1], first_read, names)
            layout = ContigLayout(list(names), list(key[1]), start.astype(np.int64), np.asarray(first_read, np.int64))
            self._dev_contigs = (key, d, layout)
            return d, layout

    def _to_device(self, ctx, contig_ranges: bool = False):
        """The reads in device memory, not yet checked (the caller holds the lock).  A host batch is uploaded: for a pass
        over one reference without QUAL and the mate fields (see :meth:`device_reads`), for a multi-reference pass
        (``contig_ranges``) with them, as the move shifts PNEXT on the device.  A file is decoded on the GPU."""
        if self._reads is not None:
            return ctx.upload(self._reads, with_qual=contig_ranges)
        kw = dict(contig_ranges=contig_ranges, sort=self.sort, primers=self.primers)
        if self.is_sam:
            d = ctx.sam_file_to_device(self.filename, **kw)
        else:
            try:
                # inflate, record index, (clip, sort) and parse on the GPU
                d = ctx.bam_file_to_device(self.filename, **kw)
            except gpu.TcError:
                # a file the device path refuses: the host reader names the broken member / record (or, should it
                # read the file after all, feeds the device parse)
                payload = bamio.read_bam_payload(self.filename)
                d = ctx.bam_to_device(payload, **kw)
                if self._written:
                    payload.release()       # the device holds the arrays now
                else:
                    self._payload = payload     # unsorted, unclipped records stay in the host payload until written
        self._hdr = (d.ref_names, d.ref_lens)
        return d

    def _write_once(self, ctx, d) -> None:
        """``output_bam`` from the first device decode that passed its checks (the caller holds the lock)."""
        if self._written:
            return
        ctx.write_bam(d, self.output_bam)
        self._written = True
        if self._payload is not None:
            self._payload.release()
            self._payload = None

    def pileup(self, *args, **kwargs):
        raise NotImplementedError("column iteration is not part of this implementation; "
                                  "use Events.ExtractInserts / indexing.BuildIndex")

    def close(self):
        pass


@dataclass
class ContigLayout:
    """Every reference of a BAM side by side: reference k (``names[k]``, ``lens[k]`` columns) occupies the global columns
    ``start[k]`` .. ``start[k+1]-1``; its reads are ``first_read[k]`` .. ``first_read[k+1]-1``."""

    names: list
    lens: list
    start: np.ndarray
    first_read: np.ndarray

    @property
    def total(self) -> int:
        return int(self.start[-1])

    def locate(self, positions) -> tuple[np.ndarray, np.ndarray]:
        """1-based global positions -> (reference index, 1-based position on that reference)."""
        p = np.asarray(positions, dtype=np.int64)
        k = np.searchsorted(self.start, p - 1, side="right") - 1
        return k, p - self.start[k]


def contig_ranges_from_tid(tid, n_ref: int, n_reads: int) -> np.ndarray:
    """``first_read[n_ref + 1]`` of a host-decoded batch (``ReadBatch.tid``, sorted): what ``tc_bam_contig_ranges`` computes
    on the device from the records."""
    t = np.zeros(n_reads, np.int32) if tid is None else np.asarray(tid)
    if t.size and (int(t.min()) < 0 or int(t.max()) >= n_ref):
        raise ValueError(f"a read's reference index lies outside the header's {n_ref} references")
    if t.size and np.any(np.diff(t.astype(np.int64)) < 0):
        raise ValueError(UNSORTED)
    return np.searchsorted(t, np.arange(n_ref + 1), side="left").astype(np.int32)


def fasta_lengths_by_name(names, ref) -> list[int]:
    """The lengths of the FASTA records named like the BAM's references (the first record of a name counts), in the
    order of ``names``.  A reference without a record is a ValueError that names it."""
    fnames, flens = bamio.read_fasta_lengths(ref)
    by_name: dict[str, int] = {}
    for n, l in zip(fnames, flens):
        by_name.setdefault(n, int(l))
    missing = [n for n in names if n not in by_name]
    if missing:
        raise ValueError(f"reference {missing[0]!r} of the BAM header has no record in {ref}"
                         + (f" (nor have {len(missing) - 1} more)" if len(missing) > 1 else ""))
    return [by_name[n] for n in names]


def gff_by_contig(df: pd.DataFrame, names) -> dict:
    """The GFF rows of every reference (by ``seqid``), in the order of ``names``, each frame indexed 0.. like a GFF file
    holding only that reference's rows.  A row whose seqid names no reference is a ValueError: dropping it would lose
    that feature's ORF corrections."""
    known = set(names)
    unknown = sorted(set(df["seqid"]) - known)
    if unknown:
        raise ValueError(f"GFF rows with seqid {unknown[0]!r} name no reference of the BAM ({len(names)} references)")
    return {n: df[df["seqid"] == n].reset_index(drop=True) for n in names}


def Readbam(f, sort: bool = False, primers=None, output_bam=None):
    """indexing.py:6-19.  A handle passed in is returned as is, so one decoded copy of the BAM can
    serve BuildIndex, ListInserts and WriteOutputs.  ``sort``: accept records that are not coordinate-sorted and put them
    in samtools' coordinate order on the GPU (``BamHandle``).  A ``.sam`` path is read as SAM text, on the GPU.
    ``primers`` (``primers.read_bed``): the amplicon primers are soft-clipped off the reads on the GPU (implies ``sort``).
    ``output_bam``: the decoded (clipped, sorted) records are also written to this path as a BAM (``BamHandle``)."""
    if isinstance(f, BamHandle):
        return f
    return BamHandle(f, sort=sort, primers=primers, output_bam=output_bam)


class _GffHeader:
    def __init__(self, raw_text: str):
        self.raw_text = raw_text


class GffIndex:
    """Stand-in for AminoExtract's GFFDataFrame (not installed here): ``.df`` with the nine GFF3
    columns (start/end int64) and ``.header.raw_text`` — all the reference reads
    (TrueConsense.py:238-241, Outputs.py:66)."""

    GFF_COLUMNS = ["seqid", "source", "type", "start", "end", "score", "strand", "phase", "attributes"]

    def __init__(self, file: str):
        header, rows = [], []
        with open(file) as fh:
            for line in fh:
                if line.startswith("#"):
                    if not rows:
                        header.append(line)
                    continue
                if not line.strip():
                    continue
                f = line.rstrip("\n").split("\t")
                f += [""] * (9 - len(f))
                rows.append(f[:9])
        self.header = _GffHeader("".join(header))
        df = pd.DataFrame(rows, columns=self.GFF_COLUMNS)
        df["start"] = df["start"].astype("int64")
        df["end"] = df["end"].astype("int64")
        self.df = df


def Gffindex(file: str) -> GffIndex:
    """indexing.py:22-36."""
    return GffIndex(file)


def read_override_index(f):
    """indexing.py:39-52."""
    return pd.read_csv(f, sep=",", compression="gzip", index_col=0)


def Override_index_positions(index, override_data):
    """indexing.py:55-72."""
    index.loc[override_data.index, :] = override_data[:]
    return index


def frame_from_counts(counts: np.ndarray) -> pd.DataFrame:
    """int32[8][L] count table -> the reference's index frame."""
    L = counts.shape[1]
    df = pd.DataFrame({c: counts[r].astype(np.int64) for r, c in enumerate(COLUMNS)},
                      index=pd.Index(np.arange(1, L + 1, dtype=np.int64)))
    df.index.name = None
    return df


def BuildIndex(bamfile, ref):
    """indexing.py:75-154."""
    handle = bamfile if isinstance(bamfile, BamHandle) else BamHandle(bamfile)
    _, lens = bamio.read_fasta_lengths(ref)
    if not lens:
        raise ValueError(f"no sequences in {ref}")
    ref_length = int(lens[0])
    counts = gpu.default_context().pileup_counts(handle.device_reads(), ref_length)
    return frame_from_counts(counts)


def BuildIndexContigs(bamfile, ref):
    """``BuildIndex`` for every reference of the BAM header in one device pass: ``{reference: frame}`` in header order, each
    frame equal to ``BuildIndex`` over a BAM holding only that reference's records and the FASTA record of its name."""
    handle = bamfile if isinstance(bamfile, BamHandle) else BamHandle(bamfile)
    names = list(handle.references)
    if not names:
        raise ValueError(f"{handle.filename}: the BAM header lists no reference")
    lens = fasta_lengths_by_name(names, ref)
    d, lay = handle.device_reads_contigs(names, lens)
    counts = gpu.default_context().pileup_counts(d, lay.total)
    return {n: frame_from_counts(counts[:, lay.start[k]:lay.start[k + 1]]) for k, n in enumerate(names)}
