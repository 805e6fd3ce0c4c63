"""ctypes binding of the C-ABI in include/trueconsense_b200.h (libtcb200.so).

There is no CPU fallback: if the library cannot be loaded or no CUDA device is usable, the
calls raise.  Arguments may be numpy arrays (host) or torch CUDA tensors (device); the library
detects which from the pointer.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from dataclasses import dataclass

import numpy as np

from . import build
from .reads import ReadBatch, TcReads

TC_NROWS = 8
ROWS = ("coverage", "A", "T", "C", "G", "X", "I")

CF_LOWCOV, CF_PRIMARY_X, CF_MINORITY_DEL, CF_INS_CANDIDATE = 0x01, 0x02, 0x04, 0x08
CF_COV_GT_MINCOV, CF_XRUN_OFF_END, CF_ZERO_COV, CF_AMBIG = 0x10, 0x20, 0x40, 0x80

ERR_NAMES = {-1: "TC_ERR_CUDA", -2: "TC_ERR_ARG", -3: "TC_ERR_UNSORTED", -4: "TC_ERR_DEPTH_CAP", -5: "TC_ERR_NOMEM",
             -6: "TC_ERR_NO_DEVICE", -7: "TC_ERR_RANGE", -8: "TC_ERR_CAPACITY"}


class TcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class PileupParams(C.Structure):
    _fields_ = [("flag_filter", C.c_uint32), ("min_mapq", C.c_int32), ("min_base_quality", C.c_int32),
                ("ignore_orphans", C.c_int32), ("max_depth", C.c_int64), ("kernel", C.c_int32), ("reserved", C.c_int32)]


class BamStats(C.Structure):
    _fields_ = [("aligned_bases", C.c_uint64), ("max_ref_span", C.c_int32), ("unsorted", C.c_int32), ("multi_contig", C.c_int32),
                ("sorted", C.c_int32), ("n_seq_words", C.c_int64), ("n_cigar_ops", C.c_int64)]


class ClipStats(C.Structure):
    _fields_ = [("n_left", C.c_int64), ("n_right", C.c_int64), ("n_unmapped", C.c_int64), ("n_columns", C.c_int64)]


class CallParams(C.Structure):
    _fields_ = [("mincov", C.c_int32), ("include_ambig", C.c_int32), ("ambig_maxdist", C.c_double),
                ("minority_del_pct", C.c_double), ("insert_pct", C.c_double)]


class CallTable(C.Structure):
    _fields_ = [("call_char", C.c_void_p), ("flags", C.c_void_p), ("xrun", C.c_void_p), ("rank_letter", C.c_void_p),
                ("rank_count", C.c_void_p), ("ambig_char", C.c_void_p)]


class InsertCall(C.Structure):
    _fields_ = [("pos", C.c_int32), ("n_entries", C.c_int32), ("mode_count", C.c_int32), ("first_read", C.c_int32),
                ("head", C.c_int32), ("indel", C.c_int32), ("bases_off", C.c_int64)]


def buildindex_params(kernel: int = 0) -> PileupParams:
    """pysam arguments of TrueConsense/indexing.py:100: stepper="nofilter" (htslib still drops
    UNMAP), max_depth=10000000, min_base_quality=0."""
    return PileupParams(flag_filter=0x4, min_mapq=0, min_base_quality=0, ignore_orphans=0, max_depth=10_000_000,
                        kernel=kernel, reserved=0)


def extractinserts_params() -> PileupParams:
    """pysam defaults used by TrueConsense/Events.py:66."""
    return PileupParams(flag_filter=0x4 | 0x100 | 0x200 | 0x400, min_mapq=0, min_base_quality=13, ignore_orphans=1,
                        max_depth=8000, kernel=0, reserved=0)


_lib = None
_lib_lock = threading.Lock()


def lib() -> C.CDLL:
    """Load libtcb200.so (built in-tree by ``trueconsense_b200.build``).  Raises if it is missing:
    there is nothing to fall back to."""
    global _lib
    with _lib_lock:
        if _lib is None:
            path = build.CUDA_LIB
            if not os.path.exists(path):
                raise RuntimeError(
                    f"{path} is missing — the CUDA extension is the only implementation of the hot path. "
                    "Build it with `python -m trueconsense_b200.build cuda` (needs nvcc).")
            l = C.CDLL(path)
            vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
            l.tc_abi_version.restype = C.c_int
            l.tc_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
            l.tc_ctx_destroy.argtypes = [vp]
            l.tc_last_error.argtypes = [vp]
            l.tc_last_error.restype = C.c_char_p
            l.tc_launch_count.argtypes = [vp]
            l.tc_launch_count.restype = i64
            l.tc_transfer_bytes.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
            l.tc_transfer_bytes.restype = C.c_int
            l.tc_ctx_set_timing.argtypes = [vp, C.c_int]
            l.tc_ctx_set_timing.restype = C.c_int
            l.tc_last_pileup_kernel_ms.argtypes = [vp]
            l.tc_last_pileup_kernel_ms.restype = C.c_float
            l.tc_reads_upload.argtypes = [vp, C.POINTER(TcReads), C.POINTER(TcReads), vp]
            l.tc_pileup_counts.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), vp, vp]
            l.tc_depth.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), vp, vp]
            l.tc_call.argtypes = [vp, vp, i32, C.POINTER(CallParams), C.POINTER(CallTable), vp]
            l.tc_is_ambiguous.argtypes = [vp, vp, vp, vp, i64, C.c_double, vp, vp]
            l.tc_extract_inserts.argtypes = [vp, C.POINTER(TcReads), i32, vp, i32, C.POINTER(PileupParams),
                                             C.POINTER(InsertCall), vp, i64, vp]
            l.tc_list_insert_candidates.argtypes = [vp, vp, i32, vp, i32, C.POINTER(i32), vp]
            l.tc_allreduce_counts.argtypes = [vp, vp, i64, vp, vp]
            l.tc_pileup_counts_allreduce.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), vp, vp, vp]
            l.tc_pileup_counts_allreduce.restype = C.c_int
            l.tc_pileup_counts_allreduce_enqueue.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), vp, vp, vp, C.POINTER(i32)]
            l.tc_pileup_counts_allreduce_enqueue.restype = C.c_int
            l.tc_pileup_counts_allreduce_finish.argtypes = [vp, i32]
            l.tc_pileup_counts_allreduce_finish.restype = C.c_int
            l.tc_pileup_call_inserts.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), C.POINTER(CallParams),
                                                 C.POINTER(PileupParams), vp, C.POINTER(CallTable), C.POINTER(InsertCall), i32,
                                                 C.POINTER(i32), vp, i64, vp]
            l.tc_bam_records_to_reads.argtypes = [vp, vp, i64, vp, i64, C.POINTER(TcReads), C.POINTER(BamStats), vp]
            l.tc_bam_records_to_reads.restype = C.c_int
            l.tc_bam_sort_records.argtypes = [vp, vp, i64, vp, i64, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(i32), vp]
            l.tc_bam_sort_records.restype = C.c_int
            l.tc_bam_clip_primers.argtypes = [vp, vp, i64, vp, i64, i32, vp, vp, vp, i32, i32, C.c_uint32, C.POINTER(vp), C.POINTER(i64),
                                              C.POINTER(vp), C.POINTER(ClipStats), vp]
            l.tc_bam_clip_primers.restype = C.c_int
            l.tc_sam_to_bam_records.argtypes = [vp, vp, i64, i64, i64, i32, vp, vp, C.POINTER(vp), C.POINTER(i64), C.POINTER(vp),
                                                C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_double), vp]
            l.tc_sam_to_bam_records.restype = C.c_int
            l.tc_bgzf_inflate.argtypes = [vp, vp, i64, vp, i64, i64, C.POINTER(vp), vp]
            l.tc_bgzf_inflate.restype = C.c_int
            l.tc_bam_index_records.argtypes = [vp, vp, i64, i64, i32, vp, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), vp]
            l.tc_bam_index_records.restype = C.c_int
            l.tc_bam_write_records.argtypes = [vp, vp, i64, vp, i64, vp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64),
                                               C.POINTER(C.c_float), vp]
            l.tc_bam_write_records.restype = C.c_int
            l.tc_download.argtypes = [vp, vp, vp, i64, vp]
            l.tc_download.restype = C.c_int
            l.tc_sample_enqueue.argtypes = [vp, C.POINTER(TcReads), i32, C.POINTER(PileupParams), C.POINTER(CallParams),
                                            C.POINTER(PileupParams), vp, C.POINTER(CallTable), vp, C.POINTER(i32)]
            l.tc_sample_finish.argtypes = [vp, i32, C.POINTER(InsertCall), i32, C.POINTER(i32), vp, i64]
            l.tc_sample_enqueue.restype = l.tc_sample_finish.restype = C.c_int
            l.tc_bam_contig_ranges.argtypes = [vp, vp, i64, vp, i64, i32, vp, vp]
            l.tc_reads_to_contig_coords.argtypes = [vp, C.POINTER(TcReads), i32, vp, vp, vp, vp]
            l.tc_call_contigs.argtypes = [vp, vp, i32, i32, vp, C.POINTER(CallParams), C.POINTER(CallTable), vp]
            l.tc_bam_contig_ranges.restype = l.tc_reads_to_contig_coords.restype = l.tc_call_contigs.restype = C.c_int
            for name in ("tc_ctx_create", "tc_ctx_destroy", "tc_reads_upload", "tc_pileup_counts", "tc_depth", "tc_call",
                         "tc_is_ambiguous", "tc_extract_inserts", "tc_list_insert_candidates", "tc_allreduce_counts", "tc_pileup_call_inserts"):
                getattr(l, name).restype = C.c_int
            _lib = l
    return _lib


def _ptr(x):
    """Raw pointer of a numpy array or a torch tensor (None passes through)."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return x.data_ptr()
    if isinstance(x, int):
        return x
    raise TypeError(type(x))


@dataclass
class CallResult:
    call_char: np.ndarray
    flags: np.ndarray
    xrun: np.ndarray
    rank_letter: np.ndarray
    rank_count: np.ndarray
    ambig_char: np.ndarray

    def slice(self, a: int, b: int) -> "CallResult":
        """Columns [a, b) of the table (views): one reference's part of a multi-reference table."""
        return CallResult(self.call_char[a:b], self.flags[a:b], self.xrun[a:b], self.rank_letter[:, a:b], self.rank_count[:, a:b],
                          self.ambig_char[a:b])


def _call_buffers(counts, L: int):
    """Host outputs of a call table of L columns, the CallTable pointing at them, and ``counts`` checked (numpy: [8][L])."""
    res = CallResult(np.empty(L, np.uint8), np.empty(L, np.uint8), np.empty(L, np.int32), np.empty((4, L), np.uint8),
                     np.empty((4, L), np.int32), np.empty(L, np.uint8))
    t = CallTable(_ptr(res.call_char), _ptr(res.flags), _ptr(res.xrun), _ptr(res.rank_letter), _ptr(res.rank_count),
                  _ptr(res.ambig_char))
    if isinstance(counts, np.ndarray):
        counts = np.ascontiguousarray(counts, dtype=np.int32)
        if counts.shape != (TC_NROWS, L):
            raise ValueError(f"counts must be [{TC_NROWS}][{L}]")
    return res, t, counts


class DeviceReads:
    """A read batch resident in context-owned device memory (see tc_reads_upload)."""

    def __init__(self, struct: TcReads, batch: ReadBatch | None, ctx=None, generation: int = 0):
        self.struct = struct
        self.n_reads = int(struct.n_reads) if batch is None else batch.n_reads
        self.host = batch           # None: parsed on the device (bam_to_device), every array lives there
        self.ctx = ctx
        self.generation = generation
        self.stats = None
        self.info = {}              # what the decode counted and how long each step took (the *_to_device routes)
        self.ref_names = None       # the header's references (the *_to_device routes)
        self.ref_lens = None
        self.first_read = None      # [n_ref + 1]: where each reference's reads begin (bam_file_to_device(contig_ranges=True))
        self.contig_start = None    # set once the reads sit in the global columns of a multi-reference pass
        self.records = None         # (BAM header bytes, payload, bytes, record offsets, count) the reads were parsed from

    def with_host_qual(self) -> "DeviceReads":
        """The same device arrays plus the batch's HOST quality and mate arrays (QNAME hash, PNEXT, TLEN):
        tc_extract_inserts then copies them only for the reads over its candidate columns."""
        if self.host is None:
            return self
        st = TcReads()
        C.memmove(C.byref(st), C.byref(self.struct), C.sizeof(TcReads))
        if not st.qual and self.host.qual is not None:
            st.qual = self.host.qual.ctypes.data
        if not st.qname_hash and self.host.qname_hash is not None and self.host.mpos is not None and self.host.isize is not None:
            st.qname_hash = self.host.qname_hash.ctypes.data
            st.mpos = self.host.mpos.ctypes.data
            st.isize = self.host.isize.ctypes.data
        return DeviceReads(st, self.host, self.ctx, self.generation)


class Context:
    """One ``tc_ctx_t``: a device, its workspace buffers and a launch counter."""

    def __init__(self, device: int = -1):
        self._lib = lib()
        h = C.c_void_p()
        rc = self._lib.tc_ctx_create(device, C.byref(h))
        if rc != 0:
            raise TcError(rc, self._lib.tc_last_error(None).decode())
        self._h = h
        self._generation = 0        # bumped whenever host arrays are staged through the context's device buffers

    def close(self):
        if getattr(self, "_h", None):
            self._lib.tc_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise TcError(rc, self._lib.tc_last_error(self._h).decode())

    @property
    def launches(self) -> int:
        return int(self._lib.tc_launch_count(self._h))

    def transfer_bytes(self) -> tuple[int, int]:
        """(host->device, device->host) bytes copied by this context so far."""
        a, b = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.tc_transfer_bytes(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def set_timing(self, enabled: bool) -> None:
        self._check(self._lib.tc_ctx_set_timing(self._h, int(enabled)))

    def last_pileup_kernel_ms(self) -> float:
        """CUDA-event duration of the dominant kernel of the last pileup_counts call (timing on)."""
        return float(self._lib.tc_last_pileup_kernel_ms(self._h))

    # ------------------------------------------------------------------ reads
    def _reads_struct(self, reads) -> TcReads:
        if isinstance(reads, DeviceReads):
            if reads.ctx is self and reads.generation != self._generation:
                raise RuntimeError("these device reads are stale: the context has staged another batch since they were uploaded")
            return reads.struct
        if isinstance(reads, ReadBatch):
            self._generation += 1           # host arrays are staged through the same device buffers
            return reads.c_struct()
        if isinstance(reads, TcReads):
            return reads
        raise TypeError(type(reads))

    def upload(self, batch: ReadBatch, stream: int = 0, with_qual: bool = True) -> DeviceReads:
        """Copy a host batch into the context's device buffers.  They are reused by the next upload — and by any
        later call that is handed host arrays — so a DeviceReads is only valid until then (checked)."""
        dev = TcReads()
        host = batch.c_struct()
        if not with_qual:       # what only tc_extract_inserts reads stays on the host (see DeviceReads.with_host_qual)
            host.qual = None
            host.qname_hash = host.mpos = host.isize = None
        self._generation += 1
        self._check(self._lib.tc_reads_upload(self._h, C.byref(host), C.byref(dev), stream))
        return DeviceReads(dev, batch, self, self._generation)

    def download(self, dev_ptr: int, count: int, dtype, stream: int = 0) -> np.ndarray:
        """``count`` elements of ``dtype`` from device memory (e.g. a field of ``DeviceReads.struct``) as a numpy array."""
        out = np.empty(int(count), dtype=dtype)
        self._check(self._lib.tc_download(self._h, _ptr(out), dev_ptr, out.nbytes, stream))
        return out

    def clip_primers(self, payload_ptr, n_bytes: int, rec_ptr, n_reads: int, names, primers, stream: int = 0):
        """``tc_bam_clip_primers``: the records (payload and refID offsets, host or device) with the primers of ``primers`` (a
        ``primers.PrimerScheme``; its chrom names mapped to ``names``, the header's references) soft-clipped off.  Returns
        (device payload, its bytes, device record offsets in input order, ``ClipStats``); the buffers stay valid until the next
        decode on this context.  A chrom the header does not list is a ValueError."""
        ref, start, end = primers.rows(names)
        p, nb, r, st = C.c_void_p(), C.c_int64(0), C.c_void_p(), ClipStats()
        self._check(self._lib.tc_bam_clip_primers(self._h, payload_ptr, n_bytes, rec_ptr, n_reads, len(names), ref.ctypes.data,
                                                  start.ctypes.data, end.ctypes.data, len(primers), int(primers.tolerance),
                                                  int(bool(primers.both_ends)), C.byref(p), C.byref(nb), C.byref(r), C.byref(st), stream))
        return p.value, int(nb.value), r.value, st

    def bam_to_device(self, payload, stream: int = 0, contig_ranges: bool = False, sort: bool = False, primers=None) -> DeviceReads:
        """GPU-side record parsing (tc_bam_records_to_reads): a ``bamio.BamPayload`` (the BAM inflated on the host, its records
        indexed) becomes the flat read arrays in the context's device buffers — the CPU never touches a record's body.
        ``.stats`` of the result: aligned bases, longest span, sortedness, whether more than one reference occurs.
        ``sort``: records that are not sorted by (refID, pos) are put in samtools' coordinate order first
        (``tc_bam_sort_records``; the payload then travels to the device once); ``.info`` says whether they moved
        (``reordered``) and what that took (``t_sort_s``).
        ``primers`` (a ``primers.PrimerScheme``): the primers are soft-clipped off the records first (``tc_bam_clip_primers``)
        and the clipped records are sorted (``sort`` is implied); ``.info`` then also holds the clip's counts and ``t_clip_s``.
        The result carries ``.ref_names`` and ``.ref_lens`` (the payload's header), and ``contig_ranges`` adds ``.first_read``
        as for :meth:`bam_file_to_device`."""
        from . import bamio

        n = 1 << 16
        while (hdr := bamio.parse_bam_header(C.string_at(payload.payload_ptr, min(n, payload.n_bytes)), payload.n_bytes)) is None:
            n *= 4
        header = C.string_at(payload.payload_ptr, hdr[2])
        self._generation += 1
        return self._records_to_device(payload.payload_ptr, payload.n_bytes, payload.rec_off_ptr, payload.n_reads,
                                       payload.ref_names, payload.ref_lens, {}, stream, contig_ranges, sort, primers, header)

    def bam_file_to_device(self, path: str, stream: int = 0, contig_ranges: bool = False, sort: bool = False,
                           primers=None) -> DeviceReads:
        """A BAM file to the flat read arrays in device memory with the GPU doing all of it: the host maps the file and walks
        the BGZF member headers (``bamio.map_bgzf``); the device inflates every member and checks its CRC-32
        (``tc_bgzf_inflate``), finds and proves the record offsets (``tc_bam_index_records``) and parses the records
        (``tc_bam_records_to_reads``).  The result carries ``.ref_names``, ``.ref_lens``, ``.stats`` and ``.info``
        (records, unplaced records dropped, timings).  ``TcError`` / ``OSError`` for a file that does not decode.
        ``contig_ranges``: also ``.first_read``, where each reference's reads begin (``tc_bam_contig_ranges``, taken while the
        payload and the record offsets are still in the context's buffers); left None for an unsorted file.
        ``sort``: a file whose records are not sorted by (refID, pos) has its record offsets put in samtools' coordinate order
        on the device before the parse (``tc_bam_sort_records``); a sorted file is parsed as written.  ``.info`` then tells
        ``reordered`` and ``t_sort_s``.
        ``primers`` (a ``primers.PrimerScheme``): the primers are soft-clipped off the records before the sort
        (``tc_bam_clip_primers``), and the sort is implied: ``.info`` adds ``n_clipped_left``, ``n_clipped_right``,
        ``n_fully_clipped``, ``clipped_columns`` and ``t_clip_s``.  A primer chrom the header does not list is a ValueError."""
        import time

        from . import bamio

        t0 = time.perf_counter()
        m = bamio.map_bgzf(path)
        t1 = time.perf_counter()
        try:
            payload = C.c_void_p()
            self._generation += 1
            self._check(self._lib.tc_bgzf_inflate(self._h, m.file_ptr, m.file_bytes, m.blocks_ptr, m.n_blocks, m.payload_bytes,
                                                  C.byref(payload), stream))
            n_bytes, info = m.payload_bytes, {"bam_bytes": m.file_bytes, "payload_bytes": m.payload_bytes, "n_members": m.n_blocks}
        finally:
            m.release()
        t2 = time.perf_counter()
        n = 1 << 16
        while True:
            head = self.download(payload.value, min(n, n_bytes), np.uint8, stream).tobytes() if n_bytes else b""
            hdr = bamio.parse_bam_header(head, n_bytes)
            if hdr is not None:
                break
            n *= 4
        names, lens, first = hdr
        ref_len = np.asarray(lens if lens else [0], dtype=np.int32)
        rec, n_placed, n_records = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        self._check(self._lib.tc_bam_index_records(self._h, payload, n_bytes, first, len(lens), ref_len.ctypes.data, C.byref(rec),
                                                   C.byref(n_placed), C.byref(n_records), stream))
        t3 = time.perf_counter()
        info.update(n_records=int(n_records.value), n_dropped_unplaced=int(n_records.value - n_placed.value), t_map_s=t1 - t0,
                    t_inflate_s=t2 - t1, t_index_s=t3 - t2)
        return self._records_to_device(payload.value, n_bytes, rec.value, n_placed.value, names, lens, info, stream, contig_ranges,
                                       sort, primers, head[:first])

    def _records_to_device(self, payload, n_bytes: int, rec, n_reads: int, names, lens, info: dict, stream: int,
                           contig_ranges: bool, sort: bool, primers=None, header: bytes = b"") -> DeviceReads:
        """The tail every route shares: BAM records (payload and the offsets of the placed ones, host or device) -> primers
        clipped when given (``tc_bam_clip_primers``, which implies the sort), sorted when asked (``tc_bam_sort_records``),
        parsed (``tc_bam_records_to_reads``), the contig ranges when asked (``tc_bam_contig_ranges``) -> ``DeviceReads``
        with ``.ref_names``, ``.ref_lens``, ``.stats`` and ``info`` plus the clip's, the sort's and the parse's timings, and
        ``.records``: the BAM header (``header``) and the final records, what :meth:`write_bam` writes.  The caller has bumped
        ``_generation``."""
        import time

        payload, rec = C.c_void_p(payload), C.c_void_p(rec)
        if primers is not None:
            t = time.perf_counter()
            p, n_bytes, r, st = self.clip_primers(payload, n_bytes, rec, n_reads, names, primers, stream)
            payload, rec = C.c_void_p(p), C.c_void_p(r)
            info.update(n_clipped_left=int(st.n_left), n_clipped_right=int(st.n_right), n_fully_clipped=int(st.n_unmapped),
                        clipped_columns=int(st.n_columns), t_clip_s=time.perf_counter() - t)
            sort = True
        t0 = time.perf_counter()
        moved = C.c_int32(0)
        if sort:
            # a host payload is staged once here: the parse and the contig ranges go on from the device copy
            self._check(self._lib.tc_bam_sort_records(self._h, payload, n_bytes, rec, n_reads, len(lens), C.byref(payload),
                                                      C.byref(rec), C.byref(moved), stream))
        t1 = time.perf_counter()
        dev = TcReads()
        st = BamStats()
        self._check(self._lib.tc_bam_records_to_reads(self._h, payload, n_bytes, rec, n_reads, C.byref(dev), C.byref(st), stream))
        t2 = time.perf_counter()
        d = DeviceReads(dev, None, self, self._generation)
        d.stats = st
        d.ref_names, d.ref_lens = names, lens
        d.records = (header, payload.value, n_bytes, rec.value, n_reads)
        if contig_ranges and lens and not st.unsorted:
            d.first_read = np.zeros(len(lens) + 1, np.int32)
            self._check(self._lib.tc_bam_contig_ranges(self._h, payload, n_bytes, rec, n_reads, len(lens), _ptr(d.first_read),
                                                       stream))
        info.update(reordered=bool(moved.value), t_sort_s=t1 - t0, t_parse_s=t2 - t1)
        d.info = info
        return d

    def sam_file_to_device(self, path: str, stream: int = 0, contig_ranges: bool = False, sort: bool = False,
                           primers=None) -> DeviceReads:
        """A SAM file (an aligner's text output) to the flat read arrays in device memory, with the contract of
        :meth:`bam_file_to_device`: the host reads the ``@`` header lines (``bamio.read_sam_header``) and maps the file; the
        device turns every line into the BAM record ``samtools view -b`` would write for it (``tc_sam_to_bam_records``)
        and the BAM route's own steps follow (sort when asked, parse, contig ranges).  Lines with RNAME ``*`` are dropped
        and counted.  ``.info``: ``sam_bytes``, ``n_lines``, ``n_records``, ``n_dropped_unplaced``, ``reordered`` and the
        timings of each step (``t_map_s``, ``t_upload_s``, ``t_line_index_s``, ``t_convert_s``, ``t_sort_s``,
        ``t_parse_s``).  A malformed line is ``OSError("<path>: line <k>: <reason>")``.  ``primers``: as for
        :meth:`bam_file_to_device`."""
        import mmap
        import time

        from . import bamio

        t0 = time.perf_counter()
        names, lens, first_off, first_no = bamio.read_sam_header(path)
        raw = [n.encode(errors="surrogateescape") for n in names]
        name_off = np.zeros(len(raw) + 1, np.int64)
        name_off[1:] = np.cumsum([len(n) for n in raw])
        name_bytes = b"".join(raw) + b"\0"
        payload, rec = C.c_void_p(), C.c_void_p()
        n_payload, n_placed, n_records, n_lines = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
        err = (C.c_int64 * 2)()
        steps = (C.c_double * 3)()
        with open(path, "rb") as fh:
            size = os.fstat(fh.fileno()).st_size
            mm = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) if size > first_off else None
            text = None
            try:
                text = np.frombuffer(mm, np.uint8) if mm is not None else None
                t1 = time.perf_counter()
                self._generation += 1
                rc = self._lib.tc_sam_to_bam_records(self._h, None if text is None else text.ctypes.data, size, first_off, first_no,
                                                     len(raw), name_bytes, name_off.ctypes.data, C.byref(payload), C.byref(n_payload),
                                                     C.byref(rec), C.byref(n_placed), C.byref(n_records), C.byref(n_lines), err,
                                                     steps, stream)
            finally:
                del text
                if mm is not None:
                    mm.close()
        if rc != 0:
            msg = self._lib.tc_last_error(self._h).decode()
            if err[0] > 0:
                raise OSError(f"{path}: {msg}")
            raise TcError(rc, msg)
        info = {"sam_bytes": size, "n_lines": int(n_lines.value), "n_records": int(n_records.value),
                "n_dropped_unplaced": int(n_records.value - n_placed.value), "t_map_s": t1 - t0, "t_upload_s": steps[0],
                "t_line_index_s": steps[1], "t_convert_s": steps[2]}
        return self._records_to_device(payload.value, int(n_payload.value), rec.value, int(n_placed.value), names, lens, info,
                                       stream, contig_ranges, sort, primers, bamio.sam_bam_header(path, names, lens, first_off))

    def write_bam(self, reads: DeviceReads, path: str, stream: int = 0) -> dict:
        """Write the records ``reads`` were parsed from as a BAM file (``tc_bam_write_records``: BGZF members compressed on the
        GPU).  The file holds the decode's placed records in the order the passes read them (clipped, sorted), byte for byte
        except ``bin``, which is recomputed; the header is the input's with ``@HD ... SO:coordinate`` (DESIGN §4).  The file is
        written beside ``path`` and renamed onto it, so a failure leaves no partial file there.  ``reads`` stay valid.
        Returns, and adds to ``reads.info``: ``bam_out_bytes``, ``n_out_members``, ``n_written``, ``t_write_s`` and
        ``t_device_ms`` (CUDA-event milliseconds of the gather, the compression and the compaction)."""
        import time

        from . import bamio

        if not isinstance(reads, DeviceReads) or reads.ctx is not self:
            raise TypeError("write_bam writes the device reads of this context")
        if reads.records is None:
            raise ValueError("these device reads were uploaded from a host ReadBatch, which holds no BAM records: only reads "
                             "decoded from a file or payload (bam_file_to_device, sam_file_to_device, bam_to_device) can be written")
        if reads.generation != self._generation:
            raise RuntimeError("these device reads are stale: the context has decoded or staged another batch since, and their "
                               "records are gone")
        t0 = time.perf_counter()
        header, payload, n_bytes, rec, n = reads.records
        header = bamio.coordinate_header(header)
        img, nb, nm = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        t_ms = (C.c_float * 3)()
        self._check(self._lib.tc_bam_write_records(self._h, header, len(header), payload, n_bytes, rec, n, C.byref(img), C.byref(nb),
                                                   C.byref(nm), t_ms, stream))
        data = self.download(img.value, nb.value, np.uint8, stream)
        tmp = f"{path}.{os.getpid()}.{threading.get_ident()}.tmp"
        try:
            with open(tmp, "xb") as fh:
                fh.write(data.data)
            os.replace(tmp, path)
        except BaseException:
            if os.path.exists(tmp):
                os.unlink(tmp)
            raise
        out = {"bam_out_bytes": int(nb.value), "n_out_members": int(nm.value), "n_written": int(n),
               "t_write_s": time.perf_counter() - t0, "t_device_ms": float(t_ms[0] + t_ms[1] + t_ms[2])}
        reads.info.update(out)
        return out

    def reads_to_contig_coords(self, reads: DeviceReads, ref_lens, first_read, names=None, stream: int = 0) -> np.ndarray:
        """Move device-resident reads to the global columns of a multi-reference pass, in place (``tc_reads_to_contig_coords``):
        reference k's reads (``first_read[k]`` .. ``first_read[k+1]-1``) shift by the sum of the lengths before it.  Returns
        those boundaries (int32[n_ref + 1]).  A batch moves once: a second call on it raises.  A read outside its reference
        is ``TcError`` (TC_ERR_RANGE) naming the reference (``names``); the batch is unusable afterwards."""
        if not isinstance(reads, DeviceReads) or reads.ctx is not self:
            raise TypeError("reads_to_contig_coords moves the device reads of this context (upload / bam_file_to_device)")
        if reads.contig_start is not None:
            raise RuntimeError("these device reads sit in contig coordinates already")
        rs = self._reads_struct(reads)
        lens = np.ascontiguousarray(ref_lens, dtype=np.int32) if not hasattr(ref_lens, "data_ptr") else ref_lens
        first = np.ascontiguousarray(first_read, dtype=np.int32) if not hasattr(first_read, "data_ptr") else first_read
        n_ref = int(lens.shape[0])
        start = np.zeros(n_ref + 1, np.int32)
        rc = self._lib.tc_reads_to_contig_coords(self._h, C.byref(rs), n_ref, _ptr(lens), _ptr(first), _ptr(start), stream)
        if rc != 0:
            msg = self._lib.tc_last_error(self._h).decode()
            if rc == -7:
                reads.generation = -1           # partly moved: stale from now on
                import re

                m = re.search(r"reference (\d+)", msg)
                if m and names is not None and int(m.group(1)) < len(names):
                    msg = msg.replace(m.group(0), f"{m.group(0)} ({names[int(m.group(1))]!r})", 1)
            raise TcError(rc, msg)
        reads.contig_start = start
        return start

    # ------------------------------------------------------------------ (1) pileup
    def pileup_counts(self, reads, ref_len: int, params: PileupParams | None = None, out=None, stream: int = 0):
        """int32[8][ref_len] count table (rows coverage,A,T,C,G,X,I,pad).  ``out`` may be a numpy
        array or a torch CUDA int32 tensor; default: a new numpy array."""
        params = params or buildindex_params()
        if out is None:
            out = np.empty((TC_NROWS, ref_len), dtype=np.int32)
        rs = self._reads_struct(reads)
        self._check(self._lib.tc_pileup_counts(self._h, C.byref(rs), int(ref_len), C.byref(params), _ptr(out), stream))
        return out

    def allreduce_counts(self, counts_dev, comm, stream: int = 0) -> None:
        """Sum a device count table over the ranks of ``comm`` (sharding.NcclComm) in place."""
        self._check(self._lib.tc_allreduce_counts(self._h, _ptr(counts_dev), int(counts_dev.numel()), comm.handle, stream))

    def pileup_counts_allreduce(self, reads, ref_len: int, params: PileupParams, out, comm, stream: int = 0):
        """This rank's shard piled up into the torch CUDA int32 tensor ``out`` and summed over the ranks of ``comm`` in one
        enqueue (tc_pileup_counts_allreduce): no synchronisation between the two, a CUDA graph from the second call on."""
        rs = self._reads_struct(reads)
        self._check(self._lib.tc_pileup_counts_allreduce(self._h, C.byref(rs), int(ref_len), C.byref(params), _ptr(out), comm.handle, stream))
        return out

    def pileup_counts_allreduce_enqueue(self, reads, ref_len: int, params: PileupParams, out, comm, stream: int = 0) -> int:
        """First half of ``pileup_counts_allreduce``: returns a ticket as soon as the pass is enqueued.  Two passes may be in
        flight (each with its own ``out``); ``reads`` / ``out`` stay untouched until ``pileup_counts_allreduce_finish``."""
        rs = self._reads_struct(reads)
        t = C.c_int32(-1)
        self._check(self._lib.tc_pileup_counts_allreduce_enqueue(self._h, C.byref(rs), int(ref_len), C.byref(params), _ptr(out), comm.handle,
                                                                 stream, C.byref(t)))
        self._rr_keep = getattr(self, "_rr_keep", {})
        self._rr_keep[t.value] = (reads, out, params, rs)
        return int(t.value)

    def pileup_counts_allreduce_finish(self, ticket: int) -> None:
        try:
            self._check(self._lib.tc_pileup_counts_allreduce_finish(self._h, int(ticket)))
        finally:
            getattr(self, "_rr_keep", {}).pop(ticket, None)

    # ------------------------------------------------------------------ (3) depth
    def depth(self, reads, ref_len: int, params: PileupParams | None = None, out=None, stream: int = 0):
        params = params or buildindex_params()
        if out is None:
            out = np.empty(ref_len, dtype=np.int32)
        rs = self._reads_struct(reads)
        self._check(self._lib.tc_depth(self._h, C.byref(rs), int(ref_len), C.byref(params), _ptr(out), stream))
        return out

    # ------------------------------------------------------------------ (4) call
    def call(self, counts, ref_len: int, mincov: int, include_ambig: bool, stream: int = 0, maxdist: float = 10.0,
             minority_del_pct: float = 15.0, insert_pct: float = 55.0) -> CallResult:
        L = int(ref_len)
        res, t, counts = _call_buffers(counts, L)
        p = CallParams(int(mincov), int(bool(include_ambig)), maxdist, minority_del_pct, insert_pct)
        self._check(self._lib.tc_call(self._h, _ptr(counts), L, C.byref(p), C.byref(t), stream))
        return res

    def call_device(self, counts, ref_len: int, mincov: int, include_ambig: bool, table: CallTable, stream: int = 0,
                    maxdist: float = 10.0, minority_del_pct: float = 15.0, insert_pct: float = 55.0) -> None:
        """tc_call with caller-provided (device) output pointers; asynchronous."""
        p = CallParams(int(mincov), int(bool(include_ambig)), maxdist, minority_del_pct, insert_pct)
        self._check(self._lib.tc_call(self._h, _ptr(counts), int(ref_len), C.byref(p), C.byref(table), stream))

    def call_contigs(self, counts, contig_start, mincov: int, include_ambig: bool, stream: int = 0, maxdist: float = 10.0,
                     minority_del_pct: float = 15.0, insert_pct: float = 55.0) -> CallResult:
        """``tc_call_contigs``: the call table of a multi-reference count table [8][total] whose references start at
        ``contig_start`` (n + 1 boundaries): X-runs stop at their reference's end."""
        cs = np.ascontiguousarray(contig_start, dtype=np.int32)
        n, L = int(cs.shape[0]) - 1, int(cs[-1])
        res, t, counts = _call_buffers(counts, L)
        p = CallParams(int(mincov), int(bool(include_ambig)), maxdist, minority_del_pct, insert_pct)
        self._check(self._lib.tc_call_contigs(self._h, _ptr(counts), L, n, _ptr(cs), C.byref(p), C.byref(t), stream))
        return res

    def is_ambiguous(self, letters: np.ndarray, cnts: np.ndarray, cov: np.ndarray, maxdist: float = 10.0, stream: int = 0) -> np.ndarray:
        letters = np.ascontiguousarray(letters, dtype=np.uint8)
        cnts = np.ascontiguousarray(cnts, dtype=np.int32)
        cov = np.ascontiguousarray(cov, dtype=np.int32)
        n = cov.shape[0]
        out = np.zeros(n, np.uint8)
        self._check(self._lib.tc_is_ambiguous(self._h, _ptr(letters), _ptr(cnts), _ptr(cov), n, maxdist, _ptr(out), stream))
        return out

    # ------------------------------------------------------------------ (2) insertions
    def list_insert_candidates(self, flags, ref_len: int, cap: int | None = None, stream: int = 0) -> np.ndarray:
        """1-based positions with TC_CF_INS_CANDIDATE.  ``stream`` must be the stream the producer of a device ``flags`` array
        (``call_device``) was enqueued on — or that work must have been synchronised."""
        cap = int(ref_len) if cap is None else cap
        out = np.empty(max(cap, 1), np.int32)
        n = C.c_int32(0)
        self._check(self._lib.tc_list_insert_candidates(self._h, _ptr(flags), int(ref_len), _ptr(out), cap, C.byref(n), stream))
        return out[: n.value].copy()

    def extract_inserts(self, reads, ref_len: int, positions, params: PileupParams | None = None, stream: int = 0):
        """ExtractInserts for the given 1-based positions.  Returns a list of dicts with the modal
        upper-cased string of each column (``None`` when pysam would have returned ``""``).

        Host-resident SEQ / QUAL / CIGAR arrays travel to the device only for the reads that can reach a
        candidate column (tc_extract_inserts stages them range by range; this pass is the only one that
        needs QUAL, 8x the size of the packed bases)."""
        params = params or extractinserts_params()
        pos = np.ascontiguousarray(positions, dtype=np.int32)
        if pos.shape[0] == 0:
            return []
        return self._extract_inserts_raw(reads, ref_len, pos, params, stream)

    @staticmethod
    def _insert_dicts(calls, n: int, bases: np.ndarray):
        out = []
        for c in calls[:n]:
            if c.n_entries == 0:
                out.append({"pos": c.pos, "n_entries": 0, "string": None, "mode_count": 0, "first_read": -1})
                continue
            s = chr(c.head)
            if c.indel > 0:
                s += f"+{c.indel}" + bytes(bases[c.bases_off:c.bases_off + c.indel]).decode("ascii")
            elif c.indel < 0:
                s += f"-{-c.indel}" + "N" * (-c.indel)
            out.append({"pos": c.pos, "n_entries": c.n_entries, "string": s, "mode_count": c.mode_count,
                        "first_read": c.first_read})
        return out

    def pileup_call_inserts(self, reads, ref_len: int, mincov: int, include_ambig: bool, counts_dev, table: CallTable,
                            pileup: PileupParams | None = None, inserts: PileupParams | None = None, stream: int = 0,
                            maxdist: float = 10.0, minority_del_pct: float = 15.0, insert_pct: float = 55.0, cap: int = 256):
        """One enqueue per sample (tc_pileup_call_inserts): pileup into ``counts_dev``, the call table into ``table``
        (device pointers), and the ExtractInserts result of every insertion candidate — one synchronisation.
        Returns the same list of dicts as :meth:`extract_inserts` for :meth:`list_insert_candidates`' positions."""
        pileup = pileup or buildindex_params()
        inserts = inserts or extractinserts_params()
        cp = CallParams(int(mincov), int(bool(include_ambig)), maxdist, minority_del_pct, insert_pct)
        rs = self._reads_struct(reads)
        bcap = 1 << 16
        while True:
            calls = (InsertCall * max(cap, 1))()
            bases = np.zeros(bcap, np.uint8)
            n = C.c_int32(0)
            rc = self._lib.tc_pileup_call_inserts(self._h, C.byref(rs), int(ref_len), C.byref(pileup), C.byref(cp), C.byref(inserts),
                                                  _ptr(counts_dev), C.byref(table), calls, cap, C.byref(n), _ptr(bases), bcap, stream)
            if rc == -8 and n.value > cap:          # more candidates than the caller made room for
                cap = n.value
                continue
            if rc == -8 and bcap < (1 << 30) and n.value <= cap and "bases buffer" in self._lib.tc_last_error(self._h).decode():
                bcap *= 16
                continue
            self._check(rc)
            return self._insert_dicts(calls, n.value, bases)

    def sample_enqueue(self, reads, ref_len: int, mincov: int, include_ambig: bool, counts_dev, table: CallTable,
                       pileup: PileupParams | None = None, inserts: PileupParams | None = None, stream: int = 0,
                       maxdist: float = 10.0, minority_del_pct: float = 15.0, insert_pct: float = 55.0) -> int:
        """First half of :meth:`pileup_call_inserts` (tc_sample_enqueue): returns a ticket as soon as the sample's work is
        enqueued.  At most two samples in flight per context, on one stream; their buffers stay valid until
        :meth:`sample_finish`."""
        pileup = pileup or buildindex_params()
        inserts = inserts or extractinserts_params()
        cp = CallParams(int(mincov), int(bool(include_ambig)), maxdist, minority_del_pct, insert_pct)
        rs = self._reads_struct(reads)
        t = C.c_int32(-1)
        self._check(self._lib.tc_sample_enqueue(self._h, C.byref(rs), int(ref_len), C.byref(pileup), C.byref(cp), C.byref(inserts),
                                                _ptr(counts_dev), C.byref(table), stream, C.byref(t)))
        return int(t.value)

    def sample_finish(self, ticket: int, cap: int = 256):
        """Second half (tc_sample_finish): waits for that sample only and returns its insertion calls."""
        buf = getattr(self, "_sample_bufs", None)
        if buf is None or buf[2] < cap:
            buf = self._sample_bufs = ((InsertCall * max(cap, 1))(), np.zeros(1 << 16, np.uint8), cap)
        calls, bases, _ = buf
        n = C.c_int32(0)
        self._check(self._lib.tc_sample_finish(self._h, int(ticket), calls, cap, C.byref(n), _ptr(bases), bases.shape[0]))
        return self._insert_dicts(calls, n.value, bases)

    def _extract_inserts_raw(self, reads, ref_len: int, pos: np.ndarray, params: PileupParams, stream: int = 0):
        n = int(pos.shape[0])
        calls = (InsertCall * n)()
        cap = 1 << 16
        rs = self._reads_struct(reads)
        while True:
            bases = np.zeros(cap, np.uint8)
            rc = self._lib.tc_extract_inserts(self._h, C.byref(rs), int(ref_len), _ptr(pos), n, C.byref(params), calls,
                                              _ptr(bases), cap, stream)
            if rc == -8 and cap < (1 << 30):
                cap *= 16
                continue
            self._check(rc)
            return self._insert_dicts(calls, n, bases)


_default_ctx: dict[int, Context] = {}
_ctx_lock = threading.Lock()


def default_context(device: int = -1) -> Context:
    """A lazily created per-device context shared by the module-level API (BuildIndex & co)."""
    with _ctx_lock:
        c = _default_ctx.get(device)
        if c is None:
            c = Context(device)
            _default_ctx[device] = c
        return c
