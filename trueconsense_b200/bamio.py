"""BAM <-> flat read arrays (ctypes over libtchost.so, csrc/host/bamio.c).

This is the decode half of what ``pysam.AlignmentFile`` does for
TrueConsense/indexing.py:96; pysam/htslib are not installed in this image (SURVEY.md §0), so
the repo carries its own BGZF/BAM reader and writer.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build
from .reads import ReadBatch


class TcHostReads(C.Structure):
    """ctypes mirror of ``tc_hostreads_t`` (include/tc_host.h)."""

    _fields_ = [
        ("n_reads", C.c_int64), ("n_seq_words", C.c_int64), ("n_cigar_ops", C.c_int64),
        ("pos", C.POINTER(C.c_int32)), ("flag", C.POINTER(C.c_uint16)), ("mapq", C.POINTER(C.c_uint8)),
        ("l_seq", C.POINTER(C.c_int32)), ("seq_off", C.POINTER(C.c_uint32)), ("cigar_off", C.POINTER(C.c_uint32)),
        ("seq4", C.POINTER(C.c_uint32)), ("qual", C.POINTER(C.c_uint8)), ("cigar", C.POINTER(C.c_uint32)),
        ("qname_hash", C.POINTER(C.c_uint64)), ("mpos", C.POINTER(C.c_int32)), ("isize", C.POINTER(C.c_int32)),
        ("tid", C.POINTER(C.c_int32)), ("mtid", C.POINTER(C.c_int32)),
        ("n_ref", C.c_int32), ("ref_len", C.POINTER(C.c_int32)), ("ref_names", C.POINTER(C.c_char)),
        ("ref_names_len", C.c_int64),
        ("n_records", C.c_int64), ("n_dropped_unplaced", C.c_int64), ("aligned_bases", C.c_int64),
        ("sorted", C.c_int32), ("max_ref_span", C.c_int32),
        ("t_inflate_s", C.c_double), ("t_parse_s", C.c_double),
    ]


class TcBamPayload(C.Structure):
    """ctypes mirror of ``tc_bampayload_t`` (include/tc_host.h)."""

    _fields_ = [
        ("payload", C.POINTER(C.c_uint8)), ("n_bytes", C.c_int64), ("rec_off", C.POINTER(C.c_int64)), ("n_reads", C.c_int64),
        ("n_records", C.c_int64), ("n_dropped_unplaced", C.c_int64), ("n_ref", C.c_int32), ("ref_len", C.POINTER(C.c_int32)),
        ("ref_names", C.POINTER(C.c_char)), ("ref_names_len", C.c_int64), ("t_inflate_s", C.c_double), ("t_index_s", C.c_double),
    ]


class BamPayload:
    """A BAM's uncompressed payload and the offsets of its placed records (host memory, freed with the object): the host half
    of the decode when the records are parsed on the GPU (``gpu.Context.bam_to_device``)."""

    def __init__(self, st: TcBamPayload, lib: C.CDLL):
        self._st, self._lib = st, lib
        self.n_reads = int(st.n_reads)
        self.n_bytes = int(st.n_bytes)
        names = []
        if st.n_ref > 0 and st.ref_names_len > 0:
            names = [x.decode() for x in C.string_at(st.ref_names, st.ref_names_len).split(b"\0")[: st.n_ref]]
        self.ref_names = names
        self.ref_lens = [int(st.ref_len[i]) for i in range(st.n_ref)] if st.n_ref > 0 else []
        self.info = {"n_records": int(st.n_records), "n_dropped_unplaced": int(st.n_dropped_unplaced),
                     "t_inflate_s": float(st.t_inflate_s), "t_index_s": float(st.t_index_s)}

    @property
    def payload_ptr(self) -> int:
        return C.cast(self._st.payload, C.c_void_p).value or 0

    @property
    def rec_off_ptr(self) -> int:
        return C.cast(self._st.rec_off, C.c_void_p).value or 0

    def release(self) -> None:
        """Free the payload and the offsets (the header fields read in __init__ stay)."""
        if self._st is not None:
            self._lib.tc_bampayload_free(C.byref(self._st))
            self._st = None
            self.n_bytes = 0

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class TcBgzfBlock(C.Structure):
    """ctypes mirror of ``tc_bgzf_block_t``: the raw DEFLATE stream file[coff : coff + csize] inflates to payload[uoff : uoff + usize]."""

    _fields_ = [("coff", C.c_int64), ("csize", C.c_int32), ("usize", C.c_int32), ("uoff", C.c_int64)]


class TcBgzfMap(C.Structure):
    """ctypes mirror of ``tc_bgzf_map_t`` (include/tc_host.h)."""

    _fields_ = [("file", C.POINTER(C.c_uint8)), ("file_bytes", C.c_int64), ("blocks", C.POINTER(TcBgzfBlock)), ("n_blocks", C.c_int64),
                ("payload_bytes", C.c_int64)]


class BgzfMap:
    """A BAM file mapped read-only plus the index of its BGZF members (``tc_bgzf_map``): what the GPU needs to inflate it
    (``gpu.Context.bam_file_to_device``).  The host has read one header per member, nothing else."""

    def __init__(self, st: TcBgzfMap, lib: C.CDLL):
        self._st, self._lib = st, lib
        self.file_bytes = int(st.file_bytes)
        self.n_blocks = int(st.n_blocks)
        self.payload_bytes = int(st.payload_bytes)

    @property
    def file_ptr(self) -> int:
        return C.cast(self._st.file, C.c_void_p).value or 0

    @property
    def blocks_ptr(self) -> int:
        return C.cast(self._st.blocks, C.c_void_p).value or 0

    def blocks(self) -> np.ndarray:
        """The member index as a structured array (a copy)."""
        dt = np.dtype([("coff", "<i8"), ("csize", "<i4"), ("usize", "<i4"), ("uoff", "<i8")])
        return np.frombuffer(C.string_at(self._st.blocks, self.n_blocks * dt.itemsize), dtype=dt).copy()

    def release(self) -> None:
        if self._st is not None:
            self._lib.tc_bgzf_unmap(C.byref(self._st))
            self._st = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


def parse_bam_header(buf: bytes, n_total: int):
    """(reference names, reference lengths, payload offset of the first record) from the first bytes of a BAM's payload;
    None when ``buf`` ends inside the header (and the payload is longer: fetch more)."""
    import struct

    def short():
        if len(buf) >= n_total:
            raise OSError("truncated BAM header")
        return None

    if len(buf) < 12:
        if n_total < 12:
            raise OSError("missing BAM magic")
        return short()
    if buf[:4] != b"BAM\1":
        raise OSError("missing BAM magic")
    l_text = struct.unpack_from("<i", buf, 4)[0]
    if l_text < 0 or 8 + l_text + 4 > n_total:
        raise OSError("truncated BAM header")
    p = 8 + l_text
    if p + 4 > len(buf):
        return short()
    n_ref = struct.unpack_from("<i", buf, p)[0]
    p += 4
    if n_ref < 0 or n_ref * 8 > n_total - p:
        raise OSError(f"bad BAM reference count {n_ref}")
    names, lens = [], []
    for _ in range(n_ref):
        if p + 4 > len(buf):
            return short()
        l_name = struct.unpack_from("<i", buf, p)[0]
        p += 4
        if l_name < 0 or p + l_name + 4 > n_total:
            raise OSError("truncated BAM reference list")
        if p + l_name + 4 > len(buf):
            return short()
        names.append(buf[p:p + l_name].split(b"\0")[0].decode(errors="replace"))
        p += l_name
        lens.append(struct.unpack_from("<i", buf, p)[0])
        p += 4
    return names, lens, p


def read_bam_header(path: str):
    """(reference names, reference lengths) of a BAM: only the members holding the header are inflated."""
    import gzip

    n = 1 << 16
    size = os.path.getsize(path)
    while True:
        with gzip.open(path, "rb") as fh:
            buf = fh.read(n)
        got = parse_bam_header(buf, len(buf) if len(buf) < n else max(n + 1, 64 * size))
        if got is not None:
            return got[0], got[1]
        n *= 4


def read_sam_header(path: str):
    """(reference names, reference lengths, byte offset of the first record, its 1-based line number) of a SAM file: the
    ``@`` lines at its start are read, no record.  ``@SQ`` lines give the references (``SN``, ``LN``) in order; ``@HD``,
    ``@RG``, ``@PG``, ``@CO`` and any other header line are skipped.  ``OSError`` names the line of an ``@SQ`` without
    ``SN``, with a name seen before, or without an ``LN`` in 1..2^31-1.  Names keep their bytes (undecodable ones as
    surrogates: ``name.encode(errors="surrogateescape")`` gives them back)."""
    names, lens, seen = [], [], set()
    off, line_no = 0, 1
    with open(path, "rb") as fh:
        while fh.peek(1)[:1] == b"@":
            line = fh.readline()
            if line[:4] in (b"@SQ\t", b"@SQ\n", b"@SQ"):
                tags = {}
                for f in line.rstrip(b"\n").split(b"\t")[1:]:
                    tags.setdefault(f[:3], f[3:])
                sn, ln = tags.get(b"SN:"), tags.get(b"LN:")
                if not sn:
                    raise OSError(f"{path}: line {line_no}: @SQ line without a reference name (SN)")
                name = sn.decode(errors="surrogateescape")
                if name in seen:
                    raise OSError(f"{path}: line {line_no}: reference {name!r} is listed twice")
                if ln is None or not ln.isdigit() or not 1 <= int(ln) <= 0x7FFFFFFF:
                    raise OSError(f"{path}: line {line_no}: reference {name!r} needs a length (LN) in 1..2147483647")
                seen.add(name)
                names.append(name)
                lens.append(int(ln))
            off += len(line)
            line_no += 1
    return names, lens, off, line_no


def sam_bam_header(path: str, names, lens, first_off: int) -> bytes:
    """The BAM header of a SAM file: its ``@`` lines (the file's first ``first_off`` bytes) as the text, then the ``@SQ``
    references ``names`` / ``lens`` (``read_sam_header``)."""
    import struct

    with open(path, "rb") as fh:
        text = fh.read(first_off)
    refs = b"".join(struct.pack("<i", len(r) + 1) + r + b"\0" + struct.pack("<i", ln)
                    for r, ln in zip((n.encode(errors="surrogateescape") for n in names), lens))
    return b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(names)) + refs


HD_COORDINATE = b"@HD\tVN:1.6\tSO:coordinate"


def coordinate_header(header: bytes) -> bytes:
    """A BAM header (magic to the last reference) whose text says the records are in coordinate order: a first ``@HD``
    line has its ``SO:`` value replaced (or ``\\tSO:coordinate`` added); without one, ``@HD\\tVN:1.6\\tSO:coordinate`` is
    inserted as the first line.  A header that says ``SO:coordinate`` already comes back as it is."""
    import struct

    l_text = struct.unpack_from("<i", header, 4)[0]
    text, rest = header[8:8 + l_text], header[8 + l_text:]
    if text.startswith(b"@HD\t") or text.startswith(b"@HD\n") or text == b"@HD":
        end = text.find(b"\n")
        end = len(text) if end < 0 else end
        fields = text[:end].split(b"\t")
        so = [k for k, f in enumerate(fields) if f.startswith(b"SO:")]
        if so:
            if fields[so[0]] == b"SO:coordinate":
                return header
            fields[so[0]] = b"SO:coordinate"
        else:
            fields.append(b"SO:coordinate")
        text = b"\t".join(fields) + text[end:]
    else:
        text = HD_COORDINATE + b"\n" + text
    return b"BAM\1" + struct.pack("<i", len(text)) + text + rest


_lib = None


def host_lib() -> C.CDLL:
    """Load (building if necessary) libtchost.so."""
    global _lib
    if _lib is None:
        path = build.HOST_LIB
        if not os.path.exists(path) or os.environ.get("TC_REBUILD"):
            build.build_host()
        lib = C.CDLL(path)
        lib.tc_bam_read.argtypes = [C.c_char_p, C.c_int, C.POINTER(TcHostReads), C.c_char_p, C.c_int]
        lib.tc_bam_read.restype = C.c_int
        lib.tc_hostreads_free.argtypes = [C.POINTER(TcHostReads)]
        lib.tc_hostreads_free.restype = None
        lib.tc_bam_write.argtypes = [C.c_char_p, C.POINTER(TcHostReads), C.c_char_p, C.c_int32, C.c_int,
                                     C.c_char_p, C.c_int]
        lib.tc_bam_write.restype = C.c_int
        lib.tc_bam_payload.argtypes = [C.c_char_p, C.c_int, C.POINTER(TcBamPayload), C.c_char_p, C.c_int]
        lib.tc_bam_payload.restype = C.c_int
        lib.tc_bampayload_free.argtypes = [C.POINTER(TcBamPayload)]
        lib.tc_bampayload_free.restype = None
        lib.tc_bgzf_map.argtypes = [C.c_char_p, C.POINTER(TcBgzfMap), C.c_char_p, C.c_int]
        lib.tc_bgzf_map.restype = C.c_int
        lib.tc_bgzf_unmap.argtypes = [C.POINTER(TcBgzfMap)]
        lib.tc_bgzf_unmap.restype = None
        lib.tc_seq2_pack.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                     C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.c_int64), C.c_int]
        lib.tc_seq2_pack.restype = C.c_int
        lib.tc_host_free.argtypes = [C.c_void_p]
        lib.tc_host_free.restype = None
        _lib = lib
    return _lib


class _Owner:
    """Frees the C-owned arrays when the last numpy view onto them is gone."""

    def __init__(self, hr: TcHostReads, lib: C.CDLL):
        self.hr = hr
        self._free = lib.tc_hostreads_free

    def __del__(self):
        try:
            self._free(C.byref(self.hr))
        except Exception:
            pass


class _CMem:
    """Array-interface carrier: ``np.asarray(_CMem(...))`` keeps this object — and through it
    the owner of the memory — alive as the array's base."""

    def __init__(self, addr: int, n: int, dtype, owner: _Owner):
        self.__array_interface__ = {"data": (addr, False), "shape": (n,), "typestr": np.dtype(dtype).str, "version": 3}
        self._owner = owner


def _wrap(ptr, n, dtype, owner):
    addr = C.cast(ptr, C.c_void_p).value
    if n <= 0 or not addr:
        return np.zeros(0, dtype=dtype)
    return np.asarray(_CMem(addr, n, dtype, owner))


def batch_from_hostreads(hr: TcHostReads, lib: C.CDLL) -> ReadBatch:
    """Zero-copy numpy views over the C-owned arrays; freed when the batch is collected."""
    n = int(hr.n_reads)
    nw = int(hr.n_seq_words)
    nc = int(hr.n_cigar_ops)
    names = []
    if hr.n_ref > 0 and hr.ref_names_len > 0:
        raw = C.string_at(hr.ref_names, hr.ref_names_len)
        names = [s.decode() for s in raw.split(b"\0")[: hr.n_ref]]
    lens = [int(hr.ref_len[i]) for i in range(hr.n_ref)] if hr.n_ref > 0 else []
    own = _Owner(hr, lib)
    b = ReadBatch(
        pos=_wrap(hr.pos, n, np.int32, own), flag=_wrap(hr.flag, n, np.uint16, own), mapq=_wrap(hr.mapq, n, np.uint8, own),
        l_seq=_wrap(hr.l_seq, n, np.int32, own), seq_off=_wrap(hr.seq_off, n + 1, np.uint32, own),
        cigar_off=_wrap(hr.cigar_off, n + 1, np.uint32, own), seq4=_wrap(hr.seq4, nw, np.uint32, own),
        qual=_wrap(hr.qual, 8 * nw, np.uint8, own), cigar=_wrap(hr.cigar, nc, np.uint32, own),
        qname_hash=_wrap(hr.qname_hash, n, np.uint64, own), mpos=_wrap(hr.mpos, n, np.int32, own),
        isize=_wrap(hr.isize, n, np.int32, own), tid=_wrap(hr.tid, n, np.int32, own), mtid=_wrap(hr.mtid, n, np.int32, own),
        ref_names=names, ref_lens=lens, aligned_bases=int(hr.aligned_bases), max_ref_span=int(hr.max_ref_span),
        sorted=bool(hr.sorted),
        info={"n_records": int(hr.n_records), "n_dropped_unplaced": int(hr.n_dropped_unplaced),
              "t_inflate_s": float(hr.t_inflate_s), "t_parse_s": float(hr.t_parse_s)},
    )
    b._owner = own
    return b


def read_bam(path: str, threads: int = 0, compact: bool = False) -> ReadBatch:
    """Decode a BAM into flat arrays (all placed records, file order).  ``compact``: also attach the transport forms every
    later upload of the batch moves instead of the full arrays (16-bit CIGARs, 2-bit SEQ + exception words)."""
    lib = host_lib()
    hr = TcHostReads()
    err = C.create_string_buffer(512)
    rc = lib.tc_bam_read(os.fsencode(path), threads, C.byref(hr), err, len(err))
    if rc != 0:
        raise OSError(f"tc_bam_read({path!r}) failed ({rc}): {err.value.decode(errors='replace')}")
    batch = batch_from_hostreads(hr, lib)
    return batch.with_cigar16().with_seq2() if compact else batch


def read_bam_payload(path: str, threads: int = 0) -> BamPayload:
    """Inflate a BAM on the host's cores and index its placed records; the records themselves are parsed on the device
    (``gpu.Context.bam_to_device``)."""
    lib = host_lib()
    st = TcBamPayload()
    err = C.create_string_buffer(512)
    rc = lib.tc_bam_payload(os.fsencode(path), threads, C.byref(st), err, len(err))
    if rc != 0:
        raise OSError(f"tc_bam_payload({path!r}) failed ({rc}): {err.value.decode(errors='replace')}")
    return BamPayload(st, lib)


def map_bgzf(path: str) -> BgzfMap:
    """Map a BAM and index its BGZF members (``tc_bgzf_map``); the device inflates them (``gpu.Context.bam_file_to_device``)."""
    lib = host_lib()
    st = TcBgzfMap()
    err = C.create_string_buffer(512)
    rc = lib.tc_bgzf_map(os.fsencode(path), C.byref(st), err, len(err))
    if rc != 0:
        raise OSError(f"tc_bgzf_map({path!r}) failed ({rc}): {err.value.decode(errors='replace')}")
    return BgzfMap(st, lib)


def hostreads_struct(batch: ReadBatch) -> TcHostReads:
    hr = TcHostReads()
    hr.n_reads = batch.n_reads
    hr.n_seq_words = int(batch.seq4.shape[0])
    hr.n_cigar_ops = int(batch.cigar.shape[0])

    def p(a, ct):
        return None if a is None else a.ctypes.data_as(C.POINTER(ct))

    hr.pos = p(batch.pos, C.c_int32); hr.flag = p(batch.flag, C.c_uint16); hr.mapq = p(batch.mapq, C.c_uint8)
    hr.l_seq = p(batch.l_seq, C.c_int32); hr.seq_off = p(batch.seq_off, C.c_uint32)
    hr.cigar_off = p(batch.cigar_off, C.c_uint32); hr.seq4 = p(batch.seq4, C.c_uint32)
    hr.qual = p(batch.qual, C.c_uint8); hr.cigar = p(batch.cigar, C.c_uint32)
    qh = batch.qname_hash if batch.qname_hash is not None else np.arange(batch.n_reads, dtype=np.uint64)
    hr._keep = qh
    hr.qname_hash = p(qh, C.c_uint64)
    hr.mpos = p(batch.mpos, C.c_int32); hr.isize = p(batch.isize, C.c_int32)
    hr.tid = p(batch.tid, C.c_int32); hr.mtid = p(batch.mtid, C.c_int32)
    return hr


def write_bam(path: str, batch: ReadBatch, ref_name: str = "ref", ref_len: int | None = None, level: int = 1) -> None:
    """Write a batch as a coordinate-sorted single-contig BAM (read names are ``q<hash>``)."""
    lib = host_lib()
    if ref_len is None:
        ref_len = batch.ref_lens[0]
    hr = hostreads_struct(batch)
    err = C.create_string_buffer(512)
    rc = lib.tc_bam_write(os.fsencode(path), C.byref(hr), ref_name.encode(), int(ref_len), int(level), err, len(err))
    if rc != 0:
        raise OSError(f"tc_bam_write({path!r}) failed ({rc}): {err.value.decode(errors='replace')}")


def read_fasta_lengths(path: str) -> tuple[list[str], list[int]]:
    """Names and lengths of the records of a FASTA file — all that
    TrueConsense/indexing.py:97-98 takes from ``pysam.FastaFile`` (``lengths[0]``)."""
    names: list[str] = []
    lens: list[int] = []
    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                names.append(line[1:].split()[0] if len(line) > 1 and line[1:].split() else "")
                lens.append(0)
            elif names:
                lens[-1] += len(line.strip())
    return names, lens


def read_fasta(path: str) -> list[tuple[str, str]]:
    out: list[tuple[str, list[str]]] = []
    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                out.append((line[1:].split()[0] if line[1:].split() else "", []))
            elif out:
                out[-1][1].append(line.strip())
    return [(n, "".join(parts)) for n, parts in out]
