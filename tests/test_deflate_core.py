"""The BGZF member compressor the GPU BAM writer is built from (csrc/cuda/deflate_core.cuh), run on the CPU: its phases on
one thread, the same bytes the kernel writes.  Every stream inflates with zlib and with inflate_core.cuh's decoder; sizes
against zlib level 1; stored fallback, member bounds, determinism.  Also the host-side rules of ``--output-bam``: the
``@HD`` line of the written header, the flag's checks and the refusals that need no device."""
import ctypes
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from conftest import GOLD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_SRC = os.path.join(ROOT, "trueconsense_b200", "csrc", "cuda")
MEMBER = 0xFF00


def _build(name, headers):
    out_dir = os.path.join(ROOT, "build", "tests")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"lib{name}.so")
    src = os.path.join(ROOT, "tests", "native", f"{name}.cpp")
    deps = [src] + [os.path.join(CUDA_SRC, h) for h in headers]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.run(["g++", "-O2", "-g", "-shared", "-fPIC", "-x", "c++", "-I", CUDA_SRC, "-o", so, src], check=True)
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def h():
    lib = _build("deflate_harness", ["deflate_core.cuh", "inflate_core.cuh"])
    lib.h_deflate.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    lib.h_deflate.restype = ctypes.c_int
    return lib


@pytest.fixture(scope="module")
def inf():
    lib = _build("inflate_harness", ["inflate_core.cuh"])
    lib.h_inflate.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]
    return lib


def deflate(lib, data: bytes, threads: int = 512):
    """(raw DEFLATE stream, CRC-32) of one member compressed by the harness."""
    src = np.frombuffer(data, np.uint8).copy() if data else np.zeros(1, np.uint8)
    out = np.zeros(len(data) + 16, np.uint8)
    crc = ctypes.c_uint32()
    n = lib.h_deflate(src.ctypes.data, len(data), out.ctypes.data, ctypes.byref(crc), threads)
    assert n >= 0
    return out[:n].tobytes(), crc.value


def check(lib, inf, data: bytes):
    comp, crc = deflate(lib, data)
    assert zlib.decompressobj(-15).decompress(comp) == data
    assert crc == zlib.crc32(data)
    raw = np.zeros(len(comp) + 80, np.uint8)               # inflate_core reads aligned 16-byte vectors around the stream
    start = (-raw.ctypes.data) % 16 + 16
    raw[start:start + len(comp)] = np.frombuffer(comp, np.uint8)
    out = np.zeros(len(data) + 1, np.uint8)
    assert inf.h_inflate(raw.ctypes.data + start, len(comp), out.ctypes.data, len(data), 1) == 0
    assert out[:len(data)].tobytes() == data
    assert 18 + len(comp) + 8 <= 65536
    return comp


def _samples(rng):
    yield b""
    yield b"a"
    yield b"abc" * 5
    yield bytes(70000 // 7 * [1, 2, 3, 4, 5, 6, 7])[:MEMBER]
    yield bytes(MEMBER)                                                  # one run: length-258 matches at distance 1
    yield rng.integers(0, 256, MEMBER, dtype=np.uint8).tobytes()          # incompressible
    yield rng.integers(33, 75, MEMBER, dtype=np.uint8).tobytes()          # quality-like: literals only
    text = b"".join(b"read%07d\tACGT" % i + bytes(rng.integers(0, 4, 40, dtype=np.uint8) + 65) for i in range(1100))
    yield text[:MEMBER]
    far = rng.integers(0, 256, 2000, dtype=np.uint8).tobytes()
    yield far + bytes(rng.integers(0, 3, 30000, dtype=np.uint8)) + far   # a match 32 000 bytes back
    yield bytes(rng.integers(0, 2, MEMBER, dtype=np.uint8))               # two symbols
    for n in (1, 2, 3, 4, 5, 7, 8, 9, 255, 256, 257, 258, 259, 260, 1000, 4095, 4096, 4097, 32767, 32768, 32769, MEMBER - 1):
        yield rng.integers(0, 5, n, dtype=np.uint8).tobytes()


def test_members_inflate_to_their_input(h, inf):
    rng = np.random.default_rng(7)
    n = 0
    for data in _samples(rng):
        check(h, inf, data)
        n += 1
    assert n > 30


def _payload(name):
    with gzip.open(f"{GOLD}/{name}.bam", "rb") as fh:
        return fh.read()


@pytest.mark.parametrize("name", ["mini_illumina", "mini_ont", "mini_long", "mini_overlap", "quirk"])
def test_golden_payloads_in_members(h, inf, name):
    p = _payload(name)
    for o in range(0, len(p), MEMBER):
        check(h, inf, p[o:o + MEMBER])
    # members that start at other offsets (a header's length shifts the records' members)
    for o in (1, 777, 40000):
        check(h, inf, p[o:o + MEMBER])


def test_size_against_zlib_level_1(h):
    """Over the three golden payloads in 0xff00-byte members, 26 bytes of framing each: at most 1.10 x zlib level 1."""
    ours = ref = 0
    for name in ("mini_illumina", "mini_ont", "mini_long"):
        p = _payload(name)
        for o in range(0, len(p), MEMBER):
            d = p[o:o + MEMBER]
            ours += len(deflate(h, d)[0]) + 26
            c = zlib.compressobj(1, zlib.DEFLATED, -15)
            ref += len(c.compress(d) + c.flush()) + 26
    assert ref == 622_390 + 1_392_455 + 832_946
    assert ours <= 1.10 * ref, (ours, ref)


def test_incompressible_member_is_stored(h, inf):
    data = np.random.default_rng(3).integers(0, 256, MEMBER, dtype=np.uint8).tobytes()
    comp = check(h, inf, data)
    assert len(comp) == MEMBER + 5 and comp[0] == 1
    assert struct.unpack_from("<HH", comp, 1) == (MEMBER, MEMBER ^ 0xFFFF)
    assert 18 + len(comp) + 8 == 65311


def test_deterministic_and_independent_of_thread_count(h):
    p = _payload("mini_ont")
    for o in (0, 3 * MEMBER, len(p) - 5000):
        d = p[o:o + MEMBER]
        first = deflate(h, d, 512)
        assert deflate(h, d, 512) == first
        assert deflate(h, d, 32) == first and deflate(h, d, 1024) == first


# ---------------------------------------------------------------------------- the written header
def _hdr(text: bytes) -> bytes:
    return b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", 1) + struct.pack("<i", 4) + b"ref\0" + struct.pack("<i", 99)


def _text(header: bytes) -> bytes:
    return header[8:8 + struct.unpack_from("<i", header, 4)[0]]


def test_header_says_coordinate():
    from trueconsense_b200 import bamio

    same = _hdr(b"@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:99\n")
    assert bamio.coordinate_header(same) == same
    assert _text(bamio.coordinate_header(_hdr(b"@HD\tVN:1.6\tSO:unsorted\tGO:query\n@CO\tx\n"))) == \
        b"@HD\tVN:1.6\tSO:coordinate\tGO:query\n@CO\tx\n"
    assert _text(bamio.coordinate_header(_hdr(b"@HD\tVN:1.6\tSO:queryname\n"))) == b"@HD\tVN:1.6\tSO:coordinate\n"
    assert _text(bamio.coordinate_header(_hdr(b"@HD\tVN:1.4\n@SQ\tSN:ref\tLN:99\n"))) == b"@HD\tVN:1.4\tSO:coordinate\n@SQ\tSN:ref\tLN:99\n"
    assert _text(bamio.coordinate_header(_hdr(b"@HD\tVN:1.4"))) == b"@HD\tVN:1.4\tSO:coordinate"
    assert _text(bamio.coordinate_header(_hdr(b"@SQ\tSN:ref\tLN:99\n"))) == b"@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:99\n"
    assert _text(bamio.coordinate_header(_hdr(b""))) == b"@HD\tVN:1.6\tSO:coordinate\n"
    # an @HD line that is not the first is a line like any other
    assert _text(bamio.coordinate_header(_hdr(b"@CO\ta\n@HD\tVN:1.6\n"))) == b"@HD\tVN:1.6\tSO:coordinate\n@CO\ta\n@HD\tVN:1.6\n"
    out = bamio.coordinate_header(_hdr(b"@HD\tVN:1.6\n"))
    assert bamio.parse_bam_header(out, len(out)) == (["ref"], [99], len(out))


def test_sam_header_bytes(tmp_path):
    from trueconsense_b200 import bamio

    p = tmp_path / "x.sam"
    text = b"@HD\tVN:1.6\n@SQ\tSN:a\tLN:10\n@SQ\tSN:bb\tLN:20\n@PG\tID:mm2\n"
    p.write_bytes(text + b"r\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\n")
    names, lens, off, _ = bamio.read_sam_header(str(p))
    hdr = bamio.sam_bam_header(str(p), names, lens, off)
    assert _text(hdr) == text
    assert bamio.parse_bam_header(hdr, len(hdr)) == (["a", "bb"], [10, 20], len(hdr))


# ---------------------------------------------------------------------------- flag and refusals
def _argv(extra):
    n = "mini_illumina"
    return ["-i", f"{GOLD}/{n}.bam", "-ref", f"{GOLD}/{n}.fasta", "-gff", f"{GOLD}/{n}.gff", "-cov", "30", "-name", "S",
            "-o", "x.fasta"] + extra


def test_output_bam_flag():
    from trueconsense_b200 import TrueConsense

    assert TrueConsense.GetArgs(_argv([])).output_bam is None
    assert TrueConsense.GetArgs(_argv(["--output-bam", "out/S.bam"])).output_bam == "out/S.bam"
    assert TrueConsense.GetArgs(_argv(["-obam", "S.bam", "--sort-input", "--all-contigs"])).output_bam == "S.bam"
    for bad in ("S.sam", "S", "S.bam.gz"):
        with pytest.raises(SystemExit) as e:
            TrueConsense.GetArgs(_argv(["--output-bam", bad]))
        assert e.value.code == 2


def test_refusals_without_a_device(host_libs, tmp_path):
    from trueconsense_b200 import bamio, gpu, indexing

    batch = bamio.read_bam(f"{GOLD}/mini_illumina.bam")
    with pytest.raises(ValueError, match="host ReadBatch"):
        indexing.BamHandle("x.bam", reads=batch, output_bam=str(tmp_path / "o.bam"))
    ctx = gpu.Context.__new__(gpu.Context)          # (no device here: only the checks in front of the library call run)
    ctx._generation = 3
    uploaded = gpu.DeviceReads(gpu.TcReads(), batch, ctx, 3)
    with pytest.raises(ValueError, match="host ReadBatch"):
        ctx.write_bam(uploaded, str(tmp_path / "o.bam"))
    stale = gpu.DeviceReads(gpu.TcReads(), None, ctx, 2)
    stale.records = (b"", None, 0, None, 0)
    with pytest.raises(RuntimeError, match="stale"):
        ctx.write_bam(stale, str(tmp_path / "o.bam"))
    assert not os.path.exists(tmp_path / "o.bam")
