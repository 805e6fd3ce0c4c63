"""The pileup kernels at the edges inside them, against the oracle (bit for bit, all 8 rows).

Variant 3 (pileup_warp.cu) keeps the reads of a window of 256, 512 or 1024 columns while their starts stay within the
window's first `slack` columns; the window is chosen from the longest reference span (warp_geometry on the host when
the caller bounds the span, warp_pileup_kernel on the device when a span pass found it) and walked in phases of 256
columns.  Variant 4 (pileup_long.cu) cuts longer reads into pieces at the borders of cells of 400 columns and runs
variant 3 over the pieces.  The cases below aim at those edges: the spans where one geometry hands over to the next,
starts on the slack's last column and one past it, ops that end on a phase or cell border, deletions and reference
skips covering whole cells, reads of more than 2048 ops, counter runs of more than 2047 pieces, and the reference's
last column.  Every batch runs through the kernel it is aimed at (an explicit kernel raises instead of falling back)
and through the library's own choice with the span bound exact, loose and absent, from host and from device reads."""
import numpy as np
import pytest

from test_gpu_parity import _chained
from test_piece_rule_cpu import PIECE_COLS, long_read_records, record

pytestmark = pytest.mark.gpu

MIN_SLACK = 64              # pileup.cuh
PHASE_COLS = 256            # the rows of variant 3 cover one phase of 256 columns
EDGES = (184, 440, 952)     # the longest span each window (256 / 512 / 1024 columns) takes
# kernel launches of one tc_pileup_counts call, by route (the coverage scan's two kernels included)
V3_BOUND = 3                # variant 3 alone: the caller's bound picks the window
V3_NO_BOUND = 6             # span pass, variant 3 in all three geometries (two return at once)
V4_BOUND = 11               # span pass, the split (count, two scans, split, finish, iota, sort), variant 3 over the pieces
V3_THEN_V4 = 17             # no bound: span pass and variant 3, which declines the batch, then variant 4
V1_AFTER = 3                # variant 4 declined (reads without SEQ): then the scatter kernel


def geometry(span: int):
    """(window width, slack) variant 3 uses for reads of at most `span` columns; (0, 0) when no window fits (warp_geometry)."""
    ms = (span + 7) & ~7
    for width in (256, 512, 1024):
        slack = (width - ms - 8) & ~7
        if slack >= MIN_SLACK:
            return width, slack
    return 0, 0


def route(bound: int, span: int, no_seq: bool) -> int:
    """The launches of kernel = 0 with the span bound `bound` (<= 0: none) over reads of longest span `span`; no_seq:
    some reads have no SEQ, which variant 4 declines."""
    if bound > 0:
        n = V3_BOUND if geometry(bound)[0] else V4_BOUND
    else:
        n = V3_NO_BOUND if geometry(span)[0] else V3_THEN_V4
    return n + (V1_AFTER if no_seq and n in (V4_BOUND, V3_THEN_V4) else 0)


@pytest.fixture(scope="module")
def orc():
    from oracle import pileup

    pileup.build()
    return pileup


@pytest.fixture(scope="module")
def ctx():
    from trueconsense_b200 import gpu

    return gpu.Context(0)


def _batch(recs):
    from trueconsense_b200.reads import ReadBatch

    recs.sort(key=lambda r: r["pos"])
    return ReadBatch.from_records(recs)


def _where(got, exp):
    bad = np.argwhere(got != exp)
    return f"{len(bad)} cells differ, first (row, column) {tuple(bad[0])}: {got[tuple(bad[0])]} != {exp[tuple(bad[0])]}" if len(bad) else ""


def _counted(ctx, fn):
    l0 = ctx.launches
    out = fn()
    return out, ctx.launches - l0


def _check(ctx, orc, b, L, kernel, declined=False, extra_bounds=(), chained=False, mincov=10):
    """b must give the oracle's table through the explicit `kernel` (or raise TC_ERR_CAPACITY when `declined`) and
    through kernel = 0 with the span bound exact, one wider, one geometry wider, `extra_bounds` and absent, from host
    and from device reads (kernel = 0: the route's launch count too, unless declined); depth must equal row 0; with
    `chained` the chained sample must equal the separate calls."""
    from trueconsense_b200 import gpu

    exp = orc.pileup_counts(b, L, threads=8)
    span = int(b.ref_spans().max())
    wider = next(e for e in (185, 441, 953, 20_000) if e > span + 1)
    bounds = (span, span + 1, wider) + tuple(extra_bounds) + (-1,)
    for dev_reads in (False, True):
        reads = ctx.upload(b) if dev_reads else b
        for bound in bounds:
            if dev_reads:
                reads.struct.max_ref_span = max(bound, 0)
            else:
                b.max_ref_span = bound
            if declined:
                with pytest.raises(gpu.TcError) as e:
                    ctx.pileup_counts(reads, L, gpu.buildindex_params(kernel))
                assert e.value.code == -8, (kernel, bound, dev_reads)
            else:
                got = ctx.pileup_counts(reads, L, gpu.buildindex_params(kernel))
                assert np.array_equal(got, exp), (f"kernel {kernel}", bound, dev_reads, _where(got, exp))
            got, n = _counted(ctx, lambda: ctx.pileup_counts(reads, L, gpu.buildindex_params(0)))
            assert np.array_equal(got, exp), ("kernel 0", bound, dev_reads, _where(got, exp))
            assert declined or n == route(bound, span, bool((b.l_seq == 0).any())), ("launches", bound, dev_reads, n)
        assert np.array_equal(ctx.depth(reads, L), exp[0]), ("depth", dev_reads)
    if chained:
        b.max_ref_span = -1
        counts = ctx.pileup_counts(b, L)
        res = ctx.call(counts, L, mincov, True)
        sep = ctx.extract_inserts(b, L, ctx.list_insert_candidates(res.flags, L))
        c2, f2, _, _, ins = _chained(ctx, b, L, mincov, ctx.upload(b))
        assert np.array_equal(c2, exp) and np.array_equal(f2, res.flags) and ins == sep
    return exp


def _short_ops(rng, pos: int, span: int, tail: str = "M"):
    """Ops of a read at `pos` covering exactly `span` columns, with clips, insertions, deletions, reference skips and
    D / N / I adjacencies; match, D and N ops are steered to end on, start on or end one off the phase borders of the
    window the read would open (multiples of 256 columns behind pos rounded down to 8).  tail: the last op covers the
    last column ("M", "D" or "N"), or "I": an insertion anchored on the last column follows."""
    end = pos + span
    tail_len = min(int(rng.integers(1, 4)), span - 1) if tail in "DN" else 0
    stop = end - tail_len
    ops = []
    if rng.random() < 0.2:
        ops.append(("S", int(rng.integers(1, 13))))
    elif rng.random() < 0.05:
        ops.append(("H", int(rng.integers(1, 20))))
    x, w0 = pos, pos & ~7
    while x < stop:
        border = w0 + PHASE_COLS * (1 + (x - w0) // PHASE_COLS)
        l = int(rng.integers(1, 50))
        if rng.random() < 0.4 and border - x < 60:
            l = border - x + int(rng.integers(-1, 2))
        l = max(1, min(l, stop - x))
        o = "M" if rng.random() < 0.95 else "="
        if stop - x - l < 2:                    # too close to the end for another op: this match op closes the read
            ops.append((o, stop - x))
            break
        ops.append((o, l))
        x += l
        room = stop - x - 1                     # a match op closes the read
        u = rng.random()
        border = w0 + PHASE_COLS * (1 + (x - w0) // PHASE_COLS)
        steer = border - x + int(rng.integers(-1, 2)) if border - x < 40 and rng.random() < 0.5 else 0
        if u < 0.3:
            ops.append(("I", int(rng.integers(1, 4))))
        elif u < 0.6:
            l = min(steer or int(rng.integers(1, 4)), room); ops.append(("D", max(l, 1))); x += max(l, 1)
        elif u < 0.7:
            l = min(steer or int(rng.integers(1, 30)), room); ops.append(("N", max(l, 1))); x += max(l, 1)
        elif u < 0.8:
            a, c = min(int(rng.integers(1, 3)), room), int(rng.integers(1, 3))
            d = "DN"[int(rng.random() < 0.3)]
            ops += [(d, a), ("I", c)] if rng.random() < 0.5 else [("I", c), (d, a)]
            x += a
    assert ops[-1][0] in "M=" and ops[-1][1] > 0
    if tail in "DN" and tail_len:
        ops.append((tail, tail_len))
    elif tail == "I":
        ops.append(("I", int(rng.integers(1, 4))))
    if rng.random() < 0.2:
        ops.append(("S", int(rng.integers(1, 13))))
    return ops


def _short_read(rng, pos, span, tail="M", no_seq=0.01):
    r = record(rng, pos, _short_ops(rng, pos, span, tail))
    if rng.random() < no_seq:
        r["seq"] = "*"                          # no SEQ: every base reads 'N' (coverage and events only)
    return r


# ---------------------------------------------------------------------------- 1. geometry edges
@pytest.mark.parametrize("span", [184, 185, 440, 441, 952, 953])
def test_geometry_edge(ctx, orc, span):
    """The longest span sits exactly on an edge of warp_geometry (184 / 440 / 952: the last span of the 256 / 512 /
    1024-column window, slack exactly MIN_SLACK) or one past it (the next geometry's first span; 953: no window, the
    reads are cut into pieces).  Reads are spread over many windows: after a read whose start is a multiple of 8, the
    next start is often exactly slack - 1, slack or slack + 1 columns on (the last start a window takes, and the
    first two it does not), and those reads take the longest span, so they reach the last column a window can.
    Variant 3 must take spans up to 952 itself and decline 953; kernel = 0 must then take variant 4.  The host's and
    the device's choice of window must agree (a window the device does not expect counts nothing)."""
    rng = np.random.default_rng(span)
    slack = geometry(span)[1] or MIN_SLACK
    no_seq = 0.01 if span <= EDGES[-1] else 0.0             # (variant 4 declines reads without SEQ)
    recs, p = [], 50
    for _ in range(min(16000 if span < 900 else 9000, int(400_000 / (0.35 * slack + 2)))):
        u = rng.random()
        if u < 0.3:
            pass                                            # the same start
        elif u < 0.55:
            p += int(rng.integers(1, 9))
        elif u < 0.65:
            p = (p | 7) + 1                                 # a multiple of 8
        else:
            d = int(rng.integers(-1, 2))
            p = (p & ~7) + slack + d                        # the slack's last column, or one or two past it
            recs.append(_short_read(rng, p, span if d == -1 or rng.random() < 0.2 else span - int(rng.integers(0, 12)), no_seq=no_seq))
            continue
        s = span if rng.random() < 0.1 else span - int(rng.integers(1, 12))
        recs.append(_short_read(rng, p, s, "MMMDNI"[int(rng.integers(0, 6))], no_seq))
    b = _batch(recs)
    L = int(max(r["pos"] for r in recs)) + span + 8
    assert int(b.ref_spans().max()) == span
    _check(ctx, orc, b, L, 3, declined=span > EDGES[-1], chained=span in (184, 953))
    if span > EDGES[-1]:
        _check(ctx, orc, b, L, 4)


def test_loose_bound_takes_the_widest_window(ctx, orc):
    """Reads of at most 150 columns under a bound of 900: the host picks the 1024-column window, which the reads
    cross in its 4 phases."""
    rng = np.random.default_rng(150)
    recs = [_short_read(rng, 20 + int(rng.integers(0, 4000)), 150 - int(rng.integers(0, 20))) for _ in range(6000)]
    recs.append(_short_read(rng, 30, 150))
    b = _batch(recs)
    _check(ctx, orc, b, 4200, 3, extra_bounds=(900,))


# ---------------------------------------------------------------------------- 2. phase edges
@pytest.mark.parametrize("span", EDGES)
def test_phase_edges(ctx, orc, span):
    """Each geometry at its longest span: reads that open their own window (starts a few columns apart, one warp's
    reads in one window) with match, D and N ops that end on, start on or end one off each 256-column phase border of
    that window, the last phase of the 1024-column window included."""
    rng = np.random.default_rng(10 + span)
    base = 1000
    recs = []
    for _ in range(3000):
        pos = base + int(rng.integers(0, 64))
        recs.append(_short_read(rng, pos, span - int(rng.integers(0, 16)) if rng.random() < 0.8 else span))
    recs.append(_short_read(rng, base, span))
    b = _batch(recs)
    _check(ctx, orc, b, base + 64 + span + 8, 3)


# ---------------------------------------------------------------------------- 3. piece cuts
def test_piece_cuts(ctx, orc):
    """Long reads (1-12 kb) with ops steered onto the cell borders (absolute multiples of 400) and one off them: match
    ops ending on a border followed by I, D, N, I D and D I; D / N of 400-5000 columns, so pieces made of one deletion
    or skip; reads starting on a border, and whose first op after the clips is an I; leading and trailing soft clips
    of 4096+ bases (variant 4 drops leading clips, so unlike variant 3 it takes them); reads ending on a border; and
    reads of 2049-6000 ops (the split works in rounds of 2048 ops, its state carried from one to the next)."""
    rng = np.random.default_rng(400)
    recs = long_read_records(rng, 2500, dense=40)
    b = _batch(recs)
    assert np.diff(b.cigar_off.astype(np.int64)).max() > 2048
    L = int(max(r["pos"] for r in recs) + b.ref_spans().max()) + 5
    _check(ctx, orc, b, L, 4, chained=True)


def test_deep_amplicon_panel(ctx, orc):
    """ONT tiled amplicons: 25 amplicons of 1000-1300 bp (too long for any window of variant 3), 2500 reads each.  All
    reads of an amplicon start within a few columns, so their pieces start on the same cell borders, thousands deep:
    more than the 2047 reads one counter run of variant 3 holds."""
    rng = np.random.default_rng(25)
    recs, start = [], 30
    for k in range(25):
        length = int(rng.integers(1000, 1301))
        if k % 3 == 0:
            start = PIECE_COLS * (start // PIECE_COLS + 1)  # some amplicons start on a cell border
        templates = []
        for _ in range(300):
            trim = int(rng.integers(0, 4))
            templates.append((start + trim, _ont_ops(rng, length - trim - int(rng.integers(0, 4)))))
        for _ in range(2500):
            pos, ops = templates[int(rng.integers(0, len(templates)))]
            recs.append(record(rng, pos, ops))
        start += length - int(rng.integers(60, 160))        # the next amplicon overlaps this one
    b = _batch(recs)
    L = start + 1400
    exp = _check(ctx, orc, b, L, 4, chained=True)
    assert exp[0].max() >= 2500


def _ont_ops(rng, span):
    """An ONT-like alignment of `span` columns: an indel every ~30 bases, soft clips at both ends."""
    ops, x = [("S", int(rng.integers(5, 60)))], 0
    while True:
        l = int(rng.integers(5, 60))
        if x + l >= span - 4:
            ops.append(("M", span - x))
            break
        ops.append(("M", l)); x += l
        if rng.random() < 0.5:
            ops.append(("I", int(rng.integers(1, 4))))
        else:
            l = int(rng.integers(1, 4)); ops.append(("D", l)); x += l
    ops.append(("S", int(rng.integers(5, 60))))
    return ops


# ---------------------------------------------------------------------------- 4. declined inputs
def _declined_read(rng, what):
    pos = 2 * PIECE_COLS + 17
    if what == "no_seq":
        r = record(rng, pos, [("M", 700), ("D", 3), ("M", 900), ("I", 2), ("M", 500)])
        r["seq"] = "*"
    elif what == "pad":
        r = record(rng, pos, [("M", 700), ("P", 2), ("I", 3), ("M", 1500)])
    else:                                   # 15 200 inserted bases in one cell: more than one piece can stage
        r = record(rng, pos, [("M", 100)] + [("I", 3800), ("M", 20)] * 3 + [("I", 3800), ("M", 1200)])
    return r


@pytest.mark.parametrize("what", ["no_seq", "pad", "huge_piece"])
def test_declined_long_reads(ctx, orc, what):
    """Inputs variant 4 declines (TC_ERR_CAPACITY with the explicit kernel): a long read without SEQ, a long read with
    a pad, a piece whose query is longer than the staging buffers.  kernel = 0 must still give the oracle's table."""
    rng = np.random.default_rng(4)
    recs = long_read_records(rng, 150, hi=4000)
    recs.append(_declined_read(rng, what))
    b = _batch(recs)
    L = int(max(r["pos"] for r in recs) + b.ref_spans().max()) + 5
    _check(ctx, orc, b, L, 4, declined=True)


# ---------------------------------------------------------------------------- 5. reference end
@pytest.mark.parametrize("L", [1, 7, 8, 9, 255, 257, 1023, 1025, 1031])
def test_reference_end(ctx, orc, L):
    """Reads over the reference's last column: ending exactly on it, with a D or N on it, or with an insertion
    anchored on it, for references shorter than one window and of lengths that are not multiples of 8 (the count
    flush and the X / I events clamp to the reference).  Each window of variant 3 through its span bound, and
    variant 4."""
    from trueconsense_b200 import gpu

    rng = np.random.default_rng(L)
    for edge in EDGES + (2000,):
        top = min(L, edge)
        recs = []
        for i in range(400):
            s = top if i % 4 == 0 else int(rng.integers(1, top + 1))
            tail = "MDNI"[int(rng.integers(0, 4))] if s > 1 else "MI"[int(rng.integers(0, 2))]
            pos = L - s if rng.random() < 0.7 else int(rng.integers(0, L - s + 1))
            recs.append(_short_read(rng, pos, s, tail, no_seq=0.01 if edge < 2000 else 0.0))
        b = _batch(recs)
        if edge < 2000:
            exp = orc.pileup_counts(b, L, threads=8)
            b.max_ref_span = edge                           # the host launches the window of this edge
            got = ctx.pileup_counts(b, L, gpu.buildindex_params(3))
            assert np.array_equal(got, exp), (edge, _where(got, exp))
        if edge in (EDGES[0], 2000):
            _check(ctx, orc, b, L, 4 if edge == 2000 else 3)
