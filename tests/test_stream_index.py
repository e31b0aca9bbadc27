"""Seek index of one long stream (zwz_inflate_stream_index*, zwz_index_*): access points chosen from the confirmed span starts of
zwz_inflate_stream, their windows, the saved blob and its checks, and ranges extracted from the points (inflate_seek.cuh), all
against system zlib. The emulator variants use spans of a few KiB so that streams of a few hundred KB get many access points."""
import bisect
import gzip
import struct
import zlib

import numpy as np
import pytest

import zwz_b200
from test_inflate_stream import _Bits, _compress, _fixed_block, _ref
from tools import corpus

END, TRUNC, BAD = zwz_b200.STREAM_END, zwz_b200.STREAM_TRUNCATED, zwz_b200.STREAM_BAD
CAREFUL = zwz_b200.INFLATE_CAREFUL
E_ARG = -3
M_BLOCK, M_START, M_MEMBER, M_STORED = 0, 1, 2, 3
PT = np.dtype([("out", "<u8"), ("bit", "<u8"), ("mode", "<u2"), ("bfinal", "u1"), ("pad", "u1"), ("wlen", "<u4")])


@pytest.fixture(scope="module")
def sctx(emu_ctx):
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    yield emu_ctx
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 0)


def _parse(blob):
    """The saved form restated: (header dict, point table, windows)."""
    assert blob[:8] == b"ZWZIDX\0\1"
    ver, fmt, comp_len, raw_len, n, spacing, crc, zero = struct.unpack_from("<IIQQQQII", blob, 8)
    assert (ver, zero) == (1, 0)
    assert crc == zlib.crc32(blob[:48] + b"\0" * 4 + blob[52:])
    pts = np.frombuffer(blob, dtype=PT, count=n, offset=56)
    wins, o = [], 56 + 24 * n
    for w in pts["wlen"]:
        wins.append(blob[o:o + int(w)])
        o += int(w)
    assert o == len(blob)
    return dict(format=fmt, comp_len=comp_len, raw_len=raw_len, n=n, spacing=spacing), pts, wins


def _member_starts(comp, fmt):
    """Output offsets where gzip members start (the stream start for zlib and raw)."""
    if fmt != "gzip":
        return [0]
    starts, pos, total = [], 0, 0
    while len(comp) - pos >= 2 and comp[pos:pos + 2] == b"\x1f\x8b":
        d = zlib.decompressobj(31)
        try:
            part = d.decompress(comp[pos:])
        except zlib.error:
            break
        starts.append(total)
        if not d.eof:
            break
        total += len(part)
        pos = len(comp) - len(d.unused_data)
    return starts or [0]


def _build(ctx, comp, fmt, spacing):
    """Build an index and check it against inflate_stream and zlib -> (index, blob, points, reference bytes)."""
    want, wst = _ref(comp, fmt)
    cap = max(len(want), 1 << 22) + 64
    out, st, ix = ctx.inflate_stream_index(comp, format=fmt, spacing=spacing, out_cap=cap)
    o2, s2 = ctx.inflate_stream(comp, format=fmt, out_cap=cap)
    assert (st, out.tobytes()) == (s2, o2.tobytes()) == (wst, want)
    assert ix is not None and (ix.raw_len, ix.comp_len, ix.format, ix.npoints) == (len(want), len(comp), zwz_b200._format(fmt), ix.npoints)
    blob = ix.save()
    hdr, pts, wins = _parse(blob)
    assert (hdr["format"], hdr["comp_len"], hdr["raw_len"], hdr["n"], hdr["spacing"]) == (ix.format, len(comp), len(want), ix.npoints, spacing)
    assert tuple(pts[0]) == (0, 0, M_START, 0, 0, 0)
    assert (np.diff(pts["out"].astype(np.int64)) >= max(spacing, 1)).all()
    assert (np.diff(pts["bit"].astype(np.int64)) > 0).all() and int(pts["bit"][-1]) < 8 * len(comp)
    ms = _member_starts(comp, fmt)
    for p, w in zip(pts, wins):
        o = int(p["out"])
        m0 = ms[bisect.bisect_right(ms, o) - 1]
        # the window is everything of the member before the point, up to 32 KiB: the INVALID entries were exactly a prefix
        assert int(p["wlen"]) == min(32768, o - m0), (o, m0, int(p["mode"]))
        assert w == want[o - len(w):o]
        if p["mode"] == M_STORED:
            assert (int(p["bit"]) + 3) % 8 == 0
    return ix, blob, pts, want


def _ranges(rng, raw_len, pts, n):
    """Seeded ranges: empty ones, the whole stream, ranges ending at raw_len, at a point, one byte before it, across points."""
    po = [int(x) for x in pts["out"]]
    off, ln = [0, 0, raw_len, max(raw_len - 5, 0), raw_len // 2], [0, raw_len, 0, min(5, raw_len), raw_len - raw_len // 2]
    for p in po[1:]:
        off += [p, p - 1]
        ln += [min(int(rng.integers(1, 3000)), raw_len - p), min(2, raw_len - p + 1)]
    if len(po) > 3:
        off.append(po[1] - 7)
        ln.append(po[3] - po[1] + 20 if po[3] + 13 <= raw_len else raw_len - po[1] + 7)
    while len(off) < n:
        a = int(rng.integers(0, raw_len + 1))
        off.append(a)
        ln.append(int(rng.integers(0, min(raw_len - a, 40000) + 1)))
    return np.array(off[:n], dtype=np.uint64), np.array(ln[:n], dtype=np.uint64)


def _extract_check(ix, comp, want, off, ln):
    for flags in (0, CAREFUL):
        data, oo, got, st = ix.extract(comp, off, ln, flags=flags)
        assert (st == END).all() and (got == ln).all(), (flags, st[st != END][:5])
        for i in range(len(off)):
            a, n = int(off[i]), int(ln[i])
            assert data[int(oo[i]):int(oo[i]) + n].tobytes() == want[a:a + n], (flags, a, n)


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_index_levels(sctx, fmt, level):
    raw = corpus.gen_text(200000, 596, level + 20).tobytes()
    comp = _compress(raw, fmt, level)
    ix, blob, pts, want = _build(sctx, comp, fmt, 0)
    big = _build(sctx, comp, fmt, 1 << 20)[0]
    assert ix.npoints > big.npoints == 1
    _extract_check(ix, comp, want, *_ranges(np.random.default_rng(level), len(want), pts, 200))


@pytest.mark.parametrize("strategy", [zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED])
def test_index_strategies(sctx, strategy):
    raw = corpus.gen_text(150000, 596, 3).tobytes() + bytes(20000) + corpus.gen_struct(30000, 596, 4).tobytes()
    comp = _compress(raw, "gzip", 6, strategy)
    ix, blob, pts, want = _build(sctx, comp, "gzip", 0)
    if strategy == zlib.Z_FIXED:
        assert ix.npoints == 1  # fixed blocks cannot be found: one span, one point
    else:
        assert ix.npoints > 1
    _extract_check(ix, comp, want, *_ranges(np.random.default_rng(strategy), len(want), pts, 120))


def test_index_gzip_members(sctx):
    """Several members, empty ones among them, written at different levels, with garbage behind the last; ranges across members."""
    parts = [corpus.gen_text(n, 596, i).tobytes() for i, n in enumerate([30000, 0, 4096, 50000, 0, 1, 40000, 25000])]
    comp = b"".join(gzip.compress(p, lv) for p, lv in zip(parts, [6, 1, 9, 0, 6, 3, 9, 1]))
    for tail in (b"", b"garbage behind the last member"):
        ix, blob, pts, want = _build(sctx, comp + tail, "gzip", 0)
        assert M_MEMBER in set(pts["mode"].tolist()) or ix.npoints > 3
        ends = np.cumsum([len(p) for p in parts])
        off = np.array([int(e) - 10 for e in ends if 10 <= e < len(want) - 10], dtype=np.uint64)
        ln = np.full(len(off), 20, dtype=np.uint64)
        _extract_check(ix, comp + tail, want, off, ln)
        _extract_check(ix, comp + tail, want, *_ranges(np.random.default_rng(7), len(want), pts, 120))


def test_index_many_members(sctx):
    """More members than one span records: spans start at member headers (MEMBER points)."""
    parts = [corpus.gen_text(40 + 7 * (i % 13), 596, i).tobytes() for i in range(400)]
    comp = b"".join(gzip.compress(p, 6) for p in parts)
    ix, blob, pts, want = _build(sctx, comp, "gzip", 0)
    assert M_MEMBER in set(pts["mode"].tolist())
    _extract_check(ix, comp, want, *_ranges(np.random.default_rng(8), len(want), pts, 150))


def test_index_bgzf(sctx):
    raw = corpus.gen_text(300000, 596, 9).tobytes()
    gz, _ = sctx.gzip_files(raw, np.array([0, len(raw)], dtype=np.uint64))
    comp = gz.tobytes()
    ix, blob, pts, want = _build(sctx, comp, "gzip", 0)
    assert want == raw
    _extract_check(ix, comp, want, *_ranges(np.random.default_rng(9), len(want), pts, 150))


def test_index_stored_padding_not_zero(sctx):
    """A stored block's key may lie in padding that is not zero: a STORED point takes the block type from its mode."""
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 1024)
    try:
        for hdr in (0x01, 0xF9):
            p1 = bytearray(corpus.gen_text(3000, 596, 1).tobytes())
            p1[1500:1505] = bytes([0, 0x10, 0x00, 0xef, 0xff])
            p2 = corpus.gen_text(600, 596, 2).tobytes()
            comp = bytes([0]) + len(p1).to_bytes(2, "little") + (len(p1) ^ 0xFFFF).to_bytes(2, "little") + bytes(p1)
            comp += bytes([hdr]) + len(p2).to_bytes(2, "little") + (len(p2) ^ 0xFFFF).to_bytes(2, "little") + p2
            ix, blob, pts, want = _build(sctx, comp, "raw", 0)
            st = [int(p["out"]) for p in pts if p["mode"] == M_STORED]
            assert st == [len(p1)]
            off = np.array([st[0], st[0], st[0] - 1, 0], dtype=np.uint64)
            ln = np.array([len(p2), 10, 2, len(want)], dtype=np.uint64)
            _extract_check(ix, comp, want, off, ln)
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)


def test_no_index_for_bad_streams(sctx):
    """Truncated, corrupted and too-far-back streams: no index, and output and status are inflate_stream's."""
    rng = np.random.default_rng(5)
    raws = [corpus.gen_text(60000, 596, 3).tobytes(), corpus.gen_struct(40000, 596, 4).tobytes()]
    streams = [("gzip", gzip.compress(raws[0], 6) + gzip.compress(raws[1], 6)), ("zlib", _compress(raws[0], "zlib")),
               ("raw", _compress(raws[1], "raw", 9))]
    b = _Bits()
    _fixed_block(b, b"abcd", 5)
    cases = [("raw", b.bytes())]
    for fmt, comp in streams:
        for _ in range(4):
            cases.append((fmt, comp[:int(rng.integers(0, len(comp)))]))
            bad = bytearray(comp)
            bad[int(rng.integers(0, len(bad)))] ^= 1 << int(rng.integers(0, 8))
            cases.append((fmt, bytes(bad)))
    for fmt, comp in cases:
        out, st, ix = sctx.inflate_stream_index(comp, format=fmt, spacing=0, out_cap=1 << 22)
        o2, s2 = sctx.inflate_stream(comp, format=fmt, out_cap=1 << 22)
        assert (st, out.tobytes()) == (s2, o2.tobytes())
        assert (ix is None) == (st != END)
    out, st, ix = sctx.inflate_stream_index(streams[1][1], format="zlib", out_cap=10)
    assert (st, ix) == (zwz_b200.STREAM_OUTPUT_FULL, None)


@pytest.mark.parametrize("fmt", ["gzip", "raw"])
def test_blobs_identical(sctx, fmt):
    """The same index from one wave and from many (tiny scratch budget), from the host and device forms, with and without output;
    and load(save(ix)) saves the same blob and extracts the same bytes."""
    raw = corpus.gen_text(250000, 596, 6).tobytes() + b"\0" * 50000 + corpus.gen_struct(60000, 596, 7).tobytes()
    comp = _compress(raw, fmt, 6)
    if fmt == "gzip":
        comp += gzip.compress(raw[:40000]) + gzip.compress(b"")
        raw += raw[:40000]
    out, st, ix = sctx.inflate_stream_index(comp, format=fmt, spacing=8192)
    assert (st, out.tobytes()) == (END, raw)
    blob = ix.save()
    _, _, ix2 = sctx.inflate_stream_index(comp, format=fmt, spacing=8192, want_output=False)
    assert ix2.save() == blob
    dc, do = sctx.malloc_device(len(comp)), sctx.malloc_device(len(raw))
    try:
        sctx.h2d(dc, np.frombuffer(comp, dtype=np.uint8))
        for d_out in (do, None):
            n, st, ix3 = sctx.inflate_stream_index_device(dc, len(comp), d_out, len(raw), format=fmt, spacing=8192)
            assert (n, st) == (len(raw), END) and ix3.save() == blob
        # device extraction into a canary: nothing outside the ranges is written
        off = np.array([10, 70000, 123456], dtype=np.uint64)
        ln = np.array([1000, 50000, 3], dtype=np.uint64)
        oo = np.array([5, 2000, 60000], dtype=np.uint64)
        canary = np.full(len(raw), 0x5A, dtype=np.uint8)
        sctx.h2d(do, canary)
        got, st = ix.extract_device(dc, len(comp), off, ln, do, oo)
        assert (st == END).all() and (got == ln).all()
        back = np.empty_like(canary)
        sctx.d2h(back, do)
        exp = canary.copy()
        for a, n, o in zip(off, ln, oo):
            exp[int(o):int(o + n)] = np.frombuffer(raw[int(a):int(a + n)], dtype=np.uint8)
        assert (back == exp).all()
    finally:
        sctx.free_device(dc)
        sctx.free_device(do)
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 40000)
    try:
        out, st, ix4 = sctx.inflate_stream_index(comp, format=fmt, spacing=8192)
        assert (st, out.tobytes()) == (END, raw) and ix4.save() == blob
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 0)
    ld = sctx.load_index(blob)
    assert ld.save() == blob and (ld.npoints, ld.raw_len, ld.comp_len, ld.format) == (ix.npoints, ix.raw_len, ix.comp_len, ix.format)
    rng = np.random.default_rng(11)
    off = rng.integers(0, len(raw), 80).astype(np.uint64)
    ln = np.minimum(rng.integers(0, 30000, 80).astype(np.uint64), len(raw) - off)
    a, b = ix.extract(comp, off, ln), ld.extract(comp, off, ln)
    assert all((x == y).all() for x, y in zip(a, b)) and (a[3] == END).all()
    for i in range(80):
        assert a[0][int(a[1][i]):int(a[1][i + 1])].tobytes() == raw[int(off[i]):int(off[i] + ln[i])]


def _blob(fmt, comp_len, raw_len, points, windows, spacing=0, version=1, fix_crc=True):
    """A hand-built index blob; points: (out, bit, mode, bfinal, wlen)."""
    b = bytearray(b"ZWZIDX\0\1" + struct.pack("<IIQQQQII", version, fmt, comp_len, raw_len, len(points), spacing, 0, 0))
    for o, bit, mode, bf, wl in points:
        b += struct.pack("<QQHBBI", o, bit, mode, bf, 0, wl)
    b += b"".join(windows)
    if fix_crc:
        struct.pack_into("<I", b, 48, zlib.crc32(bytes(b)))
    return bytes(b)


def _refused(ctx, blob):
    with pytest.raises(zwz_b200.ZwzError) as e:
        ctx.load_index(blob)
    return e.value.code == E_ARG if hasattr(e.value, "code") else True


def test_load_refusals(sctx):
    raw = corpus.gen_text(120000, 596, 12).tobytes()
    comp = _compress(raw, "gzip", 6)
    ix, blob, pts, want = _build(sctx, comp, "gzip", 0)
    n = len(pts)
    assert n >= 2
    for k in range(56 + 24 * n):  # every single-byte flip of the header and the point table
        bad = bytearray(blob)
        bad[k] ^= 0xFF
        assert _refused(sctx, bytes(bad)), k
    rng = np.random.default_rng(13)
    wbytes = len(blob) - (56 + 24 * n)
    for _ in range(200):
        bad = bytearray(blob)
        bad[56 + 24 * n + int(rng.integers(0, wbytes))] ^= 1 << int(rng.integers(0, 8))
        assert _refused(sctx, bytes(bad))
    for cut in (0, 7, 55, 56, 56 + 24 * n - 1, len(blob) - 1):
        assert _refused(sctx, blob[:cut])
    assert _refused(sctx, blob + b"\0")
    # hand-built blobs with a correct CRC, each breaking one rule; the first one is valid
    C, R = len(comp), len(want)
    w = want[1000 - 500:1000]
    good = [(0, 0, M_START, 0, 0), (1000, 4000, M_BLOCK, 0, 500)]
    assert sctx.load_index(_blob(1, C, R, good, [w])).npoints == 2
    cases = [
        _blob(1, C, R, good, [w], version=2),
        _blob(3, C, R, good, [w]),
        _blob(1, 0xFFFFFF01, R, good, [w]),
        _blob(1, C, R, good, [w + b"x"]),
        _blob(1, C, R, good, [w[1:]]),
        _blob(1, C, R, [(1, 0, M_START, 0, 0), good[1]], [w]),
        _blob(1, C, R, [(0, 8, M_START, 0, 0), good[1]], [w]),
        _blob(1, C, R, [(0, 0, M_BLOCK, 0, 0), good[1]], [w]),
        _blob(1, C, R, [(0, 0, M_START, 1, 0), good[1]], [w]),
        _blob(1, C, R, [(0, 0, M_START, 0, 1), good[1]], [b"a", w]),
        _blob(1, C, R, [good[0], (0, 4000, M_BLOCK, 0, 0)], []),
        _blob(1, C, R, [good[0], (R + 1, 4000, M_BLOCK, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 0, M_BLOCK, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 8 * C, M_BLOCK, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 4000, 4, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 4000, M_START, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 4000, M_BLOCK, 2, 0)], []),
        _blob(1, C, R, [good[0], (1000, 4000, M_MEMBER, 0, 10)], [w[-10:]]),
        _blob(1, C, R, [good[0], (1000, 4001, M_MEMBER, 0, 0)], []),
        _blob(0, C, R, [good[0], (1000, 4000, M_MEMBER, 0, 0)], []),
        _blob(1, C, R, [good[0], (1000, 4000, M_STORED, 0, 0)], []),
        _blob(1, C, R, [good[0], (100, 4000, M_BLOCK, 0, 101)], [want[:101]]),
        _blob(1, C, R, [good[0], (40000, 4000, M_BLOCK, 0, 32769)], [want[40000 - 32769:40000]]),
        _blob(1, C, R, good + [(1000, 5000, M_BLOCK, 0, 0)], [w]),
        _blob(1, C, R, good + [(2000, 4000, M_BLOCK, 0, 0)], [w]),
        _blob(1, C, R, [], []),
    ]
    for i, b in enumerate(cases):
        assert _refused(sctx, b), i


def test_extract_refusals(sctx):
    raw = corpus.gen_text(100000, 596, 14).tobytes()
    comp = _compress(raw, "zlib", 6)
    ix, blob, pts, want = _build(sctx, comp, "zlib", 0)
    L, h = sctx.lib, sctx.h
    src = np.frombuffer(comp, dtype=np.uint8)
    out = np.zeros(64, dtype=np.uint8)
    one, zero = np.array([5], dtype=np.uint64), np.array([0], dtype=np.uint64)
    got, st = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint32)
    args = lambda **k: dict(dict(ix=ix.h, comp=src.ctypes.data, clen=len(comp), off=one.ctypes.data, ln=one.ctypes.data, flags=0), **k)

    def call(a):
        return L.zwz_index_extract(h, a["ix"], a["comp"], a["clen"], 1, a["off"], a["ln"], out.ctypes.data, zero.ctypes.data, got.ctypes.data,
                                   st.ctypes.data, a["flags"])

    assert call(args()) == 0 and out[:5].tobytes() == raw[5:10]
    assert call(args(clen=len(comp) - 1)) == E_ARG
    assert call(args(ix=None)) == E_ARG
    assert call(args(comp=None)) == E_ARG
    assert call(args(off=None)) == E_ARG
    assert call(args(flags=1)) == E_ARG
    assert call(args(flags=CAREFUL | 4)) == E_ARG
    past = np.array([len(raw) - 4], dtype=np.uint64)
    assert call(args(off=past.ctypes.data)) == E_ARG
    huge = np.array([(1 << 64) - 2], dtype=np.uint64)
    assert call(args(off=one.ctypes.data, ln=huge.ctypes.data)) == E_ARG
    # an index of another context
    other = zwz_b200.Context(0, library=sctx.lib)
    try:
        ox = other.load_index(blob)
        assert call(args(ix=ox.h)) == E_ARG
        ox.close()
    finally:
        other.close()
    # points more than 4 GiB of output apart: a piece that would decode 4 GiB or more from its point is refused before any launch
    R = 5 << 30
    far = sctx.load_index(_blob(2, len(comp), R, [(0, 0, M_START, 0, 0), (R - 1000, 4000, M_BLOCK, 0, 0)], []))
    n0 = sctx.launches
    for a, n in ((4 << 30, 10), (0, R - 1000), ((4 << 30) - 5, 10)):
        with pytest.raises(zwz_b200.ZwzError):
            far.extract_device(1, len(comp), [a], [n], 1, [0])
    assert sctx.launches == n0
    far.close()


def test_other_stream_same_length(sctx):
    """A stream of the same length that is not the one indexed: valid statuses, no fault, nothing written outside the ranges."""
    raw = corpus.gen_text(150000, 596, 15).tobytes()
    comp = _compress(raw, "gzip", 6)
    ix, blob, pts, want = _build(sctx, comp, "gzip", 0)
    rng = np.random.default_rng(16)
    others = [bytes(rng.integers(0, 256, len(comp), dtype=np.uint8)), _compress(corpus.gen_struct(150000, 596, 3).tobytes(), "gzip", 6)]
    bad = bytearray(comp)
    for _ in range(20):
        bad[int(rng.integers(10, len(bad)))] ^= 1 << int(rng.integers(0, 8))
    others.append(bytes(bad))
    off = rng.integers(0, len(want), 60).astype(np.uint64)
    ln = np.minimum(rng.integers(0, 20000, 60).astype(np.uint64), len(want) - off)
    for o in others:
        o = (o + bytes(len(comp)))[:len(comp)]
        for flags in (0, CAREFUL):
            data, oo, got, st = ix.extract(o, off, ln, flags=flags)
            assert set(st.tolist()) <= {END, TRUNC, BAD} and (got <= ln).all()


# ---- GPU: full sizes ----
@pytest.mark.gpu
def test_gpu_text_gzip6_index(cuda_ctx):
    import shutil
    import subprocess
    raw = corpus.gen_text(256 << 20, 596, 1).tobytes()
    comp = gzip.compress(raw, 6) if shutil.which("gzip") is None else \
        subprocess.run(["gzip", "-6", "-c"], input=raw, capture_output=True, check=True).stdout
    out, st, ix = cuda_ctx.inflate_stream_index(comp, format="gzip")
    o2, s2 = cuda_ctx.inflate_stream(comp, format="gzip")
    assert (st, s2) == (END, END) and out.tobytes() == o2.tobytes() == raw
    assert ix.npoints > 100
    rng = np.random.default_rng(17)
    R = len(raw)
    for n, size in ((10000, 4096), (64, 16 << 20)):
        off = rng.integers(0, R - size, n).astype(np.uint64)
        data, oo, got, st = ix.extract(comp, off, np.full(n, size, dtype=np.uint64))
        assert (st == END).all() and (got == size).all()
        v = memoryview(raw)
        for i in range(n):
            assert data[int(oo[i]):int(oo[i]) + size].tobytes() == v[int(off[i]):int(off[i]) + size], i
    data, oo, got, st = ix.extract(comp, [0], [R])
    assert (int(st[0]), int(got[0])) == (END, R) and data.tobytes() == raw
    ix2 = cuda_ctx.load_index(ix.save())
    off = rng.integers(0, R - 4096, 100).astype(np.uint64)
    a, b = ix.extract(comp, off, np.full(100, 4096, dtype=np.uint64), flags=CAREFUL), ix2.extract(comp, off, np.full(100, 4096, dtype=np.uint64))
    assert a[0].tobytes() == b[0].tobytes() and (a[3] == END).all() and (b[3] == END).all()


@pytest.mark.gpu
def test_gpu_over_4gib_index(cuda_ctx):
    """The stream of test_gpu_over_4gib (more than 4 GiB of output), indexed without output; ranges above 4 GiB checked by CRC-32."""
    period = corpus.gen_text(1 << 14, 596, 7).tobytes()
    n = (4 << 30) // len(period) + 64
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    comp = bytearray()
    for _ in range(n):
        comp += co.compress(period)
    comp += co.flush()
    total = n * len(period)
    dc = cuda_ctx.malloc_device(len(comp))
    do = cuda_ctx.malloc_device(64 << 20)
    try:
        cuda_ctx.h2d(dc, np.frombuffer(bytes(comp), dtype=np.uint8))
        rl, st, ix = cuda_ctx.inflate_stream_index_device(dc, len(comp), None, total, format="gzip")
        assert (rl, st) == (total, END) and ix.raw_len == total
        rng = np.random.default_rng(18)
        size = 1 << 18
        off = np.concatenate([rng.integers(4 << 30, total - size, 30), [total - size, (4 << 30) - 100]]).astype(np.uint64)
        oo = (np.arange(len(off)) * size).astype(np.uint64)
        got, st = ix.extract_device(dc, len(comp), off, np.full(len(off), size, dtype=np.uint64), do, oo)
        assert (st == END).all() and (got == size).all()
        crc = cuda_ctx.crc32_batch_device(do, oo, np.full(len(off), size, dtype=np.uint32))
        rep = period * (size // len(period) + 2)
        for i, a in enumerate(off):
            s = int(a) % len(period)
            assert int(crc[i]) == zlib.crc32(rep[s:s + size]), i
        ix.close()
    finally:
        cuda_ctx.free_device(dc)
        cuda_ctx.free_device(do)
