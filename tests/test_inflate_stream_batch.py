"""Many gzip, zlib and raw DEFLATE streams in one call (zwz_inflate_stream_batch*): every stream must decode exactly as system zlib
and as a zwz_inflate_stream call of its own (bytes, status, and OUTPUT_FULL's size), whatever its neighbours are. The emulator runs
use 4 KiB spans, so that streams of a few hundred KB are cut into dozens of spans."""
import ctypes as C
import gzip
import random
import zlib

import numpy as np
import pytest

import zwz_b200
from test_inflate_stream import _ref, _stats
from tools import corpus

END, TRUNC, BAD, FULL = zwz_b200.STREAM_END, zwz_b200.STREAM_TRUNCATED, zwz_b200.STREAM_BAD, zwz_b200.STREAM_OUTPUT_FULL
WBITS = {"gzip": 31, "zlib": 15, "raw": -15}
E_ARG = -3


@pytest.fixture(scope="module")
def sctx(emu_ctx):
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    yield emu_ctx
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 0)


def _compress(raw, fmt, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, WBITS[fmt], 8, strategy)
    return co.compress(raw) + co.flush()


def _pack(streams):
    off = np.zeros(len(streams), dtype=np.uint64)
    if streams:
        off[1:] = np.cumsum([len(s) for s in streams])[:-1]
    return b"".join(streams), off, np.array([len(s) for s in streams], dtype=np.uint64)


def _check_batch(ctx, streams, fmt, single=True):
    """the batch against system zlib and, with `single`, against one inflate_stream call per stream"""
    comp, off, ln = _pack(streams)
    out, out_off, st = ctx.inflate_stream_batch(comp, off, ln, format=fmt)
    assert len(st) == len(streams)
    for i, s in enumerate(streams):
        got = out[int(out_off[i]):int(out_off[i + 1])].tobytes()
        want, wst = _ref(s, fmt)
        assert (int(st[i]), len(got)) == (wst, len(want)), i
        assert got == want, i
        if single:
            one, ost = ctx.inflate_stream(s, format=fmt)
            assert (ost, one.tobytes()) == (int(st[i]), got), i
    return out, out_off, st


def _mixed(fmt, seed):
    rng = random.Random(seed)
    streams = [b""]
    for i, n in enumerate([0, 1, 100, 3000, 9000, 40000, 150000, 700]):
        gen = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random][i % 4]
        streams.append(_compress(gen(n, 596, seed + i).tobytes(), fmt, rng.choice([0, 1, 6, 9])))
    return streams


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_mixed_sizes(sctx, fmt):
    """0 bytes, streams inside one span, and streams of dozens of spans, in one batch"""
    _stats(sctx)
    _check_batch(sctx, _mixed(fmt, 3), fmt)


def test_about_a_hundred_spans(sctx):
    big = _compress(corpus.gen_text(1_500_000, 596, 8).tobytes(), "gzip", 6)
    assert len(big) > 90 * 4096
    _check_batch(sctx, [gzip.compress(b"x" * 5000), big, gzip.compress(b"")], "gzip", single=False)


def test_gzip_members_levels_strategies(sctx):
    parts = [corpus.gen_text(n, 596, i).tobytes() for i, n in enumerate([5000, 0, 4096, 30000, 0, 1, 20000])]
    multi = b"".join(gzip.compress(p, 6) for p in parts)
    streams = [multi, multi + b"garbage behind the last member", multi + b"\0" * 50,
               b"".join(gzip.compress(bytes([65 + i % 26]) * (i % 7)) for i in range(70))]  # more members than a span records
    raw = corpus.gen_text(60000, 596, 4).tobytes()
    streams += [_compress(raw, "gzip", lv) for lv in (0, 1, 6, 9)]
    streams += [_compress(raw, "gzip", 6, s) for s in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)]
    bg, _ = sctx.gzip_files(raw, np.array([0, len(raw)], dtype=np.uint64))  # BGZF
    streams.append(bg.tobytes())
    _check_batch(sctx, streams, "gzip")


def test_damage_stays_in_its_stream(sctx):
    a, b, c = (corpus.gen_text(40000, 596, i).tobytes() for i in range(3))
    good = gzip.compress(a) + gzip.compress(b)
    crc = bytearray(good)
    crc[-8] ^= 1
    isz = bytearray(good)
    isz[-4] ^= 1
    rng = random.Random(11)
    flips = []
    for _ in range(3):
        f = bytearray(good)
        f[rng.randrange(20, len(f) - 20)] ^= 1 << rng.randrange(8)
        flips.append(bytes(f))
    mates = [gzip.compress(c), _compress(c, "gzip", 1)]
    for bad in [bytes(crc), bytes(isz), good[:len(good) // 2], good[:-3]] + flips:
        _, _, st = _check_batch(sctx, [mates[0], bad, mates[1]], "gzip", single=False)
        assert (int(st[0]), int(st[2])) == (END, END)
    _, _, st = _check_batch(sctx, [bytes(crc), bytes(isz)], "gzip", single=False)
    assert list(st) == [BAD, BAD]


def test_first_match_too_far_back_behind_a_neighbour(sctx):
    """A raw stream whose first symbol is a match, right behind a multi-span stream in the same wave: BAD at 0 bytes, as in a call
    of its own (its first span decodes with an empty window; test_scan_is_segmented_at_stream_starts covers the window scan)."""
    prev = _compress(corpus.gen_text(30000, 596, 1).tobytes(), "raw", 6)
    # one fixed block: length 3 distance 1 with nothing written yet, then end of block
    bits = []

    def put(v, n, rev=False):
        for k in range(n):
            bits.append((v >> (n - 1 - k)) & 1 if rev else (v >> k) & 1)
    put(1, 1)
    put(1, 2)
    put(1, 7, rev=True)        # length code 257: length 3
    put(0, 5, rev=True)        # distance code 0: distance 1
    put(0, 7, rev=True)        # end of block
    far = bytes(sum(b << k for k, b in enumerate(bits[i:i + 8])) for i in range(0, len(bits), 8))
    want, wst = _ref(far, "raw")
    assert (wst, len(want)) == (BAD, 0)
    _check_batch(sctx, [prev, far, prev, far], "raw")


def test_scan_is_segmented_at_stream_starts(sctx):
    """The window scan composes every map with all maps before it, across streams. A stream's first map holds bytes and INVALID
    only (its span starts at the stream's header with an empty window), so the resolved windows from that map on must not depend
    on anything before it: change every map in front of it and they stay the same."""
    rng = np.random.default_rng(3)
    W = 32768

    def ref_map(lo_invalid):  # a map with window references (256 + k), bytes and INVALID
        m = rng.integers(0, 256 + W, W).astype(np.uint16)
        m[rng.random(W) < lo_invalid] = 0xFFFF
        return m
    first = rng.integers(0, 256, W).astype(np.uint16)  # a stream's first span: bytes ...
    first[:5000] = 0xFFFF                                # ... and INVALID for what lies before the stream
    tail = [ref_map(0.01) for _ in range(5)]
    results = []
    for seed in (1, 2):
        rng2 = np.random.default_rng(seed)
        head = [rng2.integers(0, 256 + W, W).astype(np.uint16) for _ in range(3)]  # the maps of the streams in front
        head[0][head[0] >= 256] = 0xFFFF  # map 0 holds no window references
        maps = np.concatenate(head + [first] + tail)
        sctx.lib.zwz_emu_win_scan(C.c_void_p(maps.ctypes.data), C.c_uint32(len(head) + 1 + len(tail)))
        results.append(maps[len(head) * W:].copy())
    assert np.array_equal(results[0], results[1])
    # and the stream's own windows are resolved through its first map: nothing is left to resolve
    assert ((results[0] < 256) | (results[0] == 0xFFFF)).all()


def test_output_full_does_not_depend_on_waves(sctx):
    """A damaged stream that does not fit its region: OUTPUT_FULL with the whole size, whether it fits one wave, is cut into
    several, or sits behind neighbours that move the wave boundaries."""
    a, b = (corpus.gen_text(100000, 596, 30 + i).tobytes() for i in range(2))
    g1 = bytearray(gzip.compress(a))
    g1[-8] ^= 1  # member 1's CRC
    bad = bytes(g1) + gzip.compress(b)
    stored = [_compress(corpus.gen_text(n, 596, 40).tobytes(), "gzip", 0) for n in (12000, 40000)]
    _, _, st = sctx.inflate_stream_batch(bad, [0], [len(bad)], format="gzip", out_caps=[150000])
    assert (list(st), list(sctx.last_needed)) == ([FULL], [200000])
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 1 << 20)
    try:
        for front in ([], stored[:1], stored[1:], stored):
            comp, off, ln = _pack(front + [bad])
            caps = [1 << 20] * len(front) + [150000]
            _, _, st = sctx.inflate_stream_batch(comp, off, ln, format="gzip", out_caps=caps)
            assert (int(st[-1]), int(sctx.last_needed[-1])) == (FULL, 200000), len(front)
            out, st1 = sctx.inflate_stream(bad, format="gzip", out_cap=150000)
            assert (st1, sctx.last_needed) == (FULL, 200000)
        # with room for it, the bad CRC is found across waves
        _, _, st = sctx.inflate_stream_batch(comp, off, ln, format="gzip")
        assert int(st[-1]) == BAD and int(sctx.last_needed[-1]) == 100000
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 0)


def test_false_candidates_repaired_together(sctx):
    raw = corpus.gen_text(200000, 596, 4).tobytes()
    inner = _compress(raw, "raw", 6)
    fake = b"".join(bytes([0, 0x34, 0x12, 0xcb, 0xed]) + bytes(300) for _ in range(100))
    streams = [_compress(inner + fake + raw[:20000], "gzip", 0), _compress(fake + inner, "gzip", 0)]
    for s in streams:
        _stats(sctx)
        sctx.inflate_stream(s, format="gzip")
        alone = _stats(sctx)
        assert alone[2] > 0, alone
    _stats(sctx)
    _check_batch(sctx, streams, "gzip", single=False)
    s = _stats(sctx)
    assert s[2] > 0, s
    # the rounds of both streams share launches: no more rounds than the longer chain of repairs, not their sum
    assert s[1] < 2 * max(1, alone[1]) + 2, s


@pytest.mark.parametrize("fmt", ["gzip", "zlib"])
def test_tiny_budget_waves(sctx, fmt):
    """waves cut inside streams and between them: the same results as one wave"""
    streams = _mixed(fmt, 5) + [_compress(b"\0" * 200000, fmt, 6)]
    comp, off, ln = _pack(streams)
    caps = [1 << 20] * len(streams)  # one call each: no second call for OUTPUT_FULL streams
    _stats(sctx)
    one = sctx.inflate_stream_batch(comp, off, ln, format=fmt, out_caps=caps)
    assert _stats(sctx)[5] == 1
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 300000)
    try:
        many = sctx.inflate_stream_batch(comp, off, ln, format=fmt, out_caps=caps)
        assert _stats(sctx)[5] > 5
        if fmt == "gzip":
            bad = bytearray(streams[-3])
            bad[-6] ^= 1  # the ISIZE of a stream that spans waves
            _check_batch(sctx, [streams[-4], bytes(bad), streams[-2]], fmt, single=False)
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 0)
    for x, y in zip(one, many):
        assert np.array_equal(x, y)


def test_output_full_and_guards(sctx):
    raws = [corpus.gen_text(n, 596, i).tobytes() for i, n in enumerate([30000, 5000, 70000, 0])]
    streams = [gzip.compress(r) for r in raws]
    comp, off, ln = _pack(streams)
    caps = [30000, 4000, 70000, 0]  # stream 1 does not fit
    out, out_off, st = sctx.inflate_stream_batch(comp, off, ln, format="gzip", out_caps=caps)
    assert list(st) == [END, FULL, END, END]
    assert list(sctx.last_needed) == [len(r) for r in raws]
    assert out[int(out_off[0]):int(out_off[1])].tobytes() == raws[0] and out[int(out_off[2]):int(out_off[3])].tobytes() == raws[2]
    # the raw C call, with guard bytes around every region
    G = 16
    regions = np.zeros(len(caps) + 1, dtype=np.uint64)
    for i, c in enumerate(caps):
        regions[i + 1] = regions[i] + c + G
    buf = np.full(int(regions[-1]) + G, 0xA7, dtype=np.uint8)
    # region i is buf[regions[i] + G .. regions[i] + G + cap], with a guard in front of it
    starts = np.array([int(regions[i]) + G for i in range(len(caps))] + [0], dtype=np.uint64)
    rl = np.zeros(len(caps), dtype=np.uint64)
    sts = np.zeros(len(caps), dtype=np.uint32)
    for i in range(len(caps)):  # one stream per call, each with its own out_off pair
        o = np.array([starts[i], starts[i] + caps[i]], dtype=np.uint64)
        sctx._check(sctx.lib.zwz_inflate_stream_batch(sctx.h, comp, off[i:].ctypes.data, ln[i:].ctypes.data, 1, buf.ctypes.data, o.ctypes.data,
                                                      rl[i:].ctypes.data, sts[i:].ctypes.data, zwz_b200.FORMAT_GZIP << 8))
    assert list(sts) == [END, FULL, END, END]
    for i in range(len(caps)):
        assert (buf[int(regions[i]):int(regions[i]) + G] == 0xA7).all(), i
    assert (buf[int(regions[-1]):] == 0xA7).all()


def test_guards_in_one_call(sctx):
    raws = [corpus.gen_text(n, 596, 20 + i).tobytes() for i, n in enumerate([30000, 5000, 70000, 9000])]
    streams = [gzip.compress(r) for r in raws]
    comp, off, ln = _pack(streams)
    caps = [30000, 4000, 70000, 9000]
    G = 16
    out_off = np.zeros(len(caps) + 1, dtype=np.uint64)
    for i, c in enumerate(caps):
        out_off[i + 1] = out_off[i] + c
    # regions back to back, a guard in front of the first and behind the last; OUTPUT_FULL's region must not spill over
    buf = np.full(int(out_off[-1]) + 2 * G, 0xA7, dtype=np.uint8)
    rl = np.zeros(len(caps), dtype=np.uint64)
    st = np.zeros(len(caps), dtype=np.uint32)
    sctx._check(sctx.lib.zwz_inflate_stream_batch(sctx.h, comp, off.ctypes.data, ln.ctypes.data, len(caps), buf.ctypes.data + G, out_off.ctypes.data,
                                                  rl.ctypes.data, st.ctypes.data, zwz_b200.FORMAT_GZIP << 8))
    assert list(st) == [END, FULL, END, END] and list(rl) == [len(r) for r in raws]
    assert (buf[:G] == 0xA7).all() and (buf[G + int(out_off[-1]):] == 0xA7).all()
    for i in (0, 2, 3):
        assert buf[G + int(out_off[i]):G + int(out_off[i]) + len(raws[i])].tobytes() == raws[i]


def test_repeats_empty_and_refusals(sctx):
    s = gzip.compress(corpus.gen_text(20000, 596, 2).tobytes())
    # the same bytes given twice, and overlapping ranges
    comp = s
    off = np.array([0, 0, 0], dtype=np.uint64)
    ln = np.array([len(s), len(s), 10], dtype=np.uint64)
    out, out_off, st = sctx.inflate_stream_batch(comp, off, ln, format="gzip")
    want, _ = _ref(s, "gzip")
    assert list(st[:2]) == [END, END] and int(st[2]) == TRUNC
    assert out[int(out_off[0]):int(out_off[1])].tobytes() == want == out[int(out_off[1]):int(out_off[2])].tobytes()
    # n == 0
    out, out_off, st = sctx.inflate_stream_batch(b"", [], [], format="gzip")
    assert len(st) == 0 and list(out_off) == [0]
    L = sctx.lib
    u64 = np.zeros(4, dtype=np.uint64)
    u32 = np.zeros(4, dtype=np.uint32)
    buf = np.zeros(64, dtype=np.uint8)
    p = buf.ctypes.data
    assert L.zwz_inflate_stream_batch(sctx.h, None, None, None, 0, None, None, None, None, 0) == 0
    # NULL pointers with n > 0
    assert L.zwz_inflate_stream_batch(sctx.h, None, u64.ctypes.data, u64.ctypes.data, 1, p, u64.ctypes.data, u64.ctypes.data, u32.ctypes.data, 0) == E_ARG
    assert L.zwz_inflate_stream_batch(sctx.h, p, u64.ctypes.data, u64.ctypes.data, 1, p, None, u64.ctypes.data, u32.ctypes.data, 0) == E_ARG
    # an unknown format
    assert L.zwz_inflate_stream_batch(sctx.h, p, u64.ctypes.data, u64.ctypes.data, 1, p, u64.ctypes.data, u64.ctypes.data, u32.ctypes.data, 7 << 8) == E_ARG
    # a stream of 4 GiB or more
    big = np.array([0, 0x1_0000_0000], dtype=np.uint64)
    assert L.zwz_inflate_stream_batch_device(sctx.h, p, big.ctypes.data, big[1:].ctypes.data, 1, p, u64.ctypes.data, u64.ctypes.data,
                                             u32.ctypes.data, 0, None) == E_ARG
    # a decreasing out_off
    dec = np.array([10, 5], dtype=np.uint64)
    z = np.zeros(2, dtype=np.uint64)
    assert L.zwz_inflate_stream_batch(sctx.h, p, z.ctypes.data, z.ctypes.data, 1, p, dec.ctypes.data, u64.ctypes.data, u32.ctypes.data, 0) == E_ARG


def test_host_and_device_agree(sctx):
    streams = _mixed("zlib", 9)
    comp, off, ln = _pack(streams)
    out, out_off, st = sctx.inflate_stream_batch(comp, off, ln, format="zlib")
    # the emulator's device memory is host memory
    caps = np.diff(out_off).astype(np.uint64)
    d_out = np.zeros(max(int(out_off[-1]), 1), dtype=np.uint8)
    cbuf = np.frombuffer(comp, dtype=np.uint8).copy()
    rl, dst = sctx.inflate_stream_batch_device(cbuf.ctypes.data, off, ln, d_out.ctypes.data, out_off, format="zlib")
    assert np.array_equal(dst, st) and np.array_equal(rl, caps)
    assert np.array_equal(d_out[:int(out_off[-1])], out)
    # NO_ADLER: an Adler-32 mismatch is not looked at
    bad = bytearray(streams[5])
    bad[-1] ^= 1
    comp2, off2, ln2 = _pack([streams[4], bytes(bad)])
    _, _, st2 = sctx.inflate_stream_batch(comp2, off2, ln2, format="zlib")
    _, _, st3 = sctx.inflate_stream_batch(comp2, off2, ln2, format="zlib", flags=zwz_b200.INFLATE_NO_ADLER)
    assert list(st2) == [END, BAD] and list(st3) == [END, END]


# ---- on the GPU ----
@pytest.mark.gpu
def test_gpu_log_uniform_gzip6(cuda_ctx):
    rng = np.random.default_rng(7)
    sizes = np.exp(rng.uniform(np.log(4096), np.log(16 << 20), 512)).astype(np.int64)
    base = corpus.gen_text((16 << 20) + 65536, 596, 7).tobytes()
    raws = [base[int(o):int(o) + int(s)] for o, s in zip(rng.integers(0, 65536, 512), sizes)]
    streams = []
    for r in raws:
        co = zlib.compressobj(6, zlib.DEFLATED, 31)
        streams.append(co.compress(r) + co.flush())
    comp, off, ln = _pack(streams)
    out, out_off, st = cuda_ctx.inflate_stream_batch(comp, off, ln, format="gzip")
    assert (st == END).all()
    for i, r in enumerate(raws):
        assert out[int(out_off[i]):int(out_off[i + 1])].tobytes() == r, i


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_gpu_c2_mix(cuda_ctx, fmt):
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    raws = [gens[i % 4](int(n), 596, i).tobytes() for i, n in enumerate(np.geomspace(1000, 8 << 20, 48))]
    streams = [_compress(r, fmt, 6) for r in raws]
    comp, off, ln = _pack(streams)
    out, out_off, st = cuda_ctx.inflate_stream_batch(comp, off, ln, format=fmt)
    assert (st == END).all()
    for i, r in enumerate(raws):
        assert out[int(out_off[i]):int(out_off[i + 1])].tobytes() == r, i
