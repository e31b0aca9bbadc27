"""One gzip, zlib or raw DEFLATE stream fed piece by piece (zwz_inflater, Context.decompressobj): over every way of cutting the input
into calls, the bytes handed out and the terminal status must equal system zlib and one inflate_stream call on the whole input. The
emulator runs use 4 KiB spans, so that a feed of a few KB already holds several spans and the resume points fall everywhere."""
import ctypes as C
import gzip
import random
import struct
import zlib

import numpy as np
import pytest

import zwz_b200
from test_inflate_stream import _ref, _stats
from test_inflate_stream_batch import _compress, _mixed
from tools import corpus

END, TRUNC, BAD, MORE = zwz_b200.STREAM_END, zwz_b200.STREAM_TRUNCATED, zwz_b200.STREAM_BAD, zwz_b200.STREAM_MORE
E_ARG = -3


@pytest.fixture(scope="module")
def sctx(emu_ctx):
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    yield emu_ctx
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 0)


def _feed_all(ctx, comp, fmt, cuts, out_cap=None, flags=0):
    """comp cut at the positions `cuts`, one call per piece, then an empty final call; every call drains with out_cap bytes at most
    (None: as much as is queued). Returns (bytes, terminal status, inflater)."""
    f = ctx.decompressobj(fmt, flags)
    L, h = ctx.lib, f.h
    n = np.zeros(1, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint32)
    buf = np.empty(1 << 21, dtype=np.uint8)
    parts = []
    bounds = [0] + sorted(cuts) + [len(comp)]
    comp = np.frombuffer(comp, dtype=np.uint8)

    def call(piece, final):
        while True:
            cap = len(buf) if out_cap is None else out_cap
            ctx._check(L.zwz_inflater_feed(h, piece.ctypes.data if piece.size else None, piece.size, final, buf.ctypes.data, cap, n.ctypes.data,
                                           st.ctypes.data))
            parts.append(buf[:int(n[0])].tobytes())
            piece = piece[:0]
            if int(st[0]) != MORE or f.queued_out == 0:
                return int(st[0])
    for a, b in zip(bounds[:-1], bounds[1:]):
        s = call(comp[a:b], 0)
        if s != MORE:  # ended: the rest is ignored
            assert s in (END, BAD), s
    s = call(comp[:0], 1)
    return b"".join(parts), s, f


def _check_cuts(ctx, comp, fmt, cuts, out_cap=None, ref=None):
    want, wst = ref if ref is not None else _ref(comp, fmt)
    got, st, f = _feed_all(ctx, comp, fmt, cuts, out_cap)
    assert (st, len(got)) == (wst, len(want)), (cuts, out_cap)
    assert got == want, (cuts, out_cap)
    f.close()


# ---- a small stream with every kind of piece ----
def _body(seed):
    """raw DEFLATE: a stored block with non-zero padding bits, a fixed block, dynamic blocks, the final block (each piece ends on a
    byte boundary: Z_SYNC_FLUSH)"""
    rng = random.Random(seed)
    a = corpus.gen_text(400, 596, seed).tobytes()
    b = corpus.gen_text(600, 596, seed + 1).tobytes()
    c = corpus.gen_text(1500, 596, seed + 2).tobytes()
    stored = bytes(rng.randrange(256) for _ in range(100))
    out = bytes([0xF8]) + struct.pack("<HH", len(stored), len(stored) ^ 0xFFFF) + stored  # BFINAL 0, BTYPE 00, padding 11111
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_FIXED)
    out += co.compress(a) + co.flush(zlib.Z_SYNC_FLUSH)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    out += co.compress(b) + co.flush(zlib.Z_SYNC_FLUSH)
    co = zlib.compressobj(9, zlib.DEFLATED, -15)
    out += co.compress(c) + co.flush()
    return out, stored + a + b + c


def _gzip_member(body, raw, header=True):
    if not header:
        return b"\x1f\x8b\x08\x00\0\0\0\0\0\xff" + body + struct.pack("<II", zlib.crc32(raw), len(raw) & 0xFFFFFFFF)
    h = b"\x1f\x8b\x08" + bytes([0x02 | 0x04 | 0x08]) + b"\1\2\3\4\0\3"  # FHCRC, FEXTRA, FNAME
    h += struct.pack("<H", 6) + b"AB\2\0xy" + b"name.txt\0"
    h += struct.pack("<H", zlib.crc32(h) & 0xFFFF)
    return h + body + struct.pack("<II", zlib.crc32(raw), len(raw) & 0xFFFFFFFF)


def _small(fmt):
    body, raw = _body(1)
    if fmt == "raw":
        return body
    if fmt == "zlib":
        return b"\x78\x9c" + body + struct.pack(">I", zlib.adler32(raw))
    body2, raw2 = _body(5)
    return _gzip_member(body, raw) + gzip.compress(b"second member " * 20) + _gzip_member(body2, raw2, header=False)


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_every_split_point(sctx, fmt):
    comp = _small(fmt)
    ref = _ref(comp, fmt)
    assert ref[1] == END
    one, ost = sctx.inflate_stream(comp, format=fmt)
    assert (ost, one.tobytes()) == (ref[1], ref[0])
    for k in range(len(comp) + 1):
        _check_cuts(sctx, comp, fmt, [k], ref=ref)


def test_every_split_point_of_a_prefix(sctx):
    """final given at a prefix: TRUNCATED with zlib's bytes, cut in two anywhere"""
    comp = _small("gzip")
    for end in range(0, len(comp), 97):
        pre = comp[:end]
        ref = _ref(pre, "gzip")
        for k in range(0, end + 1, 7):
            _check_cuts(sctx, pre, "gzip", [k], ref=ref)


# ---- seeded random splits over the corpora of the batch tests ----
def _random_cuts(rng, n, how):
    if how == "bytes":
        return list(range(1, n))
    if how == "big":
        return [rng.randrange(n + 1)] if n else []
    cuts, p = [], 0
    while True:
        p += rng.choice([1, 2, 13, 100, 1000, 4096, 9000, 30000])
        if p >= n:
            return cuts
        cuts.append(p)


def _corpora(fmt):
    streams = _mixed(fmt, 3)
    raw = corpus.gen_text(60000, 596, 4).tobytes()
    streams += [_compress(raw, fmt, lv) for lv in (0, 1, 6, 9)]
    streams += [_compress(raw, fmt, 6, s) for s in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)]
    if fmt == "gzip":
        multi = b"".join(gzip.compress(bytes([65 + i % 26]) * (i % 7)) for i in range(70))  # more members than a span records
        streams += [multi, multi + b"garbage behind the last member", multi + b"\0" * 50]
    else:
        streams += [streams[-1] + b"trailing bytes", streams[-1] + b"\0" * 50]
    return streams


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_random_splits(sctx, fmt):
    rng = random.Random(17)
    for comp in _corpora(fmt):
        ref = _ref(comp, fmt)
        if len(comp) <= 3000:  # 1-byte feeds: one decode per byte
            _check_cuts(sctx, comp, fmt, _random_cuts(rng, len(comp), "bytes"), rng.choice([1, 1000, None]), ref=ref)
        cuts = _random_cuts(rng, len(comp), "random")
        for cap in (1, 1000, None):
            if cap == 1 and len(ref[0]) > 70000:
                continue
            _check_cuts(sctx, comp, fmt, cuts, cap, ref=ref)
        _check_cuts(sctx, comp, fmt, _random_cuts(rng, len(comp), "big"), ref=ref)


def test_bgzf_and_a_hundred_spans(sctx):
    rng = random.Random(5)
    raw = corpus.gen_text(150000, 596, 6).tobytes()
    bg, _ = sctx.gzip_files(raw, np.array([0, len(raw)], dtype=np.uint64))
    big = _compress(corpus.gen_text(1_500_000, 596, 8).tobytes(), "gzip", 6)
    assert len(big) > 90 * 4096
    for comp in (bg.tobytes(), big):
        ref = _ref(comp, "gzip")
        for how in ("random", "big"):
            _check_cuts(sctx, comp, "gzip", _random_cuts(rng, len(comp), how), ref=ref)
    _check_cuts(sctx, big, "gzip", list(range(65536, len(big), 65536)), 1000)


# ---- errors ----
@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_truncated_and_flipped(sctx, fmt):
    rng = random.Random(23)
    comp = _compress(corpus.gen_text(80000, 596, 9).tobytes(), fmt, 6)
    if fmt == "gzip":
        comp = gzip.compress(b"first " * 1000) + comp
    for _ in range(6):
        end = rng.randrange(len(comp))
        pre = comp[:end]
        ref = _ref(pre, fmt)
        assert ref[1] != END or fmt == "gzip"
        for how in ("random", "big"):
            _check_cuts(sctx, pre, fmt, _random_cuts(rng, len(pre), how), ref=ref)
    for _ in range(6):
        bad = bytearray(comp)
        bad[rng.randrange(len(bad))] ^= 1 << rng.randrange(8)
        ref = _ref(bytes(bad), fmt)
        for how in ("random", "big"):
            _check_cuts(sctx, bytes(bad), fmt, _random_cuts(rng, len(bad), how), ref=ref)


def _bits_to_bytes(bits):
    bits = bits + [0] * (-len(bits) % 8)
    return bytes(sum(b << k for k, b in enumerate(bits[i:i + 8])) for i in range(0, len(bits), 8))


def _far_block(dist, final=1):
    """one fixed block: a match of length 3 at distance `dist`, then end of block"""
    bits = []

    def put(v, n, rev=False):
        for k in range(n):
            bits.append((v >> (n - 1 - k)) & 1 if rev else (v >> k) & 1)
    put(final, 1)
    put(1, 2)
    put(1, 7, rev=True)  # length code 257: length 3
    # distance code and extra bits (RFC 1951 3.2.5)
    base = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289,
            16385, 24577]
    code = max(i for i, b in enumerate(base) if b <= dist)
    put(code, 5, rev=True)
    extra = max(0, code // 2 - 1)
    put(dist - base[code], extra)
    put(0, 7, rev=True)  # end of block
    return _bits_to_bytes(bits)


def test_too_far_back_across_feeds(sctx):
    text = corpus.gen_text(5000, 596, 3).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    head = co.compress(text) + co.flush(zlib.Z_SYNC_FLUSH)
    for dist, wst in ((4000, END), (6000, BAD)):
        raw = head + _far_block(dist)
        ref = _ref(raw, "raw")
        assert ref[1] == wst
        for k in range(len(head) - 3, len(raw) + 1):
            _check_cuts(sctx, raw, "raw", [k], ref=ref)
    # a gzip member that reaches into the member before it
    first = gzip.compress(text)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    small = co.compress(b"0123456789") + co.flush(zlib.Z_SYNC_FLUSH)
    body = small + _far_block(100)
    member = b"\x1f\x8b\x08\x00\0\0\0\0\0\xff" + body + b"\0" * 8
    comp = first + member
    ref = _ref(comp, "gzip")
    assert ref[1] == BAD and len(ref[0]) == 5010
    for k in list(range(len(first) - 4, len(comp) + 1)) + [100, 2000]:
        _check_cuts(sctx, comp, "gzip", [k], ref=ref)


def test_check_values_across_feeds(sctx):
    raw = corpus.gen_text(120000, 596, 12).tobytes()
    good = gzip.compress(raw[:70000]) + gzip.compress(raw[70000:])
    crc = bytearray(good)
    crc[-8] ^= 1
    isz = bytearray(good)
    isz[-4] ^= 1
    z = bytearray(_compress(raw, "zlib", 6))
    z[-1] ^= 1
    for comp, fmt in ((bytes(crc), "gzip"), (bytes(isz), "gzip"), (bytes(z), "zlib")):
        ref = _ref(comp, fmt)
        assert ref[1] == BAD
        _check_cuts(sctx, comp, fmt, list(range(5000, len(comp), 5000)), ref=ref)
        _check_cuts(sctx, comp, fmt, list(range(5000, len(comp), 5000)), 777, ref=ref)
    # NO_ADLER skips the CRC-32, ISIZE is still checked
    got, st, _ = _feed_all(sctx, bytes(crc), "gzip", list(range(5000, len(crc), 5000)), flags=zwz_b200.INFLATE_NO_ADLER)
    assert (st, got) == (END, raw)
    got, st, _ = _feed_all(sctx, bytes(isz), "gzip", [len(isz) // 2], flags=zwz_b200.INFLATE_NO_ADLER)
    assert st == BAD


# ---- state stays bounded, feeds decode many spans ----
def test_pending_stays_bounded(sctx):
    raw = corpus.gen_text(400000, 596, 2).tobytes()
    comp = _compress(raw, "gzip", 6, zlib.Z_FIXED)  # no block candidates: one span per call
    piece = 20000
    f = sctx.decompressobj("gzip")
    out, most = [], 0
    for i in range(0, len(comp), piece):
        out.append(f.decompress(comp[i:i + piece]).tobytes())
        most = max(most, f.pending_in)
        assert f.queued_out == 0
    out.append(f.flush().tobytes())
    assert (f.status, f.eof, b"".join(out)) == (END, True, raw)
    # zlib's Z_FIXED blocks hold 16 K symbols: well under 64 KiB of compressed bytes
    assert 0 < most < piece + 65536, most
    assert (f.total_in, f.total_out, f.pending_in) == (len(comp), len(raw), 0)


def test_feeds_decode_many_spans(sctx):
    raw = corpus.gen_text(600000, 596, 3).tobytes()
    comp = _compress(raw, "gzip", 6)
    f = sctx.decompressobj("gzip")
    _stats(sctx)
    got, calls = [], 0
    for i in range(0, len(comp), 65536):
        got.append(f.decompress(comp[i:i + 65536]).tobytes())
        calls += 1
    s = _stats(sctx)
    got.append(f.flush().tobytes())
    assert b"".join(got) == raw and f.status == END
    # spans decoded: a span starts at every dynamic block header found (gzip -6 text: one every 20-30 KB), so a 64 KiB feed
    # decodes two or more
    assert calls >= 3 and s[0] >= 2 * calls, (s, calls)


# ---- the interface ----
def test_status_sequence_and_python_object(sctx):
    raw = corpus.gen_text(50000, 596, 4).tobytes()
    comp = gzip.compress(raw)
    with sctx.decompressobj("gzip") as d:
        a = d.decompress(comp[:1000])
        assert d.status == MORE and not d.eof
        b = d.decompress(comp[1000:])
        assert d.status == MORE  # gzip: another member may follow the trailer
        assert d.decompress(b"xy").size == 0 and d.status == END and d.eof  # not 1f 8b: the stream ended
        assert d.decompress(b"ignored after the end").size == 0 and d.status == END
        assert (a.tobytes() + b.tobytes()) == raw
        assert d.flush().size == 0 and d.status == END
    with sctx.decompressobj("zlib") as d:  # zlib and raw streams end at their last block
        assert d.decompress(zlib.compress(raw)).tobytes() == raw and d.status == END
    # truncated: MORE until final, then TRUNCATED, sticky
    d = sctx.decompressobj("zlib")
    z = zlib.compress(raw)
    part = d.decompress(z[:-10])
    assert d.status == MORE
    rest = d.flush()
    assert d.status == TRUNC
    want, wst = _ref(z[:-10], "zlib")
    assert (part.tobytes() + rest.tobytes(), wst) == (want, TRUNC)
    n = np.zeros(1, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint32)
    buf = np.zeros(16, dtype=np.uint8)
    assert sctx.lib.zwz_inflater_feed(d.h, None, 0, 1, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data) == 0
    assert (int(n[0]), int(st[0])) == (0, TRUNC)
    d.close()
    # Context.close frees open inflaters first
    import emu_lib
    c2 = emu_lib.emu_context()
    d2 = c2.decompressobj("raw")
    d2.decompress(_compress(raw, "raw"))
    c2.close()
    assert d2.h is None


def test_refusals_leave_the_state(sctx):
    L = sctx.lib
    raw = corpus.gen_text(30000, 596, 5).tobytes()
    comp = gzip.compress(raw)
    n = np.zeros(1, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint32)
    buf = np.zeros(1 << 16, dtype=np.uint8)
    src = np.frombuffer(comp, dtype=np.uint8)
    h = C.c_void_p()
    assert L.zwz_inflater_new(sctx.h, 7 << 8, C.byref(h)) == E_ARG
    assert L.zwz_inflater_new(sctx.h, 0, None) == E_ARG
    assert L.zwz_inflater_feed(None, src.ctypes.data, 10, 0, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data) == E_ARG
    f = sctx.decompressobj("gzip")
    p = src.ctypes.data
    assert L.zwz_inflater_feed(f.h, p, 100, 0, buf.ctypes.data, 16, None, st.ctypes.data) == E_ARG
    assert L.zwz_inflater_feed(f.h, p, 100, 0, buf.ctypes.data, 16, n.ctypes.data, None) == E_ARG
    assert L.zwz_inflater_feed(f.h, None, 100, 0, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data) == E_ARG
    assert L.zwz_inflater_feed(f.h, p, 100, 0, None, 16, n.ctypes.data, st.ctypes.data) == E_ARG
    # pending input that would reach 0xffffff00 bytes (refused before anything is read)
    assert L.zwz_inflater_feed_device(f.h, p, 0xffffff00, 0, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data, None) == E_ARG
    assert f.total_in == 0 and f.pending_in == 0
    assert L.zwz_inflater_feed(f.h, p, 1000, 0, buf.ctypes.data, 0, n.ctypes.data, st.ctypes.data) == 0
    pend = f.pending_in
    assert 0 < pend <= 1000
    assert L.zwz_inflater_feed_device(f.h, p, 0xffffff00 - pend, 0, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data, None) == E_ARG
    assert (f.total_in, f.pending_in) == (1000, pend)
    got = f.decompress(src[1000:]).tobytes()
    rest = f.flush()
    assert f.status == END
    assert L.zwz_inflater_feed(f.h, p, 1, 0, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data) == E_ARG  # input after final
    assert L.zwz_inflater_feed(f.h, None, 0, 1, buf.ctypes.data, 16, n.ctypes.data, st.ctypes.data) == 0 and int(st[0]) == END
    assert f.total_in == len(comp)
    assert got + rest.tobytes() == raw  # the first call handed out nothing (out_cap 0): its output stayed queued


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_host_and_device_forms_agree(sctx, fmt):
    rng = random.Random(31)
    comp = _compress(corpus.gen_text(90000, 596, 6).tobytes(), fmt, 6)
    cuts = _random_cuts(rng, len(comp), "random")
    host, hst, _ = _feed_all(sctx, comp, fmt, cuts, 5000)
    # the emulator's device memory is host memory
    f = sctx.decompressobj(fmt)
    src = np.frombuffer(comp, dtype=np.uint8).copy()
    out = np.zeros(5000, dtype=np.uint8)
    parts = []
    bounds = [0] + cuts + [len(comp)]
    for i, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
        final = i == len(bounds) - 2
        n, st = f.feed_device(src.ctypes.data + a, b - a, out.ctypes.data, len(out), final=final)
        parts.append(out[:n].tobytes())
        while st == MORE and f.queued_out:
            n, st = f.feed_device(0, 0, out.ctypes.data, len(out), final=final)
            parts.append(out[:n].tobytes())
    assert (b"".join(parts), st) == (host, hst)
    f.close()


# ---- on the GPU ----
def _gpu_feed(ctx, comp, fmt, rng, lo, hi):
    """comp fed in random pieces of lo..hi bytes through the device form; returns (bytes, status)"""
    import torch
    f = ctx.decompressobj(fmt)
    src = torch.from_numpy(np.frombuffer(comp, dtype=np.uint8).copy()).cuda()
    out = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    parts, p = [], 0
    while True:
        k = min(len(comp) - p, rng.randrange(lo, hi + 1))
        final = p + k == len(comp)
        n, st = f.feed_device(src.data_ptr() + p, k, out.data_ptr(), out.numel(), final=final)
        parts.append(out[:n].cpu().numpy().tobytes())
        while st == MORE and f.queued_out:
            n, st = f.feed_device(0, 0, out.data_ptr(), out.numel(), final=final)
            parts.append(out[:n].cpu().numpy().tobytes())
        p += k
        if final:
            break
    f.close()
    return b"".join(parts), st


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["text", "c2"])
def test_gpu_256mib_random_feeds(cuda_ctx, kind):
    size = 256 << 20
    if kind == "text":
        raw = corpus.gen_text(size, 596, 1).tobytes()
    else:
        gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
        raw = b"".join(gens[i % 4](size // 16, 596, i).tobytes() for i in range(16))
    comp = gzip.compress(raw, 6)
    one, ost = cuda_ctx.inflate_stream(comp, format="gzip")
    assert ost == END and one.tobytes() == raw
    got, st = _gpu_feed(cuda_ctx, comp, "gzip", random.Random(3), 1 << 20, 256 << 20)
    assert (st, got == raw) == (END, True)


def _big_unit(seed, n):
    """raw DEFLATE of n seeded bytes ending in Z_FULL_FLUSH (byte-aligned, no reference behind it): repeatable"""
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    raw = b"".join(gens[i % 4](n // 4, 596, seed + i).tobytes() for i in range(4))
    co = zlib.compressobj(1, zlib.DEFLATED, -15)
    return raw, co.compress(raw) + co.flush(zlib.Z_FULL_FLUSH)


def _check_repeated(ctx, pieces, raw, total_raw, feed):
    """feed the generated pieces into one inflater; every delivered byte is compared with the repeated raw unit"""
    f = ctx.decompressobj("gzip")
    out = np.empty(1 << 30, dtype=np.uint8)
    unit = np.frombuffer(raw, dtype=np.uint8)
    n = np.zeros(1, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint32)
    pos, most_pending, most_queued, comp_len = 0, 0, 0, 0
    L, h = ctx.lib, f.h

    def check(k):
        nonlocal pos
        o = 0
        while o < k:
            u = pos % len(unit)
            m = min(k - o, len(unit) - u)
            assert np.array_equal(out[o:o + m], unit[u:u + m]), pos
            o += m
            pos += m
    for piece, final in pieces:
        comp_len += len(piece)
        a = np.frombuffer(piece, dtype=np.uint8)
        ctx._check(L.zwz_inflater_feed(h, a.ctypes.data if a.size else None, a.size, 1 if final else 0, out.ctypes.data, out.size, n.ctypes.data,
                                       st.ctypes.data))
        most_pending = max(most_pending, f.pending_in)
        most_queued = max(most_queued, f.queued_out + int(n[0]))
        check(int(n[0]))
        while int(st[0]) == MORE and f.queued_out:
            ctx._check(L.zwz_inflater_feed(h, None, 0, 1 if final else 0, out.ctypes.data, out.size, n.ctypes.data, st.ctypes.data))
            check(int(n[0]))
    assert int(st[0]) == END
    assert pos == total_raw and f.total_out == total_raw and f.total_in == comp_len
    f.close()
    return comp_len, most_pending, most_queued


def _repeated_member_pieces(raw, unit, reps, feed):
    """one gzip member whose body is `unit` repeated, then a final empty fixed block, CRC-32 and ISIZE mod 2^32; cut into feeds"""
    crc = 0
    for _ in range(reps):
        crc = zlib.crc32(raw, crc)
    tail = b"\x03\x00" + struct.pack("<II", crc, (len(raw) * reps) & 0xFFFFFFFF)
    stream = [b"\x1f\x8b\x08\x00\0\0\0\0\0\xff"] + [unit] * reps + [tail]
    buf = b""
    for i, s in enumerate(stream):
        buf += s
        while len(buf) >= feed:
            yield buf[:feed], False
            buf = buf[feed:]
    yield buf, True


@pytest.mark.gpu
def test_gpu_one_member_over_4_5_gib(cuda_ctx):
    raw, unit = _big_unit(11, 64 << 20)
    reps = -(-((9 << 29) + 4096) // len(unit))  # >= 4.5 GiB compressed
    comp_len, pend, queued = _check_repeated(cuda_ctx, _repeated_member_pieces(raw, unit, reps, 256 << 20), raw, len(raw) * reps, 256 << 20)
    assert comp_len >= 9 << 29


@pytest.mark.gpu
def test_gpu_many_members_over_4_5_gib(cuda_ctx):
    raw, unit = _big_unit(12, 64 << 20)
    member = b"\x1f\x8b\x08\x00\0\0\0\0\0\xff" + unit + b"\x03\x00" + struct.pack("<II", zlib.crc32(raw), len(raw) & 0xFFFFFFFF)
    reps = -(-((9 << 29) + 4096) // len(member))

    def pieces(feed=200 << 20):
        buf = b""
        for _ in range(reps):
            buf += member
            while len(buf) >= feed:
                yield buf[:feed], False
                buf = buf[feed:]
        yield buf, True
    comp_len, _, _ = _check_repeated(cuda_ctx, pieces(), raw, len(raw) * reps, 200 << 20)
    assert comp_len == reps * len(member) >= 9 << 29
