"""One long stream inflated by the whole GPU (zwz_inflate_stream*): gzip files of any number of members, zlib and raw DEFLATE streams,
checked against system zlib. The emulator variants use spans of a few KiB, so that streams of a few hundred KB are cut into dozens
of spans and every path (false block candidates, slot overflow, member starts inside spans, windows resolved across spans) runs."""
import ctypes as C
import gzip
import random
import shutil
import subprocess
import zlib

import numpy as np
import pytest

import zlib_ref
import zwz_b200
from tools import corpus

END, TRUNC, BAD, FULL = zwz_b200.STREAM_END, zwz_b200.STREAM_TRUNCATED, zwz_b200.STREAM_BAD, zwz_b200.STREAM_OUTPUT_FULL
WBITS = {"gzip": 31, "zlib": 15, "raw": -15}
E_ARG = -3


@pytest.fixture(scope="module")
def sctx(emu_ctx):
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    yield emu_ctx
    emu_ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 0)


def _stats(ctx, reset=True):
    s = (C.c_uint64 * 8)()
    ctx.lib.zwz_emu_stream_stats(s, 1 if reset else 0)
    return list(s)


def _compress(raw, fmt, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, WBITS[fmt], 8, strategy)
    return co.compress(raw) + co.flush()


def _ref(comp, fmt):
    """System zlib over the whole input; gzip: members one after another, as gzip -d, stopping at the first that does not end
    cleanly -> (bytes, status)."""
    if fmt != "gzip":
        return zlib_ref.inflate_wbits(comp, WBITS[fmt], cap=1 << 24)
    out, pos, first = b"", 0, True
    while True:
        if not first and (len(comp) - pos < 2 or comp[pos:pos + 2] != b"\x1f\x8b"):
            return out, END
        d = zlib.decompressobj(31)
        try:
            part = d.decompress(comp[pos:])
        except zlib.error:
            part, st = zlib_ref.inflate_wbits(comp[pos:], 31, cap=1 << 24)
            return out + part, st
        if not d.eof:
            part, st = zlib_ref.inflate_wbits(comp[pos:], 31, cap=1 << 24)
            return out + part, st
        out += part
        pos = len(comp) - len(d.unused_data)
        first = False


def _check(ctx, comp, fmt, cap=None):
    want, wst = _ref(comp, fmt)
    # room for everything the stream decodes to before a check value fails (OUTPUT_FULL is decided before the check values)
    out, st = ctx.inflate_stream(comp, format=fmt, out_cap=cap if cap is not None else max(len(want), 1 << 22) + 64)
    assert (st, len(out)) == (wst, len(want))
    assert out.tobytes() == want
    return want


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_round_trip_levels(sctx, fmt, level):
    raw = corpus.gen_text(200000, 596, level).tobytes()
    assert _check(sctx, _compress(raw, fmt, level), fmt) == raw


@pytest.mark.parametrize("strategy", [zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED])
def test_round_trip_strategies(sctx, strategy):
    raw = corpus.gen_text(150000, 596, 3).tobytes()
    assert _check(sctx, _compress(raw, "gzip", 6, strategy), "gzip") == raw


@pytest.mark.parametrize("cls", ["T", "S", "B", "J", "R"])
def test_round_trip_classes(sctx, cls):
    gen = {"T": corpus.gen_text, "S": corpus.gen_struct, "B": getattr(corpus, "gen_binary", corpus.gen_struct),
           "J": corpus.gen_jpeg_like, "R": corpus.gen_random}[cls]
    raw = gen(120000, 596, 11).tobytes()
    assert _check(sctx, _compress(raw, "gzip", 6), "gzip") == raw


@pytest.mark.skipif(shutil.which("gzip") is None, reason="no gzip binary")
def test_gzip_binary(sctx):
    raw = corpus.gen_text(250000, 596, 5).tobytes()
    comp = subprocess.run(["gzip", "-6", "-c"], input=raw, capture_output=True, check=True).stdout
    assert _check(sctx, comp, "gzip") == raw


def test_multi_member(sctx):
    parts = [corpus.gen_text(n, 596, i).tobytes() for i, n in enumerate([5000, 0, 4096, 4095, 30000, 0, 1, 20000])]
    comp = b"".join(gzip.compress(p, 6) for p in parts)
    assert _check(sctx, comp, "gzip") == b"".join(parts)
    # trailing zero padding and garbage are ignored, as gzip -d does
    _check(sctx, comp + b"\0" * 100, "gzip")
    _check(sctx, comp + b"\x1f", "gzip")
    _check(sctx, comp + b"garbage behind the last member", "gzip")


def test_many_small_members(sctx):
    parts = [bytes([65 + i % 26]) * (i % 7) for i in range(100)]  # more members than one span records
    comp = b"".join(gzip.compress(p) for p in parts)
    assert _check(sctx, comp, "gzip") == b"".join(parts)


def test_bgzf(sctx):
    raw = corpus.gen_text(300000, 596, 9).tobytes()
    gz, goff = sctx.gzip_files(raw, np.array([0, len(raw)], dtype=np.uint64))
    out, st = sctx.inflate_stream(gz.tobytes(), format="gzip")
    back, _, gst = sctx.gunzip_files(gz, goff)
    assert (st, out.tobytes()) == (int(gst[0]), back.tobytes())


def test_bad_member_check(sctx):
    a, b, c = (corpus.gen_text(20000, 596, i).tobytes() for i in range(3))
    gb = bytearray(gzip.compress(b))
    crc = bytearray(gb)
    crc[-8] ^= 1
    isz = bytearray(gb)
    isz[-4] ^= 1
    for mid in (crc, isz):
        comp = gzip.compress(a) + bytes(mid) + gzip.compress(c)
        out, st = sctx.inflate_stream(comp, format="gzip", out_cap=100000)
        assert (st, out.tobytes()) == (BAD, a + b)


def test_false_candidates(sctx):
    # a stored gzip whose payload is itself raw DEFLATE with dynamic blocks, and stored-block look-alikes (LEN, ~NLEN)
    raw = corpus.gen_text(400000, 596, 4).tobytes()
    inner = _compress(raw, "raw", 6)
    fake = b"".join(bytes([0, 0x34, 0x12, 0xcb, 0xed]) + bytes(300) for _ in range(200))
    payload = inner + fake + raw[:50000]
    _stats(sctx)
    assert _check(sctx, _compress(payload, "gzip", 0), "gzip") == payload
    s = _stats(sctx)
    assert s[2] > 0, s  # spans decoded again from their predecessor's stop


def test_stored_padding_not_zero(sctx):
    """A span decoded again from a stored block's key sits in the header's padding, which RFC 1951 leaves arbitrary: the block type
    must not be read from it. A stored block holding a LEN / ~NLEN look-alike, then a final stored block whose header byte is
    0xF9 (BFINAL 1, BTYPE 00, padding 11111)."""
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 1024)
    try:
        for hdr in (0x01, 0xF9):
            p1 = bytearray(corpus.gen_text(3000, 596, 1).tobytes())
            p1[1500:1505] = bytes([0, 0x10, 0x00, 0xef, 0xff])  # a stored header byte and LEN 16 / NLEN
            p2 = corpus.gen_text(600, 596, 2).tobytes()
            comp = bytes([0]) + len(p1).to_bytes(2, "little") + (len(p1) ^ 0xFFFF).to_bytes(2, "little") + bytes(p1)
            comp += bytes([hdr]) + len(p2).to_bytes(2, "little") + (len(p2) ^ 0xFFFF).to_bytes(2, "little") + p2
            assert _check(sctx, comp, "raw") == bytes(p1) + p2
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)


@pytest.mark.parametrize("fmt", ["gzip", "zlib"])
def test_waves(sctx, fmt):
    """A scratch budget far below the stream's output: many waves, each handing on its window and the running check value; the
    output must equal that of one wave."""
    raw = corpus.gen_text(300000, 596, 6).tobytes() + b"\0" * 100000 + corpus.gen_struct(100000, 596, 7).tobytes()
    comp = _compress(raw, fmt, 6)
    if fmt == "gzip":
        comp += gzip.compress(raw[:70000]) + gzip.compress(b"")
        raw += raw[:70000]
    _stats(sctx)
    one, st1 = sctx.inflate_stream(comp, format=fmt, out_cap=len(raw))
    assert _stats(sctx)[5] == 1
    sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 40000)
    try:
        many, st = sctx.inflate_stream(comp, format=fmt, out_cap=len(raw))
        assert _stats(sctx)[5] > 3
        # a bad CRC in the last member is still found across waves
        if fmt == "gzip":
            bad = bytearray(comp)
            bad[-28] ^= 1  # CRC of the 70000-byte member
            _check(sctx, bytes(bad), fmt)
    finally:
        sctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, 0)
    assert (st, st1) == (END, END) and many.tobytes() == one.tobytes() == raw


@pytest.mark.parametrize("raw", [b"\0" * 3_000_000, b"".join((b"\0" * 200000) + corpus.gen_text(5000, 596, i).tobytes() for i in range(6))],
                         ids=["zeros", "zeros-text"])
def test_slot_overflow(sctx, raw):
    _stats(sctx)
    assert _check(sctx, _compress(raw, "gzip", 6), "gzip") == raw
    assert _stats(sctx)[3] > 0


class _Bits:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v, n):
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def put_rev(self, code, n):  # Huffman codes go MSB first
        self.put(int(format(code, f"0{n}b")[::-1], 2), n)

    def bytes(self):
        return bytes(self.out) + (bytes([self.acc]) if self.n else b"")


def _fixed_lit(b, x):
    if x < 144:
        b.put_rev(0x30 + x, 8)
    else:
        b.put_rev(0x190 + x - 144, 9)


def _fixed_block(b, lits, dist, last=True):
    """Fixed block: the literals, then one match of length 3 at `dist`, then end of block."""
    b.put(1 if last else 0, 1)
    b.put(1, 2)
    for x in lits:
        _fixed_lit(b, x)
    b.put_rev(1, 7)  # length 3 (symbol 257)
    d = dist - 1
    if d < 4:
        b.put_rev(d, 5)
    else:
        nb = d.bit_length() - 1
        sym = 2 * nb + ((d >> (nb - 1)) & 1)
        b.put_rev(sym, 5)
        b.put(d & ((1 << (nb - 1)) - 1), nb - 1)
    b.put_rev(0, 7)


def test_distance_too_far_back(sctx):
    # in span 0
    b = _Bits()
    _fixed_block(b, b"abcd", 5)
    _check(sctx, b.bytes(), "raw")
    # a member that starts inside one span and refers back past its start from the next span
    lead = gzip.compress(corpus.gen_text(9000, 596, 1).tobytes(), 6)
    body = corpus.gen_text(6000, 596, 2).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    head = co.compress(body) + co.flush(zlib.Z_FULL_FLUSH)
    tail = _Bits()
    _fixed_block(tail, b"xy", 7000)
    deflated = head + tail.bytes()
    member = gzip.compress(b"")[:10] + deflated + b"\0" * 8
    # the member starts in one 4 KiB span, the reference that reaches back past its start lies in a later one
    assert (len(lead) + 10) // 4096 < (len(lead) + 10 + len(head)) // 4096
    _check(sctx, lead + member, "gzip")
    # right after a member start
    b = _Bits()
    _fixed_block(b, b"", 1)
    _check(sctx, lead + gzip.compress(b"")[:10] + b.bytes() + b"\0" * 8, "gzip")


def test_truncation_and_corruption(sctx):
    rng = random.Random(5)
    raws = [corpus.gen_text(60000, 596, 3).tobytes(), corpus.gen_struct(40000, 596, 4).tobytes()]
    streams = [("gzip", gzip.compress(raws[0], 6) + gzip.compress(raws[1], 6)), ("zlib", _compress(raws[0], "zlib")),
               ("raw", _compress(raws[1], "raw", 9))]
    for fmt, comp in streams:
        for _ in range(6):
            _check(sctx, comp[:rng.randrange(len(comp))], fmt)
            bad = bytearray(comp)
            bad[rng.randrange(len(bad))] ^= 1 << rng.randrange(8)
            _check(sctx, bytes(bad), fmt)


def test_output_full(sctx):
    raw = corpus.gen_text(100000, 596, 8).tobytes()
    comp = gzip.compress(raw) + gzip.compress(raw)
    out, st = sctx.inflate_stream(comp, format="gzip", out_cap=len(raw))
    assert (st, len(out), sctx.last_needed) == (FULL, 0, 2 * len(raw))
    # nothing written: a canary in device memory stays
    dc, do = sctx.malloc_device(len(comp)), sctx.malloc_device(len(raw))
    try:
        sctx.h2d(dc, np.frombuffer(comp, dtype=np.uint8))
        canary = np.full(len(raw), 0x5a, dtype=np.uint8)
        sctx.h2d(do, canary)
        n, st = sctx.inflate_stream_device(dc, len(comp), do, len(raw), format="gzip")
        assert (n, st) == (2 * len(raw), FULL)
        back = np.empty_like(canary)
        sctx.d2h(back, do)
        assert (back == canary).all()
    finally:
        sctx.free_device(dc)
        sctx.free_device(do)
    # the Python form retries once with the size reported (ISIZE of the last member is too small here)
    out, st = sctx.inflate_stream(comp, format="gzip")
    assert (st, out.tobytes()) == (END, raw + raw)


def test_refusals(sctx):
    comp = _compress(b"hello hello hello", "zlib")
    out = np.zeros(64, dtype=np.uint8)
    rl, st = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint32)
    src = np.frombuffer(comp, dtype=np.uint8)
    L = sctx.lib
    assert L.zwz_inflate_stream(sctx.h, None, len(comp), out.ctypes.data, 64, rl.ctypes.data, st.ctypes.data, 0) == E_ARG
    assert L.zwz_inflate_stream(sctx.h, src.ctypes.data, len(comp), None, 64, rl.ctypes.data, st.ctypes.data, 0) == E_ARG
    assert L.zwz_inflate_stream(sctx.h, src.ctypes.data, len(comp), out.ctypes.data, 64, None, st.ctypes.data, 0) == E_ARG
    assert L.zwz_inflate_stream(sctx.h, src.ctypes.data, len(comp), out.ctypes.data, 64, rl.ctypes.data, st.ctypes.data, 7 << 8) == E_ARG
    co = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, zdict=b"hello")
    fd = co.compress(b"hello hello") + co.flush()
    out, st = sctx.inflate_stream(fd, format="zlib", out_cap=100)
    assert (st, len(out)) == (BAD, 0)


def _scan_ref(maps):
    """Serial reference of the window resolution: window behind span i = map_i applied to the window behind span i - 1."""
    win, res = None, []
    for m in maps:
        w = m.copy()
        ref = (m >= 256) & (m != 0xFFFF)
        w[ref] = 0xFFFF if win is None else win[m[ref] - 256]
        res.append(w)
        win = w
    return res


def test_window_scan_against_serial(sctx):
    """The log-depth scan must equal the serial chain: streams whose spans refer far back into resolved windows."""
    rng = np.random.default_rng(3)
    # long-distance repeats across many spans: every span's window comes through a chain of earlier ones
    base = corpus.gen_text(30000, 596, 2).tobytes()
    raw = b"".join(base[i * 997 % 20000:][:8000] for i in range(40))
    for fmt in ("raw", "gzip"):
        assert _check(sctx, _compress(raw, fmt, 9), fmt) == raw
    # win_scan_kernel itself on random maps with INVALID entries
    maps = [rng.integers(0, 256 + 32768, 32768).astype(np.int64) for _ in range(11)]
    for m in maps:
        m[rng.integers(0, 32768, 100)] = 0xFFFF
    maps[0][(maps[0] >= 256) & (maps[0] != 0xFFFF)] = 0xFFFF  # nothing comes before the first span
    ser = _scan_ref(maps)
    buf = np.ascontiguousarray(np.stack(maps).astype(np.uint16))
    sctx.lib.zwz_emu_win_scan(C.c_void_p(buf.ctypes.data), C.c_uint32(len(maps)))
    for i, b in enumerate(ser):
        assert (buf[i] == b).all(), i


# ---- GPU: full sizes ----
@pytest.mark.gpu
def test_gpu_text_gzip6(cuda_ctx):
    raw = corpus.gen_text(256 << 20, 596, 1).tobytes()
    comp = gzip.compress(raw, 6) if shutil.which("gzip") is None else \
        subprocess.run(["gzip", "-6", "-c"], input=raw, capture_output=True, check=True).stdout
    out, st = cuda_ctx.inflate_stream(comp, format="gzip")
    assert st == END and out.tobytes() == raw


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
def test_gpu_round_trip(cuda_ctx, fmt):
    raw = corpus.gen_text(8 << 20, 596, 2).tobytes() + b"\0" * (1 << 20) + corpus.gen_struct(4 << 20, 596, 3).tobytes()
    for level in (1, 6, 9):
        assert _check(cuda_ctx, _compress(raw, fmt, level), fmt) == raw


@pytest.mark.gpu
def test_gpu_over_4gib(cuda_ctx):
    """A stream that decodes to more than 4 GiB (which the batch call cannot take), checked by CRC-32 against the source."""
    period = corpus.gen_text(1 << 14, 596, 7).tobytes()  # inside the window: long matches, quick to compress
    n = (4 << 30) // len(period) + 64
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    comp = bytearray()
    crc = 0
    for _ in range(n):
        comp += co.compress(period)
        crc = zlib.crc32(period, crc)
    comp += co.flush()
    total = n * len(period)
    dc, do = cuda_ctx.malloc_device(len(comp)), cuda_ctx.malloc_device(total)
    try:
        cuda_ctx.h2d(dc, np.frombuffer(bytes(comp), dtype=np.uint8))
        rl, st = cuda_ctx.inflate_stream_device(dc, len(comp), do, total, format="gzip")
        assert (rl, st) == (total, END)
        pieces = np.arange(0, total, 1 << 26, dtype=np.uint64)
        lens = np.minimum(1 << 26, total - pieces).astype(np.uint32)
        got = 0
        for p, c in zip(pieces, cuda_ctx.crc32_batch_device(do, pieces, lens)):
            got = _crc_combine(got, int(c), int(min(1 << 26, total - int(p))))
        assert got == crc
    finally:
        cuda_ctx.free_device(dc)
        cuda_ctx.free_device(do)


def _crc_combine(c1, c2, len2):
    """zlib's crc32_combine over GF(2)."""
    def mult(a, b):
        p = 0
        for i in range(32):
            if a & (0x80000000 >> i):
                p ^= b
            b = (b >> 1) ^ (0xEDB88320 if b & 1 else 0)
        return p
    x2n, p = [], 1 << 30
    for _ in range(32):
        x2n.append(p)
        p = mult(p, p)
    p, k = 0x80000000, 3
    while len2:
        if len2 & 1:
            p = mult(x2n[k & 31], p)
        len2 >>= 1
        k += 1
    return mult(p, c1) ^ c2
