"""One long input deflated into a single gzip, zlib or raw DEFLATE stream (zwz_deflate_stream*, Context.compress_stream) and the
streaming deflater (zwz_deflater, Context.compressobj). Every output is decoded by system zlib; the deflater's bytes must equal the
one-shot call's for every way of cutting the input. The emulator runs use chunks of 1 KiB and 4 KiB, so that inputs of a few KB
cross many chunk boundaries and windows span several chunks."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

import zwz_b200
from tools import corpus

E_ARG, E_CAPACITY = -3, -5
WBITS = {"gzip": 31, "zlib": 15, "raw": -15}
FMT = {"zlib": 0, "gzip": 1, "raw": 2}
TUNE_C = zwz_b200.TUNE_DEFLATE_STREAM_CHUNK_BYTES
KINDS = {"text": corpus.gen_text, "struct": corpus.gen_struct, "jpeg": corpus.gen_jpeg_like, "random": corpus.gen_random,
         "zeros": lambda n, s, u: np.zeros(n, dtype=np.uint8)}


@pytest.fixture
def sctx(emu_ctx):
    emu_ctx.tune(TUNE_C, 1024)
    yield emu_ctx
    emu_ctx.tune(TUNE_C, 0)


def _unzip(comp, fmt):
    """system zlib: exactly one stream that ends, nothing behind it"""
    d = zlib.decompressobj(WBITS[fmt])
    out = d.decompress(comp)
    assert d.eof and d.unused_data == b"", fmt
    return out


def _feed(ctx, fmt, pieces, level=0, out_cap=None):
    """the deflater over (data, flush) pieces; every call is drained with out_cap bytes at most (None: everything queued). Returns the
    bytes handed out by each call, joined per piece."""
    f = ctx.compressobj(fmt, level)
    L, h = ctx.lib, f.h
    n = np.zeros(1, dtype=np.uint64)
    buf = np.empty(1 << 20, dtype=np.uint8)
    outs = []
    for data, flush in pieces:
        a = np.frombuffer(data, dtype=np.uint8)
        got = []
        while True:
            cap = len(buf) if out_cap is None else out_cap
            ctx._check(L.zwz_deflater_feed(h, a.ctypes.data if a.size else None, a.size, flush, buf.ctypes.data, cap, n.ctypes.data))
            got.append(buf[:int(n[0])].tobytes())
            a = a[:0]
            if not f.queued_out:
                break
        outs.append(b"".join(got))
    assert f.queued_out == 0 and f.total_in == sum(len(d) for d, _ in pieces) and f.total_out == sum(map(len, outs))
    f.close()
    return outs


@pytest.mark.parametrize("fmt", ["gzip", "zlib", "raw"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_round_trip(sctx, fmt, level):
    C_ = 1024
    for kind, gen in KINDS.items():
        for n in (0, 1, C_ - 1, C_, C_ + 1, 5 * C_):
            raw = gen(n, 596, 3).tobytes() if n else b""
            comp = sctx.compress_stream(raw, fmt, level)
            assert _unzip(comp, fmt) == raw, (kind, n)
            if n in (C_ + 1, 5 * C_):
                one, st = sctx.inflate_stream(comp, format=fmt)
                assert st == zwz_b200.STREAM_END and one.tobytes() == raw
                d = sctx.decompressobj(fmt)
                assert d.decompress(comp).tobytes() + d.flush().tobytes() == raw and d.status == zwz_b200.STREAM_END
                d.close()


def test_round_trip_4k_chunks_and_levels(emu_ctx):
    emu_ctx.tune(TUNE_C, 4096)
    try:
        mix = b"".join(g(3000, 596, i).tobytes() for i, g in enumerate(KINDS.values()))
        for fmt in WBITS:
            for level in (0, 9):
                for n in (4095, 4096, 4097, 3 * 4096, len(mix)):
                    raw = mix[:n]
                    assert _unzip(emu_ctx.compress_stream(raw, fmt, level), fmt) == raw
    finally:
        emu_ctx.tune(TUNE_C, 0)


def test_empty_input_is_zlibs_bytes(sctx):
    assert sctx.compress_stream(b"", "raw") == b"\x03\x00"
    assert sctx.compress_stream(b"", "zlib") == zlib.compress(b"") == bytes.fromhex("789c030000000001")
    gz = sctx.compress_stream(b"", "gzip")
    assert gz == bytes.fromhex("1f8b08000000000000ff") + b"\x03\x00" + bytes(8) and len(gz) == 20
    for fmt in WBITS:
        assert b"".join(_feed(sctx, fmt, [(b"", zwz_b200.FINISH)])) == sctx.compress_stream(b"", fmt)


def test_default_chunk_crosses_64k(emu_ctx):
    raw = corpus.gen_text(200_000, 596, 5).tobytes()
    for fmt in WBITS:
        assert _unzip(emu_ctx.compress_stream(raw, fmt), fmt) == raw


def test_window_is_used(sctx):
    # 700-byte random blocks, each repeated 2 500 bytes later: every repeat is more than a chunk (1 KiB) but less than 32 KiB back
    parts = []
    for i in range(8):  # text, not noise: noise stretches are not searched against the window
        blk = corpus.gen_text(700, 596, 20 + i).tobytes()
        parts += [blk, corpus.gen_text(1800, 596, 40 + i).tobytes(), blk]
    raw = b"".join(parts)
    comp = sctx.compress_stream(raw, "raw")
    assert _unzip(comp, "raw") == raw
    off = np.arange(0, len(raw), 1024, dtype=np.uint64)
    ln = np.minimum(1024, len(raw) - off).astype(np.uint32)
    packed, _, _ = sctx.deflate_batch(raw, off, ln, format="raw")
    assert len(comp) < 0.8 * len(packed), (len(comp), len(packed))
    # a match at distance 32 768 across a chunk boundary: 3 000 bytes repeated from the window's first byte on
    x = corpus.gen_struct(32768, 596, 9).tobytes()
    raw = x + x[:3000]
    for fmt in WBITS:
        comp = sctx.compress_stream(raw, fmt)
        assert _unzip(comp, fmt) == raw
        assert len(comp) < len(sctx.compress_stream(x, fmt)) + 300


def test_deflater_equals_one_shot(sctx):
    rng = random.Random(11)
    raw = b"".join(g(2500, 596, i).tobytes() for i, g in enumerate(KINDS.values())) * 2
    for fmt in WBITS:
        for level in (0, 6):
            want = sctx.compress_stream(raw, fmt, level)
            for trial in range(4):
                cuts = sorted(rng.sample(range(1, len(raw)), rng.randrange(1, 12)))
                b = [0] + cuts + [len(raw)]
                pieces = [(raw[x:y], zwz_b200.NO_FLUSH) for x, y in zip(b[:-1], b[1:])] + [(b"", zwz_b200.FINISH)]
                out_cap = (None, 1, 1000, None)[trial]
                assert b"".join(_feed(sctx, fmt, pieces, level, out_cap)) == want, (fmt, level, cuts, out_cap)
            # the last piece may come with FINISH itself
            assert b"".join(_feed(sctx, fmt, [(raw[:3000], 0), (raw[3000:], zwz_b200.FINISH)], level)) == want


def test_deflater_one_byte_feeds(sctx):
    raw = corpus.gen_text(2600, 596, 8).tobytes()
    for fmt in WBITS:
        pieces = [(raw[i:i + 1], zwz_b200.NO_FLUSH) for i in range(len(raw))] + [(b"", zwz_b200.FINISH)]
        outs = _feed(sctx, fmt, pieces)
        assert b"".join(outs) == sctx.compress_stream(raw, fmt)
        co = sctx.compressobj(fmt)
        for i in range(len(raw)):
            co.compress(raw[i:i + 1])
            assert co.pending_in <= 1024  # a chunk is compressed once one more byte has arrived
        co.close()


def test_sync_flush(sctx):
    raw = corpus.gen_text(9000, 596, 9).tobytes()
    cuts = [0, 5, 1500, 1500, 2048, 4000, 7777, 9000]
    for fmt in WBITS:
        pieces = [(raw[a:b], zwz_b200.SYNC_FLUSH) for a, b in zip(cuts[:-1], cuts[1:])] + [(b"", zwz_b200.FINISH)]
        outs = _feed(sctx, fmt, pieces)
        d = zlib.decompressobj(WBITS[fmt])
        got = b""
        for k, o in enumerate(outs[:-1]):
            assert o.endswith(b"\x00\x00\xff\xff")
            got += d.decompress(o)
            assert got == raw[:cuts[k + 1]], (fmt, k)
        got += d.decompress(outs[-1])
        assert got == raw and d.eof and d.unused_data == b""
    # a sync flush with nothing pending writes the empty stored block, as zlib does
    a = _feed(sctx, "raw", [(b"", zwz_b200.SYNC_FLUSH), (b"", zwz_b200.FINISH)])
    assert a == [b"\x00\x00\x00\xff\xff", b"\x03\x00"]


def test_full_flush_starts_a_fresh_window(sctx):
    base = corpus.gen_text(6000, 596, 10).tobytes()
    raw = base + base  # the second half would copy from the first if the window survived
    for fmt in WBITS:
        outs = _feed(sctx, fmt, [(raw[:6000], zwz_b200.FULL_FLUSH), (raw[6000:], zwz_b200.FINISH)])
        assert _unzip(b"".join(outs), fmt) == raw
        d = zlib.decompressobj(-15)  # the bytes after the full flush alone, as raw DEFLATE with an empty window
        assert d.decompress(outs[1]) == raw[6000:] and d.eof
        assert len(d.unused_data) == {"gzip": 8, "zlib": 4, "raw": 0}[fmt]  # the trailer
    # deterministic: the output depends on the flush points only, not on how the input between them was cut
    a = _feed(sctx, "zlib", [(raw[:100], 0), (raw[100:6000], zwz_b200.FULL_FLUSH), (raw[6000:7000], 0), (raw[7000:], zwz_b200.FINISH)])
    b = _feed(sctx, "zlib", [(raw[:6000], zwz_b200.FULL_FLUSH), (raw[6000:], zwz_b200.FINISH)])
    assert b"".join(a) == b"".join(b)


def test_bound_and_capacity(sctx):
    L = sctx.lib
    for n in (0, 1, 1023, 1025, 7000):
        raw = corpus.gen_random(n, 596, 4).tobytes() if n else b""
        bound = int(L.zwz_deflate_stream_bound(n))
        assert bound == zwz_b200.deflate_stream_bound(n)
        for fmt in WBITS:
            for level in range(10):
                assert len(sctx.compress_stream(raw, fmt, level)) <= bound, (n, fmt, level)
            comp = sctx.compress_stream(raw, fmt)
            a = np.frombuffer(raw + b"\0", dtype=np.uint8)
            out = np.zeros(bound, dtype=np.uint8)
            got = C.c_uint64()
            rc = L.zwz_deflate_stream(sctx.h, a.ctypes.data, n, out.ctypes.data, len(comp) - 1, C.byref(got), 0, FMT[fmt])
            assert rc == E_CAPACITY and got.value == len(comp)
            d_in, d_out = sctx.malloc_device(n + 64), sctx.malloc_device(bound)
            try:
                if n:
                    sctx.h2d(d_in, a[:n])
                rc = L.zwz_deflate_stream_device(sctx.h, d_in, n, d_out, len(comp) - 1, C.byref(got), 0, FMT[fmt], None)
                assert rc == E_CAPACITY and got.value == len(comp)
            finally:
                sctx.free_device(d_in)
                sctx.free_device(d_out)


def test_device_forms(sctx):
    raw = corpus.gen_struct(5000, 596, 6).tobytes()
    a = np.frombuffer(raw, dtype=np.uint8)
    for fmt in WBITS:
        want = sctx.compress_stream(raw, fmt, 6)
        d_in = sctx.malloc_device(len(raw) + 64)
        d_out = sctx.malloc_device(zwz_b200.deflate_stream_bound(len(raw)))
        try:
            sctx.h2d(d_in, a)
            n = sctx.compress_stream_device(d_in, len(raw), d_out, zwz_b200.deflate_stream_bound(len(raw)), fmt, 6)
            got = np.zeros(n, dtype=np.uint8)
            sctx.d2h(got, d_out)
            assert got.tobytes() == want
            # the deflater's device form, fed in three pieces with out_cap 700
            f = sctx.compressobj(fmt, 6)
            parts, cuts = [], [0, 1000, 3100, len(raw)]
            buf = np.zeros(700, dtype=np.uint8)
            for k in range(3):
                flush = zwz_b200.FINISH if k == 2 else zwz_b200.NO_FLUSH
                p = f.feed_device(d_in + cuts[k], cuts[k + 1] - cuts[k], d_out, 700, flush)
                while True:
                    sctx.d2h(buf[:p], d_out) if p else None
                    parts.append(buf[:p].tobytes())
                    if not f.queued_out:
                        break
                    p = f.feed_device(0, 0, d_out, 700, flush)
            assert f.eof and b"".join(parts) == want
            f.close()
        finally:
            sctx.free_device(d_in)
            sctx.free_device(d_out)


def test_refusals(sctx):
    L = sctx.lib
    h = C.c_void_p()
    n = C.c_uint64()
    assert L.zwz_deflater_new(sctx.h, 0, 3, C.byref(h)) == E_ARG
    assert L.zwz_deflater_new(sctx.h, 0, 0, None) == E_ARG
    buf = np.zeros(64, dtype=np.uint8)
    assert L.zwz_deflate_stream(sctx.h, None, 5, buf.ctypes.data, 64, C.byref(n), 0, 0) == E_ARG
    assert L.zwz_deflate_stream(sctx.h, buf.ctypes.data, 5, buf.ctypes.data, 64, C.byref(n), 0, 7) == E_ARG
    assert L.zwz_deflate_stream(sctx.h, buf.ctypes.data, 5, buf.ctypes.data, 64, None, 0, 0) == E_ARG
    assert L.zwz_deflate_stream_device(sctx.h, None, 5, None, 0, C.byref(n), 0, 0, None) == E_ARG
    for v in (1, 1023, 65536):
        assert L.zwz_ctx_tune(sctx.h, TUNE_C, v) == E_ARG
    f = sctx.compressobj("zlib")
    fh = f.h
    assert L.zwz_deflater_feed(fh, None, 3, 0, buf.ctypes.data, 64, C.byref(n)) == E_ARG
    assert L.zwz_deflater_feed(fh, buf.ctypes.data, 3, 1, buf.ctypes.data, 64, C.byref(n)) == E_ARG  # Z_PARTIAL_FLUSH is not taken
    assert L.zwz_deflater_feed(fh, buf.ctypes.data, 3, 5, buf.ctypes.data, 64, C.byref(n)) == E_ARG
    assert L.zwz_deflater_feed(fh, buf.ctypes.data, 3, 0, None, 64, C.byref(n)) == E_ARG
    assert L.zwz_deflater_feed(fh, buf.ctypes.data, 3, 0, buf.ctypes.data, 64, None) == E_ARG
    assert f.total_in == 0
    # a flush asked for while output is queued waits for the queue, and takes no input until it is done
    big = corpus.gen_text(3000, 596, 1).tobytes()
    a = np.frombuffer(big, dtype=np.uint8)
    assert L.zwz_deflater_feed(fh, a.ctypes.data, a.size, 0, buf.ctypes.data, 1, C.byref(n)) == 0 and n.value == 1
    first = buf[:1].tobytes()
    assert f.queued_out > 0 and f.pending_in == 3000 - 2048
    assert L.zwz_deflater_feed(fh, None, 0, 2, buf.ctypes.data, 0, C.byref(n)) == 0 and n.value == 0
    assert L.zwz_deflater_feed(fh, a.ctypes.data, 1, 0, buf.ctypes.data, 1, C.byref(n)) == E_ARG
    assert f.total_in == len(big)
    rest = f.flush(zwz_b200.FINISH)
    assert L.zwz_deflater_feed(fh, a.ctypes.data, 1, 0, buf.ctypes.data, 64, C.byref(n)) == E_ARG  # input after FINISH
    assert f.eof and zlib.decompress(first + rest) == big
    f.close()


@pytest.mark.parametrize("fmt", ["text", "c2"])
def test_ratio_against_zlib_and_bgzf(emu_ctx, fmt):
    """a few MiB through the emulator at the default chunk size: at most 1.03 x whole-input zlib -6; on text smaller than BGZF"""
    size = 2 << 20
    if fmt == "text":
        raw = corpus.gen_text(size, 596, 1).tobytes()
    else:
        gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
        raw = b"".join(gens[i % 4](size // 16, 596, i).tobytes() for i in range(16))
    comp = emu_ctx.compress_stream(raw, "gzip")
    assert _unzip(comp, "gzip") == raw
    z6 = len(zlib.compress(raw, 6))
    assert len(comp) <= 1.03 * z6, (len(comp), z6)
    if fmt == "text":
        gz, _ = emu_ctx.gzip_files(raw, np.array([0, len(raw)], dtype=np.uint64))
        assert len(comp) < len(gz), (len(comp), len(gz))


# ---- on the GPU ----
def _corpus(kind, size):
    if kind == "text":
        return corpus.gen_text(size, 596, 1).tobytes()
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    return b"".join(gens[i % 4](size // 16, 596, i).tobytes() for i in range(16))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["text", "c2"])
def test_gpu_256mib_all_formats(cuda_ctx, kind):
    import torch
    raw = _corpus(kind, 256 << 20)
    src = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    cap = zwz_b200.deflate_stream_bound(len(raw))
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    z6 = len(zlib.compress(raw, 6))
    for fmt in WBITS:
        host = cuda_ctx.compress_stream(raw, fmt)
        assert _unzip(host, fmt) == raw
        assert len(host) <= 1.03 * z6, (fmt, len(host), z6)
        n = cuda_ctx.compress_stream_device(src.data_ptr(), len(raw), out.data_ptr(), cap, fmt)
        assert out[:n].cpu().numpy().tobytes() == host


@pytest.mark.gpu
def test_gpu_deflater_random_feeds(cuda_ctx):
    import torch
    raw = _corpus("c2", 256 << 20)
    want = cuda_ctx.compress_stream(raw, "zlib")
    src = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    out = torch.empty(zwz_b200.deflate_stream_bound(len(raw)), dtype=torch.uint8, device="cuda")
    rng = random.Random(5)
    f = cuda_ctx.compressobj("zlib")
    parts, p = [], 0
    while True:
        k = min(len(raw) - p, rng.randrange(1, 64 << 20))
        flush = zwz_b200.FINISH if p + k == len(raw) else zwz_b200.NO_FLUSH
        n = f.feed_device(src.data_ptr() + p, k, out.data_ptr(), out.numel(), flush)
        parts.append(out[:n].cpu().numpy().tobytes())
        p += k
        if flush == zwz_b200.FINISH:
            break
    assert f.queued_out == 0 and b"".join(parts) == want
    f.close()
    assert zlib.decompress(want) == raw


@pytest.mark.gpu
def test_gpu_deflater_over_4_5_gib(cuda_ctx):
    """a gzip stream of more than 4.5 GiB of input (ISIZE wraps), fed in 256 MiB pieces, read back by streaming CPU zlib"""
    unit = np.frombuffer(_corpus("c2", 256 << 20), dtype=np.uint8)
    reps = 19  # 4.75 GiB
    f = cuda_ctx.compressobj("gzip", 1)
    d = zlib.decompressobj(31)
    pos = 0
    crc = 0

    def check(b):
        nonlocal pos
        o = 0
        while o < len(b):
            u = pos % unit.size
            m = min(len(b) - o, unit.size - u)
            assert b[o:o + m] == unit[u:u + m].tobytes(), pos
            o += m
            pos += m
    for r in range(reps):
        crc = zlib.crc32(unit, crc)
        comp = f.compress(unit) if r + 1 < reps else f.compress(unit) + f.flush(zwz_b200.FINISH)
        while comp:
            check(d.decompress(comp, 1 << 28))
            comp = d.unconsumed_tail
    assert d.eof and d.unused_data == b"" and pos == unit.size * reps
    total = unit.size * reps
    assert total > 9 << 29 and f.total_in == total
    f.close()


def test_passes_do_not_change_the_bytes(sctx):
    """1 MiB sub-batches: a pass holds about 45 chunks of 1 KiB with their window records, so 150 KB take four passes, each packed
    behind the last; the bytes are those of one pass"""
    raw = b"".join(g(30000, 596, i).tobytes() for i, g in enumerate(KINDS.values()))
    want = {fmt: sctx.compress_stream(raw, fmt) for fmt in WBITS}
    sctx.tune(zwz_b200.Context.TUNE_DEFLATE_SUBBATCH_BYTES, 1 << 20)
    try:
        for fmt in WBITS:
            got = sctx.compress_stream(raw, fmt)
            assert got == want[fmt] and _unzip(got, fmt) == raw
            n = C.c_uint64()
            a = np.frombuffer(raw, dtype=np.uint8)
            out = np.zeros(len(got), dtype=np.uint8)
            rc = sctx.lib.zwz_deflate_stream(sctx.h, a.ctypes.data, a.size, out.ctypes.data, len(got) // 2, C.byref(n), 0, FMT[fmt])
            assert rc == E_CAPACITY and n.value == len(got)
    finally:
        sctx.tune(zwz_b200.Context.TUNE_DEFLATE_SUBBATCH_BYTES, 4 << 30)
