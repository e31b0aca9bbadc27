"""Preset dictionaries (zlib's deflateSetDictionary / inflateSetDictionary, Python's zdict=) in batched deflate and inflate, ZLIB
(FDICT + DICTID) and RAW, checked against system zlib. The "emu" variants run the same kernel sources under the SIMT emulator at
small sizes; every inflate case runs on the warp decoder (with its lane-parallel block decoder) and on the careful one."""
import ctypes as C
import struct
import zlib

import numpy as np
import pytest

import zlib_ref
import zwz_b200
from tools import corpus

E_ARG = -3
END, TRUNC, BAD, FULL = zwz_b200.STREAM_END, zwz_b200.STREAM_TRUNCATED, zwz_b200.STREAM_BAD, zwz_b200.STREAM_OUTPUT_FULL
WBITS = {"zlib": 15, "raw": -15}
DICT = corpus.gen_text(32768, 596, 9999).tobytes()

INFLATE = [pytest.param("emu_ctx", id="emu-warp"), pytest.param("emu_ctx_careful", id="emu-careful"),
           pytest.param("cuda_ctx_warp", id="cuda-warp", marks=pytest.mark.gpu),
           pytest.param("cuda_ctx_careful", id="cuda-careful", marks=pytest.mark.gpu)]


@pytest.fixture(params=INFLATE)
def ictx(request):
    return request.getfixturevalue(request.param)


def _offsets(parts):
    off = np.zeros(len(parts) + 1, dtype=np.uint64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return off


def _deflate(ctx, chunks, level=0, fmt="zlib", **kw):
    off = _offsets(chunks)
    packed, poff, res = ctx.deflate_batch(b"".join(chunks), off[:-1], np.diff(off).astype(np.uint32), level=level, format=fmt, **kw)
    return [packed[int(poff[i]):int(poff[i + 1])].tobytes() for i in range(len(chunks))], res


def _inflate(ctx, streams, cap, fmt="zlib", flags=0, **kw):
    so = _offsets(streams)
    ro = np.arange(len(streams) + 1, dtype=np.uint64) * np.uint64(cap)
    out, rl, st = ctx.inflate_batch(b"".join(streams), so[:-1], np.diff(so).astype(np.uint32), ro, flags=flags, format=fmt, **kw)
    return [(out[int(ro[i]):int(ro[i]) + int(rl[i])].tobytes(), int(rl[i]), int(st[i])) for i in range(len(streams))]


def _zinflate(comp: bytes, wbits: int, zdict: bytes, cap: int):
    """System zlib with a preset dictionary, keeping the bytes written before an error: inflateSetDictionary after Z_NEED_DICT
    (zlib) or before the first inflate (raw) -> (bytes, raw_len, ZWZ_STREAM_* status)."""
    L = zlib_ref._lib()
    L.inflateSetDictionary.argtypes = [C.POINTER(zlib_ref._ZStream), C.c_char_p, C.c_uint]
    src = C.create_string_buffer(bytes(comp), max(len(comp), 1))
    out = np.empty(max(cap, 1), dtype=np.uint8)
    s = zlib_ref._ZStream()
    assert L.inflateInit2_(C.byref(s), wbits, L.zlibVersion(), C.sizeof(zlib_ref._ZStream)) == 0
    s.next_in, s.avail_in = C.addressof(src), len(comp)
    s.next_out, s.avail_out = out.ctypes.data, cap
    if wbits < 0:
        assert L.inflateSetDictionary(C.byref(s), zdict, len(zdict)) == 0
    rc = L.inflate(C.byref(s), zlib_ref.Z_NO_FLUSH)
    if rc == zlib_ref.Z_NEED_DICT:
        rc = L.inflateSetDictionary(C.byref(s), zdict, len(zdict))
        if rc == 0:
            rc = L.inflate(C.byref(s), zlib_ref.Z_NO_FLUSH)
        else:
            rc = zlib_ref.Z_DATA_ERROR
    n = cap - s.avail_out
    avail_in, avail_out = s.avail_in, s.avail_out
    L.inflateEnd(C.byref(s))
    if rc == zlib_ref.Z_STREAM_END:
        st = END
    elif rc in (zlib_ref.Z_DATA_ERROR, zlib_ref.Z_NEED_DICT):
        st = BAD
    elif avail_out == 0 and avail_in != 0:
        st = FULL
    else:
        st = TRUNC
    return out[:n].tobytes(), n, st


def _zcompress(data: bytes, zdict: bytes, level=6, wbits=15, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, wbits, 9, strategy, zdict=zdict)
    return c.compress(data) + c.flush()


# ---------------------------------------------------------------------------------------------------------------------
# deflate
# ---------------------------------------------------------------------------------------------------------------------
SIZES = (0, 1, 3, 8192, 8193, 16385, 31745, 65535)


@pytest.mark.parametrize("fmt", ["zlib", "raw"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_deflate_dict_round_trip(ctx, level, fmt):
    chunks = [corpus.gen_file(cls, n, 596, 500 + 10 * ci + si).tobytes() for ci, cls in enumerate("TSBRJ") for si, n in enumerate(SIZES)]
    streams, res = _deflate(ctx, chunks, level, fmt, zdict=DICT)
    assert (res["len1"] == 0).all()
    for c, s in zip(chunks, streams):
        d = zlib.decompressobj(WBITS[fmt], zdict=DICT)
        assert d.decompress(s) == c and d.eof and not d.unused_data, len(c)
        if fmt == "zlib":
            assert s[:2] == b"\x78\xbb" and struct.unpack(">I", s[2:6])[0] == zlib.adler32(DICT)
            assert struct.unpack(">I", s[-4:])[0] == zlib.adler32(c)
            with pytest.raises(zlib.error):
                zlib.decompress(s)


def test_deflate_dict_is_used(ctx, is_gpu):
    """Text records of 64-512 B: within 1.03 x zlib-6 with the same zdict, and far smaller than without a dictionary."""
    rng = np.random.default_rng(3)
    recs = [corpus.gen_file("T", int(n), 596, 7000 + k).tobytes() for k, n in enumerate(rng.integers(64, 513, 1000 if is_gpu else 150))]
    with_d, _ = _deflate(ctx, recs, 0, "zlib", zdict=DICT)
    without, _ = _deflate(ctx, recs, 0, "zlib")
    ref = sum(len(_zcompress(r, DICT)) for r in recs)
    ours = sum(len(s) for s in with_d)
    assert ours <= 1.03 * ref, (ours, ref)
    assert ours < 0.85 * sum(len(s) for s in without)
    tail, _ = _deflate(ctx, [DICT[-1000:]], 0, "zlib", zdict=DICT)
    assert len(tail[0]) <= 24 and zlib.decompressobj(zdict=DICT).decompress(tail[0]) == DICT[-1000:]


def test_deflate_dict_window_edges(ctx):
    big = corpus.gen_text(40000, 596, 4242).tobytes()
    s, _ = _deflate(ctx, [big[:5000], big[100:3100]], 0, "zlib", zdict=big)
    for st, c in zip(s, [big[:5000], big[100:3100]]):
        assert struct.unpack(">I", st[2:6])[0] == zlib.adler32(big)  # the DICTID covers the whole dictionary
        assert zlib.decompressobj(zdict=big).decompress(st) == c
    # a record that starts with the bytes at exactly distance 32 768 (the first byte of the window)
    rec = big[40000 - 32768:40000 - 32768 + 600] + b"tail"
    for fmt in ("zlib", "raw"):
        s, _ = _deflate(ctx, [rec], 9, fmt, zdict=big)
        assert zlib.decompressobj(WBITS[fmt], zdict=big).decompress(s[0]) == rec
    # dictionaries shorter than 3 bytes, and an empty one (no FDICT: the bytes of the plain call)
    chunk = corpus.gen_text(3000, 596, 77).tobytes()
    plain, _ = _deflate(ctx, [chunk], 0, "zlib")
    for d in (b"ab", b"a"):
        s, _ = _deflate(ctx, [chunk], 0, "zlib", zdict=d)
        assert s[0][:2] == b"\x78\xbb" and zlib.decompressobj(zdict=d).decompress(s[0]) == chunk
    s, _ = _deflate(ctx, [chunk], 0, "zlib", zdict=b"")
    assert s[0] == plain[0]


def test_deflate_dict_mixed_batch(ctx):
    dicts = [DICT, corpus.gen_struct(20000, 596, 31).tobytes(), corpus.gen_text(5000, 597, 32).tobytes()]
    chunks, idx = [], []
    for k in range(24):
        which = [0, zwz_b200.NO_DICT, 1, 2][k % 4]
        src = dicts[which] if which != zwz_b200.NO_DICT else DICT
        chunks.append(src[(k * 997) % 3000:(k * 997) % 3000 + 300 + 150 * k])
        idx.append(which)
    for fmt in ("zlib", "raw"):
        s, _ = _deflate(ctx, chunks, 0, fmt, zdict=dicts, zdict_index=idx)
        plain, _ = _deflate(ctx, chunks, 0, fmt)
        for c, st, pl, k in zip(chunks, s, plain, idx):
            if k == zwz_b200.NO_DICT:
                assert st == pl
            else:
                assert zlib.decompressobj(WBITS[fmt], zdict=dicts[k]).decompress(st) == c


# ---------------------------------------------------------------------------------------------------------------------
# inflate
# ---------------------------------------------------------------------------------------------------------------------
def _inflate_vs_zlib(ctx, streams, fmt, zdict, cap=70000, flags=0):
    got = _inflate(ctx, streams, cap, fmt, flags, zdict=zdict)
    for i, (s, g) in enumerate(zip(streams, got)):
        want = _zinflate(s, WBITS[fmt], zdict, cap)
        assert g == want, (i, len(s), g[1:], want[1:])


def _cpython_streams(fmt, levels=(1, 6, 9)):
    out = []
    for li, level in enumerate(levels):
        for si, strategy in enumerate((zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_FIXED)):
            for k, n in enumerate((200, 1500, 9000)):
                data = corpus.gen_file("TST"[k], n, 596, 800 + 100 * li + 10 * si + k).tobytes() + DICT[1000:1000 + n // 3]
                out.append(_zcompress(data, DICT, level, WBITS[fmt], strategy))
    return out


@pytest.mark.parametrize("fmt", ["zlib", "raw"])
def test_inflate_dict_cpython_streams(ictx, fmt):
    streams = _cpython_streams(fmt)
    _inflate_vs_zlib(ictx, streams, fmt, DICT)
    # truncations and single-byte corruptions
    rng = np.random.default_rng(5)
    bad = []
    for s in streams[::5]:
        for cut in (1, 2, 3, 5, len(s) // 2, len(s) - 1):
            bad.append(s[:cut])
        for _ in range(3):
            b = bytearray(s)
            p = int(rng.integers(0, len(b)))
            b[p] ^= 1 << int(rng.integers(0, 8))
            bad.append(bytes(b))
    _inflate_vs_zlib(ictx, bad, fmt, DICT)


def _bits_stream(symbols):
    """A fixed-Huffman block (BFINAL=1) of literals and (length, distance) pairs -> raw DEFLATE bytes."""
    acc, nb = 0, 0

    def put(v, n):
        nonlocal acc, nb
        acc |= v << nb
        nb += n

    def put_rev(code, n):
        put(int(format(code, f"0{n}b")[::-1], 2), n)

    def lit(s):
        if s < 144:
            put_rev(0x30 + s, 8)
        elif s < 256:
            put_rev(0x190 + s - 144, 9)
        elif s < 280:
            put_rev(s - 256, 7)
        else:
            put_rev(0xC0 + s - 280, 8)

    put(1, 1)
    put(1, 2)
    for sym in symbols:
        if isinstance(sym, int):
            lit(sym)
            continue
        ln, dist = sym
        base = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
        ext = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
        k = max(i for i in range(29) if base[i] <= ln)
        lit(257 + k)
        put(ln - base[k], ext[k])
        dbase = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193,
                 12289, 16385, 24577]
        dext = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
        j = max(i for i in range(30) if dbase[i] <= dist)
        put_rev(j, 5)
        put(dist - dbase[j], dext[j])
    lit(256)
    return acc.to_bytes((nb + 7) // 8, "little")


def _zlib_wrap(body: bytes, zdict: bytes, out: bytes):
    return b"\x78\xbb" + struct.pack(">I", zlib.adler32(zdict)) + body + struct.pack(">I", zlib.adler32(out))


@pytest.mark.parametrize("fmt", ["zlib", "raw"])
def test_inflate_dict_distance_edges(ictx, fmt):
    d = corpus.gen_text(1000, 596, 55).tobytes()  # window shorter than 32 KiB: W = 1000
    W = len(d)
    cases = [
        [65, 66, (10, 2 + W)],             # distance pos + W: the first byte of the window (OK)
        [65, 66, (10, 2 + W + 1)],         # one further (BAD, after the two literals)
        [(20, 3)],                         # overlapping copy across the window / output boundary at pos 0
        [67, (40, 5), (258, 1)],           # overlap with a period < 32 that starts in the window
        [(3, W)] + [(4, W - 7 * i) for i in range(1, 100)],   # a block full of short matches into the dictionary
    ]
    streams = []
    for syms in cases:
        body = _bits_stream(syms)
        if fmt == "raw":
            streams.append(body)
        else:
            ok = _zinflate(b"\x78\xbb" + struct.pack(">I", zlib.adler32(d)) + body + b"\0\0\0\0", 15, d, 70000)[0]
            streams.append(_zlib_wrap(body, d, ok))
    _inflate_vs_zlib(ictx, streams, fmt, d)
    got = _inflate(ictx, streams[:1], 70000, fmt, zdict=d)[0]
    assert got[2] == END and got[0] == b"AB" + d[:10]
    assert _inflate(ictx, streams[1:2], 70000, fmt, zdict=d)[0][1:] == (2, BAD)
    # output capacity too small: OUTPUT_FULL with the size needed, and the first 100 bytes are zlib's
    full, n, _ = _zinflate(streams[4], WBITS[fmt], d, 70000)
    got = _inflate(ictx, streams[4:], 100, fmt, zdict=d)[0]
    assert got[1:] == (n, FULL) and got[0][:100] == full[:100] == _zinflate(streams[4], WBITS[fmt], d, 100)[0]


def test_inflate_dict_refusals(ictx):
    data = corpus.gen_text(3000, 596, 12).tobytes() + DICT[5000:6000]
    s = _zcompress(data, DICT)
    other = corpus.gen_text(32768, 596, 1234).tobytes()
    # wrong dictionary: BAD with 0 bytes, also without the Adler-32 check
    for flags in (0, zwz_b200.INFLATE_NO_ADLER):
        assert _inflate(ictx, [s], 70000, flags=flags, zdict=other)[0] == (b"", 0, BAD)
    assert _inflate(ictx, [s], 70000, flags=zwz_b200.INFLATE_NO_ADLER, zdict=DICT)[0] == (data, len(data), END)
    # FDICT without a dictionary (also with a ZWZ_NO_DICT entry in a dictionary call)
    assert _inflate(ictx, [s], 70000)[0][1:] == (0, BAD)
    assert _inflate(ictx, [s], 70000, zdict=[DICT], zdict_index=[zwz_b200.NO_DICT])[0][1:] == (0, BAD)
    # no FDICT: the dictionary is ignored, and a reference before byte 0 is BAD where zlib finds it
    plain = zlib.compress(data, 6)
    assert _inflate(ictx, [plain], 70000, zdict=DICT)[0] == (data, len(data), END)
    body = _bits_stream([72, 73, (5, 3)])
    nofd = b"\x78\x9c" + body + b"\0\0\0\0"
    _inflate_vs_zlib(ictx, [nofd], "zlib", DICT)
    assert _inflate(ictx, [nofd], 70000, zdict=DICT)[0][1:] == (2, BAD)
    # cut inside the DICTID
    for cut in (2, 3, 4, 5):
        assert _inflate(ictx, [s[:cut]], 70000, zdict=DICT)[0][1:] == (0, TRUNC)


def test_dict_argument_refusals(emu_ctx, emu_ctx_lanes):
    chunk = DICT[:2000]
    for call in (lambda: _deflate(emu_ctx, [chunk], 0, "gzip", zdict=DICT),
                 lambda: _inflate(emu_ctx, [zlib.compress(chunk)], 70000, "gzip", zdict=DICT),
                 lambda: _inflate(emu_ctx_lanes, [_zcompress(chunk, DICT)], 70000, zdict=DICT),
                 lambda: _deflate(emu_ctx, [chunk], 0, "zlib", zdict=[DICT], zdict_index=[1]),
                 lambda: _inflate(emu_ctx, [_zcompress(chunk, DICT)], 70000, zdict=[DICT, DICT], zdict_index=[2])):
        with pytest.raises(zwz_b200.ZwzError) as e:
            call()
        assert e.value.code == E_ARG


@pytest.mark.gpu
def test_dict_device_api_large(cuda_ctx):
    """200 000 text records of 64-4 096 B, one 32 KiB dictionary, deflate -> inflate through the device API (above the host
    threads' threshold): byte-exact, every status STREAM_END, and a sample decodes with CPython."""
    ctx = cuda_ctx
    rng = np.random.default_rng(17)
    sizes = rng.integers(64, 4097, 200_000).astype(np.uint32)
    text = corpus.gen_text(int(sizes.sum()) // 4 + 65536, 596, 4321).tobytes()
    starts = rng.integers(0, len(text) - 4096, len(sizes))
    raw = np.frombuffer(b"".join(text[int(a):int(a) + int(n)] for a, n in zip(starts, sizes)), dtype=np.uint8)
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off[1:])
    slot = np.zeros(len(sizes) + 1, dtype=np.uint64)
    np.cumsum(zwz_b200.deflate_bound(sizes), out=slot[1:])
    dd = np.frombuffer(DICT, dtype=np.uint8)
    d_raw, d_out, d_back, d_dict = (ctx.malloc_device(int(x)) for x in (len(raw), int(slot[-1]), len(raw), len(dd)))
    try:
        ctx.h2d(d_raw, raw)
        ctx.h2d(d_dict, dd)
        zd = (d_dict, [0, len(dd)])
        res = ctx.deflate_batch_device(d_raw, off[:-1], sizes, d_out, slot[:-1], zdict=zd)
        assert (res["len1"] == 0).all()
        rl, st = ctx.inflate_batch_device(d_out, slot[:-1], res["len0"], d_back, off, zdict=zd)
        assert (st == END).all() and (rl == sizes).all()
        back = np.empty_like(raw)
        ctx.d2h(back, d_back)
        assert np.array_equal(back, raw)
        comp = np.empty(int(slot[-1]), dtype=np.uint8)
        ctx.d2h(comp, d_out)
    finally:
        for p in (d_raw, d_out, d_back, d_dict):
            ctx.free_device(p)
    for i in rng.choice(len(sizes), 2000, replace=False):
        s = comp[int(slot[i]):int(slot[i]) + int(res["len0"][i])].tobytes()
        assert zlib.decompressobj(zdict=DICT).decompress(s) == raw[int(off[i]):int(off[i + 1])].tobytes()
