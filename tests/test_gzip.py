"""gzip (BGZF members) and raw DEFLATE next to the zlib format: the CRC-32 kernel, deflate in the three formats (same body,
different wrapper), inflate of every format against system zlib with the matching windowBits, and the whole-file calls
gzip_files / gunzip_files. The "emu" variants run the same kernel sources under the SIMT emulator at small sizes."""
import gzip
import os
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

import oracle_lib as O
import zlib_ref
import zwz_b200
from tools import corpus

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
BGZF_HEAD = bytes.fromhex("1f8b08040000000000ff060042430200")
WBITS = {"zlib": 15, "gzip": 31, "raw": -15}
E_ARG, E_CAPACITY = -3, -5


def _offsets(parts):
    off = np.zeros(len(parts) + 1, dtype=np.uint64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return off


def _deflate(ctx, chunks, level, fmt):
    off = _offsets(chunks)
    packed, poff, res = ctx.deflate_batch(b"".join(chunks), off[:-1], np.diff(off).astype(np.uint32), level=level, format=fmt)
    return [packed[int(poff[i]):int(poff[i + 1])].tobytes() for i in range(len(chunks))], res


# ---------------------------------------------------------------------------------------------------------------------
# CRC-32
# ---------------------------------------------------------------------------------------------------------------------
def test_crc32_matches_zlib(ctx, is_gpu):
    rng = np.random.default_rng(11)
    lengths = [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, 127, 511, 4095, 65535, 65536 + 123] + ([1 << 20, 3 << 20] if is_gpu else [])
    data = rng.integers(0, 256, size=4 * sum(lengths) + 8 * 4 * len(lengths) + 64, dtype=np.uint8)
    data[: len(data) // 3] = np.frombuffer(corpus.gen_text(len(data) // 3, 596, 5).tobytes(), np.uint8)
    off, ln = [], []
    p = 0
    for n in lengths:
        for a in range(4):
            p = (p + 3) & ~3
            off.append(p + a)
            ln.append(n)
            p += a + n
    d = ctx.malloc_device(len(data))
    try:
        ctx.h2d(d, data)
        crc = ctx.crc32_batch_device(d, off, ln)
    finally:
        ctx.free_device(d)
    raw = data.tobytes()
    for o, n, c in zip(off, ln, crc):
        assert int(c) == zlib.crc32(raw[o:o + n]), (o, n)


# ---------------------------------------------------------------------------------------------------------------------
# deflate in GZIP and RAW format
# ---------------------------------------------------------------------------------------------------------------------
def _deflate_chunks():
    sizes = (0, 1, 96, 65279, 65280)
    classes = "TSBRJ"
    out = []
    for ci, cls in enumerate(classes):
        for si, n in enumerate(sizes):
            out.append(corpus.gen_file(cls, n, 596, 300 + 10 * ci + si).tobytes())
    return out


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_deflate_gzip_and_raw(ctx, level):
    chunks = _deflate_chunks()
    z, _ = _deflate(ctx, chunks, level, "zlib")
    g, gres = _deflate(ctx, chunks, level, "gzip")
    r, rres = _deflate(ctx, chunks, level, "raw")
    assert (gres["len1"] == 0).all() and (rres["len1"] == 0).all()
    for c, zs, gs, rs in zip(chunks, z, g, r):
        # one BGZF member: exact header, BSIZE = length - 1, CRC-32 and ISIZE trailer
        assert gs[:16] == BGZF_HEAD and struct.unpack("<H", gs[16:18])[0] == len(gs) - 1
        assert gs[-8:] == struct.pack("<II", zlib.crc32(c), len(c))
        d = zlib.decompressobj(31)
        assert d.decompress(gs) == c and d.eof and not d.unused_data
        assert gzip.decompress(gs) == c
        d = zlib.decompressobj(-15)
        assert d.decompress(rs) == c and d.eof
        # the body does not depend on the format
        assert zs[2:-4] == gs[18:-8] == rs, len(c)
        if not c:
            assert gs == BGZF_EOF
    # size: the body is the zlib body, so the gzip total minus its wrapper is the zlib total minus its wrapper
    assert sum(len(x) - 26 for x in g) == sum(len(x) - 6 for x in z)


def test_deflate_gzip_size_within_tolerance(ctx, is_gpu):
    """Per content class, gzip members minus their 26 wrapper bytes stay within 1.03 x zlib level 6 on the same chunks."""
    n_chunks, size = (2, 30000) if not is_gpu else (24, 65280)
    for cls in "TSBJR":
        chunks = [corpus.gen_file(cls, size, 596, 1000 + k).tobytes() for k in range(n_chunks)]
        g, _ = _deflate(ctx, chunks, 0, "gzip")
        assert all(gzip.decompress(x) == c for x, c in zip(g, chunks))
        ours = sum(len(x) - 26 for x in g)
        ref = sum(O.ref_deflate_size(c) - 6 for c in chunks)
        assert ours <= 1.03 * ref, (cls, ours, ref)


def test_deflate_gzip_chunk_limit(ctx):
    raw = bytes(65281)
    with pytest.raises(zwz_b200.ZwzError) as e:
        ctx.deflate_batch(raw, [0], [65281], format="gzip")
    assert e.value.code == E_ARG
    s, _ = _deflate(ctx, [raw], 0, "raw")  # raw has no 65 280-byte limit
    assert zlib.decompressobj(-15).decompress(s[0]) == raw
    with pytest.raises(ValueError):
        ctx.deflate_batch(raw, [0], [100], format="zip")


# ---------------------------------------------------------------------------------------------------------------------
# inflate of gzip and raw streams against zlib
# ---------------------------------------------------------------------------------------------------------------------
def _gzip_member(body_raw, level=6, flags=0, extra=b"", name=b"", comment=b"", hcrc_ok=True):
    """A gzip member with hand-chosen header fields around zlib's raw DEFLATE body."""
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = co.compress(body_raw) + co.flush()
    h = bytearray(b"\x1f\x8b\x08" + bytes([flags]) + struct.pack("<I", 1234567) + b"\x00\x03")
    if flags & 4:
        h += struct.pack("<H", len(extra)) + extra
    if flags & 8:
        h += name + b"\x00"
    if flags & 16:
        h += comment + b"\x00"
    if flags & 2:
        c = zlib.crc32(bytes(h)) & 0xffff
        h += struct.pack("<H", c if hcrc_ok else c ^ 0x0101)
    return bytes(h) + body + struct.pack("<II", zlib.crc32(body_raw), len(body_raw) & 0xffffffff)


def _inflate_cases(is_gpu):
    """(format, stream) pairs: intact streams, then cuts and corruptions."""
    text = corpus.gen_text(9000 if is_gpu else 2500, 596, 21).tobytes()
    rnd = corpus.gen_random(1500, 596, 22).tobytes()
    base = {"gzip": [], "raw": []}
    for lvl in range(10):
        base["gzip"].append(gzip.compress(text, compresslevel=lvl, mtime=0))
    for strat in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED):
        for wb, fmt in ((31, "gzip"), (-15, "raw")):
            co = zlib.compressobj(6, zlib.DEFLATED, wb, 8, strat)
            base[fmt].append(co.compress(text) + co.flush())
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    base["raw"].append(co.compress(rnd + text) + co.flush())
    base["gzip"] += [_gzip_member(text, flags=4, extra=b"AB\x03\x00xyz"), _gzip_member(text, flags=8, name=b"file.txt"),
                     _gzip_member(text, flags=16, comment=b"c" * 70), _gzip_member(rnd, flags=2 | 4 | 8 | 16, extra=b"", name=b"n" * 40, comment=b"x"),
                     _gzip_member(text, flags=2 | 8, name=b"hcrc"), _gzip_member(text, flags=2 | 8, name=b"hcrc", hcrc_ok=False),
                     _gzip_member(b""), _gzip_member(text, flags=0x20), _gzip_member(text, flags=1)]
    cases = []
    for fmt, streams in base.items():
        for si, s in enumerate(streams):
            cases.append((fmt, s))
            cases.append((fmt, s + b"trailing bytes are ignored"))
            head = 40 if fmt == "gzip" else 4
            cuts = set(range(0, min(head, len(s)))) | set(range(max(0, len(s) - 10), len(s)))
            cuts |= set(range(0, len(s), max(1, len(s) // (24 if is_gpu else 8))))
            for c in sorted(cuts):
                cases.append((fmt, s[:c]))
            rng = np.random.default_rng(100 + si)
            for _ in range(24 if is_gpu else 6):
                b = bytearray(s)
                i = int(rng.integers(0, len(b)))
                b[i] ^= 1 << int(rng.integers(0, 8))
                cases.append((fmt, bytes(b)))
            if fmt == "gzip" and len(s) >= 8:
                for k in (0, 3, 4, 7):  # a CRC-32 byte, an ISIZE byte
                    b = bytearray(s)
                    b[len(b) - 8 + k] ^= 0x40
                    cases.append((fmt, bytes(b)))
    # the zlib format keeps rejecting gzip streams and the gzip format zlib streams
    cases.append(("gzip", zlib.compress(text)))
    cases.append(("zlib", base["gzip"][0]))
    return cases


def test_inflate_formats_match_zlib(ctx_inf, is_gpu, request):
    cases = _inflate_cases(is_gpu)
    cap = 1 << 16
    lanes = "lanes" in request.node.name
    for fmt in ("gzip", "raw", "zlib"):
        streams = [s for f, s in cases if f == fmt]
        so = _offsets(streams)
        ro = np.arange(len(streams) + 1, dtype=np.uint64) * np.uint64(cap)
        args = (b"".join(streams) or b"\0", so[:-1], np.diff(so).astype(np.uint32), ro)
        if lanes and fmt != "zlib":
            with pytest.raises(zwz_b200.ZwzError) as e:
                ctx_inf.inflate_batch(*args, format=fmt)
            assert e.value.code == E_ARG
            continue
        out, rl, st = ctx_inf.inflate_batch(*args, format=fmt)
        for i, s in enumerate(streams):
            want, wst = zlib_ref.inflate_wbits(s, WBITS[fmt], cap)
            got = out[int(ro[i]):int(ro[i]) + int(rl[i])].tobytes()
            assert (int(st[i]), int(rl[i])) == (wst, len(want)), (fmt, i, len(s))
            assert got == want, (fmt, i)


def test_inflate_gzip_no_check_skips_crc_only(ctx):
    text = corpus.gen_text(3000, 596, 23).tobytes()
    good = gzip.compress(text, mtime=0)
    bad_crc = good[:-8] + bytes([good[-8] ^ 1]) + good[-7:]
    bad_isize = good[:-4] + bytes([good[-4] ^ 1]) + good[-3:]
    streams = [good, bad_crc, bad_isize]
    so = _offsets(streams)
    ro = np.arange(4, dtype=np.uint64) * np.uint64(1 << 16)
    _, rl, st = ctx.inflate_batch(b"".join(streams), so[:-1], np.diff(so).astype(np.uint32), ro, flags=zwz_b200.INFLATE_NO_ADLER,
                                  format="gzip")
    assert list(st) == [O.STREAM_END, O.STREAM_END, O.STREAM_BAD] and list(rl) == [3000] * 3


def test_decompress_records_rejects_a_format(ctx):
    comp = zlib.compress(b"abc")
    with pytest.raises(zwz_b200.ZwzError) as e:
        ctx.decompress_records(comp, [0], [len(comp)], [100], [0], 1, 100, flags=1 << 8)
    assert e.value.code == E_ARG


# ---------------------------------------------------------------------------------------------------------------------
# whole files
# ---------------------------------------------------------------------------------------------------------------------
def _files(is_gpu):
    B = zwz_b200.BGZF_BLOCK
    sizes = [0, 1, B - 1, B, B + 1, 2 * B - 1, 2 * B, 2 * B + 1] + ([5 << 20] if is_gpu else [300000])
    return [corpus.gen_file("TSBRJ"[i % 5], n, 596, 500 + i).tobytes() for i, n in enumerate(sizes)]


def _bgzf_members(gz):
    """Members of a BGZF file from their BSIZE fields (host-side reference walk)."""
    out, p = [], 0
    while p < len(gz):
        xlen = struct.unpack("<H", gz[p + 10:p + 12])[0]
        assert gz[p + 12:p + 16] == b"BC\x02\x00" and xlen == 6
        n = struct.unpack("<H", gz[p + 16:p + 18])[0] + 1
        out.append(gz[p:p + n])
        p += n
    return out


def test_gzip_files(ctx, is_gpu, tmp_path):
    files = _files(is_gpu)
    fo = _offsets(files)
    gz, gz_off = ctx.gzip_files(b"".join(files), fo)
    assert len(gz) <= ctx.lib.zwz_gzip_bound(fo.ctypes.data, len(files))
    have_gzip = shutil.which("gzip") is not None
    for i, f in enumerate(files):
        g = gz[int(gz_off[i]):int(gz_off[i + 1])].tobytes()
        assert gzip.decompress(g) == f
        m = _bgzf_members(g)
        assert m[-1] == BGZF_EOF and len(m) == -(-len(f) // zwz_b200.BGZF_BLOCK) + 1
        if have_gzip:
            p = tmp_path / f"f{i}.gz"
            p.write_bytes(g)
            subprocess.run(["gzip", "-t", str(p)], check=True)
            assert subprocess.run(["gzip", "-dc", str(p)], check=True, capture_output=True).stdout == f


def _py_bgzf(data, level):
    """A BGZF writer in plain Python (bgzip's layout) over zlib at any level."""
    out = bytearray()
    for o in list(range(0, len(data), 65280)) + [None]:
        blk = b"" if o is None else data[o:o + 65280]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        body = co.compress(blk) + co.flush()
        out += BGZF_HEAD + struct.pack("<H", 18 + len(body) + 8 - 1) + body + struct.pack("<II", zlib.crc32(blk), len(blk))
    return bytes(out)


def test_gunzip_files(ctx, is_gpu):
    files = _files(is_gpu)
    fo = _offsets(files)
    gz, gz_off = ctx.gzip_files(b"".join(files), fo)
    gzs = [gz[int(gz_off[i]):int(gz_off[i + 1])].tobytes() for i in range(len(files))]
    # our own files, files of the Python writer at other levels, then broken ones
    text = corpus.gen_text(200000, 596, 31).tobytes()
    foreign = [_py_bgzf(text, lvl) for lvl in (1, 9, 0)]
    mid = bytearray(_py_bgzf(text, 6))
    m = _bgzf_members(bytes(mid))
    crc_at = len(m[0]) + len(m[1]) - 8
    mid[crc_at] ^= 0xff  # a CRC-32 byte of the second member
    plain = gzip.compress(text)
    cut = _py_bgzf(text, 6)
    cut = cut[:len(_bgzf_members(cut)[0]) + 100]
    inputs = gzs + foreign + [gzs[1], bytes(mid), plain, cut, gzs[2]]
    want = files + [text] * 3 + [files[1], None, None, None, files[2]]
    go = _offsets(inputs)
    out, out_off, st = ctx.gunzip_files(b"".join(inputs), go)
    for i, w in enumerate(want):
        got = out[int(out_off[i]):int(out_off[i + 1])].tobytes()
        if w is not None:
            assert st[i] == O.STREAM_END and got == w, i
    i_mid, i_plain, i_cut = len(files) + 4, len(files) + 5, len(files) + 6
    assert st[i_mid] == O.STREAM_BAD
    got = out[int(out_off[i_mid]):int(out_off[i_mid + 1])].tobytes()
    assert got == text[:2 * 65280]  # the first member, then what the bad one produced before its trailer
    assert st[i_plain] == O.STREAM_BAD and out_off[i_plain + 1] == out_off[i_plain]
    assert st[i_cut] == O.STREAM_TRUNCATED
    got = out[int(out_off[i_cut]):int(out_off[i_cut + 1])].tobytes()
    assert text.startswith(got) and len(got) >= 65280
    # below the bound
    bound = ctx.lib.zwz_gunzip_bound(np.frombuffer(b"".join(inputs), np.uint8).ctypes.data, go.ctypes.data, len(inputs))
    with pytest.raises(zwz_b200.ZwzError) as e:
        ctx.gunzip_files(b"".join(inputs), go, out_cap=int(bound) - 1)
    assert e.value.code == E_CAPACITY


@pytest.mark.gpu
def test_gzip_gunzip_large_mixed_corpus(cuda_ctx):
    data, file_off = corpus.mixed_buffer(256 << 20)[:2]
    gz, gz_off = cuda_ctx.gzip_files(data, file_off)
    out, out_off, st = cuda_ctx.gunzip_files(gz, gz_off)
    assert (st == O.STREAM_END).all()
    assert np.array_equal(out_off, np.asarray(file_off, dtype=np.uint64) - np.uint64(file_off[0]))
    assert np.array_equal(out, np.asarray(data)[int(file_off[0]):int(file_off[-1])])
    for i in range(0, len(file_off) - 1, max(1, (len(file_off) - 1) // 8)):
        assert gzip.decompress(gz[int(gz_off[i]):int(gz_off[i + 1])].tobytes()) == bytes(data[int(file_off[i]):int(file_off[i + 1])])
