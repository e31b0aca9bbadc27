"""ctypes loader for oracle/liboracle.so — the CHECKER. Only tests/, smoke() and bench.py's CPU legs use this."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
_LIB = None

STREAM_END, STREAM_TRUNCATED, STREAM_BAD, STREAM_OUTPUT_FULL = 0, 1, 2, 3
CHUNK = 65535


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(ORACLE_DIR, "zwz_oracle.c")):
            subprocess.run(["make", "-C", ORACLE_DIR, "liboracle.so"], check=True, capture_output=True)
        L = C.CDLL(so)
        u8p = C.POINTER(C.c_uint8)
        L.oracle_adler32.restype = C.c_uint32
        L.oracle_adler32.argtypes = [C.c_void_p, C.c_size_t]
        L.oracle_md5_hex.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p]
        L.oracle_ref_md5_hex.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p]
        L.oracle_inflate.restype = C.c_int
        L.oracle_inflate.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.oracle_ref_deflate_chunk.restype = C.c_long
        L.oracle_ref_deflate_chunk.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.oracle_ref_deflate_bound_size.restype = C.c_long
        L.oracle_ref_deflate_bound_size.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
        L.oracle_ref_inflate_chunk.restype = C.c_longlong
        L.oracle_ref_inflate_chunk.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.oracle_ref_deflate_batch.restype = C.c_uint64
        L.oracle_ref_deflate_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.oracle_ref_inflate_batch.restype = C.c_uint64
        L.oracle_ref_inflate_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.oracle_ref_md5_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        _LIB = L
    return _LIB


def _buf(b):
    a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else b
    return a, a.ctypes.data if a.size else None


def adler32(b) -> int:
    a, p = _buf(b)
    return lib().oracle_adler32(p, a.size)


def md5_hex(b) -> str:
    a, p = _buf(b)
    out = C.create_string_buffer(32)
    lib().oracle_md5_hex(p, a.size, out)
    return out.raw.decode()


def ref_md5_hex(b) -> str:
    a, p = _buf(b)
    out = C.create_string_buffer(32)
    lib().oracle_ref_md5_hex(p, a.size, out)
    return out.raw.decode()


def inflate(comp, cap=1 << 20):
    """-> (bytes produced (clipped to cap), status, full length)"""
    a, p = _buf(comp)
    out = np.empty(max(cap, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    st = lib().oracle_inflate(p, a.size, out.ctypes.data, cap, C.byref(n))
    return out[:min(n.value, cap)].tobytes(), st, n.value


def ref_deflate_chunk(raw) -> bytes:
    """compression.cpp:119-134 — including the silent truncation at 65 535 bytes."""
    a, p = _buf(raw)
    out = np.empty(CHUNK, dtype=np.uint8)
    n = lib().oracle_ref_deflate_chunk(p, a.size, out.ctypes.data)
    return out[:n].tobytes()


def ref_deflate_size(raw, level=6) -> int:
    a, p = _buf(raw)
    return lib().oracle_ref_deflate_bound_size(p, a.size, level)


def ref_inflate_chunk(comp, cap=1 << 21) -> bytes:
    """decompression.cpp:11-37 with avail_in = len(comp)."""
    a, p = _buf(comp)
    out = np.empty(cap, dtype=np.uint8)
    n = lib().oracle_ref_inflate_chunk(p, a.size, out.ctypes.data, cap)
    assert n >= 0
    return out[:n].tobytes()


def ref_decompress(arch_dir, out_dir) -> dict:
    """`main decompress <arch_dir> <out_dir>` of the reference (decompression.cpp:45-178) restated: every *.zwz is read
    record by record with per-archive, per-path state. A record whose sequence id is the expected one is inflated
    (ref_inflate_chunk) and appended to <out_dir>/<path>, followed by any waiting records that are now in order; other records
    wait in a min-heap. When the record just read is the last one, was in order and nothing waits, the file is closed and
    the MD5 of what was written is compared with the stored one (decompression.cpp:132-146). Returns the verdict counts
    {"match": m, "mismatch": k}. tests/test_oracle.py pins this to what the reference binary wrote for tests/golden/."""
    import heapq

    import zwz_format
    verdicts = {"match": 0, "mismatch": 0}
    for name in sorted(f for f in os.listdir(arch_dir) if f.endswith(".zwz")):
        files = {}   # path -> [output file, its path, expected sequence id, heap of (sequence id, payload)]
        for r in zwz_format.parse(open(os.path.join(arch_dir, name), "rb").read()):
            if r.path not in files:
                dst = os.path.join(out_dir, r.path)
                os.makedirs(os.path.dirname(dst), exist_ok=True)
                files[r.path] = [open(dst, "wb"), dst, 0, []]
            st = files[r.path]
            if r.seq != st[2]:
                heapq.heappush(st[3], (r.seq, r.payload))
                continue
            st[0].write(ref_inflate_chunk(r.payload))
            st[2] += 1
            while st[3] and st[3][0][0] == st[2]:
                st[0].write(ref_inflate_chunk(heapq.heappop(st[3])[1]))
                st[2] += 1
            if r.last and st[2] == r.seq + 1 and not st[3]:
                st[0].close()
                ok = ref_md5_hex(open(st[1], "rb").read()) == r.md5.decode()
                verdicts["match" if ok else "mismatch"] += 1
        for st in files.values():
            st[0].close()
    return verdicts


def md5_tree(root) -> dict:
    """{relative path: {"size", "md5"}} of every file under root (the form of tests/golden/manifest.json)."""
    out = {}
    for d, _, names in os.walk(root):
        for f in names:
            p = os.path.join(d, f)
            b = open(p, "rb").read()
            out[os.path.relpath(p, root)] = {"size": len(b), "md5": hashlib.md5(b).hexdigest()}
    return out
