"""Test infrastructure: system zlib's inflate() with any windowBits (15 zlib, 31 gzip, -15 raw), driven through ctypes so that
the bytes produced before an error are kept (Python's zlib module drops them when it raises). The checker of the gzip and raw
inflate tests; the product never loads it."""
import ctypes as C
import ctypes.util

import numpy as np

STREAM_END, STREAM_TRUNCATED, STREAM_BAD, STREAM_OUTPUT_FULL = 0, 1, 2, 3  # ZWZ_STREAM_*
Z_STREAM_END, Z_NEED_DICT, Z_DATA_ERROR, Z_NO_FLUSH = 1, 2, -3, 0


class _ZStream(C.Structure):
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in", C.c_ulong),
                ("next_out", C.c_void_p), ("avail_out", C.c_uint), ("total_out", C.c_ulong),
                ("msg", C.c_char_p), ("state", C.c_void_p), ("zalloc", C.c_void_p), ("zfree", C.c_void_p), ("opaque", C.c_void_p),
                ("data_type", C.c_int), ("adler", C.c_ulong), ("reserved", C.c_ulong)]


_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(ctypes.util.find_library("z") or "libz.so.1")
        L.zlibVersion.restype = C.c_char_p
        L.inflateInit2_.argtypes = [C.POINTER(_ZStream), C.c_int, C.c_char_p, C.c_int]
        L.inflate.argtypes = [C.POINTER(_ZStream), C.c_int]
        L.inflateEnd.argtypes = [C.POINTER(_ZStream)]
        _LIB = L
    return _LIB


def inflate_wbits(comp: bytes, wbits: int, cap: int = 1 << 17):
    """One inflate() call over all of `comp` into a `cap`-byte buffer -> (bytes written, ZWZ_STREAM_* status):
    Z_STREAM_END -> END, Z_DATA_ERROR / Z_NEED_DICT -> BAD, output buffer filled first -> OUTPUT_FULL, input exhausted -> TRUNCATED."""
    L = _lib()
    src = C.create_string_buffer(bytes(comp), max(len(comp), 1))
    out = np.empty(max(cap, 1), dtype=np.uint8)
    s = _ZStream()
    assert L.inflateInit2_(C.byref(s), wbits, L.zlibVersion(), C.sizeof(_ZStream)) == 0
    s.next_in, s.avail_in = C.addressof(src), len(comp)
    s.next_out, s.avail_out = out.ctypes.data, cap
    rc = L.inflate(C.byref(s), Z_NO_FLUSH)
    n = cap - s.avail_out
    avail_in, avail_out = s.avail_in, s.avail_out
    L.inflateEnd(C.byref(s))
    if rc == Z_STREAM_END:
        st = STREAM_END
    elif rc in (Z_DATA_ERROR, Z_NEED_DICT):
        st = STREAM_BAD
    elif avail_out == 0 and avail_in != 0:
        st = STREAM_OUTPUT_FULL
    else:
        st = STREAM_TRUNCATED
    return out[:n].tobytes(), st
