"""B200-native (sm_100a) hot path of the shard-based DEFLATE pipeline: Python binding of the C ABI.

The product is ``csrc/libzwz_cuda.so`` (hand-written CUDA kernels behind ``include/zwz_cuda.h``) plus the C++ host
under ``host/`` (``main compress|decompress``). This module is a thin ctypes layer over that C ABI, used by the tests
and by ``bench.py``; it mirrors the three reference call sites it replaces:

  Context.deflate_batch   <- compression.cpp:119-134   (zlib deflate per 65 535-byte chunk)
  Context.inflate_batch   <- decompression.cpp:11-37   (zlib inflate per record)
  Context.md5_batch       <- verification.cpp:13-27    (MD5 per file, 32 lowercase hex chars)

There is NO CPU fallback: importing works anywhere, but creating a ``Context`` raises unless the CUDA extension is
built (``python -c 'import __graft_entry__ as g; g.build()'``) and a Blackwell GPU is present.

The directory name contains hyphens, so import it with
``importlib.import_module("parallel-data-compression-and-decompression_b200")`` (``zwz_b200.py`` at the repo root does that).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import numpy as np

__all__ = ["Context", "ZwzError", "load_library", "library_path", "CHUNK_SIZE", "deflate_bound", "chunk_table",
           "STREAM_END", "STREAM_TRUNCATED", "STREAM_BAD", "STREAM_OUTPUT_FULL", "RESULT_DTYPE",
           "FORMAT_ZLIB", "FORMAT_GZIP", "FORMAT_RAW", "BGZF_BLOCK", "NO_DICT"]

CHUNK_SIZE = 65535  # process.hpp:12
STREAM_END, STREAM_TRUNCATED, STREAM_BAD, STREAM_OUTPUT_FULL = 0, 1, 2, 3
INFLATE_NO_ADLER = 1
# stream formats (ZWZ_FORMAT_*): the wrapper around the DEFLATE body. The ``format=`` keywords take these names.
FORMAT_ZLIB, FORMAT_GZIP, FORMAT_RAW = 0, 1, 2
BGZF_BLOCK = 65280  # largest chunk in gzip format: one BGZF member each
_FORMATS = {"zlib": FORMAT_ZLIB, "gzip": FORMAT_GZIP, "raw": FORMAT_RAW}


def _format(name: str) -> int:
    if name not in _FORMATS:
        raise ValueError(f"format must be one of {sorted(_FORMATS)}, not {name!r}")
    return _FORMATS[name]

# zdict_index entry of a chunk / stream without a preset dictionary (ZWZ_NO_DICT)
NO_DICT = 0xFFFFFFFF


class _Dicts(C.Structure):  # zwz_dicts
    _fields_ = [("data", C.c_void_p), ("off", C.c_void_p), ("ndict", C.c_uint32), ("idx", C.c_void_p)]


def _dicts(zdict, zdict_index, n: int, device: bool):
    """The zwz_dicts of a call -> (pointer argument or None, arrays to keep alive during the call). zdict: host forms take bytes
    (one dictionary for all) or a list of bytes; device forms take (device pointer, offsets[ndict+1]). zdict_index: the
    dictionary of every chunk / stream (NO_DICT for none); None = dictionary 0 for all."""
    if zdict is None:
        if zdict_index is not None:
            raise ValueError("zdict_index without zdict")
        return None, ()
    if device:
        data, off = zdict
        off = np.ascontiguousarray(off, dtype=np.uint64)
        keep = [off]
        dptr = int(data)
    else:
        parts = [zdict] if isinstance(zdict, (bytes, bytearray, memoryview)) else list(zdict)
        parts = [bytes(p) for p in parts]
        off = np.zeros(len(parts) + 1, dtype=np.uint64)
        np.cumsum([len(p) for p in parts], out=off[1:])
        data = np.frombuffer(b"".join(parts) + b"\0", dtype=np.uint8)
        keep = [off, data]
        dptr = data.ctypes.data
    idx = None
    if zdict_index is not None:
        idx = np.ascontiguousarray(zdict_index, dtype=np.uint32)
        if len(idx) != n:
            raise ValueError(f"zdict_index has {len(idx)} entries for {n} chunks / streams")
        keep.append(idx)
    s = _Dicts(dptr, off.ctypes.data, len(off) - 1, _ptr(idx) if idx is not None and idx.size else None)
    keep.append(s)
    return C.byref(s), keep


RESULT_DTYPE = np.dtype([("len0", "<u4"), ("len1", "<u4"), ("raw0", "<u4"), ("btype", "<u4")])

_HERE = os.path.dirname(os.path.abspath(__file__))


class ZwzError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"zwz error {code}: {msg}")
        self.code = code


def library_path() -> str:
    return os.path.join(_HERE, "csrc", "libzwz_cuda.so")


_LIB = None


def _declare(L):
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.zwz_abi_version.restype = i32
    L.zwz_device_count.restype = i32
    L.zwz_init.argtypes = [i32, C.POINTER(vp)]
    L.zwz_destroy.argtypes = [vp]
    L.zwz_destroy.restype = None
    L.zwz_last_error.argtypes = [vp]
    L.zwz_last_error.restype = C.c_char_p
    L.zwz_device_props.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(C.c_size_t)]
    L.zwz_launch_count.argtypes = [vp]
    L.zwz_launch_count.restype = u64
    L.zwz_malloc_device.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    L.zwz_free_device.argtypes = [vp, vp]
    L.zwz_malloc_pinned.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    L.zwz_free_pinned.argtypes = [vp, vp]
    L.zwz_memcpy_h2d.argtypes = [vp, vp, vp, C.c_size_t]
    L.zwz_memcpy_d2h.argtypes = [vp, vp, vp, C.c_size_t]
    L.zwz_sync.argtypes = [vp]
    L.zwz_deflate_batch_device.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, i32, vp]
    L.zwz_deflate_batch.argtypes = [vp, vp, vp, vp, u32, vp, u64, vp, vp, i32]
    L.zwz_pack_streams_device.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp]
    L.zwz_inflate_batch_device.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, vp, u32, vp]
    L.zwz_inflate_batch.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, vp, u32]
    L.zwz_md5_batch_device.argtypes = [vp, vp, vp, vp, u32, vp, vp]
    L.zwz_md5_batch.argtypes = [vp, vp, vp, vp, u32, vp]
    L.zwz_md5_state_init.argtypes = [vp, u32]
    L.zwz_md5_state_init.restype = None
    L.zwz_md5_update_device.argtypes = [vp, vp, vp, vp, vp, u32, vp]
    L.zwz_md5_final_device.argtypes = [vp, vp, vp, vp, vp, vp, u32, vp, vp]
    L.zwz_md5_hex.argtypes = [vp, vp]
    L.zwz_md5_hex.restype = None
    L.zwz_adler32_batch_device.argtypes = [vp, vp, vp, vp, u32, vp, vp]
    L.zwz_crc32_batch_device.argtypes = [vp, vp, vp, vp, u32, vp, vp]
    L.zwz_deflate_batch_device_ex.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, i32, i32, vp]
    L.zwz_deflate_batch_ex.argtypes = [vp, vp, vp, vp, u32, vp, u64, vp, vp, i32, i32]
    L.zwz_gzip_bound.argtypes = [vp, u32]
    L.zwz_gzip_bound.restype = u64
    L.zwz_gzip_files.argtypes = [vp, vp, vp, u32, i32, vp, u64, vp]
    L.zwz_gunzip_bound.argtypes = [vp, vp, u32]
    L.zwz_gunzip_bound.restype = u64
    L.zwz_gunzip_files.argtypes = [vp, vp, vp, u32, vp, u64, vp, vp]
    L.zwz_compress_files.argtypes = [vp, vp, vp, u32, i32, vp, u64, vp, vp, vp]
    L.zwz_decompress_records.argtypes = [vp, vp, vp, vp, vp, vp, u32, u32, vp, u64, vp, vp, vp, vp, u32]
    L.zwz_ctx_tune.argtypes = [vp, i32, u64]
    L.zwz_compress_files_async.argtypes = [vp, vp, vp, u32, i32, vp, u64, vp, vp, vp, vp]
    L.zwz_decompress_records_async.argtypes = [vp, vp, vp, vp, vp, vp, u32, u32, vp, u64, vp, vp, vp, vp, u32, vp]
    L.zwz_wait.argtypes = [vp, u64]
    L.zwz_profile_enable.argtypes = [vp, i32]
    L.zwz_profile_read.argtypes = [vp, vp, vp, i32]
    dp = C.POINTER(_Dicts)
    L.zwz_deflate_batch_device_dict.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, i32, i32, dp, vp]
    L.zwz_deflate_batch_dict.argtypes = [vp, vp, vp, vp, u32, vp, u64, vp, vp, i32, i32, dp]
    L.zwz_inflate_batch_device_dict.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, vp, u32, dp, vp]
    L.zwz_inflate_batch_dict.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp, vp, u32, dp]
    return L


def load_library(path: Optional[str] = None):
    """dlopen the CUDA extension. Fails loudly when it has not been built: there is no other implementation."""
    global _LIB
    if path is None:
        if _LIB is not None:
            return _LIB
        path = library_path()
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
                               "(or __graft_entry__.build()). This package has no CPU fallback.")
        _LIB = _declare(C.CDLL(path))
        return _LIB
    return _declare(C.CDLL(path))


def deflate_bound(raw_len) -> np.ndarray:
    """zwz_deflate_bound(): capacity a chunk's output slot must have."""
    return ((np.asarray(raw_len, dtype=np.uint64) + np.uint64(48 + 15)) & ~np.uint64(15)).astype(np.uint64)


def chunk_table(file_offs) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """The reference's chunking rule (compression.cpp:52-64): a file of S bytes yields floor(S/65535)+1 chunks, the last
    one holding S mod 65535 bytes (0 for empty files and exact multiples). file_offs[n+1] ->
    (chunk_off u64, chunk_len u32, chunk_file i32, sequence_id i32)."""
    file_offs = np.asarray(file_offs, dtype=np.int64)
    sizes = np.diff(file_offs)
    nch = sizes // CHUNK_SIZE + 1
    cfile = np.repeat(np.arange(len(sizes), dtype=np.int64), nch)
    first = np.cumsum(nch) - nch
    seq = np.arange(int(nch.sum()), dtype=np.int64) - first[cfile]
    coff = file_offs[:-1][cfile] + seq * CHUNK_SIZE
    clen = np.minimum(CHUNK_SIZE, sizes[cfile] - seq * CHUNK_SIZE)
    return coff.astype(np.uint64), clen.astype(np.uint32), cfile.astype(np.int32), seq.astype(np.int32)


def _ptr(a) -> Optional[int]:
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data if a.size else None


def _u8(a) -> np.ndarray:
    if isinstance(a, (bytes, bytearray, memoryview)):
        return np.frombuffer(a, dtype=np.uint8)
    a = np.asarray(a)
    assert a.dtype == np.uint8
    return np.ascontiguousarray(a)


class Context:
    """One GPU's worth of streams and arenas (``zwz_ctx``)."""

    def __init__(self, device: int = 0, library=None):
        self.lib = library if library is not None else load_library()
        h = C.c_void_p()
        rc = self.lib.zwz_init(device, C.byref(h))
        if rc != 0:
            raise ZwzError(rc, "zwz_init failed: no usable sm_100a device (this package has no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.zwz_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise ZwzError(rc, self.lib.zwz_last_error(self.h).decode())

    @property
    def launches(self) -> int:
        return int(self.lib.zwz_launch_count(self.h))

    PROF_KINDS = ("lz_match", "deflate_encode", "inflate", "md5", "pack", "adler32")

    TUNE_DEFLATE_SUBBATCH_BYTES = 1
    TUNE_HOST_THREADS = 2
    TUNE_HOST_PARALLEL_MIN = 3

    def tune(self, what: int, value: int):
        """zwz_ctx_tune: e.g. TUNE_DEFLATE_SUBBATCH_BYTES (raw bytes per internal deflate pass; the scratch is 6 bytes per raw byte of one pass),
        TUNE_HOST_THREADS (host threads that stage a call's descriptors; 0 = min(8, cores / 2), 1 = the calling thread alone) and
        TUNE_HOST_PARALLEL_MIN (calls with fewer entries stay on the calling thread; default 32 768)."""
        self._check(self.lib.zwz_ctx_tune(self.h, what, value))

    def profile_enable(self, on: bool = True):
        self._check(self.lib.zwz_profile_enable(self.h, 1 if on else 0))

    def profile_read(self, reset: bool = True):
        """{kernel: (milliseconds, launches)} measured with CUDA events on the launching stream since the last reset."""
        ms = np.zeros(len(self.PROF_KINDS), dtype=np.float64)
        cnt = np.zeros(len(self.PROF_KINDS), dtype=np.uint64)
        self._check(self.lib.zwz_profile_read(self.h, ms.ctypes.data, cnt.ctypes.data, 1 if reset else 0))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROF_KINDS)}

    def props(self):
        sm, ma, mi, mem = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        self._check(self.lib.zwz_device_props(self.h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "total_mem": mem.value}

    # ---- raw memory helpers (so callers without torch can keep data resident) ----
    def malloc_device(self, n: int) -> int:
        p = C.c_void_p()
        self._check(self.lib.zwz_malloc_device(self.h, n, C.byref(p)))
        return p.value

    def free_device(self, p: int):
        self._check(self.lib.zwz_free_device(self.h, p))

    def h2d(self, dptr: int, a: np.ndarray):
        self._check(self.lib.zwz_memcpy_h2d(self.h, dptr, _ptr(a), a.nbytes))

    def d2h(self, a: np.ndarray, dptr: int):
        self._check(self.lib.zwz_memcpy_d2h(self.h, _ptr(a), dptr, a.nbytes))

    def sync(self):
        self._check(self.lib.zwz_sync(self.h))

    # ---- deflate: compression.cpp:119-134 ----
    def deflate_batch(self, raw, off, length, level: int = 0, format: str = "zlib", zdict=None, zdict_index=None):
        """Host buffers. Returns (packed uint8 array, packed_off[n+1] u64, results[n] RESULT_DTYPE). format: "zlib", "gzip" (one
        BGZF member per chunk, chunks <= BGZF_BLOCK) or "raw". zdict: a preset dictionary as in Python's zlib (bytes, one for all
        chunks), or a list of them with zdict_index (the dictionary of every chunk, NO_DICT for none); not in gzip format."""
        raw = _u8(raw)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        n = len(off)
        cap = int(deflate_bound(length).sum()) if n else 0
        out = np.empty(max(cap, 1), dtype=np.uint8)
        poff = np.zeros(n + 1, dtype=np.uint64)
        res = np.zeros(n, dtype=RESULT_DTYPE)
        dicts, _keep = _dicts(zdict, zdict_index, n, device=False)
        self._check(self.lib.zwz_deflate_batch_dict(self.h, _ptr(raw), _ptr(off), _ptr(length), n, _ptr(out), cap, poff.ctypes.data,
                                                    _ptr(res), level, _format(format), dicts))
        return out[:int(poff[n])], poff, res

    def deflate_batch_device(self, d_raw: int, off, length, d_out: int, out_off, level: int = 0, stream: int = 0, format: str = "zlib",
                             zdict=None, zdict_index=None):
        """Device buffers. zdict: (device pointer, offsets[ndict+1]) of the preset dictionaries, with zdict_index as in deflate_batch."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        out_off = np.ascontiguousarray(out_off, dtype=np.uint64)
        n = len(off)
        res = np.zeros(n, dtype=RESULT_DTYPE)
        dicts, _keep = _dicts(zdict, zdict_index, n, device=True)
        self._check(self.lib.zwz_deflate_batch_device_dict(self.h, d_raw, _ptr(off), _ptr(length), n, d_out, _ptr(out_off), _ptr(res), level,
                                                           _format(format), dicts, stream or None))
        return res

    def pack_streams_device(self, d_slots: int, slot_off, res, d_packed: int, stream: int = 0) -> np.ndarray:
        """Slots -> packed payload bytes on the device; returns packed_off[n+1]."""
        slot_off = np.ascontiguousarray(slot_off, dtype=np.uint64)
        res = np.ascontiguousarray(res)
        n = len(slot_off)
        poff = np.zeros(n + 1, dtype=np.uint64)
        self._check(self.lib.zwz_pack_streams_device(self.h, d_slots, _ptr(slot_off), _ptr(res), n, d_packed, poff.ctypes.data, stream or None))
        return poff

    # ---- inflate: decompression.cpp:11-37 ----
    def inflate_batch(self, comp, off, length, raw_off, flags: int = 0, format: str = "zlib", zdict=None, zdict_index=None):
        """Host buffers. raw_off[n+1] gives every stream's output window. Returns (raw_out, raw_len[n], status[n]).
        format: "zlib", "gzip" (one member per stream, as zlib with windowBits 31) or "raw". zdict / zdict_index: preset
        dictionaries as in deflate_batch (what zlib.decompressobj(wbits, zdict=) is given); not in gzip format."""
        comp = _u8(comp)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        raw_off = np.ascontiguousarray(raw_off, dtype=np.uint64)
        n = len(off)
        out = np.zeros(max(int(raw_off[n]) if n else 0, 1), dtype=np.uint8)
        rl = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.uint32)
        dicts, _keep = _dicts(zdict, zdict_index, n, device=False)
        self._check(self.lib.zwz_inflate_batch_dict(self.h, _ptr(comp), _ptr(off), _ptr(length), n, _ptr(out), _ptr(raw_off), _ptr(rl), _ptr(st),
                                                    flags | (_format(format) << 8), dicts))
        return out, rl, st

    def inflate_batch_device(self, d_comp: int, off, length, d_raw_out: int, raw_off, flags: int = 0, stream: int = 0, format: str = "zlib",
                             zdict=None, zdict_index=None):
        """Device buffers. zdict: (device pointer, offsets[ndict+1]) of the preset dictionaries, with zdict_index as in deflate_batch."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        raw_off = np.ascontiguousarray(raw_off, dtype=np.uint64)
        n = len(off)
        rl = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.uint32)
        dicts, _keep = _dicts(zdict, zdict_index, n, device=True)
        self._check(self.lib.zwz_inflate_batch_device_dict(self.h, d_comp, _ptr(off), _ptr(length), n, d_raw_out, _ptr(raw_off), _ptr(rl), _ptr(st),
                                                           flags | (_format(format) << 8), dicts, stream or None))
        return rl, st

    def decompress_records(self, comp, off, length, rec_cap, rec_file, nf: int, out_cap: int, want_md5: bool = True, flags: int = 0):
        """Worker side of decompression.cpp:100-151 for a group of records (host buffers): inflate every record, concatenate the
        records of each file in order, MD5 every file. Returns (files, file_off[nf+1], raw_len[n], status[n], digest[nf,16])."""
        comp = _u8(comp)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        rec_cap = np.ascontiguousarray(rec_cap, dtype=np.uint32)
        rec_file = np.ascontiguousarray(rec_file, dtype=np.uint32)
        n = len(off)
        files = np.zeros(max(out_cap, 1), dtype=np.uint8)
        foff = np.zeros(nf + 1, dtype=np.uint64)
        rl = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.uint32)
        dg = np.zeros((nf, 16), dtype=np.uint8)
        self._check(self.lib.zwz_decompress_records(self.h, _ptr(comp), _ptr(off), _ptr(length), _ptr(rec_cap), _ptr(rec_file), n, nf, _ptr(files),
                                                    out_cap, _ptr(foff), _ptr(rl), _ptr(st), _ptr(dg) if want_md5 else None, flags))
        return files, foff, rl, st, dg

    # ---- the host-buffer calls with caller-owned (page-locked) buffers given by address: what host/compress_pipeline.cpp and
    # host/decompress_pipeline.cpp do per batch; bench.py times these for its end-to-end number ----
    def compress_files_into(self, data_ptr: int, file_off, level: int, out_ptr: int, out_cap: int, want_md5: bool = True):
        """zwz_compress_files on raw addresses. file_off[nf+1] is relative to data_ptr. Returns (packed_off, results, digests)."""
        file_off = np.ascontiguousarray(file_off, dtype=np.uint64)
        nf = len(file_off) - 1
        sizes = np.diff(file_off.astype(np.int64))
        nc = int((sizes // CHUNK_SIZE + 1).sum())
        poff = np.zeros(nc + 1, dtype=np.uint64)
        res = np.zeros(nc, dtype=RESULT_DTYPE)
        dg = np.zeros((nf, 16), dtype=np.uint8) if want_md5 else None
        self._check(self.lib.zwz_compress_files(self.h, data_ptr, _ptr(file_off), nf, level, out_ptr, out_cap, poff.ctypes.data, _ptr(res),
                                                _ptr(dg) if want_md5 else None))
        return poff, res, dg

    def decompress_records_into(self, comp_ptr: int, off, length, rec_cap, rec_file, nf: int, out_ptr: int, out_cap: int, want_md5: bool = True,
                                flags: int = 0):
        """zwz_decompress_records on raw addresses. Returns (file_off[nf+1], raw_len[n], status[n], digests)."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        rec_cap = np.ascontiguousarray(rec_cap, dtype=np.uint32)
        rec_file = np.ascontiguousarray(rec_file, dtype=np.uint32)
        n = len(off)
        foff = np.zeros(nf + 1, dtype=np.uint64)
        rl = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.uint32)
        dg = np.zeros((nf, 16), dtype=np.uint8) if want_md5 else None
        self._check(self.lib.zwz_decompress_records(self.h, comp_ptr, _ptr(off), _ptr(length), _ptr(rec_cap), _ptr(rec_file), n, nf, out_ptr,
                                                    out_cap, _ptr(foff), _ptr(rl), _ptr(st), _ptr(dg) if want_md5 else None, flags))
        return foff, rl, st, dg

    def deflate_batch_into(self, raw_ptr: int, off, length, out_ptr: int, out_cap: int, level: int = 0, format: str = "zlib"):
        """zwz_deflate_batch on raw addresses. Returns (packed_off[n+1], results[n])."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        n = len(off)
        poff = np.zeros(n + 1, dtype=np.uint64)
        res = np.zeros(n, dtype=RESULT_DTYPE)
        self._check(self.lib.zwz_deflate_batch_ex(self.h, raw_ptr, _ptr(off), _ptr(length), n, out_ptr, out_cap, poff.ctypes.data, _ptr(res), level,
                                                  _format(format)))
        return poff, res

    def inflate_batch_into(self, comp_ptr: int, off, length, out_ptr: int, raw_off, flags: int = 0, format: str = "zlib"):
        """zwz_inflate_batch on raw addresses (raw_off[n+1] relative to out_ptr). Returns (raw_len[n], status[n])."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        raw_off = np.ascontiguousarray(raw_off, dtype=np.uint64)
        n = len(off)
        rl = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.zwz_inflate_batch(self.h, comp_ptr, _ptr(off), _ptr(length), n, out_ptr, _ptr(raw_off), _ptr(rl), _ptr(st),
                                               flags | (_format(format) << 8)))
        return rl, st

    # ---- MD5: verification.cpp:13-27 ----
    def md5_batch(self, data, off, length) -> np.ndarray:
        data = _u8(data)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint64)
        n = len(off)
        dg = np.zeros((n, 16), dtype=np.uint8)
        self._check(self.lib.zwz_md5_batch(self.h, _ptr(data), _ptr(off), _ptr(length), n, _ptr(dg)))
        return dg

    def md5_batch_device(self, d_data: int, off, length, stream: int = 0) -> np.ndarray:
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint64)
        n = len(off)
        dg = np.zeros((n, 16), dtype=np.uint8)
        self._check(self.lib.zwz_md5_batch_device(self.h, d_data, _ptr(off), _ptr(length), n, _ptr(dg), stream or None))
        return dg

    def md5_stream_device(self, d_data: int, total_len: int, piece: int = 1 << 26) -> bytes:
        """One long file digested in pieces through the update/final pair (the MD5_Update loop of verification.cpp:16-19)."""
        state = np.zeros(4, dtype=np.uint32)
        self.lib.zwz_md5_state_init(_ptr(state), 1)
        piece -= piece % 64
        off = np.zeros(1, dtype=np.uint64)   # kept alive across the calls: ctypes only sees their addresses
        ln = np.zeros(1, dtype=np.uint64)
        tot = np.array([total_len], dtype=np.uint64)
        done = 0
        while total_len - done >= 64:
            step = min(piece, (total_len - done) // 64 * 64)
            off[0], ln[0] = done, step
            self._check(self.lib.zwz_md5_update_device(self.h, _ptr(state), d_data, _ptr(off), _ptr(ln), 1, None))
            done += step
        dg = np.zeros(16, dtype=np.uint8)
        off[0], ln[0] = done, total_len - done
        self._check(self.lib.zwz_md5_final_device(self.h, _ptr(state), d_data, _ptr(off), _ptr(ln), _ptr(tot), 1, _ptr(dg), None))
        return dg.tobytes()

    def adler32_batch_device(self, d_data: int, off, length, stream: int = 0) -> np.ndarray:
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        n = len(off)
        out = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.zwz_adler32_batch_device(self.h, d_data, _ptr(off), _ptr(length), n, _ptr(out), stream or None))
        return out

    def crc32_batch_device(self, d_data: int, off, length, stream: int = 0) -> np.ndarray:
        """CRC-32 (RFC 1952, what zlib.crc32 computes) of every range d_data[off[i] .. off[i]+length[i]), one warp each."""
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        n = len(off)
        out = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.zwz_crc32_batch_device(self.h, d_data, _ptr(off), _ptr(length), n, _ptr(out), stream or None))
        return out

    # ---- whole files <-> BGZF .gz files ----
    def gzip_files(self, data, file_off, level: int = 0):
        """File i = data[file_off[i] .. file_off[i+1]) -> its BGZF .gz file out[gz_off[i] .. gz_off[i+1]) (readable by gzip -d,
        zcat, Python's gzip, htslib). Returns (out uint8 array, gz_off[nf+1] u64)."""
        data = _u8(data)
        file_off = np.ascontiguousarray(file_off, dtype=np.uint64)
        nf = len(file_off) - 1
        cap = int(self.lib.zwz_gzip_bound(_ptr(file_off), nf))
        out = np.empty(max(cap, 1), dtype=np.uint8)
        gz_off = np.zeros(nf + 1, dtype=np.uint64)
        self._check(self.lib.zwz_gzip_files(self.h, _ptr(data), _ptr(file_off), nf, level, _ptr(out), cap, _ptr(gz_off)))
        return out[:int(gz_off[nf])], gz_off

    def gunzip_files(self, gz, gz_off, out_cap: Optional[int] = None):
        """BGZF file i = gz[gz_off[i] .. gz_off[i+1]) -> (out uint8 array, out_off[nf+1] u64, status[nf]): file i's bytes are
        out[out_off[i] .. out_off[i+1]), status[i] STREAM_END when the whole file decoded cleanly. out_cap defaults to
        zwz_gunzip_bound (a smaller one raises ZwzError with ZWZ_E_CAPACITY)."""
        gz = _u8(gz)
        gz_off = np.ascontiguousarray(gz_off, dtype=np.uint64)
        nf = len(gz_off) - 1
        if out_cap is None:
            out_cap = int(self.lib.zwz_gunzip_bound(_ptr(gz), _ptr(gz_off), nf))
        out = np.empty(max(out_cap, 1), dtype=np.uint8)
        out_off = np.zeros(nf + 1, dtype=np.uint64)
        st = np.zeros(max(nf, 1), dtype=np.uint32)
        self._check(self.lib.zwz_gunzip_files(self.h, _ptr(gz), _ptr(gz_off), nf, _ptr(out), out_cap, _ptr(out_off), _ptr(st)))
        return out[:int(out_off[nf])], out_off, st[:nf]


def md5_hex(digests: np.ndarray):
    """verification.cpp:24-27: 16 digest bytes -> 32 lowercase hex characters."""
    d = np.asarray(digests, dtype=np.uint8).reshape(-1, 16)
    return [bytes(r).hex() for r in d]
