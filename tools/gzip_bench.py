#!/usr/bin/env python
"""Cost of the gzip and raw formats next to zlib on one GPU, on a device-resident C2-shaped corpus (tools/corpus.c2_buffer)
larger than L2, cut into BGZF_BLOCK chunks for all three formats so that they run on the same chunks:

  deflate_batch_device   zlib / gzip / raw         (gzip adds crc32_kernel between the match and encode kernels)
  inflate_batch_device   on each format's output   (gzip checks CRC-32 + ISIZE instead of Adler-32, raw nothing)
  crc32_batch_device     alone
  gzip_files + gunzip_files from page-locked host buffers (upload, kernels, download)

Every leg is warmed up first, then timed over --reps calls: call time with a host clock around calls that end in a device
synchronise, kernel time from the per-kernel CUDA-event spans (Context.profile_read). Outputs are checked against the input.
Prints one JSON line, with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zwz_b200 as zwz  # noqa: E402
from tools import corpus  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def bgzf_chunks(file_off):
    """Every file cut into BGZF_BLOCK chunks (no empty tail chunks): (offsets u64, lengths u32)."""
    B = zwz.BGZF_BLOCK
    file_off = file_off.astype(np.int64)
    sizes = np.diff(file_off)
    n = (sizes + B - 1) // B
    f = np.repeat(np.arange(len(sizes)), n)
    k = np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)
    off = file_off[:-1][f] + k * B
    return off.astype(np.uint64), np.minimum(B, sizes[f] - k * B).astype(np.uint32)


def timed(ctx, reps, fn):
    fn()  # warm-up
    ctx.sync()
    ctx.profile_read(reset=True)
    t0 = time.perf_counter()
    for _ in range(reps):
        r = fn()
    wall = (time.perf_counter() - t0) / reps
    spans = {k: v[0] / reps for k, v in ctx.profile_read(reset=True).items() if v[1]}
    return r, wall, spans


def pinned(ctx, n):
    p = C.c_void_p()
    ctx._check(ctx.lib.zwz_malloc_pinned(ctx.h, max(n, 1), C.byref(p)))
    return p.value, np.ctypeslib.as_array((C.c_uint8 * max(n, 1)).from_address(p.value))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bytes", type=float, default=1.2e9, help="corpus size (>= 1 GB keeps it out of the 126 MB L2)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--level", type=int, default=0)
    a = ap.parse_args()

    sizes = corpus.c2_sizes(370_000)
    nf = int(np.searchsorted(np.cumsum(sizes), a.bytes)) + 1
    host, file_off, _ = corpus.c2_buffer(nf, sizes=sizes[:nf])
    file_off = file_off.astype(np.uint64)
    total = int(file_off[-1])
    off, ln = bgzf_chunks(file_off)
    n = len(off)
    slot = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(zwz.deflate_bound(ln), out=slot[1:])

    ctx = zwz.Context(0)
    ctx.profile_enable(True)
    d_raw = ctx.malloc_device(total + 64)
    d_out = ctx.malloc_device(int(slot[-1]) + 64)
    d_back = ctx.malloc_device(total + 64)
    ctx.h2d(d_raw, host)
    out = {"corpus": "c2", "files": nf, "chunks": n, "raw_bytes": total, "level": a.level, "reps": a.reps, **gpu_info()}

    back = np.empty(total, dtype=np.uint8)
    for fmt in ("zlib", "gzip", "raw"):
        res, wall, spans = timed(ctx, a.reps, lambda: ctx.deflate_batch_device(d_raw, off, ln, d_out, slot[:-1], level=a.level, format=fmt))
        comp = int(res["len0"].sum() + res["len1"].sum())
        out[f"deflate_{fmt}"] = {"compressed_bytes": comp, "ms": round(wall * 1e3, 3), "GBps": round(total / wall / 1e9, 2),
                                 "kernel_ms": {k: round(v, 3) for k, v in spans.items()}}
        assert (res["len1"] == 0).all(), "every chunk is <= BGZF_BLOCK: no split"
        (rl, st), wall, spans = timed(ctx, a.reps, lambda: ctx.inflate_batch_device(d_out, slot[:-1], res["len0"], d_back,
                                                                                     np.append(off, np.uint64(total)), format=fmt))
        assert (st == zwz.STREAM_END).all() and np.array_equal(rl, ln), fmt
        ctx.d2h(back, d_back)
        assert np.array_equal(back, host), fmt
        out[f"inflate_{fmt}"] = {"ms": round(wall * 1e3, 3), "GBps": round(total / wall / 1e9, 2),
                                 "kernel_ms": {k: round(v, 3) for k, v in spans.items()}}

    crc, wall, spans = timed(ctx, a.reps, lambda: ctx.crc32_batch_device(d_raw, off, ln))
    for i in range(0, n, max(1, n // 64)):
        assert int(crc[i]) == zlib.crc32(host[int(off[i]):int(off[i]) + int(ln[i])]), i
    k_ms = spans.get("adler32", float("nan"))  # the checksum-kernel span (ZWZ_PROF_ADLER)
    out["crc32"] = {"ms": round(wall * 1e3, 3), "kernel_ms": round(k_ms, 3), "kernel_GBps": round(total / (k_ms * 1e-3) / 1e9, 1)}
    for p in (d_raw, d_out, d_back):
        ctx.free_device(p)

    # whole files through page-locked host buffers
    p_in, h_in = pinned(ctx, total)
    h_in[:total] = host
    cap = int(ctx.lib.zwz_gzip_bound(file_off.ctypes.data, nf))
    p_gz, _ = pinned(ctx, cap)
    gz_off = np.zeros(nf + 1, dtype=np.uint64)
    _, wall_gz, spans_gz = timed(ctx, a.reps, lambda: ctx._check(ctx.lib.zwz_gzip_files(ctx.h, p_in, file_off.ctypes.data, nf, a.level, p_gz, cap,
                                                                                         gz_off.ctypes.data)))
    gz_bytes = int(gz_off[-1])
    ucap = int(ctx.lib.zwz_gunzip_bound(p_gz, gz_off.ctypes.data, nf))
    p_un, h_un = pinned(ctx, ucap)
    un_off = np.zeros(nf + 1, dtype=np.uint64)
    st = np.zeros(nf, dtype=np.uint32)
    _, wall_un, spans_un = timed(ctx, a.reps, lambda: ctx._check(ctx.lib.zwz_gunzip_files(ctx.h, p_gz, gz_off.ctypes.data, nf, p_un, ucap,
                                                                                           un_off.ctypes.data, st.ctypes.data)))
    assert (st == zwz.STREAM_END).all() and np.array_equal(un_off, file_off) and np.array_equal(h_un[:total], host)
    out["gzip_files"] = {"gz_bytes": gz_bytes, "ms": round(wall_gz * 1e3, 3), "GBps": round(total / wall_gz / 1e9, 2),
                         "kernel_ms": {k: round(v, 3) for k, v in spans_gz.items()}}
    out["gunzip_files"] = {"ms": round(wall_un * 1e3, 3), "GBps": round(total / wall_un / 1e9, 2),
                           "kernel_ms": {k: round(v, 3) for k, v in spans_un.items()}}
    for p in (p_in, p_gz, p_un):
        ctx.lib.zwz_free_pinned(ctx.h, p)
    # rate of the gzip leg as a share of the zlib leg's rate (same bytes: the inverse ratio of the call times)
    out["gzip_vs_zlib_deflate"] = round(out["deflate_zlib"]["ms"] / out["deflate_gzip"]["ms"], 3)
    out["gzip_vs_zlib_inflate"] = round(out["inflate_zlib"]["ms"] / out["inflate_gzip"]["ms"], 3)
    ctx.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
