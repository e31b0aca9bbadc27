#!/usr/bin/env python
"""Many ordinary gzip files in one call (Context.inflate_stream_batch_device) against the other ways to read the same set:

  corpora  text-2000x512K   2 000 files of 512 KiB text
           text-256x4M      256 files of 4 MiB text
           loguniform-512   512 files of log-uniform sizes from 4 KiB to 16 MiB (text, about 1 GiB decoded)
           c2-64x16M        64 files of 16 MiB of the C2-shaped mix (corpus.c2_buffer)
           text-1x256M      one 256 MiB file
           Every file is one gzip member written by zlib at level 6 (gzip -6's settings); they are cached in --work.
  batch    inflate_stream_batch_device: input and output resident, one call for the whole corpus
  loop     inflate_stream_device, one call per file, input and output resident
  warp     inflate_batch_device(format="gzip"): one warp per file (every file here is a single member)
  cpu      zlib.decompress of every file, on all cores (multiprocessing: the workers inherit the compressed bytes when the pool
           forks, and only file indices and lengths cross process boundaries)

Every way gets one untimed warm-up pass (the per-file loop: one call on the first file), then GB/s are decoded bytes over the best
of --reps (host clock around work that ends in a synchronise). Every output is checked against the input. Prints one JSON line
with the GPU's name and power limit read in the same run."""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zwz_b200 as zwz  # noqa: E402
from tools import corpus  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or [",,"])[0].split(",")]
    return {"gpu": f[0], "power_limit": f[1] if len(f) > 1 else "", "max_sm_clock": f[2] if len(f) > 2 else ""}


def _gz6(raw):
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    return co.compress(raw) + co.flush()


def corpus_files(name):
    """the raw files of a corpus (slices of one generated buffer at seeded offsets)"""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    if name == "text-2000x512K":
        sizes = [512 << 10] * 2000
    elif name == "text-256x4M":
        sizes = [4 << 20] * 256
    elif name == "loguniform-512":
        sizes = np.exp(np.random.default_rng(7).uniform(np.log(4096), np.log(16 << 20), 512)).astype(np.int64).tolist()
    elif name == "c2-64x16M":
        sizes = [16 << 20] * 64
    else:
        sizes = [256 << 20]
    top = max(sizes)
    if name.startswith("c2"):
        b, _, _ = corpus.c2_buffer(20000)
        b = b.tobytes()
        base = (b * ((top + (8 << 20)) // len(b) + 1))[:top + (8 << 20)]
    else:
        base = corpus.gen_text(top + (8 << 20), 596, 1).tobytes()
    offs = rng.integers(0, 8 << 20, len(sizes))
    return [base[int(o):int(o) + int(s)] for o, s in zip(offs, sizes)]


def load(work, name, pool):
    raws = corpus_files(name)
    path = os.path.join(work, name + ".npz")
    if os.path.exists(path):
        z = np.load(path)
        comp, off = z["comp"].tobytes(), z["off"]
    else:
        parts = pool.map(_gz6, raws, chunksize=1)
        off = np.zeros(len(parts) + 1, dtype=np.uint64)
        np.cumsum([len(p) for p in parts], out=off[1:])
        comp = b"".join(parts)
        np.savez(path + ".tmp.npz", comp=np.frombuffer(comp, dtype=np.uint8), off=off)
        os.replace(path + ".tmp.npz", path)
    return raws, comp, off


_FILES = None  # the compressed files of the corpus being timed, inherited by the CPU pool's workers


def _unz(i):
    return len(zlib.decompress(_FILES[i], 31))


def best(reps, fn, warm=None):
    (warm or fn)()
    ts = []
    r = None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, min(ts)


def main():
    global _FILES
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--work", default=os.path.join(tempfile.gettempdir(), "zwz_stream_batch_bench"))
    ap.add_argument("--corpora", default="text-2000x512K,text-256x4M,loguniform-512,c2-64x16M,text-1x256M")
    ap.add_argument("--ways", default="batch,loop,warp,cpu")
    a = ap.parse_args()
    os.makedirs(a.work, exist_ok=True)
    res = {"bench": "stream_batch", **gpu_info(), "cores": os.cpu_count(), "rows": []}
    ctx = zwz.Context(0)
    pool = mp.get_context("fork").Pool(os.cpu_count())
    ways = a.ways.split(",")
    for name in a.corpora.split(","):
        raws, comp, off = load(a.work, name, pool)
        n = len(raws)
        lens = np.array([len(r) for r in raws], dtype=np.uint64)
        out_off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(lens, out=out_off[1:])
        total = int(out_off[n])
        want = b"".join(raws)
        clen = np.diff(off).astype(np.uint64)
        row = {"corpus": name, "files": n, "raw_bytes": total, "comp_bytes": len(comp)}
        d_comp = ctx.malloc_device(len(comp))
        ctx.h2d(d_comp, np.frombuffer(comp, dtype=np.uint8))
        d_out = ctx.malloc_device(total + 64)
        back = np.empty(total, dtype=np.uint8)

        def check(tag):
            ctx.d2h(back, d_out)
            assert back.tobytes() == want, (name, tag)

        if "batch" in ways:
            (rl, st), t = best(a.reps, lambda: ctx.inflate_stream_batch_device(d_comp, off[:-1], clen, d_out, out_off))
            assert (st == zwz.STREAM_END).all() and np.array_equal(rl, lens), name
            check("batch")
            row.update(batch_s=t, batch_gbps=total / t / 1e9)
        if "loop" in ways:
            def loop():
                for i in range(n):
                    r = ctx.inflate_stream_device(d_comp + int(off[i]), int(clen[i]), d_out + int(out_off[i]), int(lens[i]))
                    assert r == (int(lens[i]), zwz.STREAM_END), (name, i, r)
            _, t = best(a.reps, loop, warm=lambda: ctx.inflate_stream_device(d_comp, int(clen[0]), d_out, int(lens[0])))
            check("loop")
            row.update(loop_s=t, loop_gbps=total / t / 1e9)
        if "warp" in ways:
            (rl, st), t = best(a.reps, lambda: ctx.inflate_batch_device(d_comp, off[:-1], clen.astype(np.uint32), d_out, out_off, format="gzip"))
            assert (st == zwz.STREAM_END).all() and np.array_equal(rl.astype(np.uint64), lens), name
            check("warp")
            row.update(warp_s=t, warp_gbps=total / t / 1e9)
        if "cpu" in ways:
            _FILES = [comp[int(off[i]):int(off[i + 1])] for i in range(n)]
            cpu = mp.get_context("fork").Pool(os.cpu_count())
            got, t = best(a.reps, lambda: cpu.map(_unz, range(n), chunksize=max(1, n // (4 * os.cpu_count()))))
            cpu.close()
            assert got == [len(r) for r in raws]
            row.update(cpu_s=t, cpu_gbps=total / t / 1e9)
        ctx.free_device(d_comp)
        ctx.free_device(d_out)
        res["rows"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    pool.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
