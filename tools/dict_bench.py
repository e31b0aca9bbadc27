"""Preset dictionaries on the device: deflate and inflate of ~2 GB of small text records (64-4 096 B, more than L2 holds) without a
dictionary and with one 32 KiB dictionary, through the device API.

Prints one JSON object: wall time per call (host clock around calls that end in a stream synchronise, after warm-up), GB/s of raw
bytes, the per-kernel device spans of a separate profiled pass (zwz_profile_*), the compressed ratio of both runs, the same
ratio of zlib level 6 with and without zdict on a CPU sample, and the card's name and power limit.

    python tools/dict_bench.py [--gb 2] [--reps 3] [--seed 596]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import zwz_b200  # noqa: E402
from tools import corpus  # noqa: E402


def records(total: int, seed: int):
    """Text records of 64-4 096 B drawn from a 256 MiB generated text: sizes, raw bytes."""
    rng = np.random.default_rng(seed)
    n = int(total / 2080)
    sizes = rng.integers(64, 4097, n).astype(np.uint32)
    text = corpus.gen_text(256 << 20, seed, 1).tobytes()
    starts = rng.integers(0, len(text) - 4096, n)
    raw = np.frombuffer(b"".join(text[int(a):int(a) + int(s)] for a, s in zip(starts, sizes)), dtype=np.uint8)
    return sizes, raw


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement stands without it; say so
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=596)
    ap.add_argument("--sample", type=int, default=2000, help="records compressed with zlib-6 on the CPU")
    a = ap.parse_args()

    sizes, raw = records(int(a.gb * 1e9), a.seed)
    dictionary = np.frombuffer(corpus.gen_text(32768, a.seed, 9999).tobytes(), dtype=np.uint8)
    n = len(sizes)
    off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off[1:])
    slot = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(zwz_b200.deflate_bound(sizes), out=slot[1:])

    out = {"card": card(), "records": n, "raw_bytes": int(raw.size), "dict_bytes": int(dictionary.size)}
    with zwz_b200.Context(0) as ctx:
        d_raw, d_comp, d_back, d_dict = (ctx.malloc_device(int(x)) for x in (raw.size, slot[-1], raw.size, dictionary.size))
        ctx.h2d(d_raw, raw)
        ctx.h2d(d_dict, dictionary)
        zd = (d_dict, [0, dictionary.size])
        for name, kw in (("plain", {}), ("dict", {"zdict": zd})):
            r = {}
            res = ctx.deflate_batch_device(d_raw, off[:-1], sizes, d_comp, slot[:-1], **kw)  # warm-up
            ts = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                res = ctx.deflate_batch_device(d_raw, off[:-1], sizes, d_comp, slot[:-1], **kw)
                ts.append(time.perf_counter() - t0)
            r["deflate_s"] = ts
            r["deflate_GBps"] = raw.size / min(ts) / 1e9
            clen = res["len0"].astype(np.uint32)
            r["ratio"] = float(clen.sum()) / raw.size
            rl, st = ctx.inflate_batch_device(d_comp, slot[:-1], clen, d_back, off, **kw)
            assert (st == 0).all() and (rl == sizes).all()
            ts = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                rl, st = ctx.inflate_batch_device(d_comp, slot[:-1], clen, d_back, off, **kw)
                ts.append(time.perf_counter() - t0)
            r["inflate_s"] = ts
            r["inflate_GBps"] = raw.size / min(ts) / 1e9
            back = np.empty_like(raw)
            ctx.d2h(back, d_back)
            r["exact"] = bool(np.array_equal(back, raw))
            # per-kernel device spans of one deflate and one inflate call, in a pass of their own
            ctx.profile_enable(True)
            ctx.profile_read(reset=True)
            ctx.deflate_batch_device(d_raw, off[:-1], sizes, d_comp, slot[:-1], **kw)
            r["deflate_spans_ms"] = {k: v for k, v in ctx.profile_read(reset=True).items() if v[1]}
            ctx.inflate_batch_device(d_comp, slot[:-1], clen, d_back, off, **kw)
            r["inflate_spans_ms"] = {k: v for k, v in ctx.profile_read(reset=True).items() if v[1]}
            ctx.profile_enable(False)
            if name == "dict":
                comp = np.empty(int(slot[-1]), dtype=np.uint8)
                ctx.d2h(comp, d_comp)
            out[name] = r
        for p in (d_raw, d_comp, d_back, d_dict):
            ctx.free_device(p)

    rng = np.random.default_rng(a.seed + 1)
    pick = rng.choice(n, min(a.sample, n), replace=False)
    zd_bytes = dictionary.tobytes()
    z_plain = z_dict = ours = rawb = 0
    for i in pick:
        rec = raw[int(off[i]):int(off[i + 1])].tobytes()
        c = zlib.compressobj(6, zdict=zd_bytes)
        z_dict += len(c.compress(rec) + c.flush())
        z_plain += len(zlib.compress(rec, 6))
        s = comp[int(slot[i]):int(slot[i]) + int(res["len0"][i])].tobytes()
        assert zlib.decompressobj(zdict=zd_bytes).decompress(s) == rec
        ours += len(s)
        rawb += len(rec)
    out["cpu_sample"] = {"records": len(pick), "zlib6_ratio": z_plain / rawb, "zlib6_zdict_ratio": z_dict / rawb, "ours_zdict_ratio": ours / rawb}
    out["deflate_dict_vs_plain"] = out["dict"]["deflate_GBps"] / out["plain"]["deflate_GBps"]
    out["inflate_dict_vs_plain"] = out["dict"]["inflate_GBps"] / out["plain"]["inflate_GBps"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
