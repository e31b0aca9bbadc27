"""Streaming inflater (zwz_inflater, Context.decompressobj) on the GPU: GB/s of decoded output against the size of the feeds.

Corpora: 256 MiB of text and 256 MiB of the C2 mix (text, structured, JPEG-like and random quarters in 16 pieces), each one gzip
member at level 6. For feeds of 1, 16, 64 and 256 MiB it times
  - the device form: input resident in device memory, output drained into a 1 GiB device buffer;
  - the host form: input and output in host memory (the upload and download are part of every call);
  - single-thread CPU zlib.decompressobj with the same feeds;
and one inflate_stream_device call on the same resident bytes. Each GPU way runs once to warm up, then the best of --reps counts
(host clock around calls that end in a synchronise). Every output is checked against the input.

--big: one gzip member of at least 4.5 GiB compressed (a raw-DEFLATE unit ending in Z_FULL_FLUSH repeated, then a final empty
block, CRC-32 and ISIZE), fed end to end in 256 MiB host pieces, with the largest pending_in and queued_out seen.

The GPU's name, power limit and clocks are read in the same run. Writes one JSON file.
    python tools/inflater_bench.py --out /tmp/inflater_bench.json [--reps 2] [--big]"""
import argparse
import gzip
import json
import os
import struct
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zwz_b200 as z  # noqa: E402
from tools import corpus  # noqa: E402

MiB = 1 << 20
FEEDS = [1 * MiB, 16 * MiB, 64 * MiB, 256 * MiB]


def gpu_env():
    q = "name,power.limit,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip()


def corpora(size):
    text = corpus.gen_text(size, 596, 1).tobytes()
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    c2 = b"".join(gens[i % 4](size // 16, 596, i).tobytes() for i in range(16))
    return {"text": text, "c2": c2}


def best(f, reps):
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t0)
    return min(ts)


def device_form(ctx, d_in, n, d_out, out_cap, feed, raw_len):
    f = ctx.decompressobj("gzip")
    total, p = 0, 0
    while True:
        k = min(feed, n - p)
        final = p + k == n
        got, st = f.feed_device(d_in + p, k, d_out, out_cap, final=final)
        total += got
        while st == z.STREAM_MORE and f.queued_out:
            got, st = f.feed_device(0, 0, d_out, out_cap, final=final)
            total += got
        p += k
        if final:
            break
    f.close()
    assert (st, total) == (z.STREAM_END, raw_len), (st, total)


def host_form(ctx, comp, feed, raw):
    f = ctx.decompressobj("gzip")
    a = np.frombuffer(comp, dtype=np.uint8)
    o = 0
    for p in range(0, len(comp), feed):
        got = f.decompress(a[p:p + feed])
        assert np.array_equal(got, raw[o:o + got.size])
        o += got.size
    got = f.flush()
    o += got.size
    assert (f.status, o) == (z.STREAM_END, raw.size)
    f.close()


def cpu_form(comp, feed, raw_len):
    d = zlib.decompressobj(31)
    o = 0
    for p in range(0, len(comp), feed):
        o += len(d.decompress(comp[p:p + feed]))
    o += len(d.flush())
    assert o == raw_len


def big_member(ctx):
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    raw = b"".join(gens[i % 4](16 * MiB, 596, 11 + i).tobytes() for i in range(4))
    co = zlib.compressobj(1, zlib.DEFLATED, -15)
    unit = co.compress(raw) + co.flush(zlib.Z_FULL_FLUSH)
    reps = -(-((9 << 29) + 4096) // len(unit))
    crc = 0
    for _ in range(reps):
        crc = zlib.crc32(raw, crc)
    head = b"\x1f\x8b\x08\x00\0\0\0\0\0\xff"
    tail = b"\x03\x00" + struct.pack("<II", crc, (len(raw) * reps) & 0xFFFFFFFF)
    comp_len = len(head) + reps * len(unit) + len(tail)

    def pieces(feed=256 * MiB):  # generated as they are fed: host memory stays at a few hundred MiB
        buf = head
        for _ in range(reps):
            buf += unit
            while len(buf) >= feed:
                yield buf[:feed], False
                buf = buf[feed:]
        yield buf + tail, True
    unit_raw = np.frombuffer(raw, dtype=np.uint8)
    f = ctx.decompressobj("gzip")
    most_pend = most_queue = 0
    out = np.empty(1 << 30, dtype=np.uint8)
    n = np.zeros(1, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint32)
    pos = 0
    t_feed = 0.0
    t0 = time.perf_counter()
    for piece, final in pieces():
        a = np.frombuffer(piece, dtype=np.uint8)
        while True:
            t1 = time.perf_counter()
            ctx._check(ctx.lib.zwz_inflater_feed(f.h, a.ctypes.data if a.size else None, a.size, 1 if final else 0, out.ctypes.data, out.size,
                                                 n.ctypes.data, st.ctypes.data))
            t_feed += time.perf_counter() - t1
            a = a[:0]
            info = f._info()
            most_pend = max(most_pend, info[2])
            most_queue = max(most_queue, info[3] + int(n[0]))
            k = int(n[0])
            o = 0
            while o < k:  # every byte against the repeated unit
                u = pos % unit_raw.size
                m = min(k - o, unit_raw.size - u)
                assert np.array_equal(out[o:o + m], unit_raw[u:u + m]), pos
                o += m
                pos += m
            if int(st[0]) != z.STREAM_MORE or not info[3]:
                break
    wall = time.perf_counter() - t0
    info = f._info()
    f.close()
    assert int(st[0]) == z.STREAM_END and pos == len(raw) * reps and info[0] == comp_len
    return {"compressed_bytes": comp_len, "decoded_bytes": pos, "status": int(st[0]), "total_in": info[0], "total_out": info[1],
            "feed_bytes": 256 * MiB, "calls_s": round(t_feed, 3), "wall_with_generation_and_checks_s": round(wall, 3),
            "gbps_calls": round(pos / t_feed / 1e9, 3), "max_pending_in": most_pend, "max_queued_out": most_queue}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--size", type=int, default=256 * MiB)
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    res = {"gpu": gpu_env(), "size": args.size, "feeds": FEEDS, "corpora": {}}
    ctx = z.Context(0)
    for name, raw in corpora(args.size).items():
        comp = gzip.compress(raw, 6)
        rawa = np.frombuffer(raw, dtype=np.uint8)
        d_in = ctx.malloc_device(len(comp) + 64)
        d_out = ctx.malloc_device(1 << 30)
        d_all = ctx.malloc_device(len(raw) + 64)
        ctx.h2d(d_in, np.frombuffer(comp, dtype=np.uint8))
        r = {"compressed": len(comp), "decoded": len(raw)}

        def one_call():
            assert ctx.inflate_stream_device(d_in, len(comp), d_all, len(raw) + 64) == (len(raw), z.STREAM_END)
        t = best(one_call, args.reps)
        back = np.empty(len(raw), dtype=np.uint8)
        ctx.d2h(back, d_all)
        assert np.array_equal(back, rawa)
        r["inflate_stream_device_gbps"] = round(len(raw) / t / 1e9, 3)
        r["device"], r["host"], r["cpu_zlib_1thread"] = {}, {}, {}
        for feed in FEEDS:
            reps = 1 if feed == FEEDS[0] else args.reps
            t = best(lambda: device_form(ctx, d_in, len(comp), d_out, 1 << 30, feed, len(raw)), reps)
            r["device"][feed // MiB] = round(len(raw) / t / 1e9, 3)
            t = best(lambda: host_form(ctx, comp, feed, rawa), reps)
            r["host"][feed // MiB] = round(len(raw) / t / 1e9, 3)
            if not args.no_cpu:
                t0 = time.perf_counter()
                cpu_form(comp, feed, len(raw))
                r["cpu_zlib_1thread"][feed // MiB] = round(len(raw) / (time.perf_counter() - t0) / 1e9, 3)
            print(name, feed // MiB, r["device"][feed // MiB], r["host"][feed // MiB], r["cpu_zlib_1thread"].get(feed // MiB), flush=True)
        r["device_256_over_one_call"] = round(r["device"][256] / r["inflate_stream_device_gbps"], 3)
        for p in (d_in, d_out, d_all):
            ctx.free_device(p)
        res["corpora"][name] = r
        print(json.dumps({name: r}), flush=True)
    if args.big:
        res["big_member"] = big_member(ctx)
        print(json.dumps(res["big_member"]), flush=True)
    ctx.close()
    res["gpu_after"] = gpu_env()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
