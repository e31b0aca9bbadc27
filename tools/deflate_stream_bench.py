"""One long input deflated into one stream on the GPU (zwz_deflate_stream*, zwz_deflater): GB/s of raw input, sizes, and what the
windows cost.

Corpora: those of tools/inflater_bench.py, 256 MiB of text and 256 MiB of the C2 mix. For each it times
  - compress_stream_device (zlib format) at the default level and at levels 1 and 9, input and output resident in device memory;
  - compress_stream, the host form (the upload and download are part of the call);
  - the deflater's device form with 1, 16, 64 and 256 MiB feeds (NO_FLUSH, then FINISH);
  - deflate_batch_device_ex (raw format) on the same bytes cut into independent 65 535-byte chunks: the same kernels without windows;
  - CPU zlib.compress level 6 on one thread;
  - a pigz-style CPU baseline: 128 KiB blocks, each primed with the 32 KiB in front of it as zdict and ended with Z_SYNC_FLUSH (the
    last with Z_FINISH), on all host cores with Python threads (zlib releases the GIL).
Each GPU way runs once to warm up, then the best of --reps counts (host clock around calls that end in a synchronise). The CPU ways
run once. Every stream is decoded by CPU zlib and compared with the input.
Profile spans (zwz_profile_*) of one zlib-format compress_stream_device call at the default level, in a run of its own: there the
"adler32" kind is dict_chain_kernel alone (the windows' hash chains; the zlib format launches no CRC-32).
Sizes: ours / zlib.compress(level 6) of the whole input, and ours / the BGZF file gzip_files writes.
The GPU's name, power limit and clocks are read in the same run. Writes one JSON file.
    python tools/deflate_stream_bench.py --out /tmp/deflate_stream_bench.json [--reps 3]"""
import argparse
import concurrent.futures as cf
import json
import os
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zwz_b200 as z  # noqa: E402
from tools.inflater_bench import best, corpora, gpu_env  # noqa: E402

MiB = 1 << 20
FEEDS = [1 * MiB, 16 * MiB, 64 * MiB, 256 * MiB]
WBITS = {"gzip": 31, "zlib": 15, "raw": -15}


def pigz_like(raw, threads, block=128 << 10):
    def one(i):
        a = i * block
        co = zlib.compressobj(6, zlib.DEFLATED, -15, zdict=raw[max(0, a - 32768):a]) if a else zlib.compressobj(6, zlib.DEFLATED, -15)
        last = a + block >= len(raw)
        return co.compress(raw[a:a + block]) + co.flush(zlib.Z_FINISH if last else zlib.Z_SYNC_FLUSH)
    with cf.ThreadPoolExecutor(threads) as ex:
        body = b"".join(ex.map(one, range(-(-len(raw) // block))))
    return b"\x78\x9c" + body + zlib.adler32(raw).to_bytes(4, "big")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--size-mib", type=int, default=256)
    a = ap.parse_args()
    import torch
    res = {"gpu": gpu_env(), "host_cores": os.cpu_count(), "size_bytes": a.size_mib * MiB, "corpora": {}}
    ctx = z.Context(0)
    for name, raw in corpora(a.size_mib * MiB).items():
        n = len(raw)
        r = {}
        src = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
        cap = z.deflate_stream_bound(n)
        dout = torch.empty(cap, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

        def dev(level):
            return ctx.compress_stream_device(src.data_ptr(), n, dout.data_ptr(), cap, "zlib", level)
        for level in (0, 1, 9):
            t = best(lambda: dev(level), a.reps)
            m = dev(level)
            assert zlib.decompress(dout[:m].cpu().numpy().tobytes()) == raw
            r[f"device_level{level}"] = {"s": t, "GBps": n / t / 1e9, "bytes": m}
        m0 = r["device_level0"]["bytes"]
        host = ctx.compress_stream(raw, "zlib")
        assert host == dout[:dev(0)].cpu().numpy().tobytes()
        t = best(lambda: ctx.compress_stream(raw, "zlib"), a.reps)
        r["host"] = {"s": t, "GBps": n / t / 1e9}
        qout = torch.empty(cap, dtype=torch.uint8, device="cuda")
        for feed in FEEDS:
            def deflater():
                f = ctx.compressobj("zlib")
                p = total = 0
                while True:
                    k = min(feed, n - p)
                    fl = z.FINISH if p + k == n else z.NO_FLUSH
                    total += f.feed_device(src.data_ptr() + p, k, qout.data_ptr() + total, cap - total, fl)
                    p += k
                    if fl == z.FINISH:
                        break
                assert f.queued_out == 0
                f.close()
                return total
            t = best(deflater, a.reps)
            assert deflater() == m0 and torch.equal(qout[:m0], dout[:m0])
            r[f"deflater_feed_{feed // MiB}MiB"] = {"s": t, "GBps": n / t / 1e9}
        off = np.arange(0, n, 65535, dtype=np.uint64)
        ln = np.minimum(65535, n - off).astype(np.uint32)
        boff = np.cumsum(np.concatenate([[0], z.deflate_bound(ln)[:-1]])).astype(np.uint64)
        bout = torch.empty(int(z.deflate_bound(ln).sum()), dtype=torch.uint8, device="cuda")
        t = best(lambda: ctx.deflate_batch_device(src.data_ptr(), off, ln, bout.data_ptr(), boff, format="raw"), a.reps)
        r["batch_independent_65535"] = {"s": t, "GBps": n / t / 1e9}
        r["stream_over_batch_rate"] = r["device_level0"]["GBps"] / r["batch_independent_65535"]["GBps"]
        ctx.profile_enable(True)
        ctx.profile_read(reset=True)
        t0 = time.perf_counter()
        dev(0)
        wall = time.perf_counter() - t0
        prof = ctx.profile_read(reset=True)
        ctx.profile_enable(False)
        r["profile_device_level0"] = {"wall_ms": wall * 1e3, "kernels": prof,
                                      "dict_chain_share": prof["adler32"][0] / max(1e-9, sum(v[0] for v in prof.values()))}
        t0 = time.perf_counter()
        z6 = zlib.compress(raw, 6)
        tz = time.perf_counter() - t0
        r["cpu_zlib6_1thread"] = {"s": tz, "GBps": n / tz / 1e9, "bytes": len(z6)}
        t0 = time.perf_counter()
        pz = pigz_like(raw, os.cpu_count())
        tp = time.perf_counter() - t0
        assert zlib.decompress(pz) == raw
        r["cpu_pigz_like"] = {"s": tp, "GBps": n / tp / 1e9, "bytes": len(pz), "threads": os.cpu_count()}
        gz, _ = ctx.gzip_files(raw, np.array([0, n], dtype=np.uint64))
        sizes = {"zlib6_whole": len(z6), "bgzf_gzip_files": len(gz)}
        for fmt in WBITS:
            c = ctx.compress_stream(raw, fmt)
            d = zlib.decompressobj(WBITS[fmt])
            assert d.decompress(c) == raw and d.eof and not d.unused_data
            sizes[f"stream_{fmt}"] = len(c)
        sizes["stream_gzip_over_zlib6"] = sizes["stream_gzip"] / len(z6)
        sizes["stream_gzip_over_bgzf"] = sizes["stream_gzip"] / len(gz)
        r["sizes"] = sizes
        res["corpora"][name] = r
        print(name, json.dumps(r), flush=True)
        del src, dout, qout, bout
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_env()
    ctx.close()
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
