"""A/B of two emulator builds of the library (tests/simt: libzwz_emu.so of two source trees) on the inflate paths: the batch
decoder with and without the lane-parallel block decoder (with and without preset dictionaries) and the span decoder of
zwz_inflate_stream with 4 KiB spans. Inputs are seeded: zlib, gzip and raw streams of every level and strategy, truncated at
random points and with random bit flips, and the corpora of tests/test_inflate_stream.py. Output bytes, lengths and statuses
must be identical, and so must the emulator counters zwz_emu_inflate_stats and zwz_emu_stream_stats after every group.
    python profiles/careful_core/ab_emu.py a/libzwz_emu.so b/libzwz_emu.so"""
import ctypes as C
import gzip
import hashlib
import os
import random
import subprocess
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from tools import corpus  # noqa: E402

WBITS = {"gzip": 31, "zlib": 15, "raw": -15}
CAREFUL = 2  # ZWZ_INFLATE_CAREFUL: the careful decoder only
STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]


def compress(raw, fmt, level, strategy=zlib.Z_DEFAULT_STRATEGY, zdict=None):
    co = zlib.compressobj(level, zlib.DEFLATED, WBITS[fmt], 8, strategy, **({"zdict": zdict} if zdict else {}))
    return co.compress(raw) + co.flush()


def damaged(s, rng):
    """the stream, some of its prefixes, and copies with one to three bits flipped"""
    out = [s]
    for _ in range(3):
        out.append(s[:rng.randrange(0, len(s) + 1)])
    for _ in range(4):
        b = bytearray(s)
        for _ in range(rng.randint(1, 3)):
            i = rng.randrange(len(b))
            b[i] ^= 1 << rng.randrange(8)
        out.append(bytes(b))
    return out


def batch_sets():
    rng = random.Random(20261021)
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random]
    sets = {}
    for fmt in ("zlib", "gzip", "raw"):
        streams = []
        for i in range(48):
            raw = gens[i % 4](rng.choice([1, 300, 5000, 30000, 65535]), 596, i).tobytes()
            level = rng.choice([0, 1, 6, 9])
            streams += damaged(compress(raw, fmt, level, STRATEGIES[i % 5]), rng)
        sets[fmt] = (streams, None)
    # preset dictionaries: zlib with FDICT (right and wrong dictionary, cut inside the DICTID) and raw
    zd = corpus.gen_text(40000, 596, 77).tobytes()
    for fmt in ("zlib", "raw"):
        streams = []
        for i in range(24):
            raw = corpus.gen_text(rng.choice([100, 4000, 30000]), 596, 100 + i).tobytes()
            streams += damaged(compress(raw, fmt, rng.choice([1, 6, 9]), STRATEGIES[i % 5], zdict=zd), rng)
        sets[fmt + "-dict"] = (streams, zd)
    return sets


def stream_inputs():
    rng = random.Random(5)
    out = []
    for fmt in ("gzip", "zlib", "raw"):
        for level in (0, 1, 6, 9):
            out.append((fmt, compress(corpus.gen_text(200000, 596, level).tobytes(), fmt, level)))
    for st in STRATEGIES[1:]:
        out.append(("gzip", compress(corpus.gen_text(150000, 596, 3).tobytes(), "gzip", 6, st)))
    for g in (corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random):
        out.append(("gzip", compress(g(120000, 596, 11).tobytes(), "gzip", 6)))
    parts = [corpus.gen_text(n, 596, i).tobytes() for i, n in enumerate([5000, 0, 4096, 4095, 30000, 0, 1, 20000])]
    out.append(("gzip", b"".join(gzip.compress(p, 6) for p in parts)))
    out.append(("gzip", b"".join(gzip.compress(bytes([65 + i % 26]) * (i % 7)) for i in range(100))))
    for fmt in ("gzip", "zlib", "raw"):
        s = compress(corpus.gen_text(100000, 596, 21).tobytes(), fmt, 6)
        out += [(fmt, d) for d in damaged(s, rng)[1:]]
    return out


def stats(fn):
    s = (C.c_uint64 * 8)()
    fn(s, 1)
    return list(s)


def run(lib_path):
    """one build in this process: a digest line per group"""
    import zwz_b200
    ctx = zwz_b200.Context(0, library=zwz_b200.load_library(os.path.abspath(lib_path)))
    lines = []
    stats(ctx.lib.zwz_emu_inflate_stats)
    for name, (streams, zd) in batch_sets().items():
        fmt = name.split("-")[0]
        for flags in (0, CAREFUL):
            for cap in (70000, 3000):  # 3000: OUTPUT_FULL on the longer streams
                off = np.zeros(len(streams) + 1, dtype=np.uint64)
                np.cumsum([len(s) for s in streams], out=off[1:])
                ro = np.arange(len(streams) + 1, dtype=np.uint64) * np.uint64(cap)
                kw = {"zdict": zd} if zd else {}
                out, rl, st = ctx.inflate_batch(b"".join(streams), off[:-1], np.diff(off).astype(np.uint32), ro, flags=flags, format=fmt, **kw)
                h = hashlib.sha256()
                for i in range(len(streams)):
                    h.update(out[int(ro[i]):int(ro[i]) + min(int(rl[i]), cap)].tobytes())
                h.update(rl.tobytes())
                h.update(st.tobytes())
                sts = np.bincount(st, minlength=4).tolist()
                lines.append(f"batch {name:9s} flags {flags} cap {cap:5d}: {len(streams)} streams, status counts {sts}, "
                             f"digest {h.hexdigest()[:16]}, inflate_stats {stats(ctx.lib.zwz_emu_inflate_stats)}")
    ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    stats(ctx.lib.zwz_emu_stream_stats)
    for i, (fmt, comp) in enumerate(stream_inputs()):
        out, st = ctx.inflate_stream(comp, format=fmt, out_cap=(1 << 22))
        lines.append(f"stream {i:2d} {fmt:4s} {len(comp):7d} bytes: status {st} len {len(out)} digest "
                     f"{hashlib.sha256(out.tobytes()).hexdigest()[:16]}, stream_stats {stats(ctx.lib.zwz_emu_stream_stats)}")
    ctx.close()
    return lines


def main():
    if sys.argv[1] == "--one":  # child: one build per process
        print("\n".join(run(sys.argv[2])))
        return
    a, b = sys.argv[1], sys.argv[2]
    res = [subprocess.run([sys.executable, os.path.abspath(__file__), "--one", lib], capture_output=True, text=True, check=True).stdout.splitlines()
           for lib in (a, b)]
    bad = abs(len(res[0]) - len(res[1]))
    for la, lb in zip(*res):
        bad += la != lb
        print(("identical  " + la) if la == lb else f"DIFFERENT  {la}\n           {lb}", flush=True)
    print("all results and counters identical" if not bad else f"{bad} groups differ")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
