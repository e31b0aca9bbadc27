"""A/B of two emulator builds of the library (tests/simt: libzwz_emu.so of two source trees) on the deflate path: every
compressed stream and every result record must be byte-identical. Seeded corpora: C2 files (JPEG-like and bitmap-like), C1
mixed files, C3 text, and chunks spliced from segments of different kinds (noise, text, repeats at any distance, permutation
tables, runs, ramps) with boundaries anywhere relative to the 1 024-byte stretches and 32-position tiles; levels 1, 6 and 9.
    python tools/match_ab_emu.py a/libzwz_emu.so b/libzwz_emu.so [--mb 2]"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import zwz_b200  # noqa: E402
from tools import corpus  # noqa: E402


def fuzz_chunks(total: int, seed: int):
    rng = np.random.default_rng(seed)
    text = corpus.gen_text(200000, 596, 7).tobytes()
    chunks, size = [], 0
    while size < total:
        target = int(rng.choice([rng.integers(1, 3000), rng.integers(1000, 9000), rng.integers(8000, 65536)]))
        c = b""
        while len(c) < target:
            kind = int(rng.integers(0, 6))
            n = int(rng.choice([rng.integers(1, 40), rng.integers(40, 1100), rng.integers(1000, 5000)]))
            if kind == 0:
                seg = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            elif kind == 1:
                o = int(rng.integers(0, len(text) - n))
                seg = text[o:o + n]
            elif kind == 2 and len(c) > 8:  # a copy of earlier bytes, maybe of part of a noise stretch
                o = int(rng.integers(0, len(c)))
                d = c[o:o + n]
                seg = (d * (n // max(len(d), 1) + 1))[:n]
            elif kind == 3:
                p = rng.permutation(256).astype(np.uint8).tobytes()
                seg = (p * (n // 256 + 1))[:n]
            elif kind == 4:
                seg = bytes([int(rng.integers(0, 256))]) * n
            else:
                seg = bytes((np.arange(n) * int(rng.integers(1, 7)) & 255).astype(np.uint8))
            c += seg
        chunks.append(c[:target])
        size += target
    return chunks


def corpora(mb: float):
    nbytes = int(mb * (1 << 20))
    out = {}
    buf, offs, _ = corpus.c2_buffer(max(16, nbytes // 6700), seed=corpus.BASE_SEED + 11)
    out["c2"] = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(len(offs) - 1)]
    buf, offs = corpus.mixed_buffer(nbytes)[:2]
    out["c1"] = [buf[offs[i]:offs[i + 1]].tobytes() for i in range(len(offs) - 1)]
    t = corpus.c3_buffer(nbytes, unit_bytes=1 << 20).tobytes()
    out["c3"] = [t]
    out["fuzz"] = fuzz_chunks(nbytes, 20261020)
    return out


def run(lib_path: str, files, level: int):
    ctx = zwz_b200.Context(0, library=zwz_b200.load_library(os.path.abspath(lib_path)))
    fo = np.zeros(len(files) + 1, dtype=np.int64)
    np.cumsum([len(f) for f in files], out=fo[1:])
    coff, clen, _, _ = zwz_b200.chunk_table(fo)
    raw = np.frombuffer(b"".join(files), dtype=np.uint8)
    packed, poff, res = ctx.deflate_batch(raw, coff, clen, level)
    ctx.close()
    return np.asarray(packed).tobytes(), np.asarray(poff).tobytes(), np.asarray(res).tobytes(), len(coff)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--mb", type=float, default=2.0)
    args = ap.parse_args()
    bad = 0
    for name, files in corpora(args.mb).items():
        for level in (1, 6, 9):
            ra, rb = run(args.a, files, level), run(args.b, files, level)
            same = ra[:3] == rb[:3]
            bad += not same
            print(f"{name:5s} level {level}: {sum(map(len, files)):9d} bytes, {ra[3]:6d} chunks, {len(ra[0]):9d} compressed: "
                  f"{'identical' if same else 'DIFFERENT'}", flush=True)
    print("all streams identical" if not bad else f"{bad} corpora differ")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
