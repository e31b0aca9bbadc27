"""A/B of two emulator builds of the library (tests/simt: libzwz_emu.so of two source trees, each loaded by its own tree's package) on the deflate calls that existed before
the stream deflater: zwz_deflate_batch_dict over seeded text, structured, JPEG-like, random and all-zero chunks of 0 to 65 535 bytes,
in every format and at every level, without dictionaries and with two dictionaries (chunks using dictionary 0, dictionary 1 and none
in one call; gzip takes none), plus zwz_gzip_files over five files. Packed bytes, packed offsets and results must be identical.
    python profiles/deflate_stream/ab_emu.py a/tests/simt/libzwz_emu.so b/tests/simt/libzwz_emu.so"""
import hashlib
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def chunks(seed):
    from tools import corpus
    rng = np.random.default_rng(seed)
    gens = [corpus.gen_text, corpus.gen_struct, corpus.gen_jpeg_like, corpus.gen_random, lambda n, s, u: np.zeros(n, dtype=np.uint8)]
    sizes = [0, 1, 100, 700, 4096, 20000, 65280, 65535] + [int(x) for x in rng.integers(1, 65536, 8)]
    return [gens[i % len(gens)](n, 596, seed + i).tobytes() for i, n in enumerate(sizes)]


def run(lib_path):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(lib_path)))))  # that tree's package
    import zwz_b200
    from tools import corpus
    os.environ.setdefault("ZWZ_EMU_POISON", "5")
    ctx = zwz_b200.Context(0, library=zwz_b200.load_library(os.path.abspath(lib_path)))
    lines = []
    cs = chunks(3)
    raw = b"".join(cs)
    off = np.cumsum([0] + [len(c) for c in cs[:-1]]).astype(np.uint64)
    ln = np.array([len(c) for c in cs], dtype=np.uint32)
    dicts = [corpus.gen_text(40000, 596, 77).tobytes(), corpus.gen_struct(5000, 596, 78).tobytes()]
    idx = np.array([i % 3 if i % 3 < 2 else zwz_b200.NO_DICT for i in range(len(cs))], dtype=np.uint32)
    for fmt in ("zlib", "gzip", "raw"):
        keep = ln <= zwz_b200.BGZF_BLOCK if fmt == "gzip" else np.ones(len(cs), dtype=bool)
        for level in range(10):
            for dname, zd, zi in (("none", None, None), ("two", dicts, idx[keep])):
                if fmt == "gzip" and zd is not None:
                    continue
                out, poff, res = ctx.deflate_batch(raw, off[keep], ln[keep], level=level, format=fmt, zdict=zd, zdict_index=zi)
                lines.append(f"deflate_batch {fmt:4s} level {level} dicts {dname}: bytes {hashlib.sha256(out.tobytes()).hexdigest()[:16]} "
                             f"off {hashlib.sha256(poff.tobytes()).hexdigest()[:16]} res {hashlib.sha256(res.tobytes()).hexdigest()[:16]} "
                             f"total {int(poff[-1])}")
    files = [corpus.gen_text(200000, 596, 5).tobytes(), b"", corpus.gen_random(70000, 596, 6).tobytes(), corpus.gen_struct(65280, 596, 7).tobytes(),
             corpus.gen_jpeg_like(130561, 596, 8).tobytes()]
    data = b"".join(files)
    foff = np.cumsum([0] + [len(f) for f in files]).astype(np.uint64)
    for level in (0, 1, 6, 9):
        gz, gz_off = ctx.gzip_files(data, foff, level)
        lines.append(f"gzip_files level {level}: bytes {hashlib.sha256(gz.tobytes()).hexdigest()[:16]} off {list(map(int, gz_off))}")
    ctx.close()
    return lines


def main():
    if sys.argv[1] == "--one":
        print("\n".join(run(sys.argv[2])))
        return
    res = [subprocess.run([sys.executable, os.path.abspath(__file__), "--one", lib], capture_output=True, text=True, check=True).stdout.splitlines()
           for lib in sys.argv[1:3]]
    bad = abs(len(res[0]) - len(res[1]))
    for la, lb in zip(*res):
        bad += la != lb
        print(("identical  " + la) if la == lb else f"DIFFERENT  {la}\n           {lb}", flush=True)
    print(f"{len(res[0])} groups; " + ("all bytes, offsets and results identical" if not bad else f"{bad} groups differ"))


if __name__ == "__main__":
    main()
