"""A/B of two emulator builds of the library (tests/simt: libzwz_emu.so of two source trees) on the one-stream calls, which are
the n = 1 case of the stream batch code: zwz_inflate_stream with 4 KiB spans over the seeded inputs of
profiles/careful_core/ab_emu.py (zlib, gzip and raw streams of every level and strategy, multi-member gzip, truncated and
bit-flipped streams) plus OUTPUT_FULL caps, and zwz_inflate_stream_index's saved blobs at two spacings. Output bytes, lengths,
statuses, blobs and the counters of zwz_emu_stream_stats must be identical.
    python profiles/stream_batch/ab_emu.py a/libzwz_emu.so b/libzwz_emu.so"""
import ctypes as C
import hashlib
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "careful_core"))
from ab_emu import stream_inputs  # noqa: E402


def stats(fn):
    s = (C.c_uint64 * 8)()
    fn(s, 1)
    return list(s)


def run(lib_path):
    # each build with the Python package of its own tree (<tree>/tests/simt/libzwz_emu.so)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(lib_path)))))
    import zwz_b200
    ctx = zwz_b200.Context(0, library=zwz_b200.load_library(os.path.abspath(lib_path)))
    ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    lines = []
    stats(ctx.lib.zwz_emu_stream_stats)
    for i, (fmt, comp) in enumerate(stream_inputs()):
        for cap in (1 << 22, 50000):  # 50000: OUTPUT_FULL on the longer streams
            out, st = ctx.inflate_stream(comp, format=fmt, out_cap=cap)
            need = getattr(ctx, "last_needed", None)
            lines.append(f"stream {i:2d} {fmt:4s} {len(comp):7d} bytes cap {cap:7d}: status {st} len {len(out)} needed {need} digest "
                         f"{hashlib.sha256(out.tobytes()).hexdigest()[:16]}, stream_stats {stats(ctx.lib.zwz_emu_stream_stats)}")
        for spacing in (0, 100000):
            out, st, ix = ctx.inflate_stream_index(comp, format=fmt, spacing=spacing, out_cap=1 << 22)
            blob = ix.save() if ix is not None else b""
            lines.append(f"index  {i:2d} {fmt:4s} spacing {spacing:6d}: status {st} len {len(out)} blob {len(blob)} bytes "
                         f"{hashlib.sha256(blob).hexdigest()[:16]}, stream_stats {stats(ctx.lib.zwz_emu_stream_stats)}")
            if ix is not None:
                ix.close()
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
    print(f"{len(res[0])} groups; " + ("all results, blobs and counters identical" if not bad else f"{bad} groups differ"))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
