"""A/B of two emulator builds of the library (tests/simt: libzwz_emu.so of two source trees) on the calls that existed before the
streaming inflater: the seeded inputs of profiles/stream_batch/ab_emu.py through zwz_inflate_stream (with and without OUTPUT_FULL)
and zwz_inflate_stream_index (saved blobs at two spacings), plus zwz_inflate_stream_batch over all of them at once and under a
scratch budget that cuts them into waves. Bytes, lengths, statuses, needed sizes, blobs and the zwz_emu_stream_stats counters
must be identical.
    python profiles/inflater/ab_emu.py a/tests/simt/libzwz_emu.so b/tests/simt/libzwz_emu.so"""
import hashlib
import importlib.util
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def _load(name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "profiles", rel))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


single = _load("stream_batch_ab_emu", "stream_batch/ab_emu.py")  # puts profiles/careful_core first on sys.path
from ab_emu import stream_inputs  # noqa: E402  profiles/careful_core/ab_emu.py
stats = single.stats


def run(lib_path):
    lines = single.run(lib_path)
    import zwz_b200
    ctx = zwz_b200.Context(0, library=zwz_b200.load_library(os.path.abspath(lib_path)))
    ctx.tune(zwz_b200.Context.TUNE_STREAM_SPAN_BYTES, 4096)
    by_fmt = {}
    for fmt, comp in stream_inputs():
        by_fmt.setdefault(fmt, []).append(comp)
    stats(ctx.lib.zwz_emu_stream_stats)
    for budget in (0, 300000):
        ctx.tune(zwz_b200.Context.TUNE_STREAM_SCRATCH_BYTES, budget)
        for fmt, streams in sorted(by_fmt.items()):
            comp = b"".join(streams)
            off = np.cumsum([0] + [len(s) for s in streams[:-1]]).astype(np.uint64)
            ln = np.array([len(s) for s in streams], dtype=np.uint64)
            out, out_off, st = ctx.inflate_stream_batch(comp, off, ln, format=fmt)
            lines.append(f"batch {fmt:4s} budget {budget:6d} n {len(streams)}: status {list(map(int, st))} lens {list(map(int, np.diff(out_off)))} "
                         f"needed {list(map(int, ctx.last_needed))} digest {hashlib.sha256(out.tobytes()).hexdigest()[:16]}, "
                         f"stream_stats {stats(ctx.lib.zwz_emu_stream_stats)}")
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


if __name__ == "__main__":
    main()
