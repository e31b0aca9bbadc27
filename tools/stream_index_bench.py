#!/usr/bin/env python
"""Seek index of one long stream (Context.inflate_stream_index*, StreamIndex.extract*) on the inputs of stream_inflate_bench.py:
--mib MiB of corpus.gen_text ("text") and of the C2-shaped mix ("c2"), compressed by the gzip binary at -6 (zlib level 6 with a
gzip wrapper when there is no binary). Input and output are resident on the device; a call's time is the host clock around a call
that ends in a synchronise (best of --reps).

  build    inflate_stream_device against inflate_stream_index_device (index only and with output) at spacing 0, 1 MiB and 8 MiB:
           call time, npoints, saved index size
  full     one range [0, raw_len) through a 1 MiB index, against inflate_stream_device: GB/s of output
  random   ranges of 4 KiB and 64 KiB at seeded random offsets, 1, 64 and 4 096 per call, through the 1 MiB index: calls/s,
           ranges/s, bytes delivered per second, and bytes decoded per second (the pieces decode from their access point)

Every extracted range is checked against the input. Prints one JSON line with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zwz_b200 as zwz  # noqa: E402
from tools.stream_inflate_bench import best, compressed, data, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--work", default=os.path.join(tempfile.gettempdir(), "zwz_stream_bench"))
    ap.add_argument("--kinds", default="text,c2")
    a = ap.parse_args()
    os.makedirs(a.work, exist_ok=True)
    size = a.mib << 20
    res = {"bench": "stream_index", "mib": a.mib, **gpu_info(), "rows": []}
    ctx = zwz.Context(0)
    how = "gzip6" if shutil.which("gzip") else "zlib6"
    rng = np.random.default_rng(1)
    for kind in a.kinds.split(","):
        raw = data(kind, size)
        src = np.frombuffer(raw, dtype=np.uint8)
        comp = compressed(a.work, kind, how, raw)
        row = {"data": kind, "comp": how, "raw_bytes": size, "comp_bytes": len(comp)}
        d_comp, d_out = ctx.malloc_device(len(comp)), ctx.malloc_device(size + 64)
        ctx.h2d(d_comp, np.frombuffer(comp, dtype=np.uint8))
        (n, st), t_plain, _ = best(a.reps + 1, lambda: ctx.inflate_stream_device(d_comp, len(comp), d_out, size + 64))
        assert (n, st) == (size, zwz.STREAM_END)
        row["inflate_stream_s"] = t_plain
        row["inflate_stream_gbps"] = size / t_plain / 1e9
        row["build"] = []
        ix1 = None
        for spacing in (0, 1 << 20, 8 << 20):
            (_, st, ix), t_only, _ = best(a.reps, lambda: ctx.inflate_stream_index_device(d_comp, len(comp), None, size + 64, spacing=spacing))
            (_, st2, ix2), t_out, _ = best(a.reps, lambda: ctx.inflate_stream_index_device(d_comp, len(comp), d_out, size + 64, spacing=spacing))
            assert st == st2 == zwz.STREAM_END
            blob = ix.save()
            assert ix2.save() == blob
            row["build"].append({"spacing": spacing, "index_only_s": t_only, "with_output_s": t_out, "npoints": ix.npoints, "index_bytes": len(blob)})
            if spacing == 1 << 20:
                ix1 = ix
            else:
                ix.close()
            ix2.close()
        # the whole stream through the index
        for flags, key in ((0, "full_via_index"), (zwz.INFLATE_CAREFUL, "full_via_index_careful")):
            (got, st), t_full, _ = best(a.reps, lambda: ix1.extract_device(d_comp, len(comp), [0], [size], d_out, [0], flags=flags))
            assert int(st[0]) == zwz.STREAM_END and int(got[0]) == size
            back = np.empty(size, dtype=np.uint8)
            ctx.d2h(back, d_out)
            assert (back == src).all()
            row[key + "_s"] = t_full
            row[key + "_gbps"] = size / t_full / 1e9
        # random reads
        hdr = ix1.save()
        npt = int(np.frombuffer(hdr, dtype="<u8", count=1, offset=32)[0])
        po = np.frombuffer(hdr, dtype=np.dtype([("out", "<u8"), ("bit", "<u8"), ("m", "<u2"), ("b", "u1"), ("p", "u1"), ("w", "<u4")]),
                           count=npt, offset=56)["out"].astype(np.int64)
        row["random"] = []
        for rsize in (4096, 65536):
            for per in (1, 64, 4096):
                calls = max(4, min(64, 16384 // per))
                offs = [rng.integers(0, size - rsize, per).astype(np.uint64) for _ in range(calls)]
                lens = np.full(per, rsize, dtype=np.uint64)
                oo = (np.arange(per) * rsize).astype(np.uint64)
                ix1.extract_device(d_comp, len(comp), offs[0], lens, d_out, oo)  # warm-up
                t0 = time.perf_counter()
                for o in offs:
                    got, st = ix1.extract_device(d_comp, len(comp), o, lens, d_out, oo)
                dt = time.perf_counter() - t0
                assert (st == zwz.STREAM_END).all() and (got == rsize).all()
                back = np.empty(per * rsize, dtype=np.uint8)
                ctx.d2h(back, d_out)
                o = offs[-1].astype(np.int64)
                for i in range(min(per, 64)):
                    assert (back[i * rsize:(i + 1) * rsize] == src[o[i]:o[i] + rsize]).all()
                # bytes decoded: from the last point at or before each range start to its end
                dec = 0
                for o in offs:
                    o = o.astype(np.int64)
                    p = po[np.searchsorted(po, o, side="right") - 1]
                    dec += int((o + rsize - p).sum())
                row["random"].append({"range": rsize, "per_call": per, "calls": calls, "calls_per_s": calls / dt,
                                      "ranges_per_s": calls * per / dt, "delivered_gbps": calls * per * rsize / dt / 1e9,
                                      "decoded_gbps": dec / dt / 1e9, "ms_per_call": dt / calls * 1e3})
        ix1.close()
        ctx.free_device(d_comp)
        ctx.free_device(d_out)
        res["rows"].append(row)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
