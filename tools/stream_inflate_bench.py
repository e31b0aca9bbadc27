#!/usr/bin/env python
"""One long stream on the whole GPU (Context.inflate_stream*) against the ways the library and the CPU read the same bytes:

  inputs   --mib MiB of corpus.gen_text ("text") and of a C2-shaped mix (corpus.c2_buffer, "c2"), each compressed by the gzip
           binary at -6 (when present) and by zlib at levels 1 and 9 (gzip wrapper); the compressed files are cached in --work
  device   inflate_stream_device with input and output resident (call time, host clock around a call that ends in a synchronise)
  host     inflate_stream from host memory (upload, kernels, download)
  phases   one ZWZ_TRACE run of the device call: per-phase time, span count, repair rounds and re-decoded spans
  one warp inflate_batch_device(format="gzip") on one 32 MiB member of the same data: the per-warp rate of the batch decoder
  cpu      single-threaded zlib.decompress of the same file
  bgzf     gunzip_files of the BGZF form of the same bytes: the "independent members" ceiling

Outputs are checked against the input. Prints one JSON line with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import re
import shutil
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
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def data(kind, size):
    if kind == "text":
        return corpus.gen_text(size, 596, 1).tobytes()
    buf, off, _ = corpus.c2_buffer(20000)
    b = buf.tobytes()
    return (b * (size // len(b) + 1))[:size]


def compressed(work, kind, how, raw):
    path = os.path.join(work, f"{kind}_{len(raw)}_{how}.gz")
    if not os.path.exists(path):
        if how == "gzip6":
            c = subprocess.run(["gzip", "-6", "-c"], input=raw, capture_output=True, check=True).stdout
        else:
            co = zlib.compressobj(int(how[-1]), zlib.DEFLATED, 31)
            c = co.compress(raw) + co.flush()
        with open(path + ".tmp", "wb") as f:
            f.write(c)
        os.replace(path + ".tmp", path)
    with open(path, "rb") as f:
        return f.read()


def best(reps, fn):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, min(ts), float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--work", default=os.path.join(tempfile.gettempdir(), "zwz_stream_bench"))
    ap.add_argument("--kinds", default="text,c2")
    a = ap.parse_args()
    os.makedirs(a.work, exist_ok=True)
    size = a.mib << 20
    res = {"bench": "stream_inflate", "mib": a.mib, **gpu_info(), "rows": []}
    ctx = zwz.Context(0)
    hows = (["gzip6"] if shutil.which("gzip") else []) + ["zlib1", "zlib9"]
    for kind in a.kinds.split(","):
        raw = data(kind, size)
        d_out = ctx.malloc_device(size + 64)
        for how in hows:
            comp = compressed(a.work, kind, how, raw)
            row = {"data": kind, "comp": how, "raw_bytes": size, "comp_bytes": len(comp)}
            d_comp = ctx.malloc_device(len(comp))
            ctx.h2d(d_comp, np.frombuffer(comp, dtype=np.uint8))
            (n, st), tmin, tmed = best(a.reps + 1, lambda: ctx.inflate_stream_device(d_comp, len(comp), d_out, size + 64))
            back = np.empty(size, dtype=np.uint8)
            ctx.d2h(back, d_out)
            assert (n, st) == (size, zwz.STREAM_END) and back.tobytes() == raw, (kind, how, n, st)
            row.update(device_s=tmin, device_median_s=tmed, device_gbps=size / tmin / 1e9)
            (out, st), hmin, _ = best(a.reps, lambda: ctx.inflate_stream(comp, out_cap=size + 64))
            assert st == zwz.STREAM_END and len(out) == size
            row.update(host_s=hmin, host_gbps=size / hmin / 1e9)
            # phases: a run with ZWZ_TRACE on a context of its own (every mark synchronises)
            env = dict(os.environ, ZWZ_TRACE="1")
            code = ("import sys,numpy as np;sys.path.insert(0,%r);import zwz_b200 as z;c=z.Context(0);comp=open(%r,'rb').read();"
                    "d=c.malloc_device(len(comp));o=c.malloc_device(%d);c.h2d(d,np.frombuffer(comp,dtype=np.uint8));"
                    "[c.inflate_stream_device(d,len(comp),o,%d) for _ in range(2)]") % (
                        ROOT, os.path.join(a.work, f"{kind}_{size}_{how}.gz"), size + 64, size + 64)
            tr = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True).stderr.strip().splitlines()
            line = [t for t in tr if "inflate_stream:" in t][-1:] or [""]
            row["phases_ms"] = {k: float(v) for k, v in re.findall(r" (\w+) ([0-9.]+) ms", line[0])}
            row.update({k: int(v) for k, v in re.findall(r" (spans|rounds|reruns) (\d+)", line[0])})
            ctx.free_device(d_comp)
            t0 = time.perf_counter()
            assert zlib.decompress(comp, 31) == raw
            row["cpu_zlib_gbps"] = size / (time.perf_counter() - t0) / 1e9
            res["rows"].append(row)
        # one warp: the batch decoder on one 32 MiB member
        m = raw[:32 << 20]
        c1 = zlib.compressobj(6, zlib.DEFLATED, 31)
        member = c1.compress(m) + c1.flush()
        dc, do = ctx.malloc_device(len(member)), ctx.malloc_device(len(m) + 64)
        ctx.h2d(dc, np.frombuffer(member, dtype=np.uint8))
        (rl, st), wmin, _ = best(2, lambda: ctx.inflate_batch_device(dc, [0], [len(member)], do, [0, len(m) + 64], format="gzip"))
        assert int(rl[0]) == len(m) and int(st[0]) == zwz.STREAM_END
        res[f"one_warp_{kind}_gbps"] = len(m) / wmin / 1e9
        ctx.free_device(dc)
        ctx.free_device(do)
        # independent members: BGZF of the same bytes
        gz, goff = ctx.gzip_files(raw, np.array([0, size], dtype=np.uint64))
        (back, _, gst), bmin, _ = best(a.reps, lambda: ctx.gunzip_files(gz, goff, out_cap=size + (1 << 20)))
        assert int(gst[0]) == zwz.STREAM_END and back.tobytes() == raw
        res[f"bgzf_gunzip_files_{kind}_gbps"] = size / bmin / 1e9
        ctx.free_device(d_out)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
