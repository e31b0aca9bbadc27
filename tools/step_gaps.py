#!/usr/bin/env python
"""Where the time of a device step goes that no kernel uses.

Runs the default C2 device step of bench.py (same shard builder, same five library calls, same stream) and prints one JSON line:

  step      the step as bench.py times it: CUDA events around `--steps` whole steps, the library's kernel spans
            (zwz_profile_*) summed per step, and the GPU idle time = event span - kernel time
  calls     per library call (and for records_of, the Python between pack and inflate): host ms (perf_counter around the call),
            kernel ms (the library's spans of that call), event ms (CUDA events before and after the call on the stream) and
            idle ms = event ms - kernel ms: the time the stream held no kernel while the call ran
  phases    with --trace: ZWZ_TRACE=1 phase times inside the library, averaged over the timed steps (every phase mark
            synchronises the stream, so a phase that queues device work also holds its run time; `kernels` is the kernel
            span plus its launch)
  device    name, power limit and max SM clock (nvidia-smi, read-only)

  python tools/step_gaps.py [--steps 5] [--warmup 3] [--trace] [--out FILE]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench import build_shard, fill_device, records_of  # noqa: E402

# which kernel spans belong to which call
CALL_KERNELS = {"deflate": ("lz_match", "deflate_encode", "adler32"), "md5_src": ("md5",), "pack": ("pack",), "records_of": (),
                "inflate": ("inflate",), "md5_out": ("md5",)}


def device_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        return None


def parse_trace(text):
    """{call: {phase: [ms, ...]}} from the library's `[zwz trace ...] call: phase X ms, ...` lines"""
    out = {}
    for m in re.finditer(r"\[zwz trace [^\]]*\] (\w+):(.*)", text):
        d = out.setdefault(m.group(1), {})
        for ph, ms in re.findall(r" ([\w+-]+) ([0-9.]+) ms,", m.group(2)):
            d.setdefault(ph, []).append(float(ms))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--files", type=int, default=0, help="C2 files (default: bench.py's 370 000)")
    ap.add_argument("--trace", action="store_true", help="also split each call into the library's ZWZ_TRACE phases")
    ap.add_argument("--out", help="append the JSON line to this file too")
    args = ap.parse_args()
    if args.trace:
        os.environ["ZWZ_TRACE"] = "1"   # read by zwz_init

    import torch
    import zwz_b200

    ctx = zwz_b200.Context(0)
    main_stream = torch.cuda.Stream()
    torch.cuda.set_stream(main_stream)
    stream = main_stream.cuda_stream

    sh = build_shard("c2", args.files or 370_000, 0, 1)
    U = sh.U
    coff, clen, _, _ = zwz_b200.chunk_table(sh.foffs)
    n = len(coff)
    slot_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(zwz_b200.deflate_bound(clen), out=slot_off[1:])
    raw_off = np.concatenate([coff, [np.uint64(U)]]).astype(np.uint64)
    f_off = sh.foffs[:-1].astype(np.uint64)
    f_len = np.diff(sh.foffs).astype(np.uint64)
    d_raw = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    d_slots = torch.empty(int(slot_off[-1]) + 64, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    fill_device(torch, d_raw, sh)
    torch.cuda.synchronize()
    res0 = ctx.deflate_batch_device(d_raw.data_ptr(), coff, clen, d_slots.data_ptr(), slot_off[:-1], 0, stream)
    d_packed = torch.empty(int(res0["len0"].sum() + res0["len1"].sum()) + 4096, dtype=torch.uint8, device="cuda")

    calls = {
        "deflate": lambda s: s.update(res=ctx.deflate_batch_device(d_raw.data_ptr(), coff, clen, d_slots.data_ptr(), slot_off[:-1], 0, stream)),
        "md5_src": lambda s: s.update(dg1=ctx.md5_batch_device(d_raw.data_ptr(), f_off, f_len, stream)),
        "pack": lambda s: s.update(poff=ctx.pack_streams_device(d_slots.data_ptr(), slot_off[:-1], s["res"], d_packed.data_ptr(), stream)),
        "records_of": lambda s: s.update(rec=records_of(s["res"], s["poff"], raw_off)),
        "inflate": lambda s: s.update(inf=ctx.inflate_batch_device(d_packed.data_ptr(), s["rec"][0], s["rec"][1], d_back.data_ptr(), s["rec"][2], 0,
                                                                   stream)),
        "md5_out": lambda s: s.update(dg2=ctx.md5_batch_device(d_back.data_ptr(), f_off, f_len, stream)),
    }
    state = {}

    def step():
        for f in calls.values():
            f(state)

    # the library's trace lines go to fd 2: collect them in a file, keep only what the timed steps wrote
    trace_file = tempfile.TemporaryFile(mode="w+")
    saved_err = os.dup(2)
    if args.trace:
        sys.stderr.flush()
        os.dup2(trace_file.fileno(), 2)
    try:
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        assert (state["inf"][1] == 0).all(), "inflate status"
        assert np.array_equal(state["dg1"], state["dg2"]), "MD5 verify failed"
        assert torch.equal(d_back[:U], d_raw[:U]), "round trip mismatch"
        trace_file.seek(0, os.SEEK_END)
        trace_pos = trace_file.tell()

        # 1. the step as bench.py times it
        ctx.profile_enable(True)
        ctx.profile_read(True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        host_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        step_ms = e0.elapsed_time(e1) / args.steps
        prof = ctx.profile_read(True)
        kernel_ms = {k: v[0] / args.steps for k, v in prof.items()}

        # 2. the same steps call by call: events and kernel spans of each call on its own
        per = {c: {"host_ms": 0.0, "event_ms": 0.0, "kernel_ms": 0.0} for c in calls}
        for _ in range(args.steps):
            for name, f in calls.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                t = time.perf_counter()
                f(state)
                dt = time.perf_counter() - t
                b.record()
                b.synchronize()
                k = ctx.profile_read(True)
                per[name]["host_ms"] += dt * 1e3
                per[name]["event_ms"] += a.elapsed_time(b)
                per[name]["kernel_ms"] += sum(k[x][0] for x in CALL_KERNELS[name])
        ctx.profile_enable(False)
    finally:
        if args.trace:
            sys.stderr.flush()
            os.dup2(saved_err, 2)
        os.close(saved_err)
    for d in per.values():
        for key in d:
            d[key] /= args.steps
        d["idle_ms"] = d["event_ms"] - d["kernel_ms"]

    line = {"device": device_info(), "workload": sh.desc, "chunks": n, "files": len(f_off), "steps": args.steps, "warmup": args.warmup,
            "trace": args.trace,
            "step": {"ms_per_step": step_ms, "host_ms_per_step": host_ms, "kernel_ms_per_step": kernel_ms,
                     "kernel_ms_sum": sum(kernel_ms.values()), "idle_ms": step_ms - sum(kernel_ms.values())},
            "calls": per}
    if args.trace:
        trace_file.seek(trace_pos)
        ph = parse_trace(trace_file.read())
        # the timed steps ran twice (section 1 and 2); md5_device runs twice per step
        reps = {c: 2 * args.steps * (2 if c == "md5_device" else 1) for c in ph}
        line["phases"] = {c: {p: round(sum(v) / reps[c], 3) for p, v in d.items()} for c, d in ph.items()}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
