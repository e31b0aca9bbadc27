#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on synthetic corpora of the named shapes.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|c3|c5] [--files F] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...        # the UNMODIFIED reference binary (zlib L6 / zlib inflate / OpenSSL MD5) on host cores

A "step" is one pass of the hot path over the rank's shard of the workload:
  compress side   deflate of every 65 535-byte chunk (compression.cpp:119-134) + MD5 of every source file (:95-103)
  decompress side inflate of every record (decompression.cpp:11-37) + MD5 of every output file (:136)
`value`  = uncompressed bytes of the whole job / device time of that step with the inputs already resident in HBM (CUDA
           events on the launching stream, max over ranks).
`e2e`    = the same step through the HOST-BUFFER plugin calls the C++ host (`main`) makes — zwz_compress_files +
           zwz_decompress_records (zwz_deflate_batch + zwz_inflate_batch for the single-file shape) — from page-locked host
           buffers back into page-locked host buffers: every H2D/D2H copy, arena and descriptor handling of the library is
           inside the timed region; W worker contexts per rank, like `main` (host/pipeline.hpp).
Workloads (BASELINE.json `configs`): c2 (default; configs[1]: 370 000 image-like files, ~2.5 GB), c1 (configs[0] shape),
c3 (configs[2]: one log/text file, `--files` bytes, 16 GiB = 17179869184), c5 (configs[4]: 64 GB mixed corpus cut over the
N GPUs: strong scaling). The default c2 line also carries short device-timed C1- and C3-shaped passes (`extra_workloads`).
Multi-GPU: the reference's policy — sort by size descending, rank r takes sorted files r, r+N, ... (file_sort.cpp:30-31,
compression.cpp:31-41); no data-path collective, one NCCL all-gather of per-rank counters.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from tools import corpus  # noqa: E402

CHUNK = 65535
METRIC = "deflate/inflate GB/s (uncompressed)"
UNIT = "GB/s"
C3_PERIOD = 32 << 20


# ---------------------------------------------------------------------------------------------------------------------
# workload: every rank builds ITS shard only. A shard is `period` bytes of generated content (`unit`) repeated up to `U`
# bytes (period == U for the shapes that are generated in full); `foffs` are the file boundaries inside the U bytes.
# ---------------------------------------------------------------------------------------------------------------------
class Shard:
    def __init__(self, unit, U, foffs, desc, scaling="weak"):
        self.unit = unit            # np.uint8[period]
        self.period = len(unit)
        self.U = int(U)
        self.foffs = np.asarray(foffs, dtype=np.int64)
        self.desc = desc
        self.scaling = scaling
        self.periodic = self.period < self.U

    def host_bytes(self, lo, hi):
        """bytes [lo, hi) of the shard as a numpy array (copies when the range wraps the period)"""
        if not self.periodic:
            return self.unit[lo:hi]
        idx0 = lo % self.period
        if idx0 + (hi - lo) <= self.period:
            return self.unit[idx0:idx0 + hi - lo]
        reps = (idx0 + hi - lo + self.period - 1) // self.period
        return np.tile(self.unit, reps)[idx0:idx0 + hi - lo]


def build_shard(workload: str, files: int, rank: int, world: int) -> Shard:
    seed = corpus.BASE_SEED
    if workload == "c2":
        # sizes from the global size-sorted deal; content keyed by (seed, rank, directory)
        all_sizes = corpus.c2_sizes(files * world, seed)
        order = np.argsort(-all_sizes, kind="stable")
        mine = order[rank::world]
        # every file is generated AT its dealt size, so a file is one JPEG-like or one bitmap-like file (round 1 cut a
        # buffer of generated files at the dealt boundaries, which mixed the two classes inside most files)
        want = all_sizes[mine]
        buf, foffs, _ = corpus.c2_buffer(len(mine), seed + 7919 * rank, sizes=want)
        tot = int(foffs[-1])
        return Shard(buf, tot, foffs, f"C2: {files} image-like files/GPU (70% JPEG-like, 30% bitmap-like), one chunk each")
    if workload == "c3":
        size = files  # bytes
        unit = corpus.gen_text(min(size, C3_PERIOD), seed, 0x100000 + rank)
        return Shard(unit, size, [0, size], f"C3: one {size}-byte log/text file per GPU, 65 535-byte chunks ({len(unit) >> 20} MiB period)")
    if workload == "c1":
        buf, offs, specs = corpus.mixed_buffer(files, seed + 1 + rank, 4096, 16 << 20)
        sizes = np.diff(offs)
        order = np.argsort(-sizes, kind="stable")
        parts = [buf[offs[i]:offs[i + 1]] for i in order]
        foffs = np.zeros(len(order) + 1, dtype=np.int64)
        np.cumsum(sizes[order], out=foffs[1:])
        return Shard(np.concatenate(parts), int(foffs[-1]), foffs, f"C1-shaped: {files} bytes of mixed T/S/I/R files per GPU, size-descending")
    if workload == "c5":
        # BASELINE configs[4]: 64 GB of C1-generator files (seed 597) cut over the N GPUs. Generating 64 GB takes half an hour
        # of host time, so each rank generates a POOL of such files (seed 597 + rank, size-descending) and its shard is that
        # pool's file list repeated until the rank's share (total / N) is reached. Chunks are independent streams, so the
        # repetition changes nothing for the kernels.
        total = files
        share = total // world
        pool_bytes = min(share, 768 << 20)
        buf, offs, specs = corpus.mixed_buffer(pool_bytes, seed + 1 + rank, 4096, 16 << 20)
        sizes = np.diff(offs)
        order = np.argsort(-sizes, kind="stable")
        unit = np.concatenate([buf[offs[i]:offs[i + 1]] for i in order])
        psz = sizes[order]
        reps = max(1, int(round(share / len(unit))))
        fsz = np.tile(psz, reps)
        foffs = np.zeros(len(fsz) + 1, dtype=np.int64)
        np.cumsum(fsz, out=foffs[1:])
        return Shard(unit, int(foffs[-1]), foffs,
                     f"C5: {total} bytes of mixed T/S/I/R files (C1 generator, seed 597) cut over {world} GPU(s); per-GPU pool of {len(unit)} bytes x {reps}",
                     scaling="strong")
    raise SystemExit(f"unknown workload {workload}")


# ---------------------------------------------------------------------------------------------------------------------
# clocks (nvidia-smi sampled DURING the timed region)
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU baseline: the reference's call sequences (oracle_ref_* in oracle/zwz_oracle.c: system zlib L6 deflate, zlib inflate,
# OpenSSL MD5 in 1024-byte updates), fanned out over host threads (ctypes releases the GIL).
# ---------------------------------------------------------------------------------------------------------------------
def cpu_step(buf, foffs, coff, clen, threads, do_md5=True):
    """One full step (compress side + decompress side) on the CPU. Returns (seconds, compressed_bytes, ok)."""
    from concurrent.futures import ThreadPoolExecutor

    import oracle_lib as O
    L = O.lib()
    n = len(coff)
    nf = len(foffs) - 1
    out = np.empty((n, CHUNK), dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint32)
    back = np.empty(int(foffs[-1]) + 1, dtype=np.uint8)
    raw_off = np.concatenate([coff, [np.uint64(foffs[-1])]]).astype(np.uint64)
    raw_len = np.zeros(n, dtype=np.uint32)
    hex1 = np.zeros(nf * 32, dtype=np.uint8)
    hex2 = np.zeros(nf * 32, dtype=np.uint8)
    fo = foffs[:-1].astype(np.uint64)
    fl = np.diff(foffs).astype(np.uint64)
    cs = np.linspace(0, n, threads + 1).astype(np.int64)
    fs = np.linspace(0, nf, threads + 1).astype(np.int64)

    def run(fn):
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(fn, range(threads)))

    def deflate(t):
        a, b = int(cs[t]), int(cs[t + 1])
        if b > a:
            L.oracle_ref_deflate_batch(buf.ctypes.data, coff[a:].ctypes.data, clen[a:].ctypes.data, b - a, out[a:].ctypes.data, out_len[a:].ctypes.data)

    def inflate(t):
        a, b = int(cs[t]), int(cs[t + 1])
        if b > a:
            L.oracle_ref_inflate_batch(out[a:].ctypes.data, out_len[a:].ctypes.data, b - a, back.ctypes.data, raw_off[a:].ctypes.data, raw_len[a:].ctypes.data)

    def md5(src, dst):
        def f(t):
            a, b = int(fs[t]), int(fs[t + 1])
            if b > a:
                L.oracle_ref_md5_batch(src.ctypes.data, fo[a:].ctypes.data, fl[a:].ctypes.data, b - a, dst[32 * a:].ctypes.data)
        return f

    t0 = time.perf_counter()
    run(deflate)
    if do_md5:
        run(md5(buf, hex1))
    run(inflate)
    if do_md5:
        run(md5(back, hex2))
    dt = time.perf_counter() - t0
    ok = bool((raw_len == clen).all()) and np.array_equal(hex1, hex2)
    return dt, int(out_len.sum()), ok


def reference_binary_step(main_ref, sb, so, cores):
    """Materialise the sample as a directory tree in RAM and return (step(), P): step() runs `main_ref compress` with P
    concurrently running emulated ranks (the MPI stub reads ZWZ_STUB_RANK/SIZE) and then `main_ref decompress`, and returns
    (seconds, archive bytes). The reference's per-file stdout goes to /dev/null."""
    import atexit
    import shutil
    import tempfile
    root = tempfile.mkdtemp(prefix="zwz_ref_", dir="/dev/shm")
    atexit.register(lambda: shutil.rmtree(root, ignore_errors=True))
    src = os.path.join(root, "w", "src")
    nf = len(so) - 1
    for d in range((nf + 999) // 1000):
        os.makedirs(os.path.join(src, f"dir{d:03d}"), exist_ok=True)
    for i in range(nf):
        sb[so[i]:so[i + 1]].tofile(os.path.join(src, f"dir{i // 1000:03d}", f"f{i % 1000:04d}.dat"))
    P = max(1, min(cores, nf))
    state = {"k": 0}

    def step():
        state["k"] += 1
        arch = os.path.join(root, f"arch{state['k']}")
        out = os.path.join(root, f"out{state['k']}")
        bc = os.path.join(root, f"bc{state['k']}")
        os.makedirs(bc)
        dn = open(os.devnull, "w")
        t0 = time.perf_counter()
        env0 = dict(os.environ, ZWZ_STUB_SIZE=str(P), ZWZ_STUB_RANK="0", ZWZ_STUB_DIR=bc, OMP_NUM_THREADS="2")
        p0 = subprocess.Popen([main_ref, "compress", src, arch], env=env0, stdout=dn, stderr=dn)
        while not os.path.exists(os.path.join(bc, "bcast_1")) and p0.poll() is None:
            time.sleep(0.001)  # rank 0 publishes the record file path; then the others may start
        procs = [p0] + [subprocess.Popen([main_ref, "compress", src, arch],
                                         env=dict(os.environ, ZWZ_STUB_SIZE=str(P), ZWZ_STUB_RANK=str(r), ZWZ_STUB_DIR=bc), stdout=dn, stderr=dn)
                        for r in range(1, P)]
        for p in procs:
            p.wait()
        subprocess.run([main_ref, "decompress", arch, out], stdout=dn, stderr=dn, env=dict(os.environ, ZWZ_STUB_SIZE="1"))
        dt = time.perf_counter() - t0
        comp = sum(os.path.getsize(os.path.join(arch, f)) for f in os.listdir(arch))
        shutil.rmtree(arch, ignore_errors=True)
        shutil.rmtree(out, ignore_errors=True)
        shutil.rmtree(bc, ignore_errors=True)
        return dt, comp

    return step, P


def sample_of(sh: Shard, target_bytes):
    """Bounded sample of the same workload: whole files taken evenly across the size-sorted shard."""
    foffs = sh.foffs
    nf = len(foffs) - 1
    tot = sh.U
    if tot <= target_bytes:
        return np.ascontiguousarray(sh.host_bytes(0, tot)), foffs.copy(), "whole shard"
    if nf == 1:
        n = max(1, int(target_bytes // CHUNK)) * CHUNK
        return np.ascontiguousarray(sh.host_bytes(0, n)), np.array([0, n], dtype=np.int64), f"first {n} bytes of the file"
    stride = max(1, int(round(tot / target_bytes)))
    idx = np.arange(0, nf, stride)
    sizes = np.diff(foffs)[idx]
    so = np.zeros(len(idx) + 1, dtype=np.int64)
    np.cumsum(sizes, out=so[1:])
    sb = np.empty(int(so[-1]), dtype=np.uint8)
    for k, i in enumerate(idx):
        sb[so[k]:so[k + 1]] = sh.host_bytes(int(foffs[i]), int(foffs[i + 1]))
    return sb, so, f"every {stride}-th file of the size-sorted shard ({len(idx)} files, {int(so[-1])} bytes)"


def global_totals(workload: str, files: int, world: int):
    """(chunks, files, bytes) of the WHOLE job over `world` GPUs, from sizes alone (no contents generated): both arms put the
    same numbers into `config`."""
    seed = corpus.BASE_SEED

    def chunks_of(sizes):
        return int((np.asarray(sizes, dtype=np.int64) // CHUNK + 1).sum())
    if workload == "c2":
        sz = corpus.c2_sizes(files * world, seed)
        return chunks_of(sz), len(sz), int(sz.sum())
    if workload == "c3":
        return world * (files // CHUNK + 1), world, world * files
    if workload == "c1":
        sz = [s.size for r in range(world) for s in corpus.mixed_specs(files, seed + 1 + r, 4096, 16 << 20)]
        return chunks_of(sz), len(sz), int(sum(sz))
    if workload == "c5":
        share = files // world
        pool_bytes = min(share, 768 << 20)
        nch = nfi = tot = 0
        for r in range(world):
            psz = np.array([s.size for s in corpus.mixed_specs(pool_bytes, seed + 1 + r, 4096, 16 << 20)], dtype=np.int64)
            reps = max(1, int(round(share / int(psz.sum()))))
            nch += reps * chunks_of(psz)
            nfi += reps * len(psz)
            tot += reps * int(psz.sum())
        return nch, nfi, tot
    raise SystemExit(f"unknown workload {workload}")


def config_of(args, sh: Shard, world):
    """Workload description shared VERBATIM by both arms (`--impl ours` and `--impl reference`)."""
    n_chunks_all, nf_all, U_all = global_totals(args.workload, args.files, world)
    return {"workload": sh.desc, "chunks": int(n_chunks_all), "files": int(nf_all), "uncompressed_bytes": int(U_all),
            "l2": "inputs (>= 2 GB/GPU) exceed the 126 MB L2", "level": args.level,
            "md5": bool(args.do_md5),
            "parallelism": f"files dealt size-descending round-robin over {world} GPU(s)"}


# ---------------------------------------------------------------------------------------------------------------------
def records_of(res, poff, raw_off):
    """record table (one per stream; chunks cut by the split rule give two) from the deflate results"""
    split = res["len1"] > 0
    if not split.any():
        return poff[:-1], res["len0"], raw_off, None
    k = np.nonzero(split)[0]
    r_off = np.insert(poff[:-1], k + 1, poff[:-1][k] + res["len0"][k].astype(np.uint64))
    r_len = np.insert(res["len0"], k + 1, res["len1"][k])
    r_raw = np.insert(raw_off[:-1], k + 1, raw_off[:-1][k] + res["raw0"][k].astype(np.uint64))
    return r_off, r_len, np.concatenate([r_raw, raw_off[-1:]]), k


CALL_WALL = {"compress": 0.0, "decompress": 0.0, "parts": 0}   # --e2e-profile: seconds inside the two plugin calls, summed over parts


def host_roundtrip(w, d, clen, raw_ptr, comp_ptr, comp_cap, back_ptr, level, do_md5):
    """One part of the shard through the host-buffer plugin calls (what `main` does per batch): compress side into the
    buffer at comp_ptr, then the decompress side from that buffer into back_ptr. Returns the compressed bytes."""
    c0, c1, b0, b1 = d["c0"], d["c1"], d["b0"], d["b1"]
    if "foff" in d:
        nfp = d["f1"] - d["f0"]
        # compress side: compression.cpp:106-148 for the files of this part (chunking, deflate, MD5 of every file)
        t0 = time.perf_counter()
        poff, res, dg1 = w.compress_files_into(raw_ptr, d["foff"], level, comp_ptr, comp_cap, want_md5=do_md5)
        t1 = time.perf_counter()
        # decompress side: decompression.cpp:100-151 for the records just made
        r_off, r_len, _, k = records_of(res, poff, np.zeros(c1 - c0 + 1, dtype=np.uint64))
        rfile = d["rfile"] if k is None else np.insert(d["rfile"], k + 1, d["rfile"][k])
        rcap = np.full(len(r_off), CHUNK, dtype=np.uint32)
        t2 = time.perf_counter()
        foff2, rl, st, dg2 = w.decompress_records_into(comp_ptr, r_off, r_len, rcap, rfile, nfp, back_ptr, b1 - b0, want_md5=do_md5)
        t3 = time.perf_counter()
        CALL_WALL["compress"] += t1 - t0
        CALL_WALL["decompress"] += t3 - t2
        CALL_WALL["parts"] += 1
        assert np.array_equal(foff2, d["foff"]), "file layout after decompress"
        if do_md5:
            assert np.array_equal(dg1, dg2), "MD5 verify failed"
    else:
        poff, res = w.deflate_batch_into(raw_ptr, d["coff"], clen[c0:c1], comp_ptr, comp_cap, level)
        r_off, r_len, r_raw_off, _ = records_of(res, poff, d["roff"])
        rl, st = w.inflate_batch_into(comp_ptr, r_off, r_len, back_ptr, r_raw_off, 0)
    assert (st == 0).all()
    return int(poff[-1])


def part_descriptors(sh, coff, clen, cfile, raw_off, slot_off, part_chunk, part_file, wrap):
    """Per-part descriptors that do not depend on results (prepared once, outside the timed region: `main` plans its batches
    up front the same way)."""
    out = []
    nparts = len(part_chunk) - 1
    for i in range(nparts):
        c0, c1 = int(part_chunk[i]), int(part_chunk[i + 1])
        b0, b1 = int(raw_off[c0]), int(raw_off[c1])
        d = {"c0": c0, "c1": c1, "b0": b0, "b1": b1, "y0": (b0 % wrap) if sh.periodic else b0, "hc": int(slot_off[c0])}
        if part_file is not None:
            f0, f1 = int(part_file[i]), int(part_file[i + 1])
            d.update(f0=f0, f1=f1, foff=(sh.foffs[f0:f1 + 1] - b0).astype(np.uint64), rfile=(cfile[c0:c1] - f0).astype(np.uint32))
        else:
            d.update(coff=(coff[c0:c1] - np.uint64(b0)).astype(np.uint64), roff=(raw_off[c0:c1 + 1] - np.uint64(b0)).astype(np.uint64))
        out.append(d)
    return out


def device_pass(torch, zwz_b200, ctx, stream, sh: Shard, level, do_md5, steps, warmup):
    """Short device-timed pass over a small shard (for the `extra_workloads` keys): returns a dict of rates."""
    U = sh.U
    coff, clen, cfile, cseq = zwz_b200.chunk_table(sh.foffs)
    n = len(coff)
    slot = zwz_b200.deflate_bound(clen)
    slot_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(slot, out=slot_off[1:])
    raw_off = np.concatenate([coff, [np.uint64(U)]]).astype(np.uint64)
    f_off = sh.foffs[:-1].astype(np.uint64)
    f_len = np.diff(sh.foffs).astype(np.uint64)
    d_raw = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    fill_device(torch, d_raw, sh)
    d_slots = torch.empty(int(slot_off[-1]) + 64, dtype=torch.uint8, device="cuda")
    d_packed = torch.empty(int(slot_off[-1]) + 64, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    st = {}

    def step():
        res = ctx.deflate_batch_device(d_raw.data_ptr(), coff, clen, d_slots.data_ptr(), slot_off[:-1], level, stream)
        if do_md5:
            st["dg1"] = ctx.md5_batch_device(d_raw.data_ptr(), f_off, f_len, stream)
        poff = ctx.pack_streams_device(d_slots.data_ptr(), slot_off[:-1], res, d_packed.data_ptr(), stream)
        r_off, r_len, r_raw_off, _ = records_of(res, poff, raw_off)
        rl, s = ctx.inflate_batch_device(d_packed.data_ptr(), r_off, r_len, d_back.data_ptr(), r_raw_off, 0, stream)
        if do_md5:
            st["dg2"] = ctx.md5_batch_device(d_back.data_ptr(), f_off, f_len, stream)
        st.update(res=res, s=s)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    assert (st["s"] == 0).all() and torch.equal(d_back[:U], d_raw[:U])
    ctx.profile_enable(True)
    ctx.profile_read(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    prof = ctx.profile_read(True)
    ctx.profile_enable(False)
    C = int(st["res"]["len0"].sum() + st["res"]["len1"].sum())
    k = {name: v[0] / steps for name, v in prof.items()}
    codec_ms = k["lz_match"] + k["deflate_encode"] + k["pack"] + k["inflate"]
    out = {"workload": sh.desc, "uncompressed_bytes": U, "chunks": n, "files": len(f_off), "steps": steps, "value": U / (ms * 1e-3) / 1e9, "ms_per_step": ms,
           "codec_gbs": U / (codec_ms * 1e-3) / 1e9,   # deflate + pack + inflate kernels only: a shard this small holds too few files to
                                                      # hide the MD5 chain of its longest one (16 MiB = 131 ms), which a full C1 does
           "md5_ms_per_step": k["md5"],
           "ratio": U / max(C, 1), "deflate_gbs": U / ((k["lz_match"] + k["deflate_encode"]) * 1e-3) / 1e9,
           "inflate_gbs": U / (k["inflate"] * 1e-3) / 1e9, "kernel_ms_per_step": k, "md5": bool(do_md5)}
    del d_raw, d_slots, d_packed, d_back
    torch.cuda.empty_cache()
    return out


def fill_device(torch, d_raw, sh: Shard):
    """shard bytes -> device tensor (tiled on the device when the shard is periodic)"""
    U = sh.U
    if not sh.periodic:
        d_raw[:U].copy_(torch.from_numpy(sh.unit), non_blocking=False)
        return
    d_unit = torch.from_numpy(sh.unit).cuda()
    P = sh.period
    for o in range(0, U, P):
        k = min(P, U - o)
        d_raw[o:o + k].copy_(d_unit[:k])
    del d_unit


DUMP_ROWS = 1 << 16    # --dump-outputs: rows kept of every per-chunk, per-record and per-file array
DUMP_BYTES = 1 << 20   # and bytes kept of the packed and of the inflated buffer


def dump_rows(n):
    """A fixed, seeded choice of at most DUMP_ROWS of n rows, in order (all n when there are few)."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng([596, n]).choice(n, DUMP_ROWS, replace=False))


def step_outputs(torch, state, d_packed, d_back, U):
    """What the last device step handed its caller, as float arrays for --dump-outputs (values below 2^24 as float32, byte
    offsets as float64): the deflate result of every chunk, the packed stream offsets, the inflated length and status of every
    record and the MD5 of every source and every inflated file (rows chosen by dump_rows), and the packed and the inflated
    bytes at DUMP_BYTES fixed, seeded positions."""
    res = state["res"]
    r = dump_rows(len(res))
    out = {f"deflate_{k}": res[k][r].astype(np.float32) for k in ("len0", "len1", "raw0", "btype")}
    out["packed_off"] = state["poff"][dump_rows(len(state["poff"]))].astype(np.float64)
    r = dump_rows(len(state["rl"]))
    out["inflate_len"] = state["rl"][r].astype(np.float32)
    out["inflate_status"] = state["st"][r].astype(np.float32)
    for key, name in (("dg1", "md5_src"), ("dg2", "md5_out")):
        if state[key] is not None:
            out[name] = state[key][dump_rows(len(state[key]))].astype(np.float32)
    for name, buf, size in (("packed_bytes", d_packed, int(state["poff"][-1])), ("inflated_bytes", d_back, U)):
        pos = np.sort(np.random.default_rng([596, size]).integers(0, size, DUMP_BYTES))
        out[name] = buf[torch.from_numpy(pos).to(buf.device)].cpu().numpy().astype(np.float32)
    return out


def write_dump(path, arrays):
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c1", "c5"])
    ap.add_argument("--files", type=int, default=0, help="c2: files per GPU (default 370000); c3/c1: bytes per GPU; c5: total bytes (default 64e9)")
    ap.add_argument("--level", type=int, default=0)
    ap.add_argument("--cpu-sample-mb", type=float, default=0.0, help="CPU baseline sample size (default: ~15 s of work)")
    ap.add_argument("--ref-sample-mb", type=float, default=0.0, help="--impl reference: sample size (default: 1 GB at 25 steps, scaled so the run ends in minutes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the end-to-end leg (its line then carries e2e = null)")
    ap.add_argument("--no-extra", action="store_true", help="skip the short C1/C3-shaped device passes of the default c2 line")
    ap.add_argument("--e2e-workers", type=int, default=0, help="end-to-end leg: worker contexts (stream + buffers each) per rank; 0 = min(6, host cores / ranks), at least 2")
    ap.add_argument("--e2e-profile", action="store_true", help="diagnostics for the end-to-end leg: wall time of the two plugin calls per part and "
                    "the workers' kernel spans (CUDA events; spans of concurrently running kernels overlap, so their sum is an upper bound)")
    ap.add_argument("--e2e-parts", type=int, default=32, help="end-to-end leg: parts the shard is cut into")
    ap.add_argument("--md5", default="auto", choices=["auto", "on", "off"],
                    help="auto: on for c2/c1/c5 (compress+decompress+MD5 verify), off for c3 (BASELINE.json config 3 is deflate+inflate only: "
                         "the MD5 of ONE file is a single serial chain, one lane, ~0.13 GB/s)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed device steps, write what the last one computed on rank 0 "
                    "(see step_outputs) to DIR/<name>.npy, so that two builds can be compared output for output on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps: at least one timed step")
    if args.warmup < 3:
        args.warmup = 3  # timing rule: W >= 3
    if args.files == 0:
        args.files = {"c2": 370_000, "c3": 2 << 30, "c1": 2 << 30, "c5": 64_000_000_000}[args.workload]

    args.do_md5 = do_md5 = args.md5 == "on" or (args.md5 == "auto" and args.workload != "c3")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    # ------------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        # same workload object as rank 0 of our arm builds (world = --gpus, so that config matches ours at every N)
        sh = build_shard(args.workload, args.files, 0, max(1, args.gpus))
        cfg = config_of(args, sh, max(1, args.gpus))
        if args.ref_sample_mb:
            target = int(args.ref_sample_mb * 1e6)
        else:
            # about 0.017 GB/s per core end to end (round 1: 0.266 GB/s on 16 cores); aim at <= ~150 s for all steps
            target = int(min(sh.U, max(0.25e9, min(1.0e9, 150.0 * 0.017e9 * cores / (args.steps + args.warmup)))))
        sb, so, what = sample_of(sh, target)
        main_ref = os.path.join(ROOT, "oracle", "_ref", "main_ref")
        if os.path.exists(main_ref) and os.path.isdir("/dev/shm"):
            kind = "reference"
            step = "UNMODIFIED reference binary (oracle/_ref/main_ref): compress with P emulated MPI ranks + decompress (1 process, OpenMP over archives) on a RAM-backed tree"
            run_step, P = reference_binary_step(main_ref, sb, so, cores)
            what += f"; written as files under /dev/shm; compress ranks = {P}"
        else:
            kind = "port"
            step = "deflate(zlib L6)+MD5(src)+inflate+MD5(out) per chunk/file on host cores (oracle_ref_* call sequences)"
            coff, clen, _, _ = corpus.chunk_table(so)
            run_step = lambda: cpu_step(sb, so, coff, clen, cores, do_md5)[:2]
        times = []
        comp = 0
        for i in range(args.warmup + args.steps):
            dt, comp = run_step()
            if i >= args.warmup:
                times.append(dt)
        t = sum(times)
        val = len(sb) * len(times) / t / 1e9
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t / len(times), "higher_is_better": True, "scaling": sh.scaling, "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": cfg, "pipeline": {"step": step},
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": what,
                                 "ratio": len(sb) / max(comp, 1)},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist

    import zwz_b200

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = zwz_b200.Context(local_rank)  # raises when libzwz_cuda.so or the GPU is missing: no fallback exists
    main_stream = torch.cuda.Stream()
    torch.cuda.set_stream(main_stream)       # everything below (events, copies, our kernels) is ordered on this stream
    stream = main_stream.cuda_stream

    sh = build_shard(args.workload, args.files, rank, world)
    U = sh.U
    foffs = sh.foffs
    nf = len(foffs) - 1
    coff, clen, cfile, cseq = zwz_b200.chunk_table(foffs)
    n = len(coff)
    slot = zwz_b200.deflate_bound(clen)
    slot_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(slot, out=slot_off[1:])
    raw_off = np.concatenate([coff, [np.uint64(U)]]).astype(np.uint64)
    f_off = foffs[:-1].astype(np.uint64)
    f_len = np.diff(foffs).astype(np.uint64)

    d_raw = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    d_slots = torch.empty(int(slot_off[-1]) + 64, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(U + 64, dtype=torch.uint8, device="cuda")
    fill_device(torch, d_raw, sh)
    torch.cuda.synchronize()
    # the packed buffer is sized from a first deflate (a 16 GiB text file packs into ~6 GB; slot capacity would be 16 GiB more)
    res0 = ctx.deflate_batch_device(d_raw.data_ptr(), coff, clen, d_slots.data_ptr(), slot_off[:-1], args.level, stream)
    C0 = int(res0["len0"].sum() + res0["len1"].sum())
    d_packed = torch.empty(C0 + 4096, dtype=torch.uint8, device="cuda")

    state = {}

    def device_step():
        """inputs resident in HBM"""
        res = ctx.deflate_batch_device(d_raw.data_ptr(), coff, clen, d_slots.data_ptr(), slot_off[:-1], args.level, stream)
        dg1 = ctx.md5_batch_device(d_raw.data_ptr(), f_off, f_len, stream) if do_md5 else None
        poff = ctx.pack_streams_device(d_slots.data_ptr(), slot_off[:-1], res, d_packed.data_ptr(), stream)
        r_off, r_len, r_raw_off, _ = records_of(res, poff, raw_off)   # records: one per stream (split chunks give two)
        rl, st = ctx.inflate_batch_device(d_packed.data_ptr(), r_off, r_len, d_back.data_ptr(), r_raw_off, 0, stream)
        dg2 = ctx.md5_batch_device(d_back.data_ptr(), f_off, f_len, stream) if do_md5 else None
        state.update(res=res, dg1=dg1, dg2=dg2, rl=rl, st=st, poff=poff, r_raw_off=r_raw_off)

    # ---- end-to-end through the host-buffer plugin calls: W workers (own zwz ctx = own stream + arenas, like `main`'s worker
    # pool) take parts of the shard in turn, so the H2D of one part, the kernels of another and the D2H of a third overlap.
    # Every byte starts in page-locked host memory and ends in page-locked host memory inside the timed region.
    from concurrent.futures import ThreadPoolExecutor
    W = args.e2e_workers if args.e2e_workers > 0 else max(2, min(6, (os.cpu_count() or 16) // max(world, 1)))
    first_chunk_of_file = np.concatenate([[0], np.cumsum(np.bincount(cfile, minlength=nf))]).astype(np.int64)
    if nf > 1:   # cut on file boundaries (MD5 needs whole files), parts of about equal bytes
        want = min(max(args.e2e_parts, int(U // (768 << 20))), max(1, nf // 8))
        part_file = np.unique(np.searchsorted(foffs, np.linspace(0, U, want + 1)))
        part_file[0], part_file[-1] = 0, nf
        part_file = np.unique(part_file)
        part_chunk = first_chunk_of_file[part_file]
    else:
        part_file = None
        want = min(max(args.e2e_parts, int(U // (512 << 20))), max(1, n // 512))
        part_chunk = np.unique(np.linspace(0, n, want + 1).astype(np.int64))
    nparts = len(part_chunk) - 1
    part_b0 = np.array([int(raw_off[part_chunk[i]]) for i in range(nparts + 1)], dtype=np.int64)
    max_raw = int(np.diff(part_b0).max())
    max_slot = max(int(slot_off[part_chunk[i + 1]] - slot_off[part_chunk[i]]) for i in range(nparts))
    # page-locked host windows. Generated-in-full shards: the whole shard. Periodic shards (c3 at 16 GiB, c5): a window of
    # whole periods + one part, so that any part is contiguous in it (byte x of the shard == unit[x mod period]).
    if sh.periodic:
        wrap = sh.period * max(1, (4 << 30) // sh.period)
        win = wrap + max_raw
    else:
        wrap, win = None, U
    h_raw = torch.empty(win, dtype=torch.uint8, pin_memory=True)
    hr = h_raw.numpy()
    if sh.periodic:
        for o in range(0, win, sh.period):
            k = min(sh.period, win - o)
            hr[o:o + k] = sh.unit[:k]
    else:
        hr[:] = sh.unit
    # outputs: the whole shard when it is generated in full; one region per worker when it is periodic (16 GiB would not fit)
    back_stride = (max_raw + 4095) & ~4095
    comp_stride = (max_slot + 64 + 4095) & ~4095
    h_back = torch.empty(back_stride * W if sh.periodic else U, dtype=torch.uint8, pin_memory=True)
    h_comp = torch.empty(comp_stride * W if sh.periodic else int(slot_off[-1]) + 64, dtype=torch.uint8, pin_memory=True)
    last_part = [None] * W
    hc_ptr, hr_ptr, hb_ptr = h_comp.data_ptr(), h_raw.data_ptr(), h_back.data_ptr()
    workers = [zwz_b200.Context(local_rank) for _ in range(W)]
    for w in workers:   # like `main`'s workers: scratch for 64 MiB deflate passes instead of the default 4 GiB ones
        w.tune(w.TUNE_DEFLATE_SUBBATCH_BYTES, 64 << 20)
    wlock = threading.Lock()
    wfree = list(range(W))
    comp_bytes = [0] * nparts
    part_desc = part_descriptors(sh, coff, clen, cfile, raw_off, slot_off, part_chunk, part_file, wrap)

    def run_part(i, wi):
        d = part_desc[i]
        cap = int(slot_off[d["c1"]] - slot_off[d["c0"]]) + 64
        hc = wi * comp_stride if sh.periodic else d["hc"]
        hb = wi * back_stride if sh.periodic else d["y0"]
        comp_bytes[i] = host_roundtrip(workers[wi], d, clen, hr_ptr + d["y0"], hc_ptr + hc, cap, hb_ptr + hb, args.level, do_md5)
        last_part[wi] = i

    def e2e_part(i):
        with wlock:
            wi = wfree.pop()
        try:
            run_part(i, wi)
        finally:
            with wlock:
                wfree.append(wi)

    def size_workers():
        """Warm-up: EVERY worker context takes the parts with the most chunks, files, raw bytes and slot bytes once, so that its
        device and page-locked arenas have their final size before the timed steps (`main` sizes its workers' buffers from the
        batch plan the same way). Parts are handed to whichever worker is free, so without this a worker can meet its largest part
        inside the timed region — and growing a page-locked arena synchronises the whole device, for every worker."""
        key = [lambda i: part_chunk[i + 1] - part_chunk[i], lambda i: part_b0[i + 1] - part_b0[i],
               lambda i: int(slot_off[part_chunk[i + 1]] - slot_off[part_chunk[i]])]
        if part_file is not None:
            key.append(lambda i: part_file[i + 1] - part_file[i])
        sizing = sorted({max(range(nparts), key=k) for k in key})
        with ThreadPoolExecutor(W) as sp:
            list(sp.map(lambda wi: [run_part(i, wi) for i in sizing], range(W)))

    pool = ThreadPoolExecutor(W)

    def e2e_step():
        list(pool.map(e2e_part, range(nparts)))
        state.update(C=sum(comp_bytes))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (also sizes every arena)
    for _ in range(args.warmup):
        device_step()
    barrier()
    # correctness of what we are about to time
    res = state["res"]
    Cbytes = int(res["len0"].sum() + res["len1"].sum())
    assert (state["st"] == 0).all(), "inflate status"
    assert (not do_md5) or np.array_equal(state["dg1"], state["dg2"]), "MD5 verify failed"
    for o in range(0, U, 1 << 30):
        assert torch.equal(d_back[o:min(U, o + (1 << 30))], d_raw[o:min(U, o + (1 << 30))]), "round trip mismatch"

    sampler = ClockSampler(local_rank)
    sampler.start()
    ctx.profile_enable(True)
    ctx.profile_read(True)
    launches0 = ctx.launches
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        device_step()
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = ctx.launches - launches0
    prof = ctx.profile_read(True)
    ctx.profile_enable(False)
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, step_outputs(torch, state, d_packed, d_back, U))

    # e2e (host buffers only: the device-resident copies of the shard are not needed any more — at 32 GB per GPU, C5 over two
    # GPUs, they and the workers' arenas do not fit side by side)
    del d_raw, d_slots, d_back, d_packed
    torch.cuda.empty_cache()
    e2e_ms, e2e_launches = float("nan"), 0
    if not args.no_e2e:
        size_workers()
        for _ in range(2):
            e2e_step()
        barrier()
        wl0 = sum(w.launches for w in workers)
        if args.e2e_profile:
            for w in workers:
                w.profile_enable(True)
                w.profile_read(True)
            CALL_WALL.update(compress=0.0, decompress=0.0, parts=0)
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        for _ in range(args.steps):
            e2e_step()
        e3.record()
        barrier()
        e2e_ms = e2.elapsed_time(e3)
        e2e_launches = sum(w.launches for w in workers) - wl0
        if args.e2e_profile:
            wk = {}
            for w in workers:
                for k, v in w.profile_read(True).items():
                    wk[k] = wk.get(k, 0.0) + v[0] / args.steps
                w.profile_enable(False)
            state["e2e_profile"] = {"worker_kernel_span_ms_per_step": wk, "call_wall_ms_per_part": {k: 1e3 * CALL_WALL[k] / max(CALL_WALL["parts"], 1) for k in ("compress", "decompress")},
                                    "parts_per_step": nparts, "workers": W}
    clocks = sampler.stop()
    if args.no_e2e:
        pass
    elif sh.periodic:   # what every worker wrote last
        for wi, i in enumerate(last_part):
            if i is not None:
                d = part_desc[i]
                k = d["b1"] - d["b0"]
                assert np.array_equal(h_back.numpy()[wi * back_stride:wi * back_stride + k], hr[d["y0"]:d["y0"] + k]), "e2e round trip mismatch"
    else:
        assert np.array_equal(h_back.numpy(), hr), "e2e round trip mismatch"

    # max over ranks, totals over ranks (the ONLY collective: a few counters per GPU)
    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([U, Cbytes, n, nf, launches + e2e_launches], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        allc = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(allc, cnt)
        cnt = torch.stack(allc).sum(0)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    U_all, C_all, n_all, nf_all, launches_all = [float(x) for x in cnt]

    if rank == 0:
        K = args.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        ms = {k: v[0] for k, v in prof.items()}
        nl = {k: v[1] for k, v in prof.items()}
        # dominant kernel by device time on rank 0
        dom = max(("lz_match", "deflate_encode", "inflate") + (("md5",) if do_md5 else ()), key=lambda k: ms[k])
        alg_bytes = {"lz_match": U, "deflate_encode": U + Cbytes, "inflate": U + Cbytes, "md5": 2 * U}[dom] * K  # per K steps on rank 0
        achieved = alg_bytes / (ms[dom] * 1e-3) / 1e9 if ms[dom] > 0 else 0.0
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))   # measured on one workload only
            if tj.get("workload") == args.workload and (args.files in (0, tj.get("files"))):
                traffic = tj["kernels"].get(dom) * K / max(nl[dom], 1)   # per launch, like algorithmic_bytes_per_launch
        except Exception:
            pass
        cfg = config_of(args, sh, world)
        assert (cfg["chunks"], cfg["files"], cfg["uncompressed_bytes"]) == (int(n_all), int(nf_all), int(U_all)), "config totals"
        line = {
            "metric": METRIC, "value": U_all * K / (dev_ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": sh.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg,
            "pipeline": {"step": ("deflate+MD5(src)+pack+inflate+MD5(out)" if do_md5 else "deflate+pack+inflate (no MD5: one file = one serial chain)") + ", all through the C ABI",
                         "e2e": f"{W} worker contexts x {nparts} parts per rank through " +
                                ("zwz_compress_files + zwz_decompress_records" if part_file is not None else "zwz_deflate_batch + zwz_inflate_batch") +
                                " (host buffers in, host buffers out; the calls `main` makes)"},
            "ratio": U_all / C_all,
            "deflate_gbs": U * K / ((ms["lz_match"] + ms["deflate_encode"]) * 1e-3) / 1e9,
            "inflate_gbs": U * K / (ms["inflate"] * 1e-3) / 1e9,
            "md5_gbs": (2 * U * K / (ms["md5"] * 1e-3) / 1e9) if do_md5 and ms["md5"] > 0 else None,
            "kernel_ms_per_step": {k: v / K for k, v in ms.items()},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes / max(nl[dom], 1), "launches": nl[dom]},
            "e2e": None if args.no_e2e else {"value": U_all * K / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(U + state["C"]),
                                             "d2h_bytes_per_step": int(U + state["C"]), "ms_per_step": e2e_ms / K},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
        }
        if "e2e_profile" in state:
            line["e2e_profile"] = state["e2e_profile"]
        # free the big buffers before the extra passes / CPU leg
        if args.workload == "c2" and not args.no_extra and world == 1:
            extra = {}
            try:
                s1 = build_shard("c1", 192 << 20, 0, 1)
                extra["c1"] = device_pass(torch, zwz_b200, ctx, stream, s1, args.level, True, 3, 3)
                s3 = build_shard("c3", 1 << 30, 0, 1)
                extra["c3"] = device_pass(torch, zwz_b200, ctx, stream, s3, args.level, False, 3, 3)
            except Exception as e:  # the headline line must not die on an extra
                extra["error"] = repr(e)
            line["extra_workloads"] = extra
        if not args.no_cpu_baseline and world == 1:   # the CPU leg is a rank-0, N = 1 item (at N > 1 the other ranks would wait for it)
            target = int(args.cpu_sample_mb * 1e6) if args.cpu_sample_mb else int(min(8e6 * cores, 400e6))
            sb, so, what = sample_of(sh, target)
            scoff, sclen, _, _ = corpus.chunk_table(so)
            dt, comp, ok = cpu_step(sb, so, scoff, sclen, cores, do_md5)
            # our size on the very same sample, for the ratio criterion
            sres = ctx.deflate_batch(sb, scoff, sclen, args.level)[2]
            ours = int(sres["len0"].sum() + sres["len1"].sum())
            line["cpu_baseline"] = {"value": len(sb) / dt / 1e9, "unit": UNIT, "cores": cores, "kind": "port",
                                    "what": "the reference's call sequences (zlib L6 deflate, zlib inflate, OpenSSL MD5: oracle_ref_*) over the sample's chunks in memory, all host threads",
                                    "sample": what, "ratio": len(sb) / max(comp, 1), "roundtrip_ok": ok}
            line["size_vs_zlib6"] = ours / max(comp, 1)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
