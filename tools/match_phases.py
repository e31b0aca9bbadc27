"""Where lz_match_kernel spends its cycles: the C2 device pass (deflate of 1 000-file-directory C2 files, device-resident) on
three corpora — the JPEG-like files only, the bitmap-like files only, and the real mix — with a build of csrc/ that has
-DZWZ_DM_PHASE_CLOCKS. Thread 0 of every CTA adds up the clock64() cycles between the barriers that end each phase of a chunk
(deflate_match.cuh); the table gives cycles per chunk per phase and size class, averaged over the chunks of that class. They
are CTA cycles: the CTAs of one SM (6 of class 0, 3 of class 1, 2 of class 2, 1 of class 3) run side by side.
    python tools/match_phases.py [--files N] [--reps R] [--lib clocked.so] [--out result.json]
Without --lib the clocked library is compiled into a temporary directory (nvcc, sm_100a). A --lib without the clocks gives the
lz_match times alone."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import zwz_b200  # noqa: E402
from tools import corpus  # noqa: E402

PHASES = ("stage", "noise hist", "noise bits", "head init", "hash+count", "offsets", "scatter", "chains", "search", "flags+adler")
NPH = len(PHASES)


def build_clocked(outdir: str) -> str:
    csrc = os.path.join(ROOT, "parallel-data-compression-and-decompression_b200", "csrc")
    so = os.path.join(outdir, "libzwz_cuda_clk.so")
    cmd = ["/usr/local/cuda/bin/nvcc", "-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-ccbin", "/usr/bin/g++", "-DZWZ_DM_PHASE_CLOCKS",
           "-shared", "-o", so, os.path.join(csrc, "zwz_cuda.cu"), "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    subprocess.run(cmd, check=True)
    return so


def split_c2(n_files: int):
    """(name, buffer, file offsets) of the JPEG-like files, the bitmap-like files and all of them, in corpus order."""
    buf, offs, sizes = corpus.c2_buffer(n_files)
    hdr = corpus._jpeg_header()[:8]
    starts = offs[:-1]
    is_jpeg = np.array([sizes[i] >= 8 and np.array_equal(buf[starts[i]:starts[i] + 8], hdr) for i in range(len(sizes))])
    out = []
    for name, sel in (("jpeg", is_jpeg), ("bitmap", ~is_jpeg)):
        keep = np.repeat(sel, sizes)
        fo = np.zeros(int(sel.sum()) + 1, dtype=np.int64)
        np.cumsum(sizes[sel], out=fo[1:])
        out.append((name, np.ascontiguousarray(buf[keep]), fo))
    out.append(("mix", buf, offs.astype(np.int64)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lib", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    tmp = tempfile.TemporaryDirectory()
    path = os.path.abspath(a.lib) if a.lib else build_clocked(tmp.name)
    lib = zwz_b200.load_library(path)
    clocked = hasattr(lib, "zwz_dm_phase_clocks")
    if clocked:
        lib.zwz_dm_phase_clocks.argtypes = [ctypes.c_void_p, ctypes.c_int]
        lib.zwz_dm_phase_clocks.restype = ctypes.c_int
    clk = np.zeros((4, NPH + 1), dtype=np.uint64)
    ctx = zwz_b200.Context(0, library=lib)
    result = {"lib": os.path.basename(path), "files": a.files, "reps": a.reps, "corpora": {}}
    for name, buf, foffs in split_c2(a.files):
        coff, clen, _, _ = zwz_b200.chunk_table(foffs)
        slot = zwz_b200.deflate_bound(clen)
        slot_off = np.zeros(len(coff) + 1, dtype=np.uint64)
        np.cumsum(slot, out=slot_off[1:])
        d_raw = ctx.malloc_device(len(buf) + 64)
        d_slots = ctx.malloc_device(int(slot_off[-1]) + 64)
        ctx.h2d(d_raw, buf)
        ctx.deflate_batch_device(d_raw, coff, clen, d_slots, slot_off[:-1])  # warm-up
        assert not clocked or lib.zwz_dm_phase_clocks(clk.ctypes.data, 1) == 0
        ctx.profile_enable(True)
        ctx.profile_read(True)
        for _ in range(a.reps):
            ctx.deflate_batch_device(d_raw, coff, clen, d_slots, slot_off[:-1])
        prof = ctx.profile_read(True)
        ctx.profile_enable(False)
        assert not clocked or lib.zwz_dm_phase_clocks(clk.ctypes.data, 1) == 0
        ctx.free_device(d_raw)
        ctx.free_device(d_slots)
        rows = {}
        for cls in range(4):
            nch = int(clk[cls, NPH])
            if nch:
                rows[cls] = {"chunks": nch // a.reps, "cycles_per_chunk": round(float(clk[cls, :NPH].sum()) / nch),
                             **{PHASES[k]: round(float(clk[cls, k]) / nch) for k in range(NPH)}}
        lz = prof.get("lz_match", (0.0, 0))
        result["corpora"][name] = {"MB": round(len(buf) / 1e6, 1), "lz_match_ms": round(lz[0] / a.reps, 3), "classes": rows}
        print(f"\n{name}: {len(buf) / 1e6:.1f} MB, lz_match {lz[0] / a.reps:.3f} ms per pass")
        print("class  chunks   total  " + "  ".join(f"{p:>11s}" for p in PHASES))
        for cls, r in rows.items():
            print(f"{cls:5d} {r['chunks']:7d} {r['cycles_per_chunk']:7d}  " + "  ".join(f"{r[p]:11d}" for p in PHASES))
    ctx.close()
    print(json.dumps(result))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
