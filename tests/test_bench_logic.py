"""bench.py's end-to-end leg (host_roundtrip: the host-buffer plugin calls `main` makes) and its workload bookkeeping, run on
the CPU SIMT emulator with small shards. The GPU numbers come from bench.py itself; this only keeps its host logic honest."""
import ctypes

import numpy as np
import pytest

import bench
import zwz_b200


def _run_parts(ctx, sh, nparts_want, do_md5):
    coff, clen, cfile, cseq = zwz_b200.chunk_table(sh.foffs)
    n, nf, U = len(coff), len(sh.foffs) - 1, sh.U
    slot = zwz_b200.deflate_bound(clen)
    slot_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(slot, out=slot_off[1:])
    raw_off = np.concatenate([coff, [np.uint64(U)]]).astype(np.uint64)
    if nf > 1:
        first = np.concatenate([[0], np.cumsum(np.bincount(cfile, minlength=nf))]).astype(np.int64)
        part_file = np.unique(np.searchsorted(sh.foffs, np.linspace(0, U, nparts_want + 1)))
        part_file[0], part_file[-1] = 0, nf
        part_file = np.unique(part_file)
        part_chunk = first[part_file]
    else:
        part_file = None
        part_chunk = np.unique(np.linspace(0, n, nparts_want + 1).astype(np.int64))
    wrap = sh.period if sh.periodic else None
    descs = bench.part_descriptors(sh, coff, clen, cfile, raw_off, slot_off, part_chunk, part_file, wrap)
    max_raw = max(d["b1"] - d["b0"] for d in descs)
    win = (wrap + max_raw) if sh.periodic else U
    hr = np.empty(win, dtype=np.uint8)
    for o in range(0, win, sh.period):
        k = min(sh.period, win - o)
        hr[o:o + k] = sh.unit[:k]
    hb = np.zeros(max(win, 1), dtype=np.uint8)
    hc = np.zeros(int(slot_off[-1]) + 64, dtype=np.uint8)
    total = 0
    for d in descs:
        cap = int(slot_off[d["c1"]] - slot_off[d["c0"]]) + 64
        total += bench.host_roundtrip(ctx, d, clen, hr.ctypes.data + d["y0"], hc.ctypes.data + d["hc"], cap, hb.ctypes.data + d["y0"], 0, do_md5)
        k = d["b1"] - d["b0"]
        assert np.array_equal(hb[d["y0"]:d["y0"] + k], hr[d["y0"]:d["y0"] + k])
    return total


def test_host_roundtrip_files(emu_ctx):
    sh = bench.build_shard("c2", 60, 0, 1)
    c = _run_parts(emu_ctx, sh, 3, True)
    assert 0 < c < sh.U * 1.02


def test_host_roundtrip_single_file_periodic(emu_ctx, monkeypatch):
    monkeypatch.setattr(bench, "C3_PERIOD", 100_000)
    sh = bench.build_shard("c3", 260_000, 0, 1)   # 2.6 periods, 4 chunks, parts wrap the period
    assert sh.periodic and sh.period == 100_000
    c = _run_parts(emu_ctx, sh, 2, False)
    assert 0 < c < sh.U // 2


def test_global_totals_match_shards():
    for wl, files, world in (("c2", 500, 2), ("c3", 300_000, 2), ("c1", 3 << 20, 2), ("c5", 8 << 20, 2)):
        tot = [0, 0, 0]
        for r in range(world):
            sh = bench.build_shard(wl, files, r, world)
            sizes = np.diff(sh.foffs)
            tot[0] += int((sizes // 65535 + 1).sum())
            tot[1] += len(sizes)
            tot[2] += sh.U
        assert tuple(tot) == bench.global_totals(wl, files, world)


def test_dump_outputs_sampled_seeded_and_bounded(tmp_path):
    """--dump-outputs of a step with C2's 370 000 chunks, records and files: float arrays, the same rows and byte positions on
    every run, bytes read where the sample says, at most 64 MB in all."""
    import torch
    n, U = 370_000, 40 << 20
    rng = np.random.default_rng(1)
    res = np.zeros(n, dtype=zwz_b200.RESULT_DTYPE)
    res["len0"] = rng.integers(8, 60000, n)
    res["raw0"] = 65535
    poff = np.concatenate([[0], np.cumsum(res["len0"])]).astype(np.uint64)
    state = {"res": res, "poff": poff, "rl": res["raw0"].copy(), "st": np.zeros(n, dtype=np.uint32),
             "dg1": rng.integers(0, 256, (n, 16), dtype=np.uint8), "dg2": rng.integers(0, 256, (n, 16), dtype=np.uint8)}
    packed = torch.from_numpy(rng.integers(0, 256, int(poff[-1]), dtype=np.uint8))
    back = torch.from_numpy(rng.integers(0, 256, U, dtype=np.uint8))
    a = bench.step_outputs(torch, state, packed, back, U)
    b = bench.step_outputs(torch, state, packed, back, U)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    r = bench.dump_rows(n)
    assert len(r) == bench.DUMP_ROWS and np.array_equal(a["md5_out"], state["dg2"][r]) and np.array_equal(a["deflate_len0"], res["len0"][r])
    pos = np.sort(np.random.default_rng([596, U]).integers(0, U, bench.DUMP_BYTES))
    assert np.array_equal(a["inflated_bytes"], back.numpy()[pos])
    bench.write_dump(str(tmp_path / "d"), a)
    assert np.array_equal(np.load(tmp_path / "d" / "packed_off.npy"), a["packed_off"])


def test_sample_of_periodic():
    sh = bench.Shard(np.arange(1000, dtype=np.uint8), 5000, [0, 5000], "x")
    assert np.array_equal(sh.host_bytes(990, 1010), np.concatenate([np.arange(990, 1000), np.arange(0, 10)]).astype(np.uint8))
    sb, so, what = bench.sample_of(sh, 5000)
    assert len(sb) == 5000 and np.array_equal(sb[1000:2000], sh.unit)
