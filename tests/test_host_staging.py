"""Descriptor staging of the device-API calls on the context's host threads, and the reuse of the last deflate call's slot
offsets and results by zwz_pack_streams_device.

Results must not depend on how many host threads stage a call (ZWZ_TUNE_HOST_THREADS), and pack must use the caller's arrays:
the device copies a deflate call left behind count only while the caller's slot offsets and results are byte-equal to what that
call used and returned. On the CPU the emulator build runs with ZWZ_TUNE_HOST_PARALLEL_MIN = 64, so that these small batches
take the blocked paths; the -m gpu twins run above the default threshold."""
import hashlib

import numpy as np
import pytest

import zwz_b200
from tools import corpus

# chunk sizes in all four lz_match size classes (<= 8192, <= 16384, <= 31744, <= 65535), shuffled so that no class is in order
_CLASS_SIZES = [(40, 1, 8192), (6, 8193, 16384), (3, 16385, 31744), (3, 31745, 65535)]


def _emu(threads, parallel_min=64):
    import emu_lib
    ctx = emu_lib.emu_context()
    ctx.tune(ctx.TUNE_HOST_THREADS, threads)
    ctx.tune(ctx.TUNE_HOST_PARALLEL_MIN, parallel_min)
    return ctx


@pytest.fixture(scope="module")
def emu_pair():
    a, b = _emu(1), _emu(4)
    yield a, b
    a.close()
    b.close()


def _chunks(seed, reps=1):
    rng = np.random.default_rng(seed)
    sizes = []
    for _ in range(reps):
        for k, lo, hi in _CLASS_SIZES:
            sizes += rng.integers(lo, hi + 1, k).tolist()
    sizes += [0, 1, 65535]
    rng.shuffle(sizes)
    kinds = "TSJBR"
    parts = [corpus.gen_file(kinds[i % len(kinds)], int(s), seed + i, 1).tobytes() if s else b"" for i, s in enumerate(sizes)]
    return parts


class Batch:
    """One buffer of chunks resident on the device, with the descriptor arrays of bench.py's device step."""

    def __init__(self, ctx, parts):
        self.ctx = ctx
        self.raw = np.frombuffer(b"".join(parts), dtype=np.uint8)
        self.n = len(parts)
        self.off = np.zeros(self.n + 1, dtype=np.uint64)
        np.cumsum([len(p) for p in parts], out=self.off[1:])
        self.len = np.diff(self.off).astype(np.uint32)
        self.slot_off = np.zeros(self.n + 1, dtype=np.uint64)
        np.cumsum(zwz_b200.deflate_bound(self.len), out=self.slot_off[1:])
        U, S = len(self.raw), int(self.slot_off[-1])
        self.d_raw = ctx.malloc_device(U + 64)
        self.d_slots = ctx.malloc_device(S + 64)
        self.d_packed = ctx.malloc_device(S + 64)
        self.d_back = ctx.malloc_device(U + 64)
        self.packed_cap = S
        ctx.h2d(self.d_raw, self.raw)

    def close(self):
        for p in (self.d_raw, self.d_slots, self.d_packed, self.d_back):
            self.ctx.free_device(p)

    def deflate(self):
        return self.ctx.deflate_batch_device(self.d_raw, self.off[:-1], self.len, self.d_slots, self.slot_off[:-1])

    def slots(self):
        out = np.zeros(int(self.slot_off[-1]), dtype=np.uint8)
        self.ctx.d2h(out, self.d_slots)
        return out

    def pack(self, res, fill=0xEE):
        """packed bytes (the buffer is filled with `fill` first, so that bytes pack did not write show) and packed_off"""
        self.ctx.h2d(self.d_packed, np.full(self.packed_cap, fill, dtype=np.uint8))
        poff = self.ctx.pack_streams_device(self.d_slots, self.slot_off[:-1], res, self.d_packed)
        out = np.zeros(self.packed_cap, dtype=np.uint8)
        self.ctx.d2h(out, self.d_packed)
        return out, poff

    def expected_pack(self, res, slots):
        return b"".join(slots[int(self.slot_off[i]):int(self.slot_off[i]) + int(res[i]["len0"]) + int(res[i]["len1"])].tobytes()
                        for i in range(self.n))


def _roomiest(b: Batch, res):
    """the chunk with the most room left in its slot behind its streams"""
    room = np.diff(b.slot_off).astype(np.int64) - res["len0"].astype(np.int64) - res["len1"].astype(np.int64)
    assert room.max() >= 3
    return int(np.argmax(room))


def _records(res, poff, raw_off):
    split = res["len1"] > 0
    k = np.nonzero(split)[0]
    r_off = np.insert(poff[:-1], k + 1, poff[:-1][k] + res["len0"][k].astype(np.uint64))
    r_len = np.insert(res["len0"], k + 1, res["len1"][k])
    r_raw = np.insert(raw_off[:-1], k + 1, raw_off[:-1][k] + res["raw0"][k].astype(np.uint64))
    return r_off, r_len, np.concatenate([r_raw, raw_off[-1:]])


def _step(b: Batch):
    """bench.py's device step: deflate -> md5 of the sources -> pack -> inflate -> md5 of the output"""
    ctx = b.ctx
    f_off, f_len = b.off[:-1], np.diff(b.off)
    res = b.deflate()
    dg1 = ctx.md5_batch_device(b.d_raw, f_off, f_len)
    packed, poff = b.pack(res)
    r_off, r_len, r_raw = _records(res, poff, b.off)
    rl, st = ctx.inflate_batch_device(b.d_packed, r_off, r_len, b.d_back, r_raw)
    dg2 = ctx.md5_batch_device(b.d_back, f_off, f_len)
    back = np.zeros(len(b.raw), dtype=np.uint8)
    ctx.d2h(back, b.d_back)
    return {"res": res.tobytes(), "poff": poff, "packed": packed[:int(poff[-1])].tobytes(), "rl": rl, "st": st, "dg1": dg1, "dg2": dg2,
            "back": back.tobytes()}


def _same_step(ctx_a, ctx_b, parts):
    out = []
    for ctx in (ctx_a, ctx_b):
        b = Batch(ctx, parts)
        try:
            out.append(_step(b))
        finally:
            b.close()
    a, b = out
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])) if isinstance(a[k], np.ndarray) else a[k] == b[k], k
    assert (a["st"] == 0).all()
    assert a["back"] == b"".join(parts)
    assert bytes(a["dg1"].tobytes()) == b"".join(hashlib.md5(p).digest() for p in parts)


def test_host_threads_do_not_change_results(emu_pair):
    _same_step(*emu_pair, _chunks(11, reps=2))


def test_pack_uses_caller_results_edited_in_place(emu_pair):
    ctx = emu_pair[1]
    b = Batch(ctx, _chunks(12))
    try:
        res = b.deflate()
        ctx.md5_batch_device(b.d_raw, b.off[:-1], np.diff(b.off))   # writes the context's shared descriptor arenas in between
        slots = b.slots()
        # one stream longer than deflate made it (still inside its slot): a resident copy of the old results would leave the
        # bytes past its old end unwritten
        k = _roomiest(b, res)
        res[k]["len0"] += 3
        packed, poff = b.pack(res)
        assert packed[:int(poff[-1])].tobytes() == b.expected_pack(res, slots)
        # the unedited results still pack as deflate made them
        res[k]["len0"] -= 3
        packed, poff = b.pack(res)
        assert packed[:int(poff[-1])].tobytes() == b.expected_pack(res, slots)
    finally:
        b.close()


def test_pack_uses_results_of_another_deflate_call(emu_pair):
    ctx = emu_pair[1]
    parts_a = _chunks(13)
    # same chunk sizes, other bytes: other stream lengths
    parts_b = [corpus.gen_file("T", len(p), 700 + i, 1).tobytes() if p else b"" for i, p in enumerate(parts_a)]
    a, b = Batch(ctx, parts_a), Batch(ctx, parts_b)
    try:
        res_a = a.deflate()
        res_b = b.deflate()
        assert (res_a["len0"] != res_b["len0"]).any()
        # b's slots with a's results: every stream is cut or padded from what b's deflate left
        lens = np.minimum(res_a["len0"] + res_a["len1"], np.diff(b.slot_off).astype(np.uint32))
        mixed = res_a.copy()
        mixed["len0"], mixed["len1"] = lens, 0
        packed, poff = b.pack(mixed)
        assert packed[:int(poff[-1])].tobytes() == b.expected_pack(mixed, b.slots())
        assert int(poff[-1]) == int(lens.sum())
    finally:
        a.close()
        b.close()


def test_md5_twice_with_the_same_array_mutated(emu_pair):
    ctx = emu_pair[1]
    parts = _chunks(14)
    b = Batch(ctx, parts)
    try:
        f_off, f_len = b.off[:-1].copy(), np.diff(b.off)
        d1 = ctx.md5_batch_device(b.d_raw, f_off, f_len)
        assert d1.tobytes() == b"".join(hashlib.md5(p).digest() for p in parts)
        f_off += np.uint64(1)   # every file one byte later
        f_len[f_len > 0] -= np.uint64(1)
        d2 = ctx.md5_batch_device(b.d_raw, f_off, f_len)
        want = [hashlib.md5(b.raw[int(o):int(o) + int(n)].tobytes()).digest() for o, n in zip(f_off, f_len)]
        assert d2.tobytes() == b"".join(want)
    finally:
        b.close()


def test_host_thread_knobs_are_checked(emu_pair):
    ctx = emu_pair[0]
    with pytest.raises(zwz_b200.ZwzError):
        ctx.tune(ctx.TUNE_HOST_THREADS, 1 << 20)


# ---- real size on the B200: a C2-shaped batch above the default threshold of 32 768 entries ----------------------------------
@pytest.fixture(scope="module")
def cuda_pair():
    a, b = zwz_b200.Context(0), zwz_b200.Context(0)
    a.tune(a.TUNE_HOST_THREADS, 1)   # b keeps the defaults
    yield a, b
    a.close()
    b.close()


def _c2_parts(n_files):
    buf, foffs, _ = corpus.c2_buffer(n_files)
    coff, clen, _, _ = zwz_b200.chunk_table(foffs)
    return [buf[int(o):int(o) + int(n)].tobytes() for o, n in zip(coff, clen)]


@pytest.mark.gpu
def test_host_threads_do_not_change_results_gpu(cuda_pair):
    parts = _c2_parts(40_000)
    assert len(parts) > 32_768
    _same_step(*cuda_pair, parts)


@pytest.mark.gpu
def test_pack_uses_caller_results_edited_in_place_gpu(cuda_pair):
    ctx = cuda_pair[1]
    b = Batch(ctx, _c2_parts(40_000))
    try:
        res = b.deflate()
        ctx.md5_batch_device(b.d_raw, b.off[:-1], np.diff(b.off))
        slots = b.slots()
        packed, poff = b.pack(res)
        assert packed[:int(poff[-1])].tobytes() == b.expected_pack(res, slots)
        k = _roomiest(b, res)
        res[k]["len0"] += 3
        packed, poff = b.pack(res)
        assert packed[:int(poff[-1])].tobytes() == b.expected_pack(res, slots)
    finally:
        b.close()
