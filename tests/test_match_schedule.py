"""The noise test of lz_match_kernel (deflate_match.cuh, step 1b) restated in numpy, against the skip mask the emulator build
records for every chunk: byte histograms of the 1 024-byte stretches with the top-bit prefilter, then the two bit sets of
4-byte windows (multiplier 0x9E3779B1, 2^(HB + 4) bits) and their margins. The three counts of the second test do not depend
on the order in which windows are inserted, so the kernel may visit them in any order; the verdict must not change."""
import numpy as np
import pytest

import emu_lib
from tools import corpus

HBITS = (12, 13, 13, 14)
CAPS = (8192, 16384, 31744)
NOISE_BITS = 7.7


def hb_of(n: int) -> int:
    for cls, cap in enumerate(CAPS):
        if n <= cap:
            return HBITS[cls]
    return HBITS[3]


def windows(d: np.ndarray, q: np.ndarray) -> np.ndarray:
    """little-endian 4-byte words at positions q; bytes past the end read as zero"""
    z = np.concatenate([d, np.zeros(4, dtype=np.uint8)]).astype(np.uint32)
    return z[q] | (z[q + 1] << 8) | (z[q + 2] << 16) | (z[q + 3] << 24)


def expected_mask(d: np.ndarray):
    """(skip mask, True when the entropy sum of some stretch lies too close to the threshold to call in float)"""
    n = len(d)
    nfull = n >> 10
    cand = 0
    close = False
    thr = (10.0 - NOISE_BITS) * 1024.0
    for kb in range(nfull):
        s = d[kb << 10:(kb + 1) << 10]
        tops = int((s.reshape(32, 32)[:, :4] >= 128).sum())  # word 8 * lane of the stretch, all four bytes
        if tops < 40 or tops > 88:
            continue
        c = np.bincount(s, minlength=256).astype(np.float64)
        c = c[c > 1]
        v = float((c * np.log2(c)).sum())
        close |= abs(v - thr) < 1.0
        if v < thr:
            cand |= 1 << kb
    if not cand:
        return 0, close
    bb = hb_of(n) + 4
    nh = n - 2 if n >= 3 else 0
    isc = np.zeros(max(nh, 1), dtype=bool)
    for kb in range(nfull):
        if (cand >> kb) & 1:
            isc[kb << 10:(kb + 1) << 10] = True
    isc = isc[:nh]
    h = ((windows(d, np.arange(nh)).astype(np.uint64) * 0x9E3779B1) & 0xFFFFFFFF) >> np.uint64(32 - bb)
    hc, ho = h[isc], h[~isc]
    coll = len(hc) - len(np.unique(hc))
    set2 = len(np.unique(ho))
    coll2 = int(np.isin(hc, ho).sum())
    nc = bin(cand).count("1") << 10
    allowed = ((nc * nc) >> (bb + 1)) + (nc >> 6) + 48
    allowed2 = ((set2 * nc) >> bb) + (nc >> 6) + 48
    return (0 if coll > allowed or coll2 > allowed2 else cand), close


def crafted():
    rng = np.random.default_rng(20261020)
    noise = lambda k: rng.integers(0, 256, k, dtype=np.uint8)
    out = [np.frombuffer(bytes(range(256)) * 4, dtype=np.uint8), np.frombuffer(bytes(range(256)) * 16, dtype=np.uint8)]
    for n in (1023, 1024, 1025, 1026, 2047, 2048, 2049, 4096, 4097, 4098, 8191, 8192, 8193, 16385, 31745, 65535):
        out.append(noise(n))
    nz = noise(3072)
    for part in (64, 200, 600, 1024):  # noise followed by a copy of part of it: a narrower histogram, found by the second set
        out.append(np.concatenate([nz, nz[100:100 + part], np.zeros(1024 - part % 1024 if part < 1024 else 0, np.uint8)]))
        out.append(np.concatenate([nz, nz[500:500 + part], corpus.gen_text(2000, 596, part)]))
    out.append(np.concatenate([nz, nz, nz[:7]]))                    # a noise block stored twice
    out.append(np.tile(rng.permutation(256).astype(np.uint8), 16))  # a permutation table stored 16 times
    for k in range(186, 236, 4):                                   # byte alphabets around the entropy threshold
        out.append(rng.integers(0, k, 6 * 1024 + 300, dtype=np.uint8))
    t = corpus.gen_text(5000, 596, 3)
    out.append(np.concatenate([t[:1024], noise(4096), t[:1500]]))    # text, noise, text that repeats the first stretch
    out.append(np.concatenate([noise(2048), np.zeros(1, np.uint8)]))
    out.append(np.zeros(0, np.uint8))
    out.append(noise(2))
    return out


def c2_shaped():
    out = []
    for i, n in enumerate((900, 1025, 5632, 8192, 9000, 16384, 20000, 31744, 40000, 61440)):
        out.append(corpus.gen_jpeg_like(n, 596, 100 + i))
        out.append(corpus.gen_bitmap_like(n, 596, 200 + i))
    buf, offs, sizes = corpus.c2_buffer(120, seed=corpus.BASE_SEED + 3)
    out += [buf[offs[i]:offs[i + 1]] for i in range(len(sizes))]
    return out


@pytest.fixture(scope="module")
def ctx():
    c = emu_lib.emu_context()
    yield c
    c.close()


def run_masks(ctx, chunks):
    # every chunk at a 16-byte aligned offset: the histograms read aligned words, so no neighbour byte enters them
    lens = np.array([len(c) for c in chunks], dtype=np.uint32)
    off = np.zeros(len(chunks), dtype=np.uint64)
    pos = 0
    for i, n in enumerate(lens):
        off[i] = pos
        pos += (int(n) + 15) & ~15
    raw = np.zeros(pos + 16, dtype=np.uint8)
    for i, c in enumerate(chunks):
        raw[int(off[i]):int(off[i]) + len(c)] = c
    ctx.deflate_batch(raw, off, lens)
    masks = np.zeros(len(chunks), dtype=np.uint64)
    ctx.lib.zwz_emu_match_skipmasks(masks.ctypes.data_as(__import__("ctypes").c_void_p), len(chunks))
    return masks


@pytest.mark.parametrize("kind", ["crafted", "c2"])
def test_skip_mask_matches_numpy(ctx, kind):
    chunks = crafted() if kind == "crafted" else c2_shaped()
    assert all(len(c) <= 65535 for c in chunks)
    masks = run_masks(ctx, chunks)
    seen_skip = seen_kept = 0
    for i, c in enumerate(chunks):
        want, close = expected_mask(np.asarray(c, dtype=np.uint8))
        if close:
            continue
        assert int(masks[i]) == want, (kind, i, len(c), hex(int(masks[i])), hex(want))
        seen_skip += want != 0
        seen_kept += want == 0 and len(c) >= 1024
    assert seen_skip and seen_kept  # both verdicts occur
