"""Hand-made DEFLATE streams aimed at the inflate decode tables: Huffman codes of every length 1..15, codes longer than the
table index of either alphabet (10 bits literal/length, 8 bits distance), a distance tree with a single code, incomplete
code sets and the symbols no stream may use (literal/length 286/287, distance 30/31). Every stream, and cuts of it, goes
through each inflate path; bytes, length and status must be the oracle's (zlib 1.3)."""
import zlib

import numpy as np

import oracle_lib as O

CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [i // 4 for i in range(4, 24)] + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
DIST_EXTRA = [0] * 4 + [i // 2 - 1 for i in range(4, 30)]


def canonical(lengths):
    """RFC 1951 §3.2.2: symbol -> (code, length) for every symbol with a nonzero length."""
    cnt = [0] * 16
    for ln in lengths:
        cnt[ln] += 1
    cnt[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + cnt[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, ln in enumerate(lengths):
        if ln:
            out[s] = (nxt[ln], ln)
            nxt[ln] += 1
    return out


class Writer:
    def __init__(self):
        self.acc, self.n, self.out, self.raw = 0, 0, bytearray(), bytearray()
        self.put(0x9c78, 16)

    def put(self, v, nb):
        self.acc |= v << self.n
        self.n += nb
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, v, nb):
        self.put(int(format(v, f"0{nb}b")[::-1], 2) if nb else 0, nb)

    def dynamic_header(self, ll, dl, cl=None, last=True):
        """Block header with literal/length lengths `ll` and distance lengths `dl`, every length sent as its own code-length
        symbol; `cl` (19 code-length-code lengths by symbol) defaults to a complete 4-bit code for symbols 0..15."""
        self.put(1 if last else 0, 1)
        self.put(2, 2)
        self.put(len(ll) - 257, 5)
        self.put(len(dl) - 1, 5)
        self.put(15, 4)
        cl = cl or [4] * 16 + [0, 0, 0]
        for s in CL_ORDER:
            self.put(cl[s], 3)
        clc = canonical(cl)
        for ln in list(ll) + list(dl):
            self.code(*clc[ln])
        self.ll, self.dl = canonical(ll), canonical(dl)

    def fixed_header(self, last=True):
        self.put(1 if last else 0, 1)
        self.put(1, 2)
        self.ll = canonical([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)
        self.dl = canonical([5] * 32)

    def lit(self, b):
        self.code(*self.ll[b])
        self.raw.append(b)

    def sym(self, s):   # a literal/length symbol as it is, valid or not
        self.code(*self.ll[s])

    def match(self, length, dsym, dextra=0):
        k = max(i for i in range(29) if LEN_BASE[i] <= length and (i < 28 or length == 258))
        self.code(*self.ll[257 + k])
        self.put(length - LEN_BASE[k], LEN_EXTRA[k])
        self.code(*self.dl[dsym])
        if dsym < 30:
            self.put(dextra, DIST_EXTRA[dsym])
            dist = DIST_BASE[dsym] + dextra
            for _ in range(length):
                self.raw.append(self.raw[-dist] if dist <= len(self.raw) else 0)

    def finish(self, eob=True):
        if eob:
            self.code(*self.ll[256])
        if self.n:
            self.out.append(self.acc & 255)
            self.acc, self.n = 0, 0
        return bytes(self.out) + zlib.adler32(bytes(self.raw)).to_bytes(4, "big")


# 256 literals of 9 bits, end-of-block of 2 bits, lengths 3 and 4 of 3 bits: a complete set
COMPLETE_LL = [9] * 256 + [2, 3, 3] + [0] * 27


def every_length_stream():
    """Literal/length codes of every length 1..15 (the last two of length 15 complete the set); distance codes of every
    length 1..15 as well. Codes of 11 and more bits are longer than the literal/length index, of 9 and more than the distance
    index."""
    ll = [0] * 286
    syms = [ord(c) for c in "etaoinshrdl"] + [256, 257, 258, 259, 264]   # lengths 1..11, 12..15, 15
    for i, s in enumerate(syms):
        ll[s] = min(i + 1, 15)
    dl = [0] * 30
    for i in range(16):
        dl[i] = min(i + 1, 15)
    w = Writer()
    w.dynamic_header(ll, dl)
    for i in range(300):   # distances up to 256 need that much output first
        w.lit(ord("etaoinshrdl"[(i * 5) % 11]))
    for rep in range(40):
        for c in "etaoinshrdl":
            w.lit(ord(c))
        for k, length in enumerate((3, 4, 5, 10)):
            dsym = (rep * 4 + k) % 16
            w.match(length, dsym, (rep * 7) & ((1 << DIST_EXTRA[dsym]) - 1))
    return w.finish()


def single_distance_code_stream(bad_code=False):
    """A distance tree with one code of one bit (zlib accepts that incomplete set); with `bad_code` a match uses the
    other, unassigned bit pattern, which zlib rejects as an invalid distance code."""
    w = Writer()
    w.dynamic_header(COMPLETE_LL, [1])
    for i in range(300):
        w.lit((i * 37) & 255)
        if i % 9 == 8:
            w.match(3 + (i % 2), 0)
    if bad_code:
        w.code(*w.ll[257])
        w.put(1, 1)   # distance code "1": not part of the set
        w.lit(1)
    return w.finish()


def incomplete_sets():
    out = []
    # code-length code: two codes of 2 bits
    hdr = Writer()
    hdr.put(1, 1)
    hdr.put(2, 2)
    hdr.put(0, 5)
    hdr.put(0, 5)
    hdr.put(15, 4)
    cl = [0] * 19
    cl[8], cl[0] = 2, 2
    for s in CL_ORDER:
        hdr.put(cl[s], 3)
    hdr.put(0, 30)
    out.append(hdr.finish(eob=False))
    # literal/length: 256 codes of 9 bits + EOB of 9 bits, nothing else (incomplete, more than one code)
    ll = [9] * 257 + [0] * 29
    w = Writer()
    w.dynamic_header(ll, [1])
    out.append(w.finish(eob=False))
    # distance: three codes of 2 bits
    w = Writer()
    w.dynamic_header(COMPLETE_LL, [2, 2, 2])
    out.append(w.finish())
    return out


def invalid_symbol_streams():
    """Fixed-Huffman blocks that use literal/length 286 or 287 or distance 30 or 31 after a run of valid tokens."""
    out = []
    for kind in (286, 287, 30, 31):
        for lead in (0, 5, 2000):
            w = Writer()
            w.fixed_header()
            for i in range(lead):
                w.lit((i * 11) & 255)
                if i % 13 == 12:
                    w.match(5, 3)
            if kind >= 286:
                w.sym(kind)
            else:
                w.code(*w.ll[257])
                w.code(kind, 5)
            for i in range(40):
                w.lit(i)
            out.append(w.finish())
    return out


def all_streams():
    full = [every_length_stream(), single_distance_code_stream(), single_distance_code_stream(bad_code=True)] + incomplete_sets() + \
        invalid_symbol_streams()
    cases = list(full)
    for s in full[:3]:
        cases += [s[:n] for n in sorted({3, len(s) // 3, len(s) // 2, len(s) - 5, len(s) - 1})]
    return cases


def test_crafted_streams_are_what_they_claim():
    s = every_length_stream()
    _, st, n = O.inflate(s, 1 << 20)
    assert st == O.STREAM_END and n > 1000
    assert O.inflate(single_distance_code_stream(), 1 << 20)[1] == O.STREAM_END
    assert O.inflate(single_distance_code_stream(True), 1 << 20)[1] == O.STREAM_BAD
    for s in incomplete_sets() + invalid_symbol_streams():
        assert O.inflate(s, 1 << 20)[1] == O.STREAM_BAD


def test_inflate_decode_table_edges(ctx_inf):
    cases = all_streams()
    cap = 1 << 17
    off = np.zeros(len(cases) + 1, dtype=np.uint64)
    np.cumsum([len(c) for c in cases], out=off[1:])
    raw_off = np.arange(len(cases) + 1, dtype=np.uint64) * np.uint64(cap)
    out, rl, st = ctx_inf.inflate_batch(b"".join(cases), off[:-1], np.diff(off).astype(np.uint32), raw_off)
    for i, s in enumerate(cases):
        want, wst, wn = O.inflate(s, cap)
        assert (int(rl[i]), int(st[i])) == (wn, wst), (i, len(s))
        assert out[int(raw_off[i]):int(raw_off[i]) + wn].tobytes() == want, (i, len(s))
