// inflate.cuh — batched DEFLATE decoder, one warp per stream: zlib-wrapped (the .zwz records), gzip members or raw DEFLATE,
// chosen by the format field of the flags (ZWZ_INFLATE_FORMAT). The wrapper is parsed and checked here; the block decoders
// below it are the same for all three.
//
// Replaces decompression.cpp:11-37 (inflateInit / inflate(Z_NO_FLUSH) loop / inflateEnd, return codes ignored).
// Output contract = the bytes zlib 1.3 would have written for the same input (see oracle/zwz_oracle.c for the rules):
// a literal needs its whole code inside the input, a match needs length+extra+distance+extra, a stored block copies
// min(LEN, bytes left), and whatever was produced before an error or the end of the input stays.
//
// Layout per warp
//   * the compressed stream is read as aligned 32-bit words, 32 words at a time (one coalesced 128-byte load, the next
//     128 bytes already in flight); the word feeding the bit buffer comes from a register of the owning lane by shuffle;
//   * the bit buffer and every decode decision are computed redundantly by all 32 lanes (warp-uniform control flow, no
//     divergence, no broadcast needed), so the lanes are all there when a match has to be copied;
//   * literal/length and distance codes resolve through shared-memory lookup tables (2^10 and 2^8 16-bit entries, one LDS
//     per symbol, filled by scattering each code into its slots); longer codes fall back to a canonical walk;
//   * literals are parked in the lane `position & 31` and stored 32 at a time; back-references are copied by the whole
//     warp, 32 bytes per step (pattern-replicated when distance < 32).
// Output bytes are written straight to global memory; back-references re-read them through L1/L2 (the window of one
// 65 535-byte record fits L1+L2 trivially). Shared memory holds the decode tables, the staged window and the token regions of
// inflate_fast.cuh: 10 336 bytes per warp, so with 1 KB reserved per CTA 20 one-warp CTAs fit an SM (registers would allow
// 24). The decoder is latency-bound: resident warps hide it, but so do long windows, which take fewer rounds and commit more
// per round. 20 warps with 416-bit lane ranges measured faster than 24 with 288-bit ones (profiles/inflate_smem/).
//
// Algorithmic bytes per stream: N_comp read + N_raw written (SURVEY.md §8(d)).
#pragma once
#include "zwz_common.cuh"
#include "crc32.cuh"

namespace zwz {

#define ZWZ_INF_WARPS 1 // one warp per CTA
// registers <= 80 a thread, which would allow 24 resident CTAs per SM (6 warps for each of the 4 schedulers): registers never
// bind before shared memory does
#define ZWZ_INF_MIN_CTAS 24
#define ZWZ_INF_LBITS 10
#define ZWZ_INF_DBITS 8

// Decode-table entries are 16 bits.
// literal/length: [3:0] code length, [6:4] extra bits, [15:7] literal byte (0..255) or 253 + base length (256..511).
//                 Extra-bits field 7 marks the other entries by their value: 0 end-of-block, 1 invalid code whose length is
//                 in [3:0] (zlib's op=64 entries), 2 code longer than the table index (canonical walk needed).
// distance:       [3:0] code length, [7:4] extra bits, [9:8] m, [11:10] 0 valid, 1 invalid code (length in [3:0]), 2 code
//                 longer than the index. distance - 1 = (m << extra bits) | extra: m is the symbol for symbols 0..3 and
//                 2 | (symbol & 1) above.
// code-length code: [3:0] code length, [8:4] symbol.
#define ZWZ_LL_LIT(nb, byte) ((uint32_t) (nb) | ((uint32_t) (byte) << 7))
#define ZWZ_LL_LEN(nb, eb, base) ((uint32_t) (nb) | ((uint32_t) (eb) << 4) | (((uint32_t) (base) + 253u) << 7))
#define ZWZ_LL_EOB(nb) ((uint32_t) (nb) | 0x70u)
#define ZWZ_LL_INVALID(nb) ((uint32_t) (nb) | 0x70u | (1u << 7))
#define ZWZ_LL_LONG (0x70u | (2u << 7))
#define ZWZ_LL_IS_LIT(e) (((e) & 0x8070u) == 0u)
#define ZWZ_LL_IS_LEN(e) ((e) >= 0x8000u)
#define ZWZ_LL_IS_EOB(e) (((e) >> 4) == 7u)
#define ZWZ_LL_IS_INVALID(e) (((e) >> 4) == 15u)
#define ZWZ_LL_IS_LONG(e) (((e) >> 4) == 23u)
#define ZWZ_D_ENTRY(nb, eb, m) ((uint32_t) (nb) | ((uint32_t) (eb) << 4) | ((uint32_t) (m) << 8))
#define ZWZ_D_INVALID(nb) ((uint32_t) (nb) | (1u << 10))
#define ZWZ_D_LONG (2u << 10)
#define ZWZ_D_IS_LONG(e) (((e) >> 10) == 2u)
#define ZWZ_D_IS_SPECIAL(e) (((e) >> 10) != 0u)
// distance - 1 of a valid entry, given the bits that follow its code
#define ZWZ_D_DM1(e, bits) ((((e) >> 8 & 3u) << ((e) >> 4 & 15u)) | (((bits) >> ((e) & 15u)) & ((1u << ((e) >> 4 & 15u)) - 1u)))

// Token entries (u16) a lane may emit per decode window of inflate_fast.cuh; a multiple of 4. A window whose lane fills its
// region is cut there, so the region has to hold what ZWZ_IF_SW words decode to (a literal takes one entry, a match two):
// 80 entries over 416 bits, one per 5.2 bits. 44 or 64 entries over 480 bits cut most windows of C2-shaped data.
#ifndef ZWZ_IF_R
#define ZWZ_IF_R 80u
#endif
#define ZWZ_IF_RS (ZWZ_IF_R + 2u) // region stride in u16: an odd number of words, so equal offsets in 32 regions hit 32 banks
#ifndef ZWZ_IF_SW
#define ZWZ_IF_SW 13u // words of compressed data per lane and decode window (odd: conflict-free strides)
#endif
#define ZWZ_IF_CW (32u * ZWZ_IF_SW + 8u) // staged words: 32 ranges + the overshoot of the last token

struct InflateWarpSmem {
    union {
        struct {
            uint16_t lit[1 << ZWZ_INF_LBITS];
            uint16_t dst[1 << ZWZ_INF_DBITS];
            uint16_t sorted_ll[288];
            uint16_t sorted_d[32];
            uint32_t cnt_ll[16];
            uint32_t cnt_d[16];
            uint32_t run[16];            // running offsets while sorting
            uint32_t cw[ZWZ_IF_CW];     // inflate_fast.cuh: staged window of compressed words, then the resolve staging area
            union {
                struct { // block header parsing only: dead once the tables are built, when the token regions come to life
                    uint8_t lens[352]; // [0,19) code-length-code lengths; [32, 32+316) literal/length then distance lengths
                    uint16_t clt[128]; // code-length-code table (7 bits)
                    uint16_t sorted_cl[20];
                    uint32_t cnt_cl[16];
                };
                uint16_t tok[32u * ZWZ_IF_RS]; // inflate_fast.cuh: one token region per lane
            };
        };
        // gzip: CRC-32 slice table. Only used before the first block header and after the last block, when nothing above
        // is alive, so the gzip path needs no shared memory of its own.
        uint32_t crc[1024];
    };
};
#define ZWZ_INF_SMEM (ZWZ_INF_WARPS * (uint32_t) sizeof(zwz::InflateWarpSmem))
static_assert(sizeof(InflateWarpSmem) > sizeof(uint32_t[1024]), "the CRC-32 table must not set the size of the decoder's shared memory");

ZWZ_DEV uint32_t inf_litlen_entry(uint32_t sym, uint32_t nb) {
    if (sym < 256u) return ZWZ_LL_LIT(nb, sym);
    if (sym == 256u) return ZWZ_LL_EOB(nb);
    if (sym > 285u) return ZWZ_LL_INVALID(nb);
    uint32_t k = sym - 257u, eb, base;
    if (k < 8u) {
        eb = 0;
        base = 3u + k;
    } else if (k == 28u) {
        eb = 0;
        base = 258u;
    } else {
        eb = (k - 4u) >> 2;
        base = 3u + ((4u + (k & 3u)) << eb);
    }
    return ZWZ_LL_LEN(nb, eb, base);
}
ZWZ_DEV uint32_t inf_dist_entry(uint32_t sym, uint32_t nb) {
    if (sym > 29u) return ZWZ_D_INVALID(nb);
    if (sym < 4u) return ZWZ_D_ENTRY(nb, 0, sym);
    return ZWZ_D_ENTRY(nb, (sym >> 1) - 1u, 2u | (sym & 1u));
}
ZWZ_DEV uint32_t inf_cl_entry(uint32_t sym, uint32_t nb) { return nb | (sym << 4); }

// Canonical-code walk over `bits` (LSB first), lengths 1..maxwalk. Returns entry-maker input (sym,len) or ~0u.
ZWZ_DEV uint32_t inf_canon_walk(uint32_t bits, const uint32_t *cnt, const uint16_t *sorted, uint32_t maxwalk, uint32_t &len_out) {
    int code = 0, first = 0, index = 0;
    for (uint32_t len = 1; len <= maxwalk; ++len) {
        code |= (int) (bits & 1u);
        bits >>= 1;
        int c = (int) cnt[len];
        if (code - c < first) {
            len_out = len;
            return sorted[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return 0xffffffffu;
}

// Warp-cooperative table build. kind: 0 = code-length code (must be complete), 1 = literal/length, 2 = distance.
// Returns (warp-uniform) 0 ok / 1 invalid set. max_len_out = longest code (0 = empty set).
template <int KIND>
ZWZ_DEV int inf_build(const uint8_t *lens, uint32_t n, uint32_t *cnt, uint16_t *sorted, uint32_t *run, uint16_t *table, uint32_t tbits,
                      uint32_t &max_len_out) {
    const unsigned lane = lane_id();
    if (lane < 16u) cnt[lane] = 0;
    __syncwarp();
    for (uint32_t s = lane; s < n; s += 32u) atomicAdd(&cnt[lens[s]], 1u);
    __syncwarp();
    // validity (inftrees.c rules), computed redundantly by every lane
    uint32_t max_len = 0;
    int left = 1, bad = 0;
    uint32_t acc = 0;
    for (uint32_t l = 1; l <= 15u; ++l) {
        uint32_t c = cnt[l];
        if (c) max_len = l;
        left = (left << 1) - (int) c;
        if (left < 0) bad = 1;
        acc += c;
    }
    __syncwarp();
    // running offsets per length: run[l] = start of length-l symbols in `sorted`
    if (lane == 0) {
        uint32_t o = 0;
        for (uint32_t l = 1; l <= 15u; ++l) {
            run[l] = o;
            o += cnt[l];
        }
        run[0] = 0;
    }
    __syncwarp();
    max_len_out = max_len;
    if (bad) return 1;
    if (max_len != 0 && left > 0 && (KIND == 0 || max_len != 1u)) return 1; // incomplete set
    // stable sort of symbols by (length, symbol): 32 symbols per step
    for (uint32_t base = 0; base < n; base += 32u) {
        uint32_t s = base + lane;
        uint32_t L = s < n ? lens[s] : 0u;
        unsigned grp = __match_any_sync(ZWZ_FULL, L);
        if (L) {
            uint32_t r = (uint32_t) __popc(grp & ((1u << lane) - 1u));
            sorted[run[L] + r] = (uint16_t) s;
        }
        __syncwarp();
        if (L && (grp >> lane) == 1u) run[L] += (uint32_t) __popc(grp); // highest lane of each group
        __syncwarp();
    }
    // fill. Slots that start no code of <= tbits bits: the prefix of a longer code (or of none, in an incomplete set)
    if (left > 0 || max_len > tbits) {
        const uint32_t dflt = KIND == 0 ? 0u
                                        : (max_len > tbits ? (KIND == 1 ? ZWZ_LL_LONG : ZWZ_D_LONG)
                                                           : (KIND == 1 ? ZWZ_LL_INVALID(max_len ? max_len : 1u) : ZWZ_D_INVALID(max_len ? max_len : 1u)));
        uint32_t *t2 = (uint32_t *) table;
        for (uint32_t e = lane; e < (1u << (tbits - 1u)); e += 32u) t2[e] = dflt | (dflt << 16);
        __syncwarp();
    }
    // then every code of <= tbits bits writes its 2^(tbits - len) slots: the bit-reversed code, followed by any bits.
    // The (code, replica) pairs of one length are spread over the lanes, so a short code does not keep one lane busy.
    const uint32_t top = max_len < tbits ? max_len : tbits;
    uint32_t code = 0, idx = 0; // canonical code of the first length-l code; its place in `sorted`
    for (uint32_t l = 1; l <= top; ++l) {
        const uint32_t c = cnt[l], sh = tbits - l;
        for (uint32_t t = lane; t < (c << sh); t += 32u) {
            const uint32_t i = t >> sh;
            const uint32_t sym = sorted[idx + i];
            const uint32_t r = __brev(code + i) >> (32u - l);
            table[r | ((t & ((1u << sh) - 1u)) << l)] =
                (uint16_t) (KIND == 0 ? inf_cl_entry(sym, l) : (KIND == 1 ? inf_litlen_entry(sym, l) : inf_dist_entry(sym, l)));
        }
        idx += c;
        code = (code + c) << 1;
    }
    __syncwarp();
    return 0;
}

// Warp-uniform bit reader over aligned words with a 32-word register cache per lane.
struct InfBits {
    const uint32_t *wbase;  // aligned word holding the stream's first byte
    uint32_t skew;          // byte offset of the stream inside that word
    uint32_t nbytes;        // stream length
    uint32_t nwords;        // words covering [skew, skew + nbytes)
    uint32_t nfull;         // leading words that lie entirely inside the stream: while widx <= nfull every fed bit is real
    uint32_t widx;          // next word to feed
    uint32_t cache, cache_next;
    uint32_t cache_blk;     // block (32 words) held in `cache`; cache_next holds cache_blk + 1
    uint64_t hold;
    uint32_t cnt;           // valid bits in hold
    uint64_t fed;           // stream bits fed into hold so far (may run past 8 * nbytes: zero padding)
};

// a reader over p[0, nbytes); position it with infb_seek or infb_seek_bits
ZWZ_DEV void infb_open(InfBits &b, const uint8_t *p, uint32_t nbytes) {
    b.skew = (uint32_t) ((uintptr_t) p & 3u);
    b.wbase = (const uint32_t *) (p - b.skew);
    b.nbytes = nbytes;
    b.nwords = (b.skew + nbytes + 3u) >> 2;
    b.nfull = (b.skew + nbytes) >> 2;
}
ZWZ_DEV uint32_t infb_load(const InfBits &b, uint32_t k) {
    if (k >= b.nwords) return 0u;
    uint32_t w = __ldg(b.wbase + k);
    // bytes of the last word that lie past the end of the stream belong to somebody else: zero them
    uint32_t end = b.skew + b.nbytes; // byte index one past the stream, relative to wbase
    if ((k + 1u) * 4u > end) {
        uint32_t keep = end - k * 4u; // 1..3
        w &= (1u << (keep * 8u)) - 1u;
    }
    return w;
}
ZWZ_DEV uint32_t infb_next_word(InfBits &b) {
    uint32_t blk = b.widx >> 5;
    if (blk != b.cache_blk) { // warp-uniform
        if (blk == b.cache_blk + 1u) {
            b.cache = b.cache_next;
        } else {
            b.cache = infb_load(b, blk * 32u + lane_id());
        }
        b.cache_next = infb_load(b, (blk + 1u) * 32u + lane_id());
        b.cache_blk = blk;
    }
    uint32_t w = __shfl_sync(ZWZ_FULL, b.cache, (int) (b.widx & 31u));
    b.widx++;
    return w;
}
// position the reader at stream byte `byte_pos`
ZWZ_DEV void infb_seek(InfBits &b, uint32_t byte_pos) {
    uint32_t a = b.skew + byte_pos;
    b.widx = a >> 2;
    b.cache_blk = 0xfffffff0u;
    b.hold = 0;
    b.cnt = 0;
    uint32_t w = infb_next_word(b);
    uint32_t drop = (a & 3u) * 8u;
    b.hold = (uint64_t) (w >> drop);
    b.cnt = 32u - drop;
    b.fed = (uint64_t) byte_pos * 8u + b.cnt;
}
ZWZ_DEV void infb_refill(InfBits &b) {
    if (b.cnt <= 32u) {
        uint32_t w = infb_next_word(b);
        b.hold |= (uint64_t) w << b.cnt;
        b.cnt += 32u;
        b.fed += 32u;
    }
}
ZWZ_DEV void infb_drop(InfBits &b, uint32_t n) {
    b.hold >>= n;
    b.cnt -= n;
}
// bits consumed from the stream so far
ZWZ_DEV uint64_t infb_used(const InfBits &b) { return b.fed - b.cnt; }
// position the reader at stream bit `bit_pos`
ZWZ_DEV void infb_seek_bits(InfBits &b, uint64_t bit_pos) {
    infb_seek(b, (uint32_t) (bit_pos >> 3));
    infb_drop(b, (uint32_t) bit_pos & 7u); // <= 7 of the >= 8 bits the seek left in the buffer
}
// Everything already in `hold` is real stream data while only whole words of the stream have been fed; only the tail of a
// stream (or a truncated one) needs the per-symbol availability checks that give zlib's exact stop position.
ZWZ_DEV bool infb_inside(const InfBits &b) { return b.widx <= b.nfull; }
// the next n bits (n <= the bits in `hold`) lie inside the stream
ZWZ_DEV bool infb_need(const InfBits &b, uint32_t n) { return infb_inside(b) || infb_used(b) + n <= (uint64_t) b.nbytes * 8u; }

} // namespace zwz
#include "inflate_fast.cuh"
namespace zwz {

// CRC-32 of p[0, n) by the calling warp. The slice table overlays the warp's decoder state, which is dead before the first
// block header and after the last block: the shared-memory layout stays that of the zlib path.
ZWZ_DEV_NOINLINE uint32_t inf_crc32(const uint8_t *p, uint32_t n) {
    ZWZ_DYN_SMEM(inf_raw);
    uint32_t *tab = ((InflateWarpSmem *) inf_raw)[warp_id()].crc;
    __syncwarp();
    crc32_load_table(tab, lane_id(), 32u);
    __syncwarp();
    return crc32_warp(p, n, tab);
}

// RFC 1952 member header as zlib 1.3 reads it with windowBits 31 (inflate.c HEAD, FLAGS .. HCRC): the header length << 2 with
// ZWZ_STREAM_END, or the status zlib ends with (a header cut short is TRUNCATED, a wrong ID or CM, reserved FLG bits or a header
// CRC mismatch BAD). Byte-serial and warp-uniform; the zero-terminated FNAME / FCOMMENT are scanned 32 bytes a step.
ZWZ_DEV_NOINLINE uint32_t inf_gzip_header(const uint8_t *comp, uint32_t comp_len) {
    const unsigned lane = lane_id();
    if (comp_len < 2u) return ZWZ_STREAM_TRUNCATED;
    if (comp[0] != 0x1fu || comp[1] != 0x8bu) return ZWZ_STREAM_BAD;
    if (comp_len < 4u) return ZWZ_STREAM_TRUNCATED;
    const uint32_t flg = comp[3];
    if (comp[2] != 8u || (flg & 0xe0u)) return ZWZ_STREAM_BAD;
    uint32_t p = 10u; // ID1 ID2 CM FLG MTIME(4) XFL OS
    if (comp_len < p) return ZWZ_STREAM_TRUNCATED;
    if (flg & 0x04u) { // FEXTRA: XLEN, then XLEN bytes
        if (comp_len < p + 2u) return ZWZ_STREAM_TRUNCATED;
        p += 2u + ((uint32_t) comp[p] | ((uint32_t) comp[p + 1u] << 8));
        if (comp_len < p) return ZWZ_STREAM_TRUNCATED;
    }
    for (uint32_t f = 0x08u; f <= 0x10u; f <<= 1) { // FNAME, FCOMMENT
        if (!(flg & f)) continue;
        for (;;) {
            if (p >= comp_len) return ZWZ_STREAM_TRUNCATED;
            const uint32_t q = p + lane;
            const unsigned z = __ballot_sync(ZWZ_FULL, q < comp_len && comp[q] == 0u);
            if (z) {
                p += (uint32_t) __ffs((int) z);
                break;
            }
            p += 32u;
        }
    }
    if (flg & 0x02u) { // FHCRC: low 16 bits of the CRC-32 of everything before it
        if (comp_len < p + 2u) return ZWZ_STREAM_TRUNCATED;
        const uint32_t want = (uint32_t) comp[p] | ((uint32_t) comp[p + 1u] << 8);
        if ((inf_crc32(comp, p) & 0xffffu) != want) return ZWZ_STREAM_BAD;
        p += 2u;
    }
    return (p << 2) | ZWZ_STREAM_END;
}

// 32-bit values of the trailers: RFC 1950's Adler-32 is big-endian, RFC 1952's CRC-32 and ISIZE little-endian
ZWZ_DEV uint32_t inf_be32(const uint8_t *p) { return ((uint32_t) p[0] << 24) | ((uint32_t) p[1] << 16) | ((uint32_t) p[2] << 8) | p[3]; }
ZWZ_DEV uint32_t inf_le32(const uint8_t *p) { return (uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24); }

// The decoding steps below are shared by the batch decoder (inflate_stream), the span decoder and the block finder
// (inflate_stream.cuh). Each returns ZWZ_STREAM_END when it succeeded, else the status zlib ends with there; all are warp-uniform.

// RFC 1950 header (inflate.c HEAD) at the reader: consumes CMF and FLG and returns FLG in `flg`. FDICT is BAD unless fdict_ok:
// without a dictionary it is zlib's Z_NEED_DICT, and nothing can be decoded.
ZWZ_DEV uint32_t inf_zlib_header(InfBits &B, bool fdict_ok, uint32_t &flg) {
    infb_refill(B);
    if (!infb_need(B, 16)) return ZWZ_STREAM_TRUNCATED;
    const uint32_t cmf = (uint32_t) B.hold & 0xffu;
    flg = ((uint32_t) B.hold >> 8) & 0xffu;
    if (((cmf << 8) + flg) % 31u != 0u || (cmf & 15u) != 8u || (cmf >> 4) + 8u > 15u || ((flg & 0x20u) && !fdict_ok)) return ZWZ_STREAM_BAD;
    infb_drop(B, 16);
    return ZWZ_STREAM_END;
}

// Stored block after its 3 header bits: skips to the byte boundary and reads LEN / NLEN. The block's bytes start at stream byte
// `bpos`; `len` is LEN. The caller copies min(LEN, bytes left) and then seeks to bpos + len.
ZWZ_DEV uint32_t inf_stored_header(InfBits &B, uint32_t &bpos, uint32_t &len) {
    bpos = (uint32_t) ((infb_used(B) + 7u) >> 3);
    if ((uint64_t) bpos + 4u > B.nbytes) return ZWZ_STREAM_TRUNCATED;
    infb_seek(B, bpos);
    infb_refill(B);
    const uint32_t v = (uint32_t) B.hold;
    if ((v & 0xffffu) != ((v >> 16) ^ 0xffffu)) return ZWZ_STREAM_BAD;
    len = v & 0xffffu;
    bpos += 4u;
    return ZWZ_STREAM_END;
}

// the tables of a fixed-Huffman block (RFC 1951 §3.2.6)
ZWZ_DEV void inf_fixed_tables(InflateWarpSmem &S, uint32_t &max_ll, uint32_t &max_d) {
    const unsigned lane = lane_id();
    for (uint32_t s = lane; s < 288u; s += 32u) S.lens[32u + s] = (uint8_t) (s < 144u ? 8 : (s < 256u ? 9 : (s < 280u ? 7 : 8)));
    S.lens[320u + lane] = 5;
    __syncwarp();
    inf_build<1>(S.lens + 32, 288u, S.cnt_ll, S.sorted_ll, S.run, S.lit, ZWZ_INF_LBITS, max_ll);
    inf_build<2>(S.lens + 320, 32u, S.cnt_d, S.sorted_d, S.run, S.dst, ZWZ_INF_DBITS, max_d);
}

// The tables of a dynamic block (RFC 1951 §3.2.7), read after its 3 header bits with at least 14 bits left in `hold` (what a
// refill leaves behind them): HLIT / HDIST / HCLEN, the code-length code, the code lengths, then both codes built as inf_build
// requires, with code 256 present. The block finder's candidates are the headers this accepts.
ZWZ_DEV uint32_t inf_dyn_tables(InflateWarpSmem &S, InfBits &B, uint32_t &max_ll, uint32_t &max_d) {
    const unsigned lane = lane_id();
    if (!infb_need(B, 14)) return ZWZ_STREAM_TRUNCATED;
    const uint32_t nlen = ((uint32_t) B.hold & 31u) + 257u;
    const uint32_t ndist = (((uint32_t) B.hold >> 5) & 31u) + 1u;
    const uint32_t ncode = (((uint32_t) B.hold >> 10) & 15u) + 4u;
    infb_drop(B, 14);
    if (nlen > 286u || ndist > 30u) return ZWZ_STREAM_BAD;
    if (lane < 19u) S.lens[lane] = 0;
    __syncwarp();
    for (uint32_t i = 0; i < ncode; ++i) {
        infb_refill(B);
        if (!infb_need(B, 3)) return ZWZ_STREAM_TRUNCATED;
        // permutation 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
        const uint32_t slot = i < 3u ? 16u + i : (i == 3u ? 0u : ((i & 1u) ? 7u - ((i - 5u) >> 1) : 8u + ((i - 4u) >> 1)));
        if (lane == 0) S.lens[slot] = (uint8_t) ((uint32_t) B.hold & 7u);
        infb_drop(B, 3);
    }
    __syncwarp();
    uint32_t max_cl = 0;
    if (inf_build<0>(S.lens, 19u, S.cnt_cl, S.sorted_cl, S.run, S.clt, 7u, max_cl) != 0 || max_cl == 0u) return ZWZ_STREAM_BAD;
    // code lengths for nlen + ndist symbols (warp-uniform decode, lane 0 stores)
    uint32_t have = 0, prev_len = 0;
    const uint32_t total = nlen + ndist;
    while (have < total) {
        infb_refill(B);
        const uint32_t e = S.clt[(uint32_t) B.hold & 127u];
        const uint32_t nb = e & 15u;
        if (nb == 0u) return ZWZ_STREAM_BAD; // invalid pattern is impossible for a complete code; defensive
        const uint32_t sym = e >> 4;
        const uint32_t eb = sym < 16u ? 0u : (sym == 16u ? 2u : (sym == 17u ? 3u : 7u));
        if (!infb_need(B, nb + eb)) return ZWZ_STREAM_TRUNCATED;
        infb_drop(B, nb);
        if (sym < 16u) {
            if (lane == 0) S.lens[32u + have] = (uint8_t) sym;
            prev_len = sym;
            have++;
            continue;
        }
        uint32_t rep, val = 0;
        const uint32_t x = (uint32_t) B.hold & ((1u << eb) - 1u);
        infb_drop(B, eb);
        if (sym == 16u) {
            if (have == 0u) return ZWZ_STREAM_BAD;
            val = prev_len;
            rep = 3u + x;
        } else {
            rep = (sym == 17u ? 3u : 11u) + x;
        }
        if (have + rep > total) return ZWZ_STREAM_BAD;
        // Rolled on purpose: unrolled (five predicated stores), inflate_span_kernel spills 36 / 52 bytes instead of 28 / 44 and
        // block_find_kernel needs 52 registers instead of 50.
#pragma unroll 1
        for (uint32_t r = lane; r < rep; r += 32u) S.lens[32u + have + r] = (uint8_t) val;
        prev_len = val;
        have += rep;
    }
    __syncwarp();
    if (S.lens[32u + 256u] == 0) return ZWZ_STREAM_BAD; // missing end-of-block code
    // S.lens[32 .. 32+nlen) literal/length, then ndist distance lengths. inf_build reads them in place; the two builds use
    // disjoint outputs, and the distance lengths are read before anything overwrites them.
    if (inf_build<1>(S.lens + 32, nlen, S.cnt_ll, S.sorted_ll, S.run, S.lit, ZWZ_INF_LBITS, max_ll) != 0 ||
        inf_build<2>(S.lens + 32 + nlen, ndist, S.cnt_d, S.sorted_d, S.run, S.dst, ZWZ_INF_DBITS, max_d) != 0)
        return ZWZ_STREAM_BAD;
    return ZWZ_STREAM_END;
}

// what inf_token decoded, besides ZWZ_STREAM_TRUNCATED / ZWZ_STREAM_BAD; apart from every stream status and span result, so
// that a token code passed on as a status by mistake cannot read as one
enum { INF_TOK_LIT = 16, INF_TOK_EOB = 17, INF_TOK_MATCH = 18 };

// One token of a Huffman block, from the literal/length entry `e` of the refilled reader's next bits. A code longer than the
// table index is resolved by the canonical walk. A token is consumed only when it lies completely inside the input (zlib: a
// literal needs its whole code, a match length + extra + distance + extra); an invalid code is BAD once its own bits are there.
// INF_TOK_LIT: the byte in v. INF_TOK_MATCH: length v and distance dist, which the caller checks against its window.
ZWZ_DEV uint32_t inf_token(const InflateWarpSmem &S, InfBits &B, uint32_t e, uint32_t max_ll, uint32_t max_d, uint32_t &v, uint32_t &dist) {
    uint32_t nb = e & 15u;
    if (ZWZ_LL_IS_LONG(e)) { // complete sets only get here
        uint32_t len = 0;
        const uint32_t sym = inf_canon_walk((uint32_t) B.hold, S.cnt_ll, S.sorted_ll, max_ll, len);
        e = sym == 0xffffffffu ? ZWZ_LL_INVALID(max_ll) : inf_litlen_entry(sym, len);
        nb = e & 15u;
    }
    if (ZWZ_LL_IS_INVALID(e)) return infb_need(B, nb) ? ZWZ_STREAM_BAD : ZWZ_STREAM_TRUNCATED; // zlib's invalid-code entry
    if (!infb_need(B, nb)) return ZWZ_STREAM_TRUNCATED;
    infb_drop(B, nb);
    if (ZWZ_LL_IS_LIT(e)) {
        v = e >> 7;
        return INF_TOK_LIT;
    }
    if (ZWZ_LL_IS_EOB(e)) return INF_TOK_EOB;
    // length (the code may have been the second one since the last refill: top up before the extra bits)
    infb_refill(B);
    const uint32_t eb = (e >> 4) & 7u;
    v = (e >> 7) - 253u + ((uint32_t) B.hold & ((1u << eb) - 1u));
    if (!infb_need(B, eb)) return ZWZ_STREAM_TRUNCATED;
    infb_drop(B, eb);
    infb_refill(B);
    uint32_t d = S.dst[(uint32_t) B.hold & ((1u << ZWZ_INF_DBITS) - 1u)];
    if (ZWZ_D_IS_LONG(d)) {
        uint32_t len = 0;
        const uint32_t sym = inf_canon_walk((uint32_t) B.hold, S.cnt_d, S.sorted_d, max_d, len);
        d = sym == 0xffffffffu ? ZWZ_D_INVALID(max_d) : inf_dist_entry(sym, len);
    }
    const uint32_t dnb = d & 15u;
    if (ZWZ_D_IS_SPECIAL(d)) return infb_need(B, dnb) ? ZWZ_STREAM_BAD : ZWZ_STREAM_TRUNCATED;
    const uint32_t deb = (d >> 4) & 15u;
    if (!infb_need(B, dnb + deb)) return ZWZ_STREAM_TRUNCATED;
    dist = ZWZ_D_DM1(d, (uint32_t) B.hold) + 1u;
    infb_drop(B, dnb + deb);
    return INF_TOK_MATCH;
}

// One warp decodes stream `sid`. DICT: the stream may have a preset dictionary, whose window (dwl bytes at dwin, 0 = none) comes
// before output position 0; a zlib stream asks for it with FDICT and names it by its DICTID (did), a raw stream just uses it.
template <bool DICT>
ZWZ_DEV void inflate_stream(InflateWarpSmem &S, const uint8_t *__restrict__ comp, uint32_t comp_len, uint8_t *out, uint32_t cap,
                            uint32_t flags, uint32_t &raw_len_out, uint32_t &status_out, const uint8_t *dwin, uint32_t dwl, uint32_t did) {
    const unsigned lane = lane_id();
    InfBits B;
    infb_open(B, comp, comp_len);
    infb_seek(B, 0);

    uint32_t pos = 0;       // bytes produced (counted past cap too)
    uint32_t pend_lo = 0;   // literals [pend_lo, pos) are parked in lanes (q & 31)
    uint32_t mybyte = 0;
    uint32_t status = ZWZ_STREAM_END;
    bool overflow = false;
    const uint32_t format = (flags >> 8) & 0xffu;

#define INF_FLUSH_LITS()                                                         \
    do {                                                                         \
        uint32_t q_ = (pend_lo & ~31u) + lane;                                   \
        if (q_ >= pend_lo && q_ < pos && q_ < cap) out[q_] = (uint8_t) mybyte;   \
        pend_lo = pos;                                                           \
    } while (0)

    if (format == ZWZ_FORMAT_GZIP) {
        const uint32_t h = inf_gzip_header(comp, comp_len);
        status = h & 3u;
        if (status != ZWZ_STREAM_END) goto done;
        infb_seek(B, h >> 2);
    } else if (format == ZWZ_FORMAT_ZLIB) {
        uint32_t flg = 0;
        status = inf_zlib_header(B, DICT && dwl != 0u, flg);
        if (status != ZWZ_STREAM_END) goto done;
        if (DICT) {
            if (flg & 0x20u) { // DICTID (inflate.c DICTID): it must name the dictionary given, else inflateSetDictionary's Z_DATA_ERROR
                infb_refill(B);
                if (!infb_need(B, 32)) {
                    status = ZWZ_STREAM_TRUNCATED;
                    goto done;
                }
                const uint32_t v = (uint32_t) B.hold;
                if ((((v & 0xffu) << 24) | ((v & 0xff00u) << 8) | ((v >> 8) & 0xff00u) | (v >> 24)) != did) {
                    status = ZWZ_STREAM_BAD;
                    goto done;
                }
                infb_drop(B, 32);
            } else {
                dwl = 0; // a zlib stream without FDICT ignores the dictionary (as CPython's decompressobj(zdict=) does)
            }
        }
    }

    for (;;) {
        infb_refill(B);
        if (!infb_need(B, 3)) {
            status = ZWZ_STREAM_TRUNCATED;
            goto done;
        }
        uint32_t last = (uint32_t) B.hold & 1u;
        uint32_t type = ((uint32_t) B.hold >> 1) & 3u;
        infb_drop(B, 3);

        if (type == 0u) {
            uint32_t bpos = 0, len = 0;
            status = inf_stored_header(B, bpos, len);
            if (status != ZWZ_STREAM_END) goto done;
            const uint32_t ncopy = len < comp_len - bpos ? len : comp_len - bpos;
            INF_FLUSH_LITS();
            {
                const uint32_t room = pos < cap ? cap - pos : 0u;
                inf_copy_plain(out + pos, comp + bpos, ncopy < room ? ncopy : room);
            }
            if (pos + ncopy > cap) overflow = true;
            pos += ncopy;
            pend_lo = pos;
            if (ncopy < len) {
                status = ZWZ_STREAM_TRUNCATED;
                goto done;
            }
            infb_seek(B, bpos + len);
            if (last) break;
            continue;
        }
        if (type == 3u) {
            status = ZWZ_STREAM_BAD;
            goto done;
        }

        uint32_t max_ll = 0, max_d = 0;
        uint32_t min_ll = 1; // shortest literal/length code of this block: bounds how many codes fit a 32-bit window
        if (type == 1u) {
            inf_fixed_tables(S, max_ll, max_d);
        } else {
            status = inf_dyn_tables(S, B, max_ll, max_d);
            if (status != ZWZ_STREAM_END) goto done;
        }

        for (min_ll = 1; min_ll < 15u && S.cnt_ll[min_ll] == 0u; ++min_ll) {}
        // ---- lane-parallel decode of the block (inflate_fast.cuh); the careful loop below only sees what it hands over:
        // the first token that does not lie completely inside the input, or an invalid code ----
        if (!(flags & ZWZ_INFLATE_CAREFUL)) {
            INF_FLUSH_LITS();
            __syncwarp();
            uint64_t bp = infb_used(B);
            const int fr = inf_fast_block<DICT>(S, B, bp, max_ll, max_d, out, cap, pos, overflow, dwin, dwl);
            pend_lo = pos;
            if (fr == IFR_BAD) {
                status = ZWZ_STREAM_BAD;
                goto done;
            }
            infb_seek_bits(B, bp);
            if (fr == IFR_EOB) {
                if (last) break;
                continue;
            }
        }
        // ---- symbol loop ----
        for (;;) {
            infb_refill(B); // >= 33 valid bits
            uint32_t e;
            if (infb_inside(B)) {
                // Literal runs, 32 bit offsets at a time ("warp-ballot symbol decode"): lane l decodes the code that WOULD
                // start at bit l of the buffer; the ballot says which offsets hold a complete literal; the offsets that
                // really are code starts form the chain 0 -> nb(0) -> ..., recovered with 5 rounds of pointer doubling on
                // (reach mask, jump) pairs. All literals on the chain are stored by their lanes in one go and the whole
                // run is dropped from the bit buffer at once. The chain ends at the first non-literal (handled below) or
                // past offset 31.
                const uint32_t el = S.lit[(uint32_t) (B.hold >> lane) & ((1u << ZWZ_INF_LBITS) - 1u)];
                const bool ok = (lane + 15u <= B.cnt) && ZWZ_LL_IS_LIT(el);
                const unsigned litmask = __ballot_sync(ZWZ_FULL, ok);
                if (litmask & 1u) {
                    uint32_t J = lane + (el & 15u);
                    uint32_t R = ok ? (1u << lane) : 0u;
                    // a window of 32 bits holds at most ceil(32 / min_ll) code starts and r doubling rounds reach 2^r of them:
                    // 2 rounds when no code is shorter than 8 bits (near-uniform bytes: the JPEG-like class), 3 down to 4 bits
#define INF_ROUND()                                                                  \
    do {                                                                             \
        const bool go = ok && J < 32u && ((litmask >> J) & 1u);                      \
        const int from = go ? (int) J : (int) lane;                                  \
        const uint32_t Rj = __shfl_sync(ZWZ_FULL, R, from);                          \
        const uint32_t Jj = __shfl_sync(ZWZ_FULL, J, from);                          \
        if (go) {                                                                    \
            R |= Rj;                                                                 \
            J = Jj;                                                                  \
        }                                                                            \
    } while (0)
                    INF_ROUND();
                    INF_ROUND();
                    if (min_ll < 8u) {
                        INF_ROUND();
                        if (min_ll < 4u) {
                            INF_ROUND();
                            if (min_ll < 2u) INF_ROUND();
                        }
                    }
#undef INF_ROUND
                    const uint32_t R0 = __shfl_sync(ZWZ_FULL, R, 0);
                    const uint32_t J0 = __shfl_sync(ZWZ_FULL, J, 0);
                    const uint32_t nlit = (uint32_t) __popc(R0);
                    if (pend_lo != pos) INF_FLUSH_LITS(); // only after a step of the scalar path
                    if ((R0 >> lane) & 1u) {
                        const uint32_t q = pos + (uint32_t) __popc(R0 & ((1u << lane) - 1u));
                        if (q < cap) out[q] = (uint8_t) (el >> 7);
                    }
                    if (pos + nlit > cap) overflow = true;
                    pos += nlit;
                    pend_lo = pos;
                    infb_drop(B, J0);
                    continue;
                }
                e = __shfl_sync(ZWZ_FULL, el, 0);
            } else {
                e = S.lit[(uint32_t) B.hold & ((1u << ZWZ_INF_LBITS) - 1u)];
            }
            uint32_t v = 0, dist = 0;
            const uint32_t t = inf_token(S, B, e, max_ll, max_d, v, dist);
            if (t == INF_TOK_LIT) {
                if (lane == (pos & 31u)) mybyte = v;
                pos++;
                if ((pos & 31u) == 0u) INF_FLUSH_LITS();
                continue;
            }
            if (t == INF_TOK_EOB) break;
            if (t != INF_TOK_MATCH) {
                status = t;
                goto done;
            }
            if (dist > pos + dwl) { // "invalid distance too far back" (a preset dictionary's window counts as written)
                status = ZWZ_STREAM_BAD;
                goto done;
            }
            // copy: everything before `pos` must be in memory first. Loads go through L2 (ld.global.cg): the bytes were
            // written by other lanes of this warp moments ago and L1 is not coherent for that.
            INF_FLUSH_LITS();
            __syncwarp();
            if (pos + v > cap) overflow = true;
            inf_copy_match<DICT>(out, pos, v, dist, cap, dwin, dwl);
            pos += v;
            pend_lo = pos;
        }
        if (last) break;
    }
    // ---- RFC 1950 trailer (inflate.c CHECK), RFC 1952 trailer (CHECK, LENGTH); raw streams have none ----
    if (format != ZWZ_FORMAT_RAW) {
        INF_FLUSH_LITS();
        __syncwarp();
        uint64_t used = infb_used(B);
        uint32_t bpos = (uint32_t) ((used + 7u) >> 3);
        if ((uint64_t) bpos + 4u > comp_len) {
            status = ZWZ_STREAM_TRUNCATED;
            goto done;
        }
        if (format == ZWZ_FORMAT_ZLIB) {
            if (!(flags & 1u) && !overflow) {
                const uint32_t have = inf_adler32(out, pos); // a = 1 + sum(byte), b = n + sum((n - j) * byte_j)  (mod 65521)
                if (have != inf_be32(comp + bpos)) status = ZWZ_STREAM_BAD;
            }
        } else {
            if (!(flags & 1u) && !overflow && inf_crc32(out, pos) != inf_le32(comp + bpos)) {
                status = ZWZ_STREAM_BAD;
            } else if ((uint64_t) bpos + 8u > comp_len) {
                status = ZWZ_STREAM_TRUNCATED;
            } else if (inf_le32(comp + bpos + 4u) != pos) { // ISIZE; pos counts past the capacity too
                status = ZWZ_STREAM_BAD;
            }
        }
    }
done:
    INF_FLUSH_LITS();
    __syncwarp();
    if (status == ZWZ_STREAM_END && overflow) status = ZWZ_STREAM_OUTPUT_FULL;
    raw_len_out = pos;
    status_out = status;
#undef INF_FLUSH_LITS
}

// Persistent warps: every warp pulls the next stream from a global counter, so a CTA is never kept alive by one long stream
// while its other warps idle (streams of one batch differ in length by 100x in config C2).
// DICT: some streams have a preset dictionary (dict, zwz_common.cuh); DICT = false is the kernel of the calls without.
template <bool DICT = false>
ZWZ_KERNEL __launch_bounds__(ZWZ_INF_WARPS * 32, ZWZ_INF_MIN_CTAS) inflate_kernel(const uint8_t *__restrict__ comp, const uint64_t *__restrict__ off,
                                                              const uint32_t *__restrict__ len, uint8_t *raw_out,
                                                              const uint64_t *__restrict__ raw_off, uint32_t *raw_len, uint32_t *status,
                                                              uint32_t n, uint32_t flags, uint32_t *work_counter, DictTable dict) {
    ZWZ_DYN_SMEM(inf_raw);
    InflateWarpSmem *smem = (InflateWarpSmem *) inf_raw;
    for (;;) {
        uint32_t sid = 0;
        if (lane_id() == 0) sid = atomicAdd(work_counter, 1u);
        sid = __shfl_sync(ZWZ_FULL, sid, 0);
        if (sid >= n) break;
        uint64_t cap64 = raw_off[sid + 1] - raw_off[sid];
        uint32_t cap = cap64 > 0xfffffff0ull ? 0xfffffff0u : (uint32_t) cap64;
        uint32_t rl = 0, st = 0;
        const uint8_t *dwin = nullptr;
        uint32_t dwl = 0, did = 0;
        if (DICT) {
            const uint32_t di = dict.idx[sid];
            if (di != ZWZ_NO_DICT) {
                dwin = dict.arena + (size_t) di * ZWZ_DICT_STRIDE + ZWZ_DICT_WIN;
                dwl = dict.wlen[di];
                did = dict.id[di];
            }
        }
        inflate_stream<DICT>(smem[warp_id()], comp + off[sid], len[sid], raw_out + raw_off[sid], cap, flags, rl, st, dwin, dwl, did);
        if (lane_id() == 0) {
            raw_len[sid] = rl;
            status[sid] = st;
        }
        __syncwarp();
    }
}

} // namespace zwz
