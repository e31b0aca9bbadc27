// inflate_stream.cuh — one long DEFLATE stream (gzip members, a zlib stream or raw DEFLATE) inflated by the whole GPU
// (zwz_inflate_stream*). The batch decoder of inflate.cuh gives every stream one warp; a stream written by gzip, pigz or
// zlib.compress is one long stream, so it gets cut here instead (the method of pugz / rapidgzip):
//
//   block_find_kernel    the compressed bytes are cut into spans; one warp per span finds the first bit offset inside it where a
//                        dynamic block header passes exactly the checks the decoder makes (inf_dyn_tables: precode, code
//                        lengths, both codes complete as inf_build requires, code 256 present), or where a stored block's
//                        LEN == ~NLEN sits behind a 3-bit BTYPE = 0 header. Fixed blocks cannot be found this way: almost any
//                        bit pattern is one, so a stream of fixed blocks only is decoded by one span;
//   inflate_span_kernel  one warp per span decodes from its start to the first block boundary at or after the next span's
//                        start, into a u16 slot: values < 256 are bytes, 256 + k is byte k of the 32 KiB window that precedes
//                        the span (not known yet). Gzip members that end inside a span are closed there (trailer recorded, the
//                        next member header parsed, the window reset: from then on "too far back" is tested exactly);
//   win_map_kernel,      each span's last 32 KiB is a map from its incoming window to its outgoing one (entries: a byte, a
//   win_scan_kernel      window index, or ZWZ_SPAN_INVALID for what lies before the stream or before a member start). Composing
//                        maps is a gather and associative: an inclusive scan over the spans (log2 N launches, double
//                        buffered, no CTA waits for another) gives every span its resolved incoming window;
//   stream_gather_kernel out[dst + i] = v < 256 ? v : window[v - 256]; the first position whose value resolves to INVALID is
//                        where zlib stops with "invalid distance too far back".
//
// One call may inflate many streams (zwz_inflate_stream_batch*): every job carries the byte base and length of its stream, and
// decodes exactly as it would in a call of its own. The first span of a stream starts at its header with an empty window, so its
// window map holds no window reference and the scan needs no segment flags between streams (DESIGN.md §4.10).
//
// The host (zwz_cuda.cu) confirms the spans: span 0 starts at the stream's first byte, span j is confirmed when the confirmed span
// j - 1 of the same stream stopped exactly at its start; a span behind a false candidate is decoded again from where its
// predecessor stopped.
#pragma once
#include "inflate.cuh"

namespace zwz {

#define ZWZ_SPAN_INVALID 0xffffu
#define ZWZ_SPAN_WIN 32768u
#define ZWZ_SPAN_MAXM 32u   // member trailers one span records; a span that meets more stops in front of the next member header

// BLOCK: at a block header; STORED: at a stored block's key (below), where the bits may be the header's padding, so the block
// type is known to be stored and is not read from them; FIRST / MEMBER: at the stream's (a following member's) header
enum { SPAN_MODE_BLOCK = 0, SPAN_MODE_FIRST = 1, SPAN_MODE_MEMBER = 2, SPAN_MODE_STORED = 3 };
// span results besides ZWZ_STREAM_END / TRUNCATED / BAD (which end the stream)
enum { SPAN_STOPPED = 4, SPAN_STOP_MEMBER = 5, SPAN_STOPPED_STORED = 6 }; // stopped at a block, a member header, a stored block
// SpanJob::mode flag: more input may follow the stream's last byte (zwz_inflater). Where the input runs out, the span reports the
// last point it passed where decoding can resume (a block key or a member header, its own start when it passed none) with the
// stop result and nout / nmem / reset as they were there, and sets SpanRes::more, instead of ZWZ_STREAM_TRUNCATED. Exact because
// a prefix that runs out is never ZWZ_STREAM_BAD: every other result stays what it is.
#define ZWZ_SPAN_PARTIAL 0x100u

// Where a span starts and stops is a block "key": the bit position of the block header, except for a stored block, whose key is
// the bit 3 in front of its LEN field (the header may sit anywhere in the padding before it, and decodes the same from there).
// Keys carry BFINAL in bit 0: key64 = key << 1 | BFINAL. The block finder marks a stored candidate with bit 63.
#define ZWZ_SPAN_CAND_STORED (1ull << 63)
ZWZ_DEV uint64_t span_block_key(uint64_t p, uint32_t hdr3) {
    const uint64_t k = ((hdr3 >> 1) & 3u) == 0u ? ((p + 10u) & ~(uint64_t) 7u) - 3u : p;
    return (k << 1) | (hdr3 & 1u);
}

struct SpanJob {
    uint64_t start;   // key64 of the first block (BLOCK), or byte position << 4 of the member header (FIRST, MEMBER)
    uint64_t target;  // stop at the first block whose key64 >> 1 is >= target >> 1; ~0 = run to the end of the stream
    uint16_t *slot;
    uint64_t cap;     // slot elements; the decoder counts past it
    uint64_t cbase;   // the stream's first byte in the compressed buffer; positions above are relative to it
    uint32_t mode;
    uint32_t clen;    // the stream's compressed bytes
};
struct SpanRes {
    uint64_t stop;    // SPAN_STOPPED: key64 it stopped at; SPAN_STOP_MEMBER: byte position << 4 of the next member header
    uint64_t nout;    // elements produced (counted past the slot's capacity too)
    uint64_t reset;   // position of the last member start inside the span (~0: none; 0 for FIRST / MEMBER spans)
    uint32_t status;
    uint32_t nmem;    // member trailers recorded
    uint32_t more;    // ZWZ_SPAN_PARTIAL: the input ran out, the fields above describe the last resume point passed
    uint32_t pad;
};
struct SpanMember {
    uint64_t end;     // output position (in the span) where the member ended
    uint32_t check;   // Adler-32 (zlib) or CRC-32 (gzip) from the trailer
    uint32_t isize;
    uint32_t have;    // bit 0: the check value was complete, bit 1: ISIZE was complete
    uint32_t pad;
};

// element s of the span's output, s < pos (s < 0: the unknown window, as 256 + its index)
ZWZ_DEV uint32_t span_src(const uint16_t *slot, uint64_t cap, int64_t s) {
    if (s < 0) return 256u + (uint32_t) (ZWZ_SPAN_WIN + s);
    return (uint64_t) s < cap ? (uint32_t) __ldcg(slot + s) : 0u;
}

// One warp decodes one span (the careful, warp-uniform decoder of inflate_stream, writing u16 elements).
ZWZ_DEV void span_decode(InflateWarpSmem &S, const uint8_t *__restrict__ comp_all, const SpanJob &J, uint32_t format, uint32_t flags,
                         SpanRes &R, SpanMember *mem) {
    const unsigned lane = lane_id();
    uint16_t *slot = J.slot;
    const uint64_t cap = J.cap;
    const uint32_t mode = J.mode & 3u;
    const bool partial = (J.mode & ZWZ_SPAN_PARTIAL) != 0u;
    const bool at_header = mode == SPAN_MODE_FIRST || mode == SPAN_MODE_MEMBER;
    const uint64_t bit0 = at_header ? (J.start >> 4) * 8u : J.start >> 1;
    const uint64_t byte0 = bit0 >> 3;
    const uint32_t clen = (uint32_t) (J.clen - byte0); // bytes from byte0 on
    const uint8_t *c = comp_all + J.cbase + byte0;
    InfBits B;
    infb_open(B, c, clen);
    infb_seek_bits(B, bit0 - byte0 * 8u);

    uint64_t pos = 0, pend_lo = 0, mstart = 0, reset = at_header ? 0u : ~(uint64_t) 0;
    bool first = !at_header;
    bool fresh = at_header; // a member started at or after the span's start: every back-reference must stay inside it
    uint32_t mybyte = 0, status = ZWZ_STREAM_END, nmem = 0;
    uint64_t stop = 0;
    uint32_t hp = 0; // member header position (bytes from byte0)
    // partial: lane 0 keeps the last resume point in R itself (no registers held across the decode loop); done leaves it there
    // when the input ran out
#define SPAN_RESUME_AT(stop_, status_)         \
    do {                                       \
        if (partial && lane == 0) {            \
            R.stop = (stop_);                  \
            R.status = (status_);              \
            R.nout = pos;                      \
            R.reset = reset;                   \
            R.nmem = nmem;                     \
        }                                      \
    } while (0)
    SPAN_RESUME_AT(J.start, mode == SPAN_MODE_BLOCK ? (uint32_t) SPAN_STOPPED : (mode == SPAN_MODE_STORED ? (uint32_t) SPAN_STOPPED_STORED : (uint32_t) SPAN_STOP_MEMBER));

#define SPAN_FLUSH_LITS()                                                          \
    do {                                                                           \
        const uint64_t q_ = (pend_lo & ~(uint64_t) 31u) + lane;                    \
        if (q_ >= pend_lo && q_ < pos && q_ < cap) slot[q_] = (uint16_t) mybyte;   \
        pend_lo = pos;                                                             \
    } while (0)

    if (at_header) goto header;
    for (;;) {
        { // block boundary: stop here when this block is at or past the next span's start
            infb_refill(B);
            if (!infb_need(B, 3)) {
                status = ZWZ_STREAM_TRUNCATED;
                goto done;
            }
            const uint64_t key = span_block_key(byte0 * 8u + infb_used(B), (uint32_t) B.hold & 7u);
            if ((key >> 1) >= (J.target >> 1)) {
                status = (((uint32_t) B.hold >> 1) & 3u) == 0u ? SPAN_STOPPED_STORED : SPAN_STOPPED;
                stop = key;
                goto done;
            }
            // the span's first block resumes from its own key and mode (a stored key's bits may be padding)
            if (!first) SPAN_RESUME_AT(key, (((uint32_t) B.hold >> 1) & 3u) == 0u ? (uint32_t) SPAN_STOPPED_STORED : (uint32_t) SPAN_STOPPED);
        }
        {
            // a span that starts at a stored block's key may sit in the padding behind the real header (RFC 1951 leaves padding
            // bits arbitrary): BFINAL comes from the key and the type from the mode
            const uint32_t last = first ? (uint32_t) (J.start & 1u) : (uint32_t) B.hold & 1u;
            const uint32_t type = first && mode == SPAN_MODE_STORED ? 0u : ((uint32_t) B.hold >> 1) & 3u;
            first = false;
            infb_drop(B, 3);
            if (type == 0u) {
                uint32_t bpos = 0, len = 0;
                status = inf_stored_header(B, bpos, len);
                if (status != ZWZ_STREAM_END) goto done;
                const uint32_t ncopy = len < clen - bpos ? len : clen - bpos;
                SPAN_FLUSH_LITS();
                for (uint32_t i = lane; i < ncopy; i += 32u)
                    if (pos + i < cap) slot[pos + i] = c[bpos + i];
                pos += ncopy;
                pend_lo = pos;
                if (ncopy < len) {
                    status = ZWZ_STREAM_TRUNCATED;
                    goto done;
                }
                infb_seek(B, bpos + len);
                if (last) goto member_end;
                continue;
            }
            if (type == 3u) {
                status = ZWZ_STREAM_BAD;
                goto done;
            }
            uint32_t max_ll = 0, max_d = 0;
            if (type == 1u) {
                inf_fixed_tables(S, max_ll, max_d);
            } else {
                status = inf_dyn_tables(S, B, max_ll, max_d);
                if (status != ZWZ_STREAM_END) goto done;
            }
            for (;;) { // symbol loop
                infb_refill(B);
                uint32_t v = 0, dist = 0;
                const uint32_t t = inf_token(S, B, S.lit[(uint32_t) B.hold & ((1u << ZWZ_INF_LBITS) - 1u)], max_ll, max_d, v, dist);
                if (t == INF_TOK_LIT) {
                    if (lane == (uint32_t) (pos & 31u)) mybyte = v;
                    pos++;
                    if ((pos & 31u) == 0u) SPAN_FLUSH_LITS();
                    continue;
                }
                if (t == INF_TOK_EOB) break;
                if (t != INF_TOK_MATCH) {
                    status = t;
                    goto done;
                }
                // "invalid distance too far back": exact once the member started in this span; before that the window is
                // not known here, and a reference that lands before the member start resolves to INVALID in the gather
                if (fresh && dist > pos - mstart) {
                    status = ZWZ_STREAM_BAD;
                    goto done;
                }
                SPAN_FLUSH_LITS();
                __syncwarp();
                // every source lies before pos: a run with period dist < v repeats the period already written
                const int64_t src0 = (int64_t) pos - (int64_t) dist;
                for (uint32_t i = lane; i < v; i += 32u) {
                    const uint64_t q = pos + i;
                    const uint32_t x = span_src(slot, cap, src0 + (int64_t) (i < dist ? i : i % dist));
                    if (q < cap) slot[q] = (uint16_t) x;
                }
                __syncwarp();
                pos += v;
                pend_lo = pos;
            }
            if (!last) continue;
        }
    member_end:
        // ---- trailers: RFC 1950 Adler-32, RFC 1952 CRC-32 + ISIZE; the check values themselves are compared on the host ----
        if (format == ZWZ_FORMAT_RAW) {
            status = ZWZ_STREAM_END;
            goto done;
        }
        {
            SPAN_FLUSH_LITS();
            const uint32_t bpos = (uint32_t) ((infb_used(B) + 7u) >> 3);
            const uint32_t tl = format == ZWZ_FORMAT_ZLIB ? 4u : 8u;
            uint32_t have = 0, check = 0, isize = 0;
            if ((uint64_t) bpos + 4u <= clen) {
                have = 1u;
                check = format == ZWZ_FORMAT_ZLIB ? inf_be32(c + bpos) : inf_le32(c + bpos);
            }
            if (format == ZWZ_FORMAT_GZIP && (uint64_t) bpos + 8u <= clen) {
                have |= 2u;
                isize = inf_le32(c + bpos + 4u);
            }
            if (lane == 0) {
                SpanMember m;
                m.end = pos;
                m.check = check;
                m.isize = isize;
                m.have = have;
                m.pad = 0;
                mem[nmem] = m;
            }
            nmem++;
            if ((uint64_t) bpos + tl > clen) {
                status = ZWZ_STREAM_TRUNCATED;
                goto done;
            }
            if (format == ZWZ_FORMAT_ZLIB) {
                status = ZWZ_STREAM_END;
                goto done;
            }
            // gzip: another member follows when the next two bytes are its magic; anything else behind a trailer is ignored.
            // Partial: fewer than two bytes do not tell yet, so decoding resumes at the header position.
            hp = bpos + 8u;
            SPAN_RESUME_AT((byte0 + hp) << 4, (uint32_t) SPAN_STOP_MEMBER);
            if (partial && clen - hp < 2u) {
                status = ZWZ_STREAM_TRUNCATED;
                goto done;
            }
            if (clen - hp < 2u || c[hp] != 0x1fu || c[hp + 1u] != 0x8bu) {
                status = ZWZ_STREAM_END;
                goto done;
            }
            if (nmem == ZWZ_SPAN_MAXM) {
                status = SPAN_STOP_MEMBER;
                stop = (byte0 + hp) << 4;
                goto done;
            }
        }
    header:
        if (format == ZWZ_FORMAT_GZIP) {
            if (mode == SPAN_MODE_MEMBER && nmem == 0u && (clen < 2u || c[0] != 0x1fu || c[1] != 0x8bu)) {
                status = partial && clen < 2u ? ZWZ_STREAM_TRUNCATED : ZWZ_STREAM_END;
                goto done;
            }
            const uint32_t h = inf_gzip_header(c + hp, clen - hp);
            if ((h & 3u) != ZWZ_STREAM_END) {
                status = h & 3u;
                goto done;
            }
            infb_seek(B, hp + (h >> 2));
        } else if (format == ZWZ_FORMAT_ZLIB) {
            uint32_t flg = 0;
            status = inf_zlib_header(B, false, flg); // this call takes no dictionary
            if (status != ZWZ_STREAM_END) goto done;
        }
        fresh = true;
        mstart = pos;
        reset = pos;
    }
done:
    SPAN_FLUSH_LITS();
    __syncwarp();
    if (lane == 0) {
        const bool more = partial && status == ZWZ_STREAM_TRUNCATED;
        if (!more) {
            R.stop = stop;
            R.nout = pos;
            R.reset = reset;
            R.status = status;
            R.nmem = nmem;
        }
        R.more = more ? 1u : 0u;
    }
    __syncwarp();
#undef SPAN_RESUME_AT
#undef SPAN_FLUSH_LITS
}

// Persistent warps over the span jobs of one round (spans differ in output length by orders of magnitude).
ZWZ_KERNEL __launch_bounds__(ZWZ_INF_WARPS * 32, ZWZ_INF_MIN_CTAS) inflate_span_kernel(const uint8_t *__restrict__ comp, const SpanJob *__restrict__ jobs,
                                                                                     SpanRes *res, SpanMember *mem, uint32_t n, uint32_t flags,
                                                                                     uint32_t *work_counter) {
    ZWZ_DYN_SMEM(inf_raw);
    InflateWarpSmem *smem = (InflateWarpSmem *) inf_raw;
    const uint32_t format = (flags >> 8) & 0xffu;
    for (;;) {
        uint32_t j = 0;
        if (lane_id() == 0) j = atomicAdd(work_counter, 1u);
        j = __shfl_sync(ZWZ_FULL, j, 0);
        if (j >= n) break;
        const SpanJob J = jobs[j];
        span_decode(smem[warp_id()], comp, J, format, flags, res[j], mem + (size_t) j * ZWZ_SPAN_MAXM);
    }
}

// 64 stream bits from bit p on (bytes past the end read as 0)
ZWZ_DEV uint64_t bf_peek64(const uint8_t *comp, uint64_t comp_len, uint64_t p) {
    const uint32_t skew = (uint32_t) ((uintptr_t) comp & 3u);
    const uint32_t *wb = (const uint32_t *) (comp - skew);
    const uint64_t a = (uint64_t) skew * 8u + p, end = skew + comp_len;
    const uint64_t k = a >> 5;
    uint32_t w[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const uint64_t wi = k + (uint64_t) i;
        uint32_t v = wi * 4u < end ? __ldg(wb + wi) : 0u;
        if (wi * 4u < end && wi * 4u + 4u > end) v &= (1u << ((uint32_t) (end - wi * 4u) * 8u)) - 1u;
        w[i] = v;
    }
    const uint32_t s = (uint32_t) (a & 31u);
    const uint64_t lo = (uint64_t) w[0] | ((uint64_t) w[1] << 32);
    return s ? (lo >> s) | ((uint64_t) w[2] << (64u - s)) : lo;
}

// span j >= 1 of the stream comp[base .. base + len)
struct FindJob {
    uint64_t base;
    uint32_t len, span;
};

// One warp per job: cand[job] = key64 (relative to its stream) of the first block header candidate inside bytes [j * S, (j + 1) * S)
// of its stream, or ~0. Nothing past the stream's end is read, so a candidate is a header the decoder accepts there too.
// 32 bit offsets per step, one per lane: the cheap tests (BTYPE, HLIT / HDIST, the precode's Kraft sum; a stored block's
// LEN == ~NLEN) run on every lane, the few survivors get the full table check by the whole warp, in bit order.
ZWZ_KERNEL __launch_bounds__(32) block_find_kernel(const uint8_t *__restrict__ comp_all, const FindJob *__restrict__ jobs, uint64_t span_bytes,
                                                   uint64_t *cand, uint32_t n) {
    ZWZ_DYN_SMEM(inf_raw);
    InflateWarpSmem &S = *(InflateWarpSmem *) inf_raw;
    const unsigned lane = lane_id();
    if (blockIdx.x >= n) return;
    const FindJob fj = jobs[blockIdx.x];
    const uint8_t *comp = comp_all + fj.base;
    const uint64_t comp_len = fj.len;
    const uint32_t j = fj.span;
    const uint64_t lo = (uint64_t) j * span_bytes * 8u;
    const uint64_t hi_byte = (uint64_t) (j + 1u) * span_bytes;
    const uint64_t hi = (hi_byte < comp_len ? hi_byte : comp_len) * 8u;
    for (uint64_t b0 = lo; b0 < hi; b0 += 32u) {
        const uint64_t p = b0 + lane;
        bool dyn = false, sto = false;
        uint64_t v = 0;
        if (p < hi) {
            v = bf_peek64(comp, comp_len, p);
            const uint32_t bt = ((uint32_t) v >> 1) & 3u;
            if (bt == 2u && ((v >> 3) & 31u) <= 29u && ((v >> 8) & 31u) <= 29u) {
                const uint32_t ncode = (uint32_t) ((v >> 13) & 15u) + 4u;
                const uint64_t pc = bf_peek64(comp, comp_len, p + 17u);
                uint32_t kraft = 0;
                for (uint32_t i = 0; i < ncode; ++i) {
                    const uint32_t l = (uint32_t) (pc >> (3u * i)) & 7u;
                    if (l) kraft += 128u >> l;
                }
                dyn = kraft == 128u; // the code-length code must be complete
            } else if (bt == 0u && ((p + 3u) & 7u) == 0u && ((p + 3u) >> 3) + 4u <= comp_len) {
                const uint32_t w = (uint32_t) (v >> 3);
                sto = (w & 0xffffu) == ((w >> 16) ^ 0xffffu);
            }
        }
        unsigned m = __ballot_sync(ZWZ_FULL, dyn || sto);
        while (m) {
            const int l = __ffs((int) m) - 1;
            m &= m - 1u;
            const uint64_t pp = b0 + (uint64_t) l;
            const bool is_sto = __shfl_sync(ZWZ_FULL, sto ? 1u : 0u, l) != 0u;
            bool ok = is_sto;
            if (!is_sto) {
                InfBits B;
                infb_open(B, comp + (pp >> 3), (uint32_t) (comp_len - (pp >> 3)));
                infb_seek_bits(B, pp & 7u);
                infb_drop(B, 3);
                infb_refill(B);
                uint32_t mll = 0, md = 0;
                ok = inf_dyn_tables(S, B, mll, md) == ZWZ_STREAM_END;
            }
            if (ok) {
                const uint32_t bfinal = __shfl_sync(ZWZ_FULL, (uint32_t) v & 1u, l);
                if (lane == 0) cand[blockIdx.x] = (pp << 1) | bfinal | (is_sto ? ZWZ_SPAN_CAND_STORED : 0ull);
                return;
            }
        }
    }
    if (lane == 0) cand[blockIdx.x] = ~(uint64_t) 0;
}

// ---- window resolution and gather ----
struct SpanWin {
    const uint16_t *slot;
    uint64_t nout;
    uint64_t reset; // ~0: no member starts inside the span
    uint64_t base;  // output position of its first element in its stream's part of the wave
    uint64_t dst;   // where that element goes in the gather's output
    const uint16_t *win; // the resolved window in front of the span (nullptr: none, the span starts its stream)
    uint32_t sid, pad;   // the stream's index in the wave (its first_bad entry)
};

// map[i][k] (i < m): what the k-th byte of the window behind span sp[i] is, in terms of the window in front of it (sp: the spans of
// the wave whose outgoing window a later span reads, in order)
// win_in: the resolved window in front of sp[0] when it goes on from the previous wave, nullptr = nothing comes before it
ZWZ_KERNEL win_map_kernel(const SpanWin *__restrict__ sp, const uint16_t *__restrict__ win_in, uint16_t *map, uint32_t m) {
    const uint64_t t = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t i = (uint32_t) (t >> 15), k = (uint32_t) (t & (ZWZ_SPAN_WIN - 1u));
    if (i >= m) return;
    const SpanWin s = sp[i];
    const int64_t p = (int64_t) s.nout - (int64_t) ZWZ_SPAN_WIN + (int64_t) k;
    uint32_t v;
    if (s.reset != ~(uint64_t) 0 && p < (int64_t) s.reset) v = ZWZ_SPAN_INVALID; // before a member start: nothing was written there
    else if (p >= 0) v = s.slot[p];
    else v = 256u + (uint32_t) (s.nout + k);
    if (i == 0 && v >= 256u && v != ZWZ_SPAN_INVALID) v = win_in ? win_in[v - 256u] : ZWZ_SPAN_INVALID;
    map[t] = (uint16_t) v;
}

// one step of the inclusive scan: nxt[i] = cur[i] o cur[i - d]
ZWZ_KERNEL win_scan_kernel(const uint16_t *__restrict__ cur, uint16_t *nxt, uint32_t m, uint32_t d) {
    const uint64_t t = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t i = (uint32_t) (t >> 15);
    if (i >= m) return;
    uint32_t v = cur[t];
    if (i >= d && v >= 256u && v != ZWZ_SPAN_INVALID) v = cur[((uint64_t) (i - d) << 15) | (v - 256u)];
    nxt[t] = (uint16_t) v;
}

#define ZWZ_GATHER_TILE 65536u
// one CTA per tile of ZWZ_GATHER_TILE elements of one span; first_bad: one entry per stream of the wave
ZWZ_KERNEL stream_gather_kernel(const SpanWin *__restrict__ sp, const uint64_t *__restrict__ tiles, uint8_t *out, unsigned long long *first_bad) {
    const uint64_t tl = tiles[blockIdx.x];
    const uint32_t i = (uint32_t) (tl >> 40);
    const uint64_t e0 = tl & ((1ull << 40) - 1u);
    const SpanWin s = sp[i];
    const uint64_t e1 = e0 + ZWZ_GATHER_TILE < s.nout ? e0 + ZWZ_GATHER_TILE : s.nout;
    for (uint64_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
        uint32_t v = s.slot[e];
        if (v >= 256u && v != ZWZ_SPAN_INVALID) v = s.win ? s.win[v - 256u] : ZWZ_SPAN_INVALID;
        if (v == ZWZ_SPAN_INVALID) atomicMin(first_bad + s.sid, (unsigned long long) (s.base + e));
        else out[s.dst + e] = (uint8_t) v;
    }
}

} // namespace zwz
