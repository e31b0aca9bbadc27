// inflate_seek.cuh — pieces of a long stream decoded from the access points of a seek index (zwz_index_extract*). An access
// point is a confirmed span start of zwz_inflate_stream (inflate_stream.cuh) whose 32 KiB window was resolved when the index was
// built, so a piece needs no block search, no confirmation and no u16 slots: one warp decodes it straight into bytes with the
// window as a preset dictionary, through the same steps as the batch decoder (inflate.cuh), lane-parallel blocks included.
#pragma once
#include "inflate_stream.cuh"

namespace zwz {

struct SeekJob {
    uint64_t bit;        // where decoding starts: a block header, a stored block's key, or a member header's first bit
    uint8_t *out;        // the piece's first `need` decoded bytes go to out[0 .. need)
    const uint8_t *win;  // the point's window: the wlen bytes right before it
    uint32_t wlen;
    uint32_t need;       // skip + want
    uint32_t mode;       // SPAN_MODE_*
    uint32_t bfinal;
};
struct SeekRes {
    uint64_t nout;       // bytes decoded from the point (counted past `need` up to where decoding stopped)
    uint32_t status;     // ZWZ_STREAM_END: stopped at the first block boundary at or past `need`, or where the stream ended
    uint32_t pad;
};

// One warp decodes one piece, from its point to the first block boundary at or past J.need. A gzip member that ends inside the
// piece is closed there: its trailer is skipped, the next header parsed, and the new member starts with an empty window; `out`
// and `pos` are re-based at the member start so that the shared block decoder runs unchanged.
ZWZ_DEV void seek_decode(InflateWarpSmem &S, const uint8_t *__restrict__ comp, uint64_t comp_len, const SeekJob &J, uint32_t format, uint32_t flags,
                         SeekRes &R) {
    const unsigned lane = lane_id();
    const bool at_header = J.mode == SPAN_MODE_FIRST || J.mode == SPAN_MODE_MEMBER;
    const uint64_t byte0 = J.bit >> 3;
    const uint32_t clen = (uint32_t) (comp_len - byte0); // bytes from byte0 on
    const uint8_t *c = comp + byte0;
    InfBits B;
    infb_open(B, c, clen);
    infb_seek_bits(B, J.bit & 7u);

    uint8_t *out = J.out;          // re-based at every member start inside the piece
    uint32_t cap = J.need;         // bytes of `out` that belong to the piece
    uint32_t pos = 0, pend_lo = 0, mybyte = 0;
    uint64_t before = 0;           // bytes decoded before `out`
    const uint8_t *dwin = J.win;
    uint32_t dwl = J.wlen;
    bool first = !at_header, overflow = false;
    uint32_t status = ZWZ_STREAM_END;
    uint32_t hp = 0; // member header position (bytes from byte0)

#define SEEK_FLUSH_LITS()                                                        \
    do {                                                                         \
        const uint32_t q_ = (pend_lo & ~31u) + lane;                             \
        if (q_ >= pend_lo && q_ < pos && q_ < cap) out[q_] = (uint8_t) mybyte;   \
        pend_lo = pos;                                                           \
    } while (0)

    if (at_header) goto header;
    for (;;) {
        infb_refill(B);
        if (before + pos >= J.need) goto done; // a block boundary at or past the end of the piece
        if (!infb_need(B, 3)) {
            status = ZWZ_STREAM_TRUNCATED;
            goto done;
        }
        {
            // a stored-mode point may sit in the padding behind the real header (RFC 1951 leaves padding bits arbitrary): BFINAL
            // comes from the point and the type from its mode, as in span_decode
            const uint32_t last = first ? J.bfinal : (uint32_t) B.hold & 1u;
            const uint32_t type = first && J.mode == SPAN_MODE_STORED ? 0u : ((uint32_t) B.hold >> 1) & 3u;
            first = false;
            infb_drop(B, 3);
            if (type == 0u) {
                uint32_t bpos = 0, len = 0;
                status = inf_stored_header(B, bpos, len);
                if (status != ZWZ_STREAM_END) goto done;
                const uint32_t ncopy = len < clen - bpos ? len : clen - bpos;
                SEEK_FLUSH_LITS();
                {
                    const uint32_t room = pos < cap ? cap - pos : 0u;
                    inf_copy_plain(out + pos, c + bpos, ncopy < room ? ncopy : room);
                }
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
            if (!(flags & ZWZ_INFLATE_CAREFUL)) {
                SEEK_FLUSH_LITS();
                __syncwarp();
                uint64_t bp = infb_used(B);
                const int fr = inf_fast_block<true>(S, B, bp, max_ll, max_d, out, cap, pos, overflow, dwin, dwl);
                pend_lo = pos;
                if (fr == IFR_BAD) {
                    status = ZWZ_STREAM_BAD;
                    goto done;
                }
                infb_seek_bits(B, bp);
                if (fr == IFR_EOB) {
                    if (last) goto member_end;
                    continue;
                }
            }
            for (;;) { // the careful symbol loop (all of a block with ZWZ_INFLATE_CAREFUL, else what the fast path handed over)
                infb_refill(B);
                uint32_t v = 0, dist = 0;
                const uint32_t t = inf_token(S, B, S.lit[(uint32_t) B.hold & ((1u << ZWZ_INF_LBITS) - 1u)], max_ll, max_d, v, dist);
                if (t == INF_TOK_LIT) {
                    if (lane == (pos & 31u)) mybyte = v;
                    pos++;
                    if ((pos & 31u) == 0u) SEEK_FLUSH_LITS();
                    continue;
                }
                if (t == INF_TOK_EOB) break;
                if (t != INF_TOK_MATCH) {
                    status = t;
                    goto done;
                }
                if (dist > pos + dwl) { // "invalid distance too far back": the window holds only what lies inside the member
                    status = ZWZ_STREAM_BAD;
                    goto done;
                }
                SEEK_FLUSH_LITS();
                __syncwarp();
                inf_copy_match<true>(out, pos, v, dist, cap, dwin, dwl);
                pos += v;
                pend_lo = pos;
            }
            if (!last) continue;
        }
    member_end:
        // the stream ends with the final block (zlib, raw) or with a gzip trailer that no member header follows
        if (format == ZWZ_FORMAT_RAW) goto done;
        {
            SEEK_FLUSH_LITS();
            const uint32_t bpos = (uint32_t) ((infb_used(B) + 7u) >> 3);
            if ((uint64_t) bpos + (format == ZWZ_FORMAT_ZLIB ? 4u : 8u) > clen) {
                status = ZWZ_STREAM_TRUNCATED;
                goto done;
            }
            if (format == ZWZ_FORMAT_ZLIB) goto done;
            hp = bpos + 8u;
            if (clen - hp < 2u || c[hp] != 0x1fu || c[hp + 1u] != 0x8bu) goto done;
        }
    header:
        if (format == ZWZ_FORMAT_GZIP) {
            const uint32_t h = inf_gzip_header(c + hp, clen - hp);
            if ((h & 3u) != ZWZ_STREAM_END) {
                status = h & 3u;
                goto done;
            }
            infb_seek(B, hp + (h >> 2));
        } else if (format == ZWZ_FORMAT_ZLIB) {
            uint32_t flg = 0;
            status = inf_zlib_header(B, false, flg);
            if (status != ZWZ_STREAM_END) goto done;
        }
        // a member starts here: nothing before it can be referred to
        SEEK_FLUSH_LITS();
        __syncwarp();
        {
            const uint32_t adv = pos < cap ? pos : cap;
            out += adv;
            cap -= adv;
        }
        before += pos;
        pos = 0;
        pend_lo = 0;
        dwin = nullptr;
        dwl = 0;
    }
done:
    SEEK_FLUSH_LITS();
    __syncwarp();
    if (lane == 0) {
        R.nout = before + pos;
        R.status = status;
        R.pad = 0;
    }
    __syncwarp();
#undef SEEK_FLUSH_LITS
}

// Persistent warps over the pieces of one call, longest decode first (the host sorts them).
ZWZ_KERNEL __launch_bounds__(ZWZ_INF_WARPS * 32, ZWZ_INF_MIN_CTAS) inflate_seek_kernel(const uint8_t *__restrict__ comp, uint64_t comp_len,
                                                                                     const SeekJob *__restrict__ jobs, SeekRes *res, uint32_t n,
                                                                                     uint32_t flags, uint32_t *work_counter) {
    ZWZ_DYN_SMEM(inf_raw);
    InflateWarpSmem *smem = (InflateWarpSmem *) inf_raw;
    const uint32_t format = (flags >> 8) & 0xffu;
    for (;;) {
        uint32_t j = 0;
        if (lane_id() == 0) j = atomicAdd(work_counter, 1u);
        j = __shfl_sync(ZWZ_FULL, j, 0);
        if (j >= n) break;
        const SeekJob J = jobs[j];
        seek_decode(smem[warp_id()], comp, comp_len, J, format, flags, res[j]);
    }
}

// The windows of the chosen access points, u16 window entries (win_scan_kernel's resolved windows) to bytes: point k's 32 768
// entries come from src[k] and go to dst + (k << 15). The entries that lie before the stream or before the member start
// (ZWZ_SPAN_INVALID) form a prefix; inv[k] = its length, so the window is the last 32 768 - inv[k] bytes.
ZWZ_KERNEL index_pack_kernel(const uint16_t *const *__restrict__ src, uint8_t *dst, uint32_t *inv) {
    const uint64_t t = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t k = (uint32_t) (t >> 15), e = (uint32_t) (t & (ZWZ_SPAN_WIN - 1u));
    const uint32_t v = src[k][e];
    dst[t] = (uint8_t) v;
    if (v == ZWZ_SPAN_INVALID) atomicMax(inv + k, e + 1u);
}

} // namespace zwz
