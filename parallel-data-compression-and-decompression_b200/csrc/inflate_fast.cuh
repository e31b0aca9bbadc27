// inflate_fast.cuh — lane-parallel Huffman decode of one DEFLATE block + warp-parallel LZ77 resolve (used by inflate.cuh).
//
// The careful decoder in inflate.cuh computes every symbol redundantly in all 32 lanes (~22 warp-instructions per output
// byte, profiles/round1/ncu_inflate.txt). This path spends the lanes on DIFFERENT symbols of the same block:
//
//   window   the next 32 x 416 bits of the block are staged into shared memory (14 coalesced loads);
//   decode   lane i decodes the tokens that start in ITS 416 bits, from a speculative start (the first bit of its range),
//            into its own token region in shared memory. Lane 0 starts at a known token boundary, so its result — and the
//            position where it crosses into lane 1's range — is exact. Lanes whose start disagrees with where their
//            predecessor ended decode again from there; every round proves at least one more lane, and since Huffman
//            streams re-synchronise after a few symbols, two or three rounds usually prove all 32. Same tables for all
//            lanes (one block), so the table memory is that of ONE decoder and every lane runs the same loop;
//   resolve  the proven token regions are replayed in order, 32 tokens per step: output offsets by a warp prefix sum,
//            all literals of the step stored at once, each match copied by the whole warp.
//
// Exactness: the fast path only ever commits tokens that lie completely inside the input and are valid; at the first token
// that is not (truncated stream, invalid code) it stops AT that token's first bit and the careful decoder takes over from
// there, so the bytes and the status are zlib's in every case (oracle/zwz_oracle.c states the rules). A distance that
// reaches before the start of the output is found here, at the same point where zlib finds it.
#pragma once
#include "zwz_common.cuh"

namespace zwz {

// ZWZ_IF_SW (words of compressed data per lane and window), ZWZ_IF_CW (staged words) and ZWZ_IF_R / ZWZ_IF_RS (token
// region size and stride) are defined with the shared-memory layout in inflate.cuh
#define ZWZ_IF_SBITS (ZWZ_IF_SW * 32u)         // bits per lane and window: longer than any token (48 bits)
#define ZWZ_IF_MAXIT 6                         // rounds per window; then the proven prefix is committed and a new window starts
#ifndef ZWZ_IF_MLP
#define ZWZ_IF_MLP 4u                           // 32-byte rows of a resolve step whose back-reference loads are in flight together
#endif
#define ZWZ_IF_STG (ZWZ_IF_CW * 4u > 1536u ? 1536u : ZWZ_IF_CW * 4u) // output bytes assembled per resolve step (lives in the staged-window area)

#ifdef ZWZ_EMU
// test-only counters of the emulator build: [0] windows, [1] decode rounds, [2] committed lanes, [3] token entries,
// [4] hand-overs to the careful decoder, [5] windows cut by ZWZ_IF_MAXIT, [6] windows cut by a full token region
static uint64_t g_if_stats[8];
extern "C" void zwz_emu_inflate_stats(uint64_t *out, int reset) {
    for (int i = 0; i < 8; ++i) {
        out[i] = g_if_stats[i];
        if (reset) g_if_stats[i] = 0;
    }
}
#define ZWZ_IF_STAT(i, v) do { if (lane_id() == 0) g_if_stats[i] += (v); } while (0)
#else
#define ZWZ_IF_STAT(i, v) do { } while (0)
#endif

enum { IFL_RUN = 0, IFL_EOB = 1, IFL_FULL = 2, IFL_STOP = 3 };
enum { IFR_SLOW = 0, IFR_EOB = 1, IFR_BAD = 2 };

// 32 bits of the staged window starting at bit p
ZWZ_DEV uint32_t iff_fetch(const uint32_t *cw, uint32_t p) {
    const uint32_t k = p >> 5;
    return __funnelshift_r(cw[k], cw[k + 1u], p & 31u);
}

// The byte at output position s - d of a stream. DICT: a stream with a preset dictionary (window of dwl bytes at dwin) finds the
// bytes before its output position 0 in the dictionary's window, as if they had been written right before it.
template <bool DICT> ZWZ_DEV uint32_t inf_ref(const uint8_t *out, const uint8_t *dwin, uint32_t dwl, uint32_t s, uint32_t d) {
    if (DICT && s < d) return __ldg(dwin + (dwl + s - d));
    return __ldcg(out + (s - d));
}

// back-reference copy by the whole warp: bytes [pos, pos + mlen) = bytes [pos - dist, ...), overlapping allowed (also across
// the boundary between a preset dictionary's window and the output)
template <bool DICT = false>
ZWZ_DEV void inf_copy_match(uint8_t *out, uint32_t pos, uint32_t mlen, uint32_t dist, uint32_t cap, const uint8_t *dwin = nullptr, uint32_t dwl = 0u) {
    const unsigned lane = lane_id();
    if (mlen <= 32u && dist >= mlen) { // the common case: short, non-overlapping — one step, no loop
        const uint32_t q = pos + lane;
        if (lane < mlen && q < cap) out[q] = inf_ref<DICT>(out, dwin, dwl, q, dist);
    } else if (dist >= 32u || dist >= mlen) {
        for (uint32_t base = 0; base < mlen; base += 32u) { // warp-uniform trip count
            const uint32_t q = pos + base + lane;
            if (base + lane < mlen && q < cap) out[q] = inf_ref<DICT>(out, dwin, dwl, q, dist);
            __syncwarp(); // later steps may read what this step wrote (dist < mlen)
        }
    } else { // overlapping run with a period < 32: every byte comes from the already written period
        for (uint32_t i = lane; i < mlen; i += 32u) {
            const uint32_t q = pos + i;
            if (q < cap) out[q] = inf_ref<DICT>(out, dwin, dwl, pos + (i % dist), dist);
        }
    }
    __syncwarp();
}

// Decodes the Huffman block whose next literal/length code starts at stream bit `bitpos`, as far as the fast path can.
// Returns IFR_EOB (end-of-block consumed, bitpos behind it), IFR_SLOW (bitpos = first bit of a token the careful decoder
// must look at) or IFR_BAD (distance too far back: pos = bytes before that match). All arguments and results are
// warp-uniform. DICT: the dwl bytes of a preset dictionary's window at dwin come before output position 0.
template <bool DICT, class SMEM, class BITS>
ZWZ_DEV int inf_fast_block(SMEM &S, const BITS &B, uint64_t &bitpos, uint32_t max_ll, uint32_t max_d, uint8_t *out, uint32_t cap, uint32_t &pos,
                           bool &overflow, const uint8_t *dwin, uint32_t dwl) {
    const unsigned lane = lane_id();
    const uint64_t g_end = (uint64_t) B.skew * 8u + (uint64_t) B.nbytes * 8u; // one past the last real bit, relative to wbase
    uint16_t *const my = S.tok + lane * ZWZ_IF_RS;
    for (;;) {
        // ---- window ----
        const uint64_t g = (uint64_t) B.skew * 8u + bitpos;
        const uint32_t w0 = (uint32_t) (g >> 5);
        const uint32_t base_bit = (uint32_t) g & 31u;
        const uint64_t lim64 = g_end - (uint64_t) w0 * 32u;
        const uint32_t limit = lim64 > 0x7fffffffull ? 0x7fffffffu : (uint32_t) lim64; // real bits in the window (tokens must end <= limit)
        __syncwarp();
        for (uint32_t k = lane; k < ZWZ_IF_CW; k += 32u) S.cw[k] = infb_load(B, w0 + k);
        __syncwarp();

        // ---- decode: rounds until the lanes agree ----
        // The token loop is ONE instruction stream for all lanes (warp-uniform trip count, literal and match handled by the same
        // straight-line code with selects): a loop in which every lane branches on its own symbol kind lets the lanes drift apart
        // and the warp then executes each lane's iterations separately (measured: 5x the instructions).
        const uint32_t hi = base_bit + (lane + 1u) * ZWZ_IF_SBITS;
        uint32_t start = base_bit + lane * ZWZ_IF_SBITS;
        uint32_t e = 0, ntok = 0, flag = IFL_RUN;
        bool need = true;
        uint32_t ncommit = 0;
        for (int it = 0;; ++it) {
            uint32_t p = start;
            bool run = need;
            if (need) {
                ntok = 0;
                flag = IFL_RUN;
            }
            while (__any_sync(ZWZ_FULL, run)) {
                ZWZ_IF_STAT(7, 1);
                if (run) {
                    const uint32_t bits = iff_fetch(S.cw, p);
                    uint32_t en = S.lit[bits & ((1u << ZWZ_INF_LBITS) - 1u)];
                    if (ZWZ_LL_IS_LONG(en)) { // code longer than the table index (rare)
                        uint32_t len = 0;
                        const uint32_t sym = inf_canon_walk(bits, S.cnt_ll, S.sorted_ll, max_ll, len);
                        en = sym == 0xffffffffu ? ZWZ_LL_INVALID(max_ll) : inf_litlen_entry(sym, len);
                    }
                    const bool is_len = ZWZ_LL_IS_LEN(en);
                    const bool special = ((en >> 4) & 7u) == 7u; // end-of-block or invalid code
                    const uint32_t nb = en & 15u, eb = is_len ? (en >> 4) & 7u : 0u;
                    const uint32_t val = (en >> 7) + ((bits >> nb) & ((1u << eb) - 1u)); // literal byte, or 253 + match length
                    const uint32_t p2 = p + nb + eb;
                    // the distance code behind a length code; decoded for every lane, used by the lanes that hold a length
                    const uint32_t bits2 = iff_fetch(S.cw, p2);
                    uint32_t d = S.dst[bits2 & ((1u << ZWZ_INF_DBITS) - 1u)];
                    if (is_len && ZWZ_D_IS_LONG(d)) {
                        uint32_t len = 0;
                        const uint32_t sym = inf_canon_walk(bits2, S.cnt_d, S.sorted_d, max_d, len);
                        d = sym == 0xffffffffu ? ZWZ_D_INVALID(max_d) : inf_dist_entry(sym, len);
                    }
                    const uint32_t dnb = d & 15u, deb = (d >> 4) & 15u;
                    const uint32_t dm1 = ZWZ_D_DM1(d, bits2);
                    const uint32_t pn = is_len ? p2 + dnb + deb : p2;
                    const bool bad = (special && (en >> 7) != 0u) || (is_len && ZWZ_D_IS_SPECIAL(d)) || pn > limit;
                    if (bad) { // invalid code, or a token that does not lie completely inside the input: the careful decoder's business
                        flag = IFL_STOP;
                        run = false;
                    } else if (special) { // end-of-block
                        p = pn;
                        flag = IFL_EOB;
                        run = false;
                    } else {
                        my[ntok] = (uint16_t) (is_len ? (0x8000u - 253u) + val : val);
                        if (is_len) my[ntok + 1u] = (uint16_t) dm1;
                        ntok += is_len ? 2u : 1u;
                        p = pn;
                        if (p >= hi) {
                            run = false;
                        } else if (ntok + 2u > ZWZ_IF_R) {
                            flag = IFL_FULL;
                            run = false;
                        }
                    }
                }
            }
            if (need) e = p;
            __syncwarp();
            const uint32_t pe = __shfl_up_sync(ZWZ_FULL, e, 1);
            const uint32_t pf = __shfl_up_sync(ZWZ_FULL, flag, 1);
            const bool ok = lane == 0u || (pf == IFL_RUN && pe == start);
            const unsigned okm = __ballot_sync(ZWZ_FULL, ok);
            const unsigned termm = __ballot_sync(ZWZ_FULL, flag != IFL_RUN);
            const uint32_t c = okm == ZWZ_FULL ? 32u : (uint32_t) __ffs((int) ~okm) - 1u;   // lanes [0, c) are proven
            const uint32_t ft = termm ? (uint32_t) __ffs((int) termm) - 1u : 32u;          // first lane that stopped early
            ZWZ_IF_STAT(1, 1);
            if (ft < c) { // the chain of proven lanes ends inside the window
                ncommit = ft + 1u;
                break;
            }
            if (c == 32u || it + 1 >= ZWZ_IF_MAXIT) {
                ncommit = c;
                ZWZ_IF_STAT(5, c != 32u);
                break;
            }
            need = lane >= c && !ok && pf == IFL_RUN;
            if (need) start = pe;
        }

        // ---- resolve: replay the proven regions in order, <= 32 token entries per step ----
        // Output of a step is assembled in shared memory (the staged window is dead by now) and then written out in one go.
        // Every output byte of the step is produced by its own lane: the token that covers it is found by a binary search over
        // the step's running lengths, bytes whose source lies before the step come from global memory — all loads of the step
        // are independent, so their latency overlaps — and only matches that reach into the step's own output wait for it.
        ZWZ_IF_STAT(0, 1);
        ZWZ_IF_STAT(2, ncommit);
        const uint32_t last_flag = __shfl_sync(ZWZ_FULL, flag, (int) (ncommit - 1u));
        const uint32_t last_e = __shfl_sync(ZWZ_FULL, e, (int) (ncommit - 1u));
        uint8_t *const stg = (uint8_t *) S.cw;
        for (uint32_t l = 0; l < ncommit; ++l) {
            const uint32_t nl = __shfl_sync(ZWZ_FULL, ntok, (int) l);
            ZWZ_IF_STAT(3, nl);
            const uint16_t *reg = S.tok + l * ZWZ_IF_RS;
            uint32_t j0 = 0;
            while (j0 < nl) {
                const uint32_t idx = j0 + lane;
                uint32_t t = idx < nl ? (uint32_t) reg[idx] : 0u;
                unsigned hm = __ballot_sync(ZWZ_FULL, (t & 0x8000u) != 0u);
                uint32_t take = nl - j0 < 32u ? nl - j0 : 32u;
                if (hm >> 31) { // a match head in the last lane: its distance entry belongs to the next step
                    take = 31u;
                    hm &= 0x7fffffffu;
                    if (lane == 31u) t = 0u;
                }
                if (hm == 0u) { // literals only
                    const uint32_t q = pos + lane;
                    if (lane < take && q < cap) out[q] = (uint8_t) t;
                    if (pos + take > cap) overflow = true;
                    pos += take;
                    j0 += take;
                    continue;
                }
                const bool is_head = (hm >> lane) & 1u;
                const bool is_dist = lane > 0u && ((hm >> (lane - 1u)) & 1u);
                uint32_t olen = lane >= take || is_dist ? 0u : (is_head ? (t & 0x1ffu) : 1u);
                uint32_t incl = warp_incl_scan(olen);
                // a step's output must fit the staging area: cut behind the last entry that still does
                const unsigned fits = __ballot_sync(ZWZ_FULL, incl <= ZWZ_IF_STG);
                if (fits != ZWZ_FULL) {
                    take = (uint32_t) __ffs((int) ~fits) - 1u; // >= 3: a token is at most 258 bytes
                    if (lane >= take) olen = 0u;
                    hm &= (1u << take) - 1u;
                    incl = warp_incl_scan(olen);
                }
                const uint32_t excl = incl - olen;
                const uint32_t total = __shfl_sync(ZWZ_FULL, incl, 31);
                const uint32_t dn = __shfl_down_sync(ZWZ_FULL, t, 1); // distance - 1 of a head lane
                // invalid distance too far back: zlib stops at the first such match with everything before it written
                const unsigned far = __ballot_sync(ZWZ_FULL, is_head && lane < take && dn + 1u > pos + excl + dwl);
                // matches that reach into this step's own output (source position + min(len, dist) > step start)
                const unsigned deps = __ballot_sync(ZWZ_FULL, is_head && lane < take && excl + (olen < dn + 1u ? olen : dn + 1u) > dn + 1u);
                // ---- every byte of the step by its own lane ----
                // ZWZ_IF_MLP rows of 32 bytes at a time: the rows' back-reference loads (L2, ~600 cycles each) are all issued before
                // the first value is stored, so a warp has ZWZ_IF_MLP loads in flight instead of one (long_scoreboard at the load
                // was 26 % of all stall samples on text, profiles/round2_notes.md).
                for (uint32_t b0 = 0; b0 < total; b0 += 32u * ZWZ_IF_MLP) {
                    uint32_t val[ZWZ_IF_MLP];
                    bool put[ZWZ_IF_MLP];
#pragma unroll
                    for (uint32_t u = 0; u < ZWZ_IF_MLP; ++u) {
                        const uint32_t b = b0 + 32u * u + lane;
                        val[u] = 0;
                        put[u] = false;
                        if (b0 + 32u * u >= total) continue; // warp-uniform: a short step does not pay for empty rows
                        uint32_t j = 0;
#pragma unroll
                        for (uint32_t sft = 16u; sft != 0u; sft >>= 1) {
                            const uint32_t v = __shfl_sync(ZWZ_FULL, incl, (int) (j + sft - 1u));
                            if (v <= b) j += sft;
                        }
                        j &= 31u; // lanes past `total` search past the end
                        const uint32_t tj = __shfl_sync(ZWZ_FULL, t, (int) j);
                        const uint32_t ej = __shfl_sync(ZWZ_FULL, excl, (int) j);
                        const uint32_t dj = __shfl_sync(ZWZ_FULL, dn, (int) j) + 1u;
                        val[u] = tj;
                        put[u] = b < total;
                        if (b < total && ((hm >> j) & 1u)) {
                            const uint32_t i = b - ej;                                                // byte i of the match
                            const uint32_t src = ej + (dj >= (tj & 0x1ffu) || i < dj ? i : i % dj);   // its source + dist, relative to the step
                            // before the step iff src < dj. No load for bytes that will not be written: those of a too-far match
                            // (dj > pos + ej + dwl) and those past the capacity of the output window (a sizing pass still counts them)
                            put[u] = src < dj && dj <= pos + ej + dwl && pos + b < cap;
                            if (put[u]) val[u] = inf_ref<DICT>(out, dwin, dwl, pos + src, dj);
                        }
                    }
#pragma unroll
                    for (uint32_t u = 0; u < ZWZ_IF_MLP; ++u)
                        if (put[u]) stg[b0 + 32u * u + lane] = (uint8_t) val[u];
                }
                __syncwarp();
                // ---- matches that read this step's own output, in order (their sources lie in EARLIER tokens of the step) ----
                unsigned m = deps & hm;
                if (far) m &= (far & (0u - far)) - 1u; // nothing at or behind the first too-far match is produced
                while (m) {
                    const int j = __ffs((int) m) - 1;
                    m &= m - 1u;
                    const uint32_t mlen = __shfl_sync(ZWZ_FULL, olen, j);
                    const uint32_t m0 = __shfl_sync(ZWZ_FULL, excl, j);
                    const uint32_t dist = __shfl_sync(ZWZ_FULL, dn, j) + 1u;
                    for (uint32_t i = lane; i < mlen; i += 32u) {
                        const uint32_t src = m0 + (dist >= mlen || i < dist ? i : i % dist);
                        if (src >= dist) stg[m0 + i] = stg[src - dist];
                    }
                    __syncwarp();
                }
                // ---- write the step out ----
                uint32_t wr = total;
                if (far) wr = __shfl_sync(ZWZ_FULL, excl, __ffs((int) far) - 1);
                for (uint32_t b = lane; b < wr; b += 32u) {
                    const uint32_t q = pos + b;
                    if (q < cap) out[q] = stg[b];
                }
                if (pos + wr > cap) overflow = true;
                pos += wr;
                if (far) return IFR_BAD;
                __syncwarp();
                j0 += take;
            }
        }
        bitpos += (uint64_t) (last_e - base_bit);
        if (last_flag == IFL_EOB) return IFR_EOB;
        ZWZ_IF_STAT(6, last_flag == IFL_FULL);
        if (last_flag == IFL_STOP) {
            ZWZ_IF_STAT(4, 1);
            return IFR_SLOW;
        }
        // IFL_RUN (all lanes, or the proven prefix after ZWZ_IF_MAXIT rounds) / IFL_FULL: next window
    }
}

// inf_copy_plain (vectorised plain copy for stored blocks) lives in zwz_common.cuh: the encoder's stored writers use it too

#ifdef ZWZ_EMU
ZWZ_DEV uint32_t inf_dp4a(uint32_t a, uint32_t b, uint32_t c) {
    return c + (a & 255u) * (b & 255u) + ((a >> 8) & 255u) * ((b >> 8) & 255u) + ((a >> 16) & 255u) * ((b >> 16) & 255u) + (a >> 24) * (b >> 24);
}
#else
ZWZ_DEV uint32_t inf_dp4a(uint32_t a, uint32_t b, uint32_t c) { return __dp4a(a, b, c); }
#endif

// Adler-32 of out[0..n) (bytes this warp wrote: read through L2), 16 bytes per lane and step.
ZWZ_DEV uint32_t inf_adler32(const uint8_t *out, uint32_t n) {
    const unsigned lane = lane_id();
    uint64_t s0 = 0, s1 = 0; // s0 = sum v_j, s1 = sum (j mod 65521) * v_j
    uint32_t head = (16u - (uint32_t) ((uintptr_t) out & 15u)) & 15u;
    if (head > n) head = n;
    if (lane < head) {
        const uint32_t v = __ldcg(out + lane);
        s0 += v;
        s1 += (uint64_t) lane * v;
    }
    const uint32_t nvec = (n - head) >> 4;
    for (uint32_t k = lane; k < nvec; k += 32u) {
        const uint32_t j0 = head + 16u * k;
        const uint4 w = __ldcg((const uint4 *) (out + j0));
        const uint32_t a0 = inf_dp4a(w.x, 0x01010101u, 0u), a1 = inf_dp4a(w.y, 0x01010101u, 0u), a2 = inf_dp4a(w.z, 0x01010101u, 0u),
                       a3 = inf_dp4a(w.w, 0x01010101u, 0u);
        // sum over the 16 bytes of (index inside the vector) * byte
        const uint32_t t = inf_dp4a(w.x, 0x03020100u, 0u) + inf_dp4a(w.y, 0x07060504u, 0u) + inf_dp4a(w.z, 0x0b0a0908u, 0u) +
                           inf_dp4a(w.w, 0x0f0e0d0cu, 0u);
        const uint32_t sum = a0 + a1 + a2 + a3;
        s0 += sum;
        s1 += (uint64_t) (j0 % 65521u) * sum + t;
    }
    const uint32_t done = head + (nvec << 4);
    if (done + lane < n) {
        const uint32_t j = done + lane;
        const uint32_t v = __ldcg(out + j);
        s0 += v;
        s1 += (uint64_t) (j % 65521u) * v;
    }
    s0 = warp_sum64(s0) % 65521u;
    s1 = warp_sum64(s1 % 65521u) % 65521u;
    const uint64_t nm = n % 65521u;
    const uint32_t a = (uint32_t) ((1u + s0) % 65521u);
    const uint32_t b = (uint32_t) ((nm + nm * s0 + 65521u - s1) % 65521u);
    return (b << 16) | a;
}

} // namespace zwz
