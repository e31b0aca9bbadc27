// deflate_encode.cuh — parse + dynamic Huffman + bit packing, one warp per chunk.
//
// Second half of the replacement for zlib's deflate() at compression.cpp:119-134. Input: the per-position best matches
// left in HBM scratch by lz_match_kernel and the raw chunk. Output: one complete zlib stream (78 9C, one final DEFLATE
// block — stored, fixed or dynamic, whichever is smallest — and the big-endian Adler-32), or two stored streams when
// even the smallest encoding would not fit the reader's 65 535-byte payload array (decompression.cpp:116).
// job.format selects the wrapper around the same DEFLATE body: ZLIB as above, GZIP one BGZF member (18-byte header with
// the BC extra subfield, little-endian CRC-32 and ISIZE), RAW the bare blocks. Only the zlib form has the split rule.
//
// Per warp:
//   parse   32 positions per step. Every lane decides locally "match here or literal" with zlib-style lazy evaluation
//           (a match is deferred when the next position has a longer one), which makes `next[i]` a pure function of the
//           scratch; the token path through the window is then recovered with 5 rounds of pointer doubling on
//           (jump, reach-mask) pairs exchanged by warp shuffles; tokens are compacted in place with ballot + popc and
//           the literal/length and distance histograms are updated with shared-memory atomics.
//   codes   symbols ranked by frequency (rank sort across lanes), two-queue Huffman merge, depth histogram clamped to
//           15 (7 for the code-length alphabet) with zlib's overflow repair, lengths re-assigned by rank, canonical codes
//           assigned 32 symbols per step with __match_any_sync, bit-reversed for LSB-first output.
//   header  code lengths run-length coded exactly like RFC 1951 §3.2.7 allows (16/17/18), third Huffman code over that.
//   emit    32 tokens per step: each lane builds its <= 48-bit code, a warp-shuffle inclusive prefix sum of the bit counts
//           gives every lane its bit offset, lanes OR their bits into a shared-memory staging window and full 32-bit words
//           are flushed to the output slot with one coalesced store.
//
// Algorithmic HBM bytes per chunk: N_raw read + N_comp written (SURVEY.md §8(d)); the scratch round trip (8 N_raw) is
// design traffic.
#pragma once
#include "zwz_common.cuh"

namespace zwz {

#define ZWZ_DE_WARPS 4
#define ZWZ_DE_LL 286
#define ZWZ_DE_D 30
#define ZWZ_DE_DOFF 288 // distance symbols live at freq[288 + d]
#define ZWZ_DE_BASE 4096u // tokens per base block (blocks are merged runs of these)

struct EncWarpSmem {
    uint32_t freq[320];     // [0,286) literal/length, [288,318) distance
    uint32_t code[320];     // (bit length << 16) | bit-reversed code
    uint32_t clfreq[20];    // code-length alphabet
    uint32_t clcode[20];
    uint32_t key[288];      // (freq << 9 | symbol) of used symbols, then sorted ascending
    uint32_t weight[576];   // leaves then internal nodes
    uint16_t parent[576];
    uint8_t blen[320];      // code lengths (literal/length at 0, distance at 288)
    uint8_t clblen[20];
    uint32_t bl_count[16];
    uint32_t next_code[16];
    uint8_t cl_sym[320];    // run-length coded code lengths
    uint8_t cl_ext[320];
    uint32_t stage[64];     // bit sink staging window
    uint32_t misc[8];
    uint32_t region[16];    // stored regions of the chunk: {first token, end token, first byte, end byte} x 4
    uint32_t tflags[ZWZ_SCR_FLAG_WORDS]; // bit t: the 32-position tile t holds a match (its scratch words are valid)
    uint16_t kb_tok[66];    // token count before the first parse step that STARTS inside each 1 024-byte stretch (tokens from
                            // there on start inside it or later)
    uint16_t kb_end[66];    // token count before the first parse step that REACHES into the stretch (tokens before it start earlier)
    uint16_t kb_pos[66];    // byte positions of those two steps
    uint16_t kb_endpos[66];
};
#define ZWZ_DE_SMEM (ZWZ_DE_WARPS * (uint32_t) sizeof(zwz::EncWarpSmem))

// The warp's slice of the CTA's (dynamic) shared memory. The out-of-line helpers below fetch it themselves instead of taking
// a reference, so that the compiler still knows the address space (a reference parameter would turn every access into a
// generic load). They are out of line on purpose: fully inlined, this kernel was 345 KB of SASS — three copies of the block
// emitter, nine of the Huffman construction — and with 24 warps per SM in different phases the dominant stall was
// instruction fetch (`no_instruction`, profiles/round1_notes.md).
ZWZ_DEV EncWarpSmem &enc_smem() {
    ZWZ_DYN_SMEM(enc_raw);
    return ((EncWarpSmem *) enc_raw)[warp_id()];
}

// -------------------------------------------------------------------------------------------------------------------
// Length-limited Huffman code for the `nsym` symbols whose counts are freq[0..nsym). Writes blen[] and code[].
// -------------------------------------------------------------------------------------------------------------------
ZWZ_DEV void enc_huffman_body(EncWarpSmem &S, const uint32_t *freq, uint32_t nsym, uint32_t maxbits, uint8_t *blen, uint32_t *code) {
    const unsigned lane = lane_id();
    // 1. compact used symbols into keys
    uint32_t nused = 0;
    for (uint32_t base = 0; base < nsym; base += 32u) {
        uint32_t s = base + lane;
        uint32_t f = s < nsym ? freq[s] : 0u;
        unsigned m = __ballot_sync(ZWZ_FULL, f != 0u);
        if (f) S.key[nused + (uint32_t) __popc(m & ((1u << lane) - 1u))] = (f << 9) | s;
        nused += (uint32_t) __popc(m);
        if (s < nsym) blen[s] = 0;
    }
    __syncwarp();
    // zlib's rule (trees.c build_tree): force at least two codes so the code is complete and every decoder accepts it
    if (nused < 2u) {
        if (lane == 0) {
            uint32_t have = nused ? (S.key[0] & 511u) : 0xffffu;
            uint32_t d0 = have == 0u ? 1u : 0u;
            S.key[nused] = (1u << 9) | d0;
            if (nused == 0u) S.key[1] = (1u << 9) | 1u;
        }
        nused = 2u;
        __syncwarp();
    }
    // 2. rank sort ascending by (freq, symbol) into weight[]/sorted order; keys are unique
    uint32_t mykey[9], myrank[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        uint32_t i = lane + 32u * k;
        mykey[k] = i < nused ? S.key[i] : 0xffffffffu;
        myrank[k] = 0;
    }
    for (uint32_t j = 0; j < nused; ++j) {
        uint32_t kj = S.key[j];
#pragma unroll
        for (int k = 0; k < 9; ++k) myrank[k] += kj < mykey[k] ? 1u : 0u;
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        uint32_t i = lane + 32u * k;
        if (i < nused) S.key[myrank[k]] = mykey[k];
    }
    __syncwarp();
    for (uint32_t i = lane; i < nused; i += 32u) S.weight[i] = S.key[i] >> 9;
    __syncwarp();
    // 3. two-queue merge (serial; the data is tiny and sorted, the other lanes wait). Queue heads live in registers.
    if (lane == 0) {
        uint32_t leaf = 0, inode = nused, next = nused;
        const uint32_t last = 2u * nused - 1u;
        uint32_t wl = S.weight[0], wi = 0xffffffffu; // head weights; 0xffffffff = queue empty
        while (next < last) {
            uint32_t sum = 0;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                if (wl <= wi) { // ties prefer the leaf (shallower trees)
                    sum += wl;
                    S.parent[leaf] = (uint16_t) next;
                    ++leaf;
                    wl = leaf < nused ? S.weight[leaf] : 0xffffffffu;
                } else {
                    sum += wi;
                    S.parent[inode] = (uint16_t) next;
                    ++inode;
                    wi = inode < next ? S.weight[inode] : 0xffffffffu;
                }
            }
            S.weight[next] = sum;
            if (wi == 0xffffffffu && inode == next) wi = sum; // the node just made becomes the internal head
            ++next;
        }
        S.parent[last - 1u] = 0xffffu; // root
    }
    if (lane < 16u) S.bl_count[lane] = 0;
    __syncwarp();
    // 4. leaf depths (walk to the root), histogram clamped at maxbits
    const uint32_t root = 2u * nused - 2u;
    for (uint32_t i = lane; i < nused; i += 32u) {
        uint32_t d = 0, v = i;
        while (v != root) {
            v = S.parent[v];
            ++d;
        }
        if (d > maxbits) d = maxbits;
        atomicAdd(&S.bl_count[d], 1u);
    }
    __syncwarp();
    // 5. repair after clamping (the step of zlib's gen_bitlen): the clamped lengths over-subscribe the code space by
    //    `excess` units of 2^-maxbits; each step turns a leaf at the deepest level below maxbits into an internal node
    //    whose children are that leaf and one of the clamped leaves, which frees exactly one unit.
    if (lane == 0) {
        uint32_t total = 0;
        for (uint32_t b = 1; b <= maxbits; ++b) total += S.bl_count[b] << (maxbits - b);
        int excess = (int) total - (int) (1u << maxbits);
        while (excess > 0) {
            uint32_t bits = maxbits - 1u;
            while (S.bl_count[bits] == 0u) --bits;
            S.bl_count[bits]--;
            S.bl_count[bits + 1u] += 2u;
            S.bl_count[maxbits]--;
            --excess;
        }
    }
    __syncwarp();
    // 6. lengths by rank: the rarest symbols take the longest codes
    {
        uint32_t cum[16];
        uint32_t acc = 0;
#pragma unroll
        for (int b = 15; b >= 1; --b) {
            acc += (uint32_t) b <= maxbits ? S.bl_count[b] : 0u;
            cum[b] = acc; // symbols with rank < cum[b] have length >= b
        }
        for (uint32_t i = lane; i < nused; i += 32u) {
            uint32_t L = 1;
#pragma unroll
            for (int b = 2; b <= 15; ++b)
                if (i < cum[b]) L = (uint32_t) b;
            blen[S.key[i] & 511u] = (uint8_t) L;
        }
    }
    // 7. canonical codes
    if (lane == 0) {
        uint32_t c = 0;
        S.next_code[0] = 0;
        for (uint32_t b = 1; b <= 15u; ++b) {
            c = (c + (b - 1u <= maxbits && b > 1u ? S.bl_count[b - 1u] : 0u)) << 1;
            S.next_code[b] = c;
        }
    }
    __syncwarp();
    for (uint32_t base = 0; base < nsym; base += 32u) {
        uint32_t s = base + lane;
        uint32_t L = s < nsym ? blen[s] : 0u;
        unsigned grp = __match_any_sync(ZWZ_FULL, L);
        if (s < nsym) {
            uint32_t cw = 0;
            if (L) {
                cw = S.next_code[L] + (uint32_t) __popc(grp & ((1u << lane) - 1u));
                cw = __brev(cw) >> (32u - L);
            }
            code[s] = (L << 16) | cw;
        }
        __syncwarp();
        if (L && (grp >> lane) == 1u) S.next_code[L] += (uint32_t) __popc(grp);
        __syncwarp();
    }
}

// -------------------------------------------------------------------------------------------------------------------
// bit sink: warp-collective append of (bits, nbits <= 57) per lane, in lane order
// -------------------------------------------------------------------------------------------------------------------
// which: 0 = literal/length, 1 = distance, 2 = code-length alphabet
ZWZ_DEV_NOINLINE void enc_huffman(uint32_t which) {
    EncWarpSmem &S = enc_smem();
    const uint32_t *freq = which == 0u ? S.freq : (which == 1u ? S.freq + ZWZ_DE_DOFF : S.clfreq);
    uint8_t *blen = which == 0u ? S.blen : (which == 1u ? S.blen + ZWZ_DE_DOFF : S.clblen);
    uint32_t *code = which == 0u ? S.code : (which == 1u ? S.code + ZWZ_DE_DOFF : S.clcode);
    enc_huffman_body(S, freq, which == 0u ? ZWZ_DE_LL : (which == 1u ? ZWZ_DE_D : 19u), which == 2u ? 7u : 15u, blen, code);
}

struct BitSink {
    uint32_t *outw;     // 4-byte aligned output words
    uint32_t nwords;    // words already produced (counted even when they no longer fit)
    uint32_t fill;      // bits waiting in stage[0]
    uint32_t cap_words; // words the output slot can take; past it the sink only counts
};

ZWZ_DEV void sink_init(EncWarpSmem &S, BitSink &k, uint32_t *outw, uint32_t cap_words) {
    k.outw = outw;
    k.nwords = 0;
    k.fill = 0;
    k.cap_words = cap_words;
    S.stage[lane_id()] = 0;
    S.stage[lane_id() + 32u] = 0;
    __syncwarp();
}
ZWZ_DEV void sink_put(EncWarpSmem &S, BitSink &k, uint64_t bits, uint32_t nbits) {
    const unsigned lane = lane_id();
    uint32_t incl = warp_incl_scan(nbits);
    uint32_t total = __shfl_sync(ZWZ_FULL, incl, 31);
    if (nbits) {
        uint32_t pos = k.fill + incl - nbits;
        uint32_t w = pos >> 5, sh = pos & 31u;
        uint64_t lo = bits << sh;
        uint32_t hi = sh ? (uint32_t) (bits >> (64u - sh)) : 0u;
        atomicOr(&S.stage[w], (uint32_t) lo);
        if ((uint32_t) (lo >> 32)) atomicOr(&S.stage[w + 1u], (uint32_t) (lo >> 32));
        if (hi) atomicOr(&S.stage[w + 2u], hi);
    }
    __syncwarp();
    uint32_t nf = k.fill + total;
    uint32_t full = nf >> 5;
    uint32_t v0 = S.stage[lane], v1 = S.stage[lane + 32u];
    if (lane < full && k.nwords + lane < k.cap_words) k.outw[k.nwords + lane] = v0;
    if (lane + 32u < full && k.nwords + lane + 32u < k.cap_words) k.outw[k.nwords + lane + 32u] = v1;
    uint32_t carry = __shfl_sync(ZWZ_FULL, full < 32u ? v0 : v1, (int) (full & 31u));
    __syncwarp();
    S.stage[lane] = lane == 0 ? carry : 0u;
    S.stage[lane + 32u] = 0;
    __syncwarp();
    k.nwords += full;
    k.fill = nf & 31u;
}
// store the partial last word; returns total bytes (may exceed the slot: then nothing past it was written)
ZWZ_DEV uint32_t sink_finish(EncWarpSmem &S, BitSink &k) {
    if (k.fill && lane_id() == 0 && k.nwords < k.cap_words) k.outw[k.nwords] = S.stage[0];
    return k.nwords * 4u + ((k.fill + 7u) >> 3);
}

ZWZ_DEV_NOINLINE uint32_t enc_adler_global(const uint8_t *p, uint32_t n) {
    uint64_t s0 = 0, s1 = 0;
    for (uint32_t j = lane_id(); j < n; j += 32u) {
        uint32_t v = p[j];
        s0 += v;
        s1 += (uint64_t) j * v;
    }
    s0 = warp_sum64(s0) % 65521u;
    s1 = warp_sum64(s1 % 65521u) % 65521u;
    uint64_t nm = n % 65521u;
    uint32_t a = (uint32_t) ((1u + s0) % 65521u);
    uint32_t b = (uint32_t) ((nm + nm * s0 + 65521u - s1) % 65521u);
    return (b << 16) | a;
}

// wrapper bytes in front of the DEFLATE body, and in front plus behind it
// ZWZ_WRAP_ZLIB_DICT: the wrapper of a zlib chunk with a preset dictionary, 78 BB (FDICT set) + DICTID in front. It has no split
// rule and no 65 535-byte limit (neither has GZIP or RAW): the split rule serves .zwz records, which never have a dictionary.
#define ZWZ_WRAP_ZLIB_DICT 3u
// Pieces of one longer stream (zwz_deflate_stream, zwz_deflater), always launched with the DICT kernels: the chunks' windows are
// their "dictionaries". ZWZ_WRAP_PIECES: every chunk is a non-final piece: no header, no trailer, BFINAL = 0 on every block, and
// an empty stored block behind the body (3 zero bits, padding, 00 00 ff ff: zlib's Z_SYNC_FLUSH marker), so that pieces join byte
// for byte. ZWZ_WRAP_PIECES_LAST: the same, but the launch's last chunk is the stream's final piece, written as a RAW body.
#define ZWZ_WRAP_PIECES 4u
#define ZWZ_WRAP_PIECES_LAST 5u
#define ZWZ_WRAP_PIECE 6u // per chunk: a non-final piece
ZWZ_DEV uint32_t enc_head_bytes(uint32_t format) {
    return format == ZWZ_FORMAT_GZIP ? 18u : (format == ZWZ_FORMAT_ZLIB ? 2u : (format == ZWZ_WRAP_ZLIB_DICT ? 6u : 0u));
}
ZWZ_DEV uint32_t enc_wrap_bytes(uint32_t format) { return enc_head_bytes(format) + (format == ZWZ_FORMAT_GZIP ? 8u : (format == ZWZ_FORMAT_RAW ? 0u : 4u)); }

// BSIZE of a BGZF member header (bytes 16-17): the member's length minus 1
ZWZ_DEV void enc_bgzf_bsize(uint8_t *out, uint32_t member_bytes) {
    out[16] = (uint8_t) (member_bytes - 1u);
    out[17] = (uint8_t) ((member_bytes - 1u) >> 8);
}

// one complete stream in `format` with a single stored block (check = Adler-32 for zlib, CRC-32 for gzip); returns its size
ZWZ_DEV_NOINLINE uint32_t enc_stored_stream(uint8_t *out, const uint8_t *src, uint32_t n, uint32_t check, uint32_t format, uint32_t dictid) {
    const unsigned lane = lane_id();
    const uint32_t h = enc_head_bytes(format);
    if (lane == 0) {
        if (format == ZWZ_FORMAT_ZLIB) {
            out[0] = 0x78;
            out[1] = 0x9c;
        } else if (format == ZWZ_WRAP_ZLIB_DICT) {
            out[0] = 0x78;
            out[1] = 0xbb;
            for (int i = 0; i < 4; ++i) out[2 + i] = (uint8_t) (dictid >> (24 - 8 * i));
        } else if (format == ZWZ_FORMAT_GZIP) {
            uint32_t *w = (uint32_t *) out; // the slot start: 4-byte aligned
            w[0] = 0x04088b1fu;             // 1f 8b 08 04 | MTIME 0 | XFL 0, OS ff | XLEN 6 | 'B' 'C' 2 0
            w[1] = 0u;
            w[2] = 0x0006ff00u;
            w[3] = 0x00024342u;
            enc_bgzf_bsize(out, n + 31u);
        }
        out[h] = 0x01;
        out[h + 1u] = (uint8_t) n;
        out[h + 2u] = (uint8_t) (n >> 8);
        out[h + 3u] = (uint8_t) ~n;
        out[h + 4u] = (uint8_t) (~n >> 8);
        uint8_t *t = out + h + 5u + n;
        if (format == ZWZ_FORMAT_ZLIB || format == ZWZ_WRAP_ZLIB_DICT) {
            t[0] = (uint8_t) (check >> 24);
            t[1] = (uint8_t) (check >> 16);
            t[2] = (uint8_t) (check >> 8);
            t[3] = (uint8_t) check;
        } else if (format == ZWZ_FORMAT_GZIP) {
            for (int i = 0; i < 4; ++i) {
                t[i] = (uint8_t) (check >> (8 * i));
                t[4 + i] = (uint8_t) (n >> (8 * i));
            }
        }
    }
    __syncwarp();
    inf_copy_plain(out + h + 5u, src, n);
    return n + 5u + enc_wrap_bytes(format);
}

// a non-final piece as one stored block (BFINAL 0) followed by the empty stored block; returns its size, n + 10
ZWZ_DEV_NOINLINE uint32_t enc_stored_piece(uint8_t *out, const uint8_t *src, uint32_t n) {
    const uint32_t l = enc_stored_stream(out, src, n, 0u, ZWZ_FORMAT_RAW, 0u);
    if (lane_id() == 0) {
        out[0] = 0x00;
        out[l] = out[l + 1u] = out[l + 2u] = 0x00;
        out[l + 3u] = out[l + 4u] = 0xff;
    }
    __syncwarp();
    return l + 5u;
}

// the end of a non-final Huffman-coded piece: the empty stored block (3 zero bits, padding to a byte, LEN 0000, NLEN ffff)
ZWZ_DEV_NOINLINE void enc_piece_tail(BitSink *kp) {
    EncWarpSmem &S = enc_smem();
    const unsigned lane = lane_id();
    BitSink k = *kp;
    const uint32_t hb = 3u + ((8u - ((k.nwords * 32u + k.fill + 3u) & 7u)) & 7u);
    sink_put(S, k, lane == 1u ? 0xffff0000ull : 0ull, lane == 0 ? hb : (lane == 1u ? 32u : 0u));
    *kp = k;
}

// histogram of the tokens [t0, t1) into freq[0..320) (literal/length at 0, distance at 288); returns their extra bits
// into_code: histogram into S.code (free between two Huffman builds) instead of S.freq
ZWZ_DEV_NOINLINE uint64_t enc_hist_tokens(const uint32_t *m, uint32_t t0, uint32_t t1, bool into_code) {
    EncWarpSmem &S = enc_smem();
    uint32_t *freq = into_code ? S.code : S.freq;
    const unsigned lane = lane_id();
    for (uint32_t i = lane; i < 320u; i += 32u) freq[i] = 0;
    __syncwarp();
    uint64_t extra = 0;
    for (uint32_t i = t0 + lane; i < t1; i += 32u) {
        uint32_t tok = m[i];
        uint32_t len = tok_len(tok);
        if (len == 0u) {
            atomicAdd(&freq[tok_byte(tok)], 1u);
        } else {
            uint32_t ls, le, lv, ds, de, dv;
            len_symbol(len, ls, le, lv);
            dist_symbol(tok_dist(tok), ds, de, dv);
            atomicAdd(&freq[ls], 1u);
            atomicAdd(&freq[ZWZ_DE_DOFF + ds], 1u);
            extra += le + de;
        }
    }
    extra = warp_sum64(extra);
    __syncwarp();
    return extra;
}

// empirical entropy (bits) of the two alphabets in a[0..320) (+ b[0..320) when b != nullptr), and the used-symbol count
// sel: 0 = S.freq, 1 = S.code (a second histogram), 2 = their sum
ZWZ_DEV_NOINLINE float enc_entropy_bits(uint32_t sel, uint32_t *nused_ptr) {
    EncWarpSmem &S = enc_smem();
    const uint32_t *a = sel == 1u ? S.code : S.freq;
    const uint32_t *b = sel == 2u ? S.code : nullptr;
    uint32_t nused_out;
    const unsigned lane = lane_id();
    float nl = 0.f, nd = 0.f, h = 0.f;
    uint32_t nused = 0;
    for (uint32_t s = lane; s < 320u; s += 32u) {
        float f = (float) (a[s] + (b ? b[s] : 0u));
        if (s < ZWZ_DE_DOFF) nl += f; else nd += f;
        nused += f > 0.f ? 1u : 0u;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        nl += __shfl_xor_sync(ZWZ_FULL, nl, d);
        nd += __shfl_xor_sync(ZWZ_FULL, nd, d);
    }
    for (uint32_t s = lane; s < 320u; s += 32u) {
        float f = (float) (a[s] + (b ? b[s] : 0u));
        if (f > 0.f) h += f * (zwz_log2f(s < ZWZ_DE_DOFF ? nl : nd) - zwz_log2f(f));
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) h += __shfl_xor_sync(ZWZ_FULL, h, d);
    nused_out = warp_sum(nused);
    *nused_ptr = nused_out;
    return h;
}

// One DEFLATE block over the tokens [t0, t1): S.freq must hold their histogram (without the end-of-block symbol).
// Builds the three Huffman codes, picks fixed or dynamic (whichever is smaller) and appends the block to the sink.
ZWZ_DEV void enc_emit_block_body(EncWarpSmem &S, BitSink &k, const uint32_t *m, uint32_t t0, uint32_t t1, uint64_t extra_bits, bool last) {
    const unsigned lane = lane_id();
    if (lane == 0) S.freq[256] += 1u; // end of block
    __syncwarp();
    enc_huffman(0u);
    enc_huffman(1u);
    __syncwarp();

    // HLIT / HDIST: highest used symbol + 1
    uint32_t hl = 0, hd = 0;
    for (uint32_t s = lane; s < ZWZ_DE_LL; s += 32u)
        if (S.blen[s]) hl = s + 1u;
    if (lane < ZWZ_DE_D && S.blen[ZWZ_DE_DOFF + lane]) hd = lane + 1u;
    hl = warp_max(hl);
    hd = warp_max(hd);
    if (hl < 257u) hl = 257u;
    if (hd < 1u) hd = 1u;

    // code-length run-length coding (RFC 1951 §3.2.7; same run rules as zlib's scan_tree)
    if (lane < 20u) S.clfreq[lane] = 0;
    __syncwarp();
    uint32_t ncl = 0;
    if (lane == 0) {
        for (int part = 0; part < 2; ++part) {
            const uint8_t *L = part == 0 ? S.blen : S.blen + ZWZ_DE_DOFF;
            uint32_t cnt_syms = part == 0 ? hl : hd;
            int prevlen = -1;
            uint32_t i = 0;
            while (i < cnt_syms) {
                uint32_t cur = L[i];
                uint32_t run = 1;
                uint32_t maxrun = cur == 0u ? 138u : ((int) cur == prevlen ? 6u : 7u);
                while (i + run < cnt_syms && L[i + run] == cur && run < maxrun) ++run;
                uint32_t minrun = cur == 0u ? 3u : ((int) cur == prevlen ? 3u : 4u);
                if (run < minrun) {
                    for (uint32_t r = 0; r < run; ++r) {
                        S.cl_sym[ncl] = (uint8_t) cur;
                        S.cl_ext[ncl++] = 0;
                    }
                    S.clfreq[cur] += run;
                } else if (cur != 0u) {
                    uint32_t rep = run;
                    if ((int) cur != prevlen) {
                        S.cl_sym[ncl] = (uint8_t) cur;
                        S.cl_ext[ncl++] = 0;
                        S.clfreq[cur] += 1u;
                        rep = run - 1u;
                    }
                    S.cl_sym[ncl] = 16;
                    S.cl_ext[ncl++] = (uint8_t) (rep - 3u);
                    S.clfreq[16] += 1u;
                } else if (run <= 10u) {
                    S.cl_sym[ncl] = 17;
                    S.cl_ext[ncl++] = (uint8_t) (run - 3u);
                    S.clfreq[17] += 1u;
                } else {
                    S.cl_sym[ncl] = 18;
                    S.cl_ext[ncl++] = (uint8_t) (run - 11u);
                    S.clfreq[18] += 1u;
                }
                prevlen = (int) cur;
                i += run;
            }
        }
        S.misc[0] = ncl;
    }
    __syncwarp();
    ncl = S.misc[0];
    enc_huffman(2u);
    __syncwarp();
    // HCLEN: last used entry in the transmission order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
    uint32_t ord = lane < 3u ? 16u + lane : (lane == 3u ? 0u : ((lane & 1u) ? 7u - ((lane - 5u) >> 1) : 8u + ((lane - 4u) >> 1)));
    uint32_t hc = (lane < 19u && S.clblen[ord]) ? lane + 1u : 0u;
    hc = warp_max(hc);
    if (hc < 4u) hc = 4u;

    // sizes of the two Huffman encodings of this block
    uint64_t dyn_bits = 0, fix_bits = 0, hdr_bits = 0;
    for (uint32_t s = lane; s < ZWZ_DE_LL; s += 32u) {
        uint32_t f = S.freq[s];
        dyn_bits += (uint64_t) f * S.blen[s];
        fix_bits += (uint64_t) f * (s < 144u ? 8u : (s < 256u ? 9u : (s < 280u ? 7u : 8u)));
    }
    if (lane < ZWZ_DE_D) {
        uint32_t f = S.freq[ZWZ_DE_DOFF + lane];
        dyn_bits += (uint64_t) f * S.blen[ZWZ_DE_DOFF + lane];
        fix_bits += (uint64_t) f * 5u;
    }
    if (lane < 19u) hdr_bits += (uint64_t) S.clfreq[lane] * (S.clblen[lane] + (lane == 16u ? 2u : (lane == 17u ? 3u : (lane == 18u ? 7u : 0u))));
    dyn_bits = warp_sum64(dyn_bits) + extra_bits + warp_sum64(hdr_bits) + 14u + 3u * hc;
    fix_bits = warp_sum64(fix_bits) + extra_bits;
    const bool fixed = fix_bits <= dyn_bits;
    const uint64_t bfinal = last ? 1u : 0u;

    if (fixed) {
        // fixed codes (RFC 1951 §3.2.6) into the same code[] layout
        for (uint32_t s = lane; s < 288u; s += 32u) {
            uint32_t L = s < 144u ? 8u : (s < 256u ? 9u : (s < 280u ? 7u : 8u));
            uint32_t cw = s < 144u ? 0x30u + s : (s < 256u ? 0x190u + (s - 144u) : (s < 280u ? s - 256u : 0xC0u + (s - 280u)));
            if (s < ZWZ_DE_LL) S.code[s] = (L << 16) | (__brev(cw) >> (32u - L));
        }
        if (lane < ZWZ_DE_D) S.code[ZWZ_DE_DOFF + lane] = (5u << 16) | (__brev(lane) >> 27);
        __syncwarp();
        sink_put(S, k, lane == 0 ? (bfinal | (1ull << 1)) : 0ull, lane == 0 ? 3u : 0u);
    } else {
        // BFINAL, BTYPE=10, HLIT, HDIST, HCLEN, then HCLEN 3-bit lengths (lanes 1..19)
        uint64_t v = 0;
        uint32_t nb = 0;
        if (lane == 0) {
            v = bfinal | (2ull << 1) | ((uint64_t) (hl - 257u) << 3) | ((uint64_t) (hd - 1u) << 8) | ((uint64_t) (hc - 4u) << 13);
            nb = 17u;
        } else if (lane <= hc) {
            uint32_t o = lane - 1u;
            uint32_t od = o < 3u ? 16u + o : (o == 3u ? 0u : ((o & 1u) ? 7u - ((o - 5u) >> 1) : 8u + ((o - 4u) >> 1)));
            v = S.clblen[od];
            nb = 3u;
        }
        sink_put(S, k, v, nb);
        for (uint32_t base = 0; base < ncl; base += 32u) {
            uint32_t i = base + lane;
            uint64_t b = 0;
            uint32_t nbits = 0;
            if (i < ncl) {
                uint32_t sy = S.cl_sym[i];
                uint32_t cw = S.clcode[sy];
                nbits = cw >> 16;
                b = cw & 0xffffu;
                uint32_t eb = sy == 16u ? 2u : (sy == 17u ? 3u : (sy == 18u ? 7u : 0u));
                b |= (uint64_t) S.cl_ext[i] << nbits;
                nbits += eb;
            }
            sink_put(S, k, b, nbits);
        }
    }
    // tokens, then end-of-block. The next step's token is loaded before this step's bits go through the sink (whose warp
    // barriers the compiler will not move loads across).
    uint32_t tnext = t0 + lane < t1 ? m[t0 + lane] : 0u;
    for (uint32_t base = t0; base <= t1; base += 32u) {
        const uint32_t i = base + lane;
        const uint32_t tok = tnext;
        tnext = i + 32u < t1 ? m[i + 32u] : 0u;
        uint64_t b = 0;
        uint32_t nbits = 0;
        if (i < t1) {
            uint32_t len = tok_len(tok);
            if (len == 0u) {
                uint32_t cw = S.code[tok_byte(tok)];
                nbits = cw >> 16;
                b = cw & 0xffffu;
            } else {
                uint32_t ls, le, lv, ds, de, dv;
                len_symbol(len, ls, le, lv);
                dist_symbol(tok_dist(tok), ds, de, dv);
                uint32_t cl = S.code[ls], cd = S.code[ZWZ_DE_DOFF + ds];
                b = cl & 0xffffu;
                nbits = cl >> 16;
                b |= (uint64_t) lv << nbits;
                nbits += le;
                b |= (uint64_t) (cd & 0xffffu) << nbits;
                nbits += cd >> 16;
                b |= (uint64_t) dv << nbits;
                nbits += de;
            }
        } else if (i == t1) {
            uint32_t cw = S.code[256];
            nbits = cw >> 16;
            b = cw & 0xffffu;
        }
        sink_put(S, k, b, nbits);
    }
}

// out of line (once per DEFLATE block): the sink travels through memory, the body works on a register copy
ZWZ_DEV_NOINLINE void enc_emit_block(BitSink *kp, const uint32_t *m, uint32_t t0, uint32_t t1, uint64_t extra_bits, bool last) {
    BitSink k = *kp;
    enc_emit_block_body(enc_smem(), k, m, t0, t1, extra_bits, last);
    *kp = k;
}

// The wrapper around the Huffman-coded body (out of line: the format costs the encoder's main loop no registers).
// Header: zlib 78 9C (78 BB + DICTID big-endian with a preset dictionary); gzip the 18-byte BGZF header with BSIZE left 0 (set by
// enc_wrap_tail); raw none.
ZWZ_DEV_NOINLINE void enc_wrap_head(BitSink *kp, uint32_t format, uint32_t dictid) {
    EncWarpSmem &S = enc_smem();
    const unsigned lane = lane_id();
    BitSink k = *kp;
    if (format == ZWZ_FORMAT_ZLIB) {
        sink_put(S, k, lane == 0 ? 0x9c78ull : 0ull, lane == 0 ? 16u : 0u); // RFC 1950 header 78 9C
    } else if (format == ZWZ_WRAP_ZLIB_DICT) {
        const uint32_t be = ((dictid & 0xffu) << 24) | ((dictid & 0xff00u) << 8) | ((dictid >> 8) & 0xff00u) | (dictid >> 24);
        sink_put(S, k, lane == 0 ? 0xbb78ull : (lane == 1u ? (uint64_t) be : 0ull), lane == 0 ? 16u : (lane == 1u ? 32u : 0u));
    } else if (format == ZWZ_FORMAT_GZIP) {
        // 1f 8b 08 04 | MTIME 0 | XFL 0, OS ff | XLEN 6 | 'B' 'C' 2 0 | BSIZE
        const uint32_t w = lane == 0 ? 0x04088b1fu : (lane == 2u ? 0x0006ff00u : (lane == 3u ? 0x00024342u : 0u));
        sink_put(S, k, w, lane < 4u ? 32u : (lane == 4u ? 16u : 0u));
    }
    *kp = k;
}
// Trailer: pad to a byte boundary, then Adler-32 big-endian (zlib) or CRC-32 and ISIZE little-endian (gzip). A gzip member's
// length is known here: BSIZE goes into its header (whose words the sink has written by now: a member has >= 28 bytes).
ZWZ_DEV_NOINLINE void enc_wrap_tail(BitSink *kp, uint32_t format, uint32_t check, uint32_t n) {
    EncWarpSmem &S = enc_smem();
    const unsigned lane = lane_id();
    BitSink k = *kp;
    const uint32_t padbits = (8u - ((k.nwords * 32u + k.fill) & 7u)) & 7u;
    const uint32_t be = ((check & 0xffu) << 24) | ((check & 0xff00u) << 8) | ((check >> 8) & 0xff00u) | (check >> 24);
    uint64_t v = 0;
    uint32_t nb = lane == 0 ? padbits : 0u;
    if (lane == 1u && format != ZWZ_FORMAT_RAW) {
        v = format == ZWZ_FORMAT_GZIP ? check : be;
        nb = 32u;
    } else if (lane == 2u && format == ZWZ_FORMAT_GZIP) {
        v = n;
        nb = 32u;
    }
    sink_put(S, k, v, nb);
    if (format == ZWZ_FORMAT_GZIP && lane == 0) enc_bgzf_bsize((uint8_t *) k.outw, k.nwords * 4u + (k.fill >> 3));
    *kp = k;
}

#define ZWZ_DE_STORED_MIN 512u // literal tokens in a row before a stored region is considered

// Stored-region candidates come for free from the match kernel's tile flags: a 1 024-byte stretch with matches in at most
// ZWZ_DE_QUIET_TILES of its 32 tiles is (nearly) match-free — uniformly random bytes still repeat a 3-byte string now and then.
// Runs of such stretches whose tokens leave a Huffman code less than n/256 bytes + 8 to gain over plain bytes become
// S.region[] = {first token, end token, first byte, end byte} (from the marks the parse left). At most 4 per chunk.
#define ZWZ_DE_QUIET_TILES 3
ZWZ_DEV_NOINLINE uint32_t enc_find_stored_regions(const uint32_t *m, uint32_t n, uint32_t ntok) {
    EncWarpSmem &S = enc_smem();
    const unsigned lane = lane_id();
    const uint32_t nkb = (n + 1023u) >> 10;
    const unsigned q0 = __ballot_sync(ZWZ_FULL, lane < nkb && __popc(S.tflags[lane]) <= ZWZ_DE_QUIET_TILES);
    const unsigned q1 = __ballot_sync(ZWZ_FULL, lane + 32u < nkb && __popc(S.tflags[lane + 32u]) <= ZWZ_DE_QUIET_TILES);
    uint64_t quiet = (uint64_t) q0 | ((uint64_t) q1 << 32);
    uint32_t nreg = 0;
    if (quiet == 0ull) return 0u;
    // an unset mark takes the next set one (the end of the chunk behind the last): "first step at or behind this stretch"
    if (lane == 0) {
        uint32_t t = ntok, q = n, te = ntok, qe = n;
        for (int k = 64; k >= 0; --k) {
            if (S.kb_tok[k] == 0xffffu) {
                S.kb_tok[k] = (uint16_t) t;
                S.kb_pos[k] = (uint16_t) q;
            } else {
                t = S.kb_tok[k];
                q = S.kb_pos[k];
            }
            if (S.kb_end[k] == 0xffffu) {
                S.kb_end[k] = (uint16_t) te;
                S.kb_endpos[k] = (uint16_t) qe;
            } else {
                te = S.kb_end[k];
                qe = S.kb_endpos[k];
            }
        }
    }
    __syncwarp();
    while (quiet && nreg < 4u) { // warp-uniform
        const uint32_t a = (uint32_t) __ffsll((long long) quiet) - 1u;
        uint64_t rest = ~(quiet >> a); // first zero above a ends the run
        const uint32_t len = rest ? (uint32_t) __ffsll((long long) rest) - 1u : 64u - a;
        const uint32_t b = a + len;
        quiet = b >= 64u ? 0ull : quiet & ~((1ull << b) - 1ull);
        // tokens [r0, r1) = bytes [p0, p1): from the first step that starts in stretch a up to the first step that reaches into
        // stretch b (a step that starts in b - 1 may already emit tokens of b's first positions)
        const uint32_t r0 = S.kb_tok[a], r1 = b < nkb ? S.kb_end[b] : ntok;
        const uint32_t p0 = S.kb_pos[a], p1 = b < nkb ? S.kb_endpos[b] : n;
        if (r1 > r0 && p1 > p0 && p1 - p0 >= ZWZ_DE_STORED_MIN) {
            const uint64_t xb = enc_hist_tokens(m, r0, r1, true); // into S.code: S.freq keeps the whole-chunk histogram
            uint32_t nu;
            const float h_bits = enc_entropy_bits(1u, &nu) + (float) xb;
            const float nb = (float) (p1 - p0);
            if (8.f * nb - h_bits < nb * (1.f / 32.f) + 64.f) {
                if (lane == 0) {
                    S.region[4u * nreg] = r0;
                    S.region[4u * nreg + 1u] = r1;
                    S.region[4u * nreg + 2u] = p0;
                    S.region[4u * nreg + 3u] = p1;
                }
                ++nreg;
            }
        }
    }
    __syncwarp();
    return nreg;
}

// The raw bytes src[0, nbytes) as one stored block (RFC 1951 §3.2.4): 3 header bits, pad to a byte boundary, LEN, NLEN, bytes.
ZWZ_DEV_NOINLINE void enc_emit_stored_block(BitSink *kp, const uint8_t *src, uint32_t nbytes, bool last) {
    EncWarpSmem &S = enc_smem();
    BitSink k = *kp;
    const unsigned lane = lane_id();
    const uint32_t at = k.nwords * 32u + k.fill + 3u; // nbytes <= 65 535: a chunk has no more
    const uint32_t pad = (8u - (at & 7u)) & 7u;
    uint64_t v = 0;
    uint32_t nb = 0;
    if (lane == 0) {
        v = last ? 1ull : 0ull; // BFINAL, BTYPE = 00, zero padding
        nb = 3u + pad;
    } else if (lane == 1u) {
        v = (uint64_t) nbytes | ((uint64_t) (~nbytes & 0xffffu) << 16);
        nb = 32u;
    }
    sink_put(S, k, v, nb);
    // The stream is at a byte boundary now and the payload is plain bytes: they go straight to the slot (16-byte stores) instead
    // of through the bit sink, which is then set up again behind them. Bytes the sink still holds (< 4) are written out first.
    uint8_t *ob = (uint8_t *) k.outw;
    const uint32_t cap_bytes = k.cap_words * 4u;
    const uint32_t pend = k.fill >> 3, b0 = k.nwords * 4u;
    const uint32_t held = S.stage[0];
    __syncwarp();
    if (lane < pend && b0 + lane < cap_bytes) ob[b0 + lane] = (uint8_t) (held >> (8u * lane));
    const uint32_t dst = b0 + pend, end = dst + nbytes; // nbytes >= ZWZ_DE_STORED_MIN: the last word's bytes all come from src
    const uint32_t ncopy = dst >= cap_bytes ? 0u : (end <= cap_bytes ? nbytes : cap_bytes - dst); // past the slot the sink only counts
    __syncwarp();
    if (ncopy) inf_copy_plain(ob + dst, src, ncopy);
    const uint32_t tail = end & 3u;
    uint32_t tw = 0;
    if (lane == 0)
        for (uint32_t j = 0; j < tail; ++j) tw |= (uint32_t) src[nbytes - tail + j] << (8u * j);
    __syncwarp();
    S.stage[lane] = lane == 0 ? tw : 0u;
    S.stage[lane + 32u] = 0u;
    __syncwarp();
    k.nwords = end >> 2;
    k.fill = tail * 8u;
    *kp = k;
}

// The tokens [t0, t1) as one or more Huffman blocks. whole: S.freq already holds their histogram and extra_bits their extra
// bits (the range is the whole chunk, straight from the parse).
ZWZ_DEV_NOINLINE void enc_emit_range(BitSink *kp, const uint32_t *m, uint32_t t0r, uint32_t t1r, uint64_t extra_bits, bool last, bool whole) {
    EncWarpSmem &S = enc_smem();
    const unsigned lane = lane_id();
    const uint32_t nt = t1r - t0r;
    // base blocks of equal size, about ZWZ_DE_BASE tokens each (a short tail block would pay a whole header for nothing)
    const uint32_t nbase = (nt + ZWZ_DE_BASE / 2u) / ZWZ_DE_BASE;
    if (nbase <= 1u) {
        if (!whole) extra_bits = enc_hist_tokens(m, t0r, t1r, false);
        enc_emit_block(kp, m, t0r, t1r, extra_bits, last);
        return;
    }
    const uint32_t bsz = (nt + nbase - 1u) / nbase;
    uint32_t t0 = t0r, t1 = t0r + bsz;
    uint64_t xb = enc_hist_tokens(m, t0, t1, false);
    while (t1 < t1r) {
        const uint32_t t2 = t1 + bsz < t1r ? t1 + bsz : t1r;
        uint32_t *nf = S.code; // free until the next Huffman build
        const uint64_t xn = enc_hist_tokens(m, t1, t2, true);
        uint32_t ua, ub, uab;
        const float ha = enc_entropy_bits(0u, &ua);
        const float hb = enc_entropy_bits(1u, &ub);
        const float hab = enc_entropy_bits(2u, &uab);
        const float sep = ha + hb + 200.f + 4.f * (float) (ua + ub);
        const float mer = hab + 100.f + 4.f * (float) uab;
        if (mer <= sep) {
            for (uint32_t i = lane; i < 320u; i += 32u) S.freq[i] += nf[i];
            __syncwarp();
            xb += xn;
            t1 = t2;
        } else {
            enc_emit_block(kp, m, t0, t1, xb, false);
            t0 = t1;
            t1 = t2;
            xb = enc_hist_tokens(m, t0, t1, false);
        }
    }
    enc_emit_block(kp, m, t0, t1, xb, last);
}

template <bool DICT> ZWZ_DEV void enc_chunk(EncWarpSmem &S, const DeflateJob &job, uint32_t c) {
    const unsigned lane = lane_id();
    const uint32_t n = job.raw_len[c];
    // the wrapper of this chunk: a zlib chunk with a preset dictionary names it in its header (RAW streams do not)
    uint32_t fmt = job.format, dictid = 0;
    if (DICT) {
        if (fmt == ZWZ_WRAP_PIECES || fmt == ZWZ_WRAP_PIECES_LAST)
            fmt = fmt == ZWZ_WRAP_PIECES_LAST && c + 1u == job.n ? ZWZ_FORMAT_RAW : ZWZ_WRAP_PIECE;
        const uint32_t di = job.dict.idx[c];
        if (di != ZWZ_NO_DICT && fmt == ZWZ_FORMAT_ZLIB) {
            fmt = ZWZ_WRAP_ZLIB_DICT;
            dictid = job.dict.id[di];
        }
    }
    const bool piece = DICT && fmt == ZWZ_WRAP_PIECE; // compile-time false in the kernels of the calls without dictionaries
    const uint8_t *src = job.raw + job.raw_off[c];
    uint32_t *m = job.scratch + job.scr_off[c];
    uint8_t *out = job.out + job.out_off[c];

    for (uint32_t i = lane; i < 320u; i += 32u) S.freq[i] = 0;
    __syncwarp();

    // ---------------- incompressibility shortcut ----------------
    // The match kernel reports how many positions found a match. When (almost) none did, the token stream is (almost) the
    // byte stream: its histogram comes straight from the raw bytes (coalesced, no dependent loads) and the entropy bound below
    // decides "stored" without ever walking the 4-byte-per-position scratch. Config C2 is 70 % such chunks.
    if (n >= 512u && job.nmatch[c] * 64u <= n) {
        for (uint32_t i = lane; i < n; i += 32u) atomicAdd(&S.freq[src[i]], 1u);
        __syncwarp();
        if (lane == 0) S.freq[256] = 1u;
        __syncwarp();
        uint32_t nu;
        const float hb = enc_entropy_bits(0u, &nu);
        const float bound_bytes = hb * 0.125f + 7.f + (float) (nu >> 2);
        if (bound_bytes * 0.9995f >= (float) (n + 11u) - (float) (n >> 8) && (fmt != ZWZ_FORMAT_ZLIB || n + 11u <= ZWZ_CHUNK)) {
            uint32_t l0 = piece ? enc_stored_piece(out, src, n) : enc_stored_stream(out, src, n, job.adler[c], fmt, dictid);
            if (lane == 0) {
                job.res[4u * c + 0u] = l0;
                job.res[4u * c + 1u] = 0u;
                job.res[4u * c + 2u] = n;
                job.res[4u * c + 3u] = 0u;
            }
            return;
        }
        for (uint32_t i = lane; i < 320u; i += 32u) S.freq[i] = 0;
        __syncwarp();
    }

    // ---------------- parse ----------------
    // A position's scratch word exists only if its 32-position tile holds a match (tile flags); the other tiles are literals
    // straight from the raw bytes.
    {
        const uint32_t *gflags = m + scr_flag_offset(n);
        S.tflags[lane] = gflags[lane];
        S.tflags[lane + 32u] = gflags[lane + 32u];
    }
    __syncwarp();
#define ENC_WORD_AT(x_) ((x_) < n ? (((S.tflags[(x_) >> 10] >> (((x_) >> 5) & 31u)) & 1u) ? m[(x_)] : ((uint32_t) src[(x_)] << 24)) : 0u)
    // marks of stretches in which no step starts (resp. into which none reaches first) stay "unset" and are resolved later — the
    // last, partial stretch of a chunk is the usual case
    for (uint32_t i = lane; i < 66u; i += 32u) {
        S.kb_tok[i] = 0xffffu;
        S.kb_end[i] = 0xffffu;
    }
    __syncwarp();
    uint32_t ntok = 0;
    uint32_t last_kb = 0xffffffffu, last_kbe = 0xffffffffu;
    uint64_t extra_bits = 0; // length + distance extra bits of all matches (lane-partial, summed later)
    uint32_t m0 = ENC_WORD_AT(lane);
    for (uint32_t p = 0; p < n;) {
        uint32_t q = p + lane;
        // token boundaries the stored regions can use: a step looks at positions [p, p + 32)
        if ((p >> 10) != last_kb) {
            last_kb = p >> 10;
            if (lane == 0) {
                S.kb_tok[last_kb] = (uint16_t) ntok;
                S.kb_pos[last_kb] = (uint16_t) p;
            }
        }
        if (((p + 31u) >> 10) != last_kbe) {
            last_kbe = (p + 31u) >> 10;
            if (lane == 0) {
                S.kb_end[last_kbe] = (uint16_t) ntok;
                S.kb_endpos[last_kbe] = (uint16_t) p;
            }
        }
        // the window after this one, fetched before it is known to be needed: when the window holds no match that leaves
        // it (J0 == 32: every literal-only stretch) the next step starts without waiting on a dependent load
        const uint32_t mnx = ENC_WORD_AT(q + 32u);
        // quiet step: no tile under [p, p + 32) holds a match, so all 32 positions are literals and the path through them needs
        // no pointer doubling (the bodies of JPEG-like files, noise in general: 70 % of the steps of config C2)
        {
            const uint32_t ta = p >> 5, tb = (p + 31u) >> 5;
            if (p + 32u <= n && !(((S.tflags[ta >> 5] >> (ta & 31u)) | (S.tflags[tb >> 5] >> (tb & 31u))) & 1u)) {
                atomicAdd(&S.freq[m0 >> 24], 1u);
                m[ntok + lane] = m0 & 0xff000000u;
                ntok += 32u;
                p += 32u;
                m0 = mnx;
                continue;
            }
        }
        uint32_t m1 = __shfl_down_sync(ZWZ_FULL, m0, 1);
        const uint32_t mfirst = __shfl_sync(ZWZ_FULL, mnx, 0);
        if (lane == 31u) m1 = mfirst;
        if (lane < 4u && p + 384u + 32u * lane < n) prefetch_l2(m + p + 384u + 32u * lane); // pull the scratch ahead of the parse into L2 (it sits in HBM)
        uint32_t len0 = tok_len(m0), len1 = tok_len(m1);
        bool take = len0 >= ZWZ_MIN_MATCH && !(len1 > len0);
        uint32_t J = lane + (take ? len0 : 1u);
        uint32_t R = 1u << lane;
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            int from = J < 32u ? (int) J : (int) lane;
            uint32_t Rj = __shfl_sync(ZWZ_FULL, R, from);
            uint32_t Jj = __shfl_sync(ZWZ_FULL, J, from);
            if (J < 32u) {
                R |= Rj;
                J = Jj;
            }
        }
        uint32_t R0 = __shfl_sync(ZWZ_FULL, R, 0);
        uint32_t J0 = __shfl_sync(ZWZ_FULL, J, 0);
        bool marked = ((R0 >> lane) & 1u) && q < n;
        unsigned tm = __ballot_sync(ZWZ_FULL, marked);
        if (marked) {
            uint32_t tok;
            if (take) {
                tok = m0;
                uint32_t ls, le, lv, ds, de, dv;
                len_symbol(len0, ls, le, lv);
                dist_symbol(tok_dist(m0), ds, de, dv);
                atomicAdd(&S.freq[ls], 1u);
                atomicAdd(&S.freq[ZWZ_DE_DOFF + ds], 1u);
                extra_bits += le + de;
            } else {
                tok = m0 & 0xff000000u; // literal: the byte travels in the scratch word, no second load
                atomicAdd(&S.freq[m0 >> 24], 1u);
            }
            m[ntok + (uint32_t) __popc(tm & ((1u << lane) - 1u))] = tok;
        }
        ntok += (uint32_t) __popc(tm);
        p += J0;
        if (J0 == 32u) m0 = mnx;
        else m0 = ENC_WORD_AT(p + lane);
    }
#undef ENC_WORD_AT
    if (lane == 0) S.freq[256] += 1u; // end of block
    extra_bits = warp_sum64(extra_bits);
    __syncwarp();

    // ---------------- near-incompressible chunks are STORED ----------------
    // Policy: a chunk is stored when the best Huffman encoding would save less than n/256 bytes (0.4 %). zlib would still
    // emit a dynamic block there (it takes any gain, e.g. 7 002 vs 7 011 bytes on a JPEG-like file), but such a block costs
    // one Huffman symbol per byte to decode — for our inflate and for the reference's zlib alike — and buys nothing.
    // First an exact-safe shortcut: no prefix code beats the empirical entropy, so if even the entropy bound cannot save
    // n/256 bytes the three Huffman constructions below are skipped altogether.
    // The estimates are compared with the zlib-wrapped stored size in every format, so that the choice (and the body) does not
    // depend on the wrapper; the 65 535-byte record limit applies to zlib streams only.
    const uint32_t sto_bytes = n + 5u + (piece ? 5u : enc_wrap_bytes(fmt));
    const uint32_t zsto_bytes = n + 11u;
    const uint32_t sto_slack = n >> 8;
    bool force_stored = false;
    {
        float nl = 0.f, nd = 0.f, hl_bits = 0.f;
        uint32_t nused = 0;
        for (uint32_t s = lane; s < 320u; s += 32u) {
            float f = (float) S.freq[s];
            if (s < ZWZ_DE_DOFF) nl += f; else nd += f;
            nused += f > 0.f ? 1u : 0u;
        }
        nused = warp_sum(nused);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            nl += __shfl_xor_sync(ZWZ_FULL, nl, d);
            nd += __shfl_xor_sync(ZWZ_FULL, nd, d);
        }
        for (uint32_t s = lane; s < 320u; s += 32u) {
            float f = (float) S.freq[s];
            if (f > 0.f) hl_bits += f * (zwz_log2f(s < ZWZ_DE_DOFF ? nl : nd) - zwz_log2f(f));
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) hl_bits += __shfl_xor_sync(ZWZ_FULL, hl_bits, d);
        // + zlib wrapper and block header, + ~2 bits per used symbol for a dynamic header (a small random sample sits ~23
        // bytes under 8 bits/byte of empirical entropy; its code-length header costs several times that)
        float bound_bytes = (hl_bits + (float) extra_bits) * 0.125f + 7.f + (float) (nused >> 2);
        force_stored = bound_bytes * 0.9995f >= (float) zsto_bytes - (float) sto_slack && (fmt != ZWZ_FORMAT_ZLIB || zsto_bytes <= ZWZ_CHUNK) &&
                       n >= 512u;
    }
    if (force_stored) {
        uint32_t l0 = piece ? enc_stored_piece(out, src, n) : enc_stored_stream(out, src, n, job.adler[c], fmt, dictid);
        if (lane == 0) {
            job.res[4u * c + 0u] = l0;
            job.res[4u * c + 1u] = 0u;
            job.res[4u * c + 2u] = n;
            job.res[4u * c + 3u] = 0u;
        }
        return;
    }

    // ---------------- blocks ----------------
    // Stored regions first: a stretch of >= 256 literal tokens whose bytes are (nearly) uniformly distributed — the body of a
    // JPEG-like file behind its structured header — goes out as a STORED block between the Huffman blocks of its neighbours.
    // zlib would code it with 8-bit literals (nothing gained), pay for it in every decoder (one Huffman symbol per byte instead
    // of a copy), and let it flatten the neighbours' code lengths. Then, per remaining token range: base blocks of
    // ZWZ_DE_BASE tokens are merged left to right while one Huffman code over the union is estimated (empirical entropy + a
    // header estimate) to cost no more than two separate ones; a merged run becomes one DEFLATE block. zlib cuts every 16 383
    // symbols regardless of content; adapting the cut is worth several percent on data whose statistics drift (bitmap-like),
    // nothing on homogeneous text.
    const uint32_t cap_words = ((n + ZWZ_DEFLATE_MARGIN + 15u) & ~15u) >> 2; // zwz_deflate_bound(n) / 4
    BitSink k;
    sink_init(S, k, (uint32_t *) out, cap_words);
    enc_wrap_head(&k, fmt, dictid);
    __syncwarp();
    const uint32_t nreg = enc_find_stored_regions(m, n, ntok);
    if (nreg == 0u) {
        enc_emit_range(&k, m, 0, ntok, extra_bits, !piece, true); // S.freq still holds the whole-chunk histogram from the parse
    } else {
        uint32_t t = 0;
        for (uint32_t r = 0; r < nreg; ++r) {
            const uint32_t r0 = S.region[4u * r], r1 = S.region[4u * r + 1u], p0 = S.region[4u * r + 2u], p1 = S.region[4u * r + 3u];
            if (r0 > t) enc_emit_range(&k, m, t, r0, 0, false, false);
            enc_emit_stored_block(&k, src + p0, p1 - p0, !piece && r1 == ntok);
            t = r1;
        }
        if (t < ntok) enc_emit_range(&k, m, t, ntok, 0, !piece, false);
    }
    const uint32_t adler = job.adler[c];
    if (piece) enc_piece_tail(&k);
    else enc_wrap_tail(&k, fmt, adler, n);
    const uint32_t huff_bytes = sink_finish(S, k);
    __syncwarp();

    uint32_t len0 = huff_bytes, len1 = 0, raw0 = n, btype = 2u;
    if (sto_bytes <= huff_bytes + sto_slack || (fmt == ZWZ_FORMAT_ZLIB && huff_bytes > ZWZ_CHUNK) || huff_bytes > cap_words * 4u) { // see the policy above
        btype = 0u;
        if (fmt == ZWZ_FORMAT_ZLIB && sto_bytes > ZWZ_CHUNK) {
            // split rule: two stored streams over the halves (each needs its own Adler-32)
            raw0 = 32768u;
            uint32_t a0 = enc_adler_global(src, raw0);
            uint32_t a1 = enc_adler_global(src + raw0, n - raw0);
            len0 = enc_stored_stream(out, src, raw0, a0, ZWZ_FORMAT_ZLIB, 0u);
            len1 = enc_stored_stream(out + len0, src + raw0, n - raw0, a1, ZWZ_FORMAT_ZLIB, 0u);
        } else {
            len0 = piece ? enc_stored_piece(out, src, n) : enc_stored_stream(out, src, n, adler, fmt, dictid);
        }
    }
    if (lane == 0) {
        job.res[4u * c + 0u] = len0;
        job.res[4u * c + 1u] = len1;
        job.res[4u * c + 2u] = raw0;
        job.res[4u * c + 3u] = btype;
    }
}

// Persistent warps pulling chunks from a global counter (same reason as inflate_kernel: no idle warps behind a long chunk).
// DICT: some chunks have a preset dictionary (job.dict): their zlib header names it. DICT = false is the kernel of the calls without.
template <bool DICT = false>
ZWZ_KERNEL __launch_bounds__(ZWZ_DE_WARPS * 32) deflate_encode_kernel(DeflateJob job, uint32_t *work_counter) {
    for (;;) {
        uint32_t c = 0;
        if (lane_id() == 0) c = atomicAdd(work_counter, 1u);
        c = __shfl_sync(ZWZ_FULL, c, 0);
        if (c >= job.n) break;
        enc_chunk<DICT>(enc_smem(), job, c);
        __syncwarp();
    }
}

} // namespace zwz
