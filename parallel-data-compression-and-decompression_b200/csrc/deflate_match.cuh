// deflate_match.cuh — LZ77 match finding for <= 65 535-byte chunks, everything in shared memory.
//
// First half of the replacement for zlib's deflate() at compression.cpp:119-134 (the second half is deflate_encode.cuh).
//
// Per chunk (persistent CTAs, chunks handed out by an atomic counter):
//   1. the chunk is staged HBM -> shared memory with one bulk asynchronous copy (cp.async.bulk + mbarrier, SASS UBLKCP),
//      a 16-byte aligned superset of the chunk; the chunk itself starts at byte `skew` of the staging buffer;
//   2. all threads hash every position (3-byte multiplicative hash) into prev[] in parallel, and the positions are
//      split — stably, so each list stays sorted by position — into one list per warp by the top bits of the hash
//      (ballot-based multi-split: per-warp counts, one small scan, scatter to the chunk's scratch in HBM/L2);
//   3. every warp turns ITS list into EXACT hash chains, 32 positions per step: every lane links to the old head and
//      becomes the new head; lanes sharing a hash inside the step are found by reading the head back and repaired with
//      ballot + shuffle (lowest lane keeps the old head, the others link to the nearest earlier lane, the highest stays
//      head). Lists cover disjoint hash ranges, so the builders share head[] without ever touching the same entry — the
//      serial insertion order a hash chain needs is kept per hash value, and the chunk-long serial loop of a
//      single-builder design (measured: it was the kernel's critical path) becomes NW loops 1/NW as long;
//   4. all warps pull 32-position tiles and, one lane per position, walk the chain:
//      byte checks around the current best length reject most candidates, survivors are compared 4 bytes at a time on
//      funnel-shifted aligned words; `depth` candidates at most, stop at `nice` bytes;
//   5. the best (length, distance) of EVERY position, together with the byte at that position, goes to the chunk's scratch
//      in HBM (4 bytes per input byte, coalesced); the parse in deflate_encode.cuh picks the path through them;
//   6. Adler-32 of the chunk is reduced from shared memory while it is there.
//
// Four size classes so that small chunks do not leave an SM to one serial chain builder (config C2 is 370 000 chunks of
// ~6.7 KB): the class fixes the shared-memory footprint and with it how many CTAs — each with its own builder warp — an SM
// holds.
//      class   chunk bytes   threads   smem/CTA   CTAs/SM   hash bits
//        0       <=  8 192      256     ~33 KB       6         12
//        1       <= 16 384      512     ~66 KB       3         13
//        2       <= 32 768      512    ~114 KB       2         13
//        3       <= 65 535     1024    ~227 KB       1         14
// Algorithmic HBM bytes per chunk for the roofline: N_raw read (the 4 N_raw scratch write is traffic of this design, not of
// the algorithm — reported separately in DESIGN.md).
#pragma once
#include "zwz_common.cuh"

namespace zwz {

#define ZWZ_DM_NIL 0xffffu
#ifndef ZWZ_DM_NOISE_BITS
#define ZWZ_DM_NOISE_BITS 7.7f // order-0 entropy (bits per byte, over 1 024 bytes) above which a stretch is not searched
#endif

#ifdef ZWZ_EMU
// test-only counters of the emulator build: [0] stretches left out as noise, [1] chunks whose noise candidates were kept because
// they repeat, [2] chunks seen
static uint64_t g_dm_stats[4];
extern "C" void zwz_emu_match_stats(uint64_t *out, int reset) {
    for (int i = 0; i < 4; ++i) {
        out[i] = g_dm_stats[i];
        if (reset) g_dm_stats[i] = 0;
    }
}
#define ZWZ_DM_STAT(i, v) do { g_dm_stats[i] += (v); } while (0)
// the final skip mask of each chunk of the last call (chunk index < 65 536), for the tests that restate the noise test
static uint64_t g_dm_skip[1u << 16];
extern "C" void zwz_emu_match_skipmasks(uint64_t *out, uint32_t n) {
    for (uint32_t i = 0; i < n && i < (1u << 16); ++i) out[i] = g_dm_skip[i];
}
#define ZWZ_DM_SKIP(c, m) do { if ((c) < (1u << 16)) g_dm_skip[c] = (m); } while (0)
#else
#define ZWZ_DM_STAT(i, v) do { } while (0)
#define ZWZ_DM_SKIP(c, m) do { } while (0)
#endif

// Phase clocks (nvcc build with -DZWZ_DM_PHASE_CLOCKS only, tools/match_phases.py): thread 0 of every CTA adds the clock64()
// cycles between the CTA barriers that close the phases of a chunk, per size class; [cls][ZWZ_DM_NPHASE] counts the chunks.
#define ZWZ_DM_NPHASE 10
#if defined(ZWZ_DM_PHASE_CLOCKS) && !defined(ZWZ_EMU)
__device__ unsigned long long g_dm_phase_clk[4][ZWZ_DM_NPHASE + 1];
extern "C" int zwz_dm_phase_clocks(unsigned long long *out, int reset) {
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(out, g_dm_phase_clk, sizeof(g_dm_phase_clk)) != cudaSuccess) return 1;
    static const unsigned long long zero[4][ZWZ_DM_NPHASE + 1] = {};
    return reset && cudaMemcpyToSymbol(g_dm_phase_clk, zero, sizeof(zero)) != cudaSuccess ? 1 : 0;
}
#define ZWZ_DM_CLK_DECL uint32_t dm_clk[ZWZ_DM_NPHASE + 1] = {}; long long dm_t0 = clock64();
#define ZWZ_DM_CLK(k) do { if (tid == 0) { const long long t = clock64(); dm_clk[k] += (uint32_t) (t - dm_t0); dm_clk[ZWZ_DM_NPHASE] += (k == 0); dm_t0 = t; } } while (0)
#define ZWZ_DM_CLK_FLUSH() do { if (tid == 0) for (int k = 0; k <= ZWZ_DM_NPHASE; ++k) atomicAdd(&g_dm_phase_clk[CLS][k], (unsigned long long) dm_clk[k]); } while (0)
#else
#define ZWZ_DM_CLK_DECL
#define ZWZ_DM_CLK(k) do { } while (0)
#define ZWZ_DM_CLK_FLUSH() do { } while (0)
#endif

template <int CLS> struct MatchClass;
template <> struct MatchClass<0> {
    static constexpr uint32_t kCap = 8192, kThreads = 256, kHBits = 12, kData = 8192 + 64, kListBits = 3, kCtasPerSm = 6;
    static constexpr uint32_t kPrevBytes = ((kCap + 31u) & ~31u) * 2u, kSmem = kData + kPrevBytes + (2u << kHBits) + 1024u + 2u * 8u * 8u;
};
template <> struct MatchClass<1> {
    static constexpr uint32_t kCap = 16384, kThreads = 512, kHBits = 13, kData = 16384 + 64, kListBits = 4, kCtasPerSm = 3;
    static constexpr uint32_t kPrevBytes = ((kCap + 31u) & ~31u) * 2u, kSmem = kData + kPrevBytes + (2u << kHBits) + 1024u + 2u * 16u * 16u;
};
template <> struct MatchClass<2> {
    // 31 744, not 32 768: 2 x (smem + 1 KB) must fit the SM's 228 KB for two resident CTAs (115 712 B each at most)
    static constexpr uint32_t kCap = 31744, kThreads = 512, kHBits = 13, kData = 31744 + 64, kListBits = 4, kCtasPerSm = 2;
    static constexpr uint32_t kPrevBytes = ((kCap + 31u) & ~31u) * 2u, kSmem = kData + kPrevBytes + (2u << kHBits) + 1024u + 2u * 16u * 16u;
};
template <> struct MatchClass<3> {
    static constexpr uint32_t kCap = 65535, kThreads = 1024, kHBits = 14, kData = 65600, kListBits = 5, kCtasPerSm = 1;
    static constexpr uint32_t kPrevBytes = ((kCap + 31u) & ~31u) * 2u, kSmem = kData + kPrevBytes + (2u << kHBits) + 640u + 2u * 32u * 32u;
};

// control block (after the tables); cnt[NW][NW] u16 follows it
struct MatchCtl {
    unsigned long long mbar;   // mbarrier for the bulk copy
    uint32_t cur_work;
    uint32_t next_tile;        // search: the next of the searched tiles to hand out
    uint32_t nmatch;           // positions of this chunk that found a match
    uint32_t skip[2];          // bit k: the 1 024-byte stretch k looks like noise and is left out of the search
    uint32_t coll;             // repeated 4-byte windows among the noise candidates
    uint32_t coll2;            // candidate windows that also occur (by hash) among the other positions
    uint32_t set2;             // bits set in the other positions' bit set
    uint32_t base[33];         // list k = entries [base[k], base[k+1]) of the position list
    uint8_t slist[64];         // the stretches that are searched, in order
    uint32_t adler_a[32], adler_b[32], adler_len[32];
};
static_assert(sizeof(MatchCtl) <= 640, "MatchCtl must fit its slot");
static_assert(MatchClass<0>::kPrevBytes >= (2u << MatchClass<0>::kHBits) && MatchClass<1>::kPrevBytes >= (2u << MatchClass<1>::kHBits) &&
                  MatchClass<2>::kPrevBytes >= (2u << MatchClass<2>::kHBits) && MatchClass<3>::kPrevBytes >= (2u << MatchClass<3>::kHBits),
              "the second bit set of the noise test lives in prev[]");
static_assert(2u * (MatchClass<2>::kSmem + 1024u) <= 228u * 1024u && 3u * (MatchClass<1>::kSmem + 1024u) <= 228u * 1024u &&
                  6u * (MatchClass<0>::kSmem + 1024u) <= 228u * 1024u,
              "resident CTAs per SM assumed by the launch grids");

// scratch layout of one chunk (uint32 units): [0, A) best match per position, then tokens in place (deflate_encode.cuh);
// [A, A + B) the hash-partitioned position lists (u16) used only inside lz_match_kernel
ZWZ_DEV uint32_t dm_scratch_match_words(uint32_t n) { return scr_match_words(n); }

template <int HBITS> ZWZ_DEV uint32_t dm_hash3(uint32_t b0, uint32_t b1, uint32_t b2) {
    uint32_t v = b0 | (b1 << 8) | (b2 << 16);
    return (v * 0x9E3779B1u) >> (32 - HBITS);
}

#ifndef ZWZ_EMU
ZWZ_DEV uint32_t dm_smem_addr(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
ZWZ_DEV void dm_mbar_init(unsigned long long *bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dm_smem_addr(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
ZWZ_DEV void dm_bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    // generic-proxy accesses to this smem (previous chunk) are ordered before the async-proxy write
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dm_smem_addr(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dm_smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(dm_smem_addr(bar))
                 : "memory");
}
ZWZ_DEV void dm_mbar_wait(unsigned long long *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(dm_smem_addr(bar)), "r"(parity)
                     : "memory");
    }
}
#endif

ZWZ_DEV uint32_t sD_of(const unsigned char *smem, uint32_t skew) { return smem_addr(smem) + skew; }

// DICT: chunks with a preset dictionary (job.dict) go on searching in the dictionary's chains once their own chain is exhausted
// (step 6). DICT = false is the kernel of the calls without dictionaries.
template <int CLS, bool DICT = false>
ZWZ_KERNEL __launch_bounds__(MatchClass<CLS>::kThreads, MatchClass<CLS>::kCtasPerSm) lz_match_kernel(DeflateJob job, const uint32_t *__restrict__ order, uint32_t n_work,
                                                                         uint32_t *work_counter) {
    constexpr uint32_t T = MatchClass<CLS>::kThreads, HB = MatchClass<CLS>::kHBits, DATA = MatchClass<CLS>::kData;
    constexpr uint32_t NW = T / 32u, LB = MatchClass<CLS>::kListBits;
    static_assert((1u << LB) == NW, "one position list per warp");
    ZWZ_DYN_SMEM(smem);
    const uint32_t *dataw = (const uint32_t *) smem;                                  // chunk bytes as aligned words
    uint16_t *prev = (uint16_t *) (smem + DATA);
    uint16_t *head = (uint16_t *) (smem + DATA + MatchClass<CLS>::kPrevBytes);
    MatchCtl *ctl = (MatchCtl *) (smem + DATA + MatchClass<CLS>::kPrevBytes + (2u << HB));
    uint16_t *cnt = (uint16_t *) ((unsigned char *) ctl + 640);                       // [NW][NW]: running list offsets per (warp, list)
    const uint8_t *datab = (const uint8_t *) smem;
    const unsigned tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    const unsigned lt = (1u << lane) - 1u;
    uint32_t parity = 0;

#ifndef ZWZ_EMU
    if (tid == 0) dm_mbar_init(&ctl->mbar);
#endif
    __syncthreads();
    ZWZ_DM_CLK_DECL

    for (;;) {
        if (tid == 0) ctl->cur_work = atomicAdd(work_counter, 1u);
        __syncthreads();
        const uint32_t w = ctl->cur_work;
        if (w >= n_work) {
            ZWZ_DM_CLK_FLUSH();
            break;
        }
        const uint32_t c = order[w];
        const uint32_t n = job.raw_len[c];
        const uint8_t *src = job.raw + job.raw_off[c];
        const uint32_t skew = (uint32_t) ((uintptr_t) src & 15u);
        const uint32_t stage_bytes = (skew + n + 15u) & ~15u;
        // the chunk's preset dictionary (CTA-uniform): its record in the dictionary arena and its window length, 0 = none
        const uint8_t *drec = nullptr;
        uint32_t dwl = 0;
        if (DICT) {
            const uint32_t di = job.dict.idx[c];
            if (di != ZWZ_NO_DICT) {
                drec = job.dict.arena + (size_t) di * ZWZ_DICT_STRIDE;
                dwl = job.dict.wlen[di];
            }
        }

        // ---- 1. stage the chunk ----
#ifndef ZWZ_EMU
        if (tid == 0 && stage_bytes) dm_bulk_g2s(smem, src - skew, stage_bytes, &ctl->mbar);
#else
        for (uint32_t i = tid; i < skew + n; i += T) smem[i] = i < skew ? 0 : src[i - skew];
#endif
        if (tid == 0) {
            ctl->next_tile = 0;
            ctl->nmatch = 0;
            ctl->skip[0] = 0;
            ctl->skip[1] = 0;
        }
#ifndef ZWZ_EMU
        if (stage_bytes) dm_mbar_wait(&ctl->mbar, parity);
        parity ^= (stage_bytes != 0u);
#endif
        __syncthreads();
        ZWZ_DM_CLK(0);
        // bytes past the end take part in 4-byte compares: make them deterministic (the final clamp to `maxlen` makes
        // their value irrelevant for the result)
        if (tid < 32u) smem[skew + n + tid] = 0;

        // ---- 1b. stretches of noise are left out ----
        // A 1 024-byte stretch whose bytes are (nearly) uniformly distributed — the entropy-coded body of a JPEG, anything
        // compressed or encrypted — holds no match worth a token, and everything below would be spent on proving that: its
        // positions are neither hashed nor chained nor searched (LZ4 and zstd step over such data with a growing stride; here
        // the decision is made per stretch, up front). Two tests, both in the (not yet initialised) head[] table:
        //   (1) per stretch, one warp: byte histogram in the warp's 1 KB slice; order-0 entropy of 1 024 uniformly random bytes
        //       is 7.82 +- 0.02 bits, of text ~4.5, of the structured binary classes of the corpus < 7: candidates lie above
        //       ZWZ_DM_NOISE_BITS;
        //   (2) over all candidates of the chunk: a flat histogram does not rule out repeats (a permutation table stored four
        //       times, a random block stored twice), so every 4-byte window of the candidates is hashed into a bit set
        //       (table size = 4-8 bits per position) and the windows that find their bit already set are counted. Noise of
        //       n_c positions in m bits collides n_c^2 / 2m times (+- its square root); n_c / 64 + 48 more than that and NO
        //       stretch is left out. The candidates' windows are also looked up among the windows of all other positions (below).
        // What this gives up: repeats that cover less than ~2 % of the noise (zlib would find them). The encoder emits these
        // stretches as stored blocks (deflate_encode.cuh: quiet stretches). With a preset dictionary such a stretch is not
        // searched against the dictionary either: a copy of dictionary bytes inside noise goes out as literals.
        uint64_t cand, skipmask; // bit k: stretch k passed the histogram test / is left out
        {
            uint32_t *hist = (uint32_t *) head + wid * 256u;
            const uint32_t nfull = n >> 10; // the partial last stretch is always searched
            for (uint32_t kb = wid; kb < nfull; kb += NW) {
                const uint32_t w0 = (skew + (kb << 10)) >> 2; // aligned words: up to 3 bytes of the neighbour do not matter here
                // cheap first look (text never gets past it): of 128 sampled bytes of noise, 64 +- 6 have their top bit set
                {
                    const uint32_t sv = dataw[w0 + 8u * lane] & 0x80808080u;
                    const uint32_t tops = (uint32_t) (__popc(__ballot_sync(ZWZ_FULL, sv & 0x80u)) + __popc(__ballot_sync(ZWZ_FULL, sv & 0x8000u)) +
                                                      __popc(__ballot_sync(ZWZ_FULL, sv & 0x800000u)) + __popc(__ballot_sync(ZWZ_FULL, sv & 0x80000000u)));
                    if (tops < 40u || tops > 88u) continue;
                }
#pragma unroll
                for (uint32_t j = 0; j < 8u; ++j) hist[lane + 32u * j] = 0u;
                __syncwarp();
#pragma unroll
                for (uint32_t j = 0; j < 8u; ++j) {
                    const uint32_t wv = dataw[w0 + lane + 32u * j];
                    atomicAdd(&hist[wv & 0xffu], 1u);
                    atomicAdd(&hist[(wv >> 8) & 0xffu], 1u);
                    atomicAdd(&hist[(wv >> 16) & 0xffu], 1u);
                    atomicAdd(&hist[wv >> 24], 1u);
                }
                __syncwarp();
                float sum = 0.f; // sum of c * log2(c)
#pragma unroll
                for (uint32_t j = 0; j < 8u; ++j) {
                    const float cf = (float) hist[lane + 32u * j];
                    if (cf > 1.f) sum += cf * zwz_log2f(cf);
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(ZWZ_FULL, sum, d);
                // H = 10 - sum / 1024 > ZWZ_DM_NOISE_BITS
                if (lane == 0 && sum < (10.f - ZWZ_DM_NOISE_BITS) * 1024.f) atomicOr(&ctl->skip[kb >> 5], 1u << (kb & 31u));
                __syncwarp();
            }
            __syncthreads();
            ZWZ_DM_CLK(1);
            cand = (uint64_t) ctl->skip[0] | ((uint64_t) ctl->skip[1] << 32);
            skipmask = cand;
            if (cand) { // CTA-uniform
                // (2) runs stretch by stretch: its three counts do not depend on the order of the windows, so neither does
                // the verdict. The histograms are done with (barrier above): both bit sets are cleared at once.
                constexpr uint32_t BB = HB + 4u; // head[] is 2 << HB bytes = 1 << BB bits
                uint32_t *bits = (uint32_t *) head;
                uint32_t *bits2 = (uint32_t *) prev; // >= as large as head[] in every class
                for (uint32_t i = tid; i < (1u << BB) / 32u; i += T) {
                    bits[i] = 0u;
                    bits2[i] = 0u;
                }
                if (tid == 0) {
                    ctl->coll = 0;
                    ctl->coll2 = 0;
                    ctl->set2 = 0;
                }
                __syncthreads();
                const uint32_t sD0 = sD_of(smem, skew);
                uint32_t mine = 0;
                for (uint64_t cm = cand; cm; cm &= cm - 1ull) {
                    const uint32_t q0 = (uint32_t) (__ffsll((long long) cm) - 1) << 10;
                    for (uint32_t j = wid; j < 32u; j += NW) {
                        const uint32_t h = (lds32u(sD0 + q0 + j * 32u + lane) * 0x9E3779B1u) >> (32u - BB);
                        const uint32_t old = atomicOr(&bits[h >> 5], 1u << (h & 31u));
                        mine += (uint32_t) __popc(__ballot_sync(ZWZ_FULL, (old >> (h & 31u)) & 1u));
                    }
                }
                if (lane == 0 && mine) atomicAdd(&ctl->coll, mine);
                // ... and against the OTHER positions: the copy of PART of a noise stretch need not be a candidate itself (its
                // histogram is narrower), and bytes that are not inserted cannot be found by anyone. The other positions' windows
                // set a second bit set (in the prev[] area, unused so far), the candidates' windows are looked up in it: noise
                // windows are all different, so the hits are independent — n_c * (bits set) / m of them by chance (the
                // other way round, text windows looked up in the noise set, one unlucky window repeats its hit a hundred times).
                // This set is built in the same phase as the first: the two sets are disjoint.
                const uint32_t nh = n >= 3u ? n - 2u : 0u;
                uint32_t fresh = 0; // bits this warp was the first to set: the set's load decides what chance looks like
                for (uint32_t q0 = 0; q0 < nh; q0 += 1024u) {
                    if ((cand >> (q0 >> 10)) & 1ull) continue;
                    for (uint32_t j = wid; j < 32u && q0 + j * 32u < nh; j += NW) {
                        const uint32_t q = q0 + j * 32u + lane;
                        const uint32_t h = (lds32u(sD0 + q) * 0x9E3779B1u) >> (32u - BB);
                        const uint32_t old2 = q < nh ? atomicOr(&bits2[h >> 5], 1u << (h & 31u)) : 0xffffffffu;
                        fresh += (uint32_t) __popc(__ballot_sync(ZWZ_FULL, !((old2 >> (h & 31u)) & 1u)));
                    }
                }
                if (lane == 0 && fresh) atomicAdd(&ctl->set2, fresh);
                __syncthreads();
                uint32_t hits = 0;
                for (uint64_t cm = cand; cm; cm &= cm - 1ull) {
                    const uint32_t q0 = (uint32_t) (__ffsll((long long) cm) - 1) << 10;
                    for (uint32_t j = wid; j < 32u; j += NW) {
                        const uint32_t h = (lds32u(sD0 + q0 + j * 32u + lane) * 0x9E3779B1u) >> (32u - BB);
                        hits += (uint32_t) __popc(__ballot_sync(ZWZ_FULL, (bits2[h >> 5] >> (h & 31u)) & 1u));
                    }
                }
                if (lane == 0 && hits) atomicAdd(&ctl->coll2, hits);
                __syncthreads();
                // every thread reaches the same verdict from the same counts; bits[] (in head[]) is no longer read
                const uint32_t nc = (uint32_t) __popcll((long long) cand) << 10;
                const uint32_t allowed = (uint32_t) (((uint64_t) nc * nc) >> (BB + 1u)) + (nc >> 6) + 48u;
                const uint32_t allowed2 = (uint32_t) (((uint64_t) ctl->set2 * nc) >> BB) + (nc >> 6) + 48u; // chance: n_c * (bits set) / m
                if (ctl->coll > allowed || ctl->coll2 > allowed2) {
                    skipmask = 0;
                    if (tid == 0) ZWZ_DM_STAT(1, 1);
                }
            }
        }
        ZWZ_DM_CLK(2);
        for (uint32_t i = tid; i < (1u << HB) / 2u; i += T) ((uint32_t *) head)[i] = 0xffffffffu;
        // the stretches that are searched, in order: step / tile i of the searched ones is (slist[i >> 5] << 5) | (i & 31)
        const uint32_t nstr = (n + 1023u) >> 10;
        if (wid == 0) {
#pragma unroll
            for (uint32_t k = 0; k < 2u; ++k) {
                const uint32_t sidx = 32u * k + lane;
                const bool keep = sidx < nstr && !((skipmask >> sidx) & 1ull);
                const unsigned km = __ballot_sync(ZWZ_FULL, keep);
                if (keep) ctl->slist[(k ? (uint32_t) __popc((unsigned) ~skipmask) : 0u) + (uint32_t) __popc(km & lt)] = (uint8_t) sidx;
            }
        }
        if (tid == 0) {
            ZWZ_DM_STAT(0, (uint64_t) __popcll((long long) skipmask));
            ZWZ_DM_STAT(2, 1);
            ZWZ_DM_SKIP(c, skipmask);
        }
        __syncthreads();
        ZWZ_DM_CLK(3);

        uint32_t *mout = job.scratch + job.scr_off[c];
        uint16_t *list = (uint16_t *) (mout + dm_scratch_match_words(n));
        const uint32_t nhash = n >= 3u ? n - 2u : 0u; // positions that own a 3-byte hash
        const uint32_t nskip = 32u * (uint32_t) __popcll((long long) skipmask);
        const uint32_t ntiles = ((n + 31u) >> 5) - nskip;  // searched tiles
        const uint32_t nsteps = ((nhash + 31u) >> 5) - nskip; // searched hash steps (noise stretches are whole steps < nhash)
        const uint32_t spw = (nsteps + NW - 1u) / NW;  // searched steps per warp: warp w owns [w*spw, (w+1)*spw)
        const uint32_t s_lo = wid * spw, s_hi = min(s_lo + spw, nsteps);

        const uint32_t sD = smem_addr(smem) + skew; // shared address of chunk byte 0
        const uint32_t sP = smem_addr(prev);        // prev[0]
        const uint32_t sH = smem_addr(head);        // head[0]
        const uint8_t *slist = ctl->slist;
        // ---- 2. hash every position; count, per warp, how many of its positions fall in each of the NW hash ranges ----
        // The counts stay in registers: from the LB ballots of the range bits, lane b picks out the positions of the step that
        // fall in list b. The scatter below uses the same ballots for the rank of each position inside its list, so ranks follow
        // lane (= position) order and the lists come out sorted by position.
        {
            uint32_t my = 0;
            for (uint32_t i = s_lo; i < s_hi; ++i) {
                const uint32_t p = (((uint32_t) slist[i >> 5] << 5) | (i & 31u)) * 32u + lane;
                const bool valid = p < nhash;
                uint32_t h = 0;
                if (valid) {
                    uint32_t v = lds32u(sD + p);
                    h = dm_hash3<HB>(v & 0xffu, (v >> 8) & 0xffu, (v >> 16) & 0xffu);
                    sts16(sP + 2u * p, h); // prev[p] holds hash(p) until the builder replaces it by the link
                }
                const uint32_t b = h >> (HB - LB);
                unsigned ml = __ballot_sync(ZWZ_FULL, valid);
#pragma unroll
                for (uint32_t k = 0; k < LB; ++k) {
                    const unsigned v = __ballot_sync(ZWZ_FULL, (b >> k) & 1u);
                    ml &= ((lane >> k) & 1u) ? v : ~v;
                }
                my += (uint32_t) __popc(ml);
            }
            if (lane < NW) cnt[wid * NW + lane] = (uint16_t) my;
        }
        __syncthreads();
        ZWZ_DM_CLK(4);
        // ---- 3. offsets: list b = [base[b], base[b+1]), inside it warp 0's positions first, then warp 1's, ... ----
        // Every warp scans the NW x NW counts itself: lane b ends up with where this warp's next position of list b goes.
        uint32_t off;
        {
            uint32_t before = 0, total = 0;
            if (lane < NW) {
                for (uint32_t ww = 0; ww < NW; ++ww) {
                    const uint32_t t = cnt[ww * NW + lane];
                    before += ww < wid ? t : 0u;
                    total += t;
                }
            }
            const uint32_t incl = warp_incl_scan(total);
            off = incl - total + before;
            if (wid == 0) {
                if (lane < NW) ctl->base[lane] = incl - total;
                if (lane == NW - 1u) ctl->base[NW] = incl;
            }
        }
        ZWZ_DM_CLK(5);
        // ---- 4. scatter positions into the lists (stable) ----
        for (uint32_t i = s_lo; i < s_hi; ++i) {
            const uint32_t p = (((uint32_t) slist[i >> 5] << 5) | (i & 31u)) * 32u + lane;
            const bool valid = p < nhash;
            const uint32_t h = valid ? lds16(sP + 2u * p) : 0u;
            const uint32_t b = h >> (HB - LB);
            unsigned m = __ballot_sync(ZWZ_FULL, valid), ml = m;
#pragma unroll
            for (uint32_t k = 0; k < LB; ++k) {
                const unsigned v = __ballot_sync(ZWZ_FULL, (b >> k) & 1u);
                m &= ((b >> k) & 1u) ? v : ~v;
                ml &= ((lane >> k) & 1u) ? v : ~v;
            }
            const uint32_t o = __shfl_sync(ZWZ_FULL, off, b);
            if (valid) list[o + (uint32_t) __popc(m & lt)] = (uint16_t) p;
            off += (uint32_t) __popc(ml);
        }
        __threadfence_block();
        __syncthreads();
        ZWZ_DM_CLK(6);
        // tile flags of this chunk, collected in the cnt area (free since the offsets): bit t = tile t holds a match
        uint32_t *tflags = (uint32_t *) cnt;
        for (uint32_t i = tid; i < ZWZ_SCR_FLAG_WORDS && i < NW * NW / 2u; i += T) tflags[i] = 0u;

        // ---- 5. EXACT hash chains, one warp per list, 32 positions per step ----
        // Lists hold disjoint hash ranges, so the NW builders never touch the same head[] entry. Common case (all 32 hashes
        // of a step distinct): read the old head, store it as the link, store the position as the new head. Lanes that
        // share a hash inside the step are detected by reading the head back (one of them won the store race, the others see
        // a foreign position) and repaired group by group with ballot + shuffle, which costs per COLLIDING group —
        // __match_any_sync costs per DISTINCT value (measured ~600 cycles per step on sm_100a).
        {
            const uint32_t i_end = ctl->base[wid + 1u];
            uint32_t i0 = ctl->base[wid];
            uint32_t qn = (i0 + lane < i_end) ? (uint32_t) __ldcg(list + i0 + lane) : 0u;
            for (; i0 < i_end; i0 += 32u) {
                const bool valid = i0 + lane < i_end;
                const uint32_t q = qn;
                qn = (i0 + 32u + lane < i_end) ? (uint32_t) __ldcg(list + i0 + 32u + lane) : 0u; // next step, fetched ahead
                const uint32_t h = valid ? lds16(sP + 2u * q) : 0u;
                uint32_t old = ZWZ_DM_NIL;
                if (valid) old = lds16(sH + 2u * h);
                __syncwarp(); // all reads of head[] precede the writes of this step
                if (valid) {
                    sts16(sP + 2u * q, old);
                    sts16(sH + 2u * h, q);
                }
                __syncwarp();
                uint32_t rb = valid ? lds16(sH + 2u * h) : q;
                unsigned rem = __ballot_sync(ZWZ_FULL, rb != q); // lanes that lost a store race
                while (rem) {                                    // one round per colliding group (warp-uniform loop)
                    const int leader = __ffs((int) rem) - 1;
                    const uint32_t hl = __shfl_sync(ZWZ_FULL, h, leader);
                    const bool mine = valid && h == hl;
                    const unsigned same = __ballot_sync(ZWZ_FULL, mine);
                    const unsigned lower = same & lt;
                    const int from = (mine && lower) ? 31 - __clz((int) lower) : (int) lane;
                    const uint32_t qlow = __shfl_sync(ZWZ_FULL, q, from);  // nearest earlier position of the group
                    if (mine) {
                        if (lower) sts16(sP + 2u * q, qlow);
                        if ((same >> lane) == 1u) sts16(sH + 2u * h, q);        // the latest position stays head
                    }
                    rem &= ~same;
                }
                __syncwarp();
            }
        }
        __syncthreads();
        ZWZ_DM_CLK(7);

        // ---- 6. search: one lane per position, 32-position tiles ----
        // Every lane walks the chain of its position: the cheap test (the two bytes that would extend its best match — zlib's
        // longest_match order) turns most candidates away; a survivor is compared against the first 12 bytes of the scan string,
        // which the lane holds in three registers, in straight-line code (three XORs and a find-first-set: no loop for the
        // short matches that make up text), and by words beyond that. When the walks are done the lanes INHERIT: a match (L, d)
        // at position j is a match (L - k, d) at j + k, so a prefix maximum of L_j + j over the tile (5 shuffle steps) hands
        // every lane the best such match of its left neighbours where its own walk found less (the depth limit cuts walks
        // short; in text the best match of p + 1 is usually the tail of the one at p).
        // Only the searched tiles are handed out (noise tiles are neither searched nor written: the encoder reads the raw bytes).
        // Measured and dropped: a static schedule (warp w takes the searched tiles w, w + NW, ...) saves the shared atomic per
        // tile but leaves warps idle behind the slowest one, where walk lengths vary: lz_match +33 % on text, +10 % on the
        // bitmap-like C2 files (profiles/match_overhead).
        // Measured and dropped (profiles/round2_notes.md): rounds of "walk until a candidate survives, then extend all survivors
        // together" (the walks of a tile then run one after the other: 36.2 ms against 29.8 ms per 512 MiB of text), and
        // inheriting after the first 1-4 candidates already, to raise the bar for the rest of the walk (+3 % on text, +10 % on
        // the near-incompressible C2 files, where tiles without any match pay for the shuffles).
        uint32_t wmatch = 0; // positions of this warp's tiles that found a match
        for (;;) {
            uint32_t i = 0;
            if (lane == 0) i = atomicAdd(&ctl->next_tile, 1u);
            i = __shfl_sync(ZWZ_FULL, i, 0);
            if (i >= ntiles) break;
            const uint32_t tile = ((uint32_t) slist[i >> 5] << 5) | (i & 31u);
                const uint32_t p = tile * 32u + lane;
                uint32_t best_len = 2u, best_dist = 0u;
                uint32_t maxlen = 0u;
                if (p < nhash) {
                    maxlen = (n - p) < ZWZ_MAX_MATCH ? (n - p) : ZWZ_MAX_MATCH;
                    const uint32_t limit = p > ZWZ_MAX_DIST ? p - ZWZ_MAX_DIST : 0u;
                    const uint32_t span = p - limit;            // a candidate is usable iff 0 <= cand - limit < span (NIL fails)
                    uint32_t cand = lds16(sP + 2u * p);
                    if ((cand - limit) < span || (DICT && dwl != 0u && p < ZWZ_MAX_DIST)) {
                        const uint32_t ap = sD + p;             // shared address of the scan position
                        const uint32_t ka = ap & ~3u, sa = (ap & 3u) * 8u;
                        const uint32_t a0 = lds32(ka), a1 = lds32(ka + 4u), a2 = lds32(ka + 8u), a3 = lds32(ka + 12u);
                        const uint32_t S0 = __funnelshift_r(a0, a1, sa), S1 = __funnelshift_r(a1, a2, sa), S2 = __funnelshift_r(a2, a3, sa); // bytes [0, 12)
                        uint32_t scan_end = (S0 >> 16) & 0xffu, scan_end1 = (S0 >> 8) & 0xffu; // bytes at best_len and best_len - 1
                        uint32_t budget = job.depth;
                        for (; budget != 0u && (cand - limit) < span; --budget) {
                            const uint32_t ac = sD + cand;
                            const uint32_t nxt = lds16(sP + 2u * cand); // next link is fetched while this candidate is examined
                            if (lds8(ac + best_len) == scan_end && lds8(ac + best_len - 1u) == scan_end1) {
                                const uint32_t kc = ac & ~3u, sc = (ac & 3u) * 8u;
                                const uint32_t c0 = lds32(kc), c1 = lds32(kc + 4u), c2 = lds32(kc + 8u), c3 = lds32(kc + 12u);
                                const uint32_t x0 = __funnelshift_r(c0, c1, sc) ^ S0, x1 = __funnelshift_r(c1, c2, sc) ^ S1,
                                               x2 = __funnelshift_r(c2, c3, sc) ^ S2;
                                uint32_t len;
                                if (x0) {
                                    len = ((uint32_t) __ffs((int) x0) - 1u) >> 3; // < 3: a hash collision
                                } else if (x1) {
                                    len = 4u + (((uint32_t) __ffs((int) x1) - 1u) >> 3);
                                } else if (x2) {
                                    len = 8u + (((uint32_t) __ffs((int) x2) - 1u) >> 3);
                                } else {
                                    len = 12u;
                                    while (len < maxlen) {
                                        uint32_t y = lds32u(ac + len) ^ lds32u(ap + len);
                                        if (y) {
                                            len += ((uint32_t) __ffs((int) y) - 1u) >> 3;
                                            break;
                                        }
                                        len += 4u;
                                    }
                                }
                                if (len > maxlen) len = maxlen;
                                if (len > best_len) {
                                    best_len = len;
                                    best_dist = p - cand;
                                    if (len >= job.nice || len >= maxlen) break;
                                    scan_end = lds8(ap + len);
                                    scan_end1 = lds8(ap + len - 1u);
                                }
                            }
                            cand = nxt;
                        }
                        // The chunk's own chain is exhausted with budget left and no match of `nice` bytes: the walk goes on in the
                        // dictionary's chain, most recent position first as in zlib (whose window holds the dictionary right before
                        // the chunk), within the same budget. Window position q is at distance p + dwl - q. The 14-bit hash of the
                        // scan position holds this class's hash in its top bits, so no candidate of a true match is lost. The
                        // window is read from global memory (the record is L2-resident, read by every chunk of the call); a match
                        // that starts in the window ends at its end — DEFLATE would let it run on into the chunk, zlib does.
                        if (DICT && budget != 0u && best_len < job.nice && best_len < maxlen && dwl != 0u && p < ZWZ_MAX_DIST) {
                            const uint16_t *dhead = (const uint16_t *) (drec + ZWZ_DICT_HEAD), *dprev = (const uint16_t *) (drec + ZWZ_DICT_PREV);
                            const uint8_t *dwin = drec + ZWZ_DICT_WIN;
                            const uint32_t dlim = p + dwl > ZWZ_MAX_DIST ? p + dwl - ZWZ_MAX_DIST : 0u; // oldest usable window position
                            const uint32_t dspan = dwl - dlim;                                         // NIL fails (q - dlim) < dspan
                            uint32_t q = __ldg(dhead + dm_hash3<ZWZ_DICT_HBITS>(S0 & 0xffu, (S0 >> 8) & 0xffu, (S0 >> 16) & 0xffu));
                            for (; budget != 0u && (q - dlim) < dspan; --budget) {
                                const uint32_t nxt = __ldg(dprev + q);
                                const uint32_t dmax = dwl - q < maxlen ? dwl - q : maxlen;
                                if (best_len < dmax && __ldg(dwin + q + best_len) == scan_end && __ldg(dwin + q + best_len - 1u) == scan_end1) {
                                    uint32_t len = 0;
                                    while (len < dmax) {
                                        const uint32_t y = ld32u((const uint32_t *) dwin, q + len) ^ lds32u(ap + len);
                                        if (y) {
                                            len += ((uint32_t) __ffs((int) y) - 1u) >> 3;
                                            break;
                                        }
                                        len += 4u;
                                    }
                                    if (len > dmax) len = dmax;
                                    if (len > best_len) {
                                        best_len = len;
                                        best_dist = p + dwl - q;
                                        if (len >= job.nice || len >= maxlen) break;
                                        scan_end = lds8(ap + len);
                                        scan_end1 = lds8(ap + len - 1u);
                                    }
                                }
                                q = nxt;
                            }
                        }
                    }
                }
                if (__any_sync(ZWZ_FULL, best_len >= 4u)) { // inherit (a 3-byte match has no tail worth passing on)
                    uint32_t key = best_len >= 3u ? best_len + lane : 0u, kd = best_dist;
    #pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t ok = __shfl_up_sync(ZWZ_FULL, key, d), od = __shfl_up_sync(ZWZ_FULL, kd, d);
                        if (lane >= (unsigned) d && ok > key) {
                            key = ok;
                            kd = od;
                        }
                    }
                    if (key >= lane + 3u && key - lane > best_len && key - lane <= maxlen) { // maxlen = 0: no hash here (last two bytes)
                        best_len = key - lane;
                        best_dist = kd;
                    }
                }
                if (best_len == 3u && best_dist > 4096u) best_len = 2u; // zlib's TOO_FAR: such a match costs more than 3 literals
                // a tile without a single match is not written at all: the encoder takes its literals from the raw bytes
                const unsigned hit = __ballot_sync(ZWZ_FULL, best_len >= 3u);
                if (hit) {
                    if (p < n) mout[p] = tok_make(lds8(sD + p), best_len >= 3u ? best_len : 0u, best_dist);
                    if (lane == 0) atomicOr(&tflags[tile >> 5], 1u << (tile & 31u));
                    wmatch += (uint32_t) __popc(hit);
                }
        }
        if (lane == 0 && wmatch) atomicAdd(&ctl->nmatch, wmatch);

        // ---- 7. Adler-32 of the chunk ----
        // Each warp adds its part once it is out of tiles. Thread t takes the aligned words t, t + T, ... of the staging buffer
        // (conflict-free; a contiguous byte range per thread put 32 lanes on two banks): a = sum of bytes, b = sum of
        // (n - i) * byte_i, both by byte dot products.
        AdlerPart part;
        part.a = 0;
        part.b = 0;
        part.len = 0; // b is kept position-weighted from the start: parts add up without length terms
        {
            const uint32_t nwords = (skew + n + 3u) >> 2;
            for (uint32_t j = tid; j < nwords; j += T) { // <= 17 words per thread: (n - pos0) * 1020 * 17 < 2^32
                uint32_t wv = dataw[j];
                const int pos0 = (int) (4u * j) - (int) skew; // chunk position of the word's first byte
                if (pos0 < 0) wv = pos0 <= -4 ? 0u : wv & (0xffffffffu << (8u * (uint32_t) (-pos0)));
                if (pos0 + 4 > (int) n) wv &= 0xffffffffu >> (8u * (uint32_t) (pos0 + 4 - (int) n));
                const uint32_t s4 = zwz_dp4a(wv, 0x01010101u), w4 = zwz_dp4a(wv, 0x03020100u);
                part.a += s4;
                part.b += (uint32_t) ((int) n - pos0) * s4 - w4;
            }
            part.b %= 65521u;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                AdlerPart o;
                o.a = __shfl_down_sync(ZWZ_FULL, part.a, d);
                o.b = __shfl_down_sync(ZWZ_FULL, part.b, d);
                o.len = __shfl_down_sync(ZWZ_FULL, part.len, d);
                if ((lane & (2u * d - 1u)) == 0u) part = adler_combine(part, o);
            }
            if (lane == 0) {
                ctl->adler_a[wid] = part.a;
                ctl->adler_b[wid] = part.b;
                ctl->adler_len[wid] = part.len;
            }
        }
        __syncthreads();
        ZWZ_DM_CLK(8);
        // The lists are dead now. They were written and read back through L2 by this CTA alone: tell L2 to drop the lines instead
        // of writing 2 bytes per input byte back to DRAM (profiles/round1: lz_match moved 6.9x its algorithmic bytes).
        {
            const uint32_t list_lines = (nhash * 2u + 127u) >> 7;
            for (uint32_t i = tid; i < list_lines; i += T) discard_l2_line((const unsigned char *) list + 128u * i);
        }
        {
            uint32_t *gflags = mout + scr_flag_offset(n);
            const uint32_t used = (((n + 31u) >> 5) + 31u) >> 5;
            for (uint32_t i = tid; i < ZWZ_SCR_FLAG_WORDS; i += T) gflags[i] = i < used ? tflags[i] : 0u;
        }
        if (wid == 0) {
            part.a = lane < NW ? ctl->adler_a[lane] : 0u;
            part.b = lane < NW ? ctl->adler_b[lane] : 0u;
            part.len = lane < NW ? ctl->adler_len[lane] : 0u;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                AdlerPart o;
                o.a = __shfl_down_sync(ZWZ_FULL, part.a, d);
                o.b = __shfl_down_sync(ZWZ_FULL, part.b, d);
                o.len = __shfl_down_sync(ZWZ_FULL, part.len, d);
                if ((lane & (2u * d - 1u)) == 0u) part = adler_combine(part, o);
            }
            if (lane == 0) {
                uint32_t a = (1u + part.a) % 65521u;
                uint32_t b = (n % 65521u + part.b) % 65521u;
                job.adler[c] = (b << 16) | a;
                job.nmatch[c] = ctl->nmatch;
            }
        }
        ZWZ_DM_CLK(9);
        // No barrier here: the next chunk's first writes to shared memory (staging, the control block) follow the barrier at the
        // top of the loop, and every read of this chunk's data, flags and Adler parts precedes it.
    }
}

// One CTA per preset dictionary of a call: its record in the dictionary arena (zwz_common.cuh, ZWZ_DICT_*), read by every chunk
// that uses the dictionary. Window k is data[win_off[k] .. + wlen[k]). The chains are built as in step 5 of lz_match_kernel (all
// positions hashed in parallel, then 32 positions per step with the same collision repair), by one warp over the whole window:
// exact zlib-order chains in ~1 000 steps, once per dictionary and call.
#define ZWZ_DICT_SMEM (2u * 32768u + (2u << ZWZ_DICT_HBITS))
ZWZ_KERNEL __launch_bounds__(1024) dict_chain_kernel(const uint8_t *__restrict__ data, const uint64_t *__restrict__ win_off,
                                                     const uint32_t *__restrict__ wlen, uint8_t *arena) {
    ZWZ_DYN_SMEM(smem);
    uint16_t *prev = (uint16_t *) smem;                // hash of position q until the builder replaces it by the link
    uint16_t *head = (uint16_t *) (smem + 2u * 32768u);
    const unsigned tid = threadIdx.x, lane = lane_id(), T = blockDim.x;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t k = blockIdx.x, W = wlen[k];
    const uint8_t *src = data + win_off[k];
    uint8_t *rec = arena + (size_t) k * ZWZ_DICT_STRIDE;
    const uint32_t nh = W >= 3u ? W - 2u : 0u; // positions that own a 3-byte hash inside the window
    for (uint32_t i = tid; i < W + 64u; i += T) rec[ZWZ_DICT_WIN + i] = i < W ? src[i] : (uint8_t) 0;
    for (uint32_t i = tid; i < (1u << ZWZ_DICT_HBITS); i += T) head[i] = (uint16_t) ZWZ_DM_NIL;
    for (uint32_t q = tid; q < nh; q += T) prev[q] = (uint16_t) dm_hash3<ZWZ_DICT_HBITS>(src[q], src[q + 1u], src[q + 2u]);
    __syncthreads();
    if (tid < 32u) {
        for (uint32_t i0 = 0; i0 < nh; i0 += 32u) {
            const uint32_t q = i0 + lane;
            const bool valid = q < nh;
            const uint32_t h = valid ? prev[q] : 0u;
            const uint32_t old = valid ? head[h] : (uint32_t) ZWZ_DM_NIL;
            __syncwarp(); // all reads of head[] precede the writes of this step
            if (valid) {
                prev[q] = (uint16_t) old;
                head[h] = (uint16_t) q;
            }
            __syncwarp();
            const uint32_t rb = valid ? head[h] : q;
            unsigned rem = __ballot_sync(ZWZ_FULL, rb != q); // lanes that lost a store race
            while (rem) {
                const int leader = __ffs((int) rem) - 1;
                const uint32_t hl = __shfl_sync(ZWZ_FULL, h, leader);
                const bool mine = valid && h == hl;
                const unsigned same = __ballot_sync(ZWZ_FULL, mine);
                const unsigned lower = same & lt;
                const int from = (mine && lower) ? 31 - __clz((int) lower) : (int) lane;
                const uint32_t qlow = __shfl_sync(ZWZ_FULL, q, from);
                if (mine) {
                    if (lower) prev[q] = (uint16_t) qlow;
                    if ((same >> lane) == 1u) head[h] = (uint16_t) q;
                }
                __syncwarp();
                rem &= ~same;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    uint16_t *ghead = (uint16_t *) (rec + ZWZ_DICT_HEAD), *gprev = (uint16_t *) (rec + ZWZ_DICT_PREV);
    for (uint32_t i = tid; i < (1u << ZWZ_DICT_HBITS); i += T) ghead[i] = head[i];
    for (uint32_t q = tid; q < nh; q += T) gprev[q] = prev[q];
}

} // namespace zwz
