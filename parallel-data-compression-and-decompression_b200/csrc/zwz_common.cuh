// zwz_common.cuh — shared device-side helpers for the sm_100a kernels.
//
// Every kernel source in this directory compiles two ways:
//   nvcc -gencode arch=compute_100a,code=sm_100a            -> the product (libzwz_cuda.so)
//   g++  -DZWZ_EMU -include tests/simt/simt_emu.h           -> the CPU SIMT emulator build used ONLY by tests
// so the few places that need inline PTX (bulk async copy + mbarrier) have a plain-loop twin under ZWZ_EMU.
#pragma once
#include <stdint.h>
#include "zwz_cuda.h"

#ifdef ZWZ_EMU
#define ZWZ_DEV static inline
#define ZWZ_DEV_NOINLINE static
#define ZWZ_KERNEL static void
#define ZWZ_DYN_SMEM(name) unsigned char *name = simt::dyn_smem()
#define ZWZ_SPIN_PAUSE() zwz_emu_spin_pause()
#define ZWZ_SPIN_SLEEP(ns) zwz_emu_spin_pause()
#else
#include <cuda_runtime.h>
#define ZWZ_DEV __device__ __forceinline__
#define ZWZ_DEV_NOINLINE __device__ __noinline__
#define ZWZ_KERNEL __global__ void
#define ZWZ_DYN_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#define ZWZ_SPIN_PAUSE() __nanosleep(20)
#define ZWZ_SPIN_SLEEP(ns) __nanosleep(ns)
#endif

#ifdef ZWZ_EMU
#include <cmath>
#define zwz_log2f(x) log2f(x)
#else
#define zwz_log2f(x) __log2f(x)
#endif
#define ZWZ_FULL 0xffffffffu
#define ZWZ_CHUNK 65535u
#define ZWZ_MIN_MATCH 3u
#define ZWZ_MAX_MATCH 258u
#define ZWZ_MAX_DIST 32768u

namespace zwz {

ZWZ_DEV unsigned lane_id() { return threadIdx.x & 31u; }
ZWZ_DEV unsigned warp_id() { return threadIdx.x >> 5; }

// ---- preset dictionaries (zwz_*_dict calls) ----
// Every dictionary of a call has one record in the context's dictionary arena, built by dict_chain_kernel (deflate_match.cuh):
//   [ZWZ_DICT_HEAD, +32 KiB)  head[2^14] u16: latest window position of each 14-bit hash (dm_hash3<14>), NIL = 0xffff
//   [ZWZ_DICT_PREV, +64 KiB)  prev[32 768] u16: the next older position of the same hash (exact zlib-order chains)
//   [ZWZ_DICT_WIN, +32 KiB)   the window (the dictionary's last <= 32 768 bytes), 16-byte aligned and zero padded, so that
//                             both the match search and inflate read it with aligned loads
// The last two window positions are not chained: their 3-byte hash would need the chunk's first bytes.
#define ZWZ_DICT_HBITS 14u
#define ZWZ_DICT_HEAD 0u
#define ZWZ_DICT_PREV 32768u
#define ZWZ_DICT_WIN 98304u
#define ZWZ_DICT_STRIDE (98304u + 32768u + 256u)
struct DictTable {
    const uint32_t *idx;   // [n] dictionary of chunk / stream i, or ZWZ_NO_DICT (nullptr: the call has no dictionary)
    const uint8_t *arena;  // ZWZ_DICT_STRIDE bytes per dictionary
    const uint32_t *wlen;  // [ndict] window length (1 .. 32 768)
    const uint32_t *id;    // [ndict] DICTID: Adler-32 of the whole dictionary
};

// chunk descriptor / result as laid out in device memory (structure of arrays, one entry per chunk)
struct DeflateJob {
    const uint8_t *raw;        // all chunks' raw bytes
    const uint64_t *raw_off;   // [n]
    const uint32_t *raw_len;   // [n]   <= 65535
    const uint64_t *scr_off;   // [n]   offset (in uint32 units) of this chunk's match/token scratch
    uint32_t *scratch;         // 4 bytes per raw byte (+ pad)
    uint32_t *adler;           // [n]   check value: Adler-32 written by the match kernel, in GZIP format overwritten by the CRC-32
                               //       of crc32_kernel; read by the encoder
    uint32_t *nmatch;          // [n]   positions that found a match (match kernel -> encoder: incompressibility shortcut)
    uint8_t *out;              // output slots
    const uint64_t *out_off;   // [n]   multiple of 4, capacity >= zwz_deflate_bound(len)
    uint32_t *res;             // [n*4] zwz_deflate_result
    uint32_t n;
    uint32_t depth;            // hash-chain candidates examined per position
    uint32_t nice;             // stop searching at this length
    uint32_t *work_counter;    // persistent-CTA work queue
    uint32_t format;           // ZWZ_FORMAT_*: the wrapper deflate_encode_kernel puts around the body
    DictTable dict;            // read only by the DICT instantiations of the kernels
};

// ---- unaligned little-endian loads built from aligned 32-bit words -------------------------------------------------
// `w` is a 4-byte-aligned array, `i` a byte index into it. Reads the two words covering bytes [i, i+4).
ZWZ_DEV uint32_t ld32u(const uint32_t *w, uint32_t i) {
    uint32_t k = i >> 2;
    uint32_t lo = w[k], hi = w[k + 1];
    return __funnelshift_r(lo, hi, (i & 3u) * 8u);
}

// ---- explicit shared-memory addressing for the hot loops --------------------------------------------------------------
// A 32-bit shared-window address + ld.shared keeps the inner loops at one LDS per access; going through generic pointers made
// the compiler rebuild the window base (S2R SR_CgaCtaId / LEA) inside the candidate loop. Emulator: offset into the CTA's
// dynamic shared memory. The asm statements are volatile with a memory clobber: they must not move across barriers or the
// stores of the chain builder.
#ifdef ZWZ_EMU
ZWZ_DEV uint32_t smem_addr(const void *p) { return (uint32_t) ((const unsigned char *) p - simt::dyn_smem()); }
ZWZ_DEV uint32_t lds8(uint32_t a) { return simt::dyn_smem()[a]; }
ZWZ_DEV uint32_t lds16(uint32_t a) { return *(const uint16_t *) (simt::dyn_smem() + a); }
ZWZ_DEV uint32_t lds32(uint32_t a) { return *(const uint32_t *) (simt::dyn_smem() + a); }
ZWZ_DEV void sts16(uint32_t a, uint32_t v) { *(uint16_t *) (simt::dyn_smem() + a) = (uint16_t) v; }
#else
ZWZ_DEV uint32_t smem_addr(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
ZWZ_DEV uint32_t lds8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
ZWZ_DEV uint32_t lds16(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
ZWZ_DEV uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
ZWZ_DEV void sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short) v) : "memory"); }
#endif
// unaligned little-endian 32-bit load at shared address a
ZWZ_DEV uint32_t lds32u(uint32_t a) {
    uint32_t k = a & ~3u;
    return __funnelshift_r(lds32(k), lds32(k + 4u), (a & 3u) * 8u);
}

// sum over the four bytes of a of (byte of a) * (byte of b), unsigned
#ifdef ZWZ_EMU
ZWZ_DEV uint32_t zwz_dp4a(uint32_t a, uint32_t b) {
    uint32_t r = 0;
    for (int k = 0; k < 4; ++k) r += ((a >> (8 * k)) & 0xffu) * ((b >> (8 * k)) & 0xffu);
    return r;
}
#else
ZWZ_DEV uint32_t zwz_dp4a(uint32_t a, uint32_t b) { return __dp4a(a, b, 0u); }
#endif

ZWZ_DEV uint32_t warp_incl_scan(uint32_t v) {
    unsigned l = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(ZWZ_FULL, v, d);
        if (l >= (unsigned) d) v += t;
    }
    return v;
}
ZWZ_DEV uint32_t warp_sum(uint32_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(ZWZ_FULL, v, d);
    return v;
}
ZWZ_DEV uint64_t warp_sum64(uint64_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(ZWZ_FULL, v, d);
    return v;
}
ZWZ_DEV uint32_t warp_max(uint32_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        uint32_t t = __shfl_xor_sync(ZWZ_FULL, v, d);
        v = t > v ? t : v;
    }
    return v;
}

// ---- scratch word per position / token: [31:24] literal byte at that position, [23:15] match length (0 = none, else 3..258),
//      [14:0] match distance - 1. The parser keeps the words it selects (as tokens) and drops the others.
ZWZ_DEV uint32_t tok_make(uint32_t byte, uint32_t len, uint32_t dist) { return (byte << 24) | (len << 15) | (len ? dist - 1u : 0u); }
ZWZ_DEV uint32_t tok_len(uint32_t t) { return (t >> 15) & 0x1ffu; }
ZWZ_DEV uint32_t tok_dist(uint32_t t) { return (t & 0x7fffu) + 1u; }
ZWZ_DEV uint32_t tok_byte(uint32_t t) { return t >> 24; }
#ifdef ZWZ_EMU
ZWZ_DEV void prefetch_l2(const void *) {}
ZWZ_DEV void discard_l2_line(const void *) {}
#else
ZWZ_DEV void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// The 128-byte line at p (128-byte aligned) holds dead data: drop it from L2 WITHOUT writing it back to DRAM.
ZWZ_DEV void discard_l2_line(const void *p) { asm volatile("discard.global.L2 [%0], 128;" ::"l"(p) : "memory"); }
#endif

// ---- scratch layout of one chunk of n raw bytes (uint32 units from job.scr_off[c]; keep in step with zwz_cuda.cu) --------
//   [0, A)          best match per position (lz_match_kernel) — only the 32-position tiles that HOLD a match are written —
//                   overwritten in place by the parser with the token stream (deflate_encode_kernel)
//   [A, A + B)      the hash-partitioned u16 position lists of lz_match_kernel (dead, and discarded from L2, once the chains exist)
//   [A + B, +64)    one bit per 32-position tile: the tile holds at least one match (its words in [0, A) are valid)
#define ZWZ_SCR_FLAG_WORDS 64u
ZWZ_DEV uint32_t scr_match_words(uint32_t n) { return (n + 2u + 31u) & ~31u; }
ZWZ_DEV uint32_t scr_list_words(uint32_t n) { return ((n + 1u) / 2u + 32u + 31u) & ~31u; }
ZWZ_DEV uint32_t scr_flag_offset(uint32_t n) { return scr_match_words(n) + scr_list_words(n); }

// ---- vectorised plain copy (stored blocks): out[0..n) = src[0..n), any alignment of either side ----
// 16-byte stores to the aligned middle of the destination; the source words come from aligned 32-bit loads shifted into
// place, so nothing outside the aligned words that hold src[0..n) is read.
ZWZ_DEV void inf_copy_plain(uint8_t *dst, const uint8_t *src, uint32_t n) {
    const unsigned lane = lane_id();
    uint32_t head = (16u - (uint32_t) ((uintptr_t) dst & 15u)) & 15u;
    if (head > n) head = n;
    if (lane < head) dst[lane] = src[lane];
    const uint32_t nvec = (n - head) >> 4;
    const uint8_t *s = src + head;
    uint8_t *d = dst + head;
    const uint32_t a = (uint32_t) ((uintptr_t) s & 3u);
    const uint32_t *sw = (const uint32_t *) (s - a);
    const uint32_t sh = a * 8u;
    for (uint32_t v = lane; v < nvec; v += 32u) {
        const uint32_t *w = sw + 4u * v;
        const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2), w3 = __ldg(w + 3);
        const uint32_t w4 = a ? __ldg(w + 4) : 0u; // a == 0: the fifth word is not part of the source
        uint4 o;
        o.x = __funnelshift_r(w0, w1, sh);
        o.y = __funnelshift_r(w1, w2, sh);
        o.z = __funnelshift_r(w2, w3, sh);
        o.w = __funnelshift_r(w3, w4, sh);
        *(uint4 *) (d + 16u * v) = o;
    }
    const uint32_t done = head + (nvec << 4);
    if (done + lane < n) dst[done + lane] = src[done + lane]; // tail < 16 bytes
}

// ---- DEFLATE symbol arithmetic (RFC 1951 §3.2.5) without tables ----------------------------------------------------
// length 3..258 -> (symbol 257..285, extra bit count, extra value)
ZWZ_DEV void len_symbol(uint32_t len, uint32_t &sym, uint32_t &ebits, uint32_t &eval) {
    uint32_t l = len - 3u;
    if (l < 8u) {
        sym = 257u + l;
        ebits = 0;
        eval = 0;
    } else if (len == 258u) {
        sym = 285u;
        ebits = 0;
        eval = 0;
    } else {
        uint32_t nb = 31u - (uint32_t) __clz((int) l); // >= 3
        sym = 257u + 4u * (nb - 1u) + ((l >> (nb - 2u)) & 3u);
        ebits = nb - 2u;
        eval = l & ((1u << ebits) - 1u);
    }
}
// distance 1..32768 -> (symbol 0..29, extra bit count, extra value)
ZWZ_DEV void dist_symbol(uint32_t dist, uint32_t &sym, uint32_t &ebits, uint32_t &eval) {
    uint32_t d = dist - 1u;
    if (d < 4u) {
        sym = d;
        ebits = 0;
        eval = 0;
    } else {
        uint32_t nb = 31u - (uint32_t) __clz((int) d); // >= 2
        sym = 2u * nb + ((d >> (nb - 1u)) & 1u);
        ebits = nb - 1u;
        eval = d & ((1u << ebits) - 1u);
    }
}

// Adler-32 partial sums over a byte range handled by one thread, to be combined with adler_combine.
struct AdlerPart {
    uint32_t a; // sum of bytes            (mod 65521)
    uint32_t b; // sum of (len - j) * byte (mod 65521)
    uint32_t len;
};
// (A then B) as one range: a = aA + aB ; b = bA + bB + lenB * aA
ZWZ_DEV AdlerPart adler_combine(const AdlerPart &x, const AdlerPart &y) {
    AdlerPart r;
    r.a = (x.a + y.a) % 65521u;
    r.b = (uint32_t) (((uint64_t) x.b + y.b + (uint64_t) (y.len % 65521u) * x.a) % 65521u);
    r.len = x.len + y.len;
    return r;
}

} // namespace zwz
