// crc32.cuh — CRC-32 of RFC 1952 (reflected polynomial 0xEDB88320, register preset and final xor 0xFFFFFFFF), one warp per
// byte range: the check value of gzip members.
//
// Each lane runs slice-by-4 over one contiguous slice of the range (16-byte loads; lane 0 also takes the unaligned head,
// lane 31 the tail). The 32 partial CRCs are then combined as zlib's crc32_combine does: crc(A || B) = crc(A) * x^(8|B|) ^
// crc(B) in GF(2)[x] mod P, so every lane multiplies its CRC by x^(8 * bytes behind its slice) and the warp XORs the products.
// x^(8n) is assembled from the table of x^(2^k) like zlib's x2nmodp.
//
// The 4 KB slice table is read from shared memory. Kernels of the zlib path keep their shared-memory layout: crc32_kernel
// stages the table in a static array of its own, and inflate_kernel loads it over its decoder state (tables, staged window,
// token regions) before the first block and after the last, when that is dead (inflate.cuh, gzip header and trailer).
#pragma once
#include "zwz_common.cuh"

namespace zwz {

#define ZWZ_CRC_POLY 0xEDB88320u
#define ZWZ_CRC_TAB_WORDS 1024u // slice-by-4: 4 x 256 words

struct Crc32Tables {
    uint32_t slice[4][256]; // slice[k][b]: CRC register after byte b followed by k zero bytes
    uint32_t x2n[32];       // x^(2^k) mod P (bit 31 = x^0, reflected like the register)
};

constexpr uint32_t crc32_multmodp_c(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if (a & (0x80000000u >> i)) p ^= b;
        b = (b >> 1) ^ ((b & 1u) ? ZWZ_CRC_POLY : 0u);
    }
    return p;
}

constexpr Crc32Tables crc32_make_tables() {
    Crc32Tables r{};
    for (uint32_t b = 0; b < 256u; ++b) {
        uint32_t c = b;
        for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1u) ? ZWZ_CRC_POLY : 0u);
        r.slice[0][b] = c;
    }
    for (int k = 1; k < 4; ++k)
        for (uint32_t b = 0; b < 256u; ++b) r.slice[k][b] = (r.slice[k - 1][b] >> 8) ^ r.slice[0][r.slice[k - 1][b] & 0xffu];
    uint32_t p = 1u << 30; // x^1
    for (int k = 0; k < 32; ++k) {
        r.x2n[k] = p;
        p = crc32_multmodp_c(p, p);
    }
    return r;
}
static_assert(crc32_make_tables().slice[0][1] == 0x77073096u, "CRC-32 table");

#ifdef ZWZ_EMU
static const Crc32Tables g_crc32 = crc32_make_tables();
#else
__device__ const Crc32Tables g_crc32 = crc32_make_tables();
#endif

// a * b mod P, fixed 32 steps (no data-dependent exit: the lanes stay converged)
ZWZ_DEV uint32_t crc32_multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
        p ^= (a & (0x80000000u >> i)) ? b : 0u;
        b = (b >> 1) ^ ((b & 1u) ? ZWZ_CRC_POLY : 0u);
    }
    return p;
}

// x^(8n) mod P
ZWZ_DEV uint32_t crc32_x8n(uint64_t n) {
    uint32_t p = 0x80000000u; // x^0
    for (uint32_t k = 3; n; n >>= 1, ++k)
        if (n & 1u) p = crc32_multmodp(__ldg(&g_crc32.x2n[k & 31u]), p);
    return p;
}

// the table into shared memory (every lane of the warp takes part; no barrier implied)
ZWZ_DEV void crc32_load_table(uint32_t *tab, unsigned first, unsigned step) {
    for (uint32_t i = first; i < ZWZ_CRC_TAB_WORDS; i += step) tab[i] = __ldg(&g_crc32.slice[0][0] + i);
}

ZWZ_DEV uint32_t crc32_byte(const uint32_t *tab, uint32_t c, uint32_t b) { return tab[(c ^ b) & 0xffu] ^ (c >> 8); }
ZWZ_DEV uint32_t crc32_word(const uint32_t *tab, uint32_t c, uint32_t w) {
    c ^= w;
    return tab[768u + (c & 0xffu)] ^ tab[512u + ((c >> 8) & 0xffu)] ^ tab[256u + ((c >> 16) & 0xffu)] ^ tab[c >> 24];
}

// CRC-32 of p[0, n), warp-collective; tab = the slice table in shared memory. Loads go through L2 (ld.global.cg): inflate
// checks bytes that lanes of the same warp have just written. Every lane returns the result.
ZWZ_DEV uint32_t crc32_warp(const uint8_t *p, uint32_t n, const uint32_t *tab) {
    const unsigned lane = lane_id();
    uint32_t head = (16u - (uint32_t) ((uintptr_t) p & 15u)) & 15u;
    if (head > n) head = n;
    const uint32_t nvec = (n - head) >> 4;
    const uint32_t per = (nvec + 31u) >> 5;
    const uint32_t v0 = min(lane * per, nvec), v1 = min(v0 + per, nvec);
    uint32_t c = 0xffffffffu;
    if (lane == 0)
        for (uint32_t j = 0; j < head; ++j) c = crc32_byte(tab, c, __ldcg(p + j));
    const uint4 *vp = (const uint4 *) (p + head);
    for (uint32_t v = v0; v < v1; ++v) {
        const uint4 w = __ldcg(vp + v);
        c = crc32_word(tab, c, w.x);
        c = crc32_word(tab, c, w.y);
        c = crc32_word(tab, c, w.z);
        c = crc32_word(tab, c, w.w);
    }
    uint32_t end = head + 16u * v1;
    if (lane == 31u) {
        for (uint32_t j = end; j < n; ++j) c = crc32_byte(tab, c, __ldcg(p + j));
        end = n;
    }
    c ^= 0xffffffffu; // this lane's slice as a finished CRC (0 for an empty slice)
    uint32_t r = c ? crc32_multmodp(crc32_x8n(n - end), c) : 0u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) r ^= __shfl_xor_sync(ZWZ_FULL, r, d);
    return r;
}

// CRC-32 of arbitrary ranges, one warp each: the gzip trailer of the deflate path (launched between lz_match_kernel and
// deflate_encode_kernel, into the per-chunk check array) and zwz_crc32_batch_device
ZWZ_KERNEL crc32_kernel(const uint8_t *__restrict__ data, const uint64_t *__restrict__ off, const uint32_t *__restrict__ len, uint32_t *crc,
                        uint32_t n) {
    __shared__ uint32_t tab[ZWZ_CRC_TAB_WORDS];
    crc32_load_table(tab, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint32_t c = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (c >= n) return;
    const uint32_t r = crc32_warp(data + off[c], len[c], tab);
    if (lane_id() == 0) crc[c] = r;
}

} // namespace zwz
