// zwz_cuda.cu — implementation of the C ABI in include/zwz_cuda.h over the sm_100a kernels in this directory.
//
// One zwz_ctx per GPU: a non-blocking stream, grow-only device arenas (chunk descriptors, match/token scratch, bulk
// staging for the host-buffer entry points) and a pinned arena for descriptors/results. No CPU fallback: every entry
// point either runs the CUDA kernels or returns an error.
#include "zwz_cuda.h"
#include "zwz_rt.h"

#include "zwz_common.cuh"
#include "md5.cuh"
#include "crc32.cuh"
#include "inflate.cuh"
#include "inflate_lanes.cuh"
#include "deflate_match.cuh"
#include "deflate_encode.cuh"

#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

namespace zwz {

// Host threads of one context for the O(n) descriptor work of a call (staging copies, validation, prefix sums): while the
// calling thread prepares a call the device has nothing queued, since every call of the C ABI ends in a stream synchronise.
// run(nblk, f) calls f(0..nblk-1) on the workers and the calling thread and returns when all are done.
class HostPool {
public:
    explicit HostPool(unsigned workers) {
        for (unsigned i = 0; i < workers; ++i) th_.emplace_back([this] { loop(); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        wake_.notify_all();
        for (auto &t : th_) t.join();
    }
    void run(unsigned nblk, const std::function<void(unsigned)> &f) {
        {
            std::lock_guard<std::mutex> lk(m_);
            f_ = &f;
            nblk_ = nblk;
            next_.store(0);
            busy_ = (unsigned) th_.size();
            ++gen_;
        }
        wake_.notify_all();
        drain(f, nblk);
        std::unique_lock<std::mutex> lk(m_);
        idle_.wait(lk, [this] { return busy_ == 0; });
        f_ = nullptr;
    }

private:
    void drain(const std::function<void(unsigned)> &f, unsigned nblk) {
        for (unsigned b; (b = next_.fetch_add(1)) < nblk;) f(b);
    }
    void loop() {
        uint64_t seen = 0;
        std::unique_lock<std::mutex> lk(m_);
        for (;;) {
            wake_.wait(lk, [&] { return stop_ || gen_ != seen; });
            if (stop_) return;
            seen = gen_;
            const std::function<void(unsigned)> *f = f_;
            const unsigned nblk = nblk_;
            lk.unlock();
            drain(*f, nblk);
            lk.lock();
            if (--busy_ == 0) idle_.notify_one();
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable wake_, idle_;
    const std::function<void(unsigned)> *f_ = nullptr;
    unsigned nblk_ = 0, busy_ = 0;
    std::atomic<unsigned> next_{0};
    uint64_t gen_ = 0;
    bool stop_ = false;
};

// warp-per-chunk gather of the variable-length streams out of their slots into one packed buffer
ZWZ_KERNEL pack_streams_kernel(const uint8_t *__restrict__ slots, const uint64_t *__restrict__ slot_off, const uint32_t *__restrict__ res,
                               uint8_t *packed, const uint64_t *__restrict__ packed_off, uint32_t n) {
    uint32_t c = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (c >= n) return;
    const uint8_t *s = slots + slot_off[c];
    uint8_t *d = packed + packed_off[c];
    uint32_t bytes = res[4u * c] + res[4u * c + 1u];
    unsigned lane = lane_id();
    // slots are 4-byte aligned; use word copies when the destination happens to be too
    if ((((uintptr_t) d) & 3u) == 0u) {
        uint32_t nw = bytes >> 2;
        for (uint32_t i = lane; i < nw; i += 32u) ((uint32_t *) d)[i] = ((const uint32_t *) s)[i];
        for (uint32_t i = (nw << 2) + lane; i < bytes; i += 32u) d[i] = s[i];
    } else {
        for (uint32_t i = lane; i < bytes; i += 32u) d[i] = s[i];
    }
}

// Adler-32 of arbitrary ranges, one warp each (exported for tests; the deflate path fuses it into lz_match_kernel)
ZWZ_KERNEL adler32_kernel(const uint8_t *__restrict__ data, const uint64_t *__restrict__ off, const uint32_t *__restrict__ len,
                          uint32_t *adler, uint32_t n) {
    uint32_t c = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (c >= n) return;
    uint32_t a = enc_adler_global(data + off[c], len[c]);
    if (lane_id() == 0) adler[c] = a;
}

// concatenation of inflated records into contiguous files: one warp per record
ZWZ_KERNEL gather_records_kernel(const uint8_t *__restrict__ slots, const uint64_t *__restrict__ src_off, const uint64_t *__restrict__ dst_off,
                                 const uint32_t *__restrict__ len, uint8_t *dst, uint32_t n) {
    uint32_t c = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (c >= n) return;
    const uint8_t *s = slots + src_off[c];
    uint8_t *d = dst + dst_off[c];
    uint32_t bytes = len[c];
    unsigned lane = lane_id();
    if (((((uintptr_t) d) | ((uintptr_t) s)) & 15u) == 0u) {
        uint32_t nv = bytes >> 4;
        for (uint32_t i = lane; i < nv; i += 32u) ((uint4 *) d)[i] = ((const uint4 *) s)[i];
        for (uint32_t i = (nv << 4) + lane; i < bytes; i += 32u) d[i] = s[i];
    } else {
        for (uint32_t i = lane; i < bytes; i += 32u) d[i] = s[i];
    }
}

struct Arena {
    void *p = nullptr;
    size_t cap = 0;
    bool pinned = false;
};

// Deferred MD5 of one host-buffer batch (zwz_compress_files_async / zwz_decompress_records_async): the bytes to hash stay
// resident in `data` while the digests are computed on the context's second stream; the caller collects them with zwz_wait.
// Two slots per context, used alternately: the MD5 of batch k runs while batch k+1 goes through the main stream.
struct DigestSlot {
    Arena data;   // device: compress side = the raw files of the batch; decompress side = the concatenated output files
    Arena meta;   // device: MD5 descriptors + digests
    Arena pin;    // page-locked: descriptors (upload source) + digests (download target)
    zwz_rt::zwz_sync_event_t ev_in{}, ev_done{};
    bool pending = false;
    uint32_t n = 0;
    size_t digest_off = 0;     // where the digests land inside `pin`
    uint8_t *digest_dst = nullptr;
    uint64_t ticket = 0;
};

} // namespace zwz

struct zwz_ctx {
    int device = 0;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t total_mem = 0, smem_optin = 0;
    int inf_blocks_per_sm = 1; // resident inflate_kernel CTAs per SM
    int inf_dict_blocks_per_sm = 1; // the same for inflate_kernel<true>
    zwz_stream_t stream = nullptr;
    zwz_stream_t md5_stream = nullptr; // deferred digests (DigestSlot)
    zwz::DigestSlot slot[2];
    int next_slot = 0;
    uint64_t ticket_seq = 0;
    std::string err;
    uint64_t launches = 0;
    zwz::Arena meta, scratch, bulk_in, bulk_out, packed, pin_meta, pin_aux, counter;
    int inflate_mode = 0; // 0/1 = one warp per stream, 2 = one lane per stream, 3 = one warp per stream without the lane-parallel block decoder (ZWZ_INFLATE_MODE=warp|lanes|careful)
    bool arena_async = true; // ZWZ_ARENA_SYNC=1: plain cudaMalloc/cudaFree arenas (for A/B timing)
    bool trace = false;   // ZWZ_TRACE=1: wall-clock phases of the host-buffer calls on stderr (syncs the stream at every mark)
    size_t batch_raw_bytes = (size_t) 4 << 30; // raw bytes per internal deflate sub-batch (scratch = 6x that; ZWZ_BATCH_RAW_MB overrides)
    // The last deflate call's slot offsets and results: on the device in `keep` (which only deflate writes), and as a
    // host copy in `pin_keep` that zwz_pack_streams_device compares the caller's arrays with before it uses the device copy.
    // Layout of both: [slot_off u64 x keep_n], then at keep_res_off(keep_n) [results 16 B x keep_n].
    zwz::Arena keep, pin_keep;
    // preset dictionaries of the current call (zwz_*_dict): descriptors (device + page-locked staging), the dictionary records
    // built by dict_chain_kernel, and the dictionaries' bytes when the caller gave host memory
    zwz::Arena dict_meta, pin_dict, dict_arena, dict_data;
    std::vector<uint64_t> dict_host_off;
    uint32_t keep_n = 0; // 0 = nothing valid in keep / pin_keep
    // host threads for the descriptor work of large calls (ZWZ_TUNE_HOST_THREADS, ZWZ_TUNE_HOST_PARALLEL_MIN)
    unsigned host_threads = 0; // threads per call, the calling one included; 0 = min(8, cores / 2)
    uint64_t host_parallel_min = 32768; // calls with fewer entries run on the calling thread alone
    std::unique_ptr<zwz::HostPool> pool;
    // optional per-kernel timing
    bool profiling = false;
    struct Span {
        int kind;
        zwz_rt::zwz_event_t a, b;
    };
    std::vector<Span> spans;
    double prof_ms[ZWZ_PROF_N] = {0};
    uint64_t prof_n[ZWZ_PROF_N] = {0};
};

namespace {

using zwz::Arena;

int fail(zwz_ctx *ctx, int code, const char *what) {
    if (ctx) {
        std::string cuda;
        zwz_rt::last_error(cuda);
        ctx->err = what;
        if (!cuda.empty()) ctx->err += std::string(": ") + cuda;
    }
    return code;
}

int reserve(zwz_ctx *ctx, Arena &a, size_t bytes, bool pinned) {
    if (a.cap >= bytes && a.p) return ZWZ_OK;
    const size_t old_cap = a.p ? a.cap : 0;
    if (a.p) {
        zwz_rt::stream_sync(ctx->stream);
        if (a.pinned) zwz_rt::free_pinned(a.p); else if (ctx->arena_async) zwz_rt::free_arena(a.p, ctx->stream); else zwz_rt::free_device(a.p);
        a.p = nullptr;
        a.cap = 0;
    }
    // grow-only, with headroom (batches of one job differ by a few percent) and geometric from the second time on: a job whose
    // batches hold more and more, smaller and smaller files (the size-sorted deal) would otherwise re-allocate its descriptor
    // arenas batch after batch — and a re-allocation waits for the device, i.e. for every other worker's kernels
    // (profiles/round2_notes.md: 50-500 ms `reserve` phases in the end-to-end trace)
    size_t want = bytes + bytes / 4 + 4096;
    if (old_cap) want = std::max(want, std::min(old_cap * 2, bytes + ((size_t) 1 << 30)));
    int rc = pinned ? zwz_rt::malloc_pinned(&a.p, want) : (ctx->arena_async ? zwz_rt::malloc_arena(&a.p, want, ctx->stream) : zwz_rt::malloc_device(&a.p, want));
    if (rc) {
        a.p = nullptr;
        return fail(ctx, ZWZ_E_NOMEM, pinned ? "pinned allocation failed" : "device allocation failed");
    }
    a.cap = want;
    a.pinned = pinned;
    return ZWZ_OK;
}

void release(zwz_ctx *ctx, Arena &a) {
    if (!a.p) return;
    if (a.pinned) zwz_rt::free_pinned(a.p); else if (ctx->arena_async) zwz_rt::free_arena(a.p, ctx->stream); else zwz_rt::free_device(a.p);
    a.p = nullptr;
    a.cap = 0;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

inline size_t keep_res_off(size_t n) { return align_up(n * 8, 256); }

unsigned host_thread_count(const zwz_ctx *ctx) {
    return ctx->host_threads ? ctx->host_threads : std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2));
}

// Number of blocks an O(n) host pass over n entries is cut into: one per host thread from host_parallel_min entries on, else 1.
unsigned host_blocks(zwz_ctx *ctx, size_t n) {
    const unsigned t = host_thread_count(ctx);
    return t > 1 && n >= ctx->host_parallel_min ? t : 1u;
}

// f(b, lo, hi) for the nb blocks [lo, hi) of [0, n), block b starting at n * b / nb; on the context's host threads when nb > 1
template <class F> void host_for(zwz_ctx *ctx, unsigned nb, size_t n, F &&f) {
    if (nb > 1 && !ctx->pool) {
        try {
            ctx->pool.reset(new zwz::HostPool(host_thread_count(ctx) - 1));
        } catch (...) { // no threads to be had: this call and the next ones run on the calling thread
            ctx->pool.reset();
            ctx->host_threads = 1;
            nb = 1;
        }
    }
    auto blk = [&](unsigned b) { f(b, n * b / nb, n * (b + 1) / nb); };
    if (nb <= 1) {
        f(0u, (size_t) 0, n);
        return;
    }
    ctx->pool->run(nb, std::function<void(unsigned)>(blk));
}

// Stores into page-locked memory that the copy engine reads next, from the host threads: non-temporal, so that the lines are in
// DRAM and not left dirty in the private caches of several cores, from where the DMA read of a descriptor upload ran at a
// quarter of its speed on B200 hosts (profiles/step_gaps). The calling thread alone keeps plain stores: its small batches are
// read from the cache it wrote them to.
struct Staging {
    bool nt;
    explicit Staging(unsigned nb) : nt(nb > 1) {}
    void put(uint64_t *p, uint64_t v) const {
#if defined(__x86_64__)
        if (nt) return _mm_stream_si64((long long *) p, (long long) v);
#endif
        *p = v;
    }
    void put(uint32_t *p, uint32_t v) const {
#if defined(__x86_64__)
        if (nt) return _mm_stream_si32((int *) p, (int) v);
#endif
        *p = v;
    }
    void copy(void *dst, const void *src, size_t bytes) const {
#if defined(__x86_64__)
        if (nt) {
            uint8_t *d = (uint8_t *) dst;
            const uint8_t *s = (const uint8_t *) src;
            const size_t head = std::min(bytes, (size_t) (-(uintptr_t) d & 15u));
            memcpy(d, s, head);
            size_t i = head;
            for (; i + 16 <= bytes; i += 16) _mm_stream_si128((__m128i *) (d + i), _mm_loadu_si128((const __m128i *) (s + i)));
            memcpy(d + i, s + i, bytes - i);
            return;
        }
#endif
        memcpy(dst, src, bytes);
    }
    // at the end of a block: the non-temporal stores are globally visible before the upload is queued
    void done() const {
#if defined(__x86_64__)
        if (nt) _mm_sfence();
#endif
    }
};

// memcpy of a descriptor array of `entries` entries
void host_copy(zwz_ctx *ctx, void *dst, const void *src, size_t bytes, size_t entries) {
    host_for(ctx, host_blocks(ctx, entries), bytes, [&](unsigned, size_t lo, size_t hi) {
        memcpy((uint8_t *) dst + lo, (const uint8_t *) src + lo, hi - lo);
    });
}

// RAII bracket: records an event pair around one kernel launch when profiling is on
struct ProfSpan {
    zwz_ctx *ctx;
    zwz_stream_t st;
    zwz_ctx::Span sp;
    bool on;
    ProfSpan(zwz_ctx *c, int kind, zwz_stream_t s) : ctx(c), st(s), on(c->profiling) {
        sp.kind = kind;
        if (on) zwz_rt::event_record(&sp.a, st);
    }
    ~ProfSpan() {
        if (on) {
            zwz_rt::event_record(&sp.b, st);
            ctx->spans.push_back(sp);
        }
    }
};

int check_launch(zwz_ctx *ctx, const char *what) {
    ctx->launches++;
    std::string msg;
    if (zwz_rt::last_error(msg)) {
        ctx->err = std::string(what) + ": " + msg;
        return ZWZ_E_CUDA;
    }
    return ZWZ_OK;
}

// ZWZ_TRACE=1: phase times of a call (debugging aid: every mark synchronises the call's stream, so a phase that queues
// device work also holds that work's run time)
struct Trace {
    zwz_ctx *ctx;
    const char *call;
    zwz_stream_t st;
    double t0;
    std::string line;
    static double now() {
        struct timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
    }
    Trace(zwz_ctx *c, const char *name, zwz_stream_t s = nullptr) : ctx(c), call(name), st(s ? s : c->stream), t0(c->trace ? now() : 0.0) {}
    void mark(const char *what) {
        if (!ctx->trace) return;
        zwz_rt::stream_sync(st);
        double t = now();
        char buf[64];
        snprintf(buf, sizeof buf, " %s %.2f ms,", what, (t - t0) * 1e3);
        line += buf;
        t0 = t;
    }
    ~Trace() {
        if (ctx->trace && !line.empty()) fprintf(stderr, "[zwz trace %p] %s:%s\n", (void *) ctx, call, line.c_str());
    }
};

#ifndef ZWZ_L0_DEPTH
#define ZWZ_L0_DEPTH 12
#define ZWZ_L0_NICE 48
#endif
struct LevelParams {
    uint32_t depth, nice;
};
LevelParams level_params(int level) {
    // search effort per level (hash-chain candidates per position, stop length). 0 = default: the cheapest setting that
    // stays inside the 3 % size tolerance on every corpus class (tests/test_kernels.py::test_deflate_ratio...)
    static const LevelParams t[10] = {{ZWZ_L0_DEPTH, ZWZ_L0_NICE}, {4, 16}, {6, 24}, {8, 32}, {16, 64}, {24, 96}, {32, 128}, {64, 160}, {128, 258}, {512, 258}};
    if (level < 0 || level > 9) level = 0;
    return t[level];
}

// Preset dictionaries of one call (zwz_*_dict). Checks `d` for n chunks / streams and stages the per-entry dictionary index (on
// the host threads above host_parallel_min; an empty dictionary becomes ZWZ_NO_DICT: it is no dictionary). `refuse`: the format
// or decoder takes no dictionary, so any entry that names one is ZWZ_E_ARG. When some entry has a dictionary, every dictionary
// of the table gets its record (dict_chain_kernel) and its DICTID (adler32_kernel) on stream st, and *out points at them;
// otherwise *out stays empty and the call launches what the call without dictionaries launches.
int stage_dicts(zwz_ctx *ctx, const zwz_dicts *d, uint32_t n, bool refuse, zwz_stream_t st, zwz::DictTable *out) {
    *out = zwz::DictTable{};
    if (!d) return ZWZ_OK;
    if (!d->off) return fail(ctx, ZWZ_E_ARG, "null dictionary offsets");
    const uint32_t nd = d->ndict;
    for (uint32_t k = 0; k < nd; ++k)
        if (d->off[k + 1] < d->off[k] || d->off[k + 1] - d->off[k] > ((uint64_t) 1 << 30))
            return fail(ctx, ZWZ_E_ARG, "dictionary offsets must not decrease, dictionaries hold at most 2^30 bytes");
    if (nd && d->off[nd] > d->off[0] && !d->data) return fail(ctx, ZWZ_E_ARG, "null dictionary data");
    const size_t m_off = align_up((size_t) n * 4, 256), m_woff = m_off + (size_t) nd * 8, m_len = m_woff + (size_t) nd * 8,
                 m_wlen = m_len + (size_t) nd * 4, m_id = m_wlen + (size_t) nd * 4;
    int rc;
    if ((rc = reserve(ctx, ctx->pin_dict, m_id, true))) return rc;
    uint8_t *hp = (uint8_t *) ctx->pin_dict.p;
    uint32_t *h_idx = (uint32_t *) hp;
    const unsigned nb = host_blocks(ctx, n);
    std::vector<char> bad(nb, 0), named(nb, 0), used(nb, 0);
    const Staging stg(nb);
    host_for(ctx, nb, n, [&](unsigned b, size_t lo, size_t hi) {
        bool b_bad = false, b_named = false, b_used = false; // per block in registers: the flags of all blocks share a cache line
        for (size_t i = lo; i < hi; ++i) {
            const uint32_t k = d->idx ? d->idx[i] : (nd ? 0u : ZWZ_NO_DICT);
            const bool ok = k < nd && d->off[k + 1] > d->off[k];
            b_bad |= k != ZWZ_NO_DICT && k >= nd;
            b_named |= k != ZWZ_NO_DICT;
            b_used |= ok;
            stg.put(h_idx + i, ok ? k : ZWZ_NO_DICT);
        }
        stg.done();
        bad[b] = b_bad;
        named[b] = b_named;
        used[b] = b_used;
    });
    auto any = [](const std::vector<char> &v) { return std::any_of(v.begin(), v.end(), [](char c) { return c != 0; }); };
    if (any(bad)) return fail(ctx, ZWZ_E_ARG, "dictionary index out of range");
    if (refuse && any(named)) return fail(ctx, ZWZ_E_ARG, "no preset dictionary in gzip format or with the one-lane-per-stream decoder");
    if (!any(used)) return ZWZ_OK;
    for (uint32_t k = 0; k < nd; ++k) {
        const uint64_t l = d->off[k + 1] - d->off[k], w = std::min<uint64_t>(l, ZWZ_MAX_DIST);
        ((uint64_t *) (hp + m_off))[k] = d->off[k];
        ((uint64_t *) (hp + m_woff))[k] = d->off[k] + l - w;
        ((uint32_t *) (hp + m_len))[k] = (uint32_t) l;
        ((uint32_t *) (hp + m_wlen))[k] = (uint32_t) w;
    }
    if ((rc = reserve(ctx, ctx->dict_meta, m_id + (size_t) nd * 4 + 256, false))) return rc;
    if ((rc = reserve(ctx, ctx->dict_arena, (size_t) nd * ZWZ_DICT_STRIDE, false))) return rc;
    uint8_t *dm = (uint8_t *) ctx->dict_meta.p;
    if (zwz_rt::memcpy_h2d(dm, hp, m_id, st)) return fail(ctx, ZWZ_E_CUDA, "dictionary descriptor upload failed");
    {
        ProfSpan ps(ctx, ZWZ_PROF_ADLER, st);
        ZWZ_LAUNCH(zwz::dict_chain_kernel, nd, 1024, ZWZ_DICT_SMEM, st, d->data, (const uint64_t *) (dm + m_woff), (const uint32_t *) (dm + m_wlen),
                   (uint8_t *) ctx->dict_arena.p);
    }
    if ((rc = check_launch(ctx, "dict_chain_kernel"))) return rc;
    {
        ProfSpan ps(ctx, ZWZ_PROF_ADLER, st);
        ZWZ_LAUNCH(zwz::adler32_kernel, (nd + 7) / 8, 256, 0, st, d->data, (const uint64_t *) (dm + m_off), (const uint32_t *) (dm + m_len),
                   (uint32_t *) (dm + m_id), nd);
    }
    if ((rc = check_launch(ctx, "adler32_kernel"))) return rc;
    out->idx = (const uint32_t *) dm;
    out->arena = (const uint8_t *) ctx->dict_arena.p;
    out->wlen = (const uint32_t *) (dm + m_wlen);
    out->id = (const uint32_t *) (dm + m_id);
    return ZWZ_OK;
}

// The plain (host-buffer) calls: the dictionaries' bytes go to the device once per call. *out is *d with device data and
// offsets relative to it (kept in the context until the next call).
int upload_dicts(zwz_ctx *ctx, const zwz_dicts *d, zwz_dicts *out) {
    if (!d) return ZWZ_OK;
    *out = *d;
    if (!d->off || d->ndict == 0) return ZWZ_OK; // stage_dicts names the error
    const uint64_t lo = d->off[0], hi = d->off[d->ndict];
    if (hi < lo) return fail(ctx, ZWZ_E_ARG, "dictionary offsets must not decrease");
    if (hi > lo && !d->data) return fail(ctx, ZWZ_E_ARG, "null dictionary data");
    ctx->dict_host_off.resize(d->ndict + 1);
    for (uint32_t k = 0; k <= d->ndict; ++k) ctx->dict_host_off[k] = d->off[k] - lo;
    int rc;
    if ((rc = reserve(ctx, ctx->dict_data, (size_t) (hi - lo) + 64, false))) return rc;
    if (zwz_rt::memcpy_h2d(ctx->dict_data.p, d->data + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "dictionary upload failed");
    out->data = (const uint8_t *) ctx->dict_data.p;
    out->off = ctx->dict_host_off.data();
    return ZWZ_OK;
}

} // namespace

extern "C" {

int zwz_abi_version(void) { return ZWZ_ABI_VERSION; }
int zwz_device_count(void) { return zwz_rt::device_count(); }

int zwz_init(int device, zwz_ctx **out) {
    if (!out) return ZWZ_E_ARG;
    *out = nullptr;
    if (device < 0 || device >= zwz_rt::device_count()) return ZWZ_E_NODEVICE;
    if (zwz_rt::set_device(device)) return ZWZ_E_NODEVICE;
    zwz_ctx *ctx = new (std::nothrow) zwz_ctx();
    if (!ctx) return ZWZ_E_NOMEM;
    ctx->device = device;
    if (zwz_rt::device_props(device, &ctx->sm_count, &ctx->cc_major, &ctx->cc_minor, &ctx->total_mem, &ctx->smem_optin)) {
        delete ctx;
        return ZWZ_E_NODEVICE;
    }
#ifndef ZWZ_EMU
    if (ctx->cc_major != 10) { // the fatbin holds sm_100a SASS only
        delete ctx;
        return ZWZ_E_NODEVICE;
    }
#endif
    if (ctx->smem_optin < zwz::MatchClass<3>::kSmem || zwz_rt::stream_create(&ctx->stream) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<0>, zwz::MatchClass<0>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<1>, zwz::MatchClass<1>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<2>, zwz::MatchClass<2>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<3>, zwz::MatchClass<3>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<0, true>, zwz::MatchClass<0>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<1, true>, zwz::MatchClass<1>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<2, true>, zwz::MatchClass<2>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::lz_match_kernel<3, true>, zwz::MatchClass<3>::kSmem) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::dict_chain_kernel, ZWZ_DICT_SMEM) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::inflate_kernel<true>, ZWZ_INF_SMEM) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::md5_files_staged_kernel, ZWZ_MD5S_SMEM) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::inflate_kernel<false>, ZWZ_INF_SMEM) ||
        zwz_rt::set_max_dyn_smem((const void *) zwz::inflate_lanes_kernel, ZWZ_IL_SMEM)) {
        delete ctx;
        return ZWZ_E_NODEVICE;
    }
    if (zwz_rt::max_blocks_per_sm(&ctx->inf_blocks_per_sm, (const void *) zwz::inflate_kernel<false>, ZWZ_INF_WARPS * 32, ZWZ_INF_SMEM) ||
        zwz_rt::max_blocks_per_sm(&ctx->inf_dict_blocks_per_sm, (const void *) zwz::inflate_kernel<true>, ZWZ_INF_WARPS * 32, ZWZ_INF_SMEM)) {
        delete ctx;
        return ZWZ_E_NODEVICE;
    }
    if (zwz_rt::stream_create(&ctx->md5_stream)) {
        delete ctx;
        return ZWZ_E_NODEVICE;
    }
    for (auto &sl : ctx->slot)
        if (zwz_rt::sync_event_create(&sl.ev_in) || zwz_rt::sync_event_create(&sl.ev_done)) {
            delete ctx;
            return ZWZ_E_NODEVICE;
        }
    zwz_rt::keep_pool_memory(device);
    zwz_rt::preload_kernel((const void *) zwz::deflate_encode_kernel<false>);
    zwz_rt::preload_kernel((const void *) zwz::inflate_kernel<false>);
    zwz_rt::preload_kernel((const void *) zwz::md5_files_kernel);
    zwz_rt::preload_kernel((const void *) zwz::pack_streams_kernel);
    zwz_rt::preload_kernel((const void *) zwz::gather_records_kernel);
    zwz_rt::preload_kernel((const void *) zwz::adler32_kernel);
    zwz_rt::preload_kernel((const void *) zwz::crc32_kernel);
    if (const char *e = getenv("ZWZ_ARENA_SYNC")) ctx->arena_async = !(*e && *e != '0');
    if (const char *e = getenv("ZWZ_TRACE")) ctx->trace = *e && *e != '0';
    if (const char *e = getenv("ZWZ_INFLATE_MODE")) ctx->inflate_mode = !strcmp(e, "warp") ? 1 : (!strcmp(e, "lanes") ? 2 : (!strcmp(e, "careful") ? 3 : 0));
    if (const char *e = getenv("ZWZ_BATCH_RAW_MB")) {
        long v = atol(e);
        if (v >= 1) ctx->batch_raw_bytes = (size_t) v << 20;
    }
    *out = ctx;
    return ZWZ_OK;
}

void zwz_destroy(zwz_ctx *ctx) {
    if (!ctx) return;
    zwz_rt::set_device(ctx->device);
    zwz_rt::stream_sync(ctx->stream);
    zwz_rt::stream_sync(ctx->md5_stream);
    for (auto &sl : ctx->slot) {
        release(ctx, sl.data);
        release(ctx, sl.meta);
        release(ctx, sl.pin);
        zwz_rt::sync_event_destroy(sl.ev_in);
        zwz_rt::sync_event_destroy(sl.ev_done);
    }
    release(ctx, ctx->meta);
    release(ctx, ctx->scratch);
    release(ctx, ctx->bulk_in);
    release(ctx, ctx->bulk_out);
    release(ctx, ctx->packed);
    release(ctx, ctx->pin_meta);
    release(ctx, ctx->pin_aux);
    release(ctx, ctx->counter);
    release(ctx, ctx->keep);
    release(ctx, ctx->pin_keep);
    release(ctx, ctx->dict_meta);
    release(ctx, ctx->pin_dict);
    release(ctx, ctx->dict_arena);
    release(ctx, ctx->dict_data);
    ctx->pool.reset(); // joins the host threads
    zwz_rt::stream_sync(ctx->stream);
    zwz_rt::stream_destroy(ctx->stream);
    zwz_rt::stream_destroy(ctx->md5_stream);
    delete ctx;
}

const char *zwz_last_error(const zwz_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

int zwz_ctx_tune(zwz_ctx *ctx, int what, uint64_t value) {
    if (!ctx) return ZWZ_E_ARG;
    if (what == ZWZ_TUNE_DEFLATE_SUBBATCH_BYTES) {
        if (value < ((uint64_t) 1 << 20)) return fail(ctx, ZWZ_E_ARG, "sub-batch below 1 MiB");
        ctx->batch_raw_bytes = (size_t) value;
        return ZWZ_OK;
    }
    if (what == ZWZ_TUNE_HOST_THREADS) {
        if (value > 256) return fail(ctx, ZWZ_E_ARG, "more than 256 host threads");
        ctx->pool.reset(); // the next call that wants threads starts as many as asked
        ctx->host_threads = (unsigned) value;
        return ZWZ_OK;
    }
    if (what == ZWZ_TUNE_HOST_PARALLEL_MIN) {
        ctx->host_parallel_min = value;
        return ZWZ_OK;
    }
    return fail(ctx, ZWZ_E_ARG, "unknown tuning knob");
}

int zwz_device_props(const zwz_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem) {
    if (!ctx) return ZWZ_E_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (total_mem) *total_mem = ctx->total_mem;
    return ZWZ_OK;
}

uint64_t zwz_launch_count(const zwz_ctx *ctx) { return ctx ? ctx->launches : 0; }

int zwz_profile_enable(zwz_ctx *ctx, int on) {
    if (!ctx) return ZWZ_E_ARG;
    ctx->profiling = on != 0;
    return ZWZ_OK;
}
int zwz_profile_read(zwz_ctx *ctx, double *ms, uint64_t *launches, int reset) {
    if (!ctx) return ZWZ_E_ARG;
#ifndef ZWZ_EMU
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(ctx, ZWZ_E_CUDA, "device sync failed");
#endif
    for (auto &sp : ctx->spans) {
        ctx->prof_ms[sp.kind] += zwz_rt::event_elapsed_and_free(sp.a, sp.b);
        ctx->prof_n[sp.kind] += 1;
    }
    ctx->spans.clear();
    for (int k = 0; k < ZWZ_PROF_N; ++k) {
        if (ms) ms[k] = ctx->prof_ms[k];
        if (launches) launches[k] = ctx->prof_n[k];
        if (reset) {
            ctx->prof_ms[k] = 0;
            ctx->prof_n[k] = 0;
        }
    }
    return ZWZ_OK;
}

int zwz_malloc_device(zwz_ctx *ctx, size_t bytes, void **ptr) {
    if (!ctx || !ptr) return ZWZ_E_ARG;
    zwz_rt::set_device(ctx->device);
    return zwz_rt::malloc_device(ptr, bytes) ? fail(ctx, ZWZ_E_NOMEM, "device allocation failed") : ZWZ_OK;
}
int zwz_free_device(zwz_ctx *ctx, void *ptr) {
    if (!ctx) return ZWZ_E_ARG;
    zwz_rt::set_device(ctx->device);
    zwz_rt::stream_sync(ctx->stream);
    return zwz_rt::free_device(ptr) ? fail(ctx, ZWZ_E_CUDA, "cudaFree failed") : ZWZ_OK;
}
int zwz_malloc_pinned(zwz_ctx *ctx, size_t bytes, void **ptr) {
    if (!ctx || !ptr) return ZWZ_E_ARG;
    zwz_rt::set_device(ctx->device);
    return zwz_rt::malloc_pinned(ptr, bytes) ? fail(ctx, ZWZ_E_NOMEM, "pinned allocation failed") : ZWZ_OK;
}
int zwz_free_pinned(zwz_ctx *ctx, void *ptr) {
    if (!ctx) return ZWZ_E_ARG;
    return zwz_rt::free_pinned(ptr) ? fail(ctx, ZWZ_E_CUDA, "cudaFreeHost failed") : ZWZ_OK;
}
int zwz_memcpy_h2d(zwz_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx) return ZWZ_E_ARG;
    zwz_rt::set_device(ctx->device);
    if (zwz_rt::memcpy_h2d(dst, src, bytes, ctx->stream) || zwz_rt::stream_sync(ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "h2d copy failed");
    return ZWZ_OK;
}
int zwz_memcpy_d2h(zwz_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx) return ZWZ_E_ARG;
    zwz_rt::set_device(ctx->device);
    if (zwz_rt::memcpy_d2h(dst, src, bytes, ctx->stream) || zwz_rt::stream_sync(ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "d2h copy failed");
    return ZWZ_OK;
}
int zwz_sync(zwz_ctx *ctx) {
    if (!ctx) return ZWZ_E_ARG;
    return zwz_rt::stream_sync(ctx->stream) ? fail(ctx, ZWZ_E_CUDA, "stream sync failed") : ZWZ_OK;
}

// ======================================================================================================================
// deflate
// ======================================================================================================================
int zwz_deflate_batch_device(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_out,
                             const uint64_t *out_off, zwz_deflate_result *res, int level, void *stream_v) {
    return zwz_deflate_batch_device_ex(ctx, d_raw, off, len, n, d_out, out_off, res, level, ZWZ_FORMAT_ZLIB, stream_v);
}

int zwz_deflate_batch_device_ex(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_out,
                                const uint64_t *out_off, zwz_deflate_result *res, int level, int format, void *stream_v) {
    return zwz_deflate_batch_device_dict(ctx, d_raw, off, len, n, d_out, out_off, res, level, format, nullptr, stream_v);
}

int zwz_deflate_batch_device_dict(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_out,
                                  const uint64_t *out_off, zwz_deflate_result *res, int level, int format, const zwz_dicts *dicts, void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (format < ZWZ_FORMAT_ZLIB || format > ZWZ_FORMAT_RAW) return fail(ctx, ZWZ_E_ARG, "unknown stream format");
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !out_off || !res || !d_out) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    Trace tr(ctx, "deflate_device", st);
    ctx->keep_n = 0;
    // uint32 scratch entries of a chunk: best match per position (+ pad so the parser may peek one past the end), then the u16
    // position lists of lz_match_kernel (deflate_match.cuh: dm_scratch_match_words; zwz_common.cuh: scratch layout)
    auto scr_words = [](uint32_t l) { return align_up((size_t) l + 2, 32) + align_up(((size_t) l + 1) / 2 + 32, 32) + ZWZ_SCR_FLAG_WORDS; };
    // validation, raw bytes and scratch words per block: the first bad chunk of the first block that has one names the error
    struct Part {
        uint64_t raw = 0, scr = 0;
        const char *bad = nullptr;
    };
    const unsigned nb = host_blocks(ctx, n);
    std::vector<Part> part(nb);
    host_for(ctx, nb, n, [&](unsigned k, size_t lo, size_t hi) {
        Part p;
        for (size_t i = lo; i < hi && !p.bad; ++i) {
            if (len[i] > ZWZ_CHUNK_SIZE) p.bad = "chunk longer than 65535 bytes";
            else if (format == ZWZ_FORMAT_GZIP && len[i] > ZWZ_BGZF_BLOCK) p.bad = "gzip chunk longer than ZWZ_BGZF_BLOCK bytes";
            else if (out_off[i] & 3u) p.bad = "out_off must be a multiple of 4";
            p.raw += len[i];
            p.scr += scr_words(len[i]);
        }
        part[k] = p;
    });
    uint64_t total_raw = 0, total_scr = 0;
    for (const Part &p : part) {
        if (p.bad) return fail(ctx, ZWZ_E_ARG, p.bad);
        total_raw += p.raw;
        total_scr += p.scr;
    }
    if (total_raw && !d_raw) return fail(ctx, ZWZ_E_ARG, "null raw buffer");
    zwz::DictTable dict{};
    int rc;
    if ((rc = stage_dicts(ctx, dicts, n, format == ZWZ_FORMAT_GZIP, st, &dict))) return rc;
    tr.mark("validate");

    // descriptors: [raw_off u64][scr_off u64][raw_len u32][order u32] per chunk, then Adler-32 + match counts on the device;
    // slot offsets and results in the keep arenas ([out_off u64][results 16 B] per chunk)
    const size_t meta_bytes = (size_t) n * (8 + 8 + 4 + 4), keep_bytes = keep_res_off(n) + (size_t) n * 16;
    const size_t dev_meta_bytes = align_up(meta_bytes, 256) + (size_t) n * 8 + 256;
    if ((rc = reserve(ctx, ctx->pin_meta, meta_bytes, true))) return rc;
    if ((rc = reserve(ctx, ctx->meta, dev_meta_bytes, false))) return rc;
    if ((rc = reserve(ctx, ctx->pin_keep, keep_bytes, true))) return rc;
    if ((rc = reserve(ctx, ctx->keep, keep_bytes, false))) return rc;

    uint64_t *h_raw_off = (uint64_t *) ctx->pin_meta.p;
    uint64_t *h_scr_off = h_raw_off + n;
    uint32_t *h_len = (uint32_t *) (h_scr_off + n);
    uint32_t *h_order = h_len + n;
    uint64_t *h_out_off = (uint64_t *) ctx->pin_keep.p;

    // sub-batches bounded by scratch: a new one starts at the chunk that would take the current one past batch_raw_bytes
    std::vector<uint32_t> sub_begin{0};
    if (total_raw > ctx->batch_raw_bytes) {
        uint64_t raw = 0;
        for (uint32_t i = 0; i < n; ++i) {
            if (raw + len[i] > ctx->batch_raw_bytes && i > sub_begin.back()) {
                sub_begin.push_back(i);
                raw = 0;
            }
            raw += len[i];
        }
    }
    sub_begin.push_back(n);
    const size_t nsub = sub_begin.size() - 1;
    // scratch offsets: a blocked prefix sum over all chunks, then restarted at 0 in every sub-batch
    const Staging stg(nb);
    host_for(ctx, nb, n, [&](unsigned k, size_t lo, size_t hi) {
        uint64_t scr = 0;
        for (unsigned j = 0; j < k; ++j) scr += part[j].scr;
        for (size_t i = lo; i < hi; ++i) {
            stg.put(h_raw_off + i, off[i]);
            stg.put(h_scr_off + i, scr);
            stg.put(h_out_off + i, out_off[i]);
            stg.put(h_len + i, len[i]);
            scr += scr_words(len[i]);
        }
        stg.done();
    });
    size_t max_scr = 0;
    for (size_t s = 0; s < nsub; ++s) {
        const uint64_t s0 = h_scr_off[sub_begin[s]], s1 = s + 1 < nsub ? h_scr_off[sub_begin[s + 1]] : total_scr;
        max_scr = std::max<size_t>(max_scr, s1 - s0);
        if (s)
            for (uint32_t i = sub_begin[s]; i < sub_begin[s + 1]; ++i) h_scr_off[i] -= s0;
    }
    tr.mark("stage");
    if ((rc = reserve(ctx, ctx->scratch, max_scr * 4 + 256, false))) return rc;
    // size classes (deflate_match.cuh): per sub-batch, chunk indices grouped by class in index order (one counting pass,
    // counts per class and block, then a scatter), longest first inside a class so the persistent CTAs end together
    std::vector<uint32_t> cls_begin(nsub * 5);
    static const uint32_t kClassHi[3] = {zwz::MatchClass<0>::kCap, zwz::MatchClass<1>::kCap, zwz::MatchClass<2>::kCap};
    static_assert(zwz::MatchClass<3>::kCap >= ZWZ_CHUNK_SIZE, "every chunk has a size class");
    auto cls_of = [](uint32_t l) -> unsigned { return l <= kClassHi[0] ? 0u : (l <= kClassHi[1] ? 1u : (l <= kClassHi[2] ? 2u : 3u)); };
    for (size_t s = 0; s < nsub; ++s) {
        const uint32_t b = sub_begin[s], e = sub_begin[s + 1];
        uint32_t *o = h_order + b;
        const unsigned sb = host_blocks(ctx, e - b);
        std::vector<uint32_t> pos((size_t) sb * 4);
        host_for(ctx, sb, e - b, [&](unsigned k, size_t lo, size_t hi) {
            uint32_t c[4] = {0, 0, 0, 0};
            for (size_t i = lo; i < hi; ++i) c[cls_of(len[b + i])]++;
            for (int cls = 0; cls < 4; ++cls) pos[(size_t) k * 4 + cls] = c[cls];
        });
        uint32_t k = 0;
        for (int cls = 0; cls < 4; ++cls) {
            cls_begin[s * 5 + cls] = k;
            for (unsigned j = 0; j < sb; ++j) {
                const uint32_t c = pos[(size_t) j * 4 + cls];
                pos[(size_t) j * 4 + cls] = k;
                k += c;
            }
        }
        cls_begin[s * 5 + 4] = k;
        const Staging so(sb);
        host_for(ctx, sb, e - b, [&](unsigned j, size_t lo, size_t hi) {
            uint32_t *p = &pos[(size_t) j * 4];
            for (size_t i = lo; i < hi; ++i) so.put(o + p[cls_of(len[b + i])]++, (uint32_t) i);
            so.done();
        });
        // the four classes side by side (size-sorted shards, the reference's deal, skip the sort)
        host_for(ctx, sb > 1 ? 4u : 1u, 4, [&](unsigned, size_t c0, size_t c1) {
            auto longer = [&](uint32_t x, uint32_t y) { return len[b + x] > len[b + y]; };
            for (size_t cls = c0; cls < c1; ++cls) {
                uint32_t *o0 = o + cls_begin[s * 5 + cls], *o1 = o + cls_begin[s * 5 + cls + 1];
                if (!std::is_sorted(o0, o1, longer)) std::stable_sort(o0, o1, longer);
            }
        });
    }
    tr.mark("partition");
    if ((rc = reserve(ctx, ctx->counter, nsub * 32 + 256, false))) return rc;
    if (zwz_rt::memset_device(ctx->counter.p, 0, nsub * 32, st)) return fail(ctx, ZWZ_E_CUDA, "memset failed");

    uint8_t *dm = (uint8_t *) ctx->meta.p;
    uint8_t *dk = (uint8_t *) ctx->keep.p;
    if (zwz_rt::memcpy_h2d(dm, ctx->pin_meta.p, meta_bytes, st) || zwz_rt::memcpy_h2d(dk, h_out_off, (size_t) n * 8, st))
        return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    tr.mark("upload");
    uint32_t *d_res = (uint32_t *) (dk + keep_res_off(n));
    uint32_t *d_adler = (uint32_t *) (dm + align_up(meta_bytes, 256));
    uint32_t *d_nmatch = d_adler + n;

    const LevelParams lp = level_params(level);
    for (size_t s = 0; s + 1 < sub_begin.size(); ++s) {
        uint32_t b = sub_begin[s], e = sub_begin[s + 1];
        zwz::DeflateJob job;
        job.raw = d_raw;
        job.raw_off = (const uint64_t *) dm + b;
        job.scr_off = (const uint64_t *) dm + n + b;
        job.out_off = (const uint64_t *) dk + b;
        job.raw_len = (const uint32_t *) ((const uint64_t *) dm + 2 * (size_t) n) + b;
        job.scratch = (uint32_t *) ctx->scratch.p;
        job.adler = d_adler + b;
        job.nmatch = d_nmatch + b;
        job.out = d_out;
        job.res = d_res + (size_t) b * 4;
        job.n = e - b;
        job.depth = lp.depth;
        job.nice = lp.nice;
        job.work_counter = nullptr;
        job.format = (uint32_t) format;
        job.dict = dict;
        if (dict.idx) job.dict.idx = dict.idx + b;
        const uint32_t *d_order = (const uint32_t *) ((const uint64_t *) dm + 2 * (size_t) n) + n + b;
        uint32_t *d_counters = (uint32_t *) ctx->counter.p + s * 8; // [0..3] match classes, [4] encoder
        for (int cls = 0; cls < 4; ++cls) {
            uint32_t w0 = cls_begin[s * 5 + cls], w1 = cls_begin[s * 5 + cls + 1];
            if (w1 == w0) continue;
            ProfSpan ps(ctx, ZWZ_PROF_MATCH, st);
            const uint32_t nwork = w1 - w0, sms = (uint32_t) ctx->sm_count;
            if (dict.idx) { // the DICT instantiations only when some chunk of the call has a dictionary
                auto *k0 = zwz::lz_match_kernel<0, true>, *k1 = zwz::lz_match_kernel<1, true>, *k2 = zwz::lz_match_kernel<2, true>,
                     *k3 = zwz::lz_match_kernel<3, true>;
                if (cls == 0) ZWZ_LAUNCH(k0, std::min(nwork, sms * 6u), zwz::MatchClass<0>::kThreads, zwz::MatchClass<0>::kSmem, st, job, d_order + w0, nwork, d_counters + cls);
                else if (cls == 1) ZWZ_LAUNCH(k1, std::min(nwork, sms * 3u), zwz::MatchClass<1>::kThreads, zwz::MatchClass<1>::kSmem, st, job, d_order + w0, nwork, d_counters + cls);
                else if (cls == 2) ZWZ_LAUNCH(k2, std::min(nwork, sms * 2u), zwz::MatchClass<2>::kThreads, zwz::MatchClass<2>::kSmem, st, job, d_order + w0, nwork, d_counters + cls);
                else ZWZ_LAUNCH(k3, std::min(nwork, sms), zwz::MatchClass<3>::kThreads, zwz::MatchClass<3>::kSmem, st, job, d_order + w0, nwork, d_counters + cls);
            } else if (cls == 0) {
                ZWZ_LAUNCH(zwz::lz_match_kernel<0>, std::min(nwork, sms * 6u), zwz::MatchClass<0>::kThreads, zwz::MatchClass<0>::kSmem, st, job,
                           d_order + w0, nwork, d_counters + cls);
            } else if (cls == 1) {
                ZWZ_LAUNCH(zwz::lz_match_kernel<1>, std::min(nwork, sms * 3u), zwz::MatchClass<1>::kThreads, zwz::MatchClass<1>::kSmem, st, job,
                           d_order + w0, nwork, d_counters + cls);
            } else if (cls == 2) {
                ZWZ_LAUNCH(zwz::lz_match_kernel<2>, std::min(nwork, sms * 2u), zwz::MatchClass<2>::kThreads, zwz::MatchClass<2>::kSmem, st, job,
                           d_order + w0, nwork, d_counters + cls);
            } else {
                ZWZ_LAUNCH(zwz::lz_match_kernel<3>, std::min(nwork, sms), zwz::MatchClass<3>::kThreads, zwz::MatchClass<3>::kSmem, st, job,
                           d_order + w0, nwork, d_counters + cls);
            }
            ctx->launches++;
        }
        if ((rc = check_launch(ctx, "lz_match_kernel"))) return rc;
        ctx->launches--; // check_launch counted one more
        if (format == ZWZ_FORMAT_GZIP) { // the CRC-32 replaces the Adler-32 the match kernel left in job.adler
            {
                ProfSpan ps(ctx, ZWZ_PROF_ADLER, st);
                ZWZ_LAUNCH(zwz::crc32_kernel, (job.n + 7) / 8, 256, 0, st, d_raw, job.raw_off, job.raw_len, job.adler, job.n);
            }
            if ((rc = check_launch(ctx, "crc32_kernel"))) return rc;
        }
        uint32_t grid2 = std::min<uint32_t>((job.n + ZWZ_DE_WARPS - 1) / ZWZ_DE_WARPS, (uint32_t) ctx->sm_count * 8u);
        {
            ProfSpan ps(ctx, ZWZ_PROF_ENCODE, st);
            if (dict.idx) {
                auto *ke = zwz::deflate_encode_kernel<true>;
                ZWZ_LAUNCH(ke, grid2, ZWZ_DE_WARPS * 32, ZWZ_DE_SMEM, st, job, d_counters + 4);
            } else {
                ZWZ_LAUNCH(zwz::deflate_encode_kernel<false>, grid2, ZWZ_DE_WARPS * 32, ZWZ_DE_SMEM, st, job, d_counters + 4);
            }
        }
        if ((rc = check_launch(ctx, "deflate_encode_kernel"))) return rc;
    }
    tr.mark("kernels");
    // results come back behind the slot offsets in pin_keep, which then holds what zwz_pack_streams_device compares with
    uint8_t *h_res = (uint8_t *) ctx->pin_keep.p + keep_res_off(n);
    if (zwz_rt::memcpy_d2h(h_res, d_res, (size_t) n * 16, st) || zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "deflate kernels failed");
    tr.mark("download");
    host_copy(ctx, res, h_res, (size_t) n * 16, n);
    ctx->keep_n = n;
    tr.mark("copy-out");
    return ZWZ_OK;
}

static int md5_launch(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_data, const uint64_t *off, const uint64_t *len, const uint64_t *total_len,
                      uint32_t n, uint8_t *digest, int finalize, void *stream_v);
static int slot_finish(zwz_ctx *ctx, zwz::DigestSlot &sl);
static int slot_acquire(zwz_ctx *ctx, zwz::DigestSlot **out);
static int slot_queue_md5(zwz_ctx *ctx, zwz::DigestSlot &sl, const uint64_t *off, const uint64_t *len, uint32_t n, uint8_t *digest, uint64_t *ticket);

static int deflate_host_impl(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *out, uint64_t out_cap,
                             uint64_t *packed_off, zwz_deflate_result *res, int level, int format, const uint64_t *md5_off, const uint64_t *md5_len,
                             uint32_t md5_n, uint8_t *digest, uint64_t *ticket, const zwz_dicts *dicts = nullptr) {
    if (!ctx) return ZWZ_E_ARG;
    if (ticket) *ticket = 0;
    if (!packed_off) return fail(ctx, ZWZ_E_ARG, "null argument");
    packed_off[0] = 0;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !res || !out) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    // span of the host buffer the chunks touch
    uint64_t lo = ~0ull, hi = 0;
    for (uint32_t i = 0; i < n; ++i) {
        if (len[i] > ZWZ_CHUNK_SIZE) return fail(ctx, ZWZ_E_ARG, "chunk longer than 65535 bytes");
        lo = std::min(lo, off[i]);
        hi = std::max(hi, off[i] + len[i]);
    }
    if (hi < lo) lo = hi = 0;
    std::vector<uint64_t> roff(n), slot(n + 1);
    slot[0] = 0;
    for (uint32_t i = 0; i < n; ++i) {
        roff[i] = off[i] - lo;
        slot[i + 1] = slot[i] + zwz_deflate_bound(len[i]);
    }
    int rc;
    Trace tr(ctx, "compress");
    // the raw bytes live in a digest slot: their MD5 runs on the second stream and may outlive this call (ticket != NULL)
    zwz::DigestSlot *sl = nullptr;
    if ((rc = slot_acquire(ctx, &sl))) return rc;
    if ((rc = reserve(ctx, sl->data, (size_t) (hi - lo) + 64, false))) return rc;
    if ((rc = reserve(ctx, ctx->bulk_out, (size_t) slot[n] + 64, false))) return rc;
    tr.mark("reserve");
    if (zwz_rt::memcpy_h2d(sl->data.p, raw + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "raw upload failed");
    tr.mark("h2d");
    if (digest && md5_n) { // MD5 of the source files from the same resident copy (no second upload), beside the deflate kernels
        std::vector<uint64_t> mo(md5_n);
        for (uint32_t i = 0; i < md5_n; ++i) mo[i] = md5_off[i] - lo;
        if ((rc = slot_queue_md5(ctx, *sl, mo.data(), md5_len, md5_n, digest, ticket))) return rc;
    }
    struct Disarm { // an error below must not leave a pointer into the caller's memory behind in the slot
        zwz::DigestSlot *s;
        bool ok = false;
        ~Disarm() {
            if (!ok) s->digest_dst = nullptr;
        }
    } disarm{sl};
    zwz_dicts ddev;
    if ((rc = upload_dicts(ctx, dicts, &ddev))) return rc;
    if ((rc = zwz_deflate_batch_device_dict(ctx, (const uint8_t *) sl->data.p, roff.data(), len, n, (uint8_t *) ctx->bulk_out.p, slot.data(), res,
                                            level, format, dicts ? &ddev : nullptr, nullptr)))
        return rc;
    tr.mark("md5+deflate");
    for (uint32_t i = 0; i < n; ++i) packed_off[i + 1] = packed_off[i] + res[i].len0 + res[i].len1;
    if (packed_off[n] > out_cap) return fail(ctx, ZWZ_E_CAPACITY, "output buffer too small");
    // gather on the device so only the compressed bytes cross the bus
    const size_t pm = (size_t) (n + 1) * 8;
    if ((rc = reserve(ctx, ctx->packed, (size_t) packed_off[n] + align_up(pm, 256) + 256, false))) return rc;
    if ((rc = reserve(ctx, ctx->pin_meta, pm, true))) return rc;
    tr.mark("reserve2");
    memcpy(ctx->pin_meta.p, packed_off, pm);
    uint8_t *d_poff = (uint8_t *) ctx->packed.p;
    uint8_t *d_packed = d_poff + align_up(pm, 256);
    if (zwz_rt::memcpy_h2d(d_poff, ctx->pin_meta.p, pm, ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "offset upload failed");
    // slot offsets and results are still in ctx->keep from the call above
    const uint64_t *d_slot_off = (const uint64_t *) ctx->keep.p;
    const uint32_t *d_res = (const uint32_t *) ((const uint8_t *) ctx->keep.p + keep_res_off(n));
    {
        ProfSpan ps(ctx, ZWZ_PROF_PACK, ctx->stream);
        ZWZ_LAUNCH(zwz::pack_streams_kernel, (n + 7) / 8, 256, 0, ctx->stream, (const uint8_t *) ctx->bulk_out.p, d_slot_off, d_res, d_packed,
                   (const uint64_t *) d_poff, n);
    }
    if ((rc = check_launch(ctx, "pack_streams_kernel"))) return rc;
    tr.mark("pack");
    if (zwz_rt::memcpy_d2h(out, d_packed, (size_t) packed_off[n], ctx->stream) || zwz_rt::stream_sync(ctx->stream))
        return fail(ctx, ZWZ_E_CUDA, "compressed download failed");
    tr.mark("d2h");
    disarm.ok = true;
    if (!ticket) return slot_finish(ctx, *sl); // synchronous form: the digests are part of the result
    return ZWZ_OK;
}

int zwz_pack_streams_device(zwz_ctx *ctx, const uint8_t *d_slots, const uint64_t *slot_off, const zwz_deflate_result *res, uint32_t n,
                            uint8_t *d_packed, uint64_t *packed_off, void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (!packed_off) return fail(ctx, ZWZ_E_ARG, "null argument");
    packed_off[0] = 0;
    if (n == 0) return ZWZ_OK;
    if (!slot_off || !res || !d_slots || !d_packed) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    Trace tr(ctx, "pack_device", st);
    const size_t m_poff = (size_t) n * 8, m_res = m_poff + (size_t) (n + 1) * 8, meta_bytes = m_res + (size_t) n * 16;
    int rc;
    if ((rc = reserve(ctx, ctx->pin_meta, meta_bytes, true))) return rc;
    if ((rc = reserve(ctx, ctx->meta, meta_bytes + 256, false))) return rc;
    uint8_t *hp = (uint8_t *) ctx->pin_meta.p;
    uint64_t *h_poff = (uint64_t *) (hp + m_poff);
    // packed offsets: a blocked prefix sum. Beside it, the caller's slot offsets and results are compared with what the last
    // deflate call used and returned: where they are equal, its device copies in ctx->keep are used and not uploaded again
    const unsigned nb = host_blocks(ctx, n);
    const bool kept = ctx->keep_n == n;
    const uint8_t *hk = (const uint8_t *) ctx->pin_keep.p;
    std::vector<uint64_t> sum(nb);
    std::vector<char> same(nb, 0);
    host_for(ctx, nb, n, [&](unsigned k, size_t lo, size_t hi) {
        uint64_t a = 0;
        for (size_t i = lo; i < hi; ++i) a += (uint64_t) res[i].len0 + res[i].len1;
        sum[k] = a;
        same[k] = kept && !memcmp(hk + lo * 8, slot_off + lo, (hi - lo) * 8) && !memcmp(hk + keep_res_off(n) + lo * 16, res + lo, (hi - lo) * 16);
    });
    const bool reuse = kept && std::all_of(same.begin(), same.end(), [](char c) { return c != 0; });
    tr.mark("prefix+compare");
    h_poff[0] = 0;
    const Staging stg(nb);
    host_for(ctx, nb, n, [&](unsigned k, size_t lo, size_t hi) {
        uint64_t a = 0;
        for (unsigned j = 0; j < k; ++j) a += sum[j];
        for (size_t i = lo; i < hi; ++i) {
            a += (uint64_t) res[i].len0 + res[i].len1;
            packed_off[i + 1] = a;
            stg.put(h_poff + i + 1, a);
        }
        if (!reuse) {
            stg.copy(hp + lo * 8, slot_off + lo, (hi - lo) * 8);
            stg.copy(hp + m_res + lo * 16, res + lo, (hi - lo) * 16);
        }
        stg.done();
    });
    tr.mark("stage");
    uint8_t *dm = (uint8_t *) ctx->meta.p;
    const uint8_t *d_slot_off = reuse ? (const uint8_t *) ctx->keep.p : dm;
    const uint8_t *d_res = reuse ? (const uint8_t *) ctx->keep.p + keep_res_off(n) : dm + m_res;
    if (reuse ? zwz_rt::memcpy_h2d(dm + m_poff, h_poff, (size_t) (n + 1) * 8, st) : zwz_rt::memcpy_h2d(dm, hp, meta_bytes, st))
        return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    tr.mark("upload");
    {
        ProfSpan ps(ctx, ZWZ_PROF_PACK, st);
        ZWZ_LAUNCH(zwz::pack_streams_kernel, (n + 7) / 8, 256, 0, st, d_slots, (const uint64_t *) d_slot_off, (const uint32_t *) d_res, d_packed,
                   (const uint64_t *) (dm + m_poff), n);
    }
    if ((rc = check_launch(ctx, "pack_streams_kernel"))) return rc;
    if (zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "pack kernel failed");
    tr.mark("kernels");
    return ZWZ_OK;
}

int zwz_deflate_batch(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *out, uint64_t out_cap,
                      uint64_t *packed_off, zwz_deflate_result *res, int level) {
    return deflate_host_impl(ctx, raw, off, len, n, out, out_cap, packed_off, res, level, ZWZ_FORMAT_ZLIB, nullptr, nullptr, 0, nullptr, nullptr);
}

int zwz_deflate_batch_ex(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *out, uint64_t out_cap,
                         uint64_t *packed_off, zwz_deflate_result *res, int level, int format) {
    return deflate_host_impl(ctx, raw, off, len, n, out, out_cap, packed_off, res, level, format, nullptr, nullptr, 0, nullptr, nullptr);
}

int zwz_deflate_batch_dict(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *out, uint64_t out_cap,
                           uint64_t *packed_off, zwz_deflate_result *res, int level, int format, const zwz_dicts *dicts) {
    return deflate_host_impl(ctx, raw, off, len, n, out, out_cap, packed_off, res, level, format, nullptr, nullptr, 0, nullptr, nullptr, dicts);
}

uint64_t zwz_count_chunks(const uint64_t *file_off, uint32_t nf) {
    uint64_t c = 0;
    for (uint32_t i = 0; i < nf; ++i) c += (file_off[i + 1] - file_off[i]) / ZWZ_CHUNK_SIZE + 1;
    return c;
}

static int compress_files_impl(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                               uint64_t *packed_off, zwz_deflate_result *res, uint8_t *digest, uint64_t *ticket) {
    if (!ctx) return ZWZ_E_ARG;
    if (!file_off || !packed_off) return fail(ctx, ZWZ_E_ARG, "null argument");
    uint64_t nc = zwz_count_chunks(file_off, nf);
    if (nc > 0xffffffffull) return fail(ctx, ZWZ_E_ARG, "too many chunks in one batch");
    std::vector<uint64_t> coff((size_t) nc), flen(nf);
    std::vector<uint32_t> clen((size_t) nc);
    size_t k = 0;
    for (uint32_t i = 0; i < nf; ++i) { // compression.cpp:52-64
        uint64_t S = file_off[i + 1] - file_off[i];
        flen[i] = S;
        for (uint64_t o = 0;; o += ZWZ_CHUNK_SIZE) {
            uint64_t left = S - o;
            coff[k] = file_off[i] + o;
            clen[k] = (uint32_t) (left < ZWZ_CHUNK_SIZE ? left : ZWZ_CHUNK_SIZE);
            ++k;
            if (left < ZWZ_CHUNK_SIZE) break;
        }
    }
    return deflate_host_impl(ctx, data, coff.data(), clen.data(), (uint32_t) nc, out, out_cap, packed_off, res, level, ZWZ_FORMAT_ZLIB, file_off,
                             flen.data(), digest ? nf : 0, digest, ticket);
}

int zwz_compress_files(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                       uint64_t *packed_off, zwz_deflate_result *res, uint8_t *digest) {
    return compress_files_impl(ctx, data, file_off, nf, level, out, out_cap, packed_off, res, digest, nullptr);
}

int zwz_compress_files_async(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                             uint64_t *packed_off, zwz_deflate_result *res, uint8_t *digest, uint64_t *ticket) {
    if (!ticket) return ctx ? fail(ctx, ZWZ_E_ARG, "null ticket") : ZWZ_E_ARG;
    return compress_files_impl(ctx, data, file_off, nf, level, out, out_cap, packed_off, res, digest, ticket);
}

int zwz_wait(zwz_ctx *ctx, uint64_t ticket) {
    if (!ctx) return ZWZ_E_ARG;
    if (ticket == 0) return ZWZ_OK;
    zwz_rt::set_device(ctx->device);
    for (auto &sl : ctx->slot)
        if (sl.pending && sl.ticket == ticket) return slot_finish(ctx, sl);
    return ZWZ_OK; // already delivered (a later batch needed the slot)
}

// ======================================================================================================================
// inflate
// ======================================================================================================================
int zwz_inflate_batch_device(zwz_ctx *ctx, const uint8_t *d_comp, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_raw_out,
                             const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags, void *stream_v) {
    return zwz_inflate_batch_device_dict(ctx, d_comp, off, len, n, d_raw_out, raw_off, raw_len, status, flags, nullptr, stream_v);
}

int zwz_inflate_batch_device_dict(zwz_ctx *ctx, const uint8_t *d_comp, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_raw_out,
                                  const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags, const zwz_dicts *dicts,
                                  void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !raw_off || !raw_len || !status) return fail(ctx, ZWZ_E_ARG, "null argument");
    const uint32_t format = (flags >> 8) & 0xffu;
    if (format > ZWZ_FORMAT_RAW) return fail(ctx, ZWZ_E_ARG, "unknown stream format");
    if (format != ZWZ_FORMAT_ZLIB && ctx->inflate_mode == 2) return fail(ctx, ZWZ_E_ARG, "the one-lane-per-stream decoder reads zlib streams only");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    Trace tr(ctx, "inflate_device", st);
    zwz::DictTable dict{};
    int rc;
    if ((rc = stage_dicts(ctx, dicts, n, format == ZWZ_FORMAT_GZIP || ctx->inflate_mode == 2, st, &dict))) return rc;
    // Mapping: one warp per stream (inflate.cuh) is the product path. One lane per stream (inflate_lanes.cuh,
    // ZWZ_INFLATE_MODE=lanes) needs ~40x fewer warp-instructions per byte but only three warps fit an SM next to its
    // per-lane tables, and at that occupancy it runs latency-bound: 140 ms against 68 ms per C2 step on B200. It stays as a
    // tested alternative mapping. It keeps its Adler-32 sums unreduced and its bit counts in 32 bits, hence the size limits.
    bool lanes = ctx->inflate_mode == 2; // opt-in only: measured slower than the warp mapping on B200 (DESIGN.md, inflate)
    for (uint32_t i = 0; lanes && i < n; ++i)
        if (len[i] >= (1u << 28) || raw_off[i + 1] - raw_off[i] > (1ull << 24)) lanes = false;
    const size_t m_off = 0, m_roff = (size_t) n * 8, m_len = m_roff + (size_t) (n + 1) * 8, m_order = m_len + (size_t) n * 4,
                 meta_bytes = m_order + (lanes ? (size_t) n * 4 : 0);
    const size_t r_base = align_up(meta_bytes, 256);
    if ((rc = reserve(ctx, ctx->pin_meta, std::max(meta_bytes, (size_t) n * 8), true))) return rc;
    if ((rc = reserve(ctx, ctx->meta, r_base + (size_t) n * 8 + 512, false))) return rc;
    uint8_t *hp = (uint8_t *) ctx->pin_meta.p;
    const unsigned nb = host_blocks(ctx, n);
    const Staging stg(nb);
    host_for(ctx, nb, n, [&](unsigned, size_t lo, size_t hi) {
        stg.copy(hp + m_off + lo * 8, off + lo, (hi - lo) * 8);
        stg.copy(hp + m_roff + lo * 8, raw_off + lo, (hi - lo) * 8);
        stg.copy(hp + m_len + lo * 4, len + lo, (hi - lo) * 4);
        stg.done();
    });
    ((uint64_t *) (hp + m_roff))[n] = raw_off[n];
    if (lanes) {
        // streams by decreasing compressed size (counting sort on len / 32), so that the 32 lanes of a warp finish together
        // and the longest groups start first
        constexpr uint32_t NB = 4096;
        std::vector<uint32_t> head(NB + 1, 0u);
        auto bucket = [](uint32_t l) { return NB - 1u - std::min<uint32_t>(l >> 5, NB - 1u); };
        for (uint32_t i = 0; i < n; ++i) head[bucket(len[i]) + 1]++;
        for (uint32_t b = 0; b < NB; ++b) head[b + 1] += head[b];
        uint32_t *order = (uint32_t *) (hp + m_order);
        for (uint32_t i = 0; i < n; ++i) order[head[bucket(len[i])]++] = i;
    }
    tr.mark("stage");
    uint8_t *dm = (uint8_t *) ctx->meta.p;
    if (zwz_rt::memcpy_h2d(dm, hp, meta_bytes, st)) return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    tr.mark("upload");
    uint32_t *d_rlen = (uint32_t *) (dm + r_base);
    uint32_t *d_stat = d_rlen + n;
    uint32_t *d_counter = d_stat + n; // work queue head of the persistent warps
    if (zwz_rt::memset_device(d_counter, 0, 4, st)) return fail(ctx, ZWZ_E_CUDA, "memset failed");
    {
        ProfSpan ps(ctx, ZWZ_PROF_INFLATE, st);
        if (lanes) {
            uint32_t grid = std::min<uint32_t>((n + 31u) / 32u, (uint32_t) ctx->sm_count * 3u);
            ZWZ_LAUNCH(zwz::inflate_lanes_kernel, grid, 32, ZWZ_IL_SMEM, st, d_comp, (const uint64_t *) (dm + m_off),
                       (const uint32_t *) (dm + m_len), d_raw_out, (const uint64_t *) (dm + m_roff), d_rlen, d_stat,
                       (const uint32_t *) (dm + m_order), n, flags, d_counter);
        } else {
            uint32_t grid = std::min<uint32_t>((n + ZWZ_INF_WARPS - 1) / ZWZ_INF_WARPS, (uint32_t) (ctx->sm_count * ctx->inf_blocks_per_sm));
            if (ctx->inflate_mode == 3) flags |= ZWZ_INFLATE_CAREFUL;
            if (dict.idx) { // the DICT instantiation only when some stream of the call has a dictionary
                grid = std::min<uint32_t>((n + ZWZ_INF_WARPS - 1) / ZWZ_INF_WARPS, (uint32_t) (ctx->sm_count * ctx->inf_dict_blocks_per_sm));
                auto *ki = zwz::inflate_kernel<true>;
                ZWZ_LAUNCH(ki, grid, ZWZ_INF_WARPS * 32, ZWZ_INF_SMEM, st, d_comp, (const uint64_t *) (dm + m_off), (const uint32_t *) (dm + m_len),
                           d_raw_out, (const uint64_t *) (dm + m_roff), d_rlen, d_stat, n, flags, d_counter, dict);
            } else {
                ZWZ_LAUNCH(zwz::inflate_kernel<false>, grid, ZWZ_INF_WARPS * 32, ZWZ_INF_SMEM, st, d_comp, (const uint64_t *) (dm + m_off),
                           (const uint32_t *) (dm + m_len), d_raw_out, (const uint64_t *) (dm + m_roff), d_rlen, d_stat, n, flags, d_counter, dict);
            }
        }
    }
    if ((rc = check_launch(ctx, "inflate_kernel"))) return rc;
    tr.mark("kernels");
    if (zwz_rt::memcpy_d2h(hp, d_rlen, (size_t) n * 8, st) || zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "inflate kernel failed");
    tr.mark("download");
    host_for(ctx, nb, n, [&](unsigned, size_t lo, size_t hi) {
        memcpy(raw_len + lo, hp + lo * 4, (hi - lo) * 4);
        memcpy(status + lo, hp + (size_t) n * 4 + lo * 4, (hi - lo) * 4);
    });
    tr.mark("copy-out");
    return ZWZ_OK;
}

int zwz_inflate_batch(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *raw_out,
                      const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags) {
    return zwz_inflate_batch_dict(ctx, comp, off, len, n, raw_out, raw_off, raw_len, status, flags, nullptr);
}

int zwz_inflate_batch_dict(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *raw_out,
                           const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags, const zwz_dicts *dicts) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !raw_off || !raw_len || !status) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    uint64_t lo = ~0ull, hi = 0;
    for (uint32_t i = 0; i < n; ++i) {
        lo = std::min(lo, off[i]);
        hi = std::max(hi, off[i] + len[i]);
    }
    if (hi < lo) lo = hi = 0;
    std::vector<uint64_t> coff(n), roff(n + 1);
    for (uint32_t i = 0; i < n; ++i) coff[i] = off[i] - lo;
    for (uint32_t i = 0; i <= n; ++i) roff[i] = raw_off[i] - raw_off[0];
    int rc;
    if ((rc = reserve(ctx, ctx->bulk_in, (size_t) (hi - lo) + 64, false))) return rc;
    if ((rc = reserve(ctx, ctx->bulk_out, (size_t) roff[n] + 64, false))) return rc;
    if (zwz_rt::memcpy_h2d(ctx->bulk_in.p, comp + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "compressed upload failed");
    zwz_dicts ddev;
    if ((rc = upload_dicts(ctx, dicts, &ddev))) return rc;
    if ((rc = zwz_inflate_batch_device_dict(ctx, (const uint8_t *) ctx->bulk_in.p, coff.data(), len, n, (uint8_t *) ctx->bulk_out.p, roff.data(),
                                            raw_len, status, flags, dicts ? &ddev : nullptr, nullptr)))
        return rc;
    if (zwz_rt::memcpy_d2h(raw_out + raw_off[0], ctx->bulk_out.p, (size_t) roff[n], ctx->stream) || zwz_rt::stream_sync(ctx->stream))
        return fail(ctx, ZWZ_E_CUDA, "raw download failed");
    return ZWZ_OK;
}

static int gather_files(zwz_ctx *ctx, const uint64_t *slot, const uint64_t *dst, const uint32_t *len, uint32_t n, uint64_t acc, uint8_t *files_out,
                        uint32_t nf, const uint64_t *file_off_out, uint8_t *digest, uint64_t *ticket, Trace &tr);

static int decompress_records_impl(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, const uint32_t *rec_cap,
                                   const uint32_t *rec_file, uint32_t n, uint32_t nf, uint8_t *files_out, uint64_t out_cap, uint64_t *file_off_out,
                                   uint32_t *raw_len, uint32_t *status, uint8_t *digest, uint32_t flags, uint64_t *ticket) {
    if (!ctx) return ZWZ_E_ARG;
    if (ticket) *ticket = 0;
    if (!file_off_out) return fail(ctx, ZWZ_E_ARG, "null argument");
    if ((flags >> 8) & 0xffu) return fail(ctx, ZWZ_E_ARG, "records are zlib streams: no format may be given");
    for (uint32_t f = 0; f <= nf; ++f) file_off_out[f] = 0;
    if (n == 0) {
        if (digest && nf) { // every file is empty
            std::vector<uint64_t> z(nf, 0);
            int rc0 = reserve(ctx, ctx->bulk_in, 64, false);
            if (rc0) return rc0;
            return md5_launch(ctx, nullptr, (const uint8_t *) ctx->bulk_in.p, z.data(), z.data(), nullptr, nf, digest, 1, nullptr);
        }
        return ZWZ_OK;
    }
    if (!off || !len || !rec_cap || !rec_file || !raw_len || !status) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    uint64_t lo = ~0ull, hi = 0;
    for (uint32_t i = 0; i < n; ++i) {
        lo = std::min(lo, off[i]);
        hi = std::max(hi, off[i] + len[i]);
        if (rec_file[i] >= nf || (i && rec_file[i] < rec_file[i - 1])) return fail(ctx, ZWZ_E_ARG, "rec_file must be non-decreasing and < nf");
    }
    std::vector<uint64_t> coff(n), slot(n + 1);
    slot[0] = 0;
    for (uint32_t i = 0; i < n; ++i) {
        coff[i] = off[i] - lo;
        slot[i + 1] = slot[i] + (((uint64_t) rec_cap[i] + 15u) & ~15ull);
    }
    int rc;
    Trace tr(ctx, "decompress_records");
    if ((rc = reserve(ctx, ctx->bulk_in, (size_t) (hi - lo) + 64, false))) return rc;
    if ((rc = reserve(ctx, ctx->bulk_out, (size_t) slot[n] + 64, false))) return rc;
    tr.mark("reserve");
    if (zwz_rt::memcpy_h2d(ctx->bulk_in.p, comp + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "compressed upload failed");
    tr.mark("h2d");
    // per-record capacity is rec_cap, but slots are 16-byte aligned so the gather can use 128-bit copies
    std::vector<uint64_t> cap_off(n + 1);
    for (uint32_t i = 0; i <= n; ++i) cap_off[i] = slot[i];
    // inflate_kernel takes capacity = raw_off[i+1]-raw_off[i]; the up-to-15 padding bytes per slot are harmless extra room,
    // but OUTPUT_FULL must be judged against rec_cap — checked below.
    if ((rc = zwz_inflate_batch_device(ctx, (const uint8_t *) ctx->bulk_in.p, coff.data(), len, n, (uint8_t *) ctx->bulk_out.p, cap_off.data(),
                                       raw_len, status, flags, nullptr)))
        return rc;
    tr.mark("inflate");
    bool retry = false;
    for (uint32_t i = 0; i < n; ++i) {
        if (status[i] == ZWZ_STREAM_OUTPUT_FULL || raw_len[i] > rec_cap[i]) {
            if (raw_len[i] > rec_cap[i]) {
                status[i] = ZWZ_STREAM_OUTPUT_FULL;
                retry = true;
            }
        }
    }
    if (retry) return ZWZ_OK; // caller inspects status/raw_len and calls again with larger capacities
    // layout of the concatenated files
    std::vector<uint64_t> dst(n);
    uint64_t acc = 0;
    uint32_t f = 0;
    for (uint32_t i = 0; i < n; ++i) {
        while (f < rec_file[i]) file_off_out[++f] = acc;
        dst[i] = acc;
        acc += raw_len[i];
    }
    while (f < nf) file_off_out[++f] = acc;
    if (acc > out_cap) return fail(ctx, ZWZ_E_CAPACITY, "output buffer too small");
    return gather_files(ctx, slot.data(), dst.data(), raw_len, n, acc, files_out, nf, file_off_out, digest, ticket, tr);
}

// Concatenates the n inflated records in ctx->bulk_out (record i: len[i] bytes at slot[i], 16-byte aligned) into the output files
// (record i at dst[i]; acc bytes in all), downloads them into files_out and, when digest != NULL, queues the MD5 of the nf files
// (file_off_out) beside the download.
static int gather_files(zwz_ctx *ctx, const uint64_t *slot, const uint64_t *dst, const uint32_t *len, uint32_t n, uint64_t acc, uint8_t *files_out,
                        uint32_t nf, const uint64_t *file_off_out, uint8_t *digest, uint64_t *ticket, Trace &tr) {
    int rc;
    const size_t m_dst = (size_t) n * 8, m_len = 2 * (size_t) n * 8, meta_bytes = m_len + (size_t) n * 4;
    // the concatenated files live in a digest slot: their MD5 runs on the second stream and may outlive this call
    zwz::DigestSlot *sl = nullptr;
    if ((rc = slot_acquire(ctx, &sl))) return rc;
    if ((rc = reserve(ctx, sl->data, (size_t) acc + 256, false))) return rc;
    if ((rc = reserve(ctx, ctx->packed, align_up(meta_bytes, 256) + 256, false))) return rc;
    // NOT pin_meta: other calls refill pin_meta while this upload may still be in flight (page-locked memory is read by
    // the DMA engine after cudaMemcpyAsync returns) — a reuse race that corrupted gather descriptors once per ~10^5 records.
    if ((rc = reserve(ctx, ctx->pin_aux, meta_bytes, true))) return rc;
    tr.mark("reserve2");
    uint8_t *hp = (uint8_t *) ctx->pin_aux.p;
    memcpy(hp, slot, (size_t) n * 8);
    memcpy(hp + m_dst, dst, (size_t) n * 8);
    memcpy(hp + m_len, len, (size_t) n * 4);
    uint8_t *dmeta = (uint8_t *) ctx->packed.p;
    uint8_t *d_files = (uint8_t *) sl->data.p;
    if (zwz_rt::memcpy_h2d(dmeta, hp, meta_bytes, ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    {
        ProfSpan ps(ctx, ZWZ_PROF_PACK, ctx->stream);
        ZWZ_LAUNCH(zwz::gather_records_kernel, (n + 7) / 8, 256, 0, ctx->stream, (const uint8_t *) ctx->bulk_out.p, (const uint64_t *) dmeta,
                   (const uint64_t *) (dmeta + m_dst), (const uint32_t *) (dmeta + m_len), d_files, n);
    }
    if ((rc = check_launch(ctx, "gather_records_kernel"))) return rc;
    tr.mark("gather");
    if (digest && nf) { // beside the download of the files
        std::vector<uint64_t> fo(nf), fl(nf);
        for (uint32_t i = 0; i < nf; ++i) {
            fo[i] = file_off_out[i];
            fl[i] = file_off_out[i + 1] - file_off_out[i];
        }
        if ((rc = slot_queue_md5(ctx, *sl, fo.data(), fl.data(), nf, digest, ticket))) return rc;
    }
    tr.mark("md5 queued");
    if (zwz_rt::memcpy_d2h(files_out, d_files, (size_t) acc, ctx->stream) || zwz_rt::stream_sync(ctx->stream)) {
        sl->digest_dst = nullptr;
        return fail(ctx, ZWZ_E_CUDA, "raw download failed");
    }
    tr.mark("d2h");
    if (!ticket) return slot_finish(ctx, *sl);
    return ZWZ_OK;
}

int zwz_decompress_records(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, const uint32_t *rec_cap,
                           const uint32_t *rec_file, uint32_t n, uint32_t nf, uint8_t *files_out, uint64_t out_cap, uint64_t *file_off_out,
                           uint32_t *raw_len, uint32_t *status, uint8_t *digest, uint32_t flags) {
    return decompress_records_impl(ctx, comp, off, len, rec_cap, rec_file, n, nf, files_out, out_cap, file_off_out, raw_len, status, digest, flags,
                                   nullptr);
}

int zwz_decompress_records_async(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, const uint32_t *rec_cap,
                                 const uint32_t *rec_file, uint32_t n, uint32_t nf, uint8_t *files_out, uint64_t out_cap, uint64_t *file_off_out,
                                 uint32_t *raw_len, uint32_t *status, uint8_t *digest, uint32_t flags, uint64_t *ticket) {
    if (!ticket) return ctx ? fail(ctx, ZWZ_E_ARG, "null ticket") : ZWZ_E_ARG;
    return decompress_records_impl(ctx, comp, off, len, rec_cap, rec_file, n, nf, files_out, out_cap, file_off_out, raw_len, status, digest, flags,
                                   ticket);
}

// ======================================================================================================================
// whole files <-> BGZF .gz files
// ======================================================================================================================
uint64_t zwz_gzip_bound(const uint64_t *file_off, uint32_t nf) {
    uint64_t b = 0;
    for (uint32_t i = 0; file_off && i < nf; ++i) {
        const uint64_t S = file_off[i + 1] - file_off[i], r = S % ZWZ_BGZF_BLOCK;
        b += (S / ZWZ_BGZF_BLOCK) * zwz_deflate_bound(ZWZ_BGZF_BLOCK) + (r ? zwz_deflate_bound((uint32_t) r) : 0) + zwz_deflate_bound(0);
    }
    return b;
}

int zwz_gzip_files(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                   uint64_t *gz_off) {
    if (!ctx) return ZWZ_E_ARG;
    if (!file_off || !gz_off) return fail(ctx, ZWZ_E_ARG, "null argument");
    uint64_t nc = 0;
    for (uint32_t i = 0; i < nf; ++i) {
        if (file_off[i + 1] < file_off[i]) return fail(ctx, ZWZ_E_ARG, "file offsets must not decrease");
        nc += (file_off[i + 1] - file_off[i] + ZWZ_BGZF_BLOCK - 1) / ZWZ_BGZF_BLOCK + 1;
    }
    if (nc > 0xffffffffull) return fail(ctx, ZWZ_E_ARG, "too many chunks in one batch");
    // every file: full ZWZ_BGZF_BLOCK chunks, the remainder, then the empty chunk whose member is the BGZF end-of-file marker
    std::vector<uint64_t> coff((size_t) nc), poff((size_t) nc + 1), first(nf);
    std::vector<uint32_t> clen((size_t) nc);
    std::vector<zwz_deflate_result> res((size_t) nc);
    size_t k = 0;
    for (uint32_t i = 0; i < nf; ++i) {
        first[i] = k;
        const uint64_t S = file_off[i + 1] - file_off[i];
        for (uint64_t o = 0; o < S; o += ZWZ_BGZF_BLOCK, ++k) {
            coff[k] = file_off[i] + o;
            clen[k] = (uint32_t) std::min<uint64_t>(ZWZ_BGZF_BLOCK, S - o);
        }
        coff[k] = file_off[i + 1];
        clen[k++] = 0;
    }
    int rc = deflate_host_impl(ctx, data, coff.data(), clen.data(), (uint32_t) nc, out, out_cap, poff.data(), res.data(), level, ZWZ_FORMAT_GZIP,
                               nullptr, nullptr, 0, nullptr, nullptr);
    if (rc) return rc;
    for (uint32_t i = 0; i < nf; ++i) gz_off[i] = poff[first[i]];
    gz_off[nf] = poff[nc];
    return ZWZ_OK;
}

struct BgzfMember {
    uint64_t off;
    uint32_t len, cap;
};

// Appends the BGZF members of gz[p, end) to m, each found from the BSIZE of its BC subfield; its capacity is its ISIZE trailer.
// A member cut short by the end of the range (header included) is appended with what is there and 65 536 bytes of capacity: its
// inflate says how it ends. Returns ZWZ_STREAM_BAD in front of a member that is not BGZF (not gzip with a BC subfield, a BSIZE
// shorter than header + trailer, an ISIZE above the 64 KiB of a BGZF block), else ZWZ_STREAM_END.
static uint32_t bgzf_walk(const uint8_t *gz, uint64_t p, uint64_t end, std::vector<BgzfMember> &m) {
    while (p < end) {
        const uint8_t *h = gz + p;
        const uint64_t left = end - p;
        const uint32_t xlen = left >= 12 ? (uint32_t) h[10] | ((uint32_t) h[11] << 8) : 0u;
        if (left < 12 || left < 12u + xlen) {
            m.push_back({p, (uint32_t) left, 65536u});
            return ZWZ_STREAM_END;
        }
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 0x04)) return ZWZ_STREAM_BAD;
        uint32_t bsize = 0;
        bool found = false;
        for (uint32_t x = 0; x + 4 <= xlen;) {
            const uint8_t *f = h + 12 + x;
            const uint32_t slen = (uint32_t) f[2] | ((uint32_t) f[3] << 8);
            if (f[0] == 'B' && f[1] == 'C' && slen == 2 && x + 6 <= xlen) {
                bsize = (uint32_t) f[4] | ((uint32_t) f[5] << 8);
                found = true;
                break;
            }
            x += 4 + slen;
        }
        const uint64_t len = (uint64_t) bsize + 1;
        if (!found || len < 12u + xlen + 8u) return ZWZ_STREAM_BAD;
        if (len > left) {
            m.push_back({p, (uint32_t) left, 65536u});
            return ZWZ_STREAM_END;
        }
        const uint8_t *t = h + len - 4;
        const uint32_t isize = (uint32_t) t[0] | ((uint32_t) t[1] << 8) | ((uint32_t) t[2] << 16) | ((uint32_t) t[3] << 24);
        if (isize > 65536u) return ZWZ_STREAM_BAD;
        m.push_back({p, (uint32_t) len, isize});
        p += len;
    }
    return ZWZ_STREAM_END;
}

uint64_t zwz_gunzip_bound(const uint8_t *gz, const uint64_t *gz_off, uint32_t nf) {
    std::vector<BgzfMember> m;
    for (uint32_t i = 0; gz && gz_off && i < nf; ++i)
        if (gz_off[i + 1] > gz_off[i]) bgzf_walk(gz, gz_off[i], gz_off[i + 1], m);
    uint64_t b = 0;
    for (const BgzfMember &x : m) b += x.cap;
    return b;
}

int zwz_gunzip_files(zwz_ctx *ctx, const uint8_t *gz, const uint64_t *gz_off, uint32_t nf, uint8_t *out, uint64_t out_cap, uint64_t *out_off,
                     uint32_t *status) {
    if (!ctx) return ZWZ_E_ARG;
    if (!gz_off || !out_off || (nf && !status)) return fail(ctx, ZWZ_E_ARG, "null argument");
    for (uint32_t i = 0; i <= nf; ++i) out_off[i] = 0;
    std::vector<BgzfMember> m;
    std::vector<size_t> first(nf + 1);
    std::vector<uint32_t> walk(nf);
    uint64_t bound = 0;
    for (uint32_t i = 0; i < nf; ++i) {
        if (gz_off[i + 1] < gz_off[i]) return fail(ctx, ZWZ_E_ARG, "file offsets must not decrease");
        if (gz_off[i + 1] > gz_off[i] && !gz) return fail(ctx, ZWZ_E_ARG, "null argument");
        first[i] = m.size();
        walk[i] = bgzf_walk(gz, gz_off[i], gz_off[i + 1], m);
    }
    first[nf] = m.size();
    for (const BgzfMember &x : m) bound += x.cap;
    if (out_cap < bound) return fail(ctx, ZWZ_E_CAPACITY, "output buffer below zwz_gunzip_bound");
    if (m.size() > 0xffffffffull) return fail(ctx, ZWZ_E_ARG, "too many members in one batch");
    const uint32_t n = (uint32_t) m.size();
    if (n == 0) {
        for (uint32_t i = 0; i < nf; ++i) status[i] = walk[i];
        return ZWZ_OK;
    }
    if (!out) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    Trace tr(ctx, "gunzip_files");
    uint64_t lo = ~0ull, hi = 0;
    for (const BgzfMember &x : m) {
        lo = std::min(lo, x.off);
        hi = std::max(hi, x.off + x.len);
    }
    // every member inflates into a 16-byte aligned slot of its capacity (the gather then copies with 128-bit accesses)
    std::vector<uint64_t> coff(n), slot(n + 1), dst(n);
    std::vector<uint32_t> mlen(n), raw_len(n), st(n), take(n);
    slot[0] = 0;
    for (uint32_t j = 0; j < n; ++j) {
        coff[j] = m[j].off - lo;
        mlen[j] = m[j].len;
        slot[j + 1] = slot[j] + (((uint64_t) m[j].cap + 15u) & ~15ull);
    }
    int rc;
    if ((rc = reserve(ctx, ctx->bulk_in, (size_t) (hi - lo) + 64, false))) return rc;
    if ((rc = reserve(ctx, ctx->bulk_out, (size_t) slot[n] + 64, false))) return rc;
    tr.mark("reserve");
    if (zwz_rt::memcpy_h2d(ctx->bulk_in.p, gz + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "gz upload failed");
    tr.mark("h2d");
    if ((rc = zwz_inflate_batch_device(ctx, (const uint8_t *) ctx->bulk_in.p, coff.data(), mlen.data(), n, (uint8_t *) ctx->bulk_out.p, slot.data(),
                                       raw_len.data(), st.data(), ZWZ_INFLATE_FORMAT(ZWZ_FORMAT_GZIP), nullptr)))
        return rc;
    tr.mark("inflate");
    // per file: its members' bytes in order, up to and including the first member that does not end cleanly
    uint64_t acc = 0;
    for (uint32_t i = 0; i < nf; ++i) {
        out_off[i] = acc;
        status[i] = ZWZ_STREAM_END;
        for (size_t j = first[i]; j < first[i + 1]; ++j) {
            dst[j] = acc;
            take[j] = 0;
            if (status[i] != ZWZ_STREAM_END) continue;
            uint32_t s = st[j];
            if (s == ZWZ_STREAM_OUTPUT_FULL || raw_len[j] > m[j].cap) s = ZWZ_STREAM_BAD; // more than its ISIZE
            take[j] = std::min(raw_len[j], m[j].cap);
            acc += take[j];
            status[i] = s;
        }
        if (status[i] == ZWZ_STREAM_END) status[i] = walk[i];
    }
    out_off[nf] = acc;
    return gather_files(ctx, slot.data(), dst.data(), take.data(), n, acc, out, nf, out_off, nullptr, nullptr, tr);
}

// ======================================================================================================================
// MD5 / Adler-32 / CRC-32
// ======================================================================================================================
// Queues the MD5 kernel over n files on `st`: descriptors go up from `pin`, digests (and chained states) come back into `pin`
// at *digest_off (resp. m_state). Nothing is waited for.
static int md5_enqueue(zwz_ctx *ctx, zwz_stream_t st, Arena &dev_meta, Arena &pin, uint32_t *state, const uint8_t *d_data, const uint64_t *off,
                       const uint64_t *len, const uint64_t *total_len, uint32_t n, int finalize, size_t *digest_off, Trace *tr = nullptr) {
    const size_t m_len = (size_t) n * 8, m_tot = 2 * (size_t) n * 8, m_state = 3 * (size_t) n * 8, meta_bytes = m_state + (size_t) n * 16;
    const size_t r_base = align_up(meta_bytes, 256);
    int rc;
    if ((rc = reserve(ctx, pin, r_base + (size_t) n * 16, true))) return rc;
    if ((rc = reserve(ctx, dev_meta, r_base + (size_t) n * 16 + 256, false))) return rc;
    // the total length of the files picks the kernel below: summed while the descriptors are staged
    uint8_t *hp = (uint8_t *) pin.p;
    const unsigned nb = host_blocks(ctx, n);
    const Staging stg(nb);
    std::vector<uint64_t> sum(nb);
    host_for(ctx, nb, n, [&](unsigned k, size_t lo, size_t hi) {
        stg.copy(hp + lo * 8, off + lo, (hi - lo) * 8);
        stg.copy(hp + m_len + lo * 8, len + lo, (hi - lo) * 8);
        if (total_len) stg.copy(hp + m_tot + lo * 8, total_len + lo, (hi - lo) * 8);
        if (state) stg.copy(hp + m_state + lo * 16, state + lo * 4, (hi - lo) * 16);
        stg.done();
        uint64_t a = 0;
        for (size_t i = lo; i < hi; ++i) a += len[i];
        sum[k] = a;
    });
    if (tr) tr->mark("stage");
    // only what the kernel reads goes up: the chained states and total lengths only when there are some
    const size_t up_bytes = state ? meta_bytes : (total_len ? m_state : m_tot);
    uint8_t *dm = (uint8_t *) dev_meta.p;
    if (zwz_rt::memcpy_h2d(dm, hp, up_bytes, st)) return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    if (tr) tr->mark("upload");
    uint8_t *d_digest = dm + r_base;
    {
        // few long files: the staged kernel (coalesced cp.async into shared memory); many short ones: one lane streams its file
        uint64_t total = 0;
        for (uint64_t a : sum) total += a;
        const bool staged = total / n >= 65536u;
        ProfSpan ps(ctx, ZWZ_PROF_MD5, st);
        if (staged) {
            ZWZ_LAUNCH(zwz::md5_files_staged_kernel, (n + 31u) / 32u, ZWZ_MD5S_THREADS, ZWZ_MD5S_SMEM, st, d_data, (const uint64_t *) dm,
                       (const uint64_t *) (dm + m_len), total_len ? (const uint64_t *) (dm + m_tot) : (const uint64_t *) nullptr,
                       state ? (uint32_t *) (dm + m_state) : (uint32_t *) nullptr, d_digest, n, finalize);
        } else {
            ZWZ_LAUNCH(zwz::md5_files_kernel, (n + 127) / 128, 128, 0, st, d_data, (const uint64_t *) dm, (const uint64_t *) (dm + m_len),
                       total_len ? (const uint64_t *) (dm + m_tot) : (const uint64_t *) nullptr,
                       state ? (uint32_t *) (dm + m_state) : (uint32_t *) nullptr, d_digest, n, finalize);
        }
    }
    if ((rc = check_launch(ctx, "md5_files_kernel"))) return rc;
    if (finalize && zwz_rt::memcpy_d2h(hp + r_base, d_digest, (size_t) n * 16, st)) return fail(ctx, ZWZ_E_CUDA, "digest download failed");
    if (state && zwz_rt::memcpy_d2h(hp + m_state, dm + m_state, (size_t) n * 16, st)) return fail(ctx, ZWZ_E_CUDA, "state download failed");
    *digest_off = r_base;
    return ZWZ_OK;
}

static int md5_launch(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_data, const uint64_t *off, const uint64_t *len, const uint64_t *total_len,
                      uint32_t n, uint8_t *digest, int finalize, void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || (finalize && !digest)) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    Trace tr(ctx, "md5_device", st);
    size_t doff = 0;
    int rc = md5_enqueue(ctx, st, ctx->meta, ctx->pin_meta, state, d_data, off, len, total_len, n, finalize, &doff, &tr);
    if (rc) return rc;
    if (zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "md5 kernel failed");
    tr.mark("kernels+download");
    const uint8_t *hp = (const uint8_t *) ctx->pin_meta.p;
    if (finalize) host_copy(ctx, digest, hp + doff, (size_t) n * 16, n);
    if (state) memcpy(state, hp + 3 * (size_t) n * 8, (size_t) n * 16);
    tr.mark("copy-out");
    return ZWZ_OK;
}

// ---- deferred digests (DigestSlot) ---------------------------------------------------------------------------------
// the slot a new batch may use: its previous batch's digests are delivered first if nobody has waited for them yet
static int slot_finish(zwz_ctx *ctx, zwz::DigestSlot &sl) {
    if (!sl.pending) return ZWZ_OK;
    sl.pending = false;
    if (zwz_rt::sync_event_wait(sl.ev_done)) return fail(ctx, ZWZ_E_CUDA, "md5 kernel failed");
    if (sl.digest_dst && sl.n) memcpy(sl.digest_dst, (const uint8_t *) sl.pin.p + sl.digest_off, (size_t) sl.n * 16);
    return ZWZ_OK;
}
static int slot_acquire(zwz_ctx *ctx, zwz::DigestSlot **out) {
    zwz::DigestSlot &sl = ctx->slot[ctx->next_slot];
    ctx->next_slot ^= 1;
    int rc = slot_finish(ctx, sl);
    *out = &sl;
    return rc;
}
// MD5 of n files inside sl.data, queued on the second stream behind everything the main stream has queued so far
static int slot_queue_md5(zwz_ctx *ctx, zwz::DigestSlot &sl, const uint64_t *off, const uint64_t *len, uint32_t n, uint8_t *digest, uint64_t *ticket) {
    if (zwz_rt::sync_event_record(sl.ev_in, ctx->stream) || zwz_rt::stream_wait_event(ctx->md5_stream, sl.ev_in))
        return fail(ctx, ZWZ_E_CUDA, "stream dependency failed");
    int rc = md5_enqueue(ctx, ctx->md5_stream, sl.meta, sl.pin, nullptr, (const uint8_t *) sl.data.p, off, len, nullptr, n, 1, &sl.digest_off);
    if (rc) return rc;
    if (zwz_rt::sync_event_record(sl.ev_done, ctx->md5_stream)) return fail(ctx, ZWZ_E_CUDA, "event record failed");
    sl.pending = true;
    sl.n = n;
    sl.digest_dst = digest;
    sl.ticket = ++ctx->ticket_seq;
    if (ticket) *ticket = sl.ticket;
    return ZWZ_OK;
}

int zwz_md5_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint64_t *len, uint32_t n, uint8_t *digest, void *stream) {
    return md5_launch(ctx, nullptr, d_data, off, len, nullptr, n, digest, 1, stream);
}

int zwz_md5_batch(zwz_ctx *ctx, const uint8_t *data, const uint64_t *off, const uint64_t *len, uint32_t n, uint8_t *digest) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !digest) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    uint64_t lo = ~0ull, hi = 0;
    for (uint32_t i = 0; i < n; ++i) {
        lo = std::min(lo, off[i]);
        hi = std::max(hi, off[i] + len[i]);
    }
    if (hi < lo) lo = hi = 0;
    std::vector<uint64_t> o(n);
    for (uint32_t i = 0; i < n; ++i) o[i] = off[i] - lo;
    int rc;
    if ((rc = reserve(ctx, ctx->bulk_in, (size_t) (hi - lo) + 64, false))) return rc;
    if (zwz_rt::memcpy_h2d(ctx->bulk_in.p, data + lo, (size_t) (hi - lo), ctx->stream)) return fail(ctx, ZWZ_E_CUDA, "data upload failed");
    return md5_launch(ctx, nullptr, (const uint8_t *) ctx->bulk_in.p, o.data(), len, nullptr, n, digest, 1, nullptr);
}

void zwz_md5_state_init(uint32_t *state, uint32_t n) {
    for (uint32_t i = 0; i < n; ++i) {
        state[4 * i + 0] = 0x67452301u;
        state[4 * i + 1] = 0xefcdab89u;
        state[4 * i + 2] = 0x98badcfeu;
        state[4 * i + 3] = 0x10325476u;
    }
}

int zwz_md5_update_device(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_data, const uint64_t *off, const uint64_t *len, uint32_t n, void *stream) {
    if (!ctx) return ZWZ_E_ARG;
    if (!state) return fail(ctx, ZWZ_E_ARG, "null state");
    for (uint32_t i = 0; i < n; ++i)
        if (len[i] & 63u) return fail(ctx, ZWZ_E_ARG, "md5 update length must be a multiple of 64");
    return md5_launch(ctx, state, d_data, off, len, nullptr, n, nullptr, 0, stream);
}

int zwz_md5_final_device(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_tail, const uint64_t *off, const uint64_t *len, const uint64_t *total_len,
                         uint32_t n, uint8_t *digest, void *stream) {
    if (!ctx) return ZWZ_E_ARG;
    if (!state || !total_len) return fail(ctx, ZWZ_E_ARG, "null argument");
    return md5_launch(ctx, state, d_tail, off, len, total_len, n, digest, 1, stream);
}

void zwz_md5_hex(const uint8_t digest[16], char hex[32]) {
    static const char d[] = "0123456789abcdef";
    for (int i = 0; i < 16; ++i) {
        hex[2 * i] = d[digest[i] >> 4];
        hex[2 * i + 1] = d[digest[i] & 15];
    }
}

int zwz_adler32_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint32_t *len, uint32_t n, uint32_t *adler, void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !adler) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    const size_t m_len = (size_t) n * 8, meta_bytes = m_len + (size_t) n * 4, r_base = align_up(meta_bytes, 256);
    int rc;
    if ((rc = reserve(ctx, ctx->pin_meta, meta_bytes, true))) return rc;
    if ((rc = reserve(ctx, ctx->meta, r_base + (size_t) n * 4 + 256, false))) return rc;
    uint8_t *hp = (uint8_t *) ctx->pin_meta.p;
    memcpy(hp, off, (size_t) n * 8);
    memcpy(hp + m_len, len, (size_t) n * 4);
    uint8_t *dm = (uint8_t *) ctx->meta.p;
    if (zwz_rt::memcpy_h2d(dm, hp, meta_bytes, st)) return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    {
        ProfSpan ps(ctx, ZWZ_PROF_ADLER, st);
        ZWZ_LAUNCH(zwz::adler32_kernel, (n + 7) / 8, 256, 0, st, d_data, (const uint64_t *) dm, (const uint32_t *) (dm + m_len),
                   (uint32_t *) (dm + r_base), n);
    }
    if ((rc = check_launch(ctx, "adler32_kernel"))) return rc;
    if (zwz_rt::memcpy_d2h(hp, dm + r_base, (size_t) n * 4, st) || zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "adler kernel failed");
    memcpy(adler, hp, (size_t) n * 4);
    return ZWZ_OK;
}

int zwz_crc32_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint32_t *len, uint32_t n, uint32_t *crc, void *stream_v) {
    if (!ctx) return ZWZ_E_ARG;
    if (n == 0) return ZWZ_OK;
    if (!off || !len || !crc) return fail(ctx, ZWZ_E_ARG, "null argument");
    zwz_rt::set_device(ctx->device);
    zwz_stream_t st = stream_v ? (zwz_stream_t) stream_v : ctx->stream;
    const size_t m_len = (size_t) n * 8, meta_bytes = m_len + (size_t) n * 4, r_base = align_up(meta_bytes, 256);
    int rc;
    if ((rc = reserve(ctx, ctx->pin_meta, meta_bytes, true))) return rc;
    if ((rc = reserve(ctx, ctx->meta, r_base + (size_t) n * 4 + 256, false))) return rc;
    uint8_t *hp = (uint8_t *) ctx->pin_meta.p;
    memcpy(hp, off, (size_t) n * 8);
    memcpy(hp + m_len, len, (size_t) n * 4);
    uint8_t *dm = (uint8_t *) ctx->meta.p;
    if (zwz_rt::memcpy_h2d(dm, hp, meta_bytes, st)) return fail(ctx, ZWZ_E_CUDA, "descriptor upload failed");
    {
        ProfSpan ps(ctx, ZWZ_PROF_ADLER, st);
        ZWZ_LAUNCH(zwz::crc32_kernel, (n + 7) / 8, 256, 0, st, d_data, (const uint64_t *) dm, (const uint32_t *) (dm + m_len),
                   (uint32_t *) (dm + r_base), n);
    }
    if ((rc = check_launch(ctx, "crc32_kernel"))) return rc;
    if (zwz_rt::memcpy_d2h(hp, dm + r_base, (size_t) n * 4, st) || zwz_rt::stream_sync(st)) return fail(ctx, ZWZ_E_CUDA, "crc32 kernel failed");
    memcpy(crc, hp, (size_t) n * 4);
    return ZWZ_OK;
}

} // extern "C"
