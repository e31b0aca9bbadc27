// zwz_rt.h — the handful of CUDA runtime calls the C ABI needs, behind one seam.
//
// Product build (nvcc): thin inline wrappers over the CUDA runtime.
// Emulator build (-DZWZ_EMU, tests only): "device" memory is host memory and a launch runs the kernel body through
// tests/simt/simt_emu.h. The emulator library is never loaded by the product package.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <time.h>

#ifdef ZWZ_EMU
typedef void *zwz_stream_t;
namespace zwz_rt {
inline const char *backend() { return "simt-emulator"; }
inline int device_count() { return 1; }
inline int set_device(int) { return 0; }
inline int device_props(int, int *sms, int *maj, int *min, size_t *mem, size_t *smem_optin) {
    *sms = 4;
    *maj = 10;
    *min = 0;
    *mem = (size_t) 1 << 34;
    *smem_optin = 232448;
    return 0;
}
inline int malloc_device(void **p, size_t n) {
    *p = malloc(n ? n : 1);
    if (*p) memset(*p, 0xCD, n); // cudaMalloc memory is not zeroed either
    return *p ? 0 : 2;
}
inline int free_device(void *p) { free(p); return 0; }
inline int malloc_arena(void **p, size_t n, zwz_stream_t) { return malloc_device(p, n); }
inline int free_arena(void *p, zwz_stream_t) { return free_device(p); }
inline int keep_pool_memory(int) { return 0; }
inline int preload_kernel(const void *) { return 0; }
inline int malloc_pinned(void **p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : 2; }
inline int free_pinned(void *p) { free(p); return 0; }
inline int stream_create(zwz_stream_t *s) { *s = nullptr; return 0; }
inline int stream_destroy(zwz_stream_t) { return 0; }
inline int stream_sync(zwz_stream_t) { return 0; }
inline int memcpy_h2d(void *d, const void *s, size_t n, zwz_stream_t) { if (n) memcpy(d, s, n); return 0; }
inline int memcpy_d2h(void *d, const void *s, size_t n, zwz_stream_t) { if (n) memcpy(d, s, n); return 0; }
inline int memset_device(void *d, int v, size_t n, zwz_stream_t) { if (n) memset(d, v, n); return 0; }
inline int last_error(std::string &) { return 0; }
inline int set_max_dyn_smem(const void *, size_t) { return 0; }
// resident CTAs per SM: what shared memory alone would allow on a B200 (the emulator has no register file)
inline int max_blocks_per_sm(int *blocks, const void *, int, size_t smem) {
    *blocks = (int) std::min<size_t>(32u, std::max<size_t>(1u, (228u * 1024u) / (smem + 1024u)));
    return 0;
}
typedef int zwz_sync_event_t; // ordering-only events: the emulator runs everything in call order
inline int sync_event_create(zwz_sync_event_t *e) { *e = 0; return 0; }
inline int sync_event_destroy(zwz_sync_event_t) { return 0; }
inline int sync_event_record(zwz_sync_event_t, zwz_stream_t) { return 0; }
inline int sync_event_wait(zwz_sync_event_t) { return 0; }
inline int stream_wait_event(zwz_stream_t, zwz_sync_event_t) { return 0; }
typedef double zwz_event_t; // wall-clock stamp
inline int event_record(zwz_event_t *e, zwz_stream_t) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    *e = ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
    return 0;
}
inline double event_elapsed_and_free(zwz_event_t a, zwz_event_t b) { return b - a; }
} // namespace zwz_rt
#define ZWZ_LAUNCH(kern, grid, block, smem, stream, ...) simt::launch((unsigned) (grid), (unsigned) (block), (size_t) (smem), [&] { kern(__VA_ARGS__); })
#else
#include <cuda_runtime.h>
typedef cudaStream_t zwz_stream_t;
namespace zwz_rt {
inline const char *backend() { return "cuda"; }
inline int device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
inline int set_device(int d) { return cudaSetDevice(d) == cudaSuccess ? 0 : 1; }
inline int device_props(int d, int *sms, int *maj, int *min, size_t *mem, size_t *smem_optin) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, d) != cudaSuccess) return 1;
    *sms = p.multiProcessorCount;
    *maj = p.major;
    *min = p.minor;
    *mem = p.totalGlobalMem;
    *smem_optin = p.sharedMemPerBlockOptin;
    return 0;
}
inline int malloc_device(void **p, size_t n) { return cudaMalloc(p, n ? n : 1) == cudaSuccess ? 0 : 2; }
inline int free_device(void *p) { return cudaFree(p) == cudaSuccess ? 0 : 1; }
// Arenas come from the stream-ordered allocator: cudaMalloc/cudaFree synchronise the whole device, which stalls every other
// context of the process (the host's worker pool saw ~0.7 s stalls behind another worker's long MD5 kernel).
inline int malloc_arena(void **p, size_t n, zwz_stream_t st) {
    if (cudaMallocAsync(p, n ? n : 1, st) != cudaSuccess) return 2;
    return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 2; // usable from any stream afterwards
}
inline int free_arena(void *p, zwz_stream_t st) { return cudaFreeAsync(p, st) == cudaSuccess ? 0 : 1; }
inline int keep_pool_memory(int device) { // freed arena memory stays in the pool instead of going back to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) != cudaSuccess) return 1;
    unsigned long long keep = ~0ull;
    return cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep) == cudaSuccess ? 0 : 1;
}
// with lazy module loading (the CUDA 12 default) a kernel's code is loaded at its first launch, under a process-wide lock:
// loading at init moves that cost to where the host overlaps it with its own planning
inline int preload_kernel(const void *fn) {
    cudaFuncAttributes a;
    return cudaFuncGetAttributes(&a, fn) == cudaSuccess ? 0 : 1;
}
// resident CTAs per SM for a launch of `threads` threads and `smem` bytes of dynamic shared memory (registers, shared
// memory and the CTA limit all counted by the driver)
inline int max_blocks_per_sm(int *blocks, const void *fn, int threads, size_t smem) {
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks, fn, threads, smem) == cudaSuccess && *blocks > 0 ? 0 : 1;
}
inline int malloc_pinned(void **p, size_t n) { return cudaMallocHost(p, n ? n : 1) == cudaSuccess ? 0 : 2; }
inline int free_pinned(void *p) { return cudaFreeHost(p) == cudaSuccess ? 0 : 1; }
inline int stream_create(zwz_stream_t *s) { return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) == cudaSuccess ? 0 : 1; }
inline int stream_destroy(zwz_stream_t s) { return cudaStreamDestroy(s) == cudaSuccess ? 0 : 1; }
inline int stream_sync(zwz_stream_t s) { return cudaStreamSynchronize(s) == cudaSuccess ? 0 : 1; }
inline int memcpy_h2d(void *d, const void *s, size_t n, zwz_stream_t st) {
    return n == 0 || cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : 1;
}
inline int memcpy_d2h(void *d, const void *s, size_t n, zwz_stream_t st) {
    return n == 0 || cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st) == cudaSuccess ? 0 : 1;
}
inline int memset_device(void *d, int v, size_t n, zwz_stream_t st) { return n == 0 || cudaMemsetAsync(d, v, n, st) == cudaSuccess ? 0 : 1; }
inline int last_error(std::string &msg) {
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) return 0;
    msg = cudaGetErrorString(e);
    return 1;
}
inline int set_max_dyn_smem(const void *fn, size_t bytes) {
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes) == cudaSuccess ? 0 : 1;
}
// ordering-only events (no timing): cross-stream dependencies and the completion of deferred work (zwz_wait)
typedef cudaEvent_t zwz_sync_event_t;
inline int sync_event_create(zwz_sync_event_t *e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess ? 0 : 1; }
inline int sync_event_destroy(zwz_sync_event_t e) { return cudaEventDestroy(e) == cudaSuccess ? 0 : 1; }
inline int sync_event_record(zwz_sync_event_t e, zwz_stream_t st) { return cudaEventRecord(e, st) == cudaSuccess ? 0 : 1; }
inline int sync_event_wait(zwz_sync_event_t e) { return cudaEventSynchronize(e) == cudaSuccess ? 0 : 1; }
inline int stream_wait_event(zwz_stream_t st, zwz_sync_event_t e) { return cudaStreamWaitEvent(st, e, 0) == cudaSuccess ? 0 : 1; }
typedef cudaEvent_t zwz_event_t;
inline int event_record(zwz_event_t *e, zwz_stream_t st) {
    if (cudaEventCreate(e) != cudaSuccess) return 1;
    return cudaEventRecord(*e, st) == cudaSuccess ? 0 : 1;
}
inline double event_elapsed_and_free(zwz_event_t a, zwz_event_t b) { // caller has synchronised
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return ms;
}
} // namespace zwz_rt
#define ZWZ_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif
