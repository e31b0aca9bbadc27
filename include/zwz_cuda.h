/* zwz_cuda.h — C ABI of the B200 (sm_100a) hot path of the shard-based DEFLATE pipeline.
 *
 * This is the drop-in boundary (SURVEY.md §8(b)). The reference has no plugin/FFI interface; the narrowest seams it
 * offers are three call sites of shape "bytes in a caller-owned buffer -> bytes in a caller-owned buffer, no state":
 *
 *   zwz_deflate_batch*   replaces  compression.cpp:119-134   deflateInit / deflate(Z_FINISH) / deflateEnd per 65 535-B chunk
 *   zwz_inflate_batch*   replaces  decompression.cpp:11-37   inflateInit / inflate loop / inflateEnd per record
 *   zwz_md5_batch*       replaces  verification.cpp:13-27    MD5_Init / MD5_Update* / MD5_Final per file (+ hex at :24-27)
 *
 * Every entry point is plain C: POD arguments, caller owns every buffer it passes, the library owns its device arenas,
 * return value 0 = ok / negative = ZWZ_E_*; nothing throws across the boundary. A zwz_ctx is one stream plus its device
 * and page-locked arenas on one GPU; a ctx may be driven by one host thread at a time, different ctxs — on the same GPU
 * or not — concurrently (the host keeps one per worker). There is NO CPU fallback: zwz_init fails when no CUDA device
 * is usable.
 *
 * Two flavours of each batch call:
 *   *_device : bulk buffers are DEVICE pointers (inputs already resident in HBM); chunk descriptors (offset/length
 *              arrays) and per-chunk results are small HOST arrays. `stream` is a cudaStream_t passed as void*
 *              (NULL = the ctx's own stream). The call returns after the results are back on the host.
 *   (plain)  : bulk buffers are HOST pointers; the library stages them through pinned memory, runs the same kernels
 *              and brings the packed result back — the end-to-end call the C++ host (`main compress|decompress`) makes.
 */
#ifndef ZWZ_CUDA_H
#define ZWZ_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZWZ_ABI_VERSION 1
#define ZWZ_CHUNK_SIZE 65535u        /* process.hpp:12 CHUNK_SIZE: the largest raw chunk AND the largest payload the reader accepts */
#define ZWZ_MD5_HEX_SIZE 32u         /* process.hpp:14 MD5_DATA_SIZE */
#define ZWZ_DEFLATE_MARGIN 48u       /* zwz_deflate_bound(len) = len + margin, rounded up to 16 */

/* Stream formats: the wrapper around the DEFLATE body. The body is the same in all three for the same chunk and level. */
#define ZWZ_FORMAT_ZLIB 0       /* RFC 1950 (78 9C ... Adler-32): the .zwz record format, the default everywhere        */
#define ZWZ_FORMAT_GZIP 1       /* RFC 1952, one BGZF member per chunk (SAM/BAM spec 4.1: BC extra subfield = BSIZE)   */
#define ZWZ_FORMAT_RAW 2        /* RFC 1951, no wrapper, no check value                                                 */
#define ZWZ_BGZF_BLOCK 65280u   /* largest chunk accepted in GZIP format (bgzip's 0xff00): a stored member stays <= 64 KiB */

/* error codes */
#define ZWZ_OK 0
#define ZWZ_E_NODEVICE (-1)  /* no usable CUDA device / CUDA runtime error at init: there is no CPU path */
#define ZWZ_E_CUDA (-2)      /* a CUDA call or kernel failed; zwz_last_error() has the text */
#define ZWZ_E_ARG (-3)       /* bad argument (NULL, len > 65535, unaligned output offset, ...) */
#define ZWZ_E_NOMEM (-4)     /* device or pinned allocation failed */
#define ZWZ_E_CAPACITY (-5)  /* caller's output buffer too small */

/* per-stream inflate status (same numbering as oracle/zwz_oracle.c) */
#define ZWZ_STREAM_END 0         /* end of stream reached, Adler-32 matched                       (zlib: Z_STREAM_END)  */
#define ZWZ_STREAM_TRUNCATED 1   /* input ran out first; everything decodable was produced        (zlib: Z_OK/Z_BUF_ERROR) */
#define ZWZ_STREAM_BAD 2         /* invalid stream / check value mismatch; output up to the error (zlib: Z_DATA_ERROR)  */
#define ZWZ_STREAM_OUTPUT_FULL 3 /* would produce more than the capacity given; raw_len = size needed */
#define ZWZ_STREAM_MORE 4        /* zwz_inflater: not ended; feed more input, or call again to drain queued output   (zlib: Z_OK) */

/* per-chunk deflate result */
typedef struct zwz_deflate_result {
    uint32_t len0;  /* bytes of the first (usually only) zlib stream, at out + out_off[i]                              */
    uint32_t len1;  /* 0, or bytes of a second zlib stream right behind the first (split rule, see below)             */
    uint32_t raw0;  /* raw bytes covered by the first stream (== len[i] when len1 == 0)                                */
    uint32_t btype; /* DEFLATE block type chosen for stream 0: 0 stored, 1 fixed, 2 dynamic                            */
} zwz_deflate_result;
/* Split rule: the reference's reader copies a payload into a 65 535-byte array (decompression.cpp:116), and its writer
 * silently truncates streams longer than that (compression.cpp:127-132, SURVEY.md §5.1). When a chunk's best encoding
 * would exceed 65 535 bytes (only possible for an incompressible chunk of > 65 524 bytes) it is emitted as TWO complete
 * zlib streams over the two halves; the host writes them as two consecutive records. */

typedef struct zwz_ctx zwz_ctx;

/* ---- lifecycle --------------------------------------------------------------------------------------------------- */
int zwz_abi_version(void);
int zwz_device_count(void);                         /* 0 when there is no usable GPU */
int zwz_init(int device, zwz_ctx **out);            /* ZWZ_E_NODEVICE if `device` cannot run sm_100a code */
void zwz_destroy(zwz_ctx *ctx);
const char *zwz_last_error(const zwz_ctx *ctx);     /* text of the last failure on this ctx ("" if none) */
int zwz_device_props(const zwz_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);

/* plain-C callers need no CUDA headers: */
int zwz_malloc_device(zwz_ctx *ctx, size_t bytes, void **ptr);
int zwz_free_device(zwz_ctx *ctx, void *ptr);
int zwz_malloc_pinned(zwz_ctx *ctx, size_t bytes, void **ptr);
int zwz_free_pinned(zwz_ctx *ctx, void *ptr);
int zwz_memcpy_h2d(zwz_ctx *ctx, void *dst_device, const void *src_host, size_t bytes);
int zwz_memcpy_d2h(zwz_ctx *ctx, void *dst_host, const void *src_device, size_t bytes);
int zwz_sync(zwz_ctx *ctx);

/* number of kernel launches this ctx has issued so far (bench.py's gpu_launches) */
uint64_t zwz_launch_count(const zwz_ctx *ctx);

/* Per-kernel device timing (CUDA events recorded on the launching stream around every kernel of this ctx). Used by
 * bench.py for the roofline line; off by default. zwz_profile_read syncs, then returns the accumulated milliseconds and
 * launch counts per kernel kind since the last reset. */
#define ZWZ_PROF_MATCH 0   /* lz_match_kernel        */
#define ZWZ_PROF_ENCODE 1  /* deflate_encode_kernel  */
#define ZWZ_PROF_INFLATE 2 /* inflate_kernel; block_find_kernel, inflate_span_kernel */
#define ZWZ_PROF_MD5 3     /* md5_files_kernel       */
#define ZWZ_PROF_PACK 4    /* pack_streams_kernel; win_map_kernel, win_scan_kernel, stream_gather_kernel */
#define ZWZ_PROF_ADLER 5   /* checksum kernels: adler32_kernel, crc32_kernel; dict_chain_kernel */
#define ZWZ_PROF_N 6
int zwz_profile_enable(zwz_ctx *ctx, int on);
int zwz_profile_read(zwz_ctx *ctx, double *ms /* [ZWZ_PROF_N] */, uint64_t *launches /* [ZWZ_PROF_N] */, int reset);

/* ---- deflate: compression.cpp:119-134 ---------------------------------------------------------------------------- */
static inline uint64_t zwz_deflate_bound(uint32_t raw_len) { return (((uint64_t) raw_len + ZWZ_DEFLATE_MARGIN) + 15u) & ~(uint64_t) 15u; }

/* Chunk i is raw[off[i] .. off[i]+len[i]) with len[i] <= 65535 (0 allowed: the reference emits an 8-byte stream for the
 * empty tail chunk, compression.cpp:52-64). Its stream(s) are written at out + out_off[i]; out_off[i] must be a multiple
 * of 4 and leave zwz_deflate_bound(len[i]) bytes. level: 0 = library default; 1..9 trade search depth for speed. */
int zwz_deflate_batch_device(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n,
                             uint8_t *d_out, const uint64_t *out_off, zwz_deflate_result *res, int level, void *stream);

/* Host buffers in, PACKED host buffer out: chunk i's stream(s) are at out + packed_off[i] .. packed_off[i+1]
 * (packed_off has n+1 entries and is filled by the call). out_cap >= sum(zwz_deflate_bound(len[i])) always suffices. */
int zwz_deflate_batch(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n,
                      uint8_t *out, uint64_t out_cap, uint64_t *packed_off, zwz_deflate_result *res, int level);

/* The same two calls with a stream format (the plain forms are ZWZ_FORMAT_ZLIB). GZIP: every chunk becomes one BGZF member,
 * len[i] <= ZWZ_BGZF_BLOCK (else ZWZ_E_ARG); an empty chunk gives the 28-byte BGZF end-of-file marker. GZIP and RAW never
 * split: len1 == 0. A CRC-32 kernel runs over the chunks between the match and encode kernels. */
int zwz_deflate_batch_device_ex(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n,
                                uint8_t *d_out, const uint64_t *out_off, zwz_deflate_result *res, int level, int format, void *stream);
int zwz_deflate_batch_ex(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n,
                         uint8_t *out, uint64_t out_cap, uint64_t *packed_off, zwz_deflate_result *res, int level, int format);

/* Gather the variable-length streams of a finished zwz_deflate_batch_device out of their slots into one packed device
 * buffer (what the host then writes as record payloads, compression.cpp:93): chunk i's stream(s) land at
 * d_packed + packed_off[i] .. packed_off[i+1]; packed_off (host, n+1 entries) is filled by the call. */
int zwz_pack_streams_device(zwz_ctx *ctx, const uint8_t *d_slots, const uint64_t *slot_off, const zwz_deflate_result *res, uint32_t n,
                            uint8_t *d_packed, uint64_t *packed_off, void *stream);

/* ---- inflate: decompression.cpp:11-37 ---------------------------------------------------------------------------- */
/* Stream i is comp[off[i] .. off[i]+len[i]) (a complete RFC 1950 stream, or a truncated one). Output goes to
 * raw_out + raw_off[i] with capacity raw_off[i+1] - raw_off[i] (raw_off has n+1 entries). raw_len[i] = bytes produced —
 * exactly what zlib's inflate would have written for the same input (errors ignored as in decompression.cpp:31), or the
 * size needed when status[i] == ZWZ_STREAM_OUTPUT_FULL. flags: bit 0 = skip Adler-32 verification; bit 1 = decode with the
 * careful (warp-redundant) decoder only, without the lane-parallel block decoder (same results; for A/B timing and tests). */
#define ZWZ_INFLATE_NO_ADLER 1u
#define ZWZ_INFLATE_CAREFUL 2u
/* Bits 8..15 of flags: the stream format (default ZLIB). Each format inflates exactly as zlib 1.3 does with windowBits 15
 * (ZLIB), 31 (GZIP: one member, any header fields — FEXTRA, FNAME, FCOMMENT, FHCRC with the header CRC checked; bytes behind
 * the member's trailer are ignored) and -15 (RAW: no trailer). NO_ADLER skips the gzip CRC-32 as it skips Adler-32; ISIZE is
 * always checked. Any single-member .gz file (gzip, zlib.compress(wbits=31), ...) can be read this way; whole BGZF files go
 * through zwz_gunzip_files. The one-lane-per-stream decoder (ZWZ_INFLATE_MODE=lanes) reads zlib only: ZWZ_E_ARG otherwise. */
#define ZWZ_INFLATE_FORMAT(f) ((uint32_t) (f) << 8)
int zwz_inflate_batch_device(zwz_ctx *ctx, const uint8_t *d_comp, const uint64_t *off, const uint32_t *len, uint32_t n,
                             uint8_t *d_raw_out, const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status,
                             uint32_t flags, void *stream);
int zwz_inflate_batch(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, uint32_t n,
                      uint8_t *raw_out, const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags);

/* ---- one long stream on the whole GPU ----------------------------------------------------------------------------------
 * The batch calls give every stream one warp. A .gz file written by gzip, pigz, zlib or tar is one long stream (or a few
 * concatenated members), so these calls cut it into spans of compressed bytes instead: the spans start at block headers found by
 * searching (dynamic and stored blocks; a stream made of fixed blocks only decodes as one span), are decoded in parallel with
 * their 32 KiB window still unknown, confirmed against each other (a false start is decoded again), and the windows are then
 * resolved by a log-depth scan (DESIGN.md §4.8).
 *   comp[0 .. comp_len) is ONE stream, comp_len < 4 GiB; the output may be larger than 4 GiB. A stream of 4 GiB or more, one that
 *   arrives in pieces (a pipe, a socket) or one whose output does not fit in memory at once goes through zwz_inflater (below). flags are the inflate flags with
 *   the format in bits 8..15, whatever ZWZ_INFLATE_MODE says:
 *     GZIP : every member, as gzip -d: a member follows where the previous trailer ends when the next two bytes are 1f 8b; any
 *            other bytes behind a trailer are ignored. The result is that of zlib 1.3 (windowBits 31) decoding the members one
 *            after another and stopping at the first that does not end cleanly; a CRC-32 or ISIZE mismatch is ZWZ_STREAM_BAD
 *            behind all of that member's bytes. A BGZF file is one case of this.
 *     ZLIB : one stream (windowBits 15). FDICT is ZWZ_STREAM_BAD with 0 bytes: this call takes no dictionary.
 *     RAW  : one stream (windowBits -15).
 *   Bytes and status are zlib's otherwise (ZWZ_STREAM_END / TRUNCATED / BAD, bytes before an error included); NO_ADLER skips
 *   CRC-32 / Adler-32 (ISIZE is still checked). Bytes of out past *raw_len may have been written.
 *   ZWZ_STREAM_OUTPUT_FULL: out_cap is smaller than what the stream decodes to (up to its end or first decoding error, check
 *   values and "too far back" aside); *raw_len is that size. It takes precedence over a check value or "too far back" error,
 *   whatever the scratch waves (below), so the result does not depend on ZWZ_TUNE_STREAM_SCRATCH_BYTES. Nothing is written when the stream fits one scratch wave (below); otherwise the waves
 *   before the one that would pass out_cap have been written. (The batch calls instead fill up to the capacity.)
 *   NULL pointers and an unknown format are ZWZ_E_ARG.
 * Device scratch: u16 span slots (2 bytes per output byte) and 128 KiB of window maps for each span whose outgoing window a later
 * span reads, of one wave at a time, about ZWZ_TUNE_STREAM_SCRATCH_BYTES; allocated for the call and freed after it.
 * Adversarial input with a false block start in every span costs one confirmation round per span; it still decodes exactly. */
int zwz_inflate_stream_device(zwz_ctx *ctx, const uint8_t *d_comp, uint64_t comp_len, uint8_t *d_out, uint64_t out_cap,
                              uint64_t *raw_len, uint32_t *status, uint32_t flags, void *stream);
int zwz_inflate_stream(zwz_ctx *ctx, const uint8_t *comp, uint64_t comp_len, uint8_t *out, uint64_t out_cap,
                       uint64_t *raw_len, uint32_t *status, uint32_t flags);

/* zwz_inflate_stream_batch[_device]: many such streams (a set of .gz files, say) in one call, their spans sharing the GPU and
 * their confirmation rounds sharing launches (DESIGN.md §4.10).
 *   Stream i is comp[off[i] .. off[i] + len[i]) (ranges may overlap or repeat; they are only read) and decodes into
 *   out[out_off[i] .. out_off[i + 1]). raw_len[i] and status[i] are exactly what zwz_inflate_stream returns for that stream alone
 *   with out_cap = out_off[i + 1] - out_off[i] and the same flags, and so are the bytes up to raw_len[i]. One format per call, in
 *   bits 8..15 of flags.
 *   Nothing outside a stream's own region is written, whatever its status; an OUTPUT_FULL region's contents are unspecified. No
 *   stream's result depends on the others: a bad stream leaves its neighbours alone, and no window reaches from one into the next.
 *   ZWZ_E_ARG: NULL pointers with n > 0, an unknown format, len[i] > 0xffffff00, off[i] + len[i] past 2^64, a decreasing
 *   out_off. n == 0 does nothing.
 *   The host form uploads the extent [min off, max off + len) once and downloads every wave's output.
 * Device scratch: that of zwz_inflate_stream for one wave of spans, which may hold spans of many streams; ZWZ_TUNE_STREAM_SCRATCH_BYTES
 * counts slots and window maps. */
int zwz_inflate_stream_batch_device(zwz_ctx *ctx, const uint8_t *d_comp, const uint64_t *off, const uint64_t *len, uint32_t n,
                                    uint8_t *d_out, const uint64_t *out_off, uint64_t *raw_len, uint32_t *status,
                                    uint32_t flags, void *stream);
int zwz_inflate_stream_batch(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint64_t *len, uint32_t n,
                             uint8_t *out, const uint64_t *out_off, uint64_t *raw_len, uint32_t *status, uint32_t flags);

/* ---- one stream fed piece by piece: the streaming inflater (zlib's inflate() on successive buffers, Python's decompressobj) ----
 * zwz_inflater_new: an inflater for one stream; flags are those of zwz_inflate_stream (the format in bits 8..15, NO_ADLER; other
 *   bits are ignored). An unknown format or a NULL out is ZWZ_E_ARG.
 * zwz_inflater_feed[_device](f, in, in_len, final, out, out_cap, &produced, &status): appends in[0 .. in_len) to the pending input.
 *   When no decoded output is queued, it decodes everything the pending input allows (on the whole GPU, as zwz_inflate_stream does)
 *   into the inflater's output queue. Then it hands out min(queued, out_cap) bytes to out and sets *produced to that count.
 *   final != 0 says no input follows (it may come with the last bytes or in an empty call).
 *   Equivalence: the bytes produced over all calls, concatenated, and the terminal status equal zwz_inflate_stream on the
 *   concatenated input with the same flags (END, TRUNCATED or BAD, bytes before an error included), for every way of cutting the
 *   input into calls, every out_cap and any number of empty calls. OUTPUT_FULL does not occur, and there is no limit on the
 *   stream's total length, compressed or decoded.
 *   *status: ZWZ_STREAM_MORE until the stream has ended and its queue is drained, then the terminal status, which stays.
 *   TRUNCATED needs final. A zlib or raw stream ends with its last block (and trailer); a gzip stream ends when two bytes other
 *   than 1f 8b follow a trailer, or at final. Once the stream has ended, further input is ignored, as zwz_inflate_stream ignores
 *   bytes behind the end.
 *   ZWZ_E_ARG, with the inflater unchanged: NULL f, produced or status; NULL in with in_len > 0 or NULL out with out_cap > 0; input
 *   after final; pending input that would reach 0xffffff00 bytes. Pending input is what the decoder could not use yet: the bytes
 *   from the last complete block (or member header) on. A caller that keeps feeding without ever draining the queue stops the
 *   decoding, so its pending input grows until this refusal.
 *   The _device form takes device pointers and a cudaStream_t as void* (NULL = the context's stream); both forms return after the
 *   bytes are in out. After a ZWZ_E_CUDA or ZWZ_E_NOMEM the inflater only takes zwz_inflater_free.
 * Memory, on the context's device: the pending input, a 64 KiB window and the output queue, which holds the output of one decode:
 *   what the input of one call (plus the pending bytes) decodes to. Decoding has the fixed cost of a zwz_inflate_stream call (a few
 *   launches and synchronisations): feeds of hundreds of MiB approach its rate, 64 MiB feeds reach about half of it and feeds of
 *   1 MiB a few percent (DESIGN.md §4.11).
 * zwz_inflater_info: bytes given (total_in), bytes handed out (total_out), pending input and queued output; NULL fields are skipped.
 * An inflater belongs to its context; free it with zwz_inflater_free before the context is destroyed. */
typedef struct zwz_inflater zwz_inflater;
int zwz_inflater_new(zwz_ctx *ctx, uint32_t flags, zwz_inflater **out);
void zwz_inflater_free(zwz_inflater *f);
int zwz_inflater_feed_device(zwz_inflater *f, const uint8_t *d_in, uint64_t in_len, int final, uint8_t *d_out, uint64_t out_cap,
                             uint64_t *produced, uint32_t *status, void *stream);
int zwz_inflater_feed(zwz_inflater *f, const uint8_t *in, uint64_t in_len, int final, uint8_t *out, uint64_t out_cap,
                      uint64_t *produced, uint32_t *status);
int zwz_inflater_info(const zwz_inflater *f, uint64_t *total_in, uint64_t *total_out, uint64_t *pending_in, uint64_t *queued_out);

/* ---- one long input into one gzip, zlib or raw DEFLATE stream on the whole GPU (what gzip, zlib.compress and compressobj write) ----
 * The batch calls write one complete stream per chunk of at most 64 KiB. These calls write ONE stream of any length: the input is cut
 * into chunks of C bytes (ZWZ_TUNE_DEFLATE_STREAM_CHUNK_BYTES, default 65 535), counted from the stream start or the last flush point,
 * and every chunk is compressed by the batch kernels as a piece of the stream, its window being the <= 32 KiB of input in front of it
 * (back to the stream start or the last full flush). A piece that is not the last has no header or trailer, BFINAL 0 on all its blocks,
 * and ends on a byte boundary with an empty stored block (00 00 ff ff after three zero bits, as zlib's Z_SYNC_FLUSH), so the pieces
 * are joined byte for byte; the last piece ends the stream (DESIGN.md §4.12). Limits of the window search: a match that starts in the
 * window ends at the window's end, noise stretches are not searched against the window, and its last two positions are not chained.
 *   Wrappers: gzip = one member, header 1f 8b 08 00, MTIME 0, XFL 0, OS ff, trailer CRC-32 and ISIZE (length mod 2^32) little-endian;
 *   zlib = 78 9c, trailer Adler-32 big-endian; raw = the bare blocks. An empty input gives zlib's bytes: 03 00 in raw, 78 9c 03 00 00 00
 *   00 01 in zlib, a 20-byte member in gzip.
 * zwz_deflate_stream[_device]: d_raw[0 .. raw_len) (any length; passes of ZWZ_TUNE_DEFLATE_SUBBATCH_BYTES bound the device memory) into
 *   out[0 .. *comp_len). level as in zwz_deflate_batch. ZWZ_E_CAPACITY: out_cap is smaller than the stream, *comp_len is the size needed
 *   (bytes up to out_cap may have been written). ZWZ_E_ARG: NULL comp_len, NULL raw with raw_len > 0, NULL out with out_cap > 0, an
 *   unknown format. The host form feeds a zwz_deflater in passes of up to 1 GiB; its bytes are those of the device form.
 * zwz_deflate_stream_bound(raw_len): out_cap >= this always suffices for one call, whatever the format, level and chunk size. */
uint64_t zwz_deflate_stream_bound(uint64_t raw_len);
int zwz_deflate_stream_device(zwz_ctx *ctx, const uint8_t *d_raw, uint64_t raw_len, uint8_t *d_out, uint64_t out_cap, uint64_t *comp_len,
                              int level, int format, void *stream);
int zwz_deflate_stream(zwz_ctx *ctx, const uint8_t *raw, uint64_t raw_len, uint8_t *out, uint64_t out_cap, uint64_t *comp_len, int level,
                       int format);

/* ---- one stream written piece by piece: the streaming deflater (zlib's deflate() on successive buffers, Python's compressobj) ----
 * zwz_deflater_new: a deflater for one stream in `format` at `level` (as zwz_deflate_stream); it keeps the chunk size C the context
 *   has when it is made. An unknown format or a NULL out is ZWZ_E_ARG.
 * zwz_deflater_feed[_device](f, in, in_len, flush, out, out_cap, &produced): appends in[0 .. in_len) to the pending input. When no
 *   compressed output is queued, it compresses as `flush` says (numbered as zlib's, so Python may pass zlib.Z_*):
 *     ZWZ_NO_FLUSH   every whole chunk behind which at least one more pending byte follows; at most C bytes stay pending (the stream's
 *                    last chunk must stay pending to become its final piece). The last <= 32 KiB compressed is kept as the next window.
 *     ZWZ_SYNC_FLUSH everything pending: the output so far ends with the empty stored block (written also when nothing is pending).
 *     ZWZ_FULL_FLUSH the same, and the window is dropped: the next chunk refers to nothing before it, so a decoder can start there.
 *     ZWZ_FINISH     everything pending, the final piece and the trailer. Later input is ZWZ_E_ARG; later calls only drain the queue.
 *   Then it hands out min(queued, out_cap) bytes to out and sets *produced to that count. A flush asked for while output is queued is
 *   done once the queue is empty: a call that empties the queue compresses again, so a call that returns with nothing queued has done
 *   every flush asked for. Until then call again, as with zlib, without input: input given then is ZWZ_E_ARG.
 *   Equivalence: chunk cuts are counted from the last flush point, so the output depends only on the input bytes and on where and which
 *   flushes were asked for. NO_FLUSH feeds and one FINISH give, concatenated, exactly the bytes of zwz_deflate_stream on the concatenated
 *   input, for every way of cutting it and every out_cap.
 *   ZWZ_E_ARG: NULL f or produced; NULL in with in_len > 0 or NULL out with out_cap > 0; an unknown flush; pending input that would reach
 *   0xffffff00 bytes. The _device form takes device pointers and a cudaStream_t as void* (NULL = the context's stream); both forms return
 *   after the bytes are in out. After a ZWZ_E_CUDA or ZWZ_E_NOMEM the deflater only takes zwz_deflater_free.
 * Memory, on the context's device: the pending input with its 32 KiB window in front, and the output queue, which holds what one
 *   compression wrote (at most zwz_deflate_stream_bound of the pending input). The running check value and length stay on the host.
 *   Each compression has the fixed cost of a zwz_deflate_stream call; feeds of tens of MiB or more amortise it (DESIGN.md §4.12).
 * zwz_deflater_info: bytes given (total_in), bytes handed out (total_out), pending input and queued output; NULL fields are skipped.
 * A deflater belongs to its context; free it with zwz_deflater_free before the context is destroyed. */
#define ZWZ_NO_FLUSH 0
#define ZWZ_SYNC_FLUSH 2
#define ZWZ_FULL_FLUSH 3
#define ZWZ_FINISH 4
typedef struct zwz_deflater zwz_deflater;
int zwz_deflater_new(zwz_ctx *ctx, int level, int format, zwz_deflater **out);
void zwz_deflater_free(zwz_deflater *f);
int zwz_deflater_feed_device(zwz_deflater *f, const uint8_t *d_in, uint64_t in_len, int flush, uint8_t *d_out, uint64_t out_cap,
                             uint64_t *produced, void *stream);
int zwz_deflater_feed(zwz_deflater *f, const uint8_t *in, uint64_t in_len, int flush, uint8_t *out, uint64_t out_cap, uint64_t *produced);
int zwz_deflater_info(const zwz_deflater *f, uint64_t *total_in, uint64_t *total_out, uint64_t *pending_in, uint64_t *queued_out);

/* ---- random access into one long stream: a seek index (zlib's zran.c idea) -------------------------------------------------
 * zwz_inflate_stream_index[_device] inflate exactly as zwz_inflate_stream[_device] (same output, *raw_len and *status for the same
 * input, flags, tuning and out_cap) and keep what the span decoding already found: access points, each a confirmed span start
 * with its resolved 32 KiB window (DESIGN.md §4.9).
 *   out == NULL: index only; the library decodes into its own memory and writes nothing to the caller.
 *   *index is set only with ZWZ_STREAM_END, else it is NULL (OUTPUT_FULL, truncated or bad streams, "too far back").
 *   Access points: the stream start (point 0, empty window), then greedily the first confirmed span start whose output offset is
 *   at least the previous point's + max(spacing, 1); spacing 0 = every confirmed span start that adds output. A point records its
 *   output offset, the bit where decoding starts (a block header, a stored block's key = the bit 3 in front of its LEN field, or a
 *   gzip member header's first bit), its mode (ZWZ_INDEX_MODE_*), BFINAL, and its window: the last wlen <= 32 768 output bytes
 *   before it that lie inside the same gzip member (0 at the stream start and at member headers).
 * A zwz_index belongs to the context that created or loaded it; free it with zwz_index_free before that context is destroyed.
 * Its point table is host memory, its windows one device allocation. */
typedef struct zwz_index zwz_index;
#define ZWZ_INDEX_MODE_BLOCK 0   /* a block header                                                           */
#define ZWZ_INDEX_MODE_START 1   /* the stream's first bit (zlib / gzip header, or the first raw block)      */
#define ZWZ_INDEX_MODE_MEMBER 2  /* a following gzip member's header                                          */
#define ZWZ_INDEX_MODE_STORED 3  /* a stored block's key: the block type is not read from the bits there      */
int zwz_inflate_stream_index_device(zwz_ctx *ctx, const uint8_t *d_comp, uint64_t comp_len, uint8_t *d_out, uint64_t out_cap,
                                    uint64_t *raw_len, uint32_t *status, uint32_t flags, uint64_t spacing, zwz_index **index,
                                    void *stream);
int zwz_inflate_stream_index(zwz_ctx *ctx, const uint8_t *comp, uint64_t comp_len, uint8_t *out, uint64_t out_cap,
                             uint64_t *raw_len, uint32_t *status, uint32_t flags, uint64_t spacing, zwz_index **index);
void zwz_index_free(zwz_index *ix);
int zwz_index_info(const zwz_index *ix, uint64_t *comp_len, uint64_t *raw_len, uint32_t *format, uint64_t *npoints);
/* Saved form, little-endian:
 *    0  char[8]  "ZWZIDX\0\1"
 *    8  u32      version = 1
 *   12  u32      format (ZWZ_FORMAT_*)
 *   16  u64      comp_len
 *   24  u64      raw_len
 *   32  u64      npoints
 *   40  u64      spacing asked for
 *   48  u32      CRC-32 (as zlib.crc32) of the whole blob with these four bytes read as zero
 *   52  u32      0
 *   56  npoints x { u64 out_off; u64 bit; u16 mode; u8 bfinal; u8 0; u32 wlen }   (24 bytes each)
 *       then the windows of the points in point order, back to back (sum of wlen bytes)
 * zwz_index_save: *len = the blob's size; buf == NULL asks for the size only; cap < *len is ZWZ_E_CAPACITY.
 * zwz_index_load: the blob is outside input and is checked: magic, version, CRC; len == 56 + 24 npoints + sum(wlen); format <= RAW;
 *   comp_len <= 0xffffff00; point 0 = {0, 0, START, bfinal 0, wlen 0}; out_off strictly increasing and <= raw_len; bit strictly
 *   increasing and < 8 comp_len; mode in range (START at point 0 only, MEMBER in gzip only); header points byte-aligned and stored
 *   keys 3 bits before a byte boundary; bfinal <= 1, pad bytes 0; wlen <= min(32 768, out_off), and 0 at START and MEMBER points.
 *   Anything else is ZWZ_E_ARG. */
int zwz_index_save(const zwz_index *ix, uint8_t *buf, uint64_t cap, uint64_t *len);
int zwz_index_load(zwz_ctx *ctx, const uint8_t *buf, uint64_t len, zwz_index **out);
/* zwz_index_extract[_device]: range i is bytes [off[i], off[i] + len[i]) of what zwz_inflate_stream decodes the stream to; they go to
 * out + out_off[i]. On success status[i] = ZWZ_STREAM_END and got[i] = len[i]. Each range is cut at the access points inside it; a
 * piece is decoded by one warp from the last point at or before its start, with that point's window, up to the first block
 * boundary at or past its end (inflate_seek.cuh). Pieces that start at a point are decoded straight into the output; the others
 * into scratch, from which the kept bytes are copied.
 *   ZWZ_E_ARG: a range past raw_len, a comp_len other than the index's, an index of another context, NULL pointers, flags other
 *   than ZWZ_INFLATE_CAREFUL (the careful decoder only, for tests and A/B runs), and a piece that would decode 4 GiB or more from
 *   its point (the decoder's positions are 32-bit: two points more than 4 GiB of output apart, as in a stream of fixed blocks only).
 *   Check values are not verified (as in zran.c). A stream of the same length that is not the one indexed may give another status
 *   (got[i] = the bytes delivered before the piece that came up short) or wrong bytes; it never writes outside the ranges.
 *   Device scratch: skip + want bytes per piece that does not start at a point, in batches of about ZWZ_TUNE_STREAM_SCRATCH_BYTES.
 * The host form uploads comp on every call; random reads of a resident stream should use the device form. */
int zwz_index_extract_device(zwz_ctx *ctx, const zwz_index *ix, const uint8_t *d_comp, uint64_t comp_len, uint32_t n,
                             const uint64_t *off, const uint64_t *len, uint8_t *d_out, const uint64_t *out_off,
                             uint64_t *got, uint32_t *status, uint32_t flags, void *stream);
int zwz_index_extract(zwz_ctx *ctx, const zwz_index *ix, const uint8_t *comp, uint64_t comp_len, uint32_t n,
                      const uint64_t *off, const uint64_t *len, uint8_t *out, const uint64_t *out_off,
                      uint64_t *got, uint32_t *status, uint32_t flags);

/* ---- preset dictionaries (zlib's deflateSetDictionary / inflateSetDictionary, Python's zdict=) ----------------------------
 * A table of dictionaries, and for every chunk / stream the one it uses. Dictionary k is data[off[k] .. off[k+1]) (at most
 * 2^30 bytes); only its last min(len, 32 768) bytes are the window a stream may refer into, as if they came just before the
 * stream's first byte. An empty dictionary is no dictionary. `dicts == NULL` is exactly the call without _dict.
 *   deflate ZLIB : a chunk with a dictionary is written as 78 BB + DICTID (big-endian Adler-32 of the WHOLE dictionary, as
 *                  deflateSetDictionary), body, Adler-32 of the chunk; it never splits (len1 == 0).
 *   deflate RAW  : the body may refer into the dictionary; nothing in the stream names it.
 *   deflate GZIP : a dictionary on any chunk is ZWZ_E_ARG (zlib refuses gzip dictionaries too).
 *   inflate ZLIB : FDICT with a dictionary: the DICTID must be the dictionary's Adler-32 (also with ZWZ_INFLATE_NO_ADLER), else
 *                  ZWZ_STREAM_BAD with 0 bytes; FDICT without one: ZWZ_STREAM_BAD; no FDICT: the dictionary is ignored. A
 *                  stream that ends inside the DICTID is ZWZ_STREAM_TRUNCATED.
 *   inflate RAW  : the dictionary is the window before the first byte.
 *   inflate GZIP : a dictionary is ZWZ_E_ARG; so is any dictionary with ZWZ_INFLATE_MODE=lanes.
 * Chunks / streams marked ZWZ_NO_DICT in a call with dictionaries come out exactly as in the call without. An idx[i] that is
 * neither ZWZ_NO_DICT nor < ndict, or a NULL off, is ZWZ_E_ARG. Not available for .zwz records (zwz_compress_files,
 * zwz_decompress_records): the reference's reader inflates without a dictionary. */
#define ZWZ_NO_DICT 0xffffffffu
typedef struct zwz_dicts {
    const uint8_t *data;  /* dictionary k = data[off[k] .. off[k+1]); DEVICE pointer for *_device calls, host pointer otherwise */
    const uint64_t *off;  /* host, ndict + 1 entries                                                                        */
    uint32_t ndict;
    const uint32_t *idx;  /* host, n entries: the dictionary of chunk / stream i, or ZWZ_NO_DICT; NULL = dictionary 0 for all */
} zwz_dicts;
int zwz_deflate_batch_device_dict(zwz_ctx *ctx, const uint8_t *d_raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *d_out,
                                  const uint64_t *out_off, zwz_deflate_result *res, int level, int format, const zwz_dicts *dicts, void *stream);
int zwz_deflate_batch_dict(zwz_ctx *ctx, const uint8_t *raw, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *out,
                           uint64_t out_cap, uint64_t *packed_off, zwz_deflate_result *res, int level, int format, const zwz_dicts *dicts);
int zwz_inflate_batch_device_dict(zwz_ctx *ctx, const uint8_t *d_comp, const uint64_t *off, const uint32_t *len, uint32_t n,
                                  uint8_t *d_raw_out, const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags,
                                  const zwz_dicts *dicts, void *stream);
int zwz_inflate_batch_dict(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, uint32_t n, uint8_t *raw_out,
                           const uint64_t *raw_off, uint32_t *raw_len, uint32_t *status, uint32_t flags, const zwz_dicts *dicts);

/* ---- MD5: verification.cpp:13-27 --------------------------------------------------------------------------------- */
/* File i is data[off[i] .. off[i]+len[i]) (any length, 0 included). digest = 16 raw bytes per file. */
int zwz_md5_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint64_t *len, uint32_t n,
                         uint8_t *digest /* host, n*16 */, void *stream);
int zwz_md5_batch(zwz_ctx *ctx, const uint8_t *data, const uint64_t *off, const uint64_t *len, uint32_t n,
                  uint8_t *digest /* host, n*16 */);
/* Streaming form for files larger than one staging buffer (the MD5_Update loop of verification.cpp:16-19):
 * state = 4 x uint32 per file, host memory, initialised by zwz_md5_state_init; every update but the last must be a
 * multiple of 64 bytes; the final call pads with the file's total length and writes the digest. */
void zwz_md5_state_init(uint32_t *state, uint32_t n);
int zwz_md5_update_device(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_data, const uint64_t *off, const uint64_t *len,
                          uint32_t n, void *stream);
int zwz_md5_final_device(zwz_ctx *ctx, uint32_t *state, const uint8_t *d_tail, const uint64_t *off, const uint64_t *len,
                         const uint64_t *total_len, uint32_t n, uint8_t *digest, void *stream);
/* verification.cpp:24-27: 16 digest bytes -> 32 lowercase hex characters (no terminator). */
void zwz_md5_hex(const uint8_t digest[16], char hex[32]);

/* ---- whole-batch passes used by the C++ host (one upload, one download per batch) -------------------------------------- */
/* Chunks a batch of whole files exactly like the reference's producer (compression.cpp:52-64: floor(S/65535)+1 chunks per
 * file, the last one S mod 65535 bytes, possibly empty). */
uint64_t zwz_count_chunks(const uint64_t *file_off /* nf+1 */, uint32_t nf);
/* Compress side of one batch: file i is data[file_off[i] .. file_off[i+1]). Uploads the span once, deflates every chunk,
 * MD5s every file (md5_of_file(src), compression.cpp:95-103; pass digest = NULL to skip), packs and downloads the streams.
 * Chunks come out in file order then sequence order; packed_off has zwz_count_chunks()+1 entries, res one per chunk. */
int zwz_compress_files(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                       uint64_t *packed_off, zwz_deflate_result *res, uint8_t *digest /* nf*16 or NULL */);
/* Decompress side of one batch: record i is comp[off[i] .. off[i]+len[i]); records are given in OUTPUT order (all records
 * of file 0 in sequence order, then file 1, ...), rec_file[i] = file index (non-decreasing), rec_cap[i] = capacity to give
 * record i (65 535 is enough for every record the reference or this library writes; a record that needs more comes back with
 * status ZWZ_STREAM_OUTPUT_FULL and raw_len = the size needed, and NOTHING is written to files_out — retry with larger caps).
 * On success the records' bytes are concatenated per file into files_out (file_off_out[nf+1] filled by the call) and digest
 * receives the MD5 of every file (md5_of_file(output), decompression.cpp:136; NULL to skip). Records are zlib streams: a
 * format other than ZLIB in flags (and so in the _async form) gives ZWZ_E_ARG. */
int zwz_decompress_records(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, const uint32_t *rec_cap,
                           const uint32_t *rec_file, uint32_t n, uint32_t nf, uint8_t *files_out, uint64_t out_cap, uint64_t *file_off_out,
                           uint32_t *raw_len, uint32_t *status, uint8_t *digest /* nf*16 or NULL */, uint32_t flags);

/* Tuning knobs of a context. ZWZ_TUNE_DEFLATE_SUBBATCH_BYTES: raw bytes deflated per internal pass (default 4 GiB; the
 * match/token scratch is 6 bytes per raw byte of ONE pass, so a host worker that feeds 128 MB batches asks for 32 MiB passes
 * and its context allocates 0.2 GB of scratch instead of 0.8 GB — device allocation is the larger part of a short job's
 * start-up). */
#define ZWZ_TUNE_DEFLATE_SUBBATCH_BYTES 1
/* ZWZ_TUNE_HOST_THREADS: host threads (the calling one included) that stage the descriptors of one call — copies into and out of
 * page-locked memory, validation, offset sums; the device waits for this work, since every call ends in a synchronise. 0 =
 * min(8, cores / 2) (default), 1 = the calling thread alone. The threads belong to the context and end in zwz_destroy.
 * ZWZ_TUNE_HOST_PARALLEL_MIN: calls with fewer chunks, streams or files than this (default 32 768) run on the calling thread
 * alone, so that many contexts fed by threads of their own with small batches do not oversubscribe the host. */
#define ZWZ_TUNE_HOST_THREADS 2
#define ZWZ_TUNE_HOST_PARALLEL_MIN 3
/* ZWZ_TUNE_STREAM_SPAN_BYTES: compressed bytes per span of zwz_inflate_stream* (>= 1024; 0 = default: max(64 KiB, enough for two
 * spans per resident decoder warp)). */
#define ZWZ_TUNE_STREAM_SPAN_BYTES 4
/* ZWZ_TUNE_STREAM_SCRATCH_BYTES: u16 span slots and window maps (128 KiB for each span whose outgoing window a later span reads) of
 * one wave of zwz_inflate_stream* (0 = default, 4 GiB). Larger streams are decoded
 * in waves of consecutive spans that hand on the resolved window and the running check value; a single span larger than the budget
 * still forms a wave of its own. */
#define ZWZ_TUNE_STREAM_SCRATCH_BYTES 5
/* ZWZ_TUNE_DEFLATE_STREAM_CHUNK_BYTES: the chunk size C of zwz_deflate_stream* and of the deflaters made afterwards (1 024 .. 65 535;
 * 0 = default, 65 535). Small values let tests cross many chunk boundaries, and windows that span several chunks, with small inputs. */
#define ZWZ_TUNE_DEFLATE_STREAM_CHUNK_BYTES 6
int zwz_ctx_tune(zwz_ctx *ctx, int what, uint64_t value);

/* ---- asynchronous forms: the digests are DEFERRED ----------------------------------------------------------------------
 * SURVEY.md §8(b): "asynchronous variants ... pair with a zwz_wait". A file's MD5 is one serial chain (~0.13 GB/s per file on
 * one lane), so a batch holding a 16 MiB file would wait ~130 ms for its digests while its deflate/inflate kernels take a
 * few milliseconds. The *_async calls return as soon as the BYTES are back in the caller's buffers (packed streams resp.
 * decompressed files); the MD5 kernel keeps running on the context's second stream over the batch's device-resident copy
 * and `digest` is filled in by zwz_wait(ticket). Two batches may be in flight per context; starting a third delivers the
 * oldest one's digests first (its `digest` pointer must therefore stay valid until zwz_wait or until two more *_async calls
 * on the context have returned). The host pipeline uses this to take MD5 off its batch critical path: records are
 * serialised and archive offsets handed out while the digests are still being computed (compression.cpp:95-103 appends
 * them behind the last record of a file; decompression.cpp:136-146 only needs them for the verdict line). */
int zwz_compress_files_async(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                             uint64_t *packed_off, zwz_deflate_result *res, uint8_t *digest /* nf*16 or NULL */, uint64_t *ticket);
int zwz_decompress_records_async(zwz_ctx *ctx, const uint8_t *comp, const uint64_t *off, const uint32_t *len, const uint32_t *rec_cap,
                                 const uint32_t *rec_file, uint32_t n, uint32_t nf, uint8_t *files_out, uint64_t out_cap,
                                 uint64_t *file_off_out, uint32_t *raw_len, uint32_t *status, uint8_t *digest /* nf*16 or NULL */,
                                 uint32_t flags, uint64_t *ticket);
/* Blocks until the digests of `ticket` are in the buffer given to the *_async call (ticket 0 or an already delivered
 * ticket: returns at once). */
int zwz_wait(zwz_ctx *ctx, uint64_t ticket);

/* ---- Adler-32 (the zlib trailer; exported for tests) ---------------------------------------------------------------- */
int zwz_adler32_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint32_t *len, uint32_t n,
                             uint32_t *adler /* host, n */, void *stream);
/* ---- CRC-32 (RFC 1952, the gzip trailer; one warp per range) ----------------------------------------------------------- */
int zwz_crc32_batch_device(zwz_ctx *ctx, const uint8_t *d_data, const uint64_t *off, const uint32_t *len, uint32_t n,
                           uint32_t *crc /* host, n */, void *stream);

/* ---- whole files <-> BGZF .gz files (host buffers: one upload, one download, like zwz_compress_files) --------------------
 * zwz_gzip_files: file i is data[file_off[i] .. file_off[i+1]); it is cut into ceil(S / ZWZ_BGZF_BLOCK) chunks plus one empty
 * chunk, each deflated into one BGZF member (the empty one is the EOF marker; an empty file is the marker alone). File i's .gz
 * is out[gz_off[i] .. gz_off[i+1]) (gz_off: nf+1 entries, filled). It is an ordinary multi-member gzip file: gzip -d, zcat,
 * Python's gzip and htslib read it. out_cap >= zwz_gzip_bound() always suffices. */
uint64_t zwz_gzip_bound(const uint64_t *file_off, uint32_t nf);
int zwz_gzip_files(zwz_ctx *ctx, const uint8_t *data, const uint64_t *file_off, uint32_t nf, int level, uint8_t *out, uint64_t out_cap,
                   uint64_t *gz_off);
/* zwz_gunzip_files: file i is gz[gz_off[i] .. gz_off[i+1]), a BGZF file. Its members are found on the host from their BSIZE
 * fields (a member is BSIZE+1 bytes; it must be gzip with a BC subfield and an ISIZE of at most 65 536), all members of all
 * files are inflated in one batch, and each file's output goes to out[out_off[i] .. out_off[i+1]) (out_off: nf+1 entries,
 * filled with the bytes actually produced). status[i] = ZWZ_STREAM_END when every member ended cleanly and the members tile
 * the file exactly; otherwise the status of the first failing member (a member producing more than its ISIZE counts as
 * ZWZ_STREAM_BAD; a file whose first member is not BGZF is ZWZ_STREAM_BAD with 0 bytes), and the output stops with what that
 * member produced. One bad file does not affect the others. out_cap < zwz_gunzip_bound() gives ZWZ_E_CAPACITY.
 * Plain (non-BGZF) .gz files of one member are read with zwz_inflate_batch and ZWZ_INFLATE_FORMAT(ZWZ_FORMAT_GZIP). */
uint64_t zwz_gunzip_bound(const uint8_t *gz, const uint64_t *gz_off, uint32_t nf);
int zwz_gunzip_files(zwz_ctx *ctx, const uint8_t *gz, const uint64_t *gz_off, uint32_t nf, uint8_t *out, uint64_t out_cap,
                     uint64_t *out_off, uint32_t *status);

#ifdef __cplusplus
}
#endif
#endif /* ZWZ_CUDA_H */
