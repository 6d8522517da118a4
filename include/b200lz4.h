/*
 * b200lz4.h -- C ABI of libb200lz4.so: a B200-native (sm_100a) LZ4 block codec
 * that is a drop-in for the codec path of composewell/streamly-lz4.
 *
 * The reference crosses into C through 7 `foreign import ccall` + 1 `capi value`
 * (src/Streamly/Internal/LZ4.hs:105-147, declarations cbits/lz4.h:170,182,
 * 273-274,336,358-359,409).  This header offers
 *   (1) a BATCHED interface -- the throughput path the patched Haskell shim binds
 *       (`foreign import ccall safe`, see INTEGRATION.md), and
 *   (2) LEGACY aliases of the 7 original symbols with the original signatures, so
 *       an unmodified Streamly.Internal.LZ4 links and behaves identically (one
 *       block per call; every call still runs on the GPU -- there is no CPU codec
 *       in this library).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ or torch types cross this boundary;
 *   - all functions return B200LZ4_OK (0) or a negative B200LZ4_E_* code unless
 *     stated otherwise; b200lz4_last_error() gives the text of the last failure
 *     on the calling thread;
 *   - a failing BLOCK never aborts a batch: per-block results are reported in
 *     out_len[] (compress: 0 = failed, as LZ4_compress_fast_continue
 *     cbits/lz4.c:1026,1120,1216; decompress: < 0 = failed, as
 *     LZ4_decompress_safe_continue cbits/lz4.c:2162-2163) and the call returns
 *     B200LZ4_E_BLOCK;
 *   - block header layout is the reference's (src/Streamly/Internal/LZ4.hs:177-207,
 *     :86-94): [compLen LE32][uncompLen LE32 iff header_mode == 8][LZ4 block];
 *   - "stream" = the reference's one-LZ4_stream_t-per-Haskell-stream (linked
 *     blocks, src/Streamly/Internal/LZ4.hs:367-394); "independent" = fresh state
 *     per block (test/Main.hs:57-65, the Config.hs:142-146 stub);
 *   - dictionary semantics are the canonical ones of SURVEY.md section 5 quirk 1:
 *     external-dictionary mode, dictionary = the immediately preceding array.
 *   - Device buffers handed to the *_dev entry points must be readable up to the
 *     next 16-byte boundary past their last byte (true for any cudaMalloc /
 *     torch allocation).
 *   - ONE deliberate difference on INVALID input: a match offset of 0 (which the LZ4 block
 *     format forbids) makes the block fail (out_len < 0).  LZ4 1.9.3's safe decoder accepts
 *     it and copies bytes of its own not-yet-written output (cbits/lz4.c:2122-2130), so
 *     the reference "succeeds" with data that depends on what the destination buffer held
 *     before.  Every other accept/reject decision is the reference's
 *     (tests/test_gpu_fuzz.py pins both).
 */
#ifndef B200LZ4_H
#define B200LZ4_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200LZ4_VERSION_NUMBER 100            /* 0.1.0 */
#define B200LZ4_MAX_INPUT_SIZE 0x7E000000     /* LZ4_MAX_INPUT_SIZE, cbits/lz4.h:170 */

/* header_mode: number of header bytes in front of every LZ4 block */
#define B200LZ4_HDR_NONE 0                    /* raw LZ4 block */
#define B200LZ4_HDR_COMP 4                    /* BlockMax64KB..4MB: [compLen]            (Config.hs:121-131) */
#define B200LZ4_HDR_BOTH 8                    /* BlockHasSize:      [compLen][uncompLen] */

#define B200LZ4_OK        0
#define B200LZ4_E_CUDA   (-1)                 /* CUDA runtime error / no usable sm_100 device */
#define B200LZ4_E_ARG    (-2)                 /* invalid argument */
#define B200LZ4_E_NOMEM  (-3)                 /* host or device allocation failed / dst too small */
#define B200LZ4_E_BLOCK  (-4)                 /* at least one block failed; see out_len[] */
#define B200LZ4_E_FRAME  (-5)                 /* re-frame: incomplete block / missing end mark / bad header */
#define B200LZ4_E_CHECKSUM (-6)               /* LZ4 frame: header, block or content checksum mismatch (per frame) */

/* LZ4 frame options: the FLG bits of the frame format (lz4_Frame_format.md) */
#define B200LZ4_FRAME_INDEPENDENT      0x20   /* blocks are independent (clear: each block may reference the previous 64 KiB) */
#define B200LZ4_FRAME_BLOCK_CHECKSUM   0x10   /* XXH32 of every block's data follows it */
#define B200LZ4_FRAME_CONTENT_SIZE     0x08   /* the header holds the content size */
#define B200LZ4_FRAME_CONTENT_CHECKSUM 0x04   /* XXH32 of the whole content follows the end mark */

typedef struct b200lz4_ctx b200lz4_ctx;               /* one per (host thread, device) */
typedef struct b200lz4_cstream b200lz4_cstream;       /* device-resident LZ4_stream_t equivalent (cbits/lz4.h:595-603) */
typedef struct b200lz4_dstream b200lz4_dstream;       /* device-resident LZ4_streamDecode_t equivalent (cbits/lz4.h:605-610) */
typedef struct b200lz4_dict b200lz4_dict;             /* a dictionary loaded on one ctx's device (LZ4_loadDict semantics) */

/* ---------------------------------------------------------------- misc -- */

/* LZ4_compressBound (cbits/lz4.c:674, cbits/lz4.h:170-171): n + n/255 + 16, 0 if n is out of range. */
int b200lz4_compress_bound(int n);
int b200lz4_version(void);
const char* b200lz4_last_error(void);
/* number of CUDA devices this library can drive (compute capability 10.x); <= 0 if none */
int b200lz4_device_count(void);

/* ------------------------------------------------------------- context -- */

int  b200lz4_ctx_create(int device, b200lz4_ctx** out);
void b200lz4_ctx_destroy(b200lz4_ctx* ctx);
/* page-locked host memory for batching arrays (what the Haskell shim copies chunks into) */
void* b200lz4_host_alloc(size_t bytes);
/* the same as write-combined memory: for buffers the host only WRITES (batch input): the DMA engine reads them without
 * cache snooping, which helps when several GPUs pull from one host at once; host READS of such memory are very slow */
void* b200lz4_host_alloc_wc(size_t bytes);
/* the same from any host thread: selects the ctx's device first (a helper thread that stages the next batch must
 * not create a CUDA context on device 0 as a side effect) */
void* b200lz4_ctx_host_alloc(b200lz4_ctx* ctx, size_t bytes);
void  b200lz4_host_free(void* p);

/* per-call device timings of the last *_batch call on this ctx, milliseconds
 * (CUDA events): h2d copy, kernels (codec + compaction), d2h copy */
int b200lz4_last_timing(b200lz4_ctx* ctx, float* h2d_ms, float* kernel_ms, float* d2h_ms);
/* kernels launched by this ctx since creation (codec, scan, gather kernels) */
int64_t b200lz4_launch_count(b200lz4_ctx* ctx);
/* text of the last failure of a *_batch call on this ctx, whichever OS thread made it (b200lz4_last_error() is
 * per calling thread, which an unbound Haskell thread cannot rely on between a `safe` and an `unsafe` call) */
const char* b200lz4_ctx_last_error(b200lz4_ctx* ctx);

/* Staging helper: copy n separately allocated arrays (pageable memory) to dst + dst_off[i] with `threads` host
 * threads (0 = a default), one contiguous range of arrays per thread.  This is the gather into page-locked memory
 * that precedes every batch call when the caller's arrays are not page-locked themselves (Haskell `Array Word8`). */
int b200lz4_gather_host(void* dst, const void* const* src_ptrs, const int64_t* dst_off, const int32_t* len, int n, int threads);

/* Measurement aid: one plain H2D copy (h2d_bytes from h_src) and one D2H copy (d2h_bytes into h_dst) on the ctx's two
 * copy streams at once, no kernels, returns when both are complete -- the transfer ceiling an end-to-end call is
 * compared against (bench.py `e2e.copy_ceiling`). */
int b200lz4_copy_probe(b200lz4_ctx* ctx, const void* h_src, int64_t h2d_bytes, void* h_dst, int64_t d2h_bytes);

/* -------------------------------------------------- linked-stream state -- */
/* replaces LZ4_createStream / LZ4_freeStream (cbits/lz4.c:1423-1471) and
 * LZ4_createStreamDecode / LZ4_freeStreamDecode (cbits/lz4.c:2265-2277) for the
 * batched path; state lives in HBM between calls. */
int  b200lz4_cstream_create(b200lz4_ctx* ctx, b200lz4_cstream** out);
void b200lz4_cstream_free(b200lz4_cstream* s);
int  b200lz4_dstream_create(b200lz4_ctx* ctx, b200lz4_dstream** out);
void b200lz4_dstream_free(b200lz4_dstream* s);
/* test hooks: copy the 4096-entry hash table / currentOffset of a stream to the host */
int  b200lz4_cstream_peek(b200lz4_cstream* s, uint32_t* table4096, uint32_t* current_offset);

/* ----------------------------------------------------- batched, HOST data -- */
/*
 * Compress n_blocks arrays; array i = src[src_off[i] .. src_off[i]+src_len[i]).
 * Replaces n_blocks calls of compressChunk (src/Streamly/Internal/LZ4.hs:226-281),
 * i.e. LZ4_compressBound + LZ4_compress_fast_continue + the header pokes.
 *
 *   stream_first / n_streams / streams:
 *       stream_first == NULL            -> every block independent (fresh state);
 *       else stream s owns blocks stream_first[s] .. stream_first[s+1]-1, in order,
 *       all through ONE state: streams[s] if streams != NULL (state persists
 *       across calls, like one LZ4_stream_t per Haskell stream), else a fresh one.
 *   acceleration: as LZ4_compress_fast_continue (clamped to [1,65537], cbits/lz4.c:1577-1578).
 *   dst / dst_cap: receives the framed blocks back to back:
 *       block i = dst[dst_off[i] .. dst_off[i+1]) = [header][LZ4 block], dst_off has n_blocks+1 entries.
 *       dst_cap >= sum(header_mode + b200lz4_compress_bound(src_len[i])) is always enough.
 *   out_len[i] = LZ4 payload bytes of block i (0 = that block failed).
 */
int b200lz4_compress_batch(b200lz4_ctx* ctx,
                           const void* src, int64_t src_bytes,
                           const int64_t* src_off, const int32_t* src_len, int n_blocks,
                           const int32_t* stream_first, int n_streams, b200lz4_cstream* const* streams,
                           int acceleration, int header_mode,
                           void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len);

/*
 * Decompress n_blocks framed arrays; array i = src[src_off[i] .. +src_len[i]) holds exactly
 * one [header][LZ4 block] (what resizeChunksD yields).  Replaces n_blocks calls of
 * decompressChunk (src/Streamly/Internal/LZ4.hs:290-336).
 *   header_mode 8: capacity of block i = its header's uncompLen;
 *   header_mode 4: capacity = max_block (64K/256K/1M/4M, LZ4.hs:195-198);
 *   header_mode 0: src_len[i] is the payload length, capacity = max_block.
 * Output array i = dst[dst_off[i] .. dst_off[i]+out_len[i]); out_len[i] < 0 = failed.
 * dst_cap >= sum of capacities is always enough.
 */
int b200lz4_decompress_batch(b200lz4_ctx* ctx,
                             const void* src, int64_t src_bytes,
                             const int64_t* src_off, const int32_t* src_len, int n_blocks,
                             const int32_t* stream_first, int n_streams, b200lz4_dstream* const* streams,
                             int header_mode, int max_block,
                             void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len);

/* ---------------------------------------------------------- dictionaries -- */
/*
 * A shared dictionary, byte-exact with upstream LZ4 (1.9.3 / 1.9.4):
 *   compress    = LZ4_createStream -> LZ4_loadDict(s, dict, len) -> LZ4_compress_fast_continue per array.  Only the last
 *                 64 KiB count; a dictionary shorter than 8 bytes loads nothing but still moves currentOffset to 64 KiB,
 *                 so the output differs from a fresh stream's.
 *   decompress  = LZ4_decompress_safe_usingDict(src, dst, n, cap, dict, len) for a stream's first block (linked streams:
 *                 LZ4_setStreamDecode(dict, len) then _continue).  The whole length counts for the offset check.
 * b200lz4_dict_create copies len host bytes to the ctx's device and loads them there; the dict belongs to that ctx and may
 * be used by any number of calls until b200lz4_dict_free.
 * *_batch_dict: the arguments of b200lz4_{de,}compress_batch plus the dictionary.  Every stream starts from it (independent
 * mode: every block; linked mode: the first block of each stream, later blocks see the previous array as usual).  Passing
 * persistent `streams` as well is B200LZ4_E_ARG: load the dictionary into the handles instead (b200lz4_cstream_load_dict,
 * b200lz4_dstream_set_dict), which is LZ4_loadDict / LZ4_setStreamDecode on a stream that persists across calls.
 * The multi-device calls take no dictionary.
 */
int  b200lz4_dict_create(b200lz4_ctx* ctx, const void* dict, int64_t len, b200lz4_dict** out);
void b200lz4_dict_free(b200lz4_dict* d);
int  b200lz4_cstream_load_dict(b200lz4_cstream* s, const b200lz4_dict* d);
int  b200lz4_dstream_set_dict(b200lz4_dstream* s, const b200lz4_dict* d);
int b200lz4_compress_batch_dict(b200lz4_ctx* ctx,
                                const void* src, int64_t src_bytes,
                                const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                const int32_t* stream_first, int n_streams, b200lz4_cstream* const* streams,
                                int acceleration, int header_mode,
                                void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len, const b200lz4_dict* dict);
int b200lz4_decompress_batch_dict(b200lz4_ctx* ctx,
                                  const void* src, int64_t src_bytes,
                                  const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                  const int32_t* stream_first, int n_streams, b200lz4_dstream* const* streams,
                                  int header_mode, int max_block,
                                  void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len, const b200lz4_dict* dict);

/* ------------------------------------------- batched, HOST data, N devices -- */
/* One batch striped over several GPUs of one box (SURVEY.md section 8e): contiguous ranges of blocks (independent
 * mode) or of whole streams (linked mode), balanced by source bytes; one host thread and one b200lz4_ctx per device;
 * no exchange step between devices.  Arguments as b200lz4_compress_batch / b200lz4_decompress_batch, except:
 *   - linked streams start from a fresh state (no persistent stream handles across calls);
 *   - block i occupies dst[dst_off[i] .. dst_off[i] + header_mode + out_len[i]) (compress) or
 *     dst[dst_off[i] .. dst_off[i] + out_len[i]) (decompress); blocks are in order, but dst_off[i+1] may lie beyond
 *     the end of block i where two devices' ranges meet (each device writes into its own worst-case region), so
 *     dst_cap must be >= the sum of header_mode + b200lz4_compress_bound(src_len[i]) (compress) / of the block
 *     capacities (decompress).
 * devices == NULL: the first n usable devices (n <= 0: all).  There are no dictionary variants of these calls. */
typedef struct b200lz4_mctx b200lz4_mctx;
int  b200lz4_mctx_create(const int* devices, int n, b200lz4_mctx** out);
void b200lz4_mctx_destroy(b200lz4_mctx* m);
int  b200lz4_mctx_size(b200lz4_mctx* m);
b200lz4_ctx* b200lz4_mctx_ctx(b200lz4_mctx* m, int i);          /* per-device ctx: timings, launch counts */
const char* b200lz4_mctx_last_error(b200lz4_mctx* m);
int b200lz4_compress_batch_multi(b200lz4_mctx* m, const void* src, int64_t src_bytes,
                                 const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                 const int32_t* stream_first, int n_streams,
                                 int acceleration, int header_mode,
                                 void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len);
int b200lz4_decompress_batch_multi(b200lz4_mctx* m, const void* src, int64_t src_bytes,
                                   const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                   const int32_t* stream_first, int n_streams,
                                   int header_mode, int max_block,
                                   void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len);

/* --------------------------------------------------- batched, DEVICE data -- */
/* Everything below takes DEVICE pointers (data and descriptor arrays) and only
 * enqueues work on `cuda_stream` (a cudaStream_t, NULL = legacy default stream):
 * no host synchronisation, no host<->device copy.  This is the kernel-resident
 * path measured as bench.py's `value`. */

/* bytes of one device stream-state record (compress / decompress) */
size_t b200lz4_cstate_bytes(void);
size_t b200lz4_dstate_bytes(void);
/* bytes of scratch the *_dev calls need (work counters etc.); must be zero-filled once */
size_t b200lz4_scratch_bytes(void);

/*
 * d_states: NULL (fresh state per stream, discarded) or device array of n_streams device
 * pointers to b200lz4_cstate_bytes() records (zero-filled = new stream).  A record's
 * dictionary buffer must have been sized with b200lz4_cstate_set_dict() to hold the
 * largest array of its stream.  Records (compress and decompress alike) must be 16-byte
 * aligned; both record sizes are multiples of 16, so records packed back to back from an
 * aligned start are.
 * d_dst_cap: NULL (capacity = header_mode + compress_bound, i.e. never limiting) or per-block
 * slot capacities, header included.  Block i writes only inside
 * d_dst[d_dst_off[i] .. d_dst_off[i] + d_dst_cap[i]).  It succeeds exactly when its LZ4 payload
 * fits in d_dst_cap[i] - header_mode bytes (the limitedOutput rule of LZ4_compress_fast_continue);
 * otherwise d_out_len[i] = 0.  A failed block whose slot holds the header gets compLen 0 there;
 * a slot smaller than header_mode is not written at all.
 */
int b200lz4_compress_dev(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                         const int32_t* d_stream_first, int n_streams, void* const* d_states,
                         void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                         int acceleration, int header_mode,
                         void* d_scratch, void* cuda_stream);

/* attach a device buffer that will hold a stream's previous array between calls
 * (the reference keeps the previous Haskell array alive, LZ4.hs:389) */
int b200lz4_cstate_set_dict(void* d_state, void* d_dict_buf, uint32_t dict_cap, void* cuda_stream);

int b200lz4_decompress_dev(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                           const int32_t* d_stream_first, int n_streams, void* const* d_states,
                           void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                           int header_mode, int max_block,
                           void* d_scratch, void* cuda_stream);

/*
 * Dictionaries on the device.  b200lz4_dict_load_dev enqueues LZ4_loadDict(d_dict, len) into the record d_cstate
 * (b200lz4_cstate_bytes(), 16-byte aligned; it points into d_dict, which must stay unchanged while the record is used)
 * and LZ4_setStreamDecode(d_dict, len) into d_dstate (b200lz4_dstate_bytes(); the bytes are copied in).  Either may be
 * NULL.  The *_dev_dict calls take the arguments of the *_dev calls plus such a record, which every stream starts from
 * and which no kernel writes; d_states must be NULL then (B200LZ4_E_ARG otherwise).
 */
int b200lz4_dict_load_dev(const void* d_dict, int64_t len, void* d_cstate, void* d_dstate, void* cuda_stream);
int b200lz4_compress_dev_dict(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                              const int32_t* d_stream_first, int n_streams, void* const* d_states, const void* d_dict_cstate,
                              void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                              int acceleration, int header_mode,
                              void* d_scratch, void* cuda_stream);
int b200lz4_decompress_dev_dict(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                                const int32_t* d_stream_first, int n_streams, void* const* d_states, const void* d_dict_dstate,
                                void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                                int header_mode, int max_block,
                                void* d_scratch, void* cuda_stream);

/*
 * Compaction pass: gather per-block slots into one contiguous framed stream.
 * d_out_off[0..n_blocks] receives the exclusive prefix sum of (header_mode + d_len[i])
 * (failed blocks, d_len <= 0, contribute nothing); block i is copied from
 * d_slots + d_slot_off[i] to d_out + d_out_off[i].
 */
int b200lz4_compact_dev(const void* d_slots, const int64_t* d_slot_off, const int32_t* d_len, int n_blocks,
                        int header_mode, void* d_out, int64_t* d_out_off,
                        void* d_scratch, void* cuda_stream);

/* ------------------------------------------------------------- re-frame -- */
/*
 * resizeChunksD (src/Streamly/Internal/LZ4.hs:432-523) as a function over one contiguous
 * byte range: walk the compLen header chain of `buf[0..len)` and report where each
 * [header][block] array starts.  Because the walk only needs the bytes seen so far it can be
 * called incrementally: it consumes as many COMPLETE blocks as `buf` holds.
 *   block_off[k], block_len[k] (k < *n_found <= max_blocks): start and total length
 *       (header + payload) of block k inside buf;
 *   *consumed: bytes of buf covered by the reported blocks (+ the 4-byte end mark if seen);
 *   *ended: 1 if has_end_mark and the end mark was reached (the stream stops, LZ4.hs:506-522).
 * Returns B200LZ4_OK, or B200LZ4_E_FRAME if a header carries compLen <= 0.
 * A trailing incomplete block is not an error here; the caller reports
 * "resizeChunksD: Incomplete block" (LZ4.hs:505) if the input ends with *consumed < len.
 */
int b200lz4_reframe(const void* buf, int64_t len, int header_mode, int has_end_mark,
                    int64_t* block_off, int32_t* block_len, int64_t max_blocks,
                    int64_t* n_found, int64_t* consumed, int* ended);

/*
 * The same header walk for a stream that is already in HBM (section 8f rank 4: data that never touches the host):
 * one thread follows the compLen chain of d_buf[0..len) and fills d_block_off / d_block_len (device arrays of
 * max_blocks entries, usable directly as src_off / src_len of b200lz4_decompress_dev) and
 * d_result[0..2] = {n_found, consumed, ended}; d_result[3] = 1 if a header carried compLen <= 0 (B200LZ4_E_FRAME).
 * Only enqueues work on cuda_stream.
 */
int b200lz4_reframe_dev(const void* d_buf, int64_t len, int header_mode, int has_end_mark,
                        int64_t* d_block_off, int32_t* d_block_len, int64_t max_blocks,
                        int64_t* d_result, void* cuda_stream);

/* ------------------------------------------------------------ checksums -- */
/*
 * XXH32 (seed as given) of n byte ranges buf[off[i] .. off[i]+len[i]): what the LZ4 frame format uses for its header
 * checksum byte ((xxh32(descriptor) >> 8) & 0xFF), block checksums and content checksum.  The reference parses the
 * header checksum with `satisfy (const True)` and rejects both checksum flags (src/Streamly/Internal/LZ4.hs:602,
 * :631-640); these entry points are what a complete frame reader / writer needs (SURVEY.md section 8f rank 3).
 * _dev: device pointers, enqueue only.  _batch: host pointers (copied to the device, hashed there, results copied back).
 */
int b200lz4_xxh32_dev(const void* d_buf, const int64_t* d_off, const int32_t* d_len, int n, uint32_t seed, uint32_t* d_out, void* cuda_stream);
int b200lz4_xxh32_batch(b200lz4_ctx* ctx, const void* src, int64_t src_bytes, const int64_t* off, const int32_t* len, int n,
                        uint32_t seed, uint32_t* out);

/* ---------------------------------------------------------- LZ4 frames -- */
/*
 * Standard LZ4 frames (what the `lz4` tool, LZ4F_compressFrame and lz4.frame write), n at a time: array i <-> frame i.
 *
 * b200lz4_frame_bound: the largest frame an n-byte array can become with this block maximum and these flags (header of at
 * most 15 bytes, per block 4 + its raw bytes + 4 with block checksums, the end mark, 4 with a content checksum); < 0 for
 * an invalid argument.
 *
 * b200lz4_frame_info: parse one frame header on the host (magic, version, reserved bits, block maximum, header checksum).
 * Returns B200LZ4_OK, B200LZ4_E_FRAME (not a frame header, or one with a dictionary id), B200LZ4_E_CHECKSUM (header
 * checksum) or B200LZ4_E_ARG (fewer bytes than the header needs).  *content_size = -1 if the header holds none; *flags:
 * B200LZ4_FRAME_* bits.  Any output pointer may be NULL.
 *
 * b200lz4_frame_compress_batch: array i = src[src_off[i] .. +src_len[i]) becomes frame i, cut into blocks of block_max
 * (65536, 262144, 1048576 or 4194304) bytes.  The blocks are this library's byte-exact LZ4 blocks (independent frames: a
 * fresh stream per block; linked frames: one stream per frame, the previous block as dictionary), stored raw (size bit 31)
 * when the payload is not shorter than the raw bytes.  flags: B200LZ4_FRAME_* (content size = the array's length).  Frames
 * are written back to back: frame i = dst[dst_off[i] .. dst_off[i+1]), out_len[i] = its size; dst_off has n_frames + 1
 * entries.  dst_cap >= the sum of b200lz4_frame_bound(src_len[i]) is always enough.  Not byte-identical to
 * LZ4F_compressFrame (its block tables differ below 65 547 bytes), but every frame decoder reads the output.
 *
 * b200lz4_frame_decompress_batch: range i = src[src_off[i] .. +src_len[i]) holds exactly one frame; its content goes to
 * dst[dst_off[i] ..) with capacity dst_cap[i].  out_len[i] = content bytes, or
 *     B200LZ4_E_FRAME     bad header / reserved bits / dictionary id / block above the maximum / truncation / missing end
 *                         mark / bytes after the frame / content size mismatch,
 *     B200LZ4_E_BLOCK     the safe decoder rejected a block,
 *     B200LZ4_E_CHECKSUM  header, block or content checksum mismatch,
 *     B200LZ4_E_NOMEM     the content exceeds dst_cap[i].
 * A failing frame never aborts the batch (the call returns B200LZ4_E_BLOCK then) and leaves its destination untouched,
 * except with a content checksum mismatch, found after the content was written.  Linked blocks see the last 64 KiB of
 * decoded data, as upstream's frame decoder does, whatever the sizes of earlier blocks.
 *
 * Both calls take host or device pointers for the data and for the descriptor arrays (told apart with
 * cudaPointerGetAttributes).  Device data never leaves the device; host data is copied in once and out once.
 */
int64_t b200lz4_frame_bound(int64_t n, int block_max, int flags);
int b200lz4_frame_info(const void* buf, int64_t len, int* block_max, int* flags, int64_t* content_size, int* header_len);
int b200lz4_frame_compress_batch(b200lz4_ctx* ctx, const void* src, int64_t src_bytes,
                                 const int64_t* src_off, const int32_t* src_len, int n_frames,
                                 int block_max, int flags, int acceleration,
                                 void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len);
int b200lz4_frame_decompress_batch(b200lz4_ctx* ctx, const void* src, int64_t src_bytes,
                                   const int64_t* src_off, const int32_t* src_len, int n_frames,
                                   void* dst, const int32_t* dst_cap, const int64_t* dst_off, int32_t* out_len);

/* ------------------------------------------------------ legacy aliases -- */
/* Same names, signatures and return conventions as the 7 symbols the unmodified reference
 * imports (src/Streamly/Internal/LZ4.hs:105-140; cbits/lz4.h:170,182,273-274,336,358-359,409).
 * The opaque stream objects hold device state; data is staged to the GPU per call. */
typedef struct LZ4_stream_u LZ4_stream_t;
typedef struct LZ4_streamDecode_u LZ4_streamDecode_t;
LZ4_stream_t* LZ4_createStream(void);
int LZ4_freeStream(LZ4_stream_t* s);
LZ4_streamDecode_t* LZ4_createStreamDecode(void);
int LZ4_freeStreamDecode(LZ4_streamDecode_t* s);
int LZ4_compressBound(int inputSize);
int LZ4_compress_fast_continue(LZ4_stream_t* s, const char* src, char* dst, int srcSize, int dstCapacity, int acceleration);
int LZ4_decompress_safe_continue(LZ4_streamDecode_t* s, const char* src, char* dst, int srcSize, int dstCapacity);
/* upstream's dictionary calls, same signatures and results: LZ4_loadDict returns the dictionary size it kept (the last
 * 64 KiB, 0 below 8 bytes), LZ4_setStreamDecode returns 1 (0 on a failure upstream cannot have, e.g. no device) */
int LZ4_loadDict(LZ4_stream_t* s, const char* dictionary, int dictSize);
int LZ4_setStreamDecode(LZ4_streamDecode_t* s, const char* dictionary, int dictSize);

#ifdef __cplusplus
}
#endif
#endif /* B200LZ4_H */
