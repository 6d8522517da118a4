// kernels.h -- launch interfaces between the C ABI (api.cu) and the kernels.
#pragma once
#include <cstdint>
#include <mutex>
#include <cuda_runtime.h>
#include "common.cuh"

namespace b200lz4 {

struct CompressArgs {
    const uint8_t* src; const int64_t* src_off; const int32_t* src_len; int n_blocks;
    const int32_t* stream_first; int n_streams; void* const* states;
    int first_block;            // independent mode (stream_first == NULL): stream s is block first_block + s
    uint8_t* dst; const int64_t* dst_off; const int32_t* dst_cap; int32_t* out_len;
    int accel; int header;
    Scratch* scratch;
    // streamed launch (NULL: all input is resident): the launch's blocks are still arriving over PCIe, segment by
    // segment; *arrived segments of seg_bytes (a multiple of 128) bytes of EVERY block of the launch have landed.
    // Block starts must be 128-byte aligned.  busy_cycles[0] += finder cycles net of waiting, [1] += bytes.
    const uint32_t* arrived; int seg_bytes; unsigned long long* busy_cycles;
    // dictionary (NULL: none): a stream without a record of its own (states == NULL) starts from this read-only state,
    // written by launch_load_dict; shared by every stream of the launch and never written
    const CState* dict_state;
};

struct DecompressArgs {
    const uint8_t* src; const int64_t* src_off; const int32_t* src_len; int n_blocks;
    const int32_t* stream_first; int n_streams; void* const* states;
    int first_block;
    uint8_t* dst; const int64_t* dst_off; const int32_t* dst_cap; int32_t* out_len;
    int header; int max_block;
    Scratch* scratch;
    int debug;                  // measurement switches (B200LZ4_DECODE_DEBUG): 1 = copier skips every copy (parser-bound rate)
    uint4* wide_arena;          // descriptor rings of the wide kernel: wide_ctas x kWideArenaPerCta bytes (NULL: narrow kernel only)
    int wide_ctas;
    // streamed launch (NULL: off): every block of the launch has the same capacity, cut into n_segs segments of seg_bytes;
    // seg_count[s] counts the blocks whose segment s is in global memory, the last one sets host_ready[s] (mapped host memory)
    uint32_t* seg_count; uint32_t* host_ready; int seg_bytes; int n_segs;
    // mirrored launch (NULL: off; independent blocks only): block i's output is ALSO stored at host_dst + dst_off[i], page-locked
    // host memory with host_dst congruent to dst modulo 16
    uint8_t* host_dst;
    // dictionary (NULL: none): a stream without a record of its own (states == NULL) starts with this read-only
    // previous output (launch_load_dict); never written
    const DState* dict_state;
};

// Blocks [b0, b1) of stream s of a launch: its run in stream_first, or in independent mode the one block first_block + s.
// (Two scalar functions: returning the pair as one struct changes the register allocation of the narrow decoder.)
template <class Args> __device__ __forceinline__ int stream_begin(const Args& a, int s)
{ return a.stream_first ? a.stream_first[s] : a.first_block + s; }
template <class Args> __device__ __forceinline__ int stream_end(const Args& a, int s, int b0)
{ return a.stream_first ? a.stream_first[s + 1] : b0 + 1; }

// decompress_kernel_wide keeps its parsed-ahead sequence descriptors in global memory (L2): per CTA, kWideParsers rings of
// kWideRingBatches batches of 32 descriptors of 16 bytes.
constexpr int kWideParsers = 8;
constexpr int kWideRingBatches = 256;
constexpr size_t kWideArenaPerCta = size_t(kWideParsers) * kWideRingBatches * 32 * 16;     // 1 MiB
constexpr int kWideMaxCtas = 160;
// layout of the scratch block the *_dev entry points take: [Scratch counters][wide arena]
constexpr size_t kScratchBytes = sizeof(Scratch) + kWideMaxCtas * kWideArenaPerCta;

struct CompactArgs {
    const uint8_t* slots; const int64_t* slot_off; const int32_t* len; int n_blocks;
    int header; uint8_t* out; int64_t* out_off;
    // optional mirrors in mapped pinned HOST memory (written by the scan kernel over PCIe, so the host learns the
    // sizes without a D2H memcpy that would queue behind bulk transfers on the copy engine)
    int64_t* host_off; int32_t* host_len;
};

// Per-device setup a launcher does once (dynamic shared-memory limits), safe for host threads launching on several devices.
struct PerDeviceOnce {
    std::mutex mu;
    bool done[64] = {};
    template <class F> cudaError_t run(F configure)
    {
        int dev = 0; cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
        if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
        std::lock_guard<std::mutex> lk(mu);
        if (done[dev]) return cudaSuccess;
        e = configure();
        if (e == cudaSuccess) done[dev] = true;
        return e;
    }
};

cudaError_t launch_compress(const CompressArgs& a, cudaStream_t stream);
cudaError_t launch_set_flag(uint32_t* flag, uint32_t v, cudaStream_t stream);
cudaError_t preload_compress_kernels();
cudaError_t preload_compact_kernels();
cudaError_t launch_alias_probe(const uint32_t* flag, uint32_t* result, long long timeout_cycles, cudaStream_t stream);
cudaError_t launch_decompress(const DecompressArgs& a, cudaStream_t stream);
cudaError_t launch_decompress_wide(const DecompressArgs& a, int sm_count, cudaStream_t stream);
cudaError_t device_sm_count(int* out);
cudaError_t launch_compact(const CompactArgs& a, cudaStream_t stream);
cudaError_t launch_reframe(const uint8_t* buf, int64_t len, int header, int has_end_mark,
                           int64_t* block_off, int32_t* block_len, int64_t max_blocks, int64_t* result, cudaStream_t stream);
// LZ4_loadDict on the device: d_cstate (if not NULL) becomes the state LZ4_loadDict(dict, len) leaves in a fresh stream
// (its dict_buf points into dict, which must outlive every use of the record), d_dstate (if not NULL) the decode state
// LZ4_setStreamDecode(dict, len) sets up (the last 64 KiB copied in).  len >= 0.
cudaError_t launch_load_dict(const uint8_t* dict, int64_t len, CState* d_cstate, DState* d_dstate, cudaStream_t stream);
cudaError_t launch_xxh32(const uint8_t* buf, const int64_t* off, const int32_t* len, int n, uint32_t seed, uint32_t* out, cudaStream_t stream);
int kernel_launches_per_compress();
int kernel_launches_per_decompress();
int kernel_launches_per_compact();

}  // namespace b200lz4
