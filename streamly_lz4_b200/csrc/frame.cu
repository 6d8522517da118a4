// frame.cu -- LZ4 frames (lz4_Frame_format.md) around the block kernels: the per-frame header walk and block descriptors
// of the decode side, the staging of stored blocks, the per-frame verdicts, and the block packing and header writing of the
// encode side.  The codec work itself is done by the existing compressor and decoders; XXH32 by xxh32.cu.
//
// Decode (api.cu: b200lz4_frame_decompress_batch):
//   walk (count) -> scan -> [host reads the totals] -> walk (fill) -> stage -> decoders (one launch per block maximum)
//   -> block XXH32 -> settle -> [scan] -> place -> gather -> content XXH32 -> verdict
// Encode (b200lz4_frame_compress_batch):
//   compressor (header 0, one stream per linked frame) -> sizes -> scan -> pack -> block XXH32 -> content XXH32 -> finish
#include "common.cuh"
#include "kernels.h"
#include "b200lz4.h"

namespace b200lz4 {

namespace {

constexpr uint32_t kMagic = 0x184D2204u;
constexpr uint32_t kP1 = 2654435761u, kP2 = 2246822519u, kP3 = 3266489917u, kP4 = 668265263u, kP5 = 374761393u;

__device__ __forceinline__ uint32_t rd32(const uint8_t* p)
{ return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
__device__ __forceinline__ void wr32(uint8_t* p, uint32_t v)
{ p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

// XXH32 (seed 0) of fewer than 16 bytes: the frame descriptor (api.py: _xxh32_short)
__device__ uint32_t xxh32_short(const uint8_t* p, int n)
{
    uint32_t h = kP5 + (uint32_t)n;
    int at = 0;
    for (; at + 4 <= n; at += 4) { const uint32_t x = h + rd32(p + at) * kP3; h = __funnelshift_l(x, x, 17) * kP4; }
    for (; at < n; at++) { const uint32_t x = h + (uint32_t)p[at] * kP5; h = __funnelshift_l(x, x, 11) * kP1; }
    h ^= h >> 15; h *= kP2; h ^= h >> 13; h *= kP3; h ^= h >> 16;
    return h;
}

__device__ __forceinline__ int bmax_of(int cls) { return 65536 << (2 * cls); }

// bytes of the literal-only LZ4 block that decodes to n raw bytes: token, length bytes, the bytes
__device__ __forceinline__ long long literal_block_len(long long n) { return 1 + (n >= 15 ? (n - 15) / 255 + 1 : 0) + n; }
__device__ __forceinline__ long long al16(long long v) { return (v + 15) & ~15ll; }

// Output slot of one block.  A decoder writes exactly the bytes it produces, and an LZ4 block of c bytes produces at most
// 255 bytes per input byte, so the slot does not need the whole block maximum (which stays the decoder's capacity).
__device__ __forceinline__ long long slot_of(bool stored, long long n, int bmax)
{ return al16(stored ? n : min((long long)bmax, 256 * n + 64)); }

// One thread per frame: validate the header, follow the block chain (one dependent 4-byte load per block).
// !kFill: write the frame's record (counts, class, flags); kFill: write the per-block descriptors at the scanned bases.
template <bool kFill>
__global__ void frame_walk_kernel(FrameDecodeArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (kFill && i == 0) {                  // the terminator of each class's stream_first run (the arena exists from now on)
        long long sb = 0;
        for (int c = 0; c < 4; c++) { sb += a.totals[4 + c]; a.sf[sb] = (int32_t)a.totals[c]; sb++; }
    }
    if (i >= a.n) return;
    FrameRec r{};
    const uint8_t* p = a.base + a.src_off[i];
    const long long L = a.src_len[i];
    long long at = 0;
    int err = 0;
    if (kFill) { r = a.rec[i]; if (r.err || r.nblk == 0) return; }
    r.content_size = -1;
    const int flg = L >= 6 ? p[4] : 0, bd = L >= 6 ? p[5] : 0;
    if (L < 7 || rd32(p) != kMagic || (flg >> 6) != 1 || (flg & 0x02) || (bd & 0x8F) || (flg & 0x01) || ((bd >> 4) & 7) < 4)
        err = B200LZ4_E_FRAME;                                  // magic, version, reserved bits, dictionary id, block maximum
    if (!err) {
        at = 6;
        if (flg & 0x08) {
            if (L < 15) err = B200LZ4_E_FRAME;
            else {
                unsigned long long cs = 0;
                for (int k = 7; k >= 0; k--) cs = (cs << 8) | p[6 + k];
                r.content_size = cs > 0x7FFFFFFFFFFFFFFFull ? 0x7FFFFFFFFFFFFFFFll : (long long)cs;
                at = 14;
            }
        }
        if (!err && p[at] != ((xxh32_short(p + 4, (int)at - 4) >> 8) & 0xFF)) err = B200LZ4_E_CHECKSUM;
        at += 1;
    }
    const int cls = ((bd >> 4) & 7) - 4, bmax = err ? 0 : bmax_of(cls);
    const bool linked = !(flg & 0x20), bc = flg & 0x10;
    long long nblk = 0, stage = 0, slot = 0;
    bool short_seen = false, window = false;
    // kFill: descriptors of block k at index g = blk + k; independent frames open a stream per block, linked ones one
    long long g = r.fb.blk, rel = r.fb.rel, stage_at = r.fb.stage, slot_at = r.fb.slot;
    if (kFill && linked) a.sf[r.fb.str] = (int32_t)rel;
    while (!err) {
        if (L - at < 4) { err = B200LZ4_E_FRAME; break; }       // truncated before the next block size / the end mark
        const uint32_t size = rd32(p + at);
        at += 4;
        const long long n = size & 0x7FFFFFFFu;
        if (n == 0) break;                                      // end mark (upstream reads the size without its stored bit)
        const bool stored = size >> 31;
        if (n > bmax || L - at < n + (bc ? 4 : 0)) { err = B200LZ4_E_FRAME; break; }
        // a block that may decode to less than 64 KiB, followed by another block: that one may reach past it (window mode)
        if (linked && short_seen) window = true;
        short_seen = stored ? n < 65536 : (n - n / 255 - 16) < 65536;
        const long long stage_n = stored ? al16(literal_block_len(n)) : 0, slot_n = slot_of(stored, n, bmax);
        if (kFill) {
            a.raw_off[g] = a.src_off[i] + at;
            a.meta[g] = (int32_t)n | (stored ? (int32_t)0x80000000 : 0);
            a.csum_len[g] = bc ? (int32_t)n : 0;
            a.csum_exp[g] = bc ? rd32(p + at + n) : 0u;
            a.bframe[g] = i;
            a.dsrc_off[g] = stored ? a.stage_delta + stage_at : a.src_off[i] + at;
            a.dsrc_len[g] = stored ? (int32_t)literal_block_len(n) : (int32_t)n;
            a.slot_off[g] = slot_at;
            if (!linked) a.sf[r.fb.str + nblk] = (int32_t)(rel + nblk);
            g++; stage_at += stage_n; slot_at += slot_n;
        }
        nblk++; stage += stage_n; slot += slot_n;
        at += n + (bc ? 4 : 0);
    }
    if (!err && (flg & 0x04)) {
        if (L - at < 4) err = B200LZ4_E_FRAME;
        else { r.ccsum = rd32(p + at); at += 4; }
    }
    if (!err && at != L) err = B200LZ4_E_FRAME;                 // one frame per range: nothing may follow it
    if (kFill) return;
    r.err = err; r.cls = err ? 0 : cls; r.flags = flg;
    r.nblk = err ? 0 : (int)nblk;
    r.window = !err && window;
    r.stage = err ? 0 : stage; r.slot = err ? 0 : slot;
    a.rec[i] = r;
}

// Exclusive scans of the per-frame counts: block index (per class, classes back to back), stream index (per class, one
// spare entry per class for the terminator of its stream_first run), staging and slot bytes (global).  totals: kFrameTotals
// values (see kernels.h), read back by the host to size the block arena and pick the decoder per class.
constexpr int kScanT = 256;
constexpr int kV = kFrameTotals;

__device__ __forceinline__ void frame_counts(const FrameRec& r, long long* v)
{
    for (int k = 0; k < kV; k++) v[k] = 0;
    if (r.err) return;
    v[r.cls] = r.nblk;
    v[4 + r.cls] = (r.flags & 0x20) ? r.nblk : (r.nblk ? 1 : 0);
    v[8 + r.cls] = r.window;
    v[12] = r.stage; v[13] = r.slot;
}

__global__ void __launch_bounds__(kScanT) frame_scan_kernel(FrameDecodeArgs a)
{
    __shared__ long long part[kScanT][kV];
    const int t = threadIdx.x, n = a.n;
    const int per = (n + kScanT - 1) / kScanT, lo = min(t * per, n), hi = min(lo + per, n);
    long long sum[kV], v[kV];
    for (int k = 0; k < kV; k++) sum[k] = 0;
    for (int i = lo; i < hi; i++) { frame_counts(a.rec[i], v); for (int k = 0; k < kV; k++) sum[k] += v[k]; }
    for (int k = 0; k < kV; k++) part[t][k] = sum[k];
    __syncthreads();
    for (int d = 1; d < kScanT; d <<= 1) {              // Hillis-Steele inclusive scan, as compact.cu's scan_kernel
        long long x[kV];
        for (int k = 0; k < kV; k++) x[k] = t >= d ? part[t - d][k] : 0;
        __syncthreads();
        for (int k = 0; k < kV; k++) part[t][k] += x[k];
        __syncthreads();
    }
    long long tot[kV], blk_base[4], str_base[4];
    for (int k = 0; k < kV; k++) tot[k] = part[kScanT - 1][k];
    long long bb = 0, sb = 0;
    for (int c = 0; c < 4; c++) { blk_base[c] = bb; str_base[c] = sb; bb += tot[c]; sb += tot[4 + c] + 1; }
    long long run[kV];
    for (int k = 0; k < kV; k++) run[k] = part[t][k] - sum[k];
    for (int i = lo; i < hi; i++) {
        FrameRec r = a.rec[i];
        const int c = r.cls;
        r.fb.blk = blk_base[c] + run[c]; r.fb.rel = run[c];
        r.fb.str = str_base[c] + run[4 + c];
        r.fb.stage = run[12]; r.fb.slot = run[13];
        a.rec[i].fb = r.fb;
        frame_counts(r, v);
        for (int k = 0; k < kV; k++) run[k] += v[k];
    }
    if (t == 0) for (int k = 0; k < kV; k++) a.totals[k] = tot[k];
}

// Stored blocks become literal-only LZ4 blocks in the staging area (what read_frame does on the host), so that the
// decoders take them like any other block and a stored block stays the next linked block's dictionary.
constexpr int kStageT = 256;
__global__ void __launch_bounds__(kStageT) frame_stage_kernel(FrameDecodeArgs a, int nb)
{
    for (int g = blockIdx.x; g < nb; g += gridDim.x) {
        const int32_t m = a.meta[g];
        if (m >= 0) continue;
        const uint32_t n = (uint32_t)m & 0x7FFFFFFFu;
        uint8_t* d = const_cast<uint8_t*>(a.base) + a.dsrc_off[g];
        const uint8_t* s = a.base + a.raw_off[g];
        const uint32_t ext = n >= 15 ? (n - 15) / 255 + 1 : 0;
        for (uint32_t k = threadIdx.x; k < ext; k += kStageT) d[1 + k] = k + 1 < ext ? 255 : (uint8_t)((n - 15) % 255);
        if (threadIdx.x == 0) d[0] = (uint8_t)(n >= 15 ? 0xF0 : n << 4);
        d += 1 + ext;
        for (uint32_t k = threadIdx.x; k < n; k += kStageT) d[k] = s[k];
    }
}

// One thread per frame, after the decoders and the block checksums: the frame's verdict so far (in stream order: a block
// checksum before the block's decode, then the end-of-frame checks) and its content length; per block the offset of its
// output inside the content and the number of bytes the gather moves (none for a failed frame).
__global__ void frame_settle_kernel(FrameDecodeArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const FrameRec r = a.rec[i];
    int verdict = r.err;
    long long cont = 0;
    const long long g0 = r.fb.blk;
    for (int k = 0; k < r.nblk && !verdict; k++) {
        const long long g = g0 + k;
        if (a.csum_len[g] && a.csum_got[g] != a.csum_exp[g]) { verdict = B200LZ4_E_CHECKSUM; break; }
        const int ol = a.out_len[g];
        if (ol < 0) { verdict = B200LZ4_E_BLOCK; break; }
        a.gout_off[g] = cont; a.glen[g] = ol;
        cont += ol;
    }
    if (!verdict && r.content_size >= 0 && cont != r.content_size) verdict = B200LZ4_E_FRAME;
    if (!verdict && cont > a.dst_cap[i]) verdict = B200LZ4_E_NOMEM;
    if (verdict) for (int k = 0; k < r.nblk; k++) a.glen[g0 + k] = 0;
    a.content[i] = verdict ? 0 : (int32_t)cont;
    a.cclen[i] = !verdict && (r.flags & 0x04) ? (int32_t)cont : 0;
    a.result[i] = verdict ? verdict : (int32_t)cont;
}

// Block outputs at their place in the destination: the frame's base + the offset inside its content
__global__ void frame_place_kernel(FrameDecodeArgs a, int nb, const int64_t* __restrict__ fbase)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < nb) a.gout_off[g] += fbase[a.bframe[g]];
}

__global__ void frame_verdict_kernel(FrameDecodeArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if (a.result[i] >= 0 && (a.rec[i].flags & 0x04) && a.ccsum_got[i] != a.rec[i].ccsum) a.result[i] = B200LZ4_E_CHECKSUM;
}

// ---- encode ----

__device__ __forceinline__ int header_len(int flags) { return 7 + ((flags & B200LZ4_FRAME_CONTENT_SIZE) ? 8 : 0); }

// One thread per frame: framed size of every block (size field, stored raw bytes when the payload is not shorter, block
// checksum) and of the frame (header, blocks, end mark, content checksum)
__global__ void frame_csize_kernel(FrameEncodeArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const int bc = (a.flags & B200LZ4_FRAME_BLOCK_CHECKSUM) ? 4 : 0;
    long long at = header_len(a.flags);
    for (int g = a.frame_first[i]; g < a.frame_first[i + 1]; g++) {
        const int raw = a.blk_len[g], pay = a.pay_len[g];
        const bool stored = pay <= 0 || pay >= raw;
        a.blk_at[g] = at;
        at += 4 + (stored ? raw : pay) + bc;
    }
    at += 4 + ((a.flags & B200LZ4_FRAME_CONTENT_CHECKSUM) ? 4 : 0);
    a.fsize[i] = (int32_t)at;
}

// One CTA per block: the LE32 size field (bit 31: stored) and the block data, the compressed slot or the raw input
constexpr int kPackT = 256;
__global__ void __launch_bounds__(kPackT) frame_cpack_kernel(FrameEncodeArgs a, int nb)
{
    for (int g = blockIdx.x; g < nb; g += gridDim.x) {
        const int raw = a.blk_len[g], pay = a.pay_len[g];
        const bool stored = pay <= 0 || pay >= raw;
        const int n = stored ? raw : pay;
        const long long at = a.foff[a.blk_frame[g]] + a.blk_at[g];
        uint8_t* d = a.out + at;
        const uint8_t* s = stored ? a.src + a.blk_off[g] : a.slots + a.slot_off[g];
        if (threadIdx.x == 0) wr32(d, (uint32_t)n | (stored ? 0x80000000u : 0u));
        d += 4;
        for (int k = threadIdx.x; k < n; k += kPackT) d[k] = s[k];
        if (threadIdx.x == 0) { a.csum_off[g] = at + 4; a.csum_len[g] = (a.flags & B200LZ4_FRAME_BLOCK_CHECKSUM) ? n : 0; }
    }
}

// Threads g < nb store block checksums behind their blocks; threads i < n write frame i's header, end mark and content
// checksum
__global__ void frame_cfinish_kernel(FrameEncodeArgs a, int nb)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nb && (a.flags & B200LZ4_FRAME_BLOCK_CHECKSUM)) wr32(a.out + a.csum_off[t] + a.csum_len[t], a.bsum[t]);
    if (t >= a.n) return;
    uint8_t* p = a.out + a.foff[t];
    const int flg = 0x40 | (a.flags & 0x3C);
    wr32(p, kMagic);
    p[4] = (uint8_t)flg; p[5] = (uint8_t)((4 + a.cls) << 4);
    int at = 6;
    if (flg & B200LZ4_FRAME_CONTENT_SIZE) {
        const unsigned long long cs = (unsigned long long)a.src_len[t];
        for (int k = 0; k < 8; k++) p[6 + k] = (uint8_t)(cs >> (8 * k));
        at = 14;
    }
    p[at] = (uint8_t)(xxh32_short(p + 4, at - 4) >> 8);
    uint8_t* e = a.out + a.foff[t + 1] - 4 - ((flg & B200LZ4_FRAME_CONTENT_CHECKSUM) ? 4 : 0);
    wr32(e, 0u);
    if (flg & B200LZ4_FRAME_CONTENT_CHECKSUM) wr32(e + 4, a.csum_content[t]);
}

inline int grid_for(long long n, int per) { return (int)((n + per - 1) / per); }

}  // namespace

cudaError_t launch_frame_walk(const FrameDecodeArgs& a, bool fill, cudaStream_t st)
{
    if (a.n <= 0) return cudaSuccess;
    if (fill) frame_walk_kernel<true><<<grid_for(a.n, 128), 128, 0, st>>>(a);
    else frame_walk_kernel<false><<<grid_for(a.n, 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_scan(const FrameDecodeArgs& a, cudaStream_t st)
{
    frame_scan_kernel<<<1, kScanT, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_stage(const FrameDecodeArgs& a, int nb, cudaStream_t st)
{
    if (nb <= 0) return cudaSuccess;
    int sm = 0; cudaError_t e = device_sm_count(&sm); if (e != cudaSuccess) return e;
    frame_stage_kernel<<<nb < sm * 8 ? nb : sm * 8, kStageT, 0, st>>>(a, nb);
    return cudaGetLastError();
}

cudaError_t launch_frame_settle(const FrameDecodeArgs& a, cudaStream_t st)
{
    if (a.n <= 0) return cudaSuccess;
    frame_settle_kernel<<<grid_for(a.n, 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_place(const FrameDecodeArgs& a, int nb, const int64_t* fbase, cudaStream_t st)
{
    if (nb <= 0) return cudaSuccess;
    frame_place_kernel<<<grid_for(nb, 256), 256, 0, st>>>(a, nb, fbase);
    return cudaGetLastError();
}

cudaError_t launch_frame_verdict(const FrameDecodeArgs& a, cudaStream_t st)
{
    if (a.n <= 0) return cudaSuccess;
    frame_verdict_kernel<<<grid_for(a.n, 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_csize(const FrameEncodeArgs& a, cudaStream_t st)
{
    if (a.n <= 0) return cudaSuccess;
    frame_csize_kernel<<<grid_for(a.n, 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_cpack(const FrameEncodeArgs& a, int nb, cudaStream_t st)
{
    if (nb <= 0) return cudaSuccess;
    int sm = 0; cudaError_t e = device_sm_count(&sm); if (e != cudaSuccess) return e;
    frame_cpack_kernel<<<nb < sm * 8 ? nb : sm * 8, kPackT, 0, st>>>(a, nb);
    return cudaGetLastError();
}

cudaError_t launch_frame_cfinish(const FrameEncodeArgs& a, int nb, cudaStream_t st)
{
    const int m = nb > a.n ? nb : a.n;
    if (m <= 0) return cudaSuccess;
    frame_cfinish_kernel<<<grid_for(m, 128), 128, 0, st>>>(a, nb);
    return cudaGetLastError();
}

}  // namespace b200lz4
