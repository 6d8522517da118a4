// compact.cu -- compaction pass: exclusive scan of framed block sizes, then a gather of the
// per-block slots into one contiguous stream (so D2H moves only real bytes and the host can
// slice arrays straight out of the result, headers already in place).
#include "common.cuh"
#include "kernels.h"

namespace b200lz4 {

namespace {

constexpr int kScanThreads = 1024;

__global__ void __launch_bounds__(kScanThreads)
scan_kernel(const int32_t* __restrict__ len, int n, int header, int64_t* __restrict__ out_off,
            int64_t* __restrict__ host_off, int32_t* __restrict__ host_len)
{
    __shared__ long long partial[kScanThreads];
    const int t = threadIdx.x;
    const int per = (n + kScanThreads - 1) / kScanThreads;
    const int lo = min(t * per, n), hi = min(lo + per, n);
    long long sum = 0;
    for (int i = lo; i < hi; i++) { int l = len[i]; sum += (l > 0) ? (long long)(l + header) : 0; }
    partial[t] = sum;
    __syncthreads();
    for (int d = 1; d < kScanThreads; d <<= 1) {       // Hillis-Steele inclusive scan
        long long v = (t >= d) ? partial[t - d] : 0;
        __syncthreads();
        partial[t] += v;
        __syncthreads();
    }
    long long run = partial[t] - sum;                   // exclusive prefix of this thread's chunk
    for (int i = lo; i < hi; i++) {
        const int l = len[i];
        out_off[i] = run;
        if (host_off) { host_off[i] = run; host_len[i] = l; }
        run += (l > 0) ? (long long)(l + header) : 0;
    }
    if (t == kScanThreads - 1) { out_off[n] = partial[t]; if (host_off) host_off[n] = partial[t]; }
}

constexpr int kGatherThreads = 256;

__global__ void __launch_bounds__(kGatherThreads)
gather_kernel(CompactArgs a)
{
    const uint32_t t = threadIdx.x;
    for (int b = blockIdx.x; b < a.n_blocks; b += gridDim.x) {
        const int l = a.len[b];
        if (l <= 0) continue;
        uint32_t n = (uint32_t)(l + a.header);
        const uint8_t* src = a.slots + a.slot_off[b];
        uint8_t* dst = a.out + a.out_off[b];
        uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
        if (head > n) head = n;
        if (t < head) dst[t] = __ldg(src + t);
        src += head; dst += head; n -= head;
        const uint32_t nvec = n >> 4;
        uintptr_t sa = reinterpret_cast<uintptr_t>(src);
        const uint32_t sh = (uint32_t)(sa & 3) * 8;
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t(3));
        uint4* dv = reinterpret_cast<uint4*>(dst);
        if ((sa & 15) == 0) {
            const uint4* sv = reinterpret_cast<const uint4*>(src);
            for (uint32_t v = t; v < nvec; v += kGatherThreads) dv[v] = __ldg(sv + v);
        } else if (sh == 0) {
            for (uint32_t v = t; v < nvec; v += kGatherThreads) {
                const uint32_t* q = sw + 4 * v;
                dv[v] = make_uint4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3));
            }
        } else {
            for (uint32_t v = t; v < nvec; v += kGatherThreads) {
                const uint32_t* q = sw + 4 * v;
                uint32_t x0 = __ldg(q), x1 = __ldg(q + 1), x2 = __ldg(q + 2), x3 = __ldg(q + 3), x4 = __ldg(q + 4);
                dv[v] = make_uint4(__funnelshift_r(x0, x1, sh), __funnelshift_r(x1, x2, sh),
                                   __funnelshift_r(x2, x3, sh), __funnelshift_r(x3, x4, sh));
            }
        }
        const uint32_t done = nvec << 4, tail = n - done;
        if (t < tail) dst[done + t] = __ldg(src + done + t);
    }
}

// resizeChunksD's `process` (src/Streamly/Internal/LZ4.hs:459-484) over a stream resident in HBM: a dependent chain of
// one 4-byte load per block, so one thread walks it (O(#blocks); 13 422 blocks of config 3 take a few milliseconds).
__global__ void reframe_kernel(const uint8_t* __restrict__ buf, long long len, int header, int has_end_mark,
                               int64_t* __restrict__ block_off, int32_t* __restrict__ block_len, long long max_blocks,
                               int64_t* __restrict__ result)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    long long at = 0, k = 0, ended = 0, bad = 0;
    while (k < max_blocks) {
        const long long rest = len - at;
        if (rest < 4) break;                                            // LZ4.hs:461-462
        const uint8_t* p = buf + at;
        const int comp = (int)((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24));
        if (has_end_mark && comp == 0) { at += 4; ended = 1; break; }   // LZ4.hs:464-466
        if (rest <= header) break;                                      // LZ4.hs:468-469
        if (comp <= 0) { bad = 1; break; }
        const long long required = (long long)comp + header;            // LZ4.hs:474
        if (rest < required) break;                                     // LZ4.hs:477-478
        block_off[k] = at; block_len[k] = (int32_t)required;
        k++; at += required;
    }
    result[0] = k; result[1] = at; result[2] = ended; result[3] = bad;
}

}  // namespace

cudaError_t launch_reframe(const uint8_t* buf, int64_t len, int header, int has_end_mark,
                           int64_t* block_off, int32_t* block_len, int64_t max_blocks, int64_t* result, cudaStream_t stream)
{
    reframe_kernel<<<1, 32, 0, stream>>>(buf, (long long)len, header, has_end_mark, block_off, block_len, (long long)max_blocks, result);
    return cudaGetLastError();
}

cudaError_t launch_compact(const CompactArgs& a, cudaStream_t stream)
{
    int sm_count = 0;
    cudaError_t e0 = device_sm_count(&sm_count); if (e0 != cudaSuccess) return e0;
    scan_kernel<<<1, kScanThreads, 0, stream>>>(a.len, a.n_blocks, a.header, a.out_off, a.host_off, a.host_len);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || a.n_blocks <= 0) return e;
    int grid = a.n_blocks < sm_count * 8 ? a.n_blocks : sm_count * 8;
    gather_kernel<<<grid, kGatherThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_scan(const int32_t* len, int n, int header, int64_t* out_off, cudaStream_t stream)
{
    scan_kernel<<<1, kScanThreads, 0, stream>>>(len, n, header, out_off, nullptr, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_gather(const CompactArgs& a, cudaStream_t stream)
{
    if (a.n_blocks <= 0) return cudaSuccess;
    int sm_count = 0;
    cudaError_t e = device_sm_count(&sm_count); if (e != cudaSuccess) return e;
    gather_kernel<<<a.n_blocks < sm_count * 8 ? a.n_blocks : sm_count * 8, kGatherThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

// Loads the compaction kernels now (CUDA loads a kernel lazily at its first launch, which can wait for running kernels
// to end -- the streamed call must never launch anything for the first time while its finders wait for input).
cudaError_t preload_compact_kernels()
{
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, scan_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, gather_kernel);
    return e;
}

int kernel_launches_per_compress() { return 1; }
int kernel_launches_per_decompress() { return 1; }
int kernel_launches_per_compact() { return 2; }

}  // namespace b200lz4
