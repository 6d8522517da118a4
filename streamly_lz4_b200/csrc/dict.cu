// dict.cu -- LZ4_loadDict / LZ4_setStreamDecode on the device: the read-only state records a batch's streams start from
// when they share a dictionary (CompressArgs::dict_state, DecompressArgs::dict_state).
//
// LZ4_loadDict (lz4.c 1.9.3/1.9.4) resets the stream, sets currentOffset = 64 KiB, and -- unless the dictionary is shorter
// than HASH_UNIT (8 bytes on a 64-bit target), in which case it stops there with dictSize 0 -- inserts positions
// p = start, start + 3, ... while p <= end - 8 of the last min(len, 64 KiB) bytes with index 65536 - (end - p); a later
// position overwrites an earlier one in the same bucket.  Positions only grow, so "last writer wins" is atomicMax.
#include "common.cuh"
#include "kernels.h"

namespace b200lz4 {

namespace {

constexpr int kLoadThreads = 1024;
constexpr uint32_t kHashUnit = 8;

__global__ void __launch_bounds__(kLoadThreads, 1)
load_dict_kernel(const uint8_t* dict, int64_t len, CState* cs, DState* ds)
{
    __shared__ uint32_t table[kHashEntries];
    const uint32_t kept = len < 65536 ? (uint32_t)len : 65536u;
    const uint8_t* const start = dict + (len - kept);
    if (cs) {
        for (int i = threadIdx.x; i < kHashEntries; i += blockDim.x) table[i] = 0u;
        __syncthreads();
        if (kept >= kHashUnit) {
            const uint32_t n_pos = (kept - kHashUnit) / 3 + 1;             // p = 3k <= kept - 8
            for (uint32_t k = threadIdx.x; k < n_pos; k += blockDim.x) {
                const uint8_t* p = start + 3 * k;
                const uint32_t lo4 = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
                atomicMax(&table[hash5(lo4, p[4])], 65536u - (kept - 3 * k));
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < kHashEntries; i += blockDim.x) cs->table[i] = table[i];
        if (threadIdx.x == 0) {
            const uint32_t dict_len = kept >= kHashUnit ? kept : 0u;
            cs->offset = 65536u; cs->dict_len = dict_len; cs->dict_cap = dict_len; cs->pad_ = 0u;
            cs->dict_buf = const_cast<uint8_t*>(dict + (len - dict_len));
        }
    }
    if (ds) {       // the decoder reads the dictionary whatever its length; prev_len drives the checkOffset rule
        for (uint32_t i = threadIdx.x; i < kept; i += blockDim.x) ds->tail[65536u - kept + i] = start[i];
        if (threadIdx.x == 0) {
            ds->prev_len = (uint32_t)len; ds->kept = kept; ds->pad_[0] = 0u; ds->pad_[1] = 0u;
        }
    }
}

}  // namespace

cudaError_t launch_load_dict(const uint8_t* dict, int64_t len, CState* d_cstate, DState* d_dstate, cudaStream_t stream)
{
    if (!d_cstate && !d_dstate) return cudaSuccess;
    load_dict_kernel<<<1, kLoadThreads, 0, stream>>>(dict, len, d_cstate, d_dstate);
    return cudaGetLastError();
}

}  // namespace b200lz4
