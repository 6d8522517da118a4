// common.cuh -- shared device helpers and layouts of the B200 LZ4 block codec.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200lz4 {

constexpr uint32_t kFull = 0xFFFFFFFFu;
constexpr int kHashEntries = 4096;          // LZ4_HASH_SIZE_U32 (cbits/lz4.h:578-580)
constexpr uint32_t kMaxDistance = 65535u;   // LZ4_DISTANCE_MAX (cbits/lz4.h:556-558)
constexpr int kMaxInput = 0x7E000000;       // LZ4_MAX_INPUT_SIZE
constexpr int kMinMatch = 4, kLastLiterals = 5, kMfLimit = 12, kMinLength = 13;
constexpr int kAccelMax = 65537;            // LZ4_ACCELERATION_MAX (cbits/lz4.c:57)

// Device-resident equivalent of LZ4_stream_t_internal (cbits/lz4.h:595-603).  The kernels copy the table with 16-byte
// accesses, so records must be 16-byte aligned; the padded size keeps records packed at stride b200lz4_cstate_bytes()
// aligned too.
struct alignas(16) CState {
    uint32_t table[kHashEntries];   // stream positions (byU32)
    uint32_t offset;                // currentOffset
    uint32_t dict_len;              // dictSize: full length of the previous array
    uint32_t dict_cap;              // capacity of dict_buf
    uint32_t pad_;
    uint8_t* dict_buf;              // previous array (dict_len bytes), owned by the caller
};

// Device-resident equivalent of LZ4_streamDecode_t_internal (cbits/lz4.h:605-610):
// only the last 64 KiB of the previous output are reachable (offset <= 65535), plus
// its true length for the checkOffset rule (cbits/lz4.c:1764, :2073).
struct DState {
    uint32_t prev_len;              // prefixSize of the previous block (0 = no dictionary yet)
    uint32_t kept;                  // min(prev_len, 65536) bytes, right-aligned in tail[]
    uint32_t pad_[2];
    uint8_t tail[65536];
};
static_assert(sizeof(CState) % 16 == 0 && sizeof(DState) % 16 == 0, "state records packed back to back stay 16-byte aligned");

// Zero-filled once by the caller; kernels leave it zeroed.  Each kernel that hands out streams through a work counter owns
// one pair (claim counter, CTAs done): the compress kernels 0/1, the narrow decoder 2/3.
struct Scratch {
    uint32_t work_counter[4];
    uint32_t pad_[60];
};

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt()
{ uint32_t m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

// ---- work distribution over a Scratch counter pair ------------------------
// next stream for this warp (all lanes call): lane 0 draws it from the claim counter
__device__ __forceinline__ int claim_stream(uint32_t* counter)
{
    int s = 0;
    if (lane_id() == 0) s = (int)atomicAdd(counter, 1u);
    return __shfl_sync(kFull, s, 0);
}
// all threads of the CTA call it at the end: the last CTA out resets counter pair `first` so that the scratch stays
// zeroed for the next launch
__device__ __forceinline__ void release_counters(Scratch* scratch, int first)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t done = atomicAdd(&scratch->work_counter[first + 1], 1u);
        if (done == gridDim.x - 1) { scratch->work_counter[first] = 0; scratch->work_counter[first + 1] = 0; __threadfence(); }
    }
}

// ---- shared memory, cp.async, mbarriers -----------------------------------
// All shared-memory accesses of the kernels' hot loops use explicit 32-bit shared-space addresses.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint4 lds128(uint32_t a)
{ uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{ asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory"); }

// cp_async_4 caches in L1 (.ca: the compress finder's input lines, re-read by neighbouring probes); cp_async_16 bypasses
// it (.cg: the decoders' compressed payload, read once)
__device__ __forceinline__ void cp_async_4(uint32_t smem_addr, const void* g)
{ asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(g) : "memory"); }
__device__ __forceinline__ void cp_async_16(uint32_t smem_addr, const void* g)
{ asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(g) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count)
{ asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar)
{ asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
// one attempt to wait for the phase of the given parity on the mbarrier at shared address bar_s, suspended in hardware
// for up to about suspend_ns (a waiting warp does not burn issue slots); true once the phase has completed
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar_s, uint32_t parity, uint32_t suspend_ns)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(bar_s), "r"(parity), "r"(suspend_ns) : "memory");
    return ok != 0;
}
// waits for the phase (loops inside the asm, with a 20 us suspend hint)
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
}
// the same test without a suspend hint: returns after the hardware's own short time limit (the caller sleeps in between)
__device__ __forceinline__ bool mbar_test(unsigned long long* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}

// ---- global memory: system-scope flags, L2 prefetch -------------------------
// a flag word written by the host or another stream (acquire: what it announces is visible once it is seen)
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p)
{ uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes)
{ asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory"); }

// ---- unaligned little-endian reads through the read-only path ------------
// 4 bytes at p; touches only the aligned words that contain p[0..3].
__device__ __forceinline__ uint32_t ldg_u32_unaligned(const uint8_t* p)
{
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t w0 = __ldg(w);
    uint32_t w1 = sh ? __ldg(w + 1) : 0u;
    return __funnelshift_r(w0, w1, sh);
}
// 5 bytes at p: low 4 in .x, fifth byte in .y (always spans exactly two aligned words)
__device__ __forceinline__ uint2 ldg_5bytes(const uint8_t* p)
{
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t w0 = __ldg(w), w1 = __ldg(w + 1);
    return make_uint2(__funnelshift_r(w0, w1, sh), (w1 >> sh) & 0xFFu);
}
// same, coherent loads (for memory this kernel also writes)
__device__ __forceinline__ uint32_t ld_u32_unaligned(const uint8_t* p)
{
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t w0 = w[0];
    uint32_t w1 = sh ? w[1] : 0u;
    return __funnelshift_r(w0, w1, sh);
}

// LZ4_hash5 on a little-endian 64-bit target (cbits/lz4.c:706-716): only the low
// 5 bytes of the 8 the reference reads reach the result.
// ((five << 24) * P) >> 52 == bits 28..39 of (five * P) mod 2^40, evaluated with 32-bit
// multiplies: P = 0xCF_1BBCDCBB, five = lo4 + b4 * 2^32.
__device__ __forceinline__ uint32_t hash5(uint32_t lo4, uint32_t b4)
{
    constexpr uint32_t kPl = 0x1BBCDCBBu, kPh = 0xCFu;
    const uint32_t tl = lo4 * kPl;
    const uint32_t th = __umulhi(lo4, kPl) + lo4 * kPh + b4 * kPl;
    return (tl >> 28) | ((th & 0xFFu) << 4);
}

// ---- cache-policy helpers ---------------------------------------------------
// Streaming reads/writes of the emitter and of far probe lanes must not evict the few KiB of
// L1 that serve the match finder's current lines.
__device__ __forceinline__ uint32_t ldg_na_u32(const uint32_t* p)
{ uint32_t v; asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint32_t ldg_na_u8(const uint8_t* p)
{ uint32_t v; asm volatile("ld.global.nc.L1::no_allocate.u8 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint4 ldg_na_u128(const uint4* p)
{ uint4 v; asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p)); return v; }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// ---- warp-cooperative copies ----------------------------------------------
// dst/src arbitrary alignment, non-overlapping, src read-only for the kernel.
// All 32 lanes must call with identical arguments.
__device__ __forceinline__ void warp_copy_ro(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t len)
{
    const uint32_t lane = lane_id();
    if (len < 96) {
        for (uint32_t i = lane; i < len; i += 32) dst[i] = (uint8_t)ldg_na_u8(src + i);
        return;
    }
    // head: bring dst to 16-byte alignment
    uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
    if (lane < head) dst[lane] = (uint8_t)ldg_na_u8(src + lane);
    dst += head; src += head; len -= head;
    const uint32_t nvec = len >> 4;
    uintptr_t sa = reinterpret_cast<uintptr_t>(src);
    const uint32_t sh = (uint32_t)(sa & 3) * 8;
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t(3));
    uint4* dv = reinterpret_cast<uint4*>(dst);
    if (sh == 0) {
        if ((sa & 15) == 0) {
            const uint4* sv = reinterpret_cast<const uint4*>(src);
            for (uint32_t v = lane; v < nvec; v += 32) dv[v] = ldg_na_u128(sv + v);
        } else {
            for (uint32_t v = lane; v < nvec; v += 32) {
                const uint32_t* q = sw + 4 * v;
                dv[v] = make_uint4(ldg_na_u32(q), ldg_na_u32(q + 1), ldg_na_u32(q + 2), ldg_na_u32(q + 3));
            }
        }
    } else {
        for (uint32_t v = lane; v < nvec; v += 32) {
            const uint32_t* q = sw + 4 * v;
            uint32_t a = ldg_na_u32(q), b = ldg_na_u32(q + 1), c = ldg_na_u32(q + 2), d = ldg_na_u32(q + 3), e = ldg_na_u32(q + 4);
            dv[v] = make_uint4(__funnelshift_r(a, b, sh), __funnelshift_r(b, c, sh),
                               __funnelshift_r(c, d, sh), __funnelshift_r(d, e, sh));
        }
    }
    const uint32_t done = nvec << 4;
    const uint32_t tail = len - done;
    if (lane < tail) dst[done + lane] = (uint8_t)ldg_na_u8(src + done + lane);
}

}  // namespace b200lz4
