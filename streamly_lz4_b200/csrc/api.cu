// api.cu -- the C ABI of libb200lz4.so (see include/b200lz4.h): contexts, staging,
// the batched host/device entry points, re-framing and the legacy LZ4_* aliases.
// There is no CPU codec in this library: every compress/decompress call runs the
// sm_100a kernels, and fails with B200LZ4_E_CUDA when no such device is usable.
// What the host batch calls decide before they touch the device is in host_plan.h.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <chrono>
#include <vector>

#include "b200lz4.h"
#include "host_plan.h"
#include "kernels.h"

using namespace b200lz4;
using namespace hostplan;
static_assert(kMaxInputSize == kMaxInput, "host_plan.h restates LZ4_MAX_INPUT_SIZE");

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int fail_cuda(cudaError_t e, const char* what)
{
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return B200LZ4_E_CUDA;
}
#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail_cuda(e__, #call); } while (0)

// grow-only buffer in device memory, or (kPinned) in page-locked host memory the device can see: kernels mirror sizes into it
template <bool kPinned>
struct Buf {
    void* p = nullptr; size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        release();
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = kPinned ? cudaHostAlloc(&p, want, cudaHostAllocMapped | cudaHostAllocPortable) : cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(B200LZ4_E_NOMEM, std::string(kPinned ? "cudaHostAlloc: " : "cudaMalloc: ") + cudaGetErrorString(e)); }
        cap = want;
        return 0;
    }
    void release() { if (p) { if (kPinned) cudaFreeHost(p); else cudaFree(p); } p = nullptr; cap = 0; }
};

// the device timeline of one host batch call
struct CallEvents {
    cudaEvent_t start = nullptr, h2d_end = nullptr;         // H2D stream: before the call's first and after its last copy
    cudaEvent_t k0 = nullptr;                               // before the first kernel
    cudaEvent_t d0 = nullptr, d1 = nullptr;                 // D2H stream: t_d2h
    cudaEvent_t h2d[kMaxGroups] = {}, k[kMaxGroups] = {};   // per chunk / group: its kernels may start; its kernels are done
    template <class F> void each(F f)
    {
        for (cudaEvent_t* e : {&start, &h2d_end, &k0, &d0, &d1}) f(*e);
        for (auto& e : h2d) f(e);
        for (auto& e : k) f(e);
    }
};

}  // namespace

constexpr int kKernelStreams = kMaxChunks;   // one stream per chunk: chunk kernels must be able to overlap
constexpr size_t kFlagBytes = 1024 + kMaxGroups * kMaxSegs * sizeof(uint32_t);   // ctx->d_flags: see b200lz4_ctx

struct b200lz4_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;                  // H2D + bookkeeping
    cudaStream_t kstream[kKernelStreams] = {};      // chunk kernels (run concurrently)
    cudaStream_t dstream = nullptr;                 // D2H
    Scratch* scratch = nullptr;                     // kMaxGroups records: one work counter per in-flight kernel
    Buf<false> d_src, d_slots, d_out, d_desc, d_wide;   // d_wide: descriptor rings of decompress_kernel_wide (one slice per chunk)
    Buf<true> h_desc;
    CallEvents ev;
    // streamed compress call (compress_host_streamed): per-group arrival flags + finder cycle counters in HBM, the
    // constants the copy stream writes into the flags, and what earlier calls measured (the copy schedule is tuned by it)
    uint32_t* d_flags = nullptr;            // [kMaxGroups] u32 flags, then at byte 64: u64 busy cycles, u64 bytes; at byte 1024:
                                            // [kMaxGroups][kMaxSegs] u32 segment counters of the streamed decompress call
    uint32_t* h_const = nullptr;            // pinned: h_const[i] == i
    double est_ns_per_byte = 0;             // finder time per input byte (0 = not measured yet)
    double est_h2d_gbs = 0;                 // H2D bandwidth of the last streamed call
    int clock_khz = 0;
    int streamed_calls = 0;
    cudaStream_t fstream = nullptr;         // arrival flags are raised from here (set_flag kernels behind per-piece events), so that
                                            // the copy stream's pieces run back to back
    std::vector<cudaEvent_t> ev_piece;
    int n_kgood = -1;                       // kernel streams verified not to share a hardware queue with the copy streams
                                            // or with each other (-1: not probed yet); they come first in kstream[]
    float t_h2d = 0, t_kernel = 0, t_d2h = 0;
    int64_t launches = 0;
    std::string err;                                // text of the last failure of a call on this ctx (any thread)
};

struct b200lz4_cstream {
    b200lz4_ctx* ctx; CState* d_state; uint8_t* d_dict; uint32_t dict_cap; uint32_t last_len;
};
struct b200lz4_dstream {
    b200lz4_ctx* ctx; DState* d_state;
};
// a loaded dictionary: its bytes in HBM and the state records LZ4_loadDict / LZ4_setStreamDecode make of them
struct b200lz4_dict {
    b200lz4_ctx* ctx; uint8_t* d_bytes; int64_t len; CState* d_cstate; DState* d_dstate;
};

namespace {

int fail(const Verdict& v) { return fail(v.code, v.msg); }

int set_dict_fields(CState* d_state, uint8_t* buf, uint32_t cap, cudaStream_t st)
{
    struct { uint32_t dict_cap; uint32_t pad; uint8_t* dict_buf; } f{cap, 0, buf};
    static_assert(offsetof(CState, dict_buf) == offsetof(CState, dict_cap) + 8, "CState layout");
    CU(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(d_state) + offsetof(CState, dict_cap), &f, sizeof f, cudaMemcpyHostToDevice, st));
    return 0;
}

// grow a stream's previous-array buffer, preserving its content
int cstream_reserve(b200lz4_cstream* s, uint32_t need)
{
    if (need <= s->dict_cap) return 0;
    b200lz4_ctx* c = s->ctx;
    uint32_t cap = need < 65536u ? 65536u : need;
    uint8_t* nb = nullptr;
    cudaError_t e = cudaMalloc(&nb, (size_t)cap + 16);
    if (e != cudaSuccess) return fail(B200LZ4_E_NOMEM, std::string("cudaMalloc(dict): ") + cudaGetErrorString(e));
    if (s->d_dict && s->last_len) CU(cudaMemcpyAsync(nb, s->d_dict, s->last_len, cudaMemcpyDeviceToDevice, c->stream));
    int rc = set_dict_fields(s->d_state, nb, cap, c->stream);
    if (rc) { cudaFree(nb); return rc; }
    CU(cudaStreamSynchronize(c->stream));
    if (s->d_dict) cudaFree(s->d_dict);
    s->d_dict = nb; s->dict_cap = cap;
    return 0;
}

int sync_all(b200lz4_ctx* c)
{
    CU(cudaStreamSynchronize(c->stream));
    for (auto& k : c->kstream) CU(cudaStreamSynchronize(k));
    CU(cudaStreamSynchronize(c->dstream));
    if (c->fstream) CU(cudaStreamSynchronize(c->fstream));
    return 0;
}

// ---- hardware-queue aliasing ---------------------------------------------------
// CUDA multiplexes streams onto CUDA_DEVICE_MAX_CONNECTIONS hardware work queues (8 unless the variable is set before the
// context exists; the library's load-time constructor below asks for 32).  Entries of one queue are dispatched in order, so
// anything queued behind a kernel's same-stream successor waits for that kernel to END -- harmless for the plain pipeline,
// fatal for the streamed call, whose kernels wait for copies that are queued later on the copy stream.  Which streams share
// a queue is not documented, so it is MEASURED once per ctx: a kernel that spins on a flag (bounded by a timeout), a
// successor behind it, then a write of the flag through the other stream; if the spinning kernel times out, the two
// streams share a queue.  Kernel streams that alias the H2D stream, the D2H stream or an already accepted kernel stream are
// replaced by fresh ones (up to 40 tries).
__attribute__((constructor)) void ask_for_more_hardware_queues() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }
// (CUDA_MODULE_LOADING is deliberately left alone: probe_stream_aliasing loads the few kernels that matter by hand.)

int streams_alias(b200lz4_ctx* c, cudaStream_t spinner, cudaStream_t other, bool other_writes_by_kernel, bool* aliased)
{
    uint32_t* flag = c->d_flags + 40;       // bytes 160.. of the flag block: not used by the calls themselves
    uint32_t* result = c->d_flags + 44;
    CU(cudaMemsetAsync(flag, 0, 32, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CU(launch_alias_probe(flag, result, (long long)c->clock_khz * 15, spinner));     // 15 ms
    if (other_writes_by_kernel) CU(launch_set_flag(flag, 1u, other));
    else CU(cudaMemcpyAsync(flag, c->h_const + 1, sizeof(uint32_t), cudaMemcpyHostToDevice, other));
    CU(cudaStreamSynchronize(spinner));
    CU(cudaStreamSynchronize(other));
    uint32_t r[2] = {0, 0};
    CU(cudaMemcpy(r, result, sizeof r, cudaMemcpyDeviceToHost));
    *aliased = (r[0] != 1u);
    return 0;
}

int probe_stream_aliasing(b200lz4_ctx* c)
{
    if (c->n_kgood >= 0) return 0;
    // every kernel a streamed call launches is loaded NOW: a lazy first-time load in the middle of the call waits for
    // running kernels to end, and those wait for copies the blocked host thread has not queued yet
    CU(preload_compress_kernels());
    CU(preload_compact_kernels());
    {   // ... including whatever the runtime itself uses for memset and small copies: run each once
        CU(cudaMemsetAsync(c->d_flags, 0, kFlagBytes, c->stream));
        CU(cudaMemcpyAsync(c->d_flags + 48, c->h_const + 1, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        CU(launch_set_flag(c->d_flags + 48, 0u, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    std::vector<cudaStream_t> good, rejected;
    int next_existing = 0, tries = 0, rc;
    while ((int)good.size() < kKernelStreams && tries < 40) {
        cudaStream_t cand;
        if (next_existing < kKernelStreams) cand = c->kstream[next_existing++];
        else CU(cudaStreamCreateWithFlags(&cand, cudaStreamNonBlocking));
        tries++;
        bool bad = false;
        if ((rc = streams_alias(c, cand, c->stream, false, &bad))) return rc;
        if (!bad && (rc = streams_alias(c, cand, c->dstream, false, &bad))) return rc;
        for (size_t j = 0; j < good.size() && !bad; j++) if ((rc = streams_alias(c, good[j], cand, true, &bad))) return rc;
        (bad ? rejected : good).push_back(cand);
    }
    while (next_existing < kKernelStreams) rejected.push_back(c->kstream[next_existing++]);
    // the flag stream must not sit behind a waiting kernel either
    for (int t = 0; t < 16 && !c->fstream; t++) {
        cudaStream_t cand;
        CU(cudaStreamCreateWithFlags(&cand, cudaStreamNonBlocking));
        bool bad = false;
        for (size_t j = 0; j < good.size() && !bad; j++) if ((rc = streams_alias(c, good[j], cand, true, &bad))) return rc;
        if (bad) cudaStreamDestroy(cand); else c->fstream = cand;
    }
    c->n_kgood = (int)good.size();
    int k = 0;
    for (cudaStream_t x : good) c->kstream[k++] = x;
    for (cudaStream_t x : rejected) { if (k < kKernelStreams) c->kstream[k++] = x; else cudaStreamDestroy(x); }
    if (getenv("B200LZ4_DEBUG")) fprintf(stderr, "[b200lz4] hardware queues: %d of %d kernel streams independent of the copy streams after %d tries\n", c->n_kgood, kKernelStreams, tries);
    return 0;
}

// ---- shared steps of the host pipelines ------------------------------------------------------------------------------
// A plain host batch is cut into up to kMaxChunks chunks of whole streams (independent mode: whole blocks, host_plan.h:
// plan_chunks).  Chunk k's H2D copy, its kernels and its D2H copy run on three different CUDA streams, so that transfers
// in both directions overlap the kernels of neighbouring chunks; the chunk kernels themselves run concurrently on
// kKernelStreams streams because a codec kernel is bound by per-block latency, not by the number of blocks it is given.
// The streamed calls cut the batch into groups instead, and blocks into segments.

int ensure_desc(b200lz4_ctx* c, const DescLayout& lay)
{
    const int rc = c->h_desc.ensure(lay.bytes);
    return rc ? rc : c->d_desc.ensure(lay.bytes);
}

// Range k (chunk or group): H2D copy of its source bytes (none for an empty span), then its kernels go to ks behind it
int start_range(b200lz4_ctx* c, int k, cudaStream_t ks, Span span, uint8_t* d_src, const uint8_t* hsrc)
{
    if (span.hi > span.lo) CU(cudaMemcpyAsync(d_src + span.lo, hsrc + span.lo, (size_t)(span.hi - span.lo), cudaMemcpyHostToDevice, c->stream));
    CU(cudaEventRecord(c->ev.h2d[k], c->stream));
    CU(cudaStreamWaitEvent(ks, c->ev.h2d[k], 0));
    if (k == 0) CU(cudaEventRecord(c->ev.k0, ks));
    return 0;
}

// the kernel arguments every host pipeline fills alike: the batch's descriptors in d_desc, the launch's units of range r
template <class Args>
Args launch_args(const DescLayout& lay, void* dd, const uint8_t* d_src, uint8_t* d_slots, int n, int header, const Range& r,
                 Scratch* scratch, bool linked, bool states)
{
    Args a{};
    a.src = d_src; a.src_off = lay.src_off_in(dd); a.src_len = lay.src_len_in(dd); a.n_blocks = n;
    a.first_block = r.b0; a.n_streams = r.u1 - r.u0;
    a.stream_first = linked ? lay.first_in(dd) + r.u0 : nullptr;
    a.states = states ? lay.states_in(dd) + r.u0 : nullptr;
    a.dst = d_slots; a.dst_off = lay.slot_off_in(dd); a.out_len = lay.out_len_in(dd);
    a.header = header; a.scratch = scratch;
    return a;
}

// Compress range k, then pack its blocks behind each other in d_out: the scan kernel mirrors sizes and offsets into the
// pinned descriptor block (device-visible host memory), range k's n_k + 1 offsets from entry b0 + k of out_off.
int compress_range(b200lz4_ctx* c, const CompressArgs& a, const DescLayout& lay, const Range& r, int k, uint8_t* d_out, cudaStream_t ks)
{
    void* hd = c->h_desc.p;
    CU(launch_compress(a, ks));
    CompactArgs g{a.dst, a.dst_off + r.b0, a.out_len + r.b0, r.b1 - r.b0, a.header, d_out + lay.slot_off_in(hd)[r.b0],
                  lay.out_off_in(c->d_desc.p) + r.b0 + k, lay.out_off_in(hd) + r.b0 + k, lay.out_len_in(hd) + r.b0};
    CU(launch_compact(g, ks));
    c->launches += kernel_launches_per_compress() + kernel_launches_per_compact();
    CU(cudaEventRecord(c->ev.k[k], ks));
    return 0;
}

// As each range's kernels finish, its compacted bytes go home behind those of the ranges before it
int drain_compacted(b200lz4_ctx* c, const Range* r, int nr, const DescLayout& lay, const uint8_t* d_out,
                    void* dst, int64_t dst_cap, int64_t* dst_off, int n, bool log)
{
    const int64_t* h_out_off = lay.out_off_in(c->h_desc.p);
    const int64_t* h_slot_off = lay.slot_off_in(c->h_desc.p);
    int64_t base = 0;
    int rc = 0;
    for (int k = 0; k < nr; k++) {
        CU(cudaEventSynchronize(c->ev.k[k]));
        if (log) { fprintf(stderr, "[b200lz4] streamed: group %d done\n", k); fflush(stderr); }
        const int nk = r[k].b1 - r[k].b0;
        const int64_t* off_k = h_out_off + r[k].b0 + k;
        const int64_t total_k = off_k[nk];
        for (int i = 0; i < nk; i++) dst_off[r[k].b0 + i] = base + off_k[i];
        if (base + total_k > dst_cap) { rc = fail(B200LZ4_E_NOMEM, "dst_cap too small"); break; }
        if (total_k) CU(cudaMemcpyAsync(static_cast<uint8_t*>(dst) + base, d_out + h_slot_off[r[k].b0], (size_t)total_k,
                                        cudaMemcpyDeviceToHost, c->dstream));
        base += total_k;
    }
    dst_off[n] = base;
    return rc;
}

// Segment s of every block of group grp as one pitched copy (block i at dst + i * dpitch and src + i * spitch), queued
// after a copy of its own of the share of a short last block (last_len < L).  The copy engine moves a pitched copy row by
// row: measured 9 % slower than one plain copy of the same bytes on an idle link and 15 % slower while the opposite
// direction is busy, which is why segments are not made smaller than they have to be.
int copy_piece(uint8_t* dst, size_t dpitch, const uint8_t* src, size_t spitch, const Geometry& geo, const Range& grp,
               int n, int L, int last_len, int s, cudaMemcpyKind kind, cudaStream_t st)
{
    const int lo = s * geo.seg, width = std::min(geo.seg, L - lo);
    int rows = grp.b1 - grp.b0;
    if (grp.b1 == n && last_len < L) {
        rows--;
        const int wl = std::min(width, last_len - lo);
        if (wl > 0) CU(cudaMemcpyAsync(dst + dpitch * (n - 1) + lo, src + spitch * (n - 1) + lo, (size_t)wl, kind, st));
    }
    if (rows <= 0) return 0;
    dst += dpitch * grp.b0 + lo;
    src += spitch * grp.b0 + lo;
    if (rows == 1 || ((size_t)width == dpitch && (size_t)width == spitch)) CU(cudaMemcpyAsync(dst, src, (size_t)width * rows, kind, st));
    else CU(cudaMemcpy2DAsync(dst, dpitch, src, spitch, (size_t)width, (size_t)rows, kind, st));
    return 0;
}

// Every host pipeline ends here once it has queued work, failed (rc) or not, so that nothing it queued is left running on
// the ctx's streams.  Then the timing split, the block sizes, the device timeline of its ranges (B200LZ4_DEBUG; label
// NULL: none) and the per-block check: a compressed block failed with a size <= 0, a decompressed one with a size < 0.
int finish_call(b200lz4_ctx* c, int rc, const Range* r, int nr, const char* label, const char* landed,
                const int32_t* h_out_len, int32_t* out_len, int n, bool decode)
{
    const cudaError_t e = cudaEventRecord(c->ev.d1, c->dstream);
    if (e != cudaSuccess && !rc) rc = fail_cuda(e, "cudaEventRecord(ev.d1)");
    if (const int s = sync_all(c)) return s;
    if (rc) return rc;
    cudaEventElapsedTime(&c->t_h2d, c->ev.start, c->ev.h2d_end);
    cudaEventElapsedTime(&c->t_kernel, c->ev.k0, c->ev.k[nr - 1]);
    cudaEventElapsedTime(&c->t_d2h, c->ev.d0, c->ev.d1);
    memcpy(out_len, h_out_len, sizeof(int32_t) * n);
    if (label && getenv("B200LZ4_DEBUG")) {         // ms since the call's first event
        float t = 0;
        for (int k = 0; k < nr; k++) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, c->ev.start, c->ev.h2d[k]); cudaEventElapsedTime(&b, c->ev.start, c->ev.k[k]);
            fprintf(stderr, "[b200lz4] %s %d: blocks %d..%d  %s %.2f  kernels done %.2f\n", label, k, r[k].b0, r[k].b1, landed, a, b);
        }
        cudaEventElapsedTime(&t, c->ev.start, c->ev.h2d_end); fprintf(stderr, "[b200lz4] h2d done %.2f\n", t);
        cudaEventElapsedTime(&t, c->ev.start, c->ev.d1); fprintf(stderr, "[b200lz4] d2h done %.2f\n", t);
    }
    for (int i = 0; i < n; i++)
        if (decode ? out_len[i] < 0 : out_len[i] <= 0)
            return fail(B200LZ4_E_BLOCK, "block " + std::to_string(i) + (decode ? " failed to decompress" : " failed to compress"));
    return 0;
}

// ---- streamed compress call ---------------------------------------------------
// A batch of equally long independent blocks at a constant pitch (what compressChunks over fixed-size reads produces)
// does not have to arrive block by block.  The end of the plain pipeline above is "last byte lands + one BLOCK latency"
// (a 640 000-byte block keeps one finder busy for ~7 ms, a third of the whole transfer).  Here blocks are cut into S
// segments and block groups into 2-D copies (one segment of every block of a group per copy), each followed by a 4-byte
// copy that bumps the group's arrival flag; the group's kernel is launched as soon as its FIRST segment has landed and
// its finders wait for later segments only if they get there before the data (compress.cu: kStreamed).  Pieces are sent
// in deadline order (host_plan.h: piece_order), with w chosen so that a group's segments arrive at the pace its finders
// consume them, from what the previous streamed call on this ctx measured (finder cycles per byte, H2D rate); then the
// end of the call is "last byte lands + one SEGMENT latency + the last group's D2H".  The device layout is private to the
// call (128-byte aligned block starts, 128 bytes of gap), so no L1 sector is read before it is complete.
constexpr int kStreamedGaveUp = -1000;  // internal: compress_host retries through the plain pipeline

int compress_host_streamed(b200lz4_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, int n,
                           const StreamShape& shp, int accel, int header, const CState* dict_state,
                           void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    int rc;
    const int L = shp.L;
    const int nks = c->n_kgood;             // kernel streams that cannot block the copy stream (>= 2, checked by the caller)
    const int64_t DP = ((int64_t)L + 127) / 128 * 128 + 128;       // device pitch
    const int64_t total = total_bytes(src_len, n);
    const char* env_f = getenv("B200LZ4_STREAM_FLAG");      // measurement overrides (read per call)
    const bool flag_by_kernel = env_f && env_f[0] == 'k';
    const bool flag_inline_copy = env_f && env_f[0] == 'c';
    const bool flag_separate = !flag_by_kernel && !flag_inline_copy && c->fstream != nullptr;
    const Geometry geo = compress_geometry(n, L, total, nks, c->est_ns_per_byte, c->est_h2d_gbs, getenv("B200LZ4_STREAM_G"),
                                           getenv("B200LZ4_STREAM_S"), getenv("B200LZ4_STREAM_W"));
    Range groups[kMaxGroups];
    plan_groups(geo, n, groups);

    const DescLayout lay(n, n, 0, 0, 0, n + geo.G, 0);
    if ((rc = ensure_desc(c, lay))) return rc;
    void* hd = c->h_desc.p;
    void* dd = c->d_desc.p;
    int64_t* h_src_off = lay.src_off_in(hd);
    int64_t* h_slot_off = lay.slot_off_in(hd);
    memcpy(lay.src_len_in(hd), src_len, sizeof(int32_t) * n);
    int64_t slots_total = 0;
    for (int i = 0; i < n; i++) {
        h_src_off[i] = DP * i;
        h_slot_off[i] = slots_total;
        slots_total += compress_slot(compress_cap(src_len[i], header));
    }
    if ((rc = c->d_src.ensure((size_t)(DP * n) + 256))) return rc;
    if ((rc = c->d_slots.ensure((size_t)slots_total + 64))) return rc;
    if ((rc = c->d_out.ensure((size_t)slots_total + 64))) return rc;
    const uint8_t* hsrc = static_cast<const uint8_t*>(src);
    uint8_t* d_src = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(c->d_src.p) + 127) & ~uintptr_t(127));
    uint8_t* d_slots = static_cast<uint8_t*>(c->d_slots.p);
    uint8_t* d_out = static_cast<uint8_t*>(c->d_out.p);
    unsigned long long* d_busy = reinterpret_cast<unsigned long long*>(reinterpret_cast<uint8_t*>(c->d_flags) + 64);
    const std::vector<Piece> pieces = piece_order(geo);
    const bool dbg = getenv("B200LZ4_DEBUG") != nullptr;

    cudaStream_t st = c->stream;
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(c->ev.start, st));
        CU(cudaMemsetAsync(c->d_flags, 0, 256, st));
        CU(cudaMemcpyAsync(dd, hd, lay.upload, cudaMemcpyHostToDevice, st));
        for (size_t pi = 0; pi < pieces.size(); pi++) {
            const Piece pc = pieces[pi];
            if ((rc = copy_piece(d_src, (size_t)DP, hsrc + src_off[0], (size_t)shp.P, geo, groups[pc.g], n, L, src_len[n - 1], pc.s,
                                 cudaMemcpyHostToDevice, st))) return rc;
            if (flag_separate) {                // the flag is raised from another stream: the next piece starts right behind this one
                while (c->ev_piece.size() <= pi) { cudaEvent_t e; CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); c->ev_piece.push_back(e); }
                CU(cudaEventRecord(c->ev_piece[pi], st));
                CU(cudaStreamWaitEvent(c->fstream, c->ev_piece[pi], 0));
                CU(launch_set_flag(c->d_flags + pc.g, (uint32_t)(pc.s + 1), c->fstream));
                c->launches++;
            }
            else if (flag_by_kernel) CU(launch_set_flag(c->d_flags + pc.g, (uint32_t)(pc.s + 1), st));
            else CU(cudaMemcpyAsync(c->d_flags + pc.g, c->h_const + (pc.s + 1), sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            if (pc.s != 0) continue;
            // first segment of the group is on its way: queue the group's kernels behind it
            cudaStream_t ks = c->kstream[pc.g % nks];
            if ((rc = start_range(c, pc.g, ks, Span{0, 0}, d_src, hsrc))) return rc;
            CompressArgs a = launch_args<CompressArgs>(lay, dd, d_src, d_slots, n, header, groups[pc.g], c->scratch + pc.g, false, false);
            a.accel = accel; a.arrived = c->d_flags + pc.g; a.seg_bytes = geo.seg; a.busy_cycles = d_busy;
            a.dict_state = dict_state;
            if ((rc = compress_range(c, a, lay, groups[pc.g], pc.g, d_out, ks))) return rc;
        }
        CU(cudaEventRecord(c->ev.h2d_end, st));
        if (dbg) { fprintf(stderr, "[b200lz4] streamed: %zu pieces queued (G %d S %d seg %d w %.3f)\n", pieces.size(), geo.G, geo.S, geo.seg, geo.w); fflush(stderr); }
        CU(cudaEventRecord(c->ev.d0, c->dstream));
        return drain_compacted(c, groups, geo.G, lay, d_out, dst, dst_cap, dst_off, n, dbg);
    };
    rc = finish_call(c, enqueue(), groups, geo.G, "group", "first segment landed", lay.out_len_in(hd), out_len, n, false);
    if (rc && rc != B200LZ4_E_BLOCK) return rc;
    // what this call measured tunes the next one's schedule
    unsigned long long busy[3] = {0, 0, 0};
    CU(cudaMemcpy(busy, d_busy, sizeof busy, cudaMemcpyDeviceToHost));
    if (busy[2]) { fail(B200LZ4_E_CUDA, "streamed compress: " + std::to_string(busy[2]) + " blocks gave up waiting for their input segments"); return kStreamedGaveUp; }
    if (busy[1] && c->clock_khz > 0) {
        const double ns = (double)busy[0] / (double)busy[1] / ((double)c->clock_khz * 1e-6);
        c->est_ns_per_byte = c->est_ns_per_byte > 0 ? 0.5 * c->est_ns_per_byte + 0.5 * ns : ns;
    }
    if (c->t_h2d > 0) {
        const double gbs = (double)total / ((double)c->t_h2d * 1e6);
        c->est_h2d_gbs = c->est_h2d_gbs > 0 ? 0.5 * c->est_h2d_gbs + 0.5 * gbs : gbs;
    }
    c->streamed_calls++;
    if (dbg) fprintf(stderr, "[b200lz4] streamed: G %d S %d seg %d w %.3f rho %.3f  est %.2f ns/B  h2d %.1f GB/s\n", geo.G, geo.S, geo.seg, geo.w, geo.rho, c->est_ns_per_byte, c->est_h2d_gbs);
    return rc;
}

int compress_host(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                  const int64_t* src_off, const int32_t* src_len, int n,
                  const int32_t* stream_first, int n_streams, b200lz4_cstream* const* streams,
                  int accel, int header, const int32_t* block_cap, const CState* dict_state,
                  void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const Verdict v = check_batch(Entry::Ctx, false, c, n, header, 0, src, src_bytes, src_off, src_len, dst, dst_off, out_len,
                                  stream_first, n_streams, streams != nullptr);
    if (v.code) return fail(v);
    if (n == 0) { if (dst_off) dst_off[0] = 0; return 0; }
    int rc;
    CU(cudaSetDevice(c->device));
    const int ns = stream_first ? n_streams : n;
    // (B200LZ4_NO_STREAMED is read per call: bench.py times both pipelines in one process)
    const StreamShape shp = streamed_shape(src_off, src_len, n, stream_first != nullptr, block_cap != nullptr,
                                           getenv("B200LZ4_NO_STREAMED") != nullptr);
    if (shp.ok) {
        if ((rc = probe_stream_aliasing(c))) return rc;
        if (c->n_kgood >= 2) {
            rc = compress_host_streamed(c, src, src_off, src_len, n, shp, accel, header, dict_state, dst, dst_cap, dst_off, out_len);
            if (rc != kStreamedGaveUp) return rc;
            // finders gave up waiting for their input (should not happen on verified streams): never again on this
            // ctx, and this batch goes through the plain pipeline
            c->n_kgood = 0;
            if (getenv("B200LZ4_DEBUG")) fprintf(stderr, "[b200lz4] streamed call gave up (%s): plain pipeline from now on\n", g_err.c_str());
        }
    }

    // stream state: make sure each persistent stream can keep its last array
    if (streams) {
        for (int s = 0; s < n_streams; s++) {
            if (!streams[s] || streams[s]->ctx != c) return fail(B200LZ4_E_ARG, "stream handle belongs to another ctx");
            if (stream_first[s + 1] > stream_first[s]) {
                uint32_t need = (uint32_t)src_len[stream_first[s + 1] - 1];
                if ((rc = cstream_reserve(streams[s], need))) return rc;
            }
        }
    }
    Range chunks[kMaxChunks];
    const int nchunks = plan_chunks(src_len, n, stream_first, ns, false, chunks);

    const DescLayout lay(n, n, n, ns + 1, ns, n + nchunks, 0);
    if ((rc = ensure_desc(c, lay))) return rc;
    void* hd = c->h_desc.p;
    void* dd = c->d_desc.p;
    int64_t* h_slot_off = lay.slot_off_in(hd);
    int32_t* h_cap = lay.cap_in(hd);
    memcpy(lay.src_off_in(hd), src_off, sizeof(int64_t) * n);
    memcpy(lay.src_len_in(hd), src_len, sizeof(int32_t) * n);
    int64_t slots_total = 0;
    for (int i = 0; i < n; i++) {
        h_cap[i] = block_cap ? std::max(block_cap[i], 0) + header : (int)compress_cap(src_len[i], header);
        h_slot_off[i] = slots_total;
        slots_total += compress_slot(h_cap[i]);
    }
    if (stream_first) memcpy(lay.first_in(hd), stream_first, sizeof(int32_t) * (ns + 1));
    if (streams) for (int s = 0; s < ns; s++) lay.states_in(hd)[s] = streams[s]->d_state;

    if ((rc = c->d_src.ensure((size_t)src_bytes + 64))) return rc;
    if ((rc = c->d_slots.ensure((size_t)slots_total + 64))) return rc;
    if ((rc = c->d_out.ensure((size_t)slots_total + 64))) return rc;
    const uint8_t* hsrc = static_cast<const uint8_t*>(src);
    uint8_t* d_src = static_cast<uint8_t*>(c->d_src.p);
    uint8_t* d_slots = static_cast<uint8_t*>(c->d_slots.p);
    uint8_t* d_out = static_cast<uint8_t*>(c->d_out.p);

    cudaStream_t st = c->stream;
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(c->ev.start, st));
        CU(cudaMemcpyAsync(dd, hd, lay.upload, cudaMemcpyHostToDevice, st));
        for (int k = 0; k < nchunks; k++) {
            cudaStream_t ks = c->kstream[k % kKernelStreams];
            if ((rc = start_range(c, k, ks, byte_span(src_off, src_len, chunks[k].b0, chunks[k].b1), d_src, hsrc))) return rc;
            CompressArgs a = launch_args<CompressArgs>(lay, dd, d_src, d_slots, n, header, chunks[k], c->scratch + k,
                                                       stream_first != nullptr, streams != nullptr);
            a.dst_cap = block_cap ? lay.cap_in(dd) : nullptr;
            a.accel = accel;
            a.dict_state = dict_state;
            if ((rc = compress_range(c, a, lay, chunks[k], k, d_out, ks))) return rc;
        }
        CU(cudaEventRecord(c->ev.h2d_end, st));
        CU(cudaEventRecord(c->ev.d0, c->dstream));
        return drain_compacted(c, chunks, nchunks, lay, d_out, dst, dst_cap, dst_off, n, false);
    };
    rc = finish_call(c, enqueue(), chunks, nchunks, "chunk", "h2d done", lay.out_len_in(hd), out_len, n, false);
    if (streams && (rc == 0 || rc == B200LZ4_E_BLOCK)) for (int s = 0; s < n_streams; s++)
        if (stream_first[s + 1] > stream_first[s]) streams[s]->last_len = (uint32_t)src_len[stream_first[s + 1] - 1];
    return rc;
}

int decompress_host_streamed(b200lz4_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, int n,
                             int L, int cap_last, const DState* dict_state, void* dst, int64_t dst_cap, int64_t* dst_off,
                             int32_t* out_len);

int decompress_host(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                    const int64_t* src_off, const int32_t* src_len, int n,
                    const int32_t* stream_first, int n_streams, b200lz4_dstream* const* streams,
                    int header, int max_block, const DState* dict_state,
                    void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const Verdict v = check_batch(Entry::Ctx, true, c, n, header, max_block, src, src_bytes, src_off, src_len, dst, dst_off, out_len,
                                  stream_first, n_streams, streams != nullptr);
    if (v.code) return fail(v);
    if (n == 0) { if (dst_off) dst_off[0] = 0; return 0; }
    int rc;
    CU(cudaSetDevice(c->device));
    const int ns = stream_first ? n_streams : n;
    if (streams) for (int s = 0; s < n_streams; s++)
        if (!streams[s] || streams[s]->ctx != c) return fail(B200LZ4_E_ARG, "stream handle belongs to another ctx");
    const uint8_t* hsrc = static_cast<const uint8_t*>(src);
    // How the output goes home (B200LZ4_DECODE_OUT, host_plan.h: decode_route).  Measured on config 2 (1.07 GB out,
    // 0.77 GB in): copy 27.7 ms, mirror 27.0 ms (the posted writes of 1 678 CTAs reach 40 GB/s and slow the H2D copy from
    // 15 to 18.5 ms), pieces 26.4 ms -- so mirror stays opt-in.
    const char* out_env = getenv("B200LZ4_DECODE_OUT");
    const char* dwide_env = getenv("B200LZ4_DWIDE");            // (tests force the wide kernel with it: that one has no mirror)
    uint8_t* mirror_dst = nullptr;
    if (out_env && out_env[0] == 'm') {
        cudaPointerAttributes pa{};
        if (cudaPointerGetAttributes(&pa, dst) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer)
            mirror_dst = static_cast<uint8_t*>(pa.devicePointer);
        else cudaGetLastError();
    }
    const DecodeRoute route = decode_route(hsrc, src_off, src_len, n, header, stream_first != nullptr, out_env ? out_env[0] : 0,
                                           getenv("B200LZ4_NO_STREAMED") != nullptr, dwide_env && dwide_env[0] == '1',
                                           mirror_dst != nullptr);
    if (route.out == DecodeOut::Pieces)
        return decompress_host_streamed(c, src, src_off, src_len, n, route.L, route.cap_last, dict_state, dst, dst_cap, dst_off,
                                        out_len);
    if (route.out != DecodeOut::Mirror) mirror_dst = nullptr;
    Range chunks[kMaxChunks];
    const int nchunks = plan_chunks(src_len, n, stream_first, ns, mirror_dst != nullptr, chunks);
    if (getenv("B200LZ4_DEBUG")) fprintf(stderr, "[b200lz4] decompress: %s output, %d chunks\n", mirror_dst ? "mirror" : "copy", nchunks);

    const DescLayout lay(n, n, n, ns + 1, ns, n + nchunks, 0);
    if ((rc = ensure_desc(c, lay))) return rc;
    void* hd = c->h_desc.p;
    void* dd = c->d_desc.p;
    int64_t* h_slot_off = lay.slot_off_in(hd);
    int32_t* h_cap = lay.cap_in(hd);
    memcpy(lay.src_off_in(hd), src_off, sizeof(int64_t) * n);
    memcpy(lay.src_len_in(hd), src_len, sizeof(int32_t) * n);
    int64_t slots_total = 0;
    for (int i = 0; i < n; i++) {
        h_cap[i] = decode_cap(hsrc, src_off, src_len, i, header, max_block);
        h_slot_off[i] = slots_total;
        slots_total += decode_slot(h_cap[i], header);
    }
    const bool contiguous = (header == 8);     // slots are already exactly the output layout
    if (contiguous && slots_total > dst_cap) return fail(B200LZ4_E_NOMEM, "dst_cap too small: need " + std::to_string(slots_total));
    if (stream_first) memcpy(lay.first_in(hd), stream_first, sizeof(int32_t) * (ns + 1));
    if (streams) for (int s = 0; s < ns; s++) lay.states_in(hd)[s] = streams[s]->d_state;

    if ((rc = c->d_src.ensure((size_t)src_bytes + 64))) return rc;
    if ((rc = c->d_slots.ensure((size_t)slots_total + 64 + 16))) return rc;
    if (!contiguous && (rc = c->d_out.ensure((size_t)slots_total + 64))) return rc;
    // descriptor rings for chunks the wide kernel may take (few streams): one slice of one CTA-arena per stream, per chunk
    int wide_first[kMaxChunks + 1] = {0};
    for (int k = 0; k < nchunks; k++) wide_first[k + 1] = wide_first[k] + std::min(chunks[k].u1 - chunks[k].u0, kWideMaxCtas);
    if ((rc = c->d_wide.ensure((size_t)wide_first[nchunks] * kWideArenaPerCta))) return rc;
    uint8_t* d_src = static_cast<uint8_t*>(c->d_src.p);
    uint8_t* d_slots = static_cast<uint8_t*>(c->d_slots.p);
    if (mirror_dst) d_slots += reinterpret_cast<uintptr_t>(mirror_dst) & 15;      // same address modulo 16 on both sides: 128-bit stores line up
    uint8_t* d_out = static_cast<uint8_t*>(c->d_out.p);

    cudaStream_t st = c->stream;
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(c->ev.start, st));
        CU(cudaMemcpyAsync(dd, hd, lay.upload, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(c->ev.d0, c->dstream));
        for (int k = 0; k < nchunks; k++) {
            const Range& ch = chunks[k];
            cudaStream_t ks = c->kstream[k % kKernelStreams];
            if ((rc = start_range(c, k, ks, byte_span(src_off, src_len, ch.b0, ch.b1), d_src, hsrc))) return rc;
            DecompressArgs a = launch_args<DecompressArgs>(lay, dd, d_src, d_slots, n, header, ch, c->scratch + k,
                                                           stream_first != nullptr, streams != nullptr);
            a.dst_cap = lay.cap_in(dd);
            a.max_block = max_block;
            a.wide_arena = reinterpret_cast<uint4*>(static_cast<uint8_t*>(c->d_wide.p) + (size_t)wide_first[k] * kWideArenaPerCta);
            a.wide_ctas = wide_first[k + 1] - wide_first[k];
            a.host_dst = mirror_dst;
            a.dict_state = dict_state;
            CU(launch_decompress(a, ks));
            c->launches += kernel_launches_per_decompress();
            const int nk = ch.b1 - ch.b0;
            if (!contiguous) {
                CompactArgs g{d_slots, a.dst_off + ch.b0, a.out_len + ch.b0, nk, 0, d_out + h_slot_off[ch.b0],
                              lay.out_off_in(dd) + ch.b0 + k, nullptr, nullptr};
                CU(launch_compact(g, ks));
                c->launches += kernel_launches_per_compact();
                CU(cudaMemcpyAsync(lay.out_off_in(hd) + ch.b0 + k, lay.out_off_in(dd) + ch.b0 + k, sizeof(int64_t) * (nk + 1), cudaMemcpyDeviceToHost, ks));
            }
            CU(cudaMemcpyAsync(lay.out_len_in(hd) + ch.b0, lay.out_len_in(dd) + ch.b0, sizeof(int32_t) * nk, cudaMemcpyDeviceToHost, ks));
            CU(cudaEventRecord(c->ev.k[k], ks));
            if (contiguous && !mirror_dst) {   // sizes are known from the headers: the D2H copy can be queued right away
                const int64_t lo = h_slot_off[ch.b0];
                const int64_t hi = (ch.b1 < n) ? h_slot_off[ch.b1] : slots_total;
                CU(cudaStreamWaitEvent(c->dstream, c->ev.k[k], 0));
                if (hi > lo) CU(cudaMemcpyAsync(static_cast<uint8_t*>(dst) + lo, d_slots + lo, (size_t)(hi - lo), cudaMemcpyDeviceToHost, c->dstream));
            }
        }
        CU(cudaEventRecord(c->ev.h2d_end, st));
        if (!contiguous) return drain_compacted(c, chunks, nchunks, lay, d_out, dst, dst_cap, dst_off, n, false);
        memcpy(dst_off, h_slot_off, sizeof(int64_t) * n);
        dst_off[n] = slots_total;
        return 0;
    };
    return finish_call(c, enqueue(), chunks, nchunks, nullptr, nullptr, lay.out_len_in(hd), out_len, n, true);
}

// ---- streamed decompress call --------------------------------------------------
// The mirror image of compress_host_streamed for the OUTPUT side: decompression of equally large independent blocks is
// bound by the D2H copy (1.40 x the bytes of the H2D copy on config 2), and in the plain pipeline the first byte cannot
// leave before a whole chunk has arrived AND one block latency has passed.  Here every group's kernel counts, per segment of
// the (equal) block capacity, the blocks whose flushed output has passed it (decompress.cu: kPublish); the last one raises
// a flag in page-locked host memory, the calling thread polls the flags and queues that segment of every block of the
// group as one 2-D D2H copy.  The copy engine then runs from "first group landed + one SEGMENT latency" to the end.
int decompress_host_streamed(b200lz4_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, int n,
                             int L, int cap_last, const DState* dict_state, void* dst, int64_t dst_cap, int64_t* dst_off,
                             int32_t* out_len)
{
    int rc;
    const int header = 8;
    const int64_t out_total = (int64_t)L * (n - 1) + cap_last;
    if (out_total > dst_cap) return fail(B200LZ4_E_NOMEM, "dst_cap too small: need " + std::to_string(out_total));
    const Geometry geo = decompress_geometry(n, L, getenv("B200LZ4_STREAM_G"), getenv("B200LZ4_STREAM_S"));
    Range groups[kMaxGroups];
    plan_groups(geo, n, groups);
    if ((rc = probe_stream_aliasing(c))) return rc;     // nothing can deadlock here, but kernels queued behind another group's would start late
    const int nks = c->n_kgood >= 2 ? c->n_kgood : kKernelStreams;

    const DescLayout lay(n, n, n, 0, 0, 0, kMaxGroups * kMaxSegs);
    if ((rc = ensure_desc(c, lay))) return rc;
    void* hd = c->h_desc.p;
    void* dd = c->d_desc.p;
    int64_t* h_slot_off = lay.slot_off_in(hd);
    int32_t* h_cap = lay.cap_in(hd);
    volatile uint32_t* ready = lay.ready_in(hd);
    memcpy(lay.src_off_in(hd), src_off, sizeof(int64_t) * n);
    memcpy(lay.src_len_in(hd), src_len, sizeof(int32_t) * n);
    int64_t src_hi = 0;
    for (int i = 0; i < n; i++) {
        h_cap[i] = i < n - 1 ? L : cap_last;
        h_slot_off[i] = (int64_t)L * i;
        dst_off[i] = (int64_t)L * i;
        src_hi = std::max(src_hi, src_off[i] + (int64_t)src_len[i]);
    }
    dst_off[n] = out_total;
    for (int i = 0; i < kMaxGroups * kMaxSegs; i++) ready[i] = 0;
    if ((rc = c->d_src.ensure((size_t)src_hi + 64))) return rc;
    if ((rc = c->d_slots.ensure((size_t)out_total + 64))) return rc;
    const uint8_t* hsrc = static_cast<const uint8_t*>(src);
    uint8_t* d_src = static_cast<uint8_t*>(c->d_src.p);
    uint8_t* d_slots = static_cast<uint8_t*>(c->d_slots.p);
    uint32_t* d_counts = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(c->d_flags) + 1024);
    const bool dbg = getenv("B200LZ4_DEBUG") != nullptr;
    if (dbg) fprintf(stderr, "[b200lz4] streamed decompress: G %d S %d seg %d\n", geo.G, geo.S, geo.seg);
    struct PieceLog { int g, s; double issued_ms; cudaEvent_t done; };
    std::vector<PieceLog> plog;

    cudaStream_t st = c->stream;
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(c->ev.start, st));
        CU(cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * kMaxGroups * kMaxSegs, st));
        CU(cudaMemcpyAsync(dd, hd, lay.upload, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(c->ev.d0, c->dstream));
        for (int g = 0; g < geo.G; g++) {
            cudaStream_t ks = c->kstream[g % nks];
            if ((rc = start_range(c, g, ks, byte_span(src_off, src_len, groups[g].b0, groups[g].b1), d_src, hsrc))) return rc;
            DecompressArgs a = launch_args<DecompressArgs>(lay, dd, d_src, d_slots, n, header, groups[g], c->scratch + g, false, false);
            a.dst_cap = lay.cap_in(dd);
            a.out_len = lay.out_len_in(hd);     // page-locked, device-visible: no small D2H copies that would queue behind the pieces
            a.max_block = 0;
            a.seg_count = d_counts + g * kMaxSegs;
            a.host_ready = lay.ready_in(hd) + g * kMaxSegs;
            a.seg_bytes = geo.seg; a.n_segs = geo.S;
            a.dict_state = dict_state;
            CU(launch_decompress(a, ks));
            c->launches += kernel_launches_per_decompress();
            CU(cudaEventRecord(c->ev.k[g], ks));
        }
        CU(cudaEventRecord(c->ev.h2d_end, st));

        // drain: queue every (group, segment) piece as soon as its flag is up
        int next_s[kMaxGroups] = {0};
        int remaining = geo.G * geo.S;
        const auto t_host0 = std::chrono::steady_clock::now();
        long spins = 0;
        while (remaining) {
            bool any = false;
            for (int g = 0; g < geo.G; g++) {
                while (next_s[g] < geo.S && ready[g * kMaxSegs + next_s[g]]) {
                    if ((rc = copy_piece(static_cast<uint8_t*>(dst), (size_t)L, d_slots, (size_t)L, geo, groups[g], n, L, cap_last, next_s[g],
                                         cudaMemcpyDeviceToHost, c->dstream))) return rc;
                    if (dbg) {
                        PieceLog pl{g, next_s[g], std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count(), nullptr};
                        cudaEventCreate(&pl.done); cudaEventRecord(pl.done, c->dstream);
                        plog.push_back(pl);
                    }
                    next_s[g]++; remaining--; any = true;
                }
            }
            if (any) { spins = 0; continue; }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
            if (++spins % 4096 == 0) {          // a faulted or finished kernel must not leave this loop spinning
                bool all_done = true;
                for (int g = 0; g < geo.G; g++) {
                    const cudaError_t q = cudaEventQuery(c->ev.k[g]);
                    if (q == cudaErrorNotReady) { all_done = false; break; }
                    if (q != cudaSuccess) return fail_cuda(q, "streamed decompress");
                }
                if (all_done) {                 // every block has ended, so every flag is up: one last look
                    bool missing = false;
                    for (int g = 0; g < geo.G; g++) for (int k = next_s[g]; k < geo.S; k++) if (!ready[g * kMaxSegs + k]) missing = true;
                    if (missing) return fail(B200LZ4_E_CUDA, "streamed decompress: kernels ended without raising every segment flag");
                }
            }
        }
        return 0;
    };
    rc = finish_call(c, enqueue(), groups, geo.G, "group", "input landed", lay.out_len_in(hd), out_len, n, true);
    for (auto& pl : plog) {     // (host time counts from the moment the drain loop started)
        float x = 0; cudaEventElapsedTime(&x, c->ev.start, pl.done);
        fprintf(stderr, "[b200lz4] piece g%d s%d: queued at host +%.2f ms, copied by %.2f\n", pl.g, pl.s, pl.issued_ms, x);
        cudaEventDestroy(pl.done);
    }
    return rc;
}

}  // namespace

// ============================================================== C ABI ====

extern "C" {

int b200lz4_compress_bound(int n) { return bound_of(n); }
int b200lz4_version(void) { return B200LZ4_VERSION_NUMBER; }
const char* b200lz4_last_error(void) { return g_err.c_str(); }

int b200lz4_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; d++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

int b200lz4_ctx_create(int device, b200lz4_ctx** out)
{
    if (!out) return fail(B200LZ4_E_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) { cudaGetLastError(); return fail(B200LZ4_E_CUDA, "no CUDA device: this library has no CPU path"); }
    if (device < 0 || device >= n) return fail(B200LZ4_E_ARG, "device index out of range");
    int major = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(B200LZ4_E_CUDA, "device is not compute capability 10.x (kernels are built for sm_100a only)");
    CU(cudaSetDevice(device));
    b200lz4_ctx* c = new (std::nothrow) b200lz4_ctx();
    if (!c) return fail(B200LZ4_E_NOMEM, "out of host memory");
    c->device = device;
    cudaError_t e2 = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (int i = 0; i < kKernelStreams && e2 == cudaSuccess; i++) e2 = cudaStreamCreateWithFlags(&c->kstream[i], cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&c->dstream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaMalloc(&c->scratch, sizeof(Scratch) * kMaxGroups);
    if (e2 == cudaSuccess) e2 = cudaMemset(c->scratch, 0, sizeof(Scratch) * kMaxGroups);
    if (e2 == cudaSuccess) e2 = cudaMalloc(&c->d_flags, kFlagBytes);
    if (e2 == cudaSuccess) e2 = cudaMemset(c->d_flags, 0, kFlagBytes);
    if (e2 == cudaSuccess) e2 = cudaHostAlloc(reinterpret_cast<void**>(&c->h_const), 64 * sizeof(uint32_t), cudaHostAllocPortable);
    if (e2 == cudaSuccess) for (uint32_t i = 0; i < 64; i++) c->h_const[i] = i;
    if (e2 == cudaSuccess) e2 = cudaDeviceGetAttribute(&c->clock_khz, cudaDevAttrClockRate, device);
    c->ev.each([&](cudaEvent_t& ev) { if (e2 == cudaSuccess) e2 = cudaEventCreate(&ev); });
    if (e2 != cudaSuccess) { b200lz4_ctx_destroy(c); return fail_cuda(e2, "ctx_create"); }
    *out = c;
    return 0;
}

void b200lz4_ctx_destroy(b200lz4_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    c->d_src.release(); c->d_slots.release(); c->d_out.release(); c->d_desc.release(); c->d_wide.release(); c->h_desc.release();
    if (c->scratch) cudaFree(c->scratch);
    if (c->d_flags) cudaFree(c->d_flags);
    if (c->h_const) cudaFreeHost(c->h_const);
    c->ev.each([](cudaEvent_t& e) { if (e) cudaEventDestroy(e); });
    for (auto& k : c->kstream) if (k) cudaStreamDestroy(k);
    if (c->fstream) cudaStreamDestroy(c->fstream);
    for (auto& e : c->ev_piece) if (e) cudaEventDestroy(e);
    if (c->dstream) cudaStreamDestroy(c->dstream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

void* b200lz4_host_alloc(size_t bytes)
{
    void* p = nullptr;
    cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
    if (e != cudaSuccess) { fail_cuda(e, "cudaMallocHost"); return nullptr; }
    return p;
}
void* b200lz4_host_alloc_wc(size_t bytes)
{
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocWriteCombined | cudaHostAllocPortable);
    if (e != cudaSuccess) { fail_cuda(e, "cudaHostAlloc(write-combined)"); return nullptr; }
    return p;
}
void* b200lz4_ctx_host_alloc(b200lz4_ctx* c, size_t bytes)
{
    if (!c) { fail(B200LZ4_E_ARG, "ctx is NULL"); return nullptr; }
    if (cudaSetDevice(c->device) != cudaSuccess) { fail(B200LZ4_E_CUDA, "cudaSetDevice"); return nullptr; }
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) { fail_cuda(e, "cudaHostAlloc"); return nullptr; }
    return p;
}
void b200lz4_host_free(void* p) { if (p) cudaFreeHost(p); }

int b200lz4_last_timing(b200lz4_ctx* c, float* h2d, float* kern, float* d2h)
{
    if (!c) return fail(B200LZ4_E_ARG, "ctx is NULL");
    if (h2d) *h2d = c->t_h2d;
    if (kern) *kern = c->t_kernel;
    if (d2h) *d2h = c->t_d2h;
    return 0;
}
int64_t b200lz4_launch_count(b200lz4_ctx* c) { return c ? c->launches : 0; }
const char* b200lz4_ctx_last_error(b200lz4_ctx* c) { return c ? c->err.c_str() : ""; }

// Parallel gather of separately allocated (pageable) arrays into one staging buffer: what the Haskell shim / api.py do
// before every batch call.  One contiguous range of arrays per thread, balanced by bytes.
int b200lz4_gather_host(void* dst, const void* const* src_ptrs, const int64_t* dst_off, const int32_t* len, int n, int threads)
{
    if (n < 0 || (n > 0 && (!dst || !src_ptrs || !dst_off || !len))) return fail(B200LZ4_E_ARG, "NULL argument");
    if (n == 0) return 0;
    int64_t total = 0;
    for (int i = 0; i < n; i++) { if (len[i] < 0 || (len[i] > 0 && !src_ptrs[i])) return fail(B200LZ4_E_ARG, "bad array"); total += len[i]; }
    unsigned hw = std::thread::hardware_concurrency();
    int t = threads > 0 ? threads : (int)(hw ? (hw > 16 ? 16 : hw) : 4);
    if (total < (int64_t(4) << 20)) t = 1;
    if (t > n) t = n;
    auto work = [&](int lo, int hi) {
        uint8_t* d = static_cast<uint8_t*>(dst);
        for (int i = lo; i < hi; i++) if (len[i]) memcpy(d + dst_off[i], src_ptrs[i], (size_t)len[i]);
    };
    if (t <= 1) { work(0, n); return 0; }
    std::vector<std::thread> pool;
    int lo = 0; int64_t done = 0;
    for (int k = 0; k < t; k++) {
        const int64_t target = total * (k + 1) / t;
        int hi = lo;
        while (hi < n && (done < target || k == t - 1)) done += len[hi++];
        if (hi > lo) pool.emplace_back(work, lo, hi);
        lo = hi;
    }
    for (auto& th : pool) th.join();
    return 0;
}

// Measurement aid (bench.py's copy ceiling): one plain H2D copy of h2d_bytes and one D2H copy of d2h_bytes on the ctx's
// two copy streams at once, no kernels; returns after both are complete.  Host buffers should be page-locked.
int b200lz4_copy_probe(b200lz4_ctx* c, const void* h_src, int64_t h2d_bytes, void* h_dst, int64_t d2h_bytes)
{
    if (!c || h2d_bytes < 0 || d2h_bytes < 0) return fail(B200LZ4_E_ARG, "bad argument");
    CU(cudaSetDevice(c->device));
    int rc;
    if (h2d_bytes && (rc = c->d_src.ensure((size_t)h2d_bytes + 64))) return rc;
    if (d2h_bytes && (rc = c->d_out.ensure((size_t)d2h_bytes + 64))) return rc;
    if (h2d_bytes) CU(cudaMemcpyAsync(c->d_src.p, h_src, (size_t)h2d_bytes, cudaMemcpyHostToDevice, c->stream));
    if (d2h_bytes) CU(cudaMemcpyAsync(h_dst, c->d_out.p, (size_t)d2h_bytes, cudaMemcpyDeviceToHost, c->dstream));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaStreamSynchronize(c->dstream));
    return 0;
}

int b200lz4_cstream_create(b200lz4_ctx* c, b200lz4_cstream** out)
{
    if (!c || !out) return fail(B200LZ4_E_ARG, "NULL argument");
    *out = nullptr;
    CU(cudaSetDevice(c->device));
    b200lz4_cstream* s = new (std::nothrow) b200lz4_cstream{c, nullptr, nullptr, 0, 0};
    if (!s) return fail(B200LZ4_E_NOMEM, "out of host memory");
    cudaError_t e = cudaMalloc(&s->d_state, sizeof(CState));
    if (e == cudaSuccess) e = cudaMemsetAsync(s->d_state, 0, sizeof(CState), c->stream);     // LZ4_initStream, cbits/lz4.c:1443-1451
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { if (s->d_state) cudaFree(s->d_state); delete s; return fail_cuda(e, "cstream_create"); }
    *out = s;
    return 0;
}
void b200lz4_cstream_free(b200lz4_cstream* s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    if (s->d_state) cudaFree(s->d_state);
    if (s->d_dict) cudaFree(s->d_dict);
    delete s;
}
int b200lz4_cstream_peek(b200lz4_cstream* s, uint32_t* table, uint32_t* offset)
{
    if (!s) return fail(B200LZ4_E_ARG, "NULL stream");
    CU(cudaSetDevice(s->ctx->device));
    CU(cudaStreamSynchronize(s->ctx->stream));
    if (table) CU(cudaMemcpy(table, s->d_state->table, sizeof(uint32_t) * kHashEntries, cudaMemcpyDeviceToHost));
    if (offset) CU(cudaMemcpy(offset, &s->d_state->offset, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return 0;
}
int b200lz4_dstream_create(b200lz4_ctx* c, b200lz4_dstream** out)
{
    if (!c || !out) return fail(B200LZ4_E_ARG, "NULL argument");
    *out = nullptr;
    CU(cudaSetDevice(c->device));
    b200lz4_dstream* s = new (std::nothrow) b200lz4_dstream{c, nullptr};
    if (!s) return fail(B200LZ4_E_NOMEM, "out of host memory");
    cudaError_t e = cudaMalloc(&s->d_state, sizeof(DState));
    if (e == cudaSuccess) e = cudaMemsetAsync(s->d_state, 0, 16, c->stream);                 // calloc, cbits/lz4.c:2265-2270
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { if (s->d_state) cudaFree(s->d_state); delete s; return fail_cuda(e, "dstream_create"); }
    *out = s;
    return 0;
}
void b200lz4_dstream_free(b200lz4_dstream* s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    if (s->d_state) cudaFree(s->d_state);
    delete s;
}

// ---- dictionaries (LZ4_loadDict / LZ4_setStreamDecode) ----
int b200lz4_dict_create(b200lz4_ctx* c, const void* dict, int64_t len, b200lz4_dict** out)
{
    if (!c || !out || len < 0 || (len > 0 && !dict)) return fail(B200LZ4_E_ARG, "NULL argument or negative length");
    if (len > kMaxInput) return fail(B200LZ4_E_ARG, "dictionary longer than LZ4_MAX_INPUT_SIZE");
    *out = nullptr;
    CU(cudaSetDevice(c->device));
    b200lz4_dict* d = new (std::nothrow) b200lz4_dict{c, nullptr, len, nullptr, nullptr};
    if (!d) return fail(B200LZ4_E_NOMEM, "out of host memory");
    cudaError_t e = cudaMalloc(&d->d_bytes, (size_t)len + 16);
    if (e == cudaSuccess) e = cudaMalloc(&d->d_cstate, sizeof(CState));
    if (e == cudaSuccess) e = cudaMalloc(&d->d_dstate, sizeof(DState));
    if (e == cudaSuccess && len) e = cudaMemcpyAsync(d->d_bytes, dict, (size_t)len, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = launch_load_dict(d->d_bytes, len, d->d_cstate, d->d_dstate, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { b200lz4_dict_free(d); return fail_cuda(e, "dict_create"); }
    c->launches++;
    *out = d;
    return 0;
}
void b200lz4_dict_free(b200lz4_dict* d)
{
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    sync_all(d->ctx);
    if (d->d_bytes) cudaFree(d->d_bytes);
    if (d->d_cstate) cudaFree(d->d_cstate);
    if (d->d_dstate) cudaFree(d->d_dstate);
    delete d;
}
int b200lz4_cstream_load_dict(b200lz4_cstream* s, const b200lz4_dict* d)
{
    if (!s || !d) return fail(B200LZ4_E_ARG, "NULL argument");
    if (s->ctx != d->ctx) return fail(B200LZ4_E_ARG, "dictionary belongs to another ctx");
    b200lz4_ctx* c = s->ctx;
    CU(cudaSetDevice(c->device));
    // the kernel overwrites the stream's dict_buf with its last array, so the stream keeps a copy of the dictionary's tail
    const uint32_t dict_len = d->len < 8 ? 0u : (uint32_t)std::min<int64_t>(d->len, 65536);
    int rc;
    if ((rc = cstream_reserve(s, dict_len))) return rc;
    static_assert(offsetof(CState, dict_len) == offsetof(CState, table) + sizeof(CState::table) + 4, "CState layout");
    CU(cudaMemcpyAsync(s->d_state, d->d_cstate, offsetof(CState, dict_len) + sizeof(uint32_t), cudaMemcpyDeviceToDevice, c->stream));
    if (dict_len) CU(cudaMemcpyAsync(s->d_dict, d->d_bytes + (d->len - dict_len), dict_len, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    s->last_len = dict_len;
    return 0;
}
int b200lz4_dstream_set_dict(b200lz4_dstream* s, const b200lz4_dict* d)
{
    if (!s || !d) return fail(B200LZ4_E_ARG, "NULL argument");
    if (s->ctx != d->ctx) return fail(B200LZ4_E_ARG, "dictionary belongs to another ctx");
    CU(cudaSetDevice(s->ctx->device));
    CU(cudaMemcpyAsync(s->d_state, d->d_dstate, sizeof(DState), cudaMemcpyDeviceToDevice, s->ctx->stream));
    CU(cudaStreamSynchronize(s->ctx->stream));
    return 0;
}

int b200lz4_compress_batch(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                           const int64_t* src_off, const int32_t* src_len, int n_blocks,
                           const int32_t* stream_first, int n_streams, b200lz4_cstream* const* streams,
                           int acceleration, int header_mode,
                           void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const int rc = compress_host(c, src, src_bytes, src_off, src_len, n_blocks, stream_first, n_streams, streams,
                                 acceleration, header_mode, nullptr, nullptr, dst, dst_cap, dst_off, out_len);
    if (c && rc) c->err = g_err;
    return rc;
}

int b200lz4_decompress_batch(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                             const int64_t* src_off, const int32_t* src_len, int n_blocks,
                             const int32_t* stream_first, int n_streams, b200lz4_dstream* const* streams,
                             int header_mode, int max_block,
                             void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const int rc = decompress_host(c, src, src_bytes, src_off, src_len, n_blocks, stream_first, n_streams, streams,
                                   header_mode, max_block, nullptr, dst, dst_cap, dst_off, out_len);
    if (c && rc) c->err = g_err;
    return rc;
}

namespace {
int check_dict(const b200lz4_ctx* c, const b200lz4_dict* d, bool streams_given)
{
    if (!d) return fail(B200LZ4_E_ARG, "dictionary is NULL");
    if (c && d->ctx != c) return fail(B200LZ4_E_ARG, "dictionary belongs to another ctx");
    if (streams_given) return fail(B200LZ4_E_ARG, "a dictionary together with persistent streams: load it into the streams instead");
    return 0;
}
}  // namespace

int b200lz4_compress_batch_dict(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                                const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                const int32_t* stream_first, int n_streams, b200lz4_cstream* const* streams,
                                int acceleration, int header_mode,
                                void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len, const b200lz4_dict* dict)
{
    int rc = check_dict(c, dict, streams != nullptr);
    if (!rc) rc = compress_host(c, src, src_bytes, src_off, src_len, n_blocks, stream_first, n_streams, streams,
                                acceleration, header_mode, nullptr, dict->d_cstate, dst, dst_cap, dst_off, out_len);
    if (c && rc) c->err = g_err;
    return rc;
}

int b200lz4_decompress_batch_dict(b200lz4_ctx* c, const void* src, int64_t src_bytes,
                                  const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                  const int32_t* stream_first, int n_streams, b200lz4_dstream* const* streams,
                                  int header_mode, int max_block,
                                  void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len, const b200lz4_dict* dict)
{
    int rc = check_dict(c, dict, streams != nullptr);
    if (!rc) rc = decompress_host(c, src, src_bytes, src_off, src_len, n_blocks, stream_first, n_streams, streams,
                                  header_mode, max_block, dict->d_dstate, dst, dst_cap, dst_off, out_len);
    if (c && rc) c->err = g_err;
    return rc;
}

}  // extern "C"

// ------------------------------------------------------------ several devices
// One batch striped over the GPUs of one box (SURVEY.md section 8e): contiguous ranges of blocks (independent mode) or of
// whole streams (linked mode), balanced by source bytes, one host thread and one b200lz4_ctx per device, no exchange step.

struct b200lz4_mctx {
    std::vector<b200lz4_ctx*> ctx;
    std::string err;
};

namespace {

template <class Call>
int run_striped(b200lz4_mctx* m, const int64_t* src_off, const int32_t* src_len, int n,
                const int32_t* stream_first, int n_streams, const std::vector<int64_t>& region, /* n + 1 prefix of worst-case output */
                int64_t* dst_off, int32_t* out_len, Call call)
{
    const int parts = (int)m->ctx.size();
    const std::vector<Range> st = plan_stripes(src_len, n, stream_first, n_streams, parts);
    std::vector<int> rcs(parts, 0);
    std::vector<std::string> errs(parts);
    std::vector<std::thread> pool;
    for (int d = 0; d < parts; d++) {
        const Range s = st[d];
        if (s.b1 <= s.b0) continue;
        pool.emplace_back([&, d, s]() {
            const int nb = s.b1 - s.b0;
            const Span sp = byte_span(src_off, src_len, s.b0, s.b1);
            const int64_t lo = sp.lo, hi = sp.hi;
            std::vector<int64_t> off(nb), doff(nb + 1);
            for (int i = 0; i < nb; i++) off[i] = src_off[s.b0 + i] - lo;
            std::vector<int32_t> first;
            if (stream_first) { first.resize(s.u1 - s.u0 + 1); for (int u = s.u0; u <= s.u1; u++) first[u - s.u0] = stream_first[u] - s.b0; }
            rcs[d] = call(m->ctx[d], lo, hi - lo, off.data(), src_len + s.b0, nb, stream_first ? first.data() : nullptr, s.u1 - s.u0,
                          region[s.b0], region[s.b1] - region[s.b0], doff.data(), out_len + s.b0);
            if (rcs[d]) errs[d] = g_err;
            if (rcs[d] == 0 || rcs[d] == B200LZ4_E_BLOCK) for (int i = 0; i < nb; i++) dst_off[s.b0 + i] = region[s.b0] + doff[i];
            if ((rcs[d] == 0 || rcs[d] == B200LZ4_E_BLOCK) && s.b1 == n) dst_off[n] = region[s.b0] + doff[nb];
        });
    }
    for (auto& t : pool) t.join();
    int rc = 0;
    for (int d = 0; d < parts; d++) {
        if (rcs[d] && (rc == 0 || rc == B200LZ4_E_BLOCK)) { rc = rcs[d]; m->err = "device " + std::to_string(m->ctx[d]->device) + ": " + errs[d]; }
    }
    if (rc) g_err = m->err;
    return rc;
}

}  // namespace

extern "C" {

int b200lz4_mctx_create(const int* devices, int n, b200lz4_mctx** out)
{
    if (!out) return fail(B200LZ4_E_ARG, "out is NULL");
    *out = nullptr;
    std::vector<int> devs;
    if (devices) { if (n <= 0) return fail(B200LZ4_E_ARG, "no devices"); devs.assign(devices, devices + n); }
    else {
        int cnt = 0;
        if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { cudaGetLastError(); return fail(B200LZ4_E_CUDA, "no CUDA device: this library has no CPU path"); }
        if (n > 0 && n < cnt) cnt = n;
        for (int d = 0; d < cnt; d++) devs.push_back(d);
    }
    b200lz4_mctx* m = new (std::nothrow) b200lz4_mctx();
    if (!m) return fail(B200LZ4_E_NOMEM, "out of host memory");
    for (int d : devs) {
        b200lz4_ctx* c = nullptr;
        const int rc = b200lz4_ctx_create(d, &c);
        if (rc) { for (auto* x : m->ctx) b200lz4_ctx_destroy(x); delete m; return rc; }
        m->ctx.push_back(c);
    }
    *out = m;
    return 0;
}
void b200lz4_mctx_destroy(b200lz4_mctx* m)
{
    if (!m) return;
    for (auto* c : m->ctx) b200lz4_ctx_destroy(c);
    delete m;
}
int b200lz4_mctx_size(b200lz4_mctx* m) { return m ? (int)m->ctx.size() : 0; }
b200lz4_ctx* b200lz4_mctx_ctx(b200lz4_mctx* m, int i) { return (m && i >= 0 && i < (int)m->ctx.size()) ? m->ctx[i] : nullptr; }
const char* b200lz4_mctx_last_error(b200lz4_mctx* m) { return m ? m->err.c_str() : ""; }

int b200lz4_compress_batch_multi(b200lz4_mctx* m, const void* src, int64_t src_bytes,
                                 const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                 const int32_t* stream_first, int n_streams,
                                 int acceleration, int header_mode,
                                 void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const Verdict v = check_batch(Entry::Multi, false, (m && !m->ctx.empty()) ? m : nullptr, n_blocks, header_mode, 0, src, src_bytes,
                                  src_off, src_len, dst, dst_off, out_len, stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) { if (dst_off) dst_off[0] = 0; return 0; }
    std::vector<int64_t> region(n_blocks + 1, 0);
    for (int i = 0; i < n_blocks; i++) region[i + 1] = region[i] + compress_cap(src_len[i], header_mode);
    if (region[n_blocks] > dst_cap) return fail(B200LZ4_E_NOMEM, "dst_cap too small: need " + std::to_string(region[n_blocks]));
    const uint8_t* hs = static_cast<const uint8_t*>(src);
    uint8_t* hd = static_cast<uint8_t*>(dst);
    return run_striped(m, src_off, src_len, n_blocks, stream_first, n_streams, region, dst_off, out_len,
        [&](b200lz4_ctx* c, int64_t lo, int64_t bytes, const int64_t* off, const int32_t* len, int nb, const int32_t* first, int ns,
            int64_t r0, int64_t rcap, int64_t* doff, int32_t* olen) {
            return compress_host(c, hs + lo, bytes, off, len, nb, first, ns, nullptr, acceleration, header_mode, nullptr, nullptr,
                                 hd + r0, rcap, doff, olen);
        });
}

int b200lz4_decompress_batch_multi(b200lz4_mctx* m, const void* src, int64_t src_bytes,
                                   const int64_t* src_off, const int32_t* src_len, int n_blocks,
                                   const int32_t* stream_first, int n_streams,
                                   int header_mode, int max_block,
                                   void* dst, int64_t dst_cap, int64_t* dst_off, int32_t* out_len)
{
    const Verdict v = check_batch(Entry::Multi, true, (m && !m->ctx.empty()) ? m : nullptr, n_blocks, header_mode, max_block, src,
                                  src_bytes, src_off, src_len, dst, dst_off, out_len, stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) { if (dst_off) dst_off[0] = 0; return 0; }
    const uint8_t* hs = static_cast<const uint8_t*>(src);
    uint8_t* hd = static_cast<uint8_t*>(dst);
    std::vector<int64_t> region(n_blocks + 1, 0);
    for (int i = 0; i < n_blocks; i++)
        region[i + 1] = region[i] + decode_slot(decode_cap(hs, src_off, src_len, i, header_mode, max_block), header_mode);
    if (region[n_blocks] > dst_cap) return fail(B200LZ4_E_NOMEM, "dst_cap too small: need " + std::to_string(region[n_blocks]));
    return run_striped(m, src_off, src_len, n_blocks, stream_first, n_streams, region, dst_off, out_len,
        [&](b200lz4_ctx* c, int64_t lo, int64_t bytes, const int64_t* off, const int32_t* len, int nb, const int32_t* first, int ns,
            int64_t r0, int64_t rcap, int64_t* doff, int32_t* olen) {
            return decompress_host(c, hs + lo, bytes, off, len, nb, first, ns, nullptr, header_mode, max_block, nullptr,
                                   hd + r0, rcap, doff, olen);
        });
}

}  // extern "C"

extern "C" {

// ---------------------------------------------------------------- device path

size_t b200lz4_cstate_bytes(void) { return sizeof(CState); }
size_t b200lz4_dstate_bytes(void) { return sizeof(DState); }
size_t b200lz4_scratch_bytes(void) { return kScratchBytes; }

int b200lz4_cstate_set_dict(void* d_state, void* d_dict_buf, uint32_t dict_cap, void* cuda_stream)
{
    if (!d_state) return fail(B200LZ4_E_ARG, "NULL state");
    return set_dict_fields(static_cast<CState*>(d_state), static_cast<uint8_t*>(d_dict_buf), dict_cap,
                           static_cast<cudaStream_t>(cuda_stream));
}

int b200lz4_compress_dev(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                         const int32_t* d_stream_first, int n_streams, void* const* d_states,
                         void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                         int acceleration, int header_mode, void* d_scratch, void* cuda_stream)
{
    const Verdict v = check_batch(Entry::Dev, false, d_scratch, n_blocks, header_mode, 0, d_src, 0, d_src_off, d_src_len, d_dst,
                                  d_dst_off, d_out_len, d_stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) return 0;
    CompressArgs a{};
    a.src = static_cast<const uint8_t*>(d_src); a.src_off = d_src_off; a.src_len = d_src_len; a.n_blocks = n_blocks;
    a.stream_first = d_stream_first; a.n_streams = d_stream_first ? n_streams : n_blocks; a.states = d_states;
    a.dst = static_cast<uint8_t*>(d_dst); a.dst_off = d_dst_off; a.dst_cap = d_dst_cap; a.out_len = d_out_len;
    a.accel = acceleration; a.header = header_mode; a.scratch = static_cast<Scratch*>(d_scratch);
    CU(launch_compress(a, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_decompress_dev(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                           const int32_t* d_stream_first, int n_streams, void* const* d_states,
                           void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                           int header_mode, int max_block, void* d_scratch, void* cuda_stream)
{
    const Verdict v = check_batch(Entry::Dev, true, d_scratch, n_blocks, header_mode, max_block, d_src, 0, d_src_off, d_src_len,
                                  d_dst, d_dst_off, d_out_len, d_stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) return 0;
    DecompressArgs a{};
    a.src = static_cast<const uint8_t*>(d_src); a.src_off = d_src_off; a.src_len = d_src_len; a.n_blocks = n_blocks;
    a.stream_first = d_stream_first; a.n_streams = d_stream_first ? n_streams : n_blocks; a.states = d_states;
    a.dst = static_cast<uint8_t*>(d_dst); a.dst_off = d_dst_off; a.dst_cap = d_dst_cap; a.out_len = d_out_len;
    a.header = header_mode; a.max_block = max_block; a.scratch = static_cast<Scratch*>(d_scratch);
    a.wide_arena = reinterpret_cast<uint4*>(static_cast<uint8_t*>(d_scratch) + sizeof(Scratch)); a.wide_ctas = kWideMaxCtas;
    CU(launch_decompress(a, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_dict_load_dev(const void* d_dict, int64_t len, void* d_cstate, void* d_dstate, void* cuda_stream)
{
    if (len < 0 || (len > 0 && !d_dict)) return fail(B200LZ4_E_ARG, "NULL dictionary or negative length");
    if (len > kMaxInput) return fail(B200LZ4_E_ARG, "dictionary longer than LZ4_MAX_INPUT_SIZE");
    CU(launch_load_dict(static_cast<const uint8_t*>(d_dict), len, static_cast<CState*>(d_cstate), static_cast<DState*>(d_dstate),
                        static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_compress_dev_dict(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                              const int32_t* d_stream_first, int n_streams, void* const* d_states, const void* d_dict_cstate,
                              void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                              int acceleration, int header_mode, void* d_scratch, void* cuda_stream)
{
    if (!d_dict_cstate) return fail(B200LZ4_E_ARG, "dictionary state is NULL");
    if (d_states) return fail(B200LZ4_E_ARG, "a dictionary together with stream records: load it into the records instead");
    const Verdict v = check_batch(Entry::Dev, false, d_scratch, n_blocks, header_mode, 0, d_src, 0, d_src_off, d_src_len, d_dst,
                                  d_dst_off, d_out_len, d_stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) return 0;
    CompressArgs a{};
    a.src = static_cast<const uint8_t*>(d_src); a.src_off = d_src_off; a.src_len = d_src_len; a.n_blocks = n_blocks;
    a.stream_first = d_stream_first; a.n_streams = d_stream_first ? n_streams : n_blocks;
    a.dst = static_cast<uint8_t*>(d_dst); a.dst_off = d_dst_off; a.dst_cap = d_dst_cap; a.out_len = d_out_len;
    a.accel = acceleration; a.header = header_mode; a.scratch = static_cast<Scratch*>(d_scratch);
    a.dict_state = static_cast<const CState*>(d_dict_cstate);
    CU(launch_compress(a, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_decompress_dev_dict(const void* d_src, const int64_t* d_src_off, const int32_t* d_src_len, int n_blocks,
                                const int32_t* d_stream_first, int n_streams, void* const* d_states, const void* d_dict_dstate,
                                void* d_dst, const int64_t* d_dst_off, const int32_t* d_dst_cap, int32_t* d_out_len,
                                int header_mode, int max_block, void* d_scratch, void* cuda_stream)
{
    if (!d_dict_dstate) return fail(B200LZ4_E_ARG, "dictionary state is NULL");
    if (d_states) return fail(B200LZ4_E_ARG, "a dictionary together with stream records: load it into the records instead");
    const Verdict v = check_batch(Entry::Dev, true, d_scratch, n_blocks, header_mode, max_block, d_src, 0, d_src_off, d_src_len,
                                  d_dst, d_dst_off, d_out_len, d_stream_first, n_streams, false);
    if (v.code) return fail(v);
    if (n_blocks == 0) return 0;
    DecompressArgs a{};
    a.src = static_cast<const uint8_t*>(d_src); a.src_off = d_src_off; a.src_len = d_src_len; a.n_blocks = n_blocks;
    a.stream_first = d_stream_first; a.n_streams = d_stream_first ? n_streams : n_blocks;
    a.dst = static_cast<uint8_t*>(d_dst); a.dst_off = d_dst_off; a.dst_cap = d_dst_cap; a.out_len = d_out_len;
    a.header = header_mode; a.max_block = max_block; a.scratch = static_cast<Scratch*>(d_scratch);
    a.wide_arena = reinterpret_cast<uint4*>(static_cast<uint8_t*>(d_scratch) + sizeof(Scratch)); a.wide_ctas = kWideMaxCtas;
    a.dict_state = static_cast<const DState*>(d_dict_dstate);
    CU(launch_decompress(a, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_compact_dev(const void* d_slots, const int64_t* d_slot_off, const int32_t* d_len, int n_blocks,
                        int header_mode, void* d_out, int64_t* d_out_off, void* d_scratch, void* cuda_stream)
{
    (void)d_scratch;
    if (n_blocks < 0) return fail(B200LZ4_E_ARG, "bad argument");
    CompactArgs g{static_cast<const uint8_t*>(d_slots), d_slot_off, d_len, n_blocks, header_mode,
                  static_cast<uint8_t*>(d_out), d_out_off, nullptr, nullptr};
    CU(launch_compact(g, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

// ------------------------------------------------------------------ checksums
int b200lz4_xxh32_dev(const void* d_buf, const int64_t* d_off, const int32_t* d_len, int n, uint32_t seed, uint32_t* d_out, void* cuda_stream)
{
    if (n < 0 || (n > 0 && (!d_buf || !d_off || !d_len || !d_out))) return fail(B200LZ4_E_ARG, "NULL argument");
    CU(launch_xxh32(static_cast<const uint8_t*>(d_buf), d_off, d_len, n, seed, d_out, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

int b200lz4_xxh32_batch(b200lz4_ctx* c, const void* src, int64_t src_bytes, const int64_t* off, const int32_t* len, int n,
                        uint32_t seed, uint32_t* out)
{
    if (!c) return fail(B200LZ4_E_ARG, "ctx is NULL");
    if (n < 0 || (n > 0 && (!off || !len || !out))) return fail(B200LZ4_E_ARG, "NULL argument");
    if (n == 0) return 0;
    const Verdict v = check_blocks(off, len, n, src_bytes);
    if (v.code) return fail(v);
    CU(cudaSetDevice(c->device));
    const DescLayout lay(n, 0, 0, 0, 0, 0, 0);     // out_len: the checksums
    int rc;
    if ((rc = ensure_desc(c, lay))) return rc;
    if ((rc = c->d_src.ensure((size_t)src_bytes + 64))) return rc;
    void* hd = c->h_desc.p;
    void* dd = c->d_desc.p;
    memcpy(lay.src_off_in(hd), off, sizeof(int64_t) * n); memcpy(lay.src_len_in(hd), len, sizeof(int32_t) * n);
    cudaStream_t st = c->stream;
    CU(cudaMemcpyAsync(dd, hd, lay.upload, cudaMemcpyHostToDevice, st));
    if (src_bytes) CU(cudaMemcpyAsync(c->d_src.p, src, (size_t)src_bytes, cudaMemcpyHostToDevice, st));
    CU(launch_xxh32(static_cast<const uint8_t*>(c->d_src.p), lay.src_off_in(dd), lay.src_len_in(dd), n, seed,
                    reinterpret_cast<uint32_t*>(lay.out_len_in(dd)), st));
    c->launches += 1;
    CU(cudaMemcpyAsync(lay.out_len_in(hd), lay.out_len_in(dd), sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    memcpy(out, lay.out_len_in(hd), sizeof(uint32_t) * n);
    return 0;
}

// ------------------------------------------------------------------ re-frame
// resizeChunksD's `process` (src/Streamly/Internal/LZ4.hs:459-484) applied to one contiguous range.
int b200lz4_reframe(const void* buf, int64_t len, int header_mode, int has_end_mark,
                    int64_t* block_off, int32_t* block_len, int64_t max_blocks,
                    int64_t* n_found, int64_t* consumed, int* ended)
{
    if (!n_found || !consumed || len < 0 || (len > 0 && !buf)) return fail(B200LZ4_E_ARG, "NULL argument");
    if (header_mode != 4 && header_mode != 8) return fail(B200LZ4_E_ARG, "header_mode must be 4 or 8");
    const uint8_t* p = static_cast<const uint8_t*>(buf);
    int64_t at = 0, k = 0;
    if (ended) *ended = 0;
    *n_found = 0; *consumed = 0;
    while (k < max_blocks) {
        int64_t rest = len - at;
        if (rest < 4) break;                                            // LZ4.hs:461-462
        int32_t comp = le32(p + at);
        if (has_end_mark && comp == 0) {                                // LZ4.hs:464-466 -> RFooter; footer is the 4 bytes themselves
            at += 4; if (ended) *ended = 1; break;
        }
        if (rest <= header_mode) break;                                 // LZ4.hs:468-469
        if (comp <= 0) { *n_found = k; *consumed = at; return fail(B200LZ4_E_FRAME, "block header with compLen <= 0"); }
        int64_t required = (int64_t)comp + header_mode;                 // LZ4.hs:474
        if (rest < required) break;                                     // LZ4.hs:477-478 (RAccumulate)
        if (block_off) block_off[k] = at;
        if (block_len) block_len[k] = (int32_t)required;
        k++; at += required;                                            // LZ4.hs:475-476, :479-484
    }
    *n_found = k; *consumed = at;
    return 0;
}

int b200lz4_reframe_dev(const void* d_buf, int64_t len, int header_mode, int has_end_mark,
                        int64_t* d_block_off, int32_t* d_block_len, int64_t max_blocks,
                        int64_t* d_result, void* cuda_stream)
{
    if (!d_result || len < 0 || (len > 0 && !d_buf) || max_blocks < 0 || (max_blocks > 0 && (!d_block_off || !d_block_len)))
        return fail(B200LZ4_E_ARG, "NULL argument");
    if (header_mode != 4 && header_mode != 8) return fail(B200LZ4_E_ARG, "header_mode must be 4 or 8");
    CU(launch_reframe(static_cast<const uint8_t*>(d_buf), len, header_mode, has_end_mark, d_block_off, d_block_len, max_blocks,
                      d_result, static_cast<cudaStream_t>(cuda_stream)));
    return 0;
}

// ------------------------------------------------------------ legacy aliases

struct LZ4_stream_u { b200lz4_cstream* s; };
struct LZ4_streamDecode_u { b200lz4_dstream* s; };

static std::mutex g_legacy_mu;
static b200lz4_ctx* g_legacy_ctx = nullptr;
static b200lz4_ctx* legacy_ctx()
{
    if (!g_legacy_ctx) {
        int dev = 0;
        if (const char* e = getenv("B200LZ4_DEVICE")) dev = atoi(e);
        if (b200lz4_ctx_create(dev, &g_legacy_ctx) != 0) {
            fprintf(stderr, "libb200lz4: %s\n", g_err.c_str());
            return nullptr;
        }
    }
    return g_legacy_ctx;
}

LZ4_stream_t* LZ4_createStream(void)
{
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_ctx* c = legacy_ctx();
    if (!c) return nullptr;
    LZ4_stream_u* h = new (std::nothrow) LZ4_stream_u{nullptr};
    if (!h) return nullptr;
    if (b200lz4_cstream_create(c, &h->s) != 0) { delete h; return nullptr; }
    return h;
}
int LZ4_freeStream(LZ4_stream_t* h)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_cstream_free(h->s); delete h;
    return 0;
}
LZ4_streamDecode_t* LZ4_createStreamDecode(void)
{
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_ctx* c = legacy_ctx();
    if (!c) return nullptr;
    LZ4_streamDecode_u* h = new (std::nothrow) LZ4_streamDecode_u{nullptr};
    if (!h) return nullptr;
    if (b200lz4_dstream_create(c, &h->s) != 0) { delete h; return nullptr; }
    return h;
}
int LZ4_freeStreamDecode(LZ4_streamDecode_t* h)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_dstream_free(h->s); delete h;
    return 0;
}
int LZ4_compressBound(int n) { return bound_of(n); }

int LZ4_compress_fast_continue(LZ4_stream_t* h, const char* src, char* dst, int srcSize, int dstCapacity, int acceleration)
{
    if (!h || !h->s || srcSize < 0 || !dst) return 0;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    int64_t off = 0, dst_off[2] = {0, 0}; int32_t len = srcSize, out_len = 0, cap = dstCapacity, first[2] = {0, 1};
    static const char empty = 0;
    std::vector<char> tmp((size_t)bound_of(srcSize) + 16);
    b200lz4_cstream* ss = h->s;
    int rc = compress_host(ss->ctx, srcSize ? src : &empty, srcSize, &off, &len, 1, first, 1, &ss,
                           acceleration, 0, &cap, nullptr, tmp.data(), (int64_t)tmp.size(), dst_off, &out_len);
    if (rc != 0 || out_len <= 0 || out_len > dstCapacity) return 0;
    memcpy(dst, tmp.data(), (size_t)out_len);
    return out_len;
}

int LZ4_decompress_safe_continue(LZ4_streamDecode_t* h, const char* src, char* dst, int srcSize, int dstCapacity)
{
    if (!h || !h->s || !src || srcSize < 0 || dstCapacity < 0) return -1;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    int64_t off = 0, dst_off[2] = {0, 0}; int32_t len = srcSize, out_len = -1, first[2] = {0, 1};
    std::vector<char> tmp((size_t)dstCapacity + 16);
    b200lz4_dstream* ss = h->s;
    int rc = decompress_host(ss->ctx, src, srcSize, &off, &len, 1, first, 1, &ss, 0, dstCapacity, nullptr,
                             tmp.data(), (int64_t)tmp.size(), dst_off, &out_len);
    if (rc != 0 && rc != B200LZ4_E_BLOCK) return -1;
    if (out_len > 0) memcpy(dst, tmp.data() + dst_off[0], (size_t)out_len);
    return out_len;
}

// LZ4_loadDict / LZ4_setStreamDecode: the dictionary is loaded on the device and copied into the stream, so the caller's
// buffer is not referenced afterwards (upstream keeps pointing at it; either way it must not change before the next call)
int LZ4_loadDict(LZ4_stream_t* h, const char* dict, int size)
{
    if (!h || !h->s) return 0;
    if (size < 0 || !dict) size = 0;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_dict* d = nullptr;
    if (b200lz4_dict_create(h->s->ctx, dict, size, &d) != 0) return 0;
    const int rc = b200lz4_cstream_load_dict(h->s, d);
    b200lz4_dict_free(d);
    if (rc != 0) return 0;
    return size < 8 ? 0 : std::min(size, 65536);
}

int LZ4_setStreamDecode(LZ4_streamDecode_t* h, const char* dict, int size)
{
    if (!h || !h->s) return 0;
    if (size < 0 || !dict) size = 0;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    b200lz4_dict* d = nullptr;
    if (b200lz4_dict_create(h->s->ctx, dict, size, &d) != 0) return 0;
    const int rc = b200lz4_dstream_set_dict(h->s, d);
    b200lz4_dict_free(d);
    return rc == 0 ? 1 : 0;
}

}  // extern "C"
