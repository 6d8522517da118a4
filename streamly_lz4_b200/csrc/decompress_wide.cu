// decompress_wide.cu -- LZ4 decoder for FEW streams (linked streams, a handful of large blocks): one stream per SM.
//
// Why a second kernel.  The narrow kernel (decompress.cu) gives a stream one parser warp and one copier warp, and a
// linked stream is one chain (block N's matches may read block N-1's output, cbits/lz4.c:2322-2359, :2075-2100), so
// config 4's 128 streams occupy 256 warps of a machine that holds 9 472.  Measured (profiles/r2a_*): the chain is
// PARSER-bound -- with the copier's copies switched off it runs only 10-40 % faster.  But a block's token chain does not
// depend on any other block; only match COPIES do.  So here
//
//   8 PARSER warps   parse blocks N, N+1, .. N+7 of the stream at the same time (the unchanged parse_block, all safe-
//                    decoder rules; the one rule that needs the previous block's length, cbits/lz4.c:2073, is deferred:
//                    the parser reports how far before its block a match reaches, the dispatcher compares).  Each
//                    parser writes 32-descriptor batches into its own ring in GLOBAL memory (256 batches, a whole
//                    64 KiB block: L2-resident) and a 16-byte batch header into a shared-memory ring.
//   1 DISPATCHER warp hands batches out strictly in stream order as numbered tickets (which parser's ring is next, the
//                    batch's absolute output position, flow control, in-order retirement, stream begin / end).
//   13 COPIER warps  in four roles that form a pipeline over the tickets.  The stream's last 128 KiB of output live in a
//                    shared-memory ring indexed by stream position.
//       L (6 warps)  literals: descriptor batch -> shared memory, the batch's compressed bytes -> staging (one coalesced
//                    pass, range given by the parser), every lane copies the literals of its sequence into the ring.
//                    No dependencies at all, so L runs ahead.
//       F (4 warps)  FAR matches, lane-parallel: a match of ticket t whose source ends below the start of ticket t - 2
//                    only reads bytes that are final once the serial stage has finished ticket t - 3.
//       N (1 warp)   NEAR matches (everything else: sources inside the last two batches, overlapping runs, records), in
//                    stream order, each copied by all 32 lanes -- the narrow kernel's phase B.  This is the stream's one
//                    serial chain; it carries only the matches that really depend on recent output.  Long match pieces
//                    run here too.
//       G (2 warps)  flush finished batches to global memory with 128-bit stores and report completion.
//
// Flow control: a batch may only be handed out while its end is less than 60 KiB ahead of the in-order completion
// frontier (the ring holds 128 KiB, matches reach 64 KiB back) and fewer than 16 tickets are in flight (their descriptor
// batches sit in shared memory); long sequences are cut into pieces of 16 KiB by the parser so that every batch is small
// against that window.
#include <cstdlib>
#include "decode_common.cuh"

namespace b200lz4 {

using namespace dec;

namespace {

constexpr int kWP = kWideParsers;                 // parser warps
constexpr int kWL = 6, kWF = 4, kWG = 2;           // copier warps per role: literals, far matches, flush (+ one serial warp N)
constexpr int kWC = kWL + kWF + 1 + kWG;
constexpr int kWThreads = (kWP + 1 + kWC) * 32;   // + the dispatcher warp
#ifndef B200LZ4_WIDE_DEPTH
#define B200LZ4_WIDE_DEPTH 2
#endif
constexpr int kWDepth = B200LZ4_WIDE_DEPTH;       // a match is FAR if its source ends below the start of the ticket kWDepth before its own
constexpr int kWSlots = 16;                       // descriptor batches resident in shared memory = tickets in flight
constexpr uint32_t kWOut = 131072, kWM = kWOut - 1;      // output ring (bytes), indexed by stream position
constexpr int kWR = kWideRingBatches;             // batches per parser ring
constexpr int kWStage = 1216;                     // per copier: staging of one batch's compressed bytes (32 x (token + 1 + 32 literals + offset + 1) + alignment)
constexpr int kWIn = 2048;                        // per parser: input ring
constexpr int kTickets = 64;                      // completion flags (ring)
constexpr int kRunAhead = 61440;                  // a batch may end at most this far beyond the completion frontier
constexpr uint32_t kPiece = 16384;                // long sequences are cut into pieces of this many output bytes
constexpr uint32_t kSeedBase = 65536;             // stream position of the first output byte after (re)seeding

// Cycle accounting for development builds (make stats -> build/libb200lz4_stats.so; tools/linked_probe.py --stats): every
// warp adds its clock64() intervals to 64-bit counters in the scratch block's padding.  Compiled out of the product.
#ifdef B200LZ4_WIDE_STATS
#define WSTAT_DECL(n) unsigned long long wst_[n] = {0}; long long wst_t_ = clock64();
#define WSTAT(i) { const long long now_ = clock64(); wst_[i] += (unsigned long long)(now_ - wst_t_); wst_t_ = now_; }
#define WSTAT_COUNT(i, n) { wst_[i] += (unsigned long long)(n); }
#define WSTAT_FLUSH(a, base, n) { if (lane_id() == 0) for (int q_ = 0; q_ < (n); q_++) atomicAdd(reinterpret_cast<unsigned long long*>((a).scratch->pad_) + (base) + q_, wst_[q_]); }
#else
#define WSTAT_DECL(n)
#define WSTAT(i)
#define WSTAT_COUNT(i, n)
#define WSTAT_FLUSH(a, base, n)
#endif

struct WTicket { uint32_t jn, cf, op_start, base, valid_lo; int blk; uint32_t safe, aux; };   // 32 bytes; jn = parser << 16 | ring slot; safe: everything below is final for stage F

struct WCtl {                                     // shared memory
    uint32_t pad0_;
    uint32_t finished;                            // dispatcher: no more tickets will be issued
    uint32_t t_final;                             // ... and this many were
    uint32_t pad_;
    uint32_t rd[kWP];                             // dispatcher: next batch of each parser ring to hand out
    uint32_t wr_pub[kWP];                         // parsers: batches published
    uint32_t cons[kWP];                           // dispatcher: batches retired (parsers wait on it for ring space)
    // One mbarrier per ticket slot and pipeline edge (count 1; ticket t uses phase (t / 64) & 1 of slot t % 64).  Waiting on an
    // mbarrier suspends the warp in hardware; polling flags with nanosleep() instead let a dozen idle warps issue more
    // instructions than the working ones (ncu: 11 G of 14 G warp instructions were polls).
    unsigned long long bar_ticket[kTickets];      // dispatcher -> all stages: ticket t has been issued
    unsigned long long bar_lit[kTickets];         // stage L -> F: descriptors in shared memory, literals in the ring
    unsigned long long bar_far[kTickets];         // stage F -> N
    unsigned long long bar_near[kTickets];        // stage N -> F (ticket t + kWDepth + 1 may copy its far matches) and G
    uint32_t near_mask[kWSlots], near_long[kWSlots];      // stage F -> N: which sequences of the batch have a near match / the batch is a long match piece
    uint32_t done[kTickets];                      // stage G: ticket t is in global memory <=> done[t % 64] == t + 1
    uint32_t tend[kTickets], tn[kTickets], tj[kTickets];      // dispatcher-private: end position / ring slot / parser of a ticket
    WTicket ticket[kTickets];
};

__device__ __forceinline__ uint32_t vld(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ void vst(uint32_t* p, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(p) = v; }
__device__ __forceinline__ uint4 ld_cg_128(const uint4* p)
{ uint4 v; asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory"); return v; }

// ------------------------------------------------------------- ring <-> global ----
__device__ __forceinline__ uint32_t rix(uint32_t out_s, uint32_t pos) { return out_s + (pos & kWM); }

// n bytes of global memory -> ring positions [pos, pos + n); all lanes, identical arguments.  Four loads in flight
// per lane (a serial chain of this warp: latency, not bandwidth, is what it pays for).
template <bool kReadOnly>
__device__ __forceinline__ void copy_g2r(uint32_t out_s, uint32_t pos, const uint8_t* src, uint32_t n)
{
    const uint32_t lane = lane_id();
    uint32_t head = (4u - (pos & 3u)) & 3u;
    if (head > n) head = n;
    if (lane < head) sts8(rix(out_s, pos + lane), kReadOnly ? (uint32_t)__ldg(src + lane) : (uint32_t)src[lane]);
    pos += head; src += head; n -= head;
    const uint32_t nw = n >> 2;
    auto ld = [&](uint32_t w) { return kReadOnly ? ldg_u32_unaligned(src + 4u * w) : ld_u32_unaligned(src + 4u * w); };
    uint32_t w = lane;
    for (; w + 96u < nw; w += 128u) {
        const uint32_t a = ld(w), b = ld(w + 32u), c = ld(w + 64u), d = ld(w + 96u);
        sts32(rix(out_s, pos + 4u * w), a); sts32(rix(out_s, pos + 4u * (w + 32u)), b);
        sts32(rix(out_s, pos + 4u * (w + 64u)), c); sts32(rix(out_s, pos + 4u * (w + 96u)), d);
    }
    for (; w < nw; w += 32u) sts32(rix(out_s, pos + 4u * w), ld(w));
    const uint32_t done = nw << 2, tail = n - done;
    if (lane < tail) sts8(rix(out_s, pos + done + lane), kReadOnly ? (uint32_t)__ldg(src + done + lane) : (uint32_t)src[done + lane]);
}

// ring positions [pos, pos + n) -> global memory at gdst (128-bit stores; the ring is read in aligned words)
__device__ __forceinline__ void flush_r2g(uint32_t out_s, uint8_t* gdst, uint32_t pos, uint32_t n)
{
    const uint32_t lane = lane_id();
    uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(gdst) & 15)) & 15);
    if (head > n) head = n;
    if (lane < head) gdst[lane] = (uint8_t)lds8(rix(out_s, pos + lane));
    gdst += head; pos += head; n -= head;
    const uint32_t nvec = n >> 4;
    uint4* gv = reinterpret_cast<uint4*>(gdst);
    if ((pos & 15u) == 0) {
        uint32_t v = lane;
        for (; v + 32u < nvec; v += 64u) {
            const uint4 a = lds128(rix(out_s, pos + 16u * v)), b = lds128(rix(out_s, pos + 16u * (v + 32u)));
            gv[v] = a; gv[v + 32u] = b;
        }
        for (; v < nvec; v += 32u) gv[v] = lds128(rix(out_s, pos + 16u * v));
    } else {
        const uint32_t sh = (pos & 3u) * 8u;
        for (uint32_t v = lane; v < nvec; v += 32) {
            const uint32_t a = (pos + 16u * v) & ~3u;
            const uint32_t x0 = lds32(rix(out_s, a)), x1 = lds32(rix(out_s, a + 4)), x2 = lds32(rix(out_s, a + 8)), x3 = lds32(rix(out_s, a + 12));
            const uint32_t x4 = sh ? lds32(rix(out_s, a + 16)) : 0u;
            gv[v] = make_uint4(__funnelshift_r(x0, x1, sh), __funnelshift_r(x1, x2, sh), __funnelshift_r(x2, x3, sh), __funnelshift_r(x3, x4, sh));
        }
    }
    const uint32_t done = nvec << 4, tail = n - done;
    if (lane < tail) gdst[done + lane] = (uint8_t)lds8(rix(out_s, pos + done + lane));
}

// One lane copies n bytes to ring position dst from shared address space `src_s` at byte offset `src` masked by
// `smask` (the ring itself, or the staging buffer with an all-ones mask): four bytes per step (two aligned word loads, a
// funnel shift, four byte stores that need not wait for each other), then the odd bytes.  The source may overlap the
// destination from below by 4 bytes or more (an LZ4 match with offset >= 4).
__device__ __forceinline__ void lane_copy4(uint32_t out_s, uint32_t dst, uint32_t src_s, uint32_t src, uint32_t smask, uint32_t n)
{
    uint32_t i = 0;
    for (; i + 4u <= n; i += 4u) {
        const uint32_t a = src + i, al = a & ~3u;
        const uint32_t w0 = lds32(src_s + (al & smask)), w1 = lds32(src_s + ((al + 4u) & smask));
        const uint32_t v = __funnelshift_r(w0, w1, (a & 3u) * 8u);
        sts8(rix(out_s, dst + i), v & 0xFFu); sts8(rix(out_s, dst + i + 1u), (v >> 8) & 0xFFu);
        sts8(rix(out_s, dst + i + 2u), (v >> 16) & 0xFFu); sts8(rix(out_s, dst + i + 3u), v >> 24);
    }
    for (; i < n; i++) sts8(rix(out_s, dst + i), lds8(src_s + ((src + i) & smask)));
}

// A long match piece inside the ring, all lanes: rounds of one period each (the period's source is complete before
// the round starts; several periods per round once they have been written); periods below 32 are replicated from
// registers.
__device__ __forceinline__ void coop_long_match(uint32_t out_s, uint32_t dst, uint32_t len, uint32_t dist)
{
    const uint32_t lane = lane_id();
    const uint32_t src = dst - dist;
    if (dist >= 32u) {
        const uint32_t kmax = dist < 4096u ? 4096u / dist : 1u;
        uint32_t done = 0;                              // bytes [0, done) written
        while (done < len) {
            uint32_t k = (done + dist) / dist;          // whole periods available below dst + done: any multiple of dist is a valid offset
            if (k > kmax) k = kmax;
            const uint32_t P = k * dist;
            const uint32_t n = min(P, len - done);
            for (uint32_t i = lane; i < n; i += 32) sts8(rix(out_s, dst + done + i), lds8(rix(out_s, dst + done + i - P)));
            __syncwarp();
            done += n;
        }
    } else {
        const uint32_t pat = lds8(rix(out_s, src + (lane < dist ? lane : 0u)));
        uint32_t k = lane % dist;
        const uint32_t adv = 32u % dist;
        for (uint32_t i0 = 0; i0 < len; i0 += 32) {
            const uint32_t bb = __shfl_sync(kFull, pat, k);
            if (i0 + lane < len) sts8(rix(out_s, dst + i0 + lane), bb);
            k += adv; if (k >= dist) k -= dist;
        }
    }
}

// (re)start the ring at stream position kSeedBase: the dictionary (at most 64 KiB) lies right-aligned below it
__device__ void wseed(uint32_t out_s, const uint8_t* tail_src, uint32_t kept)
{
    if (kept) copy_g2r<false>(out_s, kSeedBase - kept, tail_src, kept);
    __threadfence_block();
    __syncwarp();
}

// ------------------------------------------------------------------ parser sink ----
struct WParser {
    static constexpr bool kWide = true;
    static constexpr int kRing = kWIn;
    uint32_t ring_s;            // shared address of this parser's input ring
    const uint8_t* gbase;       // global address of ring-space position 0
    int end, issued_end, ready_end, cur_start;
    uint4* gring;               // this parser's descriptor ring (global memory)
    uint32_t hdr_s;             // shared address of its header ring: {count | flags, first output position, end position, reach}
    uint32_t* wr_pub; uint32_t* cons;
    uint32_t batch;             // batches published so far
    int fill, flags;
    int op_start, op_end;       // block-relative output range of the batch being filled
    int need;                   // bytes before the block start the furthest-reaching match reads (deferred cbits/lz4.c:2073)
#ifdef B200LZ4_WIDE_STATS
    unsigned long long ring_wait = 0;
#endif

    __device__ __forceinline__ uint32_t at(int p) const { return lds8(ring_s + ((uint32_t)p & (kRing - 1))); }
    __device__ __forceinline__ void begin()
    {   // the ring slot of this batch must have been retired
#ifdef B200LZ4_WIDE_STATS
        const long long w0_ = clock64();
#endif
        while (batch - vld(cons) >= (uint32_t)kWR) __nanosleep(2000);      // (a full ring is >= 200 us of copier work)
#ifdef B200LZ4_WIDE_STATS
        ring_wait += (unsigned long long)(clock64() - w0_);
#endif
        fill = 0;
    }
    __device__ __forceinline__ uint4* slot() const { return gring + (size_t)(batch & (kWR - 1)) * 32; }
    __device__ __forceinline__ void put(uint32_t rank, uint32_t x, uint32_t y, uint32_t z, uint32_t w) { slot()[fill + rank] = make_uint4(x, y, z, w); }
    __device__ __forceinline__ void advance(int n, int op_after) { fill += n; op_end = op_after; }
    __device__ __forceinline__ void push(uint32_t x, uint32_t y, uint32_t z, uint32_t w, int op_after)
    {
        if (lane_id() == 0) slot()[fill] = make_uint4(x, y, z, w);
        fill++; op_end = op_after;
    }
    __device__ __forceinline__ void note_reach(int r) { need = r > need ? r : need; }
    __device__ void publish(int extra, int result, int ip)
    {
        uint32_t cf = (uint32_t)(fill | flags | extra);
        if ((extra & kEndBlock) && result < 0) cf |= (uint32_t)kFailed;
        if (extra & kEndBlock) cp_async_wait_all();      // nothing of this block's input may land after the next block starts
        __threadfence();                                 // descriptor stores (several lanes) before the header
        __syncwarp();
        uint32_t aux = (uint32_t)need;
        if (!(extra & (kEndBlock | kBulk))) {            // where the batch's literals lie: [cur_start, ip) of the payload, in 16-byte vectors
            const uint32_t lo = (uint32_t)cur_start & ~15u, nv = ((uint32_t)ip - lo + 15u) >> 4;
            aux = lo;
            if (nv <= (uint32_t)(kWStage / 16)) cf |= nv << 8;
        }
        if (lane_id() == 0) {
            sts128(hdr_s + 16u * (batch & (kWR - 1)), cf, (uint32_t)op_start, (uint32_t)op_end, aux);
            __threadfence_block();
            vst(wr_pub, batch + 1);
        }
        batch++;
        flags = 0; op_start = op_end; cur_start = ip;
        begin();
    }
    // a long sequence: pieces of at most kPiece output bytes, one batch each (descriptor: literal start, literals, match bytes, offset)
    __device__ void push_bulk(uint32_t lit_src, uint32_t lit, uint32_t mlen, uint32_t dist, int op_seq, int ip_after)
    {
        int op = op_seq;
        while (lit) {
            const uint32_t n = lit < kPiece ? lit : kPiece;
            op_start = op;
            push(lit_src, n, 0u, 0u, op + (int)n);
            publish(kBulk, 0, ip_after);
            lit_src += n; lit -= n; op += (int)n;
        }
        while (mlen) {
            const uint32_t n = mlen < kPiece ? mlen : kPiece;
            op_start = op;
            push(0u, 0u, n, dist, op + (int)n);
            publish(kBulk, 0, ip_after);
            mlen -= n; op += (int)n;
        }
    }
    __device__ __forceinline__ void top_up(int ip)
    {   // only this warp reads its ring, and it never looks back: 1.5 KiB ahead always fits the 2 KiB ring
        while (issued_end < end && issued_end - ip < 1024) {
            const int p = issued_end + 16 * (int)lane_id();
            if (p < end) cp_async_16(ring_s + ((uint32_t)p & (kRing - 1)), gbase + p);
            cp_async_commit();
            issued_end += kFill;
        }
    }
    __device__ void ensure(int ip, int need_pos)
    {
        if (need_pos <= ready_end) return;
        if (ip >= issued_end) {                         // jumped over everything requested so far: restart at ip
            cp_async_wait_all();
            issued_end = ip & ~(kFill - 1);
            ready_end = issued_end;
        }
        top_up(ip);
        cp_async_wait_all();
        __syncwarp();
        ready_end = issued_end;
    }
};

__device__ void wparser_main(const DecompressArgs& a, int j, WCtl* ctl, uint32_t ring_s, uint32_t hdr_s, uint4* gring)
{
    WParser P;
    P.ring_s = ring_s; P.gbase = nullptr; P.end = P.issued_end = P.ready_end = P.cur_start = 0;
    P.gring = gring; P.hdr_s = hdr_s; P.wr_pub = &ctl->wr_pub[j]; P.cons = &ctl->cons[j];
    P.batch = 0; P.fill = 0; P.flags = 0; P.op_start = P.op_end = 0; P.need = 0;
#ifdef B200LZ4_WIDE_STATS
    const long long p0_ = clock64();
#endif
    for (int s = blockIdx.x; s < a.n_streams; s += gridDim.x) {
        const int b0 = stream_begin(a, s), b1 = stream_end(a, s, b0);
        for (int b = b0 + j; b < b1; b += kWP) {        // block (b - b0) of a stream belongs to parser (b - b0) % 8
            const BlockGeom g = block_geom(a, b);
            P.flags = kBegin; P.need = 0; P.op_start = P.op_end = 0;
            int r = -1;
            if (g.ok) {
                const int skew = (int)(reinterpret_cast<uintptr_t>(g.payload) & 15);
                P.gbase = g.payload - skew;
                r = parse_block(P, skew, g.comp_len, g.cap, 0u);
            }
            P.publish(kEndBlock, r, 0);
        }
    }
#ifdef B200LZ4_WIDE_STATS
    if (lane_id() == 0) {
        unsigned long long* st = reinterpret_cast<unsigned long long*>(a.scratch->pad_);
        atomicAdd(st + 0, (unsigned long long)(clock64() - p0_)); atomicAdd(st + 1, P.ring_wait); atomicAdd(st + 2, (unsigned long long)P.batch);
    }
#endif
}

// ------------------------------------------------------------------ dispatcher ----
// One warp; every lane runs the same scalar code on the same shared-memory words (loads broadcast, stores coincide), the
// cooperative parts (seeding the ring, keeping the stream tail) use all lanes.
struct WDispatch {
    WCtl* c;
    uint32_t T, F, fpos;        // tickets issued / retired in order; stream position below which all output is final

    // retire finished tickets in order; free their ring slots for the parsers
    __device__ __forceinline__ void advance()
    {
        while (F != T && vld(&c->done[F & (kTickets - 1)]) == F + 1) {
            const uint32_t k = F & (kTickets - 1);
            fpos = vld(&c->tend[k]);
            vst(&c->cons[vld(&c->tj[k])], vld(&c->tn[k]) + 1);
            F++;
        }
    }
    __device__ __forceinline__ void drain()
    {
        for (;;) { advance(); if (F == T) break; __nanosleep(100); }
        __threadfence_block();
    }
};

__device__ void wdispatch_main(const DecompressArgs& a, WCtl* ctl, uint32_t out_s, uint32_t hdrs_s)
{
    const uint32_t lane = lane_id();
    WDispatch D{ctl, 0u, 0u, kSeedBase};
    WSTAT_DECL(4)       // 0 other, 1 waiting for the parser, 2 waiting for flow control, 3 stream open / close
    for (int s = blockIdx.x; s < a.n_streams; s += gridDim.x) {
        const int b0 = stream_begin(a, s), b1 = stream_end(a, s, b0);
        DState* st = a.states ? reinterpret_cast<DState*>(a.states[s]) : nullptr;
        const DState* init = a.states ? st : a.dict_state;              // what the stream starts from: its record, or the dictionary's
        // ---- open the stream: the ring restarts at kSeedBase with the kept tail of the previous call as dictionary
        WSTAT(0)
        D.drain();
        uint32_t dict_len = 0, kept = 0;
        if (init && init->prev_len) { dict_len = init->prev_len; kept = init->kept; wseed(out_s, init->tail + 65536 - kept, kept); }
        else wseed(out_s, nullptr, 0u);
        uint32_t base = kSeedBase, valid_lo = kSeedBase - kept;
        D.fpos = kSeedBase;
        uint32_t hist[kWDepth];                                          // start positions of the last kWDepth tickets (nothing in flight: all final)
        #pragma unroll
        for (int q = 0; q < kWDepth; q++) hist[q] = kSeedBase;
        const uint8_t* last_out = nullptr; int last_len = 0;
        WSTAT(3)
        for (int blk = b0; blk < b1; blk++) {
            const uint32_t j = (uint32_t)(blk - b0) % (uint32_t)kWP;
            for (;;) {                                                      // the batches of this block, in order
                const uint32_t n = vld(&ctl->rd[j]);
                WSTAT(0)
                while (vld(&ctl->wr_pub[j]) == n) { D.advance(); __nanosleep(20); }    // (retiring slots may be what a parser waits for)
                WSTAT(1)
                __threadfence_block();
                const uint4 h = lds128(hdrs_s + (j * kWR + (n & (kWR - 1))) * 16u);
                const uint32_t e = base + h.z;
                // flow control: the ring holds 128 KiB and matches reach 64 KiB back, so nothing may be written more than
                // 60 KiB beyond the completion frontier; ticket slots are reused after 64
                for (;;) {
                    D.advance();
                    if ((int)(e - D.fpos) <= kRunAhead && D.T - D.F < (uint32_t)(kWSlots - 1)) break;
                    __nanosleep(20);
                }
                WSTAT(2)
                const uint32_t k = D.T & (kTickets - 1);
                vst(&ctl->tend[k], e); vst(&ctl->tj[k], j); vst(&ctl->tn[k], n);
                if (lane == 0) {
                    WTicket* tk = &ctl->ticket[k];
                    tk->jn = (j << 16) | (n & (kWR - 1)); tk->cf = h.x; tk->op_start = h.y; tk->base = base; tk->valid_lo = valid_lo; tk->blk = blk; tk->safe = hist[kWDepth - 1]; tk->aux = h.w;
                    __threadfence_block();
                    mbar_arrive(&ctl->bar_ticket[k]);
                }
                __syncwarp();
                D.T++;
                vst(&ctl->rd[j], n + 1);
                #pragma unroll
                for (int q = kWDepth - 1; q > 0; q--) hist[q] = hist[q - 1];
                hist[0] = base + h.y;
                if ((int)h.x & kEndBlock) {
                    int r = ((int)h.x & kFailed) ? -1 : (int)h.z;
                    if (r >= 0 && dict_len < 65536u && h.w > dict_len) r = -1;      // cbits/lz4.c:2073, deferred: a match reached below the dictionary
                    if (lane == 0) a.out_len[blk] = r;
                    if (r > 0) {                                            // cbits/lz4.c:2353-2355: this output is the next dictionary
                        base += (uint32_t)r; dict_len = (uint32_t)r;
                        valid_lo = base - ((uint32_t)r < 65536u ? (uint32_t)r : 65536u);
                        last_out = a.dst + a.dst_off[blk]; last_len = r;
                    } else if (r < 0 && blk + 1 < b1) {
                        // what the failed block wrote into the ring is garbage: restart the ring from the last good output
                        // (which stays the dictionary), taken from global memory
                        D.drain();
                        kept = 0; dict_len = 0;
                        if (last_out) {
                            dict_len = (uint32_t)last_len; kept = dict_len < 65536u ? dict_len : 65536u;
                            wseed(out_s, last_out + last_len - kept, kept);
                        } else if (init && init->prev_len) {
                            dict_len = init->prev_len; kept = init->kept;
                            wseed(out_s, init->tail + 65536 - kept, kept);
                        } else wseed(out_s, nullptr, 0u);
                        base = kSeedBase; valid_lo = kSeedBase - kept; D.fpos = kSeedBase;
                        #pragma unroll
                        for (int q = 0; q < kWDepth; q++) hist[q] = kSeedBase;
                    }
                    break;
                }
            }
        }
        // ---- close the stream: keep the reachable tail of the last output for the next call
        if (st && last_out) {
            D.drain();
            const uint32_t kp = last_len < 65536 ? (uint32_t)last_len : 65536u;
            warp_copy_rw(st->tail + 65536 - kp, last_out + last_len - kp, kp);
            __syncwarp();
            if (lane == 0) { st->prev_len = (uint32_t)last_len; st->kept = kp; }
        }
    }
    D.drain();
    vst(&ctl->t_final, D.T);
    __threadfence_block();
    vst(&ctl->finished, 1u);
    WSTAT(3)
    WSTAT_FLUSH(a, 4, 4)
}

// ---------------------------------------------------------------------- copiers ----
// one attempt to wait (suspended in hardware for up to ~1 us) for the phase of ticket t on its slot's barrier
__device__ __forceinline__ bool bar_try(unsigned long long* bars, uint32_t t)
{ return mbar_try_wait(smem_u32(&bars[t & (kTickets - 1)]), (t >> 6) & 1u, 1000u); }
__device__ __forceinline__ void bar_wait(unsigned long long* bars, uint32_t t) { while (!bar_try(bars, t)) { } }
// all lanes' earlier writes, then one arrival for ticket t
__device__ __forceinline__ void bar_signal(unsigned long long* bars, uint32_t t)
{
    __threadfence_block();
    __syncwarp();
    if (lane_id() == 0) mbar_arrive(&bars[t & (kTickets - 1)]);
}
// wait until ticket t has been issued; false: the dispatcher has finished and never issued it
__device__ __forceinline__ bool wait_ticket(WCtl* ctl, uint32_t t)
{
    while (!bar_try(ctl->bar_ticket, t))
        if (vld(&ctl->finished) && (int)(t - vld(&ctl->t_final)) >= 0) return false;
    return true;
}
struct WTk { uint32_t j, slot, base, op_start, valid_lo, safe, aux; int cf, blk; };
__device__ __forceinline__ WTk read_ticket(WCtl* ctl, uint32_t t)
{
    const uint32_t a = smem_u32(&ctl->ticket[t & (kTickets - 1)]);
    const uint4 x = lds128(a), y = lds128(a + 16u);
    WTk k; k.j = x.x >> 16; k.slot = x.x & 0xFFFFu; k.cf = (int)x.y; k.op_start = x.z; k.base = x.w;
    k.valid_lo = y.x; k.blk = (int)y.y; k.safe = y.z; k.aux = y.w;
    return k;
}

// stage L: descriptors into shared memory, literals into the ring (tickets w, w + kWL, ...)
__device__ void wstage_literals(const DecompressArgs& a, int w, WCtl* ctl, uint32_t out_s, uint32_t desc_s, uint32_t stage_s, const uint4* garena)
{
    constexpr uint32_t M = kWM;
    const uint32_t lane = lane_id();
    int cached_blk = -1; const uint8_t* blk_gbase = nullptr;
    WSTAT_DECL(4)       // 0 waiting for a ticket, 1 loads, 2 copy, 3 tickets
    for (uint32_t t = (uint32_t)w;; t += kWL) {
        if (!wait_ticket(ctl, t)) break;
        WSTAT(0) WSTAT_COUNT(3, 1)
        const WTk k = read_ticket(ctl, t);
        const int cnt = k.cf & 0xFF;
        uint32_t nvec = ((uint32_t)k.cf >> 8) & 0xFFu, lo = k.aux;       // where the batch's literals lie (0 vectors: not given)
        uint4 d = make_uint4(0, 0, 0, 0);
        if ((int)lane < cnt) d = ld_cg_128(garena + ((size_t)k.j * kWR + k.slot) * 32 + lane);
        if (k.blk != cached_blk && cnt) {
            const BlockGeom g = block_geom(a, k.blk);
            blk_gbase = g.payload - (reinterpret_cast<uintptr_t>(g.payload) & 15);
            cached_blk = k.blk;
        }
        const uint32_t dslot = desc_s + (t & (kWSlots - 1)) * 512u;
        if (k.cf & kBulk) {
            const uint32_t lit_src = __shfl_sync(kFull, d.x, 0), lit = __shfl_sync(kFull, d.y, 0);
            sts128(dslot + 16u * lane, d.x, d.y, d.z, d.w);
            if (lit) copy_g2r<true>(out_s, k.base + k.op_start, blk_gbase + lit_src, lit);
        } else if (cnt) {
            sts128(dslot + 16u * lane, d.x, d.y, d.z, d.w);
            const uint32_t lit = d.y & 0xFFu;
            if (nvec == 0) {
                lo = __shfl_sync(kFull, d.x, 0) & ~15u;
                nvec = (__shfl_sync(kFull, d.x + lit, cnt - 1) - lo + 15u) >> 4;
            }
            const bool staged = nvec <= (uint32_t)(kWStage / 16);
            if (staged) {
                const uint4* gv = reinterpret_cast<const uint4*>(blk_gbase + lo);
                uint4 x0 = make_uint4(0, 0, 0, 0), x1 = x0, x2 = x0;       // (at most 76 vectors: three per lane, all in flight at once)
                if (lane < nvec) x0 = ldg_na_u128(gv + lane);
                if (lane + 32u < nvec) x1 = ldg_na_u128(gv + lane + 32u);
                if (lane + 64u < nvec) x2 = ldg_na_u128(gv + lane + 64u);
                if (lane < nvec) sts128(stage_s + 16u * lane, x0.x, x0.y, x0.z, x0.w);
                if (lane + 32u < nvec) sts128(stage_s + 16u * (lane + 32u), x1.x, x1.y, x1.z, x1.w);
                if (lane + 64u < nvec) sts128(stage_s + 16u * (lane + 64u), x2.x, x2.y, x2.z, x2.w);
            }
            __syncwarp();
            WSTAT(1)
            const uint32_t lit_pos = k.base + d.z;
            if ((int)lane < cnt && lit) {
                if (staged) lane_copy4(out_s, lit_pos, stage_s, d.x - lo, 0xFFFFFFFFu, lit);
                else { const uint8_t* gp = blk_gbase + d.x; for (uint32_t i = 0; i < lit; i++) sts8(out_s + ((lit_pos + i) & M), (uint32_t)__ldg(gp + i)); }
            }
        }
        bar_signal(ctl->bar_lit, t);
        WSTAT(2)
    }
    WSTAT_FLUSH(a, 8, 4)
}

// stage F: matches whose source is final before the ticket starts, lane-parallel (tickets w, w + kWF, ...).  It also
// prepares the serial stage's work: the parameters of every match (see copy_near_matches) replace the (consumed)
// descriptors, and one word says which of them are NEAR, so that stage N spends nothing on bookkeeping.
__device__ void wstage_far(const DecompressArgs& a, int w, WCtl* ctl, uint32_t out_s, uint32_t desc_s)
{
    const uint32_t lane = lane_id();
    WSTAT_DECL(3)       // 0 waiting (ticket, descriptors), 1 waiting for the serial stage, 2 copy
    for (uint32_t t = (uint32_t)w;; t += kWF) {
        if (!wait_ticket(ctl, t)) break;
        const WTk k = read_ticket(ctl, t);
        const int cnt = k.cf & 0xFF;
        const uint32_t dslot = desc_s + (t & (kWSlots - 1)) * 512u;
        uint32_t nmask = 0, nlong = 0;
        if (cnt) {
            bar_wait(ctl->bar_lit, t);                                      // (the descriptors are in shared memory)
            WSTAT(0)
            const uint4 d = lds128(dslot + 16u * lane);
            if (k.cf & kBulk) {
                const uint32_t lit = __shfl_sync(kFull, d.y, 0), mlen = __shfl_sync(kFull, d.z, 0), dist = __shfl_sync(kFull, d.w, 0);
                const uint32_t m_pos = k.base + k.op_start + lit;
                if (mlen && (int)(m_pos - dist - k.valid_lo) >= 0) {        // (else: the block is rejected at its end)
                    nlong = 1;
                    __syncwarp();
                    if (lane == 0) sts128(dslot, m_pos, mlen, dist, 0u);
                }
            } else {
                const uint32_t lit = d.y & 0xFFu, mlen = (d.y >> 8) & 0xFFu, dist = d.y >> 16;
                const uint32_t m_pos = k.base + d.z + lit, from = m_pos - dist;
                const bool live = (int)lane < cnt && mlen != 0 && (int)(from - k.valid_lo) >= 0;     // (a match below the dictionary: block rejected)
                const bool far = live && (int)(from + mlen - k.safe) <= 0;
                nmask = __ballot_sync(kFull, live && !far);
                if (nmask) sts128(dslot + 16u * lane, m_pos, mlen, dist, overlap_inv(dist, mlen));     // (every lane has read its own descriptor)
                // everything below `safe` (the start of ticket t - kWDepth) is final once stage N has finished ticket t - kWDepth - 1
                if (__ballot_sync(kFull, far)) {
                    if (t > (uint32_t)kWDepth) bar_wait(ctl->bar_near, t - kWDepth - 1);
                    WSTAT(1)
                    if (far) lane_copy4(out_s, m_pos, out_s, from, kWM, mlen);
                }
            }
        }
        if (lane == 0) { vst(&ctl->near_mask[t & (kWSlots - 1)], nmask); vst(&ctl->near_long[t & (kWSlots - 1)], nlong); }
        bar_signal(ctl->bar_far, t);
        WSTAT(2)
    }
    WSTAT_FLUSH(a, 12, 3)
}

// stage N: the serial chain -- near matches in stream order, each copied by all lanes; long match pieces
__device__ void wstage_near(const DecompressArgs& a, WCtl* ctl, uint32_t out_s, uint32_t desc_s)
{
    const uint32_t lane = lane_id();
    WSTAT_DECL(4)       // 0 waiting for stage F, 1 near matches, 2 long matches, 3 near matches (count)
    for (uint32_t t = 0;; t++) {
        bool fin = false;
        while (!bar_try(ctl->bar_far, t))                                   // (stage F has waited for the ticket and for stage L)
            if (vld(&ctl->finished) && (int)(t - vld(&ctl->t_final)) >= 0) { fin = true; break; }
        if (fin) break;
        const uint32_t dep = vld(&ctl->near_mask[t & (kWSlots - 1)]);
        const uint32_t is_long = vld(&ctl->near_long[t & (kWSlots - 1)]);
        const uint32_t dslot = desc_s + (t & (kWSlots - 1)) * 512u;
        WSTAT(0)
        if (is_long) {
            const uint4 d = lds128(dslot);
            coop_long_match(out_s, d.x, d.y, d.z);
            WSTAT(2)
        } else if (dep) {
            copy_near_matches<kWM>(out_s, dslot, dep, lane);
            WSTAT_COUNT(3, __popc(dep))
            WSTAT(1)
        }
        bar_signal(ctl->bar_near, t);
    }
    WSTAT_FLUSH(a, 15, 4)
}

// stage G: finished batches leave for global memory (tickets w, w + kWG, ...)
__device__ void wstage_flush(const DecompressArgs& a, int w, WCtl* ctl, uint32_t out_s)
{
    const uint32_t lane = lane_id();
    int cached_blk = -1; uint8_t* blk_out = nullptr;
    WSTAT_DECL(2)       // 0 waiting, 1 flush
    for (uint32_t t = (uint32_t)w;; t += kWG) {
        if (!wait_ticket(ctl, t)) break;
        const WTk k = read_ticket(ctl, t);
        const uint32_t e = vld(&ctl->tend[t & (kTickets - 1)]);
        bar_wait(ctl->bar_near, t);
        WSTAT(0)
        const uint32_t s_pos = k.base + k.op_start;
        if (e != s_pos) {
            if (k.blk != cached_blk) { blk_out = a.dst + a.dst_off[k.blk]; cached_blk = k.blk; }
#ifdef B200LZ4_BOUNDS_CHECK
            { const BlockGeom g = block_geom(a, k.blk); BCHK(a, (long long)k.op_start + (e - s_pos) <= (long long)g.cap && (e - s_pos) <= 65536u); }
#endif
            flush_r2g(out_s, blk_out + k.op_start, s_pos, e - s_pos);
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0) vst(&ctl->done[t & (kTickets - 1)], t + 1);
        WSTAT(1)
    }
    WSTAT_FLUSH(a, 19, 2)
}

constexpr size_t kWSmem = 128 /* alignment slack */ + kWOut + kWP * kWIn + kWP * kWR * 16 + kWSlots * 512 + kWL * kWStage + sizeof(WCtl);

__global__ void __launch_bounds__(kWThreads, 1)
decompress_kernel_wide(DecompressArgs a)
{
    extern __shared__ __align__(16) uint8_t smem_dyn[];
    uint8_t* base = smem_dyn + ((128u - (smem_u32(smem_dyn) & 127u)) & 127u);
    uint8_t* out_ring = base;
    uint8_t* in_rings = out_ring + kWOut;
    uint8_t* hdrs = in_rings + kWP * kWIn;
    uint8_t* descs = hdrs + kWP * kWR * 16;
    uint8_t* stages = descs + kWSlots * 512;
    WCtl* ctl = reinterpret_cast<WCtl*>(stages + kWL * kWStage);
    for (uint32_t i = threadIdx.x; i < sizeof(WCtl) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(ctl)[i] = 0u;
    __syncthreads();
    if (threadIdx.x < kTickets) {
        mbar_init(&ctl->bar_ticket[threadIdx.x], 1); mbar_init(&ctl->bar_lit[threadIdx.x], 1);
        mbar_init(&ctl->bar_far[threadIdx.x], 1); mbar_init(&ctl->bar_near[threadIdx.x], 1);
    }
    __syncthreads();
    const int warp = (int)(threadIdx.x >> 5);
    uint4* garena = a.wide_arena + (size_t)blockIdx.x * (kWideArenaPerCta / 16);
    uint32_t out_s;             // laundered so that the compiler keeps it in a register
    asm volatile("mov.u32 %0, %1;" : "=r"(out_s) : "r"(smem_u32(out_ring)));
    const uint32_t desc_s = smem_u32(descs);
    int r = warp;
    if (r < kWP) { wparser_main(a, r, ctl, smem_u32(in_rings) + (uint32_t)r * kWIn, smem_u32(hdrs) + (uint32_t)r * kWR * 16u, garena + (size_t)r * kWR * 32); return; }
    r -= kWP;
    if (r == 0) { wdispatch_main(a, ctl, out_s, smem_u32(hdrs)); return; }
    r -= 1;
    if (r < kWL) { wstage_literals(a, r, ctl, out_s, desc_s, smem_u32(stages) + (uint32_t)r * kWStage, garena); return; }
    r -= kWL;
    if (r < kWF) { wstage_far(a, r, ctl, out_s, desc_s); return; }
    r -= kWF;
    if (r == 0) { wstage_near(a, ctl, out_s, desc_s); return; }
    wstage_flush(a, r - 1, ctl, out_s);
}

}  // namespace

cudaError_t launch_decompress_wide(const DecompressArgs& a, int sm_count, cudaStream_t stream)
{
    static PerDeviceOnce once;
    const cudaError_t e = once.run([] {
        return cudaFuncSetAttribute(decompress_kernel_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWSmem);
    });
    if (e != cudaSuccess) return e;
    int grid = a.n_streams < sm_count ? a.n_streams : sm_count;
    if (grid > a.wide_ctas) grid = a.wide_ctas;
    if (grid <= 0) return cudaErrorInvalidValue;
    decompress_kernel_wide<<<grid, kWThreads, kWSmem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace b200lz4
