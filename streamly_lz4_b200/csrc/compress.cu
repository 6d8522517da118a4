// compress.cu -- byte-exact LZ4 block compressor for sm_100a.
//
// Reproduces LZ4_compress_fast_continue in external-dictionary mode
// (cbits/lz4.c:1565-1637 -> LZ4_compress_generic_validated :851-1240 with
// limitedOutput/byU32/usingExtDict) bit for bit, organised for a SIMT machine.
//
// One stream (independent mode: one block) is owned by a PAIR of warps:
//
//   FINDER warp  -- runs the match finder, the only inherently serial part.  It keeps the
//     16 KiB position table in shared memory and produces (literal run, match length,
//     offset) triples.
//       * After a match the reference inserts ip-2 and immediately re-tests ip
//         (cbits/lz4.c:1146-1196).  This "match follows match" regime dominates
//         compressible data, so it is a warp-uniform scalar path: one broadcast load of
//         the bytes around ip, two hashes, one table read/write, then ONE 32-lane byte
//         compare + ballot that both verifies the candidate and gives the match length.
//       * Otherwise the serial "probe, overwrite, test" recurrence (cbits/lz4.c:959-1014)
//         is evaluated up to 32 probes at a time.  Probe positions follow a closed-form
//         schedule (step_k = (acc*64 + k - 1) >> 6), lane l speculatively evaluates probe
//         j0+l; same-bucket forwarding inside the window is resolved with
//         __match_any_sync (a lane's candidate is the nearest lower lane with the same
//         hash, else the table), the lowest accepting lane wins, lanes up to the winner
//         commit their table writes in order (last writer per bucket wins), later lanes
//         are discarded.  The window width adapts (4 or 32) so that large accelerations
//         do not touch far cache lines that the serial algorithm would never read.
//       * upcoming input is pulled into L2 with cp.async.bulk.prefetch.L2.
//   EMITTER warp -- receives the triples through a double-buffered shared-memory queue
//     (mbarrier full/empty handshakes), turns 32 of them at a time into LZ4 sequences:
//     encoded sizes -> warp prefix sum -> every lane writes its own token / length bytes /
//     offset, literal runs are copied per lane (short) or cooperatively (long, 128-bit).
//
// Three kernels share this code (template parameters of find_block / finder_main), chosen per launch by the number
// of streams it carries (launch_compress):
//   compress_kernel          classic: 4 pairs per CTA, 3 CTAs per SM, 16 KiB tables      (up to 12 streams per SM)
//   compress_kernel_wide     one pair per CTA, one CTA per SM, 128 KiB stream-indexed data ring that also holds the
//                            dictionary                                                   (no more streams than SMs)
//   compress_kernel_compact  8.5 KiB tables (16-bit entries + epoch bit, periodic sweeps), 4 CTAs per SM
//                                                                                        (more than one classic wave)
// All three produce the reference's bytes; tests/test_gpu_modes.py forces each of them in turn.
//
// The compaction pass (compact.cu) then gathers the per-block slots into one stream.
#include <cstdio>
#include <cstdlib>
#include "common.cuh"
#include "kernels.h"

namespace b200lz4 {

namespace {

constexpr int kPairs = 4;                        // stream-owning warp pairs per CTA
constexpr int kQueueDepth = 16;                  // descriptors per queue buffer
constexpr uint32_t kPrefetchAhead = 16384;       // bytes of input kept ahead in L2
constexpr uint32_t kPrefetchChunk = 4096;

struct __align__(16) Queue {
    uint4 desc[2][kQueueDepth];                  // {literal start, literal length, match code, offset (0 = final literals)}
    unsigned long long full[2], empty[2];        // mbarriers
    int count[2];                                // descriptors in buffer; bit 30 = block ends here, bit 29 = terminate
    int block[2];                                // block index the buffer belongs to
    int pad_[4];
};
constexpr int kEndBlock = 1 << 30, kTerminate = 1 << 29;

// offset (from the run start) and step of probe j >= 0 of a search run (cbits/lz4.c:957-967).
__device__ __forceinline__ void probe_schedule(long long j, int accel, long long& off, int& step)
{
    if (j <= 0) { off = 0; step = 1; return; }
    long long m = j - 1, q = m >> 6, r = m & 63;
    off = 1 + m * accel + 32 * q * (q - 1) + q * r;
    step = accel + (int)q;
}

// Common-prefix length of a[0..cap) and b[0..cap), 4 bytes per lane per round (what LZ4_count
// computes, cbits/lz4.c:603-626).  a, b read-only global memory.
__device__ __forceinline__ uint32_t warp_common_prefix(const uint8_t* a, const uint8_t* b, uint32_t cap)
{
    const uint32_t lane = lane_id();
    uint32_t base = 0;
    for (;;) {
        const uint32_t at = base + lane * 4;
        uint32_t nb = 0;
        bool stop = true;
        if (at + 4 <= cap) {
            uint32_t x = ldg_u32_unaligned(a + at) ^ ldg_u32_unaligned(b + at);
            nb = x ? ((uint32_t)(__ffs(x) - 1) >> 3) : 4u;
            stop = (nb < 4);
        } else if (at < cap) {
            const uint32_t room = cap - at;
            while (nb < room && __ldg(a + at + nb) == __ldg(b + at + nb)) nb++;
        }
        const uint32_t sb = __ballot_sync(kFull, stop);
        if (sb) {
            const int l = __ffs(sb) - 1;
            const uint32_t res = __shfl_sync(kFull, at + nb, l);
            return res < cap ? res : cap;
        }
        base += 128;
    }
}

// Number of equal bytes walking backwards from a[-1], b[-1], at most cap (the catch-up loop,
// cbits/lz4.c:1019), 4 bytes per lane per round.
__device__ __forceinline__ uint32_t warp_common_suffix(const uint8_t* a, const uint8_t* b, uint32_t cap)
{
    const uint32_t lane = lane_id();
    if (cap <= 32) {                    // the usual case (a few literals at most): one byte per lane, one ballot
        uint32_t x = 0, y = 1;          // lanes at or past the cap differ by construction
        if (lane < cap) { x = __ldg(a - 1 - lane); y = __ldg(b - 1 - lane); }
        const uint32_t ne = __ballot_sync(kFull, x != y);
        return ne ? (uint32_t)__ffs(ne) - 1u : 32u;     // ne == 0 only when cap == 32 and all 32 bytes agree
    }
    uint32_t base = 0;
    for (;;) {
        const uint32_t at = base + lane * 4;        // this lane covers bytes [-(at+4), -at)
        uint32_t nb = 0;
        bool stop = true;
        if (at + 4 <= cap) {
            uint32_t x = ldg_u32_unaligned(a - at - 4) ^ ldg_u32_unaligned(b - at - 4);
            nb = x ? ((uint32_t)__clz(x) >> 3) : 4u;
            stop = (nb < 4);
        } else if (at < cap) {
            const uint32_t room = cap - at;
            while (nb < room && __ldg(a - at - nb - 1) == __ldg(b - at - nb - 1)) nb++;
        }
        const uint32_t sb = __ballot_sync(kFull, stop);
        if (sb) {
            const int l = __ffs(sb) - 1;
            const uint32_t res = __shfl_sync(kFull, at + nb, l);
            return res < cap ? res : cap;
        }
        base += 128;
    }
}

// ---- shared-memory input window of the finder ---------------------------------
// Four 128-byte lines of the input around ip (data ring, keyed by global line index & 3,
// filled with cp.async one line ahead of use) plus the LZ4 hash of every position in them
// (hash ring, computed 128 positions at a time by all lanes when a line lands).  The scalar
// re-test path takes hash(ip-2), hash(ip) and the bytes it compares from these rings, so its
// dependent chain is shared-memory latency only and a few dozen instructions long.
//   invariant while ip is in line L:  lines L-1, L, L+1 complete, L+2 in flight;
//   data readable for positions [lo_pos, ready_end), hashes valid for [lo_pos, ready_end - 4).
// All accesses use explicit 32-bit shared-space addresses (ld.shared / st.shared).
constexpr int kWinLines = 4, kWinBytes = kWinLines * 128;
// WIDE mode (at most one stream per SM): the data ring is 128 KiB and indexed by stream position, so it holds the
// previous array too -- every candidate within reach (65535 back, dictionary included), every catch-up and every
// count is then served from shared memory and a block costs its instruction chain, not L2 round trips.
constexpr int kWideLines = 1024, kWideBytes = kWideLines * 128;
constexpr int kHashPos = 512;                    // hash ring: u16 hashes of the 512 most recent ring positions

struct BlockIn {
    const uint8_t* src; int n;
    const uint8_t* dict_end;    // one past the last dictionary byte (meaningful iff dict_len > 0)
    uint32_t dict_len;
    uint32_t start;             // currentOffset before this block
    int accel;
    int block;                  // block index (for the emitter)
    // wide mode, carried from block to block of a stream: ring position one past the previous array, lowest ring
    // position of contiguously loaded data, and whether both mean anything
    uint32_t w_end, w_lo; bool w_ok;
    uint32_t tbase;             // compact table: stream position of rel == 1 (carried from block to block)
    // streamed launches (the block is still arriving over PCIe, see CompressArgs::arrived): flag word, segment size,
    // cycles this finder spent waiting for data
    const uint32_t* arrived; int seg; long long stall; bool timed_out;
};

// Producer side of the queue (finder warp).  The buffer being filled is always already acquired.
struct Producer {
    Queue* q;
    uint32_t batch;     // batches pushed so far
    int fill;           // descriptors in the current buffer
    uint32_t slot_s;    // shared address of the next descriptor slot

    __device__ __forceinline__ void begin()
    {   // wait until the buffer we are about to fill has been drained, point at its first slot
        const uint32_t b = batch & 1, t = batch >> 1;
        if (t) mbar_wait(&q->empty[b], (t - 1) & 1);
        slot_s = smem_u32(&q->desc[b][0]);
        fill = 0;
    }
    __device__ __forceinline__ void push(uint32_t lit_pos, uint32_t lit_len, uint32_t mcode, uint32_t off, int block)
    {
        sts128(slot_s, lit_pos, lit_len, mcode, off);     // all lanes store the same 16 bytes: no lane predicate on the hot path
        slot_s += 16;
        if (++fill == kQueueDepth) flush(block, 0);
    }
    __device__ __forceinline__ void flush(int block, int flags)
    {
        if (fill == 0 && flags == 0) return;
        const uint32_t b = batch & 1;
        if (lane_id() == 0) { q->count[b] = fill | flags; q->block[b] = block; }
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(&q->full[b]);
        batch++;
        begin();
    }
};

// (x & mask) | base in one LOP3 (base must have no bits inside mask: rings are aligned to their size)
__device__ __forceinline__ uint32_t and_or(uint32_t x, uint32_t mask, uint32_t base)
{ uint32_t d; asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(x), "r"(mask), "r"(base)); return d; }

// Match finder for one block: pushes sequence descriptors, ends with the final-literals descriptor.
// data_s (512-byte aligned) / hash_s (1024-byte aligned): shared addresses of this finder's rings.
// COMPACT table (kCompact): 16-bit entries plus one epoch bit per bucket, 8.5 KiB instead of 16 KiB, so that more
// finders fit an SM.  A bucket holds rel = pos - tbase + 1 (17 bits: u16 + the bucket's bit; 0 = empty).  Positions are
// inserted in non-decreasing order, so when the current position reaches tbase + 131071 every entry in the lower half
// (rel <= 65536) is more than 65535 behind every future position -- the reference rejects such candidates -- and a
// SWEEP drops them, moves the upper half down (clear all bits) and advances tbase by 65536.  An empty bucket decodes to
// tbase - 1, which the distance test rejects by itself.
constexpr uint32_t kEpoch = 65536u, kRelMax = 2 * kEpoch - 1;       // rel in [1, 131071]

// STREAMED launches (kStreamed): the block's bytes land in HBM segment by segment while the finder runs.  `avail` is the
// number of leading bytes of the block that have arrived (a multiple of 128 or n; block starts are 128-byte aligned, so
// no 32-byte L1 sector is ever read before it is complete); every read AHEAD of ip -- ring fills, L2 prefetches, probe
// windows, forward counts -- first makes sure the bytes it touches lie below it (wait_for polls the flag word the
// copy stream bumps after each segment).  Reads at or behind ip need no check.
constexpr long long kArrivalTimeoutCycles = 2000000000LL;        // ~1 s at 2 GHz

template <bool kWide, bool kCompact, bool kStreamed>
__device__ void find_block(BlockIn& in, uint32_t* table, const uint32_t data_s, const uint32_t hash_s, Producer& out,
                           const uint32_t off0, const uint32_t step0, const uint32_t off1, const uint32_t step1)
{
    constexpr uint32_t kRingBytes = kWide ? kWideBytes : kWinBytes;
    const uint32_t lane = lane_id();
    const uint8_t* const src = in.src;
    const int n = in.n;
    const uint32_t S = in.start;
    const bool dict_small = (in.dict_len < 65536u) && (in.dict_len < S);   // cbits/lz4.c:1627
    const uint32_t low_index = S - in.dict_len;                             // prefixIdxLimit, :879
    const int mfl = n - kMfLimit + 1;          // mflimitPlusOne as an index
    const int mlimit = n - kLastLiterals;      // matchlimit
    const uint32_t table_s = smem_u32(table);
    int anchor = 0;
    if (kWide && n < kMinLength) in.w_ok = false;       // nothing of a tiny array reaches the ring
    int avail = kStreamed ? 0 : n;
    auto wait_for = [&](long long upto) {               // block until bytes [0, min(upto, n)) of the block have arrived
        if (!kStreamed) return;
        const int want = upto < (long long)n ? (int)upto : n;
        if (want <= avail) return;
        const long long t0 = clock64();
        for (;;) {
            const long long got = (long long)ld_acquire_sys(in.arrived) * in.seg;
            avail = got < (long long)n ? (int)got : n;
            if (want <= avail) break;
            if (clock64() - t0 > kArrivalTimeoutCycles) {       // the copy stream died under us: do not spin forever, let the host fail the call
                in.timed_out = true; avail = n;
                break;
            }
            __nanosleep(2000);
        }
        in.stall += clock64() - t0;
    };
    // forward count whose first operand runs ahead of ip: a = src + p
    auto count_ahead = [&](int p, const uint8_t* b, uint32_t cap) -> uint32_t {
        if (!kStreamed || p + (int)cap <= avail) return warp_common_prefix(src + p, b, cap);
        uint32_t L = 0;
        for (;;) {
            wait_for((long long)p + L + 1);
            const uint32_t piece = min(cap - L, (uint32_t)(avail - (p + (int)L)));
            const uint32_t x = warp_common_prefix(src + p + L, b + L, piece);
            L += x;
            if (x < piece || L == cap) return L;
        }
    };

    // ---- position table access (classic: u32 per bucket; compact: see above)
    uint32_t tbase = in.tbase;
    const uint32_t tfl_s = table_s + 2 * kHashEntries;  // compact: the epoch bits, one u32 per 32 buckets
    auto t_get = [&](uint32_t h) -> uint32_t {          // stream position held by bucket h
        if (!kCompact) return lds32(table_s + h * 4);
        const uint32_t lo = lds16(table_s + h * 2);
        const uint32_t fw = lds32(tfl_s + ((h >> 5) << 2));
        return tbase + (lo | (((fw >> (h & 31u)) & 1u) << 16)) - 1u;
    };
    auto t_put = [&](uint32_t h, uint32_t pos) {        // warp-uniform insert (every lane stores the same values)
        if (!kCompact) { sts32(table_s + h * 4, pos); return; }
        const uint32_t rel = pos - tbase + 1u;
        sts16(table_s + h * 2, rel & 0xFFFFu);
        const uint32_t a = tfl_s + ((h >> 5) << 2), bit = 1u << (h & 31u);
        const uint32_t fw = lds32(a), nw = (rel >> 16) ? (fw | bit) : (fw & ~bit);
        if (nw != fw) sts32(a, nw);
    };
    auto t_swap = [&](uint32_t h, uint32_t pos) -> uint32_t {      // warp-uniform: read bucket h, then insert pos (one flag-word load)
        if (!kCompact) { const uint32_t m = lds32(table_s + h * 4); sts32(table_s + h * 4, pos); return m; }
        const uint32_t a = tfl_s + ((h >> 5) << 2), bit = 1u << (h & 31u);
        const uint32_t lo = lds16(table_s + h * 2);
        const uint32_t fw = lds32(a);
        const uint32_t rel = pos - tbase + 1u;
        sts16(table_s + h * 2, rel & 0xFFFFu);
        const uint32_t nw = (rel >> 16) ? (fw | bit) : (fw & ~bit);
        if (nw != fw) sts32(a, nw);
        return tbase + (lo | ((fw & bit) ? kEpoch : 0u)) - 1u;
    };
    auto t_put_lane = [&](uint32_t h, uint32_t pos) {   // per-lane insert (distinct buckets in one warp instruction)
        if (!kCompact) { sts32(table_s + h * 4, pos); return; }
        const uint32_t rel = pos - tbase + 1u;
        sts16(table_s + h * 2, rel & 0xFFFFu);
        uint32_t* w = table + kHashEntries / 2 + (h >> 5);
        if (rel >> 16) atomicOr(w, 1u << (h & 31u)); else atomicAnd(w, ~(1u << (h & 31u)));
    };
    auto t_sweep_to = [&](uint32_t cur) {               // make position cur insertable: rel(cur) <= kRelMax
        if (!kCompact) return;
        while (cur - tbase >= kRelMax) {
            __syncwarp();
            if (cur - tbase >= 2 * kRelMax) {           // a long skip: everything is stale
                for (int i = lane; i < kHashEntries / 8; i += 32) sts128(table_s + 16 * i, 0u, 0u, 0u, 0u);
                for (int i = lane; i < kHashEntries / 32; i += 32) sts32(tfl_s + 4 * i, 0u);
                tbase = cur - (kEpoch - 1);
            } else {
                for (int j = lane; j < kHashEntries / 32; j += 32) {
                    const uint32_t fw = lds32(tfl_s + 4 * j);
                    uint32_t clr = ~fw;                 // lower-half entries: out of reach from now on
                    while (clr) { const int b = __ffs(clr) - 1; clr &= clr - 1; sts16(table_s + 2 * (32 * j + b), 0u); }
                    sts32(tfl_s + 4 * j, 0u);
                }
                tbase += kEpoch;
            }
            __syncwarp();
        }
    };

    if (n >= kMinLength) {
        // ---- window state (see the invariant above)
        const uintptr_t base = reinterpret_cast<uintptr_t>(src), end = base + (uintptr_t)n;
        // Ring position of block position p is g32 + p (as u32).  Dense mode: g32 = the block's global address, the
        // ring is a 512-byte cache of the lines around ip.  Wide mode: g32 continues the previous array's positions
        // when the word alignment of both agrees, so positions below 0 are the dictionary, still resident.
        uint32_t g32 = (uint32_t)base;
        int lo_pos = 0;                        // lowest block position whose bytes are in the ring (wide: may be negative)
        if (kWide) {
            if (in.w_ok && in.dict_len && ((in.w_end - g32) & 3u) == 0 && (base & 3) == 0) {
                g32 = in.w_end;
                const uint32_t have = in.w_end - in.w_lo;           // contiguously loaded bytes before this block
                lo_pos = -(int)min(min(have, in.dict_len), (uint32_t)(kWideBytes - 65536 - 1024));
            }
            in.w_ok = false;
        }
        const uint32_t glane = g32 + 4 * lane;
        uintptr_t cur_line = ~uintptr_t(0) - 8;
        int ready_end = 0, trigger = -1;
        uint32_t pf_next = 0;                  // next input byte not yet requested into L2

        auto raddr = [&](uint32_t a, uint32_t mask) -> uint32_t {     // shared address of ring position a (mask selects the granule)
            if (kWide) return data_s + (a & mask);
            return and_or(a, mask, data_s);
        };
        auto ring32 = [&](uint32_t a) {        // 4 bytes of the data ring at ring position a
            return __funnelshift_r(lds32(raddr(a, kRingBytes - 4)), lds32(raddr(a + 4, kRingBytes - 4)), a << 3);
        };
        auto ring8 = [&](uint32_t a) { return lds8(raddr(a, kRingBytes - 1)); };
        auto hash_at = [&](uint32_t a) { return lds16(and_or(a << 1, 2 * kHashPos - 2, hash_s)); };
        auto issue = [&](uintptr_t line) {     // one 4-byte cp.async per lane; lines outside the block are not touched
            const uintptr_t wa = (line << 7) + 4 * lane;       // this lane's aligned word: copied only if it holds a byte of the block
            if (wa < end && wa + 4 > base)
                cp_async_4(raddr(g32 + (uint32_t)(wa - base), kRingBytes - 4), reinterpret_cast<const void*>(wa));
            cp_async_commit();
        };
        auto hash_round = [&](int p0) {        // hashes of the 128 positions from p0 on ((g32 + p0) % 4 == 0)
            const uint32_t a = glane + (uint32_t)p0;
            const uint32_t w0 = lds32(raddr(a, kRingBytes - 4)), w1 = lds32(raddr(a + 4, kRingBytes - 4));
            const uint32_t h0 = hash5(w0, w1 & 0xFFu);
            const uint32_t h1 = hash5(__funnelshift_r(w0, w1, 8), (w1 >> 8) & 0xFFu);
            const uint32_t h2 = hash5(__funnelshift_r(w0, w1, 16), (w1 >> 16) & 0xFFu);
            const uint32_t h3 = hash5(__funnelshift_r(w0, w1, 24), w1 >> 24);
            sts64(and_or(a << 1, 2 * kHashPos - 8, hash_s), h0 | (h1 << 16), h2 | (h3 << 16));
        };
        auto l2_prefetch = [&](int ip) {       // keep the next kPrefetchAhead bytes of input on their way into L2
            if (pf_next < (uint32_t)ip) pf_next = (uint32_t)ip & ~(kPrefetchChunk - 1);
            if (kStreamed && avail < n && pf_next + kPrefetchChunk > (uint32_t)avail) return;   // not there yet (no poll here: wait_for refreshes avail)
            if (pf_next < (uint32_t)n) {
                const uintptr_t pbase = (base + pf_next) & ~uintptr_t(15);
                const uint32_t room = (uint32_t)n - pf_next;
                const uint32_t bytes = room < kPrefetchChunk ? (room & ~15u) : kPrefetchChunk;
                if (lane == 0 && bytes) prefetch_l2_bulk(reinterpret_cast<const void*>(pbase), bytes);
            }
            pf_next += kPrefetchChunk;
        };
        auto move_window = [&](int ip) {       // (re)centre the window on ip's line
            const uintptr_t L = (base + (uintptr_t)ip) >> 7;
            if (kStreamed) wait_for((long long)((L + 3) << 7) - (long long)base);       // lines L-1 .. L+2 are touched below
            __syncwarp();
            cp_async_wait<0>();
            __syncwarp();
            if (kWide) {
                // the ring keeps everything behind ip: advance over up to 96 lines without leaving a hole
                const bool near = trigger >= 0 && L > cur_line && L - cur_line <= 96;
                int new_ready;
                if (near) {
                    for (uintptr_t l = cur_line + 3; l <= L + 1; l++) issue(l);
                    if (L > cur_line + 1) { cp_async_wait<0>(); __syncwarp(); }
                    new_ready = (int)(((L + 2) << 7) - base);
                } else {                       // first window of the block, or a long skip (leaves a hole behind it)
                    issue(L - 1); issue(L); issue(L + 1);
                    cp_async_wait<0>();
                    __syncwarp();
                    const long long lo = (long long)((L - 1) << 7) - (long long)base;
                    if (lo > 0) lo_pos = (int)lo;           // else: the window reaches the block start, what precedes it stays valid
                    new_ready = (int)lo + 384;
                    hash_round((int)lo); hash_round((int)lo + 128); hash_round((int)lo + 256);
                }
                if (near) for (int r = max(ready_end, new_ready - 384); r < new_ready; r += 128) hash_round(r - 4);
                ready_end = new_ready;
                lo_pos = max(lo_pos, new_ready + 128 - kWideBytes);
                issue(L + 2);
                __syncwarp();
                cur_line = L;
                trigger = (int)(((L + 1) << 7) - base);
                if ((uint32_t)ip + kPrefetchAhead > pf_next) l2_prefetch(ip);
                return;
            }
            if (L == cur_line + 1) {           // steady state: line L+1 has just landed
                hash_round(ready_end - 4);
                ready_end += 128;
                const int lo = (int)(((L - 1) << 7) - base);
                lo_pos = lo_pos > lo ? lo_pos : lo;
            } else {                           // jump: reload L-1, L, L+1
                issue(L - 1); issue(L); issue(L + 1);
                cp_async_wait<0>();
                __syncwarp();
                const long long lo = (long long)((L - 1) << 7) - (long long)base;
                const int p0 = (int)lo;
                hash_round(p0); hash_round(p0 + 128); hash_round(p0 + 256);
                lo_pos = lo < 0 ? 0 : p0;
                ready_end = p0 + 384;
            }
            issue(L + 2);
            __syncwarp();
            cur_line = L;
            trigger = (int)(((L + 1) << 7) - base);
            if ((uint32_t)ip + kPrefetchAhead > pf_next) l2_prefetch(ip);
        };

        // Scalar probe at position p (every lane computes the same thing; the only 32-wide step is the
        // verify+count).  kRetest: the post-match probe, which first inserts p-2 and has no literals.
        // On a hit fills mip / mlen / dist and returns true.
        int mip = 0; uint32_t mlen = 0, dist = 0;

        // ---- wide mode: extensions served from the ring.  Block positions; c < p; c may be negative (dictionary).
        // common prefix of p.. and c.., at most cap, as far as the ring reaches; `more`: the ring ended first
        auto ring_prefix = [&](int p, int c, uint32_t cap, bool& more) -> uint32_t {
            const uint32_t lim = min(cap, (uint32_t)(ready_end - p));
            const uint32_t pa = g32 + (uint32_t)p, ca = g32 + (uint32_t)c;
            uint32_t k0 = 0;
            for (;;) {
                const uint32_t at = k0 + lane * 4;
                uint32_t nb = 0;
                bool stop = true;
                if (at + 4 <= lim) {
                    const uint32_t x = ring32(pa + at) ^ ring32(ca + at);
                    nb = x ? ((uint32_t)(__ffs(x) - 1) >> 3) : 4u;
                    stop = (nb < 4);
                } else if (at < lim) {
                    const uint32_t room = lim - at;
                    while (nb < room && ring8(pa + at + nb) == ring8(ca + at + nb)) nb++;
                }
                const uint32_t sb = __ballot_sync(kFull, stop);
                if (sb) {
                    uint32_t res = __shfl_sync(kFull, at + nb, __ffs(sb) - 1);
                    res = res < lim ? res : lim;
                    more = (res == lim) && (lim < cap);
                    return res;
                }
                k0 += 128;
            }
        };
        // full forward count: ring first, then global memory (two segments when the candidate is still in the dictionary)
        auto count_wide = [&](int p, int c, uint32_t cap) -> uint32_t {
            bool more = false;
            uint32_t L = ring_prefix(p, c, cap, more);
            if (more) {
                int cc = c + (int)L;
                const uint8_t* a = src + p + L;
                uint32_t rest = cap - L;
                if (cc < 0) {                                                                        // :1080-1089
                    const uint32_t seg = min(rest, (uint32_t)(-cc));
                    const uint32_t x = warp_common_prefix(a, in.dict_end + cc, seg);
                    L += x;
                    if (x < seg || rest == seg) return L;
                    a += x; rest -= x; cc = 0;
                }
                L += warp_common_prefix(a, src + cc, rest);
            }
            return L;
        };
        // number of equal bytes walking backwards from p-1 / c-1, at most cap; needs c - cap >= lo_pos
        auto ring_suffix = [&](int p, int c, uint32_t cap) -> uint32_t {
            const uint32_t pa = g32 + (uint32_t)p, ca = g32 + (uint32_t)c;
            if (cap <= 32) {            // the usual case: one byte per lane, one ballot
                uint32_t x = 0, y = 1;
                if (lane < cap) { x = ring8(pa - 1 - lane); y = ring8(ca - 1 - lane); }
                const uint32_t ne = __ballot_sync(kFull, x != y);
                return ne ? (uint32_t)__ffs(ne) - 1u : 32u;
            }
            uint32_t k0 = 0;
            for (;;) {
                const uint32_t at = k0 + lane * 4;
                uint32_t nb = 0;
                bool stop = true;
                if (at + 4 <= cap) {
                    const uint32_t x = ring32(pa - at - 4) ^ ring32(ca - at - 4);
                    nb = x ? ((uint32_t)__clz(x) >> 3) : 4u;
                    stop = (nb < 4);
                } else if (at < cap) {
                    const uint32_t room = cap - at;
                    while (nb < room && ring8(pa - at - nb - 1) == ring8(ca - at - nb - 1)) nb++;
                }
                const uint32_t sb = __ballot_sync(kFull, stop);
                if (sb) {
                    const uint32_t res = __shfl_sync(kFull, at + nb, __ffs(sb) - 1);
                    return res < cap ? res : cap;
                }
                k0 += 128;
            }
        };
        // verify candidate index m for position p and count the match (table already updated)
        auto verify_count = [&](int p, uint32_t m, bool retest) -> bool {
            const uint32_t cur = S + (uint32_t)p;
            if (kWide) {
                const int cpos = (int)(m - S);                      // negative: in the dictionary, still a ring position
                if (cpos >= lo_pos) {
                    uint32_t L = count_wide(p, cpos, (uint32_t)(mlimit - p));
                    if (L < 4) return false;                                                         // :1009 / :1189
                    uint32_t back = 0;
                    if (!retest) {                                                                   // :1019
                        const uint32_t room_c = (m >= S) ? (uint32_t)cpos : in.dict_len - (S - m);
                        const uint32_t real = min((uint32_t)(p - anchor), room_c);
                        const uint32_t in_ring = min(real, (uint32_t)(cpos - lo_pos));      // part of the walk the ring can serve
                        if (in_ring && ring8(g32 + (uint32_t)p - 1) == ring8(g32 + (uint32_t)cpos - 1)) back = ring_suffix(p, cpos, in_ring);
                        if (back == in_ring && back < real) {       // the ring ended before the walk did: finish it in global memory
                            const uint8_t* cand_g = (m >= S) ? (src + cpos) : (in.dict_end - (S - m));
                            back += warp_common_suffix(src + p - back, cand_g - back, real - back);
                        }
                    }
                    mip = p - (int)back; mlen = L + back; dist = cur - m;
                    return true;
                }
            }
            const uint32_t mine = ring32(glane + (uint32_t)p);      // lane's 4 bytes of p..
            uint32_t cap = (uint32_t)(mlimit - p);
            uint32_t L;
            const uint8_t* cand;
            uint32_t room_c;                    // bytes available before the candidate (catch-up limit)
            if (m >= S) {
                const int cpos = (int)(m - S);
                cand = src + cpos; room_c = (uint32_t)cpos;
                const uint32_t cap1 = min(cap, 128u);
                const uint32_t at = lane * 4;
                uint32_t x = 0xFFu;                                 // lanes wholly past cap1 read nothing
                if (at < cap1)
                    x = mine ^ ((cpos >= lo_pos) ? ring32(glane + (uint32_t)cpos) : ldg_u32_unaligned(cand + at));
                const uint32_t nb = min((uint32_t)(__ffs(x) - 1) >> 3, 4u);   // x == 0 -> 4
                const uint32_t sb = __ballot_sync(kFull, (nb < 4) || (at + 4 >= cap1));   // never empty
                const uint32_t res = __shfl_sync(kFull, at + nb, __ffs(sb) - 1);
                L = res < cap1 ? res : cap1;
                if (res >= cap1 && cap > 128u) L += count_ahead(p + 128, cand + 128, cap - 128u);
            } else {                                                                                 // candidate in the dictionary
                cand = in.dict_end - (S - m); room_c = in.dict_len - (S - m);
                cap = min(cap, (uint32_t)(in.dict_end - cand));
                L = count_ahead(p, cand, cap);
                if (L >= 4 && L == cap && (int)(p + L) < mlimit)                                     // :1085-1089
                    L += count_ahead(p + (int)L, src, (uint32_t)(mlimit - (p + (int)L)));
            }
            if (L < 4) return false;                                                                 // :1009 / :1189
            uint32_t back = 0;
            if (!retest) {                      // catch up (cbits/lz4.c:1019): usually nothing to do
                const uint32_t maxback = min((uint32_t)(p - anchor), room_c);
                if (maxback && __ldg(src + p - 1) == __ldg(cand - 1)) back = warp_common_suffix(src + p, cand, maxback);
            }
            mip = p - (int)back; mlen = L + back; dist = cur - m;
            return true;
        };
        auto scalar_probe = [&](int p, bool retest) -> bool {
            if (p >= trigger) move_window(p);
            const uint32_t ap = g32 + (uint32_t)p;
            const uint32_t h = hash_at(ap);
            const uint32_t cur = S + (uint32_t)p;
            // every lane performs the same accesses in program order: no warp sync needed
            t_sweep_to(cur);
            if (retest) t_put(hash_at(ap - 2), cur - 2);                                             // :1146
            const uint32_t m = t_swap(h, cur);                                                       // :998 / :1185
            if ((dict_small && m < low_index) || (m + kMaxDistance < cur)) return false;             // :1001-1006 / :1187-1188
            return verify_count(p, m, retest);
        };

        // The post-match probe (put(ip-2), re-test ip; cbits/lz4.c:1146, :1159-1196), the hot loop on compressible data.
        // Lane l compares BYTE p+l with byte cand+l, so the match length is one ballot away (no per-lane
        // word assembly, no shuffle); only matches of 32 bytes and more take a second, word-granular step.
        auto retest_probe = [&](int p) -> bool {
            if (p >= trigger) move_window(p);
            const uint32_t ap = g32 + (uint32_t)p;
            const uint32_t capb = min((uint32_t)(mlimit - p), 32u);
            const uint32_t mine = ring8(ap + lane);             // issued early: overlaps the table chain
            const uint32_t h = hash_at(ap);
            const uint32_t cur = S + (uint32_t)p;
            t_sweep_to(cur);
            t_put(hash_at(ap - 2), cur - 2);                                                         // :1146
            const uint32_t m = t_swap(h, cur);                                                       // :1185
            if ((dict_small && m < low_index) || (m + kMaxDistance < cur)) return false;             // :1187-1188
            const int cpos = (int)(m - S);
            if (m < S && !(kWide && cpos >= lo_pos)) return verify_count(p, m, true);                // candidate in the dictionary, not in the ring
            uint32_t theirs = 0x100u;                           // lanes past the cap differ by construction
            if (lane < capb)
                theirs = (cpos >= lo_pos) ? ring8(g32 + (uint32_t)cpos + lane) : (uint32_t)__ldg(src + cpos + lane);
            const uint32_t ne = __ballot_sync(kFull, mine != theirs);
            uint32_t L;
            if (ne) L = (uint32_t)__ffs(ne) - 1u;
            else {                                              // 32 equal bytes and room for more
                const uint32_t cap = (uint32_t)(mlimit - p);
                L = 32u;
                if (cap > 32u) {
                    if (kWide && cpos >= lo_pos) L += count_wide(p + 32, cpos + 32, cap - 32u);
                    else L += count_ahead(p + 32, src + cpos + 32, cap - 32u);
                }
            }
            if (L < 4) return false;                                                                 // :1189
            mip = p; mlen = L; dist = cur - m;
            return true;
        };

        // A run of re-tests in the classic geometry without a dictionary (dict_len == 0, so the only lower bound on a
        // candidate is S and every candidate that passes it lies in the block): the same steps as retest_probe + push,
        // arranged so that one sequence costs one dependent chain and one branch.  Inside the inner loop ip stays below
        // both the next ring window (no move_window) and mlimit - 31 (32-byte compares need no cap); the hash-ring and
        // byte loads of the next sequence are issued as soon as this one's length is known, ahead of the descriptor
        // store; the queue is flushed when the loop leaves it full.  Anything else -- a miss, a match of 32+ bytes, the
        // window edge, a full queue -- leaves the inner loop and is settled here.
        // Returns 0: the re-test at ip missed (ip unchanged), 1: ip reached mflimit, 2: ip is within 32 bytes of
        // matchlimit (the caller finishes the run with retest_probe).
        auto retest_run = [&](int& ip) -> int {
            const uint32_t gl_s = g32 + lane - S;                   // ring position of byte lane of candidate index cand: gl_s + cand
            const uint8_t* const src_s = src + lane - S;            // its global address: src_s + cand (cand >= S)
            for (;;) {
                if (ip >= trigger) move_window(ip);
                if (ip > mlimit - 32) return 2;
                const int lim = min(trigger, mlimit - 31);
                const uint32_t ring_lo = S + (uint32_t)lo_pos;         // candidates from here on are in the ring
                const uint32_t slot0 = out.slot_s, slot_end = slot0 + 16u * (uint32_t)(kQueueDepth - out.fill);
                uint32_t slot = slot0;
                const uint32_t ap = g32 + (uint32_t)ip;
                uint32_t cur = S + (uint32_t)ip;
                uint32_t h = hash_at(ap), h2 = hash_at(ap - 2), mine = ring8(ap + lane);
                uint32_t m, ne;
                bool near, hit;
                do {
                    t_put(h2, cur - 2);                                                              // :1146
                    m = t_swap(h, cur);                                                              // :1185
                    near = (m >= S) && (m + kMaxDistance >= cur);                                    // :1187-1188
                    // ring bytes unless the candidate is older than the ring (a far miss compares garbage: near decides)
                    uint32_t theirs = ring8(gl_s + m);
                    if (near && m < ring_lo) theirs = __ldg(src_s + m);
                    ne = __ballot_sync(kFull, mine != theirs);
                    const uint32_t L = (uint32_t)__ffs(ne) - 1u;
                    hit = near && L - 4u < 28u;                                                      // 4 <= L < 32
                    // The next sequence's loads.  On the iteration that leaves the loop (a miss, where L may be
                    // ffs(0) - 1, or ip + L at the window edge) they may read ring bytes past ready_end, including the
                    // line cp.async is still filling: on purpose -- the addresses are masked into this finder's rings,
                    // the values are dropped, and the outer loop reloads h / h2 / mine after move_window.
                    const uint32_t na = g32 + (uint32_t)ip + L;
                    const uint32_t nh = hash_at(na), nh2 = hash_at(na - 2), nmine = ring8(na + lane);
                    sts128(slot, (uint32_t)ip, 0u, L - 4, cur - m);      // after a miss: a stale slot past the fill mark
                    if (hit) { slot += 16; ip += (int)L; cur += L; h = nh; h2 = nh2; mine = nmine; }
                } while (hit && ip < lim && slot != slot_end);
                out.fill += (int)((slot - slot0) >> 4);
                out.slot_s = slot;
                anchor = ip;
                if (!hit) {
                    // a miss: out of reach, or fewer than 4 equal bytes (4..31 would have been a hit)      :1187-1189
                    if (!near || ne != 0) return 0;
                    // 32 equal bytes; cap >= 32 below lim
                    const uint32_t cap = (uint32_t)(mlimit - ip);
                    uint32_t L = 32u;
                    if (cap > 32u) L += count_ahead(ip + 32, src + (m - S) + 32, cap - 32u);
                    out.push((uint32_t)ip, 0u, L - 4, cur - m, in.block);
                    ip += (int)L;
                    anchor = ip;
                } else if (out.fill == kQueueDepth) {
                    out.flush(in.block, 0);
                }
                if (ip >= mfl) return 1;                                                             // :1143
            }
        };

        wait_for(128);
        { t_sweep_to(S); uint2 v = ldg_5bytes(src); t_put(hash5(v.x, v.y), S); }    // :924
        __syncwarp();
        int ip = 1;                            // :925  (search runs start here)
        bool after_match = false;
        bool narrow = false;                   // adaptive probe-window width
        bool first_scalar = false;             // predictor: the previous run hit on its first probe
        const bool ring_probes = in.accel <= 8; // the first probes of a run are (nearly) consecutive positions
        for (;;) {
            bool have = false;
            if (after_match) {
                // ---- put(ip-2), re-test ip (cbits/lz4.c:1146, :1159-1196); ip == anchor here.
                // Loops for as long as a match immediately follows a match.
                int run = 2;
                if constexpr (!kWide && !kCompact) {
                    if (in.dict_len == 0) run = retest_run(ip);
                }
                if (run == 1) goto tail;
                if (run == 2) while (retest_probe(ip)) {
                    out.push((uint32_t)ip, 0u, mlen - 4, dist, in.block);
                    ip += (int)mlen;
                    anchor = ip;
                    if (ip >= mfl) goto tail;                                                        // :1143
                }
                ip++;                                                                                // :1200
            }
            if ((uint32_t)ip + kPrefetchAhead > pf_next) l2_prefetch(ip);
            // ---- a search run starts at ip (cbits/lz4.c:956-1014)
            if (ring_probes && ip >= trigger) move_window(ip);      // dense probing: keep the rings under the first window
            long long jbase = 0;
            if (first_scalar) {                // probe 0 of the run on the scalar path
                if (ip + 1 > mfl) break;                                                             // :969
                have = scalar_probe(ip, false);
                jbase = 1;
            }
            if (!have) {
                // ---- speculative probe windows
                int mpos = 0; uint32_t midx = 0;
                uint32_t width = narrow ? 4u : 32u;
                bool found = false; int hit_index = 0;
                for (;;) {
                    long long off; int step;
                    if (jbase == 0) { off = off0; step = (int)step0; }
                    else if (jbase == 1) { off = off1; step = (int)step1; }
                    else probe_schedule(jbase + lane, in.accel, off, step);
                    const long long pos64 = (long long)ip + off;
                    if (kStreamed && avail < n) {       // the window's farthest probe reads 8 bytes at its position
                        const long long far = __shfl_sync(kFull, pos64, (int)width - 1);
                        wait_for(far + 8);
                    }
                    const bool active = lane < width;
                    bool valid = active && (pos64 + step <= (long long)mfl);                         // :969
                    bool clipped = false;               // compact table: probes past the epoch boundary wait for the sweep
                    if (kCompact) {
                        // lane 0's position becomes insertable -- only if it is a real probe: sweeping to a position that is
                        // never reached would break the "positions only grow" rule the sweep relies on
                        if (__shfl_sync(kFull, (int)valid, 0)) t_sweep_to(S + (uint32_t)__shfl_sync(kFull, (int)pos64, 0));
                        const bool beyond = valid && ((S + (uint32_t)pos64) - tbase >= kRelMax);
                        clipped = __ballot_sync(kFull, beyond) != 0;
                        valid = valid && !beyond;
                    }
                    uint32_t h = 0, seq = 0, cur = 0;
                    const int pos = valid ? (int)pos64 : 0;
                    if (valid) {
                        cur = S + (uint32_t)pos;
                        if (pos >= lo_pos && pos + 8 <= ready_end) {    // bytes and hash are already in the rings
                            seq = ring32(g32 + (uint32_t)pos); h = hash_at(g32 + (uint32_t)pos);
                        } else {
                            uint2 v = ldg_5bytes(src + pos);
                            seq = v.x; h = hash5(v.x, v.y);
                        }
                    }
                    const uint32_t peers = __match_any_sync(kFull, valid ? h : (0x1000u + lane));
                    const uint32_t lower = peers & lanemask_lt();
                    const int from_lane = lower ? (31 - __clz(lower)) : (int)lane;
                    const uint32_t fwd = __shfl_sync(kFull, cur, from_lane);
                    bool ok = false; uint32_t m = 0;
                    if (valid) {
                        m = lower ? fwd : t_get(h);
                        if (!(dict_small && m < low_index) && (m + kMaxDistance >= cur)) {           // :1001-1006
                            if (kWide && (int)(m - S) >= lo_pos && (int)(m - S) + 4 <= ready_end) {      // (a run may have outrun the loaded lines)
                                ok = (ring32(g32 + (m - S)) == seq);
                            } else {
                                const uint8_t* c = (m < S) ? (in.dict_end - (S - m)) : (src + (m - S));  // :985-993
                                ok = (ldg_u32_unaligned(c) == seq);                                  // :1009
                            }
                        }
                    }
                    const uint32_t okb = __ballot_sync(kFull, ok);
                    const uint32_t vb = __ballot_sync(kFull, valid);
                    const int nvalid = __popc(vb);                      // valid lanes form a prefix
                    const int w = okb ? (__ffs(okb) - 1) : 32;
                    const int ncommit = min(w + 1, nvalid);
                    if ((int)lane < ncommit) {                          // ordered commit: last writer per bucket
                        const uint32_t grp = peers & (ncommit >= 32 ? kFull : ((1u << ncommit) - 1u));
                        if ((31 - __clz(grp)) == (int)lane) t_put_lane(h, cur);                      // :998
                    }
                    __syncwarp();
                    if (w < 32) {
                        found = true; hit_index = (int)jbase + w;
                        mpos = __shfl_sync(kFull, pos, w); midx = __shfl_sync(kFull, m, w);
                        break;
                    }
                    if (nvalid < (int)width) {
                        if (kCompact && clipped) { jbase += nvalid; continue; }      // the rest of this window after the sweep
                        break;                                          // ran into mflimit: last literals
                    }
                    jbase += width;
                    width = 32;
                }
                if (!found) break;
                narrow = (in.accel > 16) && (hit_index < 3);
                first_scalar = (hit_index == 0);

                // catch up (cbits/lz4.c:1019), then count (:1076-1095)
                // The backward and the forward extension are independent: the byte pair that decides whether there
                // is anything to catch up is requested before the forward count, so both round trips overlap.
                const bool in_dict = midx < S;
                if (kWide && (int)(midx - S) >= lo_pos && mpos + 4 <= ready_end) {
                    // 4 bytes are known equal; verify_count redoes them from the ring and handles catch-up
                    const bool hit = verify_count(mpos, midx, false);
                    (void)hit;                  // always true: the candidate was accepted on the same bytes
                } else {
                const uint8_t* cand = in_dict ? (in.dict_end - (S - midx)) : (src + (midx - S));
                const uint32_t room_c = in_dict ? (in.dict_len - (S - midx)) : (midx - S);
                const uint32_t maxback = min((uint32_t)(mpos - anchor), room_c);
                uint32_t b_src = 0, b_cand = 1;
                if (maxback) { b_src = __ldg(src + mpos - 1); b_cand = __ldg(cand - 1); }
                uint32_t cap = (uint32_t)(mlimit - mpos);
                if (in_dict) cap = min(cap, (uint32_t)(in.dict_end - cand));
                uint32_t L = 4 + count_ahead(mpos + 4, cand + 4, cap - 4);
                if (in_dict && L == cap && mpos + (int)L < mlimit)
                    L += count_ahead(mpos + (int)L, src, (uint32_t)(mlimit - (mpos + (int)L)));
                const uint32_t back = (b_src == b_cand) ? warp_common_suffix(src + mpos, cand, maxback) : 0u;
                mip = mpos - (int)back;
                mlen = L + back; dist = (S + (uint32_t)mpos) - midx;
                }
            }
            out.push((uint32_t)anchor, (uint32_t)(mip - anchor), mlen - 4, dist, in.block);
            ip = mip + (int)mlen;
            anchor = ip;
            if (ip >= mfl) break;                                                                    // :1143
            after_match = true;
        }
    tail:
        if (kWide) {                    // this array is the next block's dictionary: bring its tail into the ring
            if (n - 1 >= trigger) move_window(n - 1);
            in.w_end = g32 + (uint32_t)n; in.w_lo = g32 + (uint32_t)lo_pos; in.w_ok = true;
        }
        cp_async_wait<0>();             // nothing of this block's window may land after the next block starts
        __syncwarp();
    }
    in.tbase = tbase;
    // last literals, :1204-1231
    out.push((uint32_t)anchor, (uint32_t)(n - anchor), 0u, 0u, in.block);
}

template <bool kWide, bool kCompact, bool kStreamed = false>
__device__ void finder_main(const CompressArgs& a, uint32_t* table, uint32_t* ring, uint16_t* hring, Queue* q)
{
    const uint32_t lane = lane_id();
    uint32_t* counter = &a.scratch->work_counter[0];
    const int accel = a.accel < 1 ? 1 : (a.accel > kAccelMax ? kAccelMax : a.accel);   // :1577-1578
    Producer out{q, 0, 0, 0};
    out.begin();
    const uint32_t data_s = smem_u32(ring), hash_s = smem_u32(hring);
    long long off0, off1; int step0, step1;
    probe_schedule(lane, accel, off0, step0);           // first window of a search run, starting at probe 0
    probe_schedule(lane + 1, accel, off1, step1);       // ... starting at probe 1 (probe 0 was taken by the scalar path)

    for (;;) {
        const int s = claim_stream(counter);
        if (s >= a.n_streams) break;
        const int b0 = stream_begin(a, s), b1 = stream_end(a, s, b0);
        CState* st = a.states ? reinterpret_cast<CState*>(a.states[s]) : nullptr;
        const CState* init = a.states ? st : a.dict_state;                 // where the stream starts from (read only)

        uint32_t offset = 0, dict_len = 0;
        const uint8_t* dict_end = nullptr;
        uint32_t tbase = 0;
        uint16_t* const t16 = reinterpret_cast<uint16_t*>(table);          // compact layout: 4096 x u16, then 128 x u32 epoch bits
        uint32_t* const tfl = table + kHashEntries / 2;
        {   // table: zero (fresh LZ4_initStream, :1443-1451) or restored (the stream's record, or the dictionary's)
            uint4* t4 = reinterpret_cast<uint4*>(table);
            if (init) {
                offset = init->offset; dict_len = init->dict_len;
                dict_end = init->dict_buf + dict_len;
                if (kCompact) {         // positions within reach become rel = pos - tbase + 1 in the lower half, the rest is dropped
                    // (d == 65535 only for the zero entries of a stream that has not compressed anything yet: position 0 == offset)
                    tbase = offset - (kEpoch - 1);
                    for (int k = 0; k < kHashEntries / 32; k++) {
                        const int i = (int)lane + 32 * k;
                        const uint32_t d = init->table[i] - tbase;
                        const uint32_t rel = (d <= kEpoch - 1) ? d + 1u : 0u;
                        t16[i] = (uint16_t)rel;
                        const uint32_t hi = __ballot_sync(kFull, (rel >> 16) != 0);
                        if (lane == 0) tfl[k] = hi;
                    }
                } else {
                    const uint4* g4 = reinterpret_cast<const uint4*>(init->table);
                    for (int i = lane; i < kHashEntries / 4; i += 32) t4[i] = g4[i];
                }
            } else if (kCompact) {      // every bucket = stream position 0 (what a zero-filled table means): rel = 65536
                tbase = 0u - (kEpoch - 1);
                for (int i = lane; i < kHashEntries / 8; i += 32) t4[i] = make_uint4(0, 0, 0, 0);
                for (int i = lane; i < kHashEntries / 32; i += 32) tfl[i] = 0xFFFFFFFFu;
            } else {
                for (int i = lane; i < kHashEntries / 4; i += 32) t4[i] = make_uint4(0, 0, 0, 0);
            }
            __syncwarp();
        }
        auto compact_pos = [&](int i) -> uint32_t {     // stream position held by bucket i of the compact table
            return tbase + ((uint32_t)t16[i] | (((tfl[i >> 5] >> (i & 31)) & 1u) << 16)) - 1u;
        };
        const uint8_t* last_src = nullptr; int last_n = -1;
        uint32_t w_end = 0, w_lo = 0; bool w_ok = false;
        for (int b = b0; b < b1; b++) {
            const uint8_t* src = a.src + a.src_off[b];
            const int n = a.src_len[b];
            if (n >= 0 && n <= kMaxInput) {                                                  // :1262
                if (offset + (uint32_t)n > 0x80000000u) {                                    // LZ4_renormDictT, :1545-1562
                    uint32_t delta = offset - 65536u;
                    if (kCompact) {     // re-express what is still within reach relative to the new origin (tbase = 1), drop the rest
                        uint32_t keep[kHashEntries / 32];
                        #pragma unroll 1
                        for (int k = 0; k < kHashEntries / 32; k++) {
                            const uint32_t p = compact_pos(lane + 32 * k);
                            keep[k] = (offset - p <= kMaxDistance + 1u) ? (p - delta) : 0u;      // new rel = new pos (tbase = 1)
                        }
                        __syncwarp();
                        #pragma unroll 1
                        for (int k = 0; k < kHashEntries / 32; k++) t16[lane + 32 * k] = (uint16_t)keep[k];
                        for (int i = lane; i < kHashEntries / 32; i += 32) tfl[i] = 0u;
                        tbase = 1u;
                    } else {
                        for (int i = lane; i < kHashEntries; i += 32) { uint32_t v = table[i]; table[i] = v < delta ? 0u : v - delta; }
                    }
                    offset = 65536u;
                    if (dict_len > 65536u) dict_len = 65536u;
                    __syncwarp();
                }
                if (dict_len >= 1 && dict_len <= 3) dict_len = 0;                            // :1581-1587
                BlockIn in{src, n, dict_end, dict_len, offset, accel, b, w_end, w_lo, w_ok, tbase, a.arrived, a.seg_bytes, 0, false};
                if (n > 0) offset += (uint32_t)n;                                            // :918 (n == 0 never reaches it, :1263-1273)
                const long long t_begin = kStreamed ? clock64() : 0;
                find_block<kWide, kCompact, kStreamed>(in, table, data_s, hash_s, out, (uint32_t)off0, (uint32_t)step0, (uint32_t)off1, (uint32_t)step1);
                if (kStreamed && a.busy_cycles && lane == 0) {      // what the host's copy schedule is tuned by: finder time net of waiting
                    atomicAdd(a.busy_cycles, (unsigned long long)(clock64() - t_begin - in.stall));
                    atomicAdd(a.busy_cycles + 1, (unsigned long long)n);
                    if (in.timed_out) atomicAdd(a.busy_cycles + 2, 1ull);
                }
                w_end = in.w_end; w_lo = in.w_lo; w_ok = in.w_ok; tbase = in.tbase;
                __syncwarp();
                dict_end = src + n; dict_len = (uint32_t)n;                                  // :1633-1634
                last_src = src; last_n = n;
                out.flush(b, kEndBlock);
            } else {
                out.flush(b, kEndBlock | (1 << 28));      // unsupported size: the emitter reports 0
                w_ok = false;
            }
        }
        if (st) {   // persist the stream (what the reference keeps in LZ4_stream_t + the live previous array)
            if (kCompact) {
                __syncwarp();
                for (int i = lane; i < kHashEntries; i += 32) st->table[i] = compact_pos(i);     // (an empty bucket saves as tbase - 1: out of reach for good)
            } else {
                uint4* g4 = reinterpret_cast<uint4*>(st->table);
                const uint4* t4 = reinterpret_cast<const uint4*>(table);
                for (int i = lane; i < kHashEntries / 4; i += 32) g4[i] = t4[i];
            }
            if (last_n >= 0) {
                uint32_t keep = (uint32_t)last_n <= st->dict_cap ? (uint32_t)last_n : 0u;   // host sizes dict_buf; 0 only on misuse
                if (keep) warp_copy_ro(st->dict_buf, last_src, keep);
                if (lane == 0) { st->offset = offset; st->dict_len = keep; }
            } else if (lane == 0) {
                st->offset = offset; st->dict_len = dict_len;
            }
        }
        __syncwarp();
    }
    out.flush(-1, kTerminate);
}

// encoded length-extension byte count for a nibble value v (0 if v < 15)
__device__ __forceinline__ uint32_t ext_bytes(uint32_t v) { return v >= 15 ? (v - 15) / 255 + 1 : 0; }
__device__ __forceinline__ void write_ext(uint8_t* p, uint32_t v)
{   // v >= 15
    uint32_t rest = v - 15;
    while (rest >= 255) { *p++ = 255; rest -= 255; }
    *p = (uint8_t)rest;
}

__device__ void emitter_main(const CompressArgs& a, Queue* q)
{
    const uint32_t lane = lane_id();
    uint32_t batch = 0;
    long long op = 0;               // bytes of the current block emitted so far
    bool failed = false;
    for (;;) {
        const uint32_t b = batch & 1, t = batch >> 1;
        while (!mbar_test(&q->full[b], t & 1)) __nanosleep(2500);      // idle emitters must not steal issue slots from finders (a queue buffer takes the finder >= 6 us to fill)
        const int cnt_flags = q->count[b];
        const int blk = q->block[b];
        const int cnt = cnt_flags & 0xFFFF;
        if (cnt_flags & kTerminate) break;
        const uint8_t* src = nullptr; uint8_t* dst = nullptr; long long cap = 0;
        if (blk >= 0) {
            src = a.src + a.src_off[blk];
            const int n = a.src_len[blk];
            dst = a.dst + a.dst_off[blk] + a.header;
            cap = a.dst_cap ? (long long)a.dst_cap[blk] - a.header : (long long)n + n / 255 + 16;
        }
        if (cnt_flags & (1 << 28)) failed = true;
        uint4 d = make_uint4(0, 0, 0, 0);
        if ((int)lane < cnt) d = q->desc[b][lane];
        __syncwarp();
        if (lane == 0) mbar_arrive(&q->empty[b]);       // descriptors are in registers: hand the buffer back
        batch++;

        const uint32_t lit = d.y, mcode = d.z, off = d.w;
        const bool is_seq = (int)lane < cnt;
        const uint32_t le = ext_bytes(lit);
        uint32_t size = 0;
        if (is_seq) size = 1 + le + lit + (off ? 2 + ext_bytes(mcode) : 0);
        // inclusive warp scan of sizes (64-bit safe: one block is < 2 GiB + bound)
        uint32_t incl = size;
        #pragma unroll
        for (int dlt = 1; dlt < 32; dlt <<= 1) { uint32_t v = __shfl_up_sync(kFull, incl, dlt); if ((int)lane >= dlt) incl += v; }
        const long long start = op + (long long)(incl - size);
        // limitedOutput guards of the reference, evaluated at this sequence's output position
        bool bad = false;
        if (is_seq) {
            if (off) {
                bad = (start + 1 + lit + (2 + 1 + kLastLiterals) + lit / 255 > cap)                       // :1024-1027
                   || (start + 1 + le + lit + 2 + (1 + kLastLiterals) + (mcode + 240) / 255 > cap);      // :1097-1121
            } else {
                bad = (start + lit + 1 + ((lit + 255 - 15) / 255) > cap);                                // :1207-1217
            }
        }
        if (__ballot_sync(kFull, bad)) failed = true;
        if (!failed && is_seq) {
            uint8_t* p = dst + start;
            *p++ = (uint8_t)((min(lit, 15u) << 4) | (off ? min(mcode, 15u) : 0u));
            if (le) { write_ext(p, lit); p += le; }
            if (lit <= 16) { const uint8_t* s = src + d.x; for (uint32_t i = 0; i < lit; i++) p[i] = (uint8_t)ldg_na_u8(s + i); }
            p += lit;
            if (off) {
                p[0] = (uint8_t)off; p[1] = (uint8_t)(off >> 8);                                         // :1068
                if (mcode >= 15) write_ext(p + 2, mcode);                                                // :1123-1135
            }
        }
        // long literal runs: cooperative copies, one run at a time
        uint32_t longs = __ballot_sync(kFull, !failed && is_seq && lit > 16);
        while (longs) {
            const int l = __ffs(longs) - 1; longs &= longs - 1;
            const uint32_t l_pos = __shfl_sync(kFull, d.x, l), l_len = __shfl_sync(kFull, lit, l);
            const uint32_t l_le = __shfl_sync(kFull, le, l);
            const uint32_t l_rel = __shfl_sync(kFull, incl - size, l);
            warp_copy_ro(dst + op + l_rel + 1 + l_le, src + l_pos, l_len);
        }
        op += (long long)__shfl_sync(kFull, incl, 31);
        if (cnt_flags & kEndBlock) {
            const int r = failed ? 0 : (int)op;
            if (lane == 0 && blk >= 0) {
                uint8_t* slot = a.dst + a.dst_off[blk];
                a.out_len[blk] = r;
                // a slot smaller than its header has failed (cap < 0 above) and is left untouched: the header would land
                // in the next block's slot
                const bool room = !a.dst_cap || a.dst_cap[blk] >= a.header;
                if (room && a.header >= 4) { uint32_t v = (uint32_t)r; for (int k = 0; k < 4; k++) slot[k] = (uint8_t)(v >> (8 * k)); }                 // LZ4.hs:262
                if (room && a.header == 8) { uint32_t v = (uint32_t)a.src_len[blk]; for (int k = 0; k < 4; k++) slot[4 + k] = (uint8_t)(v >> (8 * k)); }   // LZ4.hs:261
            }
            op = 0; failed = false;
        }
    }
}

// Compact tables (see find_block): u16 entries + epoch bits, 8.5 KiB instead of 16 KiB
constexpr int kCompactTableBytes = kHashEntries * 2 + kHashEntries / 8;

// Dynamic shared memory of a compress CTA of kP finder/emitter pairs: hash rings | data rings | tables | queues from a
// 1024-byte aligned start, plus the alignment slack.
template <int kP, bool kWide, bool kCompact>
constexpr size_t compress_smem()
{
    return 1024 + kP * (kHashPos * sizeof(uint16_t) + (kWide ? kWideBytes : kWinBytes)
                        + (kCompact ? kCompactTableBytes : kHashEntries * sizeof(uint32_t)) + sizeof(Queue));
}

// One compress CTA: warps 0 .. kP-1 are the finders, warps kP .. 2kP-1 their emitters.
template <int kP, bool kWide, bool kCompact, bool kStreamed>
__device__ __forceinline__ void compress_cta(const CompressArgs& a)
{
    constexpr uint32_t kRingWords = (kWide ? kWideBytes : kWinBytes) / 4;
    constexpr uint32_t kTableWords = (kCompact ? kCompactTableBytes : kHashEntries * sizeof(uint32_t)) / 4;
    extern __shared__ __align__(16) uint8_t smem_dyn[];
    uint8_t* smem_raw = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    uint16_t* hrings = reinterpret_cast<uint16_t*>(smem_raw);
    uint32_t* rings = reinterpret_cast<uint32_t*>(smem_raw + kP * kHashPos * sizeof(uint16_t));
    uint32_t* tables = rings + kP * kRingWords;
    Queue* queues = reinterpret_cast<Queue*>(tables + kP * kTableWords);
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t pair = warp & (kP - 1);
    if (threadIdx.x < kP) {
        Queue* q = &queues[threadIdx.x];
        mbar_init(&q->full[0], 1); mbar_init(&q->full[1], 1);
        mbar_init(&q->empty[0], 1); mbar_init(&q->empty[1], 1);
    }
    __syncthreads();
    if (warp < kP) finder_main<kWide, kCompact, kStreamed>(a, tables + pair * kTableWords, rings + pair * kRingWords,
                                                            hrings + pair * kHashPos, &queues[pair]);
    else emitter_main(a, &queues[pair]);
    release_counters(a.scratch, 0);
}

__global__ void __launch_bounds__(kPairs * 64, 3)
compress_kernel(CompressArgs a) { compress_cta<kPairs, false, false, false>(a); }

// Streamed launches (host batch calls, see api.cu): the classic geometry, finders wait for their input segment by segment.
__global__ void __launch_bounds__(kPairs * 64, 3)
compress_kernel_streamed(CompressArgs a) { compress_cta<kPairs, false, false, true>(a); }

// Compact mode: the dense kernel with 8.5 KiB position tables (see find_block): 4 CTAs of 4 pairs per SM = 16 streams in
// flight per SM instead of 12.  Used for launches of more than one wave of the classic kernel.
__global__ void __launch_bounds__(kPairs * 64, 4)
compress_kernel_compact(CompressArgs a) { compress_cta<kPairs, false, true, false>(a); }

// Wide mode: one finder/emitter pair per CTA, one CTA per SM (144 KiB: hash ring | 128 KiB data ring | table | queue).
// Used when a launch has no more streams than the device has SMs (few linked streams, few large blocks, the tail
// chunk of a host batch): per-stream latency is all that matters then.
__global__ void __launch_bounds__(64, 1)
compress_kernel_wide(CompressArgs a) { compress_cta<1, true, false, false>(a); }

__global__ void set_flag_kernel(uint32_t* flag, uint32_t v) { *flag = v; __threadfence(); }

// Stream-aliasing self-test (api.cu: probe_stream_aliasing): spins until *flag != 0 or `timeout` cycles have passed and
// reports which; `successor_kernel` is the entry queued behind it in the same stream.
__global__ void alias_probe_kernel(const uint32_t* flag, uint32_t* result, long long timeout)
{
    const long long t0 = clock64();
    uint32_t v = 0;
    for (;;) {
        v = ld_acquire_sys(flag);
        if (v || clock64() - t0 > timeout) break;
        __nanosleep(500);
    }
    *result = v ? 1u : 2u;
}
__global__ void successor_kernel(uint32_t* result) { result[1] = 1u; }

}  // namespace

// stream-ordered store of one arrival flag (the alternative to a 4-byte copy: B200LZ4_STREAM_FLAG=kernel)
cudaError_t launch_set_flag(uint32_t* flag, uint32_t v, cudaStream_t stream)
{
    set_flag_kernel<<<1, 1, 0, stream>>>(flag, v);
    return cudaGetLastError();
}

cudaError_t preload_compress_kernels()
{
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, compress_kernel_streamed);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, set_flag_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, compress_kernel);
    return e;
}

cudaError_t launch_alias_probe(const uint32_t* flag, uint32_t* result, long long timeout_cycles, cudaStream_t stream)
{
    alias_probe_kernel<<<1, 1, 0, stream>>>(flag, result, timeout_cycles);
    successor_kernel<<<1, 1, 0, stream>>>(result);
    return cudaGetLastError();
}

cudaError_t launch_compress(const CompressArgs& a, cudaStream_t stream)
{
    constexpr size_t smem = compress_smem<kPairs, false, false>();         // classic and streamed
    constexpr size_t kCompactSmem = compress_smem<kPairs, false, true>(), kWideSmem = compress_smem<1, true, false>();
    int sm_count = 0;
    cudaError_t e = device_sm_count(&sm_count); if (e != cudaSuccess) return e;
    static PerDeviceOnce once;
    e = once.run([&] {
        cudaError_t r = cudaFuncSetAttribute(compress_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (r == cudaSuccess) r = cudaFuncSetAttribute(compress_kernel_streamed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (r == cudaSuccess) r = cudaFuncSetAttribute(compress_kernel_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWideSmem);
        if (r == cudaSuccess) r = cudaFuncSetAttribute(compress_kernel_compact, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCompactSmem);
        if (r == cudaSuccess && getenv("B200LZ4_DEBUG")) {
            int occ = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, compress_kernel, kPairs * 64, smem);
            fprintf(stderr, "[b200lz4] compress_kernel: %zu B dynamic smem, %d CTAs/SM, %d SMs\n", smem, occ, sm_count);
        }
        return r;
    });
    if (e != cudaSuccess) return e;
    if (a.n_streams <= 0) return cudaSuccess;
    if (a.arrived) {                             // input still arriving: classic geometry, finders poll a.arrived
        const int want = (a.n_streams + kPairs - 1) / kPairs, max_ctas = sm_count * 3;
        compress_kernel_streamed<<<want < max_ctas ? want : max_ctas, kPairs * 64, smem, stream>>>(a);
        return cudaGetLastError();
    }
    static const bool no_wide = getenv("B200LZ4_NO_WIDE") != nullptr;     // A/B switch for measurements
    if (a.n_streams <= sm_count && !no_wide) {   // few streams: one per SM with everything in shared memory
        compress_kernel_wide<<<a.n_streams, 64, kWideSmem, stream>>>(a);
        return cudaGetLastError();
    }
    static const char* compact_env = getenv("B200LZ4_COMPACT");           // A/B switch: "0" never, "1" always (when not wide)
    const bool compact = compact_env ? (compact_env[0] == '1') : (a.n_streams > sm_count * 3 * kPairs);
    if (compact) {                               // more than one wave of the classic kernel: 16 streams per SM instead of 12
        const int max_c = sm_count * 4, want_c = (a.n_streams + kPairs - 1) / kPairs;
        compress_kernel_compact<<<want_c < max_c ? want_c : max_c, kPairs * 64, kCompactSmem, stream>>>(a);
        return cudaGetLastError();
    }
    const int ctas_per_sm = 3;                   // 3 x (64 KiB of tables + queues) per SM
    const int max_ctas = sm_count * ctas_per_sm;
    const int want = (a.n_streams + kPairs - 1) / kPairs;
    const int grid = want < max_ctas ? want : max_ctas;
    compress_kernel<<<grid, kPairs * 64, smem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace b200lz4
