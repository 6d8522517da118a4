// decompress.cu -- LZ4 block decoder for sm_100a.
//
// Semantics: LZ4_decompress_safe_continue restricted to non-adjacent outputs
// (cbits/lz4.c:2322-2359), i.e. LZ4_decompress_generic(endOnInputSize,
// decode_full_block, {noDict | usingExtDict with the previous output})
// (cbits/lz4.c:1737-2165; the safe loop :1929-2151 defines the accept/reject rules).
//
// Organisation: one CTA of two warps per stream (independent mode: per block).
//
//   PARSER warp -- walks the token chain, the only inherently serial part
//     (token -> literal length -> offset -> match length -> next token).  The compressed
//     payload is streamed into a 4 KiB shared-memory ring with cp.async (16 bytes per lane,
//     well ahead of the parse point), so one step of the chain costs a couple of
//     shared-memory round trips.  The parser applies every accept/reject rule of the safe
//     decoder (it tracks the output position) and hands (literal start, literal length,
//     match length, offset) descriptors to the copier through a double-buffered queue
//     (mbarrier full/empty handshakes).
//   COPIER warp -- executes up to 32 sequences at a time.  Output is assembled in an 8 KiB
//     shared-memory ring and flushed to global memory with 128-bit stores, so matches with
//     near offsets never touch L2 and global writes are coalesced.
//       phase A  lane j copies the literals of sequence j (input ring -> output ring) and,
//                if the match of sequence j only reads bytes produced before this batch,
//                its match bytes as well: 32 sequences in parallel;
//       phase B  matches that read bytes produced inside the batch run in order, each one
//                copied by all lanes (overlapping matches are a periodic source);
//       bulk     sequences with a long literal run or a long match travel alone and are
//                copied cooperatively global -> global.
#include <cstdlib>
#include <mutex>
#include "decode_common.cuh"

namespace b200lz4 {

using namespace dec;

namespace {

struct __align__(16) DQueue {
    uint4 desc[2][kQDepth];              // short: {literal start (ring space), lit | mlen << 8 | offset << 16, output position, -}
                                         // bulk:  {literal start (ring space), literal length, match length (0 = none), offset}
    unsigned long long full[2], empty[2];
    int count[2];
    int block[2];
    int stream[2];
    int result[2];
};

// ------------------------------------------------------------------ parser ----

struct Parser {
    static constexpr bool kWide = false;
    static constexpr int kRing = kInRing;
    DQueue* q;
    uint32_t ring_s;            // shared address of the input ring
    // queue producer state
    uint32_t batch;             // batches published so far
    int fill;                   // descriptors in the buffer being filled
    uint32_t slot_s;            // shared address of the next descriptor slot
    int flags;                  // flags to attach to the buffer being filled
    // batch bounds (ring space / output space)
    int cur_start;              // ring-space position where the current batch starts
    int prev_start;             // ... where the previously published batch starts
    bool prev_pending;          // that batch may still be read by the copier
    // input ring state (ring space: payload index + skew, so that 16-byte granules are aligned in both spaces)
    const uint8_t* gbase;       // global address of ring-space position 0
    int end;                    // ring-space end of the payload
    int issued_end, ready_end;  // fills issued / complete and visible, ring space (multiples of kFill)
    int block, stream;

    __device__ __forceinline__ void begin()
    {   // wait until the buffer we are about to fill has been drained
        const uint32_t b = batch & 1, t = batch >> 1;
        if (t) mbar_wait(&q->empty[b], (t - 1) & 1);
        slot_s = smem_u32(&q->desc[b][0]);
        fill = 0;
    }
    // publish the current buffer (possibly empty) with extra flags
    __device__ __forceinline__ void publish(int extra, int result, int ip)
    {
        const uint32_t b = batch & 1;
        cp_async_wait_all();            // literal bytes of this batch must have landed before the copier is told
        if (lane_id() == 0) { q->count[b] = fill | flags | extra; q->block[b] = block; q->stream[b] = stream; q->result[b] = result; }
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(&q->full[b]);
        ready_end = issued_end;
        batch++;
        flags = 0;
        prev_start = cur_start; prev_pending = true;
        cur_start = ip;
        begin();                        // the buffer of the batch before the one just published is now free ...
        // ... so only the batch just published can still be pending
    }
    __device__ __forceinline__ void push(uint32_t lit_src, uint32_t lit, uint32_t mlen, uint32_t off, int /*op_after*/ = 0)
    {
        if (lane_id() == 0) sts128(slot_s, lit_src, lit, mlen, off);
        slot_s += 16;
        fill++;
    }
    // window path: lane-parallel descriptor stores, then the batch grows by n
    __device__ __forceinline__ void put(uint32_t rank, uint32_t x, uint32_t y, uint32_t z, uint32_t w) { sts128(slot_s + 16u * rank, x, y, z, w); }
    __device__ __forceinline__ void advance(int n, int /*op_after*/) { slot_s += 16u * (uint32_t)n; fill += n; }
    // a long sequence travels alone
    __device__ __forceinline__ void push_bulk(uint32_t lit_src, uint32_t lit, uint32_t mlen, uint32_t off, int /*op_seq*/, int ip_after)
    { push(lit_src, lit, mlen, off); publish(kBulk, 0, ip_after); }
    __device__ __forceinline__ void note_reach(int) {}
    __device__ __forceinline__ uint32_t at(int p) const { return lds8(ring_s + ((uint32_t)p & (kInRing - 1))); }

    // issue ring fills ahead of ip as far as the copier's needs allow
    __device__ __forceinline__ void top_up(int ip)
    {
        const int lo_needed = prev_pending ? prev_start : cur_start;
        while (issued_end < end && issued_end - ip < 2048 && issued_end + kFill - kInRing <= lo_needed) {
            const int p = issued_end + 16 * (int)lane_id();
            if (p < end) cp_async_16(ring_s + ((uint32_t)p & (kInRing - 1)), gbase + p);
            cp_async_commit();
            issued_end += kFill;
        }
    }
    // make ring bytes [.., need) readable, need <= ip + 64 (or report that the payload ends before)
    __device__ void ensure(int ip, int need)
    {
        if (need <= ready_end) return;
        if (ip >= issued_end) {                         // jumped over everything requested so far: restart at ip
            cp_async_wait_all();
            issued_end = ip & ~(kFill - 1);
            ready_end = issued_end;
        }
        for (;;) {
            top_up(ip);
            if (need <= issued_end || issued_end >= end) break;
            // blocked: the ring would overwrite bytes the copier may still read
            if (prev_pending) {
                const uint32_t pb = (batch - 1) & 1, t = (batch - 1) >> 1;
                mbar_wait(&q->empty[pb], t & 1);
                prev_pending = false;
            } else {
                publish(0, 0, ip);                      // the current batch itself pins the ring: hand it over
            }
        }
        cp_async_wait_all();
        __syncwarp();
        ready_end = issued_end;
    }
};

template <bool kWindow>
__device__ void parser_main(const DecompressArgs& a, DQueue* q, uint32_t ring_s)
{
    uint32_t* counter = &a.scratch->work_counter[2];
    Parser P;
    P.q = q; P.ring_s = ring_s; P.batch = 0; P.fill = 0; P.flags = 0; P.prev_pending = false; P.prev_start = 0; P.cur_start = 0;
    P.block = -1; P.stream = -1;
    P.begin();
    for (;;) {
        const int s = claim_stream(counter);
        if (s >= a.n_streams) break;
        const int b0 = stream_begin(a, s), b1 = stream_end(a, s, b0);
        const DState* st = a.states ? reinterpret_cast<const DState*>(a.states[s]) : a.dict_state;   // the stream's record, or the dictionary's
        uint32_t dict_len = st ? st->prev_len : 0u;
        for (int b = b0; b < b1; b++) {
            const BlockGeom g = block_geom(a, b);
            P.block = b; P.stream = s;
            if (P.prev_pending) {       // the copier may still read literals of the previous block from the ring
                const uint32_t pb = (P.batch - 1) & 1, t = (P.batch - 1) >> 1;
                mbar_wait(&q->empty[pb], t & 1);
                P.prev_pending = false;
            }
            P.flags = kBegin | (b == b0 ? kStreamBegin : 0);
            int r = -1;
            if (g.ok) {
                const int skew = (int)(reinterpret_cast<uintptr_t>(g.payload) & 15);
                P.gbase = g.payload - skew;
                r = parse_block(P, skew, g.comp_len, g.cap, dict_len);
            }
            P.publish(kEndBlock | (b == b1 - 1 ? kStreamEnd : 0), r, 0);
            if (kWindow) { if (r > 0) dict_len = min(65536u, dict_len + (uint32_t)r); }   // the last 64 KiB of the stream's output
            else if (r > 0) dict_len = (uint32_t)r;                    // cbits/lz4.c:2353-2355
        }
    }
    P.publish(kTerminate, 0, 0);
}

// ------------------------------------------------------------------ copier ----

struct Copier {
    uint32_t in_s, out_s;       // shared addresses of the rings
    uint8_t* dst;               // output of the current block
    uint8_t* hdst;              // kMirror: the block's place in the caller's page-locked HOST buffer (same address modulo 16 as dst)
    uint32_t oskew;             // (address of dst) & 15: ring index of output position q is (q + oskew) & (kOutRing - 1)
    int op;                     // output bytes produced so far
    int flushed;                // output positions below this are in global memory
    int ring_lo;                // output positions below this are NOT in the ring (bulk copies bypass it)
    const uint8_t* dict_end; uint32_t dict_len;
    int cap;                    // capacity of the current block's destination (bounds-check builds)

    __device__ __forceinline__ uint32_t oidx(int q) const { return out_s + (((uint32_t)q + oskew) & (kOutRing - 1)); }

    // Make the ring hold the 64 output positions below `upto` (taken from global memory / the previous output),
    // so that a short match that reaches back across a block start or a bulk copy still reads the ring.
    __device__ void preload(int upto)
    {
        const uint32_t lane = lane_id();
        #pragma unroll
        for (int k = 0; k < 2; k++) {
            const int qd = upto - 64 + (int)lane + 32 * k;
            uint32_t bb = 0;
            if (qd >= 0) bb = dst[qd];
            else if ((uint32_t)(-qd) <= dict_len && (uint32_t)(-qd) <= 65536u) bb = dict_end[qd];
            sts8(oidx(qd), bb);
        }
        ring_lo = upto - 64;
    }
    // ring -> global for output positions [flushed, upto); unless `all`, stops at the last 16-byte boundary.
    // kMirror: every store goes to the host buffer as well (posted PCIe writes, 512 contiguous bytes per warp instruction), so
    // the output is on its way home while the block is still being decoded and no D2H copy follows the kernel.
    template <bool kMirror>
    __device__ void flush(int upto, bool all)
    {
        const uint32_t lane = lane_id();
        int lo = flushed, hi = upto;
        if (!all) hi = (int)((((uint32_t)upto + oskew) & ~15u) - oskew);
        if (hi <= lo) return;
#ifdef B200LZ4_BOUNDS_CHECK
        if (lo < 0 || hi > cap) __trap();
#endif
        uint32_t head = (16u - (((uint32_t)lo + oskew) & 15u)) & 15u;
        if (head > (uint32_t)(hi - lo)) head = (uint32_t)(hi - lo);
        if (lane < head) { const uint8_t bb = (uint8_t)lds8(oidx(lo + (int)lane)); dst[lo + (int)lane] = bb; if (kMirror) hdst[lo + (int)lane] = bb; }
        lo += (int)head;
        const uint32_t nvec = (uint32_t)(hi - lo) >> 4;
        for (uint32_t v = lane; v < nvec; v += 32) {
            const int qv = lo + (int)(v << 4);
            const uint4 x = lds128(oidx(qv));
            *reinterpret_cast<uint4*>(dst + qv) = x;
            if (kMirror) *reinterpret_cast<uint4*>(hdst + qv) = x;
        }
        lo += (int)(nvec << 4);
        const uint32_t tail = (uint32_t)(hi - lo);
        if (lane < tail) { const uint8_t bb = (uint8_t)lds8(oidx(lo + (int)lane)); dst[lo + (int)lane] = bb; if (kMirror) hdst[lo + (int)lane] = bb; }
        flushed = hi;
    }
};

// kPublish (streamed host call, api.cu: decompress_host_streamed): the launch's blocks all have the same capacity and the
// host sends their output home segment by segment while they are still being decoded.  Whenever a block's flushed
// prefix crosses a segment boundary the copier counts it in seg_count[s]; the block that completes segment s for the
// whole launch raises host_ready[s] (page-locked host memory the calling thread polls).
template <bool kPublish, bool kMirror, bool kWindow>
__device__ void copier_main(const DecompressArgs& a, DQueue* q, uint32_t in_s, uint32_t out_s)
{
    const uint32_t lane = lane_id();
    int pub = 0;                            // segments of the current block already counted
    auto publish = [&](int upto) {          // upto: number of leading segments of the current block that are in global memory
        if (!kPublish) return;
        if (pub >= upto) return;
        __threadfence();                    // every lane's stores of those segments are visible device-wide ...
        __syncwarp();
        if (lane == 0) {
            for (int sgm = pub; sgm < upto; sgm++) {
                const uint32_t before = atomicAdd(a.seg_count + sgm, 1u);       // ... before the block is counted
                if (before + 1u == (uint32_t)a.n_streams) {
                    __threadfence_system();
                    *(volatile uint32_t*)(a.host_ready + sgm) = 1u;
                }
            }
        }
        __syncwarp();
        pub = upto;
    };
    Copier C;
    C.in_s = in_s; C.out_s = out_s; C.dst = nullptr; C.hdst = nullptr; C.oskew = 0; C.op = 0; C.flushed = 0; C.ring_lo = 0;
    C.dict_end = nullptr; C.dict_len = 0; C.cap = 0;
    const uint8_t* gbase = nullptr;         // global address of input ring-space position 0
    const uint8_t* last_out = nullptr; int last_len = 0;
    uint32_t batch = 0;
    for (;;) {
        const uint32_t b = batch & 1, t = batch >> 1;
        mbar_wait(&q->full[b], t & 1);
        const int cf = q->count[b];
        const int blk = q->block[b];
        const int cnt = cf & kCountMask;
        if (cf & kTerminate) break;
        uint4 d = make_uint4(0, 0, 0, 0);
        if ((int)lane < cnt) d = q->desc[b][lane];
        if (cf & kBegin) {
            const BlockGeom g = block_geom(a, blk);
            C.dst = g.out; C.oskew = (uint32_t)(reinterpret_cast<uintptr_t>(g.out) & 15); C.cap = g.cap;
            if (kMirror) C.hdst = a.host_dst + a.dst_off[blk];
            C.op = 0; C.flushed = 0; C.ring_lo = 0;
            pub = 0;
            gbase = g.payload - (reinterpret_cast<uintptr_t>(g.payload) & 15);
            if (cf & kStreamBegin) {
                const DState* st = a.states ? reinterpret_cast<const DState*>(a.states[q->stream[b]]) : a.dict_state;
                C.dict_end = nullptr; C.dict_len = 0; last_out = nullptr; last_len = 0;
                if (st && st->prev_len) { C.dict_len = st->prev_len; C.dict_end = st->tail + 65536; }
            }
            if (C.dict_len) { C.preload(0); __syncwarp(); }
        }
        const int result = q->result[b];
        const int stream = q->stream[b];
        uint8_t* const dst = C.dst;

        if (a.debug & 1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&q->empty[b]);
        } else if (cf & kBulk) {
            // ---- one long sequence, copied cooperatively global -> global
            __syncwarp();
            if (lane == 0) mbar_arrive(&q->empty[b]);
            const uint32_t lit_src = __shfl_sync(kFull, d.x, 0), lit = __shfl_sync(kFull, d.y, 0);
            const uint32_t mlen = __shfl_sync(kFull, d.z, 0), dist = __shfl_sync(kFull, d.w, 0);
            C.template flush<kMirror>(C.op, true);
            __syncwarp();
            BCHK(a, C.op >= 0 && (long long)C.op + lit + mlen <= (long long)C.cap);
            const int bulk_start = C.op;
            if (lit) warp_copy_ro(dst + C.op, gbase + lit_src, lit);
            int op = C.op + (int)lit;
            __syncwarp();
            if (mlen) {
                int from = op - (int)dist;
                uint8_t* out = dst + op;
                uint32_t mrest = mlen;
                if (from < 0) {                                        // starts in the previous output (:2075-2100):
                    const uint32_t nd = min(mrest, (uint32_t)(-from)); // that part first, the rest is an ordinary match from position 0
                    for (uint32_t i = lane; i < nd; i += 32) out[i] = C.dict_end[from + (int)i];
                    __syncwarp();
                    out += nd; from += (int)nd; mrest -= nd;
                }
                const uint32_t mlen = mrest;                           // (shadows: what is left to copy from this block's own output)
                if (mlen == 0) {
                } else if (dist >= mlen) {
                    warp_copy_rw(out, dst + from, mlen);
                } else if (dist >= 32) {                               // overlapping: rounds of one period each
                    for (uint32_t done = 0; done < mlen; done += dist) {
                        const uint32_t n = min(dist, mlen - done);
                        warp_copy_rw(out + done, dst + from + done, n);
                        __syncwarp();
                    }
                } else {                                               // short period: the source is dist bytes repeated
                    const uint32_t pat = dst[from + (int)(lane < dist ? lane : 0u)];
                    uint32_t k = lane % dist;
                    const uint32_t adv = 32 % dist;
                    for (uint32_t i0 = 0; i0 < mlen; i0 += 32) {
                        const uint32_t i = i0 + lane;
                        const uint32_t bb = __shfl_sync(kFull, pat, k);
                        if (i < mlen) out[i] = (uint8_t)bb;
                        k += adv; if (k >= dist) k -= dist;
                    }
                }
            }
            op += (int)mlen;
            __syncwarp();
            if (kMirror) { warp_copy_rw(C.hdst + bulk_start, dst + bulk_start, (uint32_t)(op - bulk_start)); __syncwarp(); }
            C.op = op; C.flushed = op;
            C.preload(op);
            __syncwarp();
            if (kPublish && C.flushed >= (pub + 1) * a.seg_bytes) publish(min(C.flushed / a.seg_bytes, a.n_segs - 1));
        } else if (cnt) {
            // ---- up to 32 short sequences
            constexpr uint32_t M = kOutRing - 1;
            const uint32_t lit = d.y & 0xFFu, mlen = (d.y >> 8) & 0xFFu, dist = d.y >> 16;
            const int lit_dst = (int)d.z;
            const int op0 = C.op;
            const int op1 = __shfl_sync(kFull, lit_dst + (int)(lit + mlen), cnt - 1);
            const int m_dst = lit_dst + (int)lit;
            const int from = m_dst - (int)dist;
            C.template flush<kMirror>(op0, false);     // previous batches leave for global memory (128-bit stores)
            if (kPublish && C.flushed >= (pub + 1) * a.seg_bytes) publish(min(C.flushed / a.seg_bytes, a.n_segs - 1));
            BCHK(a, op0 >= 0 && op1 >= op0 && op1 <= C.cap);
            const int ring_base = max(C.ring_lo, op1 - kOutRing);       // output positions >= this are in the ring; below: in global memory
            const uint32_t oskew = C.oskew;
            // phase A: literals (lane per sequence)
            {
                const uint32_t sl = d.x, dl = (uint32_t)lit_dst + oskew;
                for (uint32_t i = 0; i < lit; i++) sts8(out_s + ((dl + i) & M), lds8(in_s + ((sl + i) & (kInRing - 1))));
            }
            __syncwarp();
            // phase A: matches whose source was complete before this batch
            const bool has_match = mlen != 0;
            const bool indep = has_match && (from + (int)mlen <= op0);
            const uint32_t sa = (uint32_t)from + oskew, da = (uint32_t)m_dst + oskew;     // ring-space source / destination
            if (indep) {
                if (from >= ring_base) {                                // source in the ring
                    for (uint32_t i = 0; i < mlen; i++) sts8(out_s + ((da + i) & M), lds8(out_s + ((sa + i) & M)));
                } else if (from >= 0) {                                 // source already flushed (from + mlen <= flushed)
                    // aligned 32-bit loads, four bytes per round trip (never touches a word that holds no source byte)
                    const uintptr_t ga = reinterpret_cast<uintptr_t>(dst + from);
                    const uint32_t* gw = reinterpret_cast<const uint32_t*>(ga & ~uintptr_t(3));
                    const uint32_t sh = (uint32_t)(ga & 3) * 8;
                    const uint32_t nwords = ((uint32_t)(ga & 3) + mlen + 3) >> 2;
                    uint32_t w0 = gw[0];
                    for (uint32_t i = 0, k = 1; i < mlen; i += 4, k++) {
                        const uint32_t w1 = k < nwords ? gw[k] : 0u;
                        const uint32_t v = __funnelshift_r(w0, w1, sh);
                        w0 = w1;
                        const uint32_t n = min(4u, mlen - i);
                        sts8(out_s + ((da + i) & M), v & 0xFFu);
                        if (n > 1) sts8(out_s + ((da + i + 1) & M), (v >> 8) & 0xFFu);
                        if (n > 2) sts8(out_s + ((da + i + 2) & M), (v >> 16) & 0xFFu);
                        if (n > 3) sts8(out_s + ((da + i + 3) & M), v >> 24);
                    }
                } else {                                                // starts in the previous output (:2075-2100)
                    for (uint32_t i = 0; i < mlen; i++) {
                        const int f = from + (int)i;
                        uint32_t bb;
                        if (f < 0) bb = C.dict_end[f];
                        else if (f >= ring_base) bb = lds8(out_s + ((sa + i) & M));
                        else bb = dst[f];
                        sts8(out_s + ((da + i) & M), bb);
                    }
                }
            }
            __syncwarp();
            // phase B: matches that read bytes of this batch, in order, each copied by all lanes.  Their sources lie
            // within 64 bytes of the batch start, which the ring always holds (see preload()).
            const uint32_t dep = __ballot_sync(kFull, has_match && !indep);
            if (dep) {
                // every lane leaves the parameters of its match in the (already consumed) descriptor slot, so the loop
                // reads one broadcast 128-bit word per match instead of shuffling
                const uint32_t par_s = smem_u32(&q->desc[b][0]);
                sts128(par_s + 16u * lane, da, mlen, dist, overlap_inv(dist, mlen));
                __syncwarp();
                copy_near_matches<M>(out_s, par_s, dep, lane);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&q->empty[b]);  // literals copied, descriptor slots no longer in use
            C.op = op1;
        } else {
            __syncwarp();
            if (lane == 0) mbar_arrive(&q->empty[b]);
        }
        batch++;

        if (cf & kEndBlock) {
            if (result >= 0 && dst) { C.template flush<kMirror>(C.op, true); __syncwarp(); }
            if (kPublish) publish(a.n_segs);           // the block is over (short, failed or complete): nothing more will come
            if (lane == 0) a.out_len[blk] = result;
            if (kWindow) {                                 // the next block starts where this one ended; its dictionary is the
                if (!(cf & kStreamEnd) && lane == 0)       // stream's last min(64 KiB, bytes so far) bytes, right below it
                    const_cast<int64_t*>(a.dst_off)[blk + 1] = a.dst_off[blk] + (result > 0 ? result : 0);
                if (result > 0) { C.dict_end = dst + result; C.dict_len = min(65536u, C.dict_len + (uint32_t)result); }
            } else if (result > 0) { C.dict_end = dst + result; C.dict_len = (uint32_t)result; last_out = dst; last_len = result; }   // cbits/lz4.c:2353-2355
            if ((cf & kStreamEnd) && a.states && last_out) {   // keep the reachable tail of the last output for the next call
                DState* st = reinterpret_cast<DState*>(a.states[stream]);
                const uint32_t kept = last_len < 65536 ? (uint32_t)last_len : 65536u;
                const uint8_t* fromp = last_out + last_len - kept;
                uint8_t* to = st->tail + 65536 - kept;
                __syncwarp();
                for (uint32_t i = lane; i < kept; i += 32) to[i] = fromp[i];
                if (lane == 0) { st->prev_len = (uint32_t)last_len; st->kept = kept; }
            }
            __syncwarp();
        }
    }
}

// Two register budgets: 16 CTAs per SM (64 registers, a few spilled bytes) when a launch has more than 12 streams per SM
// to keep busy, 12 CTAs per SM (80 registers, no spills) when everything is resident anyway -- measured +6 % on config 2's
// single wave, -12 % on 16 384 blocks of 64 KiB if used there.
template <int kCtasPerSm, bool kPublish = false, bool kMirror = false, bool kWindow = false>
__global__ void __launch_bounds__(64, kCtasPerSm)
decompress_kernel(DecompressArgs a)
{
    __shared__ __align__(16) uint8_t in_ring[kInRing];
    __shared__ __align__(16) uint8_t out_ring[kOutRing];
    __shared__ DQueue queue;
    if (threadIdx.x == 0) {
        mbar_init(&queue.full[0], 1); mbar_init(&queue.full[1], 1);
        mbar_init(&queue.empty[0], 1); mbar_init(&queue.empty[1], 1);
    }
    __syncthreads();
    uint32_t in_s, out_s;       // laundered so that the compiler keeps them in registers instead of re-deriving them in the hot loops
    asm volatile("mov.u32 %0, %1;" : "=r"(in_s) : "r"(smem_u32(in_ring)));
    asm volatile("mov.u32 %0, %1;" : "=r"(out_s) : "r"(smem_u32(out_ring)));
    if (threadIdx.x < 32) parser_main<kWindow>(a, &queue, in_s);
    else copier_main<kPublish, kMirror, kWindow>(a, &queue, in_s, out_s);
    release_counters(a.scratch, 2);
}

// 12 CTAs per SM while every stream gets a CTA of its own, else 16 per SM (one wave; CTAs claim further streams)
template <bool kPublish, bool kMirror, bool kWindow = false>
cudaError_t launch_narrow(const DecompressArgs& a, int sm_count, cudaStream_t stream)
{
    if (a.n_streams <= sm_count * 12) decompress_kernel<12, kPublish, kMirror, kWindow><<<a.n_streams, 64, 0, stream>>>(a);
    else {
        const int max_ctas = sm_count * 16;
        decompress_kernel<16, kPublish, kMirror, kWindow><<<a.n_streams < max_ctas ? a.n_streams : max_ctas, 64, 0, stream>>>(a);
    }
    return cudaGetLastError();
}

}  // namespace

// SM count per device, looked up once (thread-safe: several host threads launch on different devices)
cudaError_t device_sm_count(int* out)
{
    static std::mutex mu;
    static int sm_counts[64] = {0};
    int dev = 0; cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lk(mu);
    if (!sm_counts[dev]) { e = cudaDeviceGetAttribute(&sm_counts[dev], cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e; }
    *out = sm_counts[dev];
    return cudaSuccess;
}

cudaError_t launch_decompress(const DecompressArgs& a, cudaStream_t stream)
{
    int sm_count = 0;
    cudaError_t e0 = device_sm_count(&sm_count); if (e0 != cudaSuccess) return e0;
    if (a.n_streams <= 0) return cudaSuccess;
    static const char* dbg = getenv("B200LZ4_DECODE_DEBUG");
    static const char* wide_env = getenv("B200LZ4_DWIDE");           // A/B switch: "0" never, "1" whenever the arena allows
    DecompressArgs b = a;
    b.debug = dbg ? atoi(dbg) : 0;
    // Wide kernel (one stream per SM: parallel block parsers + a copier pipeline): LINKED streams when there are few enough of
    // them that the narrow kernel would leave most of the GPU idle (measured: 128 streams 17 -> 35 GB/s on mixed data, 11 ->
    // 49 GB/s on text; with more than two streams per SM the narrow kernel's 16 CTAs per SM win).  Independent blocks gain
    // nothing from it -- a block has ONE token chain, so only one of the eight parsers would work.
    if (a.host_dst)                         // host call with a page-locked destination: the output goes home from inside the kernel
        return launch_narrow<false, true>(b, sm_count, stream);
    if (a.seg_count)                        // streamed host call: independent blocks, output leaves segment by segment
        return launch_narrow<true, false>(b, sm_count, stream);
    bool wide = a.stream_first != nullptr && a.n_streams <= 2 * sm_count;
    if (wide_env) wide = wide_env[0] == '1';
    if (wide && a.wide_arena) return launch_decompress_wide(b, sm_count, stream);
    return launch_narrow<false, false>(b, sm_count, stream);
}

cudaError_t launch_decompress_window(const DecompressArgs& a, cudaStream_t stream)
{
    int sm_count = 0;
    cudaError_t e0 = device_sm_count(&sm_count); if (e0 != cudaSuccess) return e0;
    if (a.n_streams <= 0) return cudaSuccess;
    return launch_narrow<false, false, true>(a, sm_count, stream);
}

}  // namespace b200lz4
