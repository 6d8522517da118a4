// decode_common.cuh -- what the two decoder kernels share: constants, the in-order copy of matches that read recent
// output (copy_near_matches, with overlap_inv), the block geometry of decompressChunk and the block PARSER (parse_block),
// which walks the token chain of one LZ4 block with every accept/reject rule of the reference's safe decoder
// (cbits/lz4.c:1929-2151) and hands sequence descriptors to a sink PT:
//     decompress.cu       Parser   -- shared-memory double buffer read by ONE copier warp        (kWide == false)
//     decompress_wide.cu  WParser  -- global-memory descriptor ring read by several copier warps (kWide == true)
// Sink interface: kWide, kRing; ring_s, end, issued_end, ready_end, cur_start, fill; at(p), top_up(ip), ensure(ip, need),
// put(rank, x, y, z, w) / advance(n, op_after) for the lane-parallel window path, push(x, y, z, w, op_after) for one short
// sequence, push_bulk(lit_src, lit, mlen, dist, op_seq, ip_after) for a long one, publish(extra, result, ip),
// note_reach(bytes before the block start a match reads; wide mode only).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace b200lz4 {

namespace dec {

// Debug build (make bounds -> streamly_lz4_b200/libb200lz4_bounds.so, exercised by tests/test_gpu_modes.py): every global
// store range of the decoder is checked against the destination capacity of its block; a violation records the source
// line in the scratch block and traps.  compute-sanitizer is not available on the GPU pool, so this is the memory-safety
// evidence for malformed input.  Compiled out of the product.
#ifdef B200LZ4_BOUNDS_CHECK
#define BCHK(a, cond) do { if (!(cond)) { atomicExch(&(a).scratch->pad_[59], (uint32_t)__LINE__); __trap(); } } while (0)
#else
#define BCHK(a, cond) do { } while (0)
#endif

constexpr int kInRing = 4096;            // bytes of compressed payload resident in shared memory
constexpr int kFill = 512;               // ring fill unit (32 lanes x 16 bytes)
constexpr int kOutRing = 8192;           // bytes of recent output resident in shared memory
constexpr int kQDepth = 32;              // descriptors per queue buffer
constexpr uint32_t kShortLit = 32;       // sequences within these limits take the lane-parallel path
constexpr uint32_t kShortMatch = 64;
constexpr int kWindowSeqs = 11;          // most sequences one 32-byte parse window can hold (3 bytes each)
// A batch is at most kQDepth short sequences: <= 32 * (1 + 32 + 2 + 1) = 1152 compressed bytes (plus skipped
// length bytes, which nobody reads again) and <= 32 * (32 + 64) = 3072 output bytes.

constexpr int kCountMask = 0xFFFF;
constexpr int kBulk = 1 << 16;           // the batch is one sequence to be copied cooperatively
constexpr int kBegin = 1 << 17;          // first batch of a block
constexpr int kStreamBegin = 1 << 18;    // ... of the first block of a stream
constexpr int kStreamEnd = 1 << 19;      // with kEndBlock: last block of the stream
constexpr int kEndBlock = 1 << 30;       // block finished; result[] holds what to report
constexpr int kTerminate = 1 << 29;
constexpr int kFailed = 1 << 28;          // wide mode, with kEndBlock: the parser rejected the block

__device__ __forceinline__ int read_le32(const uint8_t* p)
{ return (int)((uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16) | ((uint32_t)__ldg(p + 3) << 24)); }

// coherent (not read-only-path) cooperative copy, non-overlapping, arbitrary alignment
__device__ __forceinline__ void warp_copy_rw(uint8_t* dst, const uint8_t* src, uint32_t len)
{
    const uint32_t lane = lane_id();
    if (len < 96) {
        for (uint32_t i = lane; i < len; i += 32) dst[i] = src[i];
        return;
    }
    uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
    if (lane < head) dst[lane] = src[lane];
    dst += head; src += head; len -= head;
    const uint32_t nvec = len >> 4;
    uintptr_t sa = reinterpret_cast<uintptr_t>(src);
    const uint32_t sh = (uint32_t)(sa & 3) * 8;
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t(3));
    uint4* dv = reinterpret_cast<uint4*>(dst);
    if ((sa & 15) == 0) {
        const uint4* sv = reinterpret_cast<const uint4*>(src);
        for (uint32_t v = lane; v < nvec; v += 32) dv[v] = sv[v];
    } else {
        for (uint32_t v = lane; v < nvec; v += 32) {
            const uint32_t* qd = sw + 4 * v;
            uint32_t x0 = qd[0], x1 = qd[1], x2 = qd[2], x3 = qd[3], x4 = sh ? qd[4] : 0u;
            dv[v] = make_uint4(__funnelshift_r(x0, x1, sh), __funnelshift_r(x1, x2, sh),
                               __funnelshift_r(x2, x3, sh), __funnelshift_r(x3, x4, sh));
        }
    }
    const uint32_t done = nvec << 4, tail = len - done;
    if (lane < tail) dst[done + lane] = src[done + lane];
}

// Overlapping match (offset < length <= 64): byte i comes from source byte i mod offset.  i mod offset through a 16-bit
// fixed-point reciprocal, exact for i < 64 (inv = 65536/offset plus at most 3); inv = 0 makes it the identity for
// ordinary matches.
__device__ __forceinline__ uint32_t overlap_inv(uint32_t dist, uint32_t mlen)
{ return (dist < mlen) ? (uint32_t)(65536.0f * __frcp_rn((float)dist)) + 2u : 0u; }

// Matches that read recent output, in order, each copied by all lanes within the output ring at out_s (kMask: ring size
// - 1).  par_s + 16 * i holds {destination, length <= 64, offset, overlap_inv} of match i, for every bit i of dep != 0;
// lane is the caller's lane_id().
template <uint32_t kMask>
__device__ __forceinline__ void copy_near_matches(uint32_t out_s, uint32_t par_s, uint32_t dep, const uint32_t lane)
{
    const uint32_t i1 = lane + 32;
    uint4 nx = lds128(par_s + 16u * (uint32_t)(__ffs(dep) - 1));
    for (;;) {
        dep &= dep - 1;
        const uint4 cu = nx;
        if (dep) nx = lds128(par_s + 16u * (uint32_t)(__ffs(dep) - 1));      // next match's parameters, early
        const uint32_t csa = cu.x - cu.z;
        const uint32_t k0 = lane - ((lane * cu.w) >> 16) * cu.z, k1 = i1 - ((i1 * cu.w) >> 16) * cu.z;
        if (lane < cu.y) sts8(out_s + ((cu.x + lane) & kMask), lds8(out_s + ((csa + k0) & kMask)));
        if (i1 < cu.y) sts8(out_s + ((cu.x + i1) & kMask), lds8(out_s + ((csa + k1) & kMask)));
        __syncwarp();
        if (!dep) break;
    }
}

// Header fields and the checks of decompressChunk (src/Streamly/Internal/LZ4.hs:303-318): both warps
// derive the same block geometry from the descriptor arrays.
struct BlockGeom { const uint8_t* payload; int comp_len; int cap; uint8_t* out; bool ok; };
__device__ __forceinline__ BlockGeom block_geom(const DecompressArgs& a, int b)
{
    BlockGeom g;
    const uint8_t* arr = a.src + a.src_off[b];
    const int avail = a.src_len[b] - a.header;
    g.payload = arr + a.header; g.out = a.dst + a.dst_off[b];
    g.comp_len = 0; g.cap = 0; g.ok = false;
    if (avail >= 0) {
        g.comp_len = a.header >= 4 ? read_le32(arr) : avail;                  // LZ4.hs:303
        g.cap = a.header == 8 ? read_le32(arr + 4) : a.max_block;             // LZ4.hs:189-198
        g.ok = g.comp_len > 0 && g.comp_len == avail && g.cap >= 0;           // LZ4.hs:309-318 (array length bounds the read)
        if (a.dst_cap && g.cap > a.dst_cap[b]) g.ok = false;
    }
    return g;
}

// Parse one block; pushes descriptors; returns the value to report (bytes produced, or < 0).
// Positions ip* are in ring space (payload index + skew).
//
// Two paths.  WINDOW: lane l decodes the 32 bytes from ip on as if a token started at ip + l (token, offset,
// one optional length byte), then the true token chain is followed through the window with one shuffle
// per sequence; the lanes on the chain write their descriptors side by side.  Only sequences without a
// literal-length extension, with at most one match-length byte and a short match qualify, and only away
// from the end of the block, where none of the end-of-block rules can fire.  SERIAL: everything else,
// one sequence at a time with the complete rule set of the safe decoder.
template <class PT>
__device__ int parse_block(PT& P, int skew, int src_len, int cap, uint32_t dict_len)
{
    const uint32_t lane = lane_id();
    constexpr uint32_t kRM = PT::kRing - 1;
    const bool check_offset = !PT::kWide && dict_len < 65536u;         // cbits/lz4.c:1764 (wide mode: deferred, see P.need)
    const int iend = skew + src_len;                                   // ring-space end of the payload
    const uint32_t ring_s = P.ring_s;
    int ip = skew, op = 0;
    P.end = iend;
    P.issued_end = P.ready_end = skew & ~(kFill - 1);
    P.cur_start = ip;
    if (cap == 0) {                                                    // :1781-1785
        if (src_len != 1) return -1;
        P.ensure(ip, ip + 1);
        return P.at(ip) == 0 ? 0 : -1;
    }
    if (src_len == 0) return -1;                                       // :1787
    for (;;) {
        if (P.fill + kWindowSeqs > kQDepth) P.publish(0, 0, ip);
        if (P.issued_end - ip < 1024) P.top_up(ip);
        if (ip + 72 > P.ready_end) P.ensure(ip, ip + 72);
        if (ip + 80 <= iend && op + 1024 <= cap) {
            // ---- window path
            const int p = ip + (int)lane;
            const uint32_t tok = lds8(ring_s + ((uint32_t)p & kRM));
            const uint32_t e1 = lds8(ring_s + (((uint32_t)p + 1u) & kRM));   // the byte after the token (issued with it): a literal-length byte if the nibble is 15
            const uint32_t ml = tok & 15u;
            const bool lext = (tok >> 4) == 15u;                       // one literal-length byte, e1 <= 17: 15 .. 32 literals (:1977-1983)
            const uint32_t lit = lext ? 15u + e1 : (tok >> 4);
            const uint32_t lsrc = (uint32_t)p + 1u + (lext ? 1u : 0u);  // first literal
            const uint32_t o = lsrc + (lit <= kShortLit ? lit : 0u);   // offset field
            const uint32_t b0 = lds8(ring_s + (o & kRM));
            const uint32_t b1 = lds8(ring_s + ((o + 1) & kRM));
            const uint32_t b2 = lds8(ring_s + ((o + 2) & kRM));
            const uint32_t dist = b0 | (b1 << 8);                      // :2055
            const bool ext = ml == 15u;
            const uint32_t mlen = ext ? 19u + b2 : ml + 4u;            // one length byte b2 != 255, :2062-2067
            const uint32_t nxt = (o - (uint32_t)ip) + 2u + (ext ? 1u : 0u);    // next token, relative to ip
            const bool simple = lit <= kShortLit && !(ext && b2 == 255u) && mlen <= kShortMatch;
            const uint32_t packed = nxt | ((lit + mlen) << 8) | (simple ? 0u : 0x80000000u);
            uint32_t cur = 0, real = 0;
            int opr = op, my_op = 0;
            for (;;) {
                const uint32_t info = __shfl_sync(kFull, packed, cur);
                if ((int)info < 0) break;
                if (lane == cur) my_op = opr;
                real |= 1u << cur;
                opr += (int)((info >> 8) & 0xFFFFu);
                cur = info & 0xFFu;
                if (cur >= 32u) break;
            }
            if (real) {
                const bool mine = (real >> lane) & 1u;
                // rules that can fire here: offset beyond the dictionary start (:2073), zero offset
                const bool bad = mine && (dist == 0u || (check_offset && (uint32_t)my_op + lit + dict_len < dist));
                if (__ballot_sync(kFull, bad)) return -1;
                if (PT::kWide && op < 65536) {       // the dictionary length is not known yet: remember how far back the block reaches
                    const int reach = mine ? (int)dist - (int)((uint32_t)my_op + lit) : 0;
                    P.note_reach(__reduce_max_sync(kFull, reach));
                }
                const uint32_t rank = __popc(real & lanemask_lt());
                if (mine) P.put(rank, lsrc, lit | (mlen << 8) | (dist << 16), (uint32_t)my_op, 0u);
                P.advance(__popc(real), opr);
                op = opr; ip += (int)cur;
                continue;
            }
        }
        // ---- serial path: one sequence
        const uint32_t token = P.at(ip); ip++;
        uint32_t len = token >> 4;
        if (len == 15) {                                               // :1977-1983 with reader :1707-1729
            const int lim = iend - 15;
            if (ip >= lim) return -1;                                  // initial_error
            for (;;) {
                P.ensure(ip, ip + 32);
                const int p = ip + (int)lane;
                const uint32_t s = (p < lim) ? P.at(p) : 0u;
                const bool stop = (p >= lim - 1) || (s != 255u);       // reading position lim-1 ends the run (loop_error keeps the sum)
                const uint32_t sb = __ballot_sync(kFull, stop);
                if (sb) {
                    const int t = __ffs(sb) - 1;
                    len += 255u * (uint32_t)t + __shfl_sync(kFull, s, t);
                    ip += t + 1;
                    break;
                }
                len += 255u * 32u; ip += 32;
            }
            if (len > 0x7FFFFFFFu) return -1;                          // cannot be a valid run; keeps the int arithmetic below exact
        }
        // end rule, :1991-2047
        const bool last = ((long long)op + len > (long long)cap - kMfLimit) || ((long long)ip + len > (long long)iend - (2 + 1 + kLastLiterals));
        if (last && ((long long)ip + len != (long long)iend || (long long)op + len > (long long)cap)) return -1;
        const bool bulk_lit = len > kShortLit;
        if (last) {
            if (len) {
                if (bulk_lit) { if (P.fill) P.publish(0, 0, ip); P.push_bulk((uint32_t)ip, len, 0u, 0u, op, ip + (int)len); }
                else { P.ensure(ip, ip + (int)len); P.push((uint32_t)ip, len, (uint32_t)op, 0u, op + (int)len); }
            }
            return op + (int)len;
        }
        const int lit_src = ip;
        ip += (int)len;
        P.ensure(ip, ip + 34);
        const uint32_t dist = P.at(ip) | (P.at(ip + 1) << 8); ip += 2;  // :2055
        uint32_t mlen = token & 15;
        if (mlen == 15) {                                              // :2062-2067
            const int lim = iend - kLastLiterals + 1;
            for (;;) {
                P.ensure(ip, ip + 32);
                const int p = ip + (int)lane;
                const uint32_t s = (p < iend) ? P.at(p) : 0u;
                const bool stop = (p >= iend) || (s != 255u);
                const uint32_t sb = __ballot_sync(kFull, stop);
                if (sb) {
                    const int t = __ffs(sb) - 1;
                    if (ip + t + 1 >= lim) return -1;                  // loop_error
                    mlen += 255u * (uint32_t)t + __shfl_sync(kFull, s, t);
                    ip += t + 1;
                    break;
                }
                if (ip + 32 >= lim) return -1;
                mlen += 255u * 32u; ip += 32;
            }
        }
        mlen += kMinMatch;
        const int op_seq = op;
        op += (int)len;
        const int from = op - (int)dist;
        if (check_offset && (long long)from + (long long)dict_len < 0) return -1;        // :2073
        if (PT::kWide && from < 0) P.note_reach(-from);
        if ((long long)op + mlen > (long long)cap - kLastLiterals) return -1;             // :2076-2078, :2139
        if (dist == 0) return -1;          // format violation (the reference copies garbage here, :2122-2130)
        if (bulk_lit || mlen > kShortMatch) {
            if (P.fill) P.publish(0, 0, lit_src);
            P.push_bulk((uint32_t)lit_src, len, mlen, dist, op_seq, ip);
        } else {
            P.push((uint32_t)lit_src, len | (mlen << 8) | (dist << 16), (uint32_t)op_seq, 0u, op + (int)mlen);
        }
        op += (int)mlen;
    }
}


}  // namespace dec

}  // namespace b200lz4
