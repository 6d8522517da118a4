// host_plan.h -- what the host batch calls of api.cu decide before they touch the device: argument checks, slot
// capacities, how a batch is cut into chunks (one ctx), stripes (several devices) and groups (streamed calls), which
// pipeline a call takes, the streamed geometry and piece order, and the layout of the descriptor block.  Pure functions
// of the call's arguments (no CUDA, no environment), so that tests/test_host_plan.py can pin them without a GPU: a
// mistake here changes the speed of a call, not its bytes.
#pragma once
#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <string>
#include <vector>

#include "b200lz4.h"

namespace hostplan {
namespace {     // internal linkage: nothing of this header shows up among libb200lz4.so's exported symbols

constexpr int kMaxInputSize = 0x7E000000;   // LZ4_MAX_INPUT_SIZE (common.cuh: kMaxInput, checked in api.cu)
constexpr int kMaxChunks = 6;       // pipeline depth of the plain host calls (H2D + D2H + chunk streams must fit the
                                    // 8 hardware queues of the default CUDA_DEVICE_MAX_CONNECTIONS, else chunks serialize)
constexpr int kMaxGroups = 16;      // streamed calls: block groups (events, work counters, arrival flags)
constexpr int kMaxSegs = 16;        // ... and segments a block is cut into on its way to / from the device

inline int bound_of(int n) { return ((unsigned)n > (unsigned)kMaxInputSize) ? 0 : n + n / 255 + 16; }
inline int64_t align16(int64_t v) { return (v + 15) & ~int64_t(15); }
inline int32_t le32(const uint8_t* p)
{ return (int32_t)((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24)); }

// ---- argument checks ---------------------------------------------------------------------------------------------------
struct Verdict { int code; std::string msg; };      // code 0: the call may go on (and has nothing to do if n == 0)

inline Verdict check_blocks(const int64_t* off, const int32_t* len, int n, int64_t bytes)
{
    for (int i = 0; i < n; i++) {
        if (len[i] < 0 || off[i] < 0 || off[i] + (int64_t)len[i] > bytes)
            return {B200LZ4_E_ARG, "block " + std::to_string(i) + " lies outside the source buffer"};
    }
    return {0, ""};
}

enum class Entry { Ctx, Multi, Dev };   // b200lz4_{de,}compress_batch, ..._batch_multi, ..._dev

// Every check a batch entry point makes, in the order it makes them.  owner: the ctx, the mctx (NULL when it has no
// devices) or d_scratch.  The device entry points cannot read their (device) arrays and take max_block as given.
inline Verdict check_batch(Entry who, bool decode, const void* owner, int n, int header, int max_block,
                           const void* src, int64_t src_bytes, const int64_t* src_off, const int32_t* src_len,
                           const void* dst, const int64_t* dst_off, const int32_t* out_len,
                           const int32_t* stream_first, int n_streams, bool streams_given)
{
    const Verdict ok{0, ""};
    const bool arrays = src_off && src_len && dst_off && out_len;
    if (who == Entry::Dev && (n < 0 || !owner)) return {B200LZ4_E_ARG, "bad argument"};
    if (who == Entry::Ctx && !owner) return {B200LZ4_E_ARG, "ctx is NULL"};
    if (who == Entry::Ctx && (n < 0 || (n > 0 && !arrays))) return {B200LZ4_E_ARG, "NULL descriptor array"};
    if (who == Entry::Multi && !owner) return {B200LZ4_E_ARG, "mctx is NULL"};
    if (who == Entry::Multi && (n < 0 || (n > 0 && !(arrays && src && dst)))) return {B200LZ4_E_ARG, "NULL argument"};
    if (header != 0 && header != 4 && header != 8) return {B200LZ4_E_ARG, "header_mode must be 0, 4 or 8"};
    if (who == Entry::Dev) return ok;
    if (decode && header != 8 && max_block < 0) return {B200LZ4_E_ARG, "max_block"};
    if (streams_given && !stream_first) return {B200LZ4_E_ARG, "streams given without stream_first"};
    if (n == 0) return ok;
    if (!src || !dst) return {B200LZ4_E_ARG, "NULL data buffer"};
    Verdict v = check_blocks(src_off, src_len, n, src_bytes);
    if (v.code || !stream_first) return v;
    if (n_streams < 0 || n_streams == 0) return {B200LZ4_E_ARG, "n_streams"};     // (n > 0 here)
    if (stream_first[0] != 0 || stream_first[n_streams] != n) return {B200LZ4_E_ARG, "stream_first must start at 0 and end at n_blocks"};
    for (int s = 0; s < n_streams; s++)
        if (stream_first[s] > stream_first[s + 1]) return {B200LZ4_E_ARG, "stream_first must be non-decreasing"};
    return ok;
}

// ---- capacities ----------------------------------------------------------------------------------------------------------
// compress: a block's output (header included) needs at most header + bound_of(len) bytes; its device slot has 16 bytes more
inline int64_t compress_cap(int32_t len, int header) { return (int64_t)header + bound_of(len); }
inline int64_t compress_slot(int64_t cap_with_header) { return align16(cap_with_header + 16); }
// decompress: the header's uncompLen (BlockHasSize) or the configured maximum (LZ4.hs:189-198), and the bytes the block
// takes in the device slots and in the (multi-device) output: exact with sizes in the headers, else rounded up to 16
inline int decode_cap(const uint8_t* src, const int64_t* off, const int32_t* len, int i, int header, int max_block)
{
    int cap = max_block;
    if (header == 8) cap = len[i] >= 8 ? le32(src + off[i] + 4) : 0;
    return cap < 0 ? 0 : cap;
}
inline int64_t decode_slot(int cap, int header) { return header == 8 ? (int64_t)cap : align16((int64_t)cap); }

// ---- ranges ----------------------------------------------------------------------------------------------------------------
// Blocks [b0, b1) = units [u0, u1): a unit is a whole stream when stream_first is given, else one block.
struct Range { int u0, u1, b0, b1; };

// Contiguous ranges of units: range k takes units while the bytes taken so far are below target(k) (INT64_MAX: all that
// are left); the last of max_parts ranges takes the rest.  all_parts: always max_parts ranges, the trailing ones possibly
// empty; else ranges end with the units.  A range whose predecessor overshot its share is empty and still counts.
template <class Target>
int cut_ranges(const int32_t* len, int n, const int32_t* first, int ns, int max_parts, bool all_parts, Target target, Range* out)
{
    const int units = first ? ns : n;
    auto block = [&](int u) { return first ? first[u] : u; };
    int k = 0, u = 0;
    int64_t done = 0;
    for (; k < max_parts && (all_parts || u < units); k++) {
        Range r{u, u, block(u), block(u)};
        const int64_t t = k == max_parts - 1 ? INT64_MAX : target(k);
        for (; u < units && done < t; u++) for (int i = block(u); i < block(u + 1); i++) done += len[i];
        r.u1 = u; r.b1 = block(u);
        out[k] = r;
    }
    return k;
}

inline int64_t total_bytes(const int32_t* len, int n)
{
    int64_t t = 0;
    for (int i = 0; i < n; i++) t += len[i];
    return t;
}

// Plain pipeline: up to kMaxChunks chunks.  Chunk k becomes ready when its H2D copy lands and finishes one block latency
// later, so the end of the call is "last byte arrives + block latency + D2H of the last chunk": keep the last chunk small.
// early_start (mirrored decompress: the output leaves from inside the kernels, so the call ends one PCIe-bound stretch
// after the FIRST chunk has landed): a small first chunk instead of a small last one.  Below 48 MiB: one chunk.
inline int plan_chunks(const int32_t* len, int n, const int32_t* first, int ns, bool early_start, Range* out)
{
    static const double kShareTail[kMaxChunks] = {0.14, 0.20, 0.20, 0.20, 0.18, 0.08};
    static const double kShareHead[kMaxChunks] = {0.03, 0.09, 0.18, 0.24, 0.24, 0.22};
    const double* kShare = early_start ? kShareHead : kShareTail;
    const int64_t total = total_bytes(len, n);
    const bool small = total < (int64_t(48) << 20);
    return cut_ranges(len, n, first, ns, kMaxChunks, false, [&](int k) {
        double upto = 0;
        for (int q = 0; q <= k; q++) upto += kShare[q];
        return small ? INT64_MAX : (int64_t)(upto * (double)total);
    }, out);
}

// Several devices: exactly `parts` stripes with about equal source bytes
inline std::vector<Range> plan_stripes(const int32_t* len, int n, const int32_t* first, int ns, int parts)
{
    const int64_t total = total_bytes(len, n);
    std::vector<Range> out(parts);
    cut_ranges(len, n, first, ns, parts, true, [&](int k) { return total * (k + 1) / parts; }, out.data());
    return out;
}

// the bytes of the source buffer blocks b0..b1 span ({0, 0} for none)
struct Span { int64_t lo, hi; };
inline Span byte_span(const int64_t* off, const int32_t* len, int b0, int b1)
{
    Span s{INT64_MAX, 0};
    for (int i = b0; i < b1; i++) { s.lo = std::min(s.lo, off[i]); s.hi = std::max(s.hi, off[i] + (int64_t)len[i]); }
    if (s.lo > s.hi) s.lo = s.hi = 0;
    return s;
}

// ---- which pipeline --------------------------------------------------------------------------------------------------------
// Streamed compress: at least 96 equally long independent blocks of >= 64 KiB, >= 96 MiB in all, at a constant pitch (the
// last block may be shorter).  L: the block length, P: the pitch.
struct StreamShape { int L; int64_t P; bool ok; };
inline StreamShape streamed_shape(const int64_t* off, const int32_t* len, int n, bool linked, bool block_cap, bool disabled)
{
    const StreamShape no{0, 0, false};
    if (disabled || linked || block_cap || n < 96) return no;
    const int L = len[0];
    if (L < 65536 || (int64_t)L * n < (int64_t(96) << 20)) return no;
    const int64_t P = off[1] - off[0];
    if (P < L) return no;
    for (int i = 0; i < n; i++) {
        if (off[i] != off[0] + P * i) return no;
        if (i < n - 1 ? len[i] != L : (len[i] <= 0 || len[i] > L)) return no;
    }
    return {L, P, true};
}

// How decompressed output goes home (B200LZ4_DECODE_OUT, first letter `out`): Copy = D2H copies behind each chunk's
// kernel; Pieces = segment by segment while the blocks are being decoded (the streamed call: at least 96 independent
// blocks whose headers (mode 8) give them all the same capacity L >= 64 KiB, >= 96 MiB in all, the last one may be
// smaller; the default where it applies); Mirror = independent blocks with their sizes in the headers and a destination
// in mapped page-locked memory (dst_mapped): the kernels store every output byte to the host buffer as well (opt-in).
// wide_forced: B200LZ4_DWIDE=1, whose kernel has no mirror.
enum class DecodeOut { Copy, Pieces, Mirror };
struct DecodeRoute { DecodeOut out; int L, cap_last; };
inline DecodeRoute decode_route(const uint8_t* src, const int64_t* off, const int32_t* len, int n, int header, bool linked,
                                char out, bool disabled, bool wide_forced, bool dst_mapped)
{
    if (out == 'm' && header == 8 && !linked && !wide_forced && dst_mapped) return {DecodeOut::Mirror, 0, 0};
    const DecodeRoute copy{DecodeOut::Copy, 0, 0};
    if (disabled || out == 'c' || header != 8 || linked || n < 96 || len[0] < 8) return copy;
    const int L = le32(src + off[0] + 4);
    if (L < 65536 || (int64_t)L * n < (int64_t(96) << 20)) return copy;
    for (int i = 0; i < n - 1; i++) if (decode_cap(src, off, len, i, 8, 0) != L) return copy;
    const int cap_last = decode_cap(src, off, len, n - 1, 8, 0);
    if (cap_last <= 0 || cap_last > L) return copy;
    return {DecodeOut::Pieces, L, cap_last};
}

// ---- streamed geometry -----------------------------------------------------------------------------------------------------
// G groups of per_group consecutive blocks (one kernel launch each), blocks cut into S segments of seg bytes (a multiple of
// 128), pieces (g, s) sent in order of g + s * w.  rho: one block's finder time over the whole H2D time (compress).
struct Geometry { int G, S, seg, per_group; double w, rho; };

// the clamps and the recount shared by both directions: G and S as asked (overrides included), then what they come to
inline Geometry clamp_geometry(int n, int L, int G, int S)
{
    G = std::min(std::max(G, 1), kMaxGroups);
    S = std::min(std::max(S, 1), kMaxSegs);
    const int seg = (int)((((int64_t)L + S - 1) / S + 127) / 128 * 128);
    S = (L + seg - 1) / seg;
    const int per_group = (n + G - 1) / G;
    G = (n + per_group - 1) / per_group;
    return {G, S, seg, per_group, (double)G, 0};
}

constexpr double kStreamSpread = 1.5;   // measured: a little later is better than a little early (the D2H copies of finished groups
                                        // share the link, and a starved finder only waits while an early piece delays everyone else's)

// Compress: from what the previous streamed call on the ctx measured (0: nothing yet) and the kernel streams that cannot
// block the copy stream (nks).  env_*: the B200LZ4_STREAM_G / _S / _W overrides (NULL: none).
inline Geometry compress_geometry(int n, int L, int64_t total, int nks, double est_ns_per_byte, double est_h2d_gbs,
                                  const char* env_g, const char* env_s, const char* env_w)
{
    const double ns_per_byte = est_ns_per_byte > 0 ? est_ns_per_byte : 12.0;       // first call: ~85 MB/s per finder
    const double h2d_gbs = est_h2d_gbs > 0 ? est_h2d_gbs : 50.0;
    const double t_block_ms = ns_per_byte * 1.1 * L * 1e-6, t_h2d_ms = (double)total / (h2d_gbs * 1e6);
    const double rho = t_block_ms / t_h2d_ms;
    // a group runs behind group g - nks on its stream.  Segments of ~160 000 bytes (rows of a pitched copy: smaller ones
    // cost copy-engine efficiency while the D2H direction is busy, larger ones lengthen the tail, which is one segment's
    // worth of finder time): 4 for 640 000-byte blocks, 16 from 2.5 MB
    Geometry g = clamp_geometry(n, L, env_g ? atoi(env_g) : (rho <= 0.45 ? 2 * nks : nks),
                                env_s ? atoi(env_s) : (int)std::min<int64_t>(kMaxSegs, std::max<int64_t>(4, ((int64_t)L + 80000) / 160000)));
    g.rho = rho;
    // a group's S pieces are (S - 1) * w key units apart, the whole schedule spans (G - 1) + (S - 1) * w units in t_h2d:
    // the last piece of a group should land when its finders get there, (S - 1) / S of a block time after the first
    if (g.S - rho * (g.S - 1) > 0.01) g.w = kStreamSpread * rho * (g.G - 1) / (g.S - rho * (g.S - 1));
    if (env_w) g.w = atof(env_w);
    if (g.w > g.G) g.w = g.G;
    return g;
}

inline Geometry decompress_geometry(int n, int L, const char* env_g, const char* env_s)
{
    return clamp_geometry(n, L, env_g ? atoi(env_g) : 12, env_s ? atoi(env_s) : 8);
}

inline int plan_groups(const Geometry& geo, int n, Range* out)
{
    for (int g = 0; g < geo.G; g++) {
        const int b0 = g * geo.per_group, b1 = std::min(n, b0 + geo.per_group);
        out[g] = Range{b0, b1, b0, b1};
    }
    return geo.G;
}

// every (group, segment) piece once, in deadline order key(g, s) = g + s * w: w = 0 is the plain block order, a large w
// sends segment 0 of every block first
struct Piece { int g, s; };
inline std::vector<Piece> piece_order(const Geometry& geo)
{
    struct Keyed { int g, s; double key; };
    std::vector<Keyed> k;
    k.reserve((size_t)geo.G * geo.S);
    for (int g = 0; g < geo.G; g++) for (int s = 0; s < geo.S; s++) k.push_back({g, s, g + s * geo.w});
    std::stable_sort(k.begin(), k.end(), [](const Keyed& x, const Keyed& y) { return x.key < y.key; });
    std::vector<Piece> out;
    out.reserve(k.size());
    for (const Keyed& x : k) out.push_back({x.g, x.s});
    return out;
}

// ---- descriptor block --------------------------------------------------------------------------------------------------------
// Typed arrays at 16-byte aligned offsets of one host (pinned) and one device block of the same layout; the arrays before
// `upload` go to the device in one copy.  An array of 0 entries takes no room.
struct DescLayout {
    size_t src_off, slot_off, src_len, cap, first, states, upload, out_len, out_off, ready, bytes;

    DescLayout(int n, int n_slot, int n_cap, int n_first, int n_states, int n_out_off, int n_ready)
    {
        size_t at = 0;
        auto take = [&](size_t b) { const size_t o = at; at = (at + b + 15) & ~size_t(15); return o; };
        src_off = take(sizeof(int64_t) * n);
        slot_off = take(sizeof(int64_t) * n_slot);
        src_len = take(sizeof(int32_t) * n);
        cap = take(sizeof(int32_t) * n_cap);
        first = take(sizeof(int32_t) * n_first);
        states = take(sizeof(void*) * n_states);
        upload = at;
        out_len = take(sizeof(int32_t) * n);
        out_off = take(sizeof(int64_t) * n_out_off);
        ready = take(sizeof(uint32_t) * n_ready);
        bytes = at;
    }
    template <class T> static T* at(void* base, size_t o) { return reinterpret_cast<T*>(static_cast<uint8_t*>(base) + o); }
    int64_t* src_off_in(void* b) const { return at<int64_t>(b, src_off); }
    int64_t* slot_off_in(void* b) const { return at<int64_t>(b, slot_off); }
    int32_t* src_len_in(void* b) const { return at<int32_t>(b, src_len); }
    int32_t* cap_in(void* b) const { return at<int32_t>(b, cap); }
    int32_t* first_in(void* b) const { return at<int32_t>(b, first); }
    void** states_in(void* b) const { return at<void*>(b, states); }
    int32_t* out_len_in(void* b) const { return at<int32_t>(b, out_len); }
    int64_t* out_off_in(void* b) const { return at<int64_t>(b, out_off); }
    uint32_t* ready_in(void* b) const { return at<uint32_t>(b, ready); }
};

}  // namespace
}  // namespace hostplan
