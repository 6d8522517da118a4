"""The host batch calls' planning (csrc/host_plan.h) without a GPU: which pipeline a call takes, how a batch is cut into
chunks, stripes and groups, the streamed geometry and piece order, the descriptor layout and the argument checks.  A
mistake here changes the speed of a call, not its bytes, so the GPU parity tests cannot see it.  A small C++ driver is
compiled against the header with g++; the pinned plans were produced by the same driver run against the planning code
as it stood inside csrc/api.cu before it moved to the header.  The GPU part runs the error path of every host pipeline
through the ABI (dst_cap too small) and checks that the ctx is still good afterwards."""
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MiB = 1 << 20

DRIVER = r"""
// one command per input line, one answer per output line
#include <cstdio>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>
#include "host_plan.h"
using namespace hostplan;

template <class T> std::vector<T> take(std::istream& in, int n) { std::vector<T> v(n > 0 ? n : 0); for (auto& x : v) in >> x; return v; }
static const char* opt(const std::string& s) { return s == "-" ? nullptr : s.c_str(); }
static void ranges(const Range* r, int k) { for (int i = 0; i < k; i++) printf("%s%d %d %d %d", i ? " | " : "", r[i].u0, r[i].u1, r[i].b0, r[i].b1); printf("\n"); }

int main()
{
    std::string line;
    while (std::getline(std::cin, line)) {
        std::istringstream in(line);
        std::string cmd;
        in >> cmd;
        if (cmd == "chunks" || cmd == "stripes") {          // chunks EARLY | stripes PARTS, then n ns len[n] first[ns+1] (ns -1: no streams)
            int arg, n, ns;
            in >> arg >> n >> ns;
            auto len = take<int32_t>(in, n);
            auto first = take<int32_t>(in, ns + 1);
            const int32_t* f = ns >= 0 ? first.data() : nullptr;
            if (cmd == "chunks") { Range r[kMaxChunks]; ranges(r, plan_chunks(len.data(), n, f, ns, arg != 0, r)); }
            else { auto r = plan_stripes(len.data(), n, f, ns, arg); ranges(r.data(), (int)r.size()); }
        } else if (cmd == "shape") {                        // n linked block_cap disabled off[n] len[n]
            int n, linked, cap, dis;
            in >> n >> linked >> cap >> dis;
            auto off = take<int64_t>(in, n);
            auto len = take<int32_t>(in, n);
            const StreamShape s = streamed_shape(off.data(), len.data(), n, linked, cap, dis);
            printf("%d %d %lld\n", (int)s.ok, s.L, (long long)s.P);
        } else if (cmd == "cgeo" || cmd == "dgeo") {        // cgeo n L total nks est_ns est_gbs G S W | dgeo n L G S  (-: no override)
            int n, L, nks = 0; long long total = 0; double est_ns = 0, est_gbs = 0; std::string g, s, w = "-";
            in >> n >> L;
            if (cmd == "cgeo") in >> total >> nks >> est_ns >> est_gbs >> g >> s >> w; else in >> g >> s;
            const Geometry geo = cmd == "cgeo" ? compress_geometry(n, L, total, nks, est_ns, est_gbs, opt(g), opt(s), opt(w))
                                               : decompress_geometry(n, L, opt(g), opt(s));
            printf("G %d S %d seg %d per_group %d w %.17g rho %.17g |", geo.G, geo.S, geo.seg, geo.per_group, geo.w, geo.rho);
            for (const Piece& p : piece_order(geo)) printf(" %d.%d", p.g, p.s);
            printf("\n");
        } else if (cmd == "route") {                        // n header linked out disabled wide mapped len[n] cap[n]: block i at 8 i
            int n, header, linked, dis, wide, mapped; std::string out;
            in >> n >> header >> linked >> out >> dis >> wide >> mapped;
            auto len = take<int32_t>(in, n);
            auto cap = take<int32_t>(in, n);
            std::vector<uint8_t> src(8 * (size_t)n + 8);
            std::vector<int64_t> off(n);
            for (int i = 0; i < n; i++) { off[i] = 8 * (int64_t)i; for (int b = 0; b < 4; b++) src[8 * i + 4 + b] = (uint8_t)((uint32_t)cap[i] >> (8 * b)); }
            const DecodeRoute r = decode_route(src.data(), off.data(), len.data(), n, header, linked, out == "-" ? 0 : out[0], dis, wide, mapped);
            printf("%d %d %d\n", (int)r.out, r.L, r.cap_last);
#ifndef LEGACY
        } else if (cmd == "check") {    // who decode owner n header max_block src src_bytes dst arrays(4 bits) streams_given ns first[ns+1] off[n] len[n]
            int who, decode, owner, n, header, max_block, src, dst, mask, given, ns; long long bytes;
            in >> who >> decode >> owner >> n >> header >> max_block >> src >> bytes >> dst >> mask >> given >> ns;
            auto first = take<int32_t>(in, ns + 1);
            auto off = take<int64_t>(in, n);
            auto len = take<int32_t>(in, n);
            static int dummy;
            auto p = [&](bool on) -> const void* { return on ? &dummy : nullptr; };
            const Verdict v = check_batch((Entry)who, decode, p(owner), n, header, max_block, p(src), bytes,
                                          mask & 1 ? off.data() : nullptr, mask & 2 ? len.data() : nullptr, p(dst),
                                          mask & 4 ? reinterpret_cast<const int64_t*>(&dummy) : nullptr,
                                          mask & 8 ? reinterpret_cast<const int32_t*>(&dummy) : nullptr,
                                          ns >= 0 ? first.data() : nullptr, ns, given);
            printf("%d %s\n", v.code, v.msg.c_str());
        } else if (cmd == "layout") {                       // n n_slot n_cap n_first n_states n_out_off n_ready
            int a[7];
            for (int& x : a) in >> x;
            const DescLayout d(a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
            printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", d.src_off, d.slot_off, d.src_len, d.cap, d.first, d.states,
                   d.upload, d.out_len, d.out_off, d.ready, d.bytes);
#endif
        } else {
            printf("? %s\n", cmd.c_str());
        }
        fflush(stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    d = tmp_path_factory.mktemp("host_plan")
    (d / "driver.cpp").write_text(DRIVER)
    exe = d / "driver"
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(ROOT, "streamly_lz4_b200", "csrc"), str(d / "driver.cpp"), "-o", str(exe)], check=True)

    def run(*cmds):
        out = subprocess.run([str(exe)], input="\n".join(cmds) + "\n", capture_output=True, text=True, check=True).stdout
        lines = out.splitlines()
        assert len(lines) == len(cmds)
        return lines
    return run


def ints(v):
    return " ".join(str(int(x)) for x in v)


def chunks(lens, first=None, early=False):
    ns = -1 if first is None else len(first) - 1
    return f"chunks {int(early)} {len(lens)} {ns} {ints(lens)} {ints(first or [])}"


def stripes(parts, lens, first=None):
    ns = -1 if first is None else len(first) - 1
    return f"stripes {parts} {len(lens)} {ns} {ints(lens)} {ints(first or [])}"


def shape(offs, lens, linked=False, cap=False, disabled=False):
    return f"shape {len(lens)} {int(linked)} {int(cap)} {int(disabled)} {ints(offs)} {ints(lens)}"


def cgeo(n, L, total, nks, est_ns=0, est_gbs=0, g="-", s="-", w="-"):
    return f"cgeo {n} {L} {total} {nks} {est_ns} {est_gbs} {g} {s} {w}"


def dgeo(n, L, g="-", s="-"):
    return f"dgeo {n} {L} {g} {s}"


def route(lens, caps, header=8, linked=False, out="-", disabled=False, wide=False, mapped=False):
    return f"route {len(lens)} {header} {int(linked)} {out} {int(disabled)} {int(wide)} {int(mapped)} {ints(lens)} {ints(caps)}"


def equal(n, L, last=None):
    lens = [L] * n
    if last is not None:
        lens[-1] = last
    return lens


def pitched(n, pitch):
    return [i * pitch for i in range(n)]


def total(lens):
    return sum(lens)


# config 2 (1 678 x 640 000), the shapes of test_gpu_streamed.py, the odd-geometry overrides, a batch whose second and third
# chunks are empty, a batch below 48 MiB (one chunk), a linked batch with uneven streams, and 2 and 8 stripes
CFG2 = equal(1678, 640000)
EMPTY_MIDDLE = [60 * MiB] + [MiB] * 40
SMALL = [MiB] * 10 + [12345]
LINKED_FIRST = [0, 3, 4, 50, 51, 60, 90, 91]
LINKED = [MiB + 7 * i for i in range(91)]
CASES = {
    "cfg2-chunks": chunks(CFG2),
    "cfg2-chunks-mirror": chunks(CFG2, early=True),
    "cfg2-shape": shape(pitched(1678, 640000), CFG2),
    "cfg2-cgeo-2": cgeo(1678, 640000, total(CFG2), 2),
    "cfg2-cgeo-6": cgeo(1678, 640000, total(CFG2), 6),
    "cfg2-dgeo": dgeo(1678, 640000),
    "cfg2-route": route([300000] * 1678, CFG2),
    "s170-last5-shape": shape(pitched(170, 640016), equal(170, 640000, 5)),
    "s170-last123457-shape": shape(pitched(170, 640000), equal(170, 640000, 123457)),
    "s170-pitch650000-shape": shape(pitched(170, 650000), equal(170, 640000)),
    "s170-cgeo-2": cgeo(170, 640000, total(equal(170, 640000, 5)), 2),
    "s170-cgeo-6": cgeo(170, 640000, total(equal(170, 640000, 123457)), 6),
    "s170-dgeo": dgeo(170, 640000),
    "s170-route-last5": route([70000] * 170, equal(170, 640000, 5)),
    "s1100-shape": shape(pitched(1100, 100003), equal(1100, 100003, 77)),
    "s1100-cgeo-2": cgeo(1100, 100003, total(equal(1100, 100003, 77)), 2),
    "s1100-cgeo-6": cgeo(1100, 100003, total(equal(1100, 100003, 77)), 6),
    "s1100-dgeo": dgeo(1100, 100003),
    "s97-shape": shape(pitched(97, 4 * MiB), equal(97, 4 * MiB)),
    "s97-cgeo-2": cgeo(97, 4 * MiB, total(equal(97, 4 * MiB)), 2),
    "s97-cgeo-6": cgeo(97, 4 * MiB, total(equal(97, 4 * MiB)), 6),
    "s97-dgeo": dgeo(97, 4 * MiB),
    "odd-cgeo": cgeo(170, 640000, total(equal(170, 640000)), 6, g="5", s="13", w="0.7"),
    "odd-dgeo": dgeo(170, 640000, g="5", s="13"),
    "empty-middle-chunks": chunks(EMPTY_MIDDLE),
    "small-chunks": chunks(SMALL),
    "linked-chunks": chunks(LINKED, LINKED_FIRST),
    "cfg2-stripes-2": stripes(2, CFG2),
    "cfg2-stripes-8": stripes(8, CFG2),
    "linked-stripes-2": stripes(2, LINKED, LINKED_FIRST),
    "linked-stripes-8": stripes(8, LINKED, LINKED_FIRST),
}

PINNED = {
    'cfg2-chunks':
        '0 235 0 235 | 235 571 235 571 | 571 907 571 907 | 907 1242 907 1242 | 1242 1544 1242 1544 | 1544 1678 1544 1678',
    'cfg2-chunks-mirror':
        '0 51 0 51 | 51 202 51 202 | 202 504 202 504 | 504 907 504 907 | 907 1309 907 1309 | 1309 1678 1309 1678',
    'cfg2-shape':
        '1 640000 640000',
    'cfg2-cgeo-2':
        'G 4 S 4 seg 160000 per_group 420 w 0.62764158918005086 rho 0.39332538736591183 | 0.0 0.1 1.0 0.2 1.1 0.3 2.0 1.2 2.1 1.3 3.0 2.2 3.1 2.3 3.2 3.3',
    'cfg2-cgeo-6':
        'G 12 S 4 seg 160000 per_group 140 w 2.3013524936601866 rho 0.39332538736591183 | 0.0 1.0 2.0 0.1 3.0 1.1 4.0 2.1 0.2 5.0 3.1 1.2 6.0 4.1 2.2 0.3 7.0 5.1 3.2 1.3 8.0 6.1 4.2 2.3 9.0 7.1 5.2 3.3 10.0 8.1 6.2 4.3 11.0 9.1 7.2 5.3 10.1 8.2 6.3 11.1 9.2 7.3 10.2 8.3 11.2 9.3 10.3 11.3',
    'cfg2-dgeo':
        'G 12 S 8 seg 80000 per_group 140 w 12 rho 0 | 0.0 1.0 2.0 3.0 4.0 5.0 6.0 7.0 8.0 9.0 10.0 11.0 0.1 1.1 2.1 3.1 4.1 5.1 6.1 7.1 8.1 9.1 10.1 11.1 0.2 1.2 2.2 3.2 4.2 5.2 6.2 7.2 8.2 9.2 10.2 11.2 0.3 1.3 2.3 3.3 4.3 5.3 6.3 7.3 8.3 9.3 10.3 11.3 0.4 1.4 2.4 3.4 4.4 5.4 6.4 7.4 8.4 9.4 10.4 11.4 0.5 1.5 2.5 3.5 4.5 5.5 6.5 7.5 8.5 9.5 10.5 11.5 0.6 1.6 2.6 3.6 4.6 5.6 6.6 7.6 8.6 9.6 10.6 11.6 0.7 1.7 2.7 3.7 4.7 5.7 6.7 7.7 8.7 9.7 10.7 11.7',
    'cfg2-route':
        '1 640000 640000',
    's170-last5-shape':
        '1 640000 640016',
    's170-last123457-shape':
        '1 640000 640000',
    's170-pitch650000-shape':
        '1 640000 650000',
    's170-cgeo-2':
        'G 2 S 4 seg 160000 per_group 85 w 2 rho 3.9053252632523456 | 0.0 1.0 0.1 1.1 0.2 1.2 0.3 1.3',
    's170-cgeo-6':
        'G 6 S 4 seg 160000 per_group 29 w 6 rho 3.9008728729449418 | 0.0 1.0 2.0 3.0 4.0 5.0 0.1 1.1 2.1 3.1 4.1 5.1 0.2 1.2 2.2 3.2 4.2 5.2 0.3 1.3 2.3 3.3 4.3 5.3',
    's170-dgeo':
        'G 12 S 8 seg 80000 per_group 15 w 12 rho 0 | 0.0 1.0 2.0 3.0 4.0 5.0 6.0 7.0 8.0 9.0 10.0 11.0 0.1 1.1 2.1 3.1 4.1 5.1 6.1 7.1 8.1 9.1 10.1 11.1 0.2 1.2 2.2 3.2 4.2 5.2 6.2 7.2 8.2 9.2 10.2 11.2 0.3 1.3 2.3 3.3 4.3 5.3 6.3 7.3 8.3 9.3 10.3 11.3 0.4 1.4 2.4 3.4 4.4 5.4 6.4 7.4 8.4 9.4 10.4 11.4 0.5 1.5 2.5 3.5 4.5 5.5 6.5 7.5 8.5 9.5 10.5 11.5 0.6 1.6 2.6 3.6 4.6 5.6 6.6 7.6 8.6 9.6 10.6 11.6 0.7 1.7 2.7 3.7 4.7 5.7 6.7 7.7 8.7 9.7 10.7 11.7',
    's170-route-last5':
        '1 640000 5',
    's1100-shape':
        '1 100003 100003',
    's1100-cgeo-2':
        'G 2 S 4 seg 25088 per_group 550 w 0.40976768955023896 rho 0.60054553011266054 | 0.0 0.1 0.2 1.0 0.3 1.1 1.2 1.3',
    's1100-cgeo-6':
        'G 6 S 4 seg 25088 per_group 184 w 2.0488384477511947 rho 0.60054553011266054 | 0.0 1.0 2.0 0.1 3.0 1.1 4.0 2.1 0.2 5.0 3.1 1.2 4.1 2.2 0.3 5.1 3.2 1.3 4.2 2.3 5.2 3.3 4.3 5.3',
    's1100-dgeo':
        'G 12 S 8 seg 12544 per_group 92 w 12 rho 0 | 0.0 1.0 2.0 3.0 4.0 5.0 6.0 7.0 8.0 9.0 10.0 11.0 0.1 1.1 2.1 3.1 4.1 5.1 6.1 7.1 8.1 9.1 10.1 11.1 0.2 1.2 2.2 3.2 4.2 5.2 6.2 7.2 8.2 9.2 10.2 11.2 0.3 1.3 2.3 3.3 4.3 5.3 6.3 7.3 8.3 9.3 10.3 11.3 0.4 1.4 2.4 3.4 4.4 5.4 6.4 7.4 8.4 9.4 10.4 11.4 0.5 1.5 2.5 3.5 4.5 5.5 6.5 7.5 8.5 9.5 10.5 11.5 0.6 1.6 2.6 3.6 4.6 5.6 6.6 7.6 8.6 9.6 10.6 11.6 0.7 1.7 2.7 3.7 4.7 5.7 6.7 7.7 8.7 9.7 10.7 11.7',
    's97-shape':
        '1 4194304 4194304',
    's97-cgeo-2':
        'G 2 S 16 seg 262144 per_group 49 w 2 rho 6.804123711340206 | 0.0 1.0 0.1 1.1 0.2 1.2 0.3 1.3 0.4 1.4 0.5 1.5 0.6 1.6 0.7 1.7 0.8 1.8 0.9 1.9 0.10 1.10 0.11 1.11 0.12 1.12 0.13 1.13 0.14 1.14 0.15 1.15',
    's97-cgeo-6':
        'G 6 S 16 seg 262144 per_group 17 w 6 rho 6.804123711340206 | 0.0 1.0 2.0 3.0 4.0 5.0 0.1 1.1 2.1 3.1 4.1 5.1 0.2 1.2 2.2 3.2 4.2 5.2 0.3 1.3 2.3 3.3 4.3 5.3 0.4 1.4 2.4 3.4 4.4 5.4 0.5 1.5 2.5 3.5 4.5 5.5 0.6 1.6 2.6 3.6 4.6 5.6 0.7 1.7 2.7 3.7 4.7 5.7 0.8 1.8 2.8 3.8 4.8 5.8 0.9 1.9 2.9 3.9 4.9 5.9 0.10 1.10 2.10 3.10 4.10 5.10 0.11 1.11 2.11 3.11 4.11 5.11 0.12 1.12 2.12 3.12 4.12 5.12 0.13 1.13 2.13 3.13 4.13 5.13 0.14 1.14 2.14 3.14 4.14 5.14 0.15 1.15 2.15 3.15 4.15 5.15',
    's97-dgeo':
        'G 11 S 8 seg 524288 per_group 9 w 11 rho 0 | 0.0 1.0 2.0 3.0 4.0 5.0 6.0 7.0 8.0 9.0 10.0 0.1 1.1 2.1 3.1 4.1 5.1 6.1 7.1 8.1 9.1 10.1 0.2 1.2 2.2 3.2 4.2 5.2 6.2 7.2 8.2 9.2 10.2 0.3 1.3 2.3 3.3 4.3 5.3 6.3 7.3 8.3 9.3 10.3 0.4 1.4 2.4 3.4 4.4 5.4 6.4 7.4 8.4 9.4 10.4 0.5 1.5 2.5 3.5 4.5 5.5 6.5 7.5 8.5 9.5 10.5 0.6 1.6 2.6 3.6 4.6 5.6 6.6 7.6 8.6 9.6 10.6 0.7 1.7 2.7 3.7 4.7 5.7 6.7 7.7 8.7 9.7 10.7',
    'odd-cgeo':
        'G 5 S 13 seg 49280 per_group 34 w 0.69999999999999996 rho 3.8823529411764706 | 0.0 0.1 1.0 0.2 1.1 2.0 0.3 1.2 2.1 0.4 3.0 1.3 2.2 0.5 3.1 1.4 4.0 2.3 0.6 3.2 1.5 4.1 2.4 0.7 3.3 1.6 4.2 2.5 0.8 3.4 1.7 4.3 2.6 0.9 3.5 1.8 4.4 2.7 0.10 3.6 1.9 4.5 2.8 0.11 3.7 1.10 4.6 2.9 0.12 3.8 1.11 4.7 2.10 3.9 1.12 4.8 2.11 3.10 4.9 2.12 3.11 4.10 3.12 4.11 4.12',
    'odd-dgeo':
        'G 5 S 13 seg 49280 per_group 34 w 5 rho 0 | 0.0 1.0 2.0 3.0 4.0 0.1 1.1 2.1 3.1 4.1 0.2 1.2 2.2 3.2 4.2 0.3 1.3 2.3 3.3 4.3 0.4 1.4 2.4 3.4 4.4 0.5 1.5 2.5 3.5 4.5 0.6 1.6 2.6 3.6 4.6 0.7 1.7 2.7 3.7 4.7 0.8 1.8 2.8 3.8 4.8 0.9 1.9 2.9 3.9 4.9 0.10 1.10 2.10 3.10 4.10 0.11 1.11 2.11 3.11 4.11 0.12 1.12 2.12 3.12 4.12',
    'empty-middle-chunks':
        '0 1 0 1 | 1 1 1 1 | 1 1 1 1 | 1 15 1 15 | 15 33 15 33 | 33 41 33 41',
    'small-chunks':
        '0 11 0 11',
    'linked-chunks':
        '0 3 0 50 | 3 3 50 50 | 3 3 50 50 | 3 6 50 90 | 6 6 90 90 | 6 7 90 91',
    'cfg2-stripes-2':
        '0 839 0 839 | 839 1678 839 1678',
    'cfg2-stripes-8':
        '0 210 0 210 | 210 420 210 420 | 420 630 420 630 | 630 839 630 839 | 839 1049 839 1049 | 1049 1259 1049 1259 | 1259 1469 1259 1469 | 1469 1678 1469 1678',
    'linked-stripes-2':
        '0 3 0 50 | 3 7 50 91',
    'linked-stripes-8':
        '0 3 0 50 | 3 3 50 50 | 3 3 50 50 | 3 3 50 50 | 3 5 50 60 | 5 6 60 90 | 6 6 90 90 | 6 7 90 91',
}


def test_plans_are_pinned(plan):
    names = list(CASES)
    got = dict(zip(names, plan(*[CASES[k] for k in names])))
    assert set(PINNED) == set(CASES)
    for k in names:
        assert got[k] == PINNED[k], k


def test_empty_middle_chunk_still_counts(plan):
    r = [tuple(map(int, x.split())) for x in plan(CASES["empty-middle-chunks"])[0].split(" | ")]
    assert len(r) == 6 and r[1][2] == r[1][3] and r[2][2] == r[2][3]      # two empty chunks among six
    assert len(plan(CASES["small-chunks"])[0].split(" | ")) == 1


def parse_ranges(line):
    return [tuple(map(int, x.split())) for x in line.split(" | ")] if line else []


def check_ranges(r, n, first, exact=None, limit=None):
    units = len(first) - 1 if first else n
    assert r[0][0] == 0 and r[-1][1] == units
    for k, (u0, u1, b0, b1) in enumerate(r):
        assert u0 <= u1 and (b0, b1) == ((first[u0], first[u1]) if first else (u0, u1))     # whole streams only
        if k:
            assert u0 == r[k - 1][1]
    if exact is not None:
        assert len(r) == exact
    if limit is not None:
        assert 1 <= len(r) <= limit


def random_batch(rng):
    n = rng.choice([1, 2, 5, 40, 97, 300])
    big = rng.random() < 0.5
    lens = [rng.choice([0, 1, rng.randrange(1, 4 * MiB if big else 65536)]) for _ in range(n)]
    first = None
    if rng.random() < 0.5:
        cuts = sorted(rng.sample(range(1, n), rng.randrange(0, n)) if n > 1 else [])
        first = [0] + cuts + [n]
    return lens, first


def test_ranges_cover_the_batch_and_never_split_a_stream(plan):
    rng = random.Random(20261020)
    batches = [random_batch(rng) for _ in range(300)]
    cmds = []
    for lens, first in batches:
        cmds += [chunks(lens, first), chunks(lens, first, early=True), stripes(3, lens, first), stripes(8, lens, first)]
    out = plan(*cmds)
    for i, (lens, first) in enumerate(batches):
        for line in out[4 * i:4 * i + 2]:
            r = parse_ranges(line)
            check_ranges(r, len(lens), first, limit=6)
            if sum(lens) < 48 * MiB:
                assert len(r) == 1
        check_ranges(parse_ranges(out[4 * i + 2]), len(lens), first, exact=3)
        check_ranges(parse_ranges(out[4 * i + 3]), len(lens), first, exact=8)


def test_every_piece_once(plan):
    rng = random.Random(7)
    cmds, shapes = [], []
    for _ in range(300):
        n, L = rng.randrange(96, 3000), rng.randrange(65536, 8 * MiB)
        g, s = rng.choice(["-", str(rng.randrange(-2, 20))]), rng.choice(["-", str(rng.randrange(-2, 20))])
        w = rng.choice(["-", "0", str(rng.uniform(0, 30))])
        cmds.append(cgeo(n, L, n * L, rng.choice([2, 3, 6]), rng.choice([0, rng.uniform(1, 30)]), rng.choice([0, rng.uniform(5, 60)]), g, s, w))
        shapes.append((n, L))
        cmds.append(dgeo(n, L, g, s))
        shapes.append((n, L))
    for (n, L), line in zip(shapes, plan(*cmds)):
        head, pieces = line.split(" |")
        f = head.split()
        G, S, seg, per_group = int(f[1]), int(f[3]), int(f[5]), int(f[7])
        assert 1 <= G <= 16 and 1 <= S <= 16 and seg % 128 == 0 and (S - 1) * seg < L <= S * seg
        assert (G - 1) * per_group < n <= G * per_group
        got = [tuple(map(int, p.split("."))) for p in pieces.split()]
        assert sorted(got) == [(g, s) for g in range(G) for s in range(S)]
        for g in range(G):      # a group's segments go in order
            assert [s for gg, s in got if gg == g] == list(range(S))


def shape_rule(offs, lens, linked, cap, disabled):
    n = len(lens)
    if disabled or linked or cap or n < 96:
        return False
    L, P = lens[0], offs[1] - offs[0]
    return (L >= 65536 and L * n >= 96 * MiB and P >= L and all(o == offs[0] + P * i for i, o in enumerate(offs))
            and all(x == L for x in lens[:-1]) and 0 < lens[-1] <= L)


def route_rule(lens, caps, header, linked, out, disabled, wide, mapped):
    if out == "m" and header == 8 and not linked and not wide and mapped:
        return 2
    n = len(lens)
    if disabled or out == "c" or header != 8 or linked or n < 96 or lens[0] < 8:
        return 0
    cap = [c if x >= 8 else 0 for x, c in zip(lens, caps)]
    L = cap[0]
    ok = L >= 65536 and L * n >= 96 * MiB and all(c == L for c in cap[:-1]) and 0 < cap[-1] <= L
    return 1 if ok else 0


def test_streamed_eligibility_follows_the_rule(plan):
    rng = random.Random(96)
    cmds, want = [], []
    for _ in range(300):
        n = rng.choice([95, 96, 97, 170, 1678])
        L = rng.choice([65535, 65536, 640000, 1 << 20])
        lens = [L] * n
        lens[-1] = rng.choice([L, L + 1, 1, 0, L // 3])
        if rng.random() < 0.2:
            lens[rng.randrange(n)] = L - 1
        pitch = rng.choice([L, L + 16, L - 1])
        offs = [7 + i * pitch for i in range(n)]
        if rng.random() < 0.2:
            offs[rng.randrange(1, n)] += 1
        flags = [rng.random() < 0.1 for _ in range(3)]
        cmds.append(shape(offs, lens, *flags))
        want.append(f"{int(shape_rule(offs, lens, *flags))}")
        clens = [rng.choice([300000, 8, 7]) if rng.random() < 0.05 else 300000 for _ in range(n)]
        args = dict(header=rng.choice([8, 8, 8, 4, 0]), linked=rng.random() < 0.1, out=rng.choice(["-", "-", "c", "m", "p"]),
                    disabled=rng.random() < 0.1, wide=rng.random() < 0.1, mapped=rng.random() < 0.5)
        cmds.append(route(clens, lens, **args))
        want.append(f"{route_rule(clens, lens, **args)}")
    got = plan(*cmds)
    for c, g, w in zip(cmds, got, want):
        assert g.split()[0] == w, c[:120]


def carve(*sizes):
    """api.cu's descriptor blocks were carved as consecutive 16-byte aligned arrays"""
    at, offs = 0, []
    for b in sizes:
        offs.append(at)
        at = (at + b + 15) & ~15
    return offs, at


@pytest.mark.parametrize("n,ns,k", [(1, 1, 1), (7, 3, 2), (1678, 1678, 6), (97, 5, 6)])
def test_descriptor_layouts(plan, n, ns, k):
    # plain pipelines: src_off slot_off src_len cap first states | out_len out_off
    (o, end) = carve(8 * n, 8 * n, 4 * n, 4 * n, 4 * (ns + 1), 8 * ns, 4 * n, 8 * (n + k))
    got = list(map(int, plan(f"layout {n} {n} {n} {ns + 1} {ns} {n + k} 0")[0].split()))
    assert got == o[:6] + [o[6]] + o[6:8] + [end, end]
    # streamed compress: src_off slot_off src_len | out_len out_off (one extra entry per group)
    (o, end) = carve(8 * n, 8 * n, 4 * n, 4 * n, 8 * (n + k))
    got = list(map(int, plan(f"layout {n} {n} 0 0 0 {n + k} 0")[0].split()))
    assert [got[0], got[1], got[2], got[6], got[7], got[8], got[10]] == [o[0], o[1], o[2], o[3], o[3], o[4], end]
    # streamed decompress: src_off slot_off src_len cap | out_len ready flags
    (o, end) = carve(8 * n, 8 * n, 4 * n, 4 * n, 4 * n, 4 * 256)
    got = list(map(int, plan(f"layout {n} {n} {n} 0 0 0 256")[0].split()))
    assert [got[0], got[1], got[2], got[3], got[6], got[7], got[9], got[10]] == [o[0], o[1], o[2], o[3], o[4], o[4], o[5], end]
    # checksums: off len | out
    (o, end) = carve(8 * n, 4 * n, 4 * n)
    got = list(map(int, plan(f"layout {n} 0 0 0 0 0 0")[0].split()))
    assert [got[0], got[2], got[6], got[7], got[10]] == [o[0], o[1], o[2], o[2], end]


CTX, MULTI, DEV = 0, 1, 2
ARG = -2


def check(who, n=2, decode=0, owner=1, header=8, max_block=0, src=1, nbytes=100, dst=1, mask=15, given=0, first=None,
          off=None, lens=None):
    off = off if off is not None else [0, 50][:n] + [0] * max(0, n - 2)
    lens = lens if lens is not None else [10] * n
    ns = -1 if first is None else len(first) - 1
    return (f"check {who} {decode} {owner} {n} {header} {max_block} {src} {nbytes} {dst} {mask} {given} {ns} "
            f"{ints(first or [])} {ints(off if n > 0 else [])} {ints(lens if n > 0 else [])}")


REJECTIONS = [
    (check(CTX, owner=0), "ctx is NULL"),
    (check(CTX, n=-1), "NULL descriptor array"),
    (check(CTX, mask=7), "NULL descriptor array"),
    (check(CTX, header=5), "header_mode must be 0, 4 or 8"),
    (check(CTX, decode=1, header=4, max_block=-1), "max_block"),
    (check(CTX, given=1), "streams given without stream_first"),
    (check(CTX, src=0), "NULL data buffer"),
    (check(CTX, dst=0), "NULL data buffer"),
    (check(CTX, nbytes=59), "block 1 lies outside the source buffer"),
    (check(CTX, off=[0, -1]), "block 1 lies outside the source buffer"),
    (check(CTX, lens=[-1, 10]), "block 0 lies outside the source buffer"),
    (check(CTX, first=[0]), "n_streams"),
    (check(CTX, first=[1, 2]), "stream_first must start at 0 and end at n_blocks"),
    (check(CTX, first=[0, 1]), "stream_first must start at 0 and end at n_blocks"),
    (check(CTX, first=[0, 2, 1, 2]), "stream_first must be non-decreasing"),
    (check(MULTI, owner=0), "mctx is NULL"),
    (check(MULTI, n=-1), "NULL argument"),
    (check(MULTI, mask=14), "NULL argument"),
    (check(MULTI, src=0), "NULL argument"),
    (check(MULTI, dst=0), "NULL argument"),
    (check(MULTI, header=1), "header_mode must be 0, 4 or 8"),
    (check(MULTI, decode=1, header=0, max_block=-5), "max_block"),
    (check(MULTI, nbytes=10), "block 1 lies outside the source buffer"),
    (check(MULTI, first=[0, 3]), "stream_first must start at 0 and end at n_blocks"),
    (check(DEV, owner=0), "bad argument"),
    (check(DEV, n=-1), "bad argument"),
    (check(DEV, header=2), "header_mode must be 0, 4 or 8"),
]
ACCEPTED = [
    check(CTX), check(CTX, n=0, src=0, dst=0, mask=0), check(CTX, decode=1, header=8, max_block=-1),
    check(CTX, first=[0, 1, 2], given=1), check(CTX, first=[0, 0, 2]), check(MULTI, n=0, src=0, dst=0, mask=0),
    check(DEV, decode=1, header=0, max_block=-1, src=0, dst=0, mask=0, nbytes=0), check(DEV, n=0),
]


def test_argument_checks(plan):
    got = plan(*[c for c, _ in REJECTIONS], *ACCEPTED)
    for (c, msg), g in zip(REJECTIONS, got):
        assert g == f"{ARG} {msg}", c
    for c, g in zip(ACCEPTED, got[len(REJECTIONS):]):
        assert g == "0 ", c


# ---- GPU: the error path of every host pipeline leaves the ctx usable -----------------------------------------------

def _blocks(kind, seed, n, block):
    from streamly_lz4_b200 import datagen
    data = datagen.make(kind, seed, n * block)
    return data, np.arange(n, dtype=np.int64) * block, np.full(n, block, dtype=np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["compress-plain", "compress-streamed", "decompress-plain-h4", "decompress-plain-h8",
                                  "decompress-streamed"])
def test_dst_cap_too_small_then_a_good_call(ctx, ref, monkeypatch, case):
    streamed = case.endswith("streamed")
    n, block = (100, MiB) if streamed else (12, 100000)
    data, offs, lens = _blocks("mixed", 31, n, block)
    src = ctx.pinned("hp_src", data.size)[:data.size]       # (the pinned buffers are reused and may be larger)
    src[:] = data
    header = 4 if case.endswith("h4") else 8
    bound = int(sum(int(x) + int(x) // 255 + 16 + header for x in lens))
    if case.startswith("compress"):
        dst = ctx.pinned("hp_dst", bound)[:bound]
        n_before = ctx.launch_count()
        rc, _, _ = ctx.compress_batch(src, offs, lens, 1, header, dst[:64])
        assert rc == -3 and "dst_cap too small" in ctx.last_error(), (rc, ctx.last_error())
        assert ctx.launch_count() > n_before        # the call failed after it had queued work
        rc, doff, olen = ctx.compress_batch(src, offs, lens, 1, header, dst)
        assert rc == 0, ctx.last_error()
        want = ref.compress_chunks([data[i * block:(i + 1) * block].tobytes() for i in range(n)], 1, linked=False, threads=8)
        for i in range(n):
            assert dst[int(doff[i]):int(doff[i]) + header + int(olen[i])].tobytes() == want[i], i
        return
    arrays = [data[i * block:(i + 1) * block].tobytes() for i in range(n)]
    framed = ref.compress_chunks(arrays, 1, block_size="BlockHasSize" if header == 8 else "BlockMax256KB", linked=False, threads=8)
    blob = b"".join(framed)
    csrc = ctx.pinned("hp_csrc", len(blob))[:len(blob)]
    csrc[:] = np.frombuffer(blob, dtype=np.uint8)
    coff = np.cumsum([0] + [len(f) for f in framed[:-1]]).astype(np.int64)
    clen = np.array([len(f) for f in framed], dtype=np.int32)
    max_block = 0 if header == 8 else 256 << 10
    out = ctx.pinned("hp_out", n * block + 16 * n)[:n * block + 16 * n]
    if not streamed:
        monkeypatch.setenv("B200LZ4_DECODE_OUT", "copy")
    rc, _, _ = ctx.decompress_batch(csrc, coff, clen, header, max_block, out[:64])
    assert rc == -3 and "dst_cap too small" in ctx.last_error(), (rc, ctx.last_error())
    rc, boff, blen = ctx.decompress_batch(csrc, coff, clen, header, max_block, out)
    assert rc == 0, ctx.last_error()
    assert (blen == block).all()
    for i in range(n):
        assert out[int(boff[i]):int(boff[i]) + block].tobytes() == arrays[i], i
