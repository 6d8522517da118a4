"""Both decoders' copy paths on hand-built VALID blocks whose sequences sit exactly at the boundaries those paths are built
around: overlapping matches at every offset 1..64, batch and parse-window positions, the narrow copier's 8 KiB output ring
and its 64 preloaded bytes, the bulk path's period loops, the wide decoder's 16 KiB pieces and far/near split, the
dictionary and the DState tail kept across calls.  Encoder-made blocks reach these shapes only by chance.

Every case is an explicit list of sequences (literal length, match length, offset).  A plain Python model applies them
byte by byte and gives the plaintext.  Each case is checked three ways: the model equals the `ref` fixture's decode
(which also proves the block valid), and the GPU's output equals both, with nothing outside an output slot changed.

Routes, picked by launch_decompress's rule: the wide decoder (at most 2 x SM linked streams), the narrow decoder with 12
CTAs per SM, the narrow decoder with 16 CTAs per SM (more streams than CTAs: a CTA takes several streams one after
another), all through b200lz4_decompress_dev into sentinel-filled slots that start at every residue mod 16; and the host
call with the output mirrored from inside the kernel (B200LZ4_DECODE_OUT=mirror, header 8, independent blocks).
tests/test_gpu_modes.py re-runs this file with each decoder forced and on the bounds-checked build."""
import functools
import os

import numpy as np
import pytest

from test_gpu_device_abi import SENTINEL, Dev, framed, place, stream_firsts

KPIECE = 16384                       # decompress_wide.cu: long sequences are cut into pieces of this many output bytes
OVERLAP_LENGTHS = list(range(4, 21)) + [31, 32, 33, 34, 63, 64, 65, 66, 100, 273, 274, 275, 528, 529, 530, 2000]
FILLERS_BEFORE = [1, 10, 11, 12, 31]  # around kWindowSeqs (11 sequences per parse window) and kQDepth (32 per batch)


# ---- block builder and model ----------------------------------------------------------------------------------------------

def _emit_len(out, v):
    v -= 15
    while v >= 255:
        out.append(255)
        v -= 255
    out.append(v)


class Block:
    """One LZ4 block from an explicit sequence list.  seqs: (literal length, match length, offset); `last`: the final
    literal run.  The literal bytes come from `pool` starting at `at`.  `dictionary`: the previous block's output of a
    linked stream (None: independent).  `empty`: the one valid block of an empty array."""

    def __init__(self, seqs, last, pool, at=0, dictionary=None, empty=False):
        self.seqs, self.last = list(seqs), last
        if empty:
            self.seqs, self.last, self.payload, self.plain, self.starts = [], 0, b"\x00", b"", np.zeros(0, np.int64)
            return
        assert self.seqs == [] or last >= 12, "a block with matches ends with >= 12 literals (MFLIMIT)"
        n_lit = sum(s[0] for s in self.seqs) + last
        lits = pool[at:at + n_lit]
        assert len(lits) == n_lit, "literal pool too small"
        d = bytes(dictionary[-65536:]) if dictionary else b""
        out = bytearray(d)
        enc = bytearray()
        starts = []
        li = 0
        for k, (lit, ml, off) in enumerate(self.seqs):
            assert lit >= 0 and ml >= 4 and 1 <= off <= 65535, (k, lit, ml, off)
            starts.append(len(out) - len(d))
            enc.append((min(lit, 15) << 4) | min(ml - 4, 15))
            if lit >= 15:
                _emit_len(enc, lit)
            enc += lits[li:li + lit]
            out += lits[li:li + lit]
            li += lit
            enc += bytes((off & 255, off >> 8))
            if ml - 4 >= 15:
                _emit_len(enc, ml - 4)
            src = len(out) - off
            assert src >= 0, f"sequence {k} {(lit, ml, off)} reaches before the dictionary"
            if off >= ml:
                out += out[src:src + ml]
            else:                                   # overlapping: the source period repeated
                out += (out[src:src + off] * (ml // off + 1))[:ml]
        enc.append(min(last, 15) << 4)
        if last >= 15:
            _emit_len(enc, last)
        enc += lits[li:li + last]
        out += lits[li:li + last]
        self.payload, self.plain = bytes(enc), bytes(out[len(d):])
        self.starts = np.array(starts, dtype=np.int64)

    @property
    def n(self):
        return len(self.plain)

    def where(self, pos):
        """The sequence that produced output byte `pos`."""
        if not self.seqs or pos >= self.n - self.last:
            return f"the final literal run ({self.last} bytes)"
        k = int(np.searchsorted(self.starts, pos, side="right")) - 1
        return f"sequence {k} (lit, ml, off) = {self.seqs[k]}"


class Family:
    """Streams (lists of Blocks; a block's dictionary is the stream's last non-empty output before it)."""

    def __init__(self, name, streams, independent):
        self.name, self.streams, self.independent = name, streams, independent

    @property
    def blocks(self):
        return [b for s in self.streams for b in s]


class StreamBuilder:
    def __init__(self, pool):
        self.pool, self.at, self.blocks, self.prev = pool, 0, [], None

    def add(self, seqs, last, empty=False):
        b = Block(seqs, last, self.pool, self.at, self.prev, empty)
        self.at = (self.at + sum(s[0] for s in b.seqs) + b.last) % (len(self.pool) // 2)
        if b.n:
            self.prev = b.plain
        self.blocks.append(b)
        return b


def _pool(seed, n=1 << 19):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8).tobytes()


def _single_blocks(pool, block_seqs):
    out, at = [], 0
    for seqs, last in block_seqs:
        b = Block(seqs, last, pool, at)
        at = (at + sum(s[0] for s in seqs) + last) % (len(pool) // 2)
        out.append([b])
    return out


# ---- case families ----------------------------------------------------------------------------------------------------------

def _fillers(j):
    """j short sequences (window path); returns (seqs, bytes produced)."""
    seqs = [(8, 4, 3)] + [(1, 4, 1 + (k * 5) % 8) for k in range(1, j)]
    return seqs, sum(a + b for a, b, _ in seqs)


def fam_overlap():
    """Every offset 1..64 x OVERLAP_LENGTHS, placed as the first sequence of a block (first of its batch), after j short
    fillers, and right after a bulk sequence (its source in the ring's 64 preloaded bytes)."""
    cases = []
    for off in range(1, 65):
        for i, ml in enumerate(OVERLAP_LENGTHS):
            cases.append(([(off + ml % 5, ml, off)], 16))
            for j in FILLERS_BEFORE:
                seqs, made = _fillers(j)
                cases.append((seqs + [(max(0, off - made), ml, off)], 16))
            bulk = (70, 4, 7) if i % 2 == 0 else (8, 200, 3)          # a long literal run / a long match
            cases.append(([bulk, (0, ml, off)], 16))
    return Family("overlap", _single_blocks(_pool(1), cases), True)


LIT_RUNS = [14, 15, 16, 31, 32, 33, 269, 270, 271, 524, 525, 526, 2047, 2048, 2049, 4095, 4096, 4097, 16383, 16384, 16385,
            3 * KPIECE + 1, 70000]
MATCH_LENGTHS = [64, 65, 16383, 16384, 16385, 49153, 100000]
OFFSETS = [1, 3, 31, 32, 33, 4095, 8191, 8192, 8193, 20000, 65535]


def fam_lengths():
    """Literal runs and match lengths at the 15 / 255 extension steps, kShortLit / kShortMatch and the wide decoder's
    16 KiB pieces, with offsets below, at and above the ring sizes (offset < length across piece boundaries)."""
    cases = []
    for r in LIT_RUNS:
        cases.append(([(r, 8, 3)], 16))                    # as a sequence's literals
        cases.append(([(8, 4, 3)], r))                     # as the final run
        cases.append(([(5, 4, 1), (r, 70, 20)], 13))       # followed by a bulk match
    for ml in MATCH_LENGTHS:
        for off in OFFSETS:
            cases.append(([(off, ml, off)], 16))
    cases.append(([(3, 100000, 1), (2, 49153, 3), (40, 16385, 33)], 20))
    return Family("lengths", _single_blocks(_pool(2, 1 << 20), cases), True)


def fam_ring_alias():
    """After a long literal run, batches of 22 long-ish literal runs (one sequence per parse window) in which every third
    match has an offset 8100..8192: its source lies in [op0 - 8192, op1 - 8192), ring slots this batch's own literals
    have already overwritten, so it must come from global memory."""
    blocks = []
    for variant in range(2):
        seqs = [(9000, 4, 1)]
        q_all = 0
        for g in range(40):
            for q in range(22):
                if q % 3 == 1:
                    seqs.append((17 + (q_all + variant) % 16, 4 + (g * 7 + q) % 61, 8100 + (q_all * 5 + variant) % 93))
                else:
                    seqs.append((32 - variant * (q % 4), 4 + (q * 5 + g) % 30, 1 + (q * 13 + g) % 64))
                q_all += 1
        blocks.append((seqs, 16))
    return Family("ring_alias", _single_blocks(_pool(3), blocks), True)


def fam_far_near():
    """Linked streams whose match sources end exactly at, one before and one after the output start of each of the
    previous 3 x 32 sequences: the source end walks across every ticket boundary of the wide decoder."""
    streams = []
    for s in range(2):
        sb = StreamBuilder(_pool(40 + s))
        for blk in range(4):
            seqs, starts, op = [], [], 0
            for i in range(2400):
                if i < 96:
                    lit, ml = 8 + i % 20, 4 + i % 40
                    off = 1 + (i * 7) % min(op + lit, 64)
                else:
                    lit, ml = (i * 7 + blk + s) % 33, 4 + (i * 11 + s) % 61
                    k, d = 1 + (i // 3) % 96, i % 3 - 1
                    off = op + lit + ml - starts[i - k] - d
                starts.append(op)
                seqs.append((lit, ml, off))
                op += lit + ml
            sb.add(seqs, 16)
        streams.append(sb.blocks)
    return Family("far_near", streams, False)


DICT_SIZES = [1, 5, 64, 65, 8191, 65535, 65536, 70000]


def _reach_seqs(d):
    """Matches reaching exactly to the dictionary start and 1..64 bytes before the block start."""
    reach = min(d, 65535)
    seqs, op = [(0, 4 + reach % 7, reach)], 0
    op += seqs[0][1]
    for r in range(1, min(64, d) + 1):
        ml = [4, 5, 17, 33, 64][r % 5]
        seqs.append((0, ml, op + r))
        op += ml
    return seqs


def fam_dict_reach():
    """Dictionaries of DICT_SIZES bytes; the next block reaches exactly to their start and 1..64 bytes back; bulk matches
    (length > 64, offset < length) start in the dictionary and run on into the block; an empty block between a
    dictionary and its user (the reference decides what it means)."""
    streams = []
    for i, d in enumerate(DICT_SIZES):
        for kind in ("reach", "bulk", "empty_between"):
            sb = StreamBuilder(_pool(50 + i, 1 << 18))
            sb.add([], d)
            if kind == "empty_between":
                sb.add([], 0, empty=True)
            if kind == "bulk":
                for j, r in enumerate(r for r in sorted({1, 2, 3, 17, 31, 32, 33, 63, 64, 65, 100, 1000, min(d, 65535)})
                                      if r <= d):
                    if j:
                        sb.add([], d)                      # a fresh dictionary for each
                    sb.add([(0, max(100, 2 * r + 70), r)], 16)
            else:
                sb.add(_reach_seqs(d), 16)
            streams.append(sb.blocks)
    return Family("dict_reach", streams, False)


def fam_many_seqs():
    """9 000, 70 000 and 2^20 minimal sequences (no literals, length 4, offsets 1..64): more batches than a parser ring
    holds; the last block is 4 MiB."""
    blocks = []
    for count in (9000, 70000, 1 << 20):
        seqs = [(64, 4, 1)] + [(0, 4, 1 + (i * 37) % 64) for i in range(1, count)]
        blocks.append((seqs, 16))
    return Family("many_seqs", _single_blocks(_pool(6, 1 << 16), blocks), True)


FAMILIES = {f.__name__[4:]: f for f in (fam_overlap, fam_lengths, fam_ring_alias, fam_far_near, fam_dict_reach,
                                        fam_many_seqs)}


@functools.lru_cache(maxsize=None)
def family(name):
    return FAMILIES[name]()


def across_calls_streams():
    """(streams, cut) for decoding over two calls: the first block of the second call reaches into the kept tail (DState)
    of a previous block shorter than and longer than 64 KiB, up to 65 535 bytes back."""
    streams = []
    for s, size in enumerate((40000, 100000, 65536)):
        sb = StreamBuilder(_pool(70 + s, 1 << 18))
        if s == 2:
            sb.add([(30, 50, 20)], 500)                    # an earlier block: the cut comes after two
        sb.add([(size - 984, 600, 7)], 384)               # exactly `size` bytes
        reaches = [r for r in (65535, 50000, 32769, 32768, 32767, 1000, 64, 1) if r <= min(size, 65535)]
        seqs, op = [], 0
        for r in reaches:
            off = op + r
            if off > 65535:
                continue
            ml = 20 + len(seqs)
            seqs.append((0, ml, off))
            op += ml
        seqs.append((0, 300, op + 40))                     # a bulk match that starts in the tail
        sb.add(seqs, 16)
        sb.add([(0, 70, 300)], 16)                         # and a block after it that reaches into it
        streams.append(sb.blocks)
    return streams


# ---- checks ------------------------------------------------------------------------------------------------------------------

def ref_outputs(ref, streams):
    frames = [framed(b.payload, b.n, 8) for s in streams for b in s]
    sf = stream_firsts([len(s) for s in streams])
    return ref.decompress_chunks_raw(frames, stream_first=sf, threads=8)


def first_diff(got, want):
    g, w = np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8)
    m = min(len(g), len(w))
    bad = np.flatnonzero(g[:m] != w[:m])
    return int(bad[0]) if bad.size else m


def check_block(label, b, got):
    if got != b.plain:
        p = first_diff(got, b.plain)
        gv = f"0x{got[p]:02x}" if p < len(got) else "nothing"
        wv = f"0x{b.plain[p]:02x}" if p < b.n else "nothing"
        raise AssertionError(f"{label} ({b.n} bytes, {len(b.seqs)} sequences): first wrong byte {p} in {b.where(p)}: "
                             f"got {gv}, want {wv}")


def check_model(ref, name, streams):
    want = ref_outputs(ref, streams)
    i = 0
    for s, st in enumerate(streams):
        for k, b in enumerate(st):
            check_block(f"{name}: model vs reference, stream {s} block {k}", b, want[i])
            i += 1


@pytest.mark.parametrize("name", list(FAMILIES) + ["across_calls"])
def test_model_matches_reference(ref, name):
    """The builder makes valid blocks and the model decodes them as the reference does (no GPU needed)."""
    streams = across_calls_streams() if name == "across_calls" else family(name).streams
    check_model(ref, name, streams)


# ---- GPU routes ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def dev(ctx):
    import torch
    from streamly_lz4_b200 import _lib
    return Dev(torch, _lib.load())


@functools.lru_cache(maxsize=None)
def _filler():
    return Block([(8, 4, 3), (1, 6, 5)], 12, _pool(9, 4096))


def residue_slots(sizes, salt):
    """Slot starts: each slot begins at the first position at or after the previous slot's end whose residue mod 16 is
    (7 i + salt) % 16, so the slots of a launch start at every residue and most of them touch their neighbours."""
    offs, at = [], 0
    for i, n in enumerate(sizes):
        at += ((7 * i + salt) - at) % 16
        offs.append(at)
        at += int(n)
    return np.array(offs, dtype=np.int64), at


def launch_groups(dev, route, streams, linked):
    """Split `streams` into launches and pad each so that launch_decompress picks `route`.  Returns a list of
    (streams of the launch, index of each in `streams` or -1 for filler, pass stream_first)."""
    sm = dev.sm
    if route == "wide":
        lim = 2 * sm
        if not linked:                       # one-block streams regrouped into at most 2 x SM linked streams
            k = -(-len(streams) // lim)
            groups = [list(range(i, min(i + k, len(streams)))) for i in range(0, len(streams), k)]
            merged = [[streams[i][0] for i in g] for g in groups]
            return [(merged, [("merged", g) for g in groups], True)]
        return [(streams[i:i + lim], list(range(i, min(i + lim, len(streams)))), True)
                for i in range(0, len(streams), lim)]
    lo, hi = (2 * sm + 1, 12 * sm) if route == "narrow12" else (16 * sm + 200, 1 << 30)
    if not linked and route == "narrow12":
        lo = 1
    out = []
    for i in range(0, len(streams), hi):
        part = list(range(i, min(i + hi, len(streams))))
        total = max(len(part), lo)
        idx = [-1] * total                   # our streams spread evenly among the fillers
        for j, p in enumerate(part):
            idx[j * total // len(part)] = p
        out.append(([streams[p] if p >= 0 else [_filler()] for p in idx], idx, linked or route == "wide"))
    return out


def run_dev(dev, streams, use_sf, salt, states=None):
    """One decompress_dev launch (header 8, every slot exactly its block's size); returns the blocks' outputs and checks
    that nothing outside the slots changed and the scratch header is clean."""
    torch = dev.torch
    blocks = [b for s in streams for b in s]
    frames = [framed(b.payload, b.n, 8) for b in blocks]
    rng = np.random.default_rng(salt)
    src, src_off, lens = place(frames, "odd", rng)
    sizes = np.array([b.n for b in blocks], dtype=np.int32)
    dst_off, end = residue_slots(sizes, salt)
    out = dev.put(np.full(end + 64, SENTINEL, dtype=np.uint8))
    out_len = dev.put(np.full(len(blocks), -7, dtype=np.int32))
    sf = dev.put(stream_firsts([len(s) for s in streams])) if use_sf else None
    dev.decompress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), dev.put(sizes), out_len, 8, 0,
                   sf=sf, states=states)
    dev.sync_and_check_scratch()
    got, got_len = dev.get(out), dev.get(out_len)
    outside = np.ones(end + 64, dtype=bool)
    res = []
    for b, o, n, r in zip(blocks, dst_off, sizes, got_len):
        outside[o:o + n] = False
        res.append((int(r), got[o:o + n].tobytes()))
    bad = np.flatnonzero(outside & (got != SENTINEL))
    assert not bad.size, f"a byte outside every slot changed: buffer position {bad[0]} (slots end at {end})"
    return res


def check_stream(label, st, res):
    """The blocks of one stream against their (out_len, bytes) from run_dev."""
    for k, (b, (r, got)) in enumerate(zip(st, res)):
        assert r == b.n, f"{label} block {k}: out_len {r}, want {b.n}"
        check_block(f"{label} block {k}", b, got)


def run_route(dev, route, fam):
    for g, (streams, idx, use_sf) in enumerate(launch_groups(dev, route, fam.streams, not fam.independent)):
        res = run_dev(dev, streams, use_sf, salt=g + 3)
        i = 0
        for (st, where) in zip(streams, idx):
            if isinstance(where, tuple):         # one-block streams where[1] merged into one linked stream
                for k, b in enumerate(st):
                    check_stream(f"{fam.name} on {route}: launch {g}, stream {where[1][k]} (merged)", [b], res[i + k:i + k + 1])
            else:
                check_stream(f"{fam.name} on {route}: launch {g}, " + (f"stream {where}" if where >= 0 else "filler stream"),
                             st, res[i:i + len(st)])
            i += len(st)


def run_mirror(ctx, fam):
    """The host call with B200LZ4_DECODE_OUT=mirror (read per call): independent blocks, header 8."""
    import streamly_lz4_b200 as lz
    frames = [framed(s[0].payload, s[0].n, 8) for s in fam.streams]
    old = os.environ.get("B200LZ4_DECODE_OUT")
    os.environ["B200LZ4_DECODE_OUT"] = "mirror"
    try:
        src, offs, plens = lz.api._gather(ctx, "geom_src", frames)
        total = sum(s[0].n for s in fam.streams)
        dst = ctx.pinned("geom_dst", total + 4096)
        dst[:total + 4096] = SENTINEL
        rc, doff, olen = ctx.decompress_batch(src, offs, plens, 8, 0, dst)
    finally:
        if old is None:
            del os.environ["B200LZ4_DECODE_OUT"]
        else:
            os.environ["B200LZ4_DECODE_OUT"] = old
    assert rc == 0, rc
    for s, st in enumerate(fam.streams):
        b = st[0]
        assert olen[s] == b.n, f"{fam.name} on mirror: block {s}: out_len {olen[s]}, want {b.n}"
        check_block(f"{fam.name} on mirror: block {s}", b, dst[doff[s]:doff[s] + b.n].tobytes())
    assert (dst[int(doff[-1]):total + 4096] == SENTINEL).all(), "the call wrote past its output"


INDEPENDENT = ["overlap", "lengths", "ring_alias", "many_seqs"]       # the families of one-block streams without dictionary
ROUTES = [(name, route) for name in FAMILIES for route in ("wide", "narrow12", "narrow16", "mirror")
          if route != "mirror" or name in INDEPENDENT]             # (the mirrored host call takes independent blocks only)


@pytest.mark.gpu
@pytest.mark.parametrize("name,route", ROUTES, ids=[f"{n}-{r}" for n, r in ROUTES])
def test_family_decodes_like_the_model(dev, ctx, ref, name, route):
    fam = family(name)
    assert fam.independent == (name in INDEPENDENT)
    check_model(ref, name, fam.streams)
    if route == "mirror":
        run_mirror(ctx, fam)
    else:
        run_route(dev, route, fam)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["wide", "narrow12", "narrow16"])
def test_linked_stream_across_calls(dev, ref, route):
    """The same linked streams decoded in one call and in two: the second call's first block reaches up to 65 535 bytes
    back into the tail the previous call kept in the caller's DState record."""
    streams = across_calls_streams()
    check_model(ref, "across_calls", streams)
    sb = dev.lib.b200lz4_dstate_bytes()
    sm = dev.sm
    n_total = {"wide": len(streams), "narrow12": 2 * sm + 9, "narrow16": 16 * sm + 200}[route]
    spread = [j * n_total // len(streams) for j in range(len(streams))]
    for calls in (1, 2):
        states = dev.zeros(n_total * sb)
        ptrs = dev.put(np.array([states.data_ptr() + s * sb for s in range(n_total)], dtype=np.uint64).view(np.int64))
        cuts = [len(s) - 2 if calls == 2 else len(s) for s in streams]
        for part in range(calls):
            mine = {p: (st[:c] if part == 0 else st[c:]) for p, st, c in zip(spread, streams, cuts)}
            launch = [mine.get(p, [_filler()]) for p in range(n_total)]
            res = run_dev(dev, launch, True, salt=11 + part, states=ptrs)
            i = 0
            for p, st in enumerate(launch):
                label = f"across_calls on {route}, {calls} call(s), call {part}, " + \
                        (f"stream {spread.index(p)}" if p in mine else "filler stream")
                check_stream(label, st, res[i:i + len(st)])
                i += len(st)
