"""Hand-built LZ4 frames for the window decoder: linked frames whose blocks reach back across the last 64 KiB of the
frame's content, not just the previous block (LZ4F_decompress's window).  Pure Python and deterministic; upstream's
verdict on every case is stored in tests/golden/frames/window_checks.json (frame_golden.py window), and the tests
(test_frame_golden.py on the CPU, test_gpu_frame_window.py on the device) rebuild the cases from this module.

Each block is a test_gpu_decode_geometry.Block given the frame's content so far as its dictionary, so the Block model is
the content a stock reader produces.  A block meant to be rejected (an offset one past the content so far) is built
against the content with `phantom` zero bytes in front: its payload is the intended one, its model output is unused.

Families:
  reach     sources 1, 2 or many blocks back, over earlier blocks of 1 .. 65535 bytes
  straddle  a match whose source starts in earlier blocks and runs into the current one, at every offset 1 .. 64, short
            and bulk lengths (overlapping and not), with literals below and above the bulk threshold
  clamp     offset 65535 after 65535, 65536, 65537 and about 200 000 bytes of earlier content
  limit     an offset equal to the bytes decoded so far, and one more, at block starts after the frame start
  stored    stored blocks of 14 .. 525 bytes (length bytes of the staged literal block) with matches reaching across them
  empty     blocks that decode to nothing between real ones
  bmax      a block decoding to exactly the block maximum, and to one byte more, in each class
  expand    blocks that expand as much as their payload allows, back to back, linked and independent
  fail      a failing block in the middle of a frame, valid blocks after it
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.dirname(HERE)):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import frame  # noqa: E402
from test_gpu_decode_geometry import Block, _pool  # noqa: E402

BMAX = frame.BD_SIZES
KB64 = 65536


class Case:
    """One frame: `blob`, and `plain` -- the content a stock reader produces, or None when a block is built to be
    rejected."""

    def __init__(self, cid, blob, plain, block_max):
        self.id, self.blob, self.plain, self.block_max = cid, blob, plain, block_max


class FrameBuilder:
    """A frame block by block.  `pool`: the literal bytes (default: drawn from `seed`); `dictionary`: content in front of
    the frame that its blocks may reference (LZ4F_decompress_usingDict), not part of the frame's content."""

    def __init__(self, seed, bd_code=4, independent=False, block_checksum=False, content_size=False,
                 content_checksum=False, pool=None, dictionary=b""):
        self.pool, self.at = pool if pool is not None else _pool(seed), 0
        self.code, self.independent = bd_code, independent
        self.bc, self.cs, self.cc = block_checksum, content_size, content_checksum
        self.content, self.blocks, self.valid, self.skip = bytearray(dictionary), [], True, len(dictionary)

    def _take(self, n):
        assert n <= len(self.pool) // 2
        if self.at + n > len(self.pool) // 2:
            self.at = 0
        s = self.at
        self.at += n
        return s

    def seqs(self, seqs, last, phantom=0):
        """A compressed block of (literal length, match length, offset) sequences and `last` final literals."""
        dic = bytes(self.content[:self.skip]) if self.independent else (b"\0" * phantom + bytes(self.content[-KB64:]))
        b = Block(seqs, last, self.pool, self._take(sum(s[0] for s in seqs) + last), dic)
        assert len(b.payload) <= BMAX[self.code]
        self.blocks.append((False, b.payload))
        if phantom:
            self.valid = False
        self.content += b.plain
        return self

    def lits(self, n):
        return self.seqs([], n)

    def stored(self, n):
        s = self._take(n)
        raw = self.pool[s:s + n]
        self.blocks.append((True, raw))
        self.content += raw
        return self

    def empty(self):
        self.blocks.append((False, b"\x00"))
        return self

    def raw(self, payload):
        """A compressed block given as bytes (rejected ones)"""
        self.blocks.append((False, payload))
        self.valid = False
        return self

    def case(self, cid):
        content = bytes(self.content[self.skip:])
        out = [frame.header(self.code, self.independent, self.bc, len(content) if self.cs else None, self.cc)]
        for stored, data in self.blocks:
            out.append((len(data) | (0x80000000 if stored else 0)).to_bytes(4, "little") + data)
            if self.bc:
                out.append(frame.xxh32(data).to_bytes(4, "little"))
        out.append(b"\0\0\0\0")
        if self.cc:
            out.append(frame.xxh32(content).to_bytes(4, "little"))
        return Case(cid, b"".join(out), content if self.valid else None, BMAX[self.code])


def _reach(seed):
    out = []
    for size in (1, 5, 11, 12, 31, 32, 33, 64, 65, 100, 4096, 65535):
        count = 2 if size == 65535 else 6
        f = FrameBuilder(seed + size, bd_code=5 if size == 65535 else 4)
        for _ in range(count):
            f.lits(size)
        n = len(f.content)
        seqs, op = [], 0
        for back in (1, 2, count):             # a source inside the block `back` blocks before the current one
            for within in (0, size // 2, size - 1):
                lit = 1 + within % 3
                src = n - back * size + within
                off = n + op + lit - src
                ml = 4 + (size + within) % 70
                if off > 65535:                 # (beyond the window: 65 535-byte blocks, back 2)
                    continue
                seqs.append((lit, ml, off))
                op += lit + ml
        out.append(f.seqs(seqs, 12).case(f"reach_{size}"))
    return out


def _straddle(seed):
    """one frame per shape: three packed earlier blocks (64 bytes), then one block per offset 1 .. 64 whose first match
    starts before the block start and runs into the block"""
    out = []
    shapes = {"short": lambda off, lit: off - lit + 3,               # match <= 64 ending inside the current block
              "bulk": lambda off, lit: 65 + off,                    # > 64, overlapping (offset <= 64)
              "bulklit": lambda off, lit: off - lit + 2}            # literals > 32 before it (bulk literal path)
    for name, ml_of in shapes.items():
        f = FrameBuilder(seed + len(out))
        for n in (5, 11, 48):
            f.lits(n)
        for off in range(1, 65):
            lit = (33 if off > 33 else off - 1) if name == "bulklit" else off // 2
            if lit >= off:
                continue
            f.seqs([(lit, max(4, ml_of(off, lit)), off)], 12)
        out.append(f.case(f"straddle_{name}"))
    # bulk and not overlapping: offset >= match length > 64, source across two earlier blocks and the block start
    f = FrameBuilder(seed + 10)
    for n in (40, 70, 90):
        f.lits(n)
    for off, lit, ml in ((100, 40, 80), (150, 10, 150), (200, 33, 180), (129, 64, 65), (300, 0, 300)):
        f.seqs([(lit, ml, off)], 12)
    out.append(f.case("straddle_bulk_disjoint"))
    return out


def _clamp(seed):
    out = []
    for total, code, parts in ((65535, 5, [65535]), (65536, 5, [65536]), (65537, 5, [65536, 1]), (200_000, 5, [200_000]),
                               (65535, 4, [30000, 35535]), (65537, 4, [60000, 5537]), (200_000, 4, [65536] * 3 + [3392])):
        f = FrameBuilder(seed + total + code, bd_code=code)
        for n in parts:
            if code == 4 and n > 60000:
                f.stored(n)
            else:
                f.lits(n)
        assert len(f.content) == total
        f.seqs([(0, 20, 65535), (5, 100, 65535), (0, 4, 65535 - 105 + 7)], 12)
        out.append(f.case(f"clamp_{total}_b{code}_{len(parts)}"))
    return out


def _limit(seed):
    out = []
    for k, (parts, lit) in enumerate((([1000, 2000], 0), ([10, 20, 30], 3), ([1, 1], 0), ([5, 7], 2), ([4096, 1], 15),
                                     ([33], 40))):
        for extra in (0, 1):
            f = FrameBuilder(seed + k)
            for n in parts:
                f.lits(n)
            n = len(f.content)
            f.seqs([(lit, 8, n + lit + extra)], 12, phantom=extra)
            f.lits(20)                          # a valid block after it
            out.append(f.case(f"limit_{k}_{'over' if extra else 'equal'}"))
    return out


def _stored(seed):
    out = []
    for n in (14, 15, 16, 269, 270, 271, 524, 525):
        f = FrameBuilder(seed + n, block_checksum=n % 2 == 0, content_checksum=True)
        f.lits(50).stored(n)
        m = len(f.content)
        # into the stored block (its first and last byte), back across it into the first block, and a straddle of its end
        f.seqs([(0, 10, n), (2, 30, 12 + n + 40), (1, 6, 1), (3, 4, m + 45)], 12)
        f.stored(n).seqs([(0, 8, n + 4)], 12)
        out.append(f.case(f"stored_{n}"))
    return out


def _empty(seed):
    f = FrameBuilder(seed, content_size=True)
    f.lits(500).empty().empty().lits(300).empty()
    f.seqs([(0, 40, 790), (4, 64, 301), (0, 5, 500)], 12).empty()
    out = [f.case("empty_between")]
    f = FrameBuilder(seed + 1)
    f.empty().lits(3).empty().seqs([(1, 4, 4)], 12)
    out.append(f.case("empty_first"))
    return out


def _bmax(seed):
    out = []
    for code in (4, 5, 6, 7):
        for extra in (0, 1):
            f = FrameBuilder(seed + code, bd_code=code)
            f.lits(100)
            ml = BMAX[code] - 12 - 1 + extra
            f.seqs([(1, ml, 50)], 12)          # decodes to block max + extra; the +1 block is rejected
            if extra:
                f.valid = False
            f.lits(30)
            out.append(f.case(f"bmax_b{code}_{'over' if extra else 'exact'}"))
    return out


def _expand(seed):
    out = []
    for code in (4, 6):
        for ind in (False, True):
            f = FrameBuilder(seed + code + ind, bd_code=code, independent=ind)
            for k in range(3):
                f.seqs([(1 + k, BMAX[code] - 13 - k, 1)], 12)
            out.append(f.case(f"expand_b{code}_{'ind' if ind else 'lnk'}"))
    return out


def _fail(seed):
    f = FrameBuilder(seed, block_checksum=True)
    f.lits(200).seqs([(0, 10, 201)], 12, phantom=1).lits(40).seqs([(0, 20, 100)], 12)
    out = [f.case("fail_offset_mid")]
    f = FrameBuilder(seed + 1)
    f.lits(200).raw(bytes([0xF0, 40]) + b"x" * 20).lits(40)       # literals past the end of the block
    out.append(f.case("fail_cut_mid"))
    return out


def cases():
    """Every case, in a fixed order."""
    out = []
    for k, fam in enumerate((_reach, _straddle, _clamp, _limit, _stored, _empty, _bmax, _expand, _fail)):
        out += fam(7000 + 1000 * k)
    assert len({c.id for c in out}) == len(out)
    return out
