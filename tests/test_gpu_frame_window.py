"""The frame decoder's window mode (decompress_kernel<..., kWindow = true>): in a linked frame a block may reference the
last 64 KiB of the frame's content, across any number of earlier blocks, as LZ4F_decompress does.  Every hand-built case
of tests/golden/window_cases.py in one call (host and device pointers), more window frames than 12 x SM (several frames
per CTA, the window reset at each frame start), about 5 000 shuffled frames of every class, mode, flag set and
corruption, read_frame on short linked blocks, and the frame encoder at block-split sizes and on every compressor route.

Each frame is checked against the CPU window reference (oracle/frame.py: verdict, decode), whose verdicts on the
hand-built cases are pinned to upstream LZ4F by tests/golden/frames/window_checks.json.  The destination is filled with a
sentinel, and every byte outside [dst_off, dst_off + content) must keep it; a failing frame writes nothing (a content
checksum mismatch is found after the content is in place, so only that verdict leaves bytes behind).
tests/test_gpu_modes.py re-runs this file with each decoder forced and on the bounds-checked build."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

import streamly_lz4_b200 as lz
from oracle import frame
from streamly_lz4_b200 import api, datagen

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import window_cases  # noqa: E402
from window_cases import FrameBuilder  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
GAP = 48                  # sentinel bytes between two frames' destinations
CLASSES = {4: 65536, 5: 262144, 6: 1 << 20, 7: 4 << 20}
NAMES = {65536: "BlockMax64KB", 262144: "BlockMax256KB", 1 << 20: "BlockMax1MB", 4 << 20: "BlockMax4MB"}


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def cases():
    return window_cases.cases()


def decode(ctx, blobs, caps, device=False):
    """(rc, out_len, dst, dst_off) of one frame_decompress_batch call; destinations GAP bytes apart, sentinel-filled"""
    src = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy()
    ln = np.array([len(b) for b in blobs], dtype=np.int32)
    off = np.concatenate([[0], np.cumsum(ln.astype(np.int64))[:-1]]).astype(np.int64)
    caps = np.asarray(caps, dtype=np.int32)
    doff = (GAP + np.concatenate([[0], np.cumsum(caps.astype(np.int64) + GAP)[:-1]])).astype(np.int64)
    dst = np.full(int(doff[-1] + caps[-1] + GAP), SENTINEL, dtype=np.uint8)
    if device:
        import torch
        t = lambda a: torch.from_numpy(a).cuda()
        d_dst = t(dst)
        rc, out = ctx.frame_decompress_batch(t(src), t(off), t(ln), d_dst, t(doff), t(caps))
        dst = d_dst.cpu().numpy()
    else:
        rc, out = ctx.frame_decompress_batch(src, off, ln, dst, doff, caps)
    return rc, out, dst, doff


def check(labels, blobs, caps, want_code, want_plain, rc, out, dst, doff):
    """every frame's code and content; the sentinel everywhere else"""
    assert rc == (api.E_BLOCK if any(c < 0 for c in want_code) else 0)
    written = np.zeros(len(dst), dtype=bool)
    for i, label in enumerate(labels):
        assert int(out[i]) == want_code[i], (label, int(out[i]), want_code[i])
        if want_code[i] >= 0 or want_code[i] == api.E_CHECKSUM and want_plain[i] is not None:
            p = want_plain[i]
            got = dst[doff[i]:doff[i] + len(p)].tobytes()
            assert got == p, (label, next((k for k in range(len(p)) if got[k] != p[k]), None))
            written[doff[i]:doff[i] + len(p)] = True
    stray = np.nonzero(~written & (dst != SENTINEL))[0]
    assert len(stray) == 0, f"byte {int(stray[0])} written outside every content (frame destinations at {doff[:8]}...)"


def reference(blobs, caps):
    """(code, content) of every frame from the CPU window reference; content also after a content checksum mismatch"""
    codes, plains = [], []
    for b, c in zip(blobs, caps):
        code, p = frame.decode_result(b, c, b"", False)
        codes.append(code)
        plains.append(p)
    return codes, plains


# ---- the hand-built cases ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_window_cases_one_call(ctx, cases, device):
    with open(os.path.join(HERE, "golden", "frames", "window_checks.json")) as fh:
        checks = json.load(fh)["cases"]
    blobs = [c.blob for c in cases]
    caps = [len(c.plain) if c.plain is not None else c.block_max + 64 for c in cases]
    codes, plains = reference(blobs, caps)
    for c, code, p in zip(cases, codes, plains):        # the model, the reference and upstream agree
        if checks[c.id]["upstream"] == "accept":
            assert p == c.plain and code == len(p) and hashlib.sha256(p).hexdigest() == checks[c.id]["sha256"], c.id
        else:
            assert c.plain is None and code == api.E_BLOCK, c.id
    rc, out, dst, doff = decode(ctx, blobs, caps, device)
    check([c.id for c in cases], blobs, caps, codes, plains, rc, out, dst, doff)


def _limit_frame(pool, k, extra):
    """a window frame: a short block, then a match whose offset is the bytes decoded so far in this frame (+ extra)"""
    f = FrameBuilder(0, pool=pool)
    f.at = (97 * k) % 4096
    a, lit = 1 + k % 37, k % 5
    f.lits(a)
    f.seqs([(lit, 4 + k % 9, a + lit + extra)], 12, phantom=extra)
    return f.case(f"limit_{k}_{extra}")


def _good_frame(pool, k):
    f = FrameBuilder(0, pool=pool)
    f.at = (131 * k) % 4096
    f.lits(2 + k % 23).lits(1 + k % 7)
    n = len(f.content)
    f.seqs([(k % 3, 4 + k % 11, n - k % 2 + k % 3)], 12)
    return f.case(f"good_{k}")


def test_many_window_frames_per_cta(ctx, sm_count):
    """More window frames than 12 x SM: the 16-CTA decoder, each CTA taking several frames in turn.  Every other frame
    has, in its second block, a match whose offset equals the bytes decoded so far in that frame (accepted) or is one
    more, which would read the previous frame's output if the window were not reset at the frame start (rejected)."""
    pool = np.random.default_rng(11).integers(0, 256, 1 << 14, dtype=np.uint8).tobytes()
    n = 12 * sm_count + 301
    cases = [_good_frame(pool, k) if k % 2 == 0 else _limit_frame(pool, k, (k // 2) % 2) for k in range(n)]
    assert sum(c.plain is None for c in cases) > 12 * sm_count // 4
    blobs = [c.blob for c in cases]
    caps = [len(c.plain) if c.plain is not None else 4096 for c in cases]
    codes, plains = reference(blobs, caps)
    assert [p for p in plains] == [c.plain for c in cases]
    rc, out, dst, doff = decode(ctx, blobs, caps)
    check([c.id for c in cases], blobs, caps, codes, plains, rc, out, dst, doff)


# ---- many mixed frames in one call --------------------------------------------------------------------------------------

def _rehc(b):
    at = 14 if b[4] & 0x08 else 6
    b[at] = (frame.xxh32(bytes(b[4:at])) >> 8) & 0xFF
    return b


def _corrupt(blob, kind, rng):
    """one corruption of a valid frame (the kinds of the golden set, at a random block where it applies)"""
    b = bytearray(blob)
    flg = b[4]
    hl = 15 if flg & 0x08 else 7
    if kind == "hc":
        b[hl - 1] ^= 1 << int(rng.integers(0, 8))
    elif kind == "reserved":
        b[[4, 5, 5][int(rng.integers(0, 3))]] |= [0x02, 0x80, 0x01][int(rng.integers(0, 3))]
        _rehc(b)
    elif kind == "above_max":
        b[hl:hl + 4] = (frame.BD_SIZES[(b[5] >> 4) & 7] + 1).to_bytes(4, "little")
    elif kind == "trunc":
        b = b[:int(rng.integers(1, len(b)))]
    elif kind == "no_end":
        cc = 4 if flg & 0x04 else 0
        b = b[:len(b) - 4 - cc] + b[len(b) - cc:]
    elif kind == "trailing":
        b.append(int(rng.integers(0, 256)))
    elif kind == "size_plus" or kind == "size_minus":
        n = int.from_bytes(b[6:14], "little") + (1 if kind == "size_plus" else -1)
        b[6:14] = (n % (1 << 64)).to_bytes(8, "little")
        _rehc(b)
    elif kind == "block_csum" or kind == "content_csum":
        b[-1 if kind == "content_csum" else hl + 4 + (int.from_bytes(b[hl:hl + 4], "little") & 0x7FFFFFFF)] ^= 0x40
    return bytes(b)


def _mixed_frames(rng, ora):
    pool = rng.integers(0, 256, 1 << 18, dtype=np.uint8).tobytes()
    kinds = list(datagen.KINDS)
    blobs, labels = [], []
    # encoder-made frames: every class, block mode and flag set, stored blocks included
    for code, bm in CLASSES.items():
        for ind in (False, True):
            for fl in range(8):
                for j in range(6 if code < 6 else 2):
                    n = int(rng.integers(0, 3 * bm // (4 if code < 6 else 16)))
                    data = datagen.make(kinds[j % len(kinds)], int(rng.integers(0, 1 << 30)), n).tobytes() if n else b""
                    arrays = [data[k:k + bm] for k in range(0, len(data), bm)]
                    blobs.append(frame.encode(ora, arrays, code, 1, ind, bool(fl & 4), bool(fl & 2), bool(fl & 1)))
                    labels.append(f"enc_b{code}_{'ind' if ind else 'lnk'}_{fl}_{j}")
    # hand-built window frames with random short blocks, and stored blocks between them
    for k in range(3000):
        fl = k % 8
        f = FrameBuilder(0, bd_code=4 + (k % 5 == 0), block_checksum=bool(fl & 4), content_size=bool(fl & 2),
                         content_checksum=bool(fl & 1), pool=pool)
        f.at = int(rng.integers(0, 1 << 16))
        for _ in range(int(rng.integers(1, 6))):
            r = int(rng.integers(0, 10))
            if r == 0:
                f.stored(int(rng.integers(1, 600)))
            elif r == 1:
                f.empty()
            elif r < 4 or not f.content:
                f.lits(int(rng.integers(1, 300)))
            else:
                seqs, op = [], 0
                for _ in range(int(rng.integers(1, 8))):
                    lit = int(rng.integers(0, 40))
                    off = int(rng.integers(1, min(65535, len(f.content) + op + lit) + 1))
                    ml = int(rng.integers(4, 200))
                    seqs.append((lit, ml, off)); op += lit + ml
                f.seqs(seqs, 12)
        blobs.append(f.case("").blob)
        labels.append(f"win_{k}")
    # corruptions of both kinds of frames
    kinds_bad = ["hc", "reserved", "above_max", "trunc", "no_end", "trailing", "size_plus", "size_minus", "block_csum",
                 "content_csum"]
    valid = list(range(len(blobs)))
    for k in range(2000):
        kind = kinds_bad[k % len(kinds_bad)]
        i = valid[int(rng.integers(0, len(valid)))]
        b = blobs[i]
        need = {"size_plus": 0x08, "size_minus": 0x08, "block_csum": 0x10, "content_csum": 0x04}.get(kind, 0)
        if need and not b[4] & need or kind == "block_csum" and int.from_bytes(b[(15 if b[4] & 8 else 7):][:4], "little") == 0:
            continue
        blobs.append(_corrupt(b, kind, rng))
        labels.append(f"bad_{kind}_{labels[i]}")
    return blobs, labels


def test_mixed_frames_one_call(ctx, ref, cases):
    """About 5 000 shuffled frames in one call: every class, linked and independent, window and not, stored and
    compressed blocks, every flag set, the golden set's corruptions, the hand-built cases, and capacities equal to the
    content and one byte short.  Each frame gets the reference's verdict and bytes, and the same result alone."""
    rng = np.random.default_rng(2024)
    blobs, labels = _mixed_frames(rng, ref)
    blobs += [c.blob for c in cases]
    labels += [c.id for c in cases]
    with open(os.path.join(HERE, "golden", "frames", "frames.json")) as fh:
        for r in json.load(fh)["frames"]:
            with open(os.path.join(HERE, "golden", "frames", r["file"]), "rb") as g:
                blobs.append(g.read())
            labels.append(r["file"])
    full = [frame.decode_result(b, None, b"", False) for b in blobs]
    caps = []
    for k, (code, p) in enumerate(full):
        n = len(p) if p is not None else 256
        caps.append(max(n - (k % 3 == 0 and n > 0), 0))       # every third frame one byte short
    order = rng.permutation(len(blobs))
    blobs, labels, caps = [blobs[i] for i in order], [labels[i] for i in order], [caps[i] for i in order]
    assert len(blobs) > 4500
    codes, plains = reference(blobs, caps)
    assert {api.E_NOMEM, api.E_BLOCK, api.E_FRAME, api.E_CHECKSUM} <= set(codes) and sum(c >= 0 for c in codes) > 2000
    rc, out, dst, doff = decode(ctx, blobs, caps)
    check(labels, blobs, caps, codes, plains, rc, out, dst, doff)
    step = max(1, len(blobs) // 600)
    for i in range(0, len(blobs), step):                     # the same verdict alone
        rc1, out1, dst1, doff1 = decode(ctx, [blobs[i]], [caps[i]])
        assert int(out1[0]) == int(out[i]), labels[i]
        if out1[0] >= 0:
            assert dst1[doff1[0]:doff1[0] + out1[0]].tobytes() == dst[doff[i]:doff[i] + out[i]].tobytes(), labels[i]


# ---- read_frame -----------------------------------------------------------------------------------------------------------

def test_read_frame_golden_frames(ctx):
    """read_frame decodes every golden frame upstream accepts (the flushed ones: short linked blocks reached across by
    matches) from fragmented input, and refuses what the C ABI refuses"""
    with open(os.path.join(HERE, "golden", "frames", "frames.json")) as fh:
        recs = json.load(fh)["frames"]
    for r in recs:
        with open(os.path.join(HERE, "golden", "frames", r["file"]), "rb") as g:
            blob = g.read()
        if r["code"] != "ok":
            with pytest.raises(lz.LZ4Error):
                b"".join(lz.read_frame([blob], ctx=ctx))
            continue
        for size in ((7, 1000) if r["file"].startswith("flushed_") else (4096,)):
            got = b"".join(lz.read_frame([blob[k:k + size] for k in range(0, len(blob), size)], ctx=ctx))
            assert hashlib.sha256(got).hexdigest() == r["sha256"], r["file"]
        if r["file"].startswith("flushed_"):
            assert b"".join(lz.read_frame([blob], ctx=ctx, verify=False)) == got


def test_read_frame_window_cases(ctx, cases):
    for c in cases:
        if c.plain is None:
            with pytest.raises(lz.LZ4Error):
                b"".join(lz.read_frame([c.blob], ctx=ctx))
        elif len(c.plain) < (2 << 20):
            assert b"".join(lz.read_frame([c.blob], ctx=ctx)) == c.plain, c.id


@pytest.mark.parametrize("independent", [False, True], ids=["linked", "independent"])
def test_read_frame_dictionary_short_blocks(ctx, ref, independent):
    """A frame with a dictionary whose short blocks reach back into the dictionary and across each other: each block
    sees the dictionary followed by the content before it, last 64 KiB (LZ4F_decompress_usingDict)"""
    dic = datagen.make("text", 5, 70_000).tobytes()
    f = FrameBuilder(41, independent=independent, content_checksum=True, dictionary=dic)
    f.seqs([(3, 20, 1000), (0, 30, 65535)], 12)
    for k in range(6):
        n = len(f.content) - len(dic)
        back = 65535 if independent else min(65535, n + 60000)
        f.seqs([(k, 10 + k, back - 7 * k), (1, 8, 40 + k)], 12)
    c = f.case("dict_short")
    assert frame.decode(ref, c.blob, dic) == c.plain
    d = ctx.dictionary(dic)
    for size in (5, 1 << 20):
        assert b"".join(lz.read_frame([c.blob[k:k + size] for k in range(0, len(c.blob), size)], ctx=ctx,
                                      dictionary=d)) == c.plain


# ---- the encoder ----------------------------------------------------------------------------------------------------------

def _encode(ctx, arrays, bm, flags):
    src = np.frombuffer(b"".join(arrays) + b"\0", dtype=np.uint8).copy()
    ln = np.array([len(a) for a in arrays], dtype=np.int32)
    off = np.concatenate([[0], np.cumsum(ln.astype(np.int64))[:-1]]).astype(np.int64)
    rc, dst, doff, out = ctx.frame_compress_batch(src, off, ln, bm, flags, 1)
    assert rc == 0, ctx.last_error()
    return [dst[doff[i]:doff[i + 1]].tobytes() for i in range(len(arrays))]


def _check_blocks(ref, arrays, frames, bm, independent):
    for a, f in zip(arrays, frames):
        d, blocks, _ = frame.parse(f)
        split = [a[k:k + bm] for k in range(0, len(a), bm)]
        want = ref.compress_chunks(split, 1, block_size=NAMES[bm], linked=not independent) if split else []
        assert len(blocks) == len(split)
        for raw, w, (stored, data) in zip(split, want, blocks):
            assert stored == (len(w) - 4 >= len(raw)) and data == (raw if stored else w[4:])


@pytest.mark.parametrize("bm", sorted(NAMES))
def test_compress_block_split(ctx, ref, bm):
    """k x bm - 1, k x bm and k x bm + 1 bytes for k = 1..3, linked and independent: every block byte for byte"""
    sizes = [k * bm + e for k in (1, 2, 3) for e in (-1, 0, 1)]
    arrays = [datagen.make(("mixed", "text", "records")[i % 3], 900 + i, n).tobytes() for i, n in enumerate(sizes)]
    for independent in (False, True):
        flags = api.FRAME_CONTENT_CHECKSUM | api.FRAME_CONTENT_SIZE | (api.FRAME_INDEPENDENT if independent else 0)
        frames = _encode(ctx, arrays, bm, flags)
        _check_blocks(ref, arrays, frames, bm, independent)
        assert [frame.decode(ref, f) for f in frames] == arrays


@pytest.mark.parametrize("route", ["wide", "classic", "compact"])
def test_compress_routes_byte_parity(ctx, ref, sm_count, route):
    """one call per compressor route (at most SM linked frames, up to 12 x SM, more): every block byte for byte"""
    n = {"wide": sm_count, "classic": 6 * sm_count, "compact": 12 * sm_count + 77}[route]
    rng = np.random.default_rng({"wide": 1, "classic": 2, "compact": 3}[route])
    sizes = rng.integers(0, 150_000 if route == "wide" else 20_000, n)
    kinds = list(datagen.KINDS)
    arrays = [datagen.make(kinds[i % len(kinds)], 5000 + i, int(s)).tobytes() if s else b"" for i, s in enumerate(sizes)]
    frames = _encode(ctx, arrays, 65536, api.FRAME_BLOCK_CHECKSUM)
    _check_blocks(ref, arrays, frames, 65536, False)
    rc, out, dst, doff = decode(ctx, frames, [max(len(a), 1) for a in arrays])
    assert rc == 0 and all(dst[doff[i]:doff[i] + len(a)].tobytes() == a for i, a in enumerate(arrays))
