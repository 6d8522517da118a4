"""LZ4 frames on the device (b200lz4_frame_compress_batch / b200lz4_frame_decompress_batch): upstream's golden frames,
valid and corrupted, in one call; many frames and one large frame; the encoder against the checker's blocks over every
block maximum, block mode, flag combination, data kind and acceleration; linked frames whose short blocks are reached
across by matches (window mode)."""
import hashlib
import json
import os

import numpy as np
import pytest

import streamly_lz4_b200 as lz
from streamly_lz4_b200 import api, datagen

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FRAMES = os.path.join(HERE, "golden", "frames")
CODE = {"ok": None, "frame": api.E_FRAME, "checksum": api.E_CHECKSUM, "block": api.E_BLOCK}
NAMES = {65536: "BlockMax64KB", 262144: "BlockMax256KB", 1 << 20: "BlockMax1MB", 4 << 20: "BlockMax4MB"}
FLAG_SETS = [f1 | f2 | f3 for f1 in (0, api.FRAME_BLOCK_CHECKSUM) for f2 in (0, api.FRAME_CONTENT_SIZE)
             for f3 in (0, api.FRAME_CONTENT_CHECKSUM)]


@pytest.fixture(scope="module")
def ctx():
    c = lz.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def oracle():
    from oracle.oracle import Oracle
    return Oracle("auto")


def content(kind, seed, n):
    return datagen.make(kind, seed, n).tobytes() if n else b""


def pack(blobs):
    off = np.zeros(len(blobs), dtype=np.int64)
    at = 0
    for i, b in enumerate(blobs):
        off[i] = at
        at += len(b)
    buf = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy()
    return buf, off, np.array([len(b) for b in blobs], dtype=np.int32)


def decode(ctx, blobs, caps, device=False):
    """(rc, out_len, [content or None]) of one frame_decompress_batch call; destination pre-filled with 0xA5"""
    src, off, ln = pack(blobs)
    caps = np.asarray(caps, dtype=np.int32)
    doff = np.concatenate([[0], np.cumsum(caps.astype(np.int64))[:-1]]).astype(np.int64)
    dst = np.full(int(caps.sum()) + 1, 0xA5, dtype=np.uint8)
    if device:
        import torch
        t = lambda a: torch.from_numpy(a).cuda()
        d_dst = t(dst)
        rc, out = ctx.frame_decompress_batch(t(src), t(off), t(ln), d_dst, t(doff), t(caps))
        dst = d_dst.cpu().numpy()
    else:
        rc, out = ctx.frame_decompress_batch(src, off, ln, dst, doff, caps)
    return rc, out, dst, doff


def golden():
    with open(os.path.join(FRAMES, "frames.json")) as fh:
        recs = json.load(fh)["frames"]
    blobs = []
    for r in recs:
        with open(os.path.join(FRAMES, r["file"]), "rb") as fh:
            blobs.append(fh.read())
    return recs, blobs


def check_golden(recs, out, dst, doff, caps):
    for i, r in enumerate(recs):
        want = CODE[r["code"]]
        if want is None:
            assert out[i] == r["length"], r["file"]
            got = dst[doff[i]:doff[i] + r["length"]].tobytes()
            assert hashlib.sha256(got).hexdigest() == r["sha256"], r["file"]
        else:
            assert out[i] == want, (r["file"], int(out[i]), want)
            if want != api.E_CHECKSUM or r["file"] != "bad_content_checksum.lz4":
                assert (dst[doff[i]:doff[i] + caps[i]] == 0xA5).all(), r["file"]      # a failing frame writes nothing


def test_golden_frames_one_call(ctx):
    recs, blobs = golden()
    caps = [max(r["length"], 1) for r in recs]
    rc, out, dst, doff = decode(ctx, blobs, caps)
    assert rc == api.E_BLOCK, ctx.last_error()
    check_golden(recs, out, dst, doff, caps)
    rc2, out2, dst2, _ = decode(ctx, blobs, caps, device=True)
    assert rc2 == rc and (out2 == out).all() and (dst2 == dst).all()


def test_golden_capacity_short_by_one(ctx):
    recs, blobs = golden()
    pick = [i for i, r in enumerate(recs) if r["code"] == "ok" and r["length"] > 0][:6]
    rc, out, _, _ = decode(ctx, [blobs[i] for i in pick], [recs[i]["length"] - 1 for i in pick])
    assert rc == api.E_BLOCK and (out == api.E_NOMEM).all()
    assert lz.api.frame_info(blobs[pick[0]])[0] in NAMES


def compress(ctx, arrays, block_max, flags, accel, device=False):
    src, off, ln = pack(arrays)
    if device:
        import torch
        t = lambda a: torch.from_numpy(a).cuda()
        cap = sum(api.frame_bound(len(a), block_max, flags) for a in arrays) + 1
        d_dst = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        rc, _, doff, out = ctx.frame_compress_batch(t(src), t(off), t(ln), block_max, flags, accel, dst=d_dst)
        dst = d_dst.cpu().numpy()
    else:
        rc, dst, doff, out = ctx.frame_compress_batch(src, off, ln, block_max, flags, accel)
    assert rc == 0, ctx.last_error()
    return [dst[doff[i]:doff[i + 1]].tobytes() for i in range(len(arrays))], out


@pytest.mark.parametrize("block_max", sorted(NAMES))
@pytest.mark.parametrize("independent", [False, True])
def test_compress_matrix(ctx, oracle, block_max, independent):
    from oracle import frame
    kinds = list(datagen.KINDS)
    for fi, fl in enumerate(FLAG_SETS):
        flags = fl | (api.FRAME_INDEPENDENT if independent else 0)
        accel = (1, 12, 65537)[fi % 3]
        sizes = [0, 1, block_max, block_max + 1] + ([3 << 20] if fi % 4 == 0 else [])
        arrays = [content(k, 1000 * fi + 10 * j + si, n) for si, n in enumerate(sizes) for j, k in enumerate(kinds)
                  if n < block_max or j % 2 == fi % 2]
        frames, out = compress(ctx, arrays, block_max, flags, accel)
        if fi in (0, 7):
            dframes, dout = compress(ctx, arrays, block_max, flags, accel, device=True)
            assert dframes == frames and (dout == out).all()
        for a, f, n in zip(arrays, frames, out):
            assert n == len(f) <= api.frame_bound(len(a), block_max, flags)
            assert frame.decode(oracle, f) == a
            d, blocks, _ = frame.parse(f)
            assert d["independent"] == independent and (d["content_size"] is not None) == bool(flags & api.FRAME_CONTENT_SIZE)
            split = [a[k:k + block_max] for k in range(0, len(a), block_max)]
            ref = oracle.compress_chunks(split, accel, block_size=NAMES[block_max], linked=not independent) if split else []
            assert len(blocks) == len(split)
            for raw, r, (stored, data) in zip(split, ref, blocks):
                payload = r[4:]
                assert stored == (len(payload) >= len(raw))
                assert data == (raw if stored else payload)
        rc, back, dst, doff = decode(ctx, frames, [max(len(a), 1) for a in arrays])
        assert rc == 0 and list(back) == [len(a) for a in arrays]
        assert all(dst[doff[i]:doff[i] + len(a)].tobytes() == a for i, a in enumerate(arrays))


def test_many_small_frames_and_one_large(ctx):
    rng = np.random.default_rng(5)
    sizes = rng.integers(0, 5000, 4096)
    arrays = [content(("text", "records", "mixed", "random")[i % 4], i, int(n)) for i, n in enumerate(sizes)]
    for flags in (api.FRAME_CONTENT_CHECKSUM | api.FRAME_INDEPENDENT, api.FRAME_BLOCK_CHECKSUM | api.FRAME_CONTENT_SIZE):
        frames, _ = compress(ctx, arrays, 65536, flags, 1)
        rc, back, dst, doff = decode(ctx, frames, [max(len(a), 1) for a in arrays])
        assert rc == 0 and all(dst[doff[i]:doff[i] + len(a)].tobytes() == a for i, a in enumerate(arrays))
    big = content("mixed", 77, 16 << 20)
    for flags in (api.FRAME_CONTENT_CHECKSUM, api.FRAME_INDEPENDENT | api.FRAME_BLOCK_CHECKSUM):
        frames, _ = compress(ctx, [big], 65536, flags, 1)
        rc, back, dst, _ = decode(ctx, frames, [len(big)])
        assert rc == 0 and back[0] == len(big) and dst[:len(big)].tobytes() == big


# ---- window mode: hand-built linked frames with short blocks ----

def token_block(seqs, tail):
    """An LZ4 block: sequences (literals, offset, match length) then the literal-only tail"""
    out = bytearray()

    def length(n):
        while n >= 255:
            out.append(255); n -= 255
        out.append(n)
    for lits, off, ml in seqs:
        out.append((min(len(lits), 15) << 4) | min(ml - 4, 15))
        if len(lits) >= 15:
            length(len(lits) - 15)
        out += lits
        out += off.to_bytes(2, "little")
        if ml - 4 >= 15:
            length(ml - 4 - 15)
    out.append(min(len(tail), 15) << 4)
    if len(tail) >= 15:
        length(len(tail) - 15)
    out += tail
    return bytes(out)


def window_frame(block_sizes, offsets, seed):
    """Linked 64 KiB-max frame: literal-only blocks of the given sizes, then a block of matches at the given offsets
    (each reaching back across the short blocks).  Returns (frame, content as a stock decoder builds it)."""
    from oracle import frame
    rnd = content("random", seed, sum(block_sizes) + 64 * len(offsets) + 64)
    at, blocks, plain = 0, [], bytearray()
    for n in block_sizes:
        blocks.append(token_block([], rnd[at:at + n])); plain += rnd[at:at + n]; at += n
    seqs = []
    for off in offsets:
        lits = rnd[at:at + 3]; at += 3
        seqs.append((lits, off, 20))
    tail = rnd[at:at + 16]
    blk = token_block(seqs, tail)
    blocks.append(blk)
    for lits, off, ml in seqs:
        plain += lits
        for _ in range(ml):
            plain.append(plain[-off] if off <= len(plain) else 0)     # (invalid offsets: rejected, content unused)
    plain += tail
    body = b"".join(len(b).to_bytes(4, "little") + b for b in blocks)
    return frame.header(4, independent=False) + body + b"\0\0\0\0", bytes(plain)


def upstream_decode(blob, n):
    import ctypes.util
    path = ctypes.util.find_library("lz4")
    if not path:
        return None
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    from frame_golden import LZ4F
    ok, got = LZ4F(path).decompress(blob, n)
    return got if ok else False


def test_window_mode(ctx):
    cases = [([1000, 2000], [1, 30, 2500, 3000]),
             ([20000, 20000, 20000, 9000], [65535, 60000, 40001, 20000, 1, 7]),
             ([5000, 100, 100, 100, 30000], [35300, 35299, 30150, 100, 2]),
             ([40000, 30000], [65535, 30001])]
    blobs, plains = [], []
    for k, (sizes, offs) in enumerate(cases):
        offs = [o for o in offs if o <= min(sum(sizes), 65535)]
        blob, plain = window_frame(sizes, offs, 300 + k)
        blobs.append(blob); plains.append(plain)
        up = upstream_decode(blob, len(plain))
        if up is not None:
            assert up == plain
    # offsets one past the bytes decoded so far (the blocks and the 3 literals in front of the match): rejected
    bad = [window_frame([1000, 2000], [3004], 400)[0], window_frame([10, 20, 30], [64], 401)[0]]
    for b in bad:
        assert upstream_decode(b, 4096) in (None, False)
    rc, out, dst, doff = decode(ctx, blobs + bad, [len(p) for p in plains] + [4096, 4096])
    assert rc == api.E_BLOCK
    for i, p in enumerate(plains):
        assert out[i] == len(p) and dst[doff[i]:doff[i] + len(p)].tobytes() == p, i
    assert list(out[len(plains):]) == [api.E_BLOCK, api.E_BLOCK]
