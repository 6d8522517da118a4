"""Golden LZ4 frames written by upstream LZ4F (the system liblz4, 1.9.x), with upstream's accept/reject verdicts.

  python tests/golden/frame_golden.py [LIB]         -> tests/golden/frames/*.lz4 + tests/golden/frames/frames.json
  python tests/golden/frame_golden.py window [LIB]  -> tests/golden/frames/window_checks.json: upstream's verdict and
                                                       content digest for every hand-built case of window_cases.py

Every frame's content is datagen(kind, seed)[:length]; frames.json holds, per file, the content's SHA-256, upstream's
verdict (LZ4F_decompress over the whole range: accept = no error, frame complete, every byte consumed) and the code
b200lz4_frame_decompress_batch must report ("ok", or the B200LZ4_E_* class of the corruption: frame, checksum, block).
Valid frames cover the four block maxima, independent and linked blocks, every combination of block checksum, content
size and content checksum, stored blocks (incompressible data and LZ4F_uncompressedUpdate), linked frames flushed after
small updates (blocks shorter than 64 KiB referenced across several blocks), empty and 1-byte content, and content of
exactly the block maximum and one byte more.  The corrupted copies are derived from a few of them.
"""
from __future__ import annotations

import ctypes
import ctypes.util
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "frames")
sys.path.insert(0, ROOT)

BMAX = {4: 64 << 10, 5: 256 << 10, 6: 1 << 20, 7: 4 << 20}


class _FrameInfo(ctypes.Structure):
    _fields_ = [("blockSizeID", ctypes.c_int), ("blockMode", ctypes.c_int), ("contentChecksumFlag", ctypes.c_int),
                ("frameType", ctypes.c_int), ("contentSize", ctypes.c_ulonglong), ("dictID", ctypes.c_uint),
                ("blockChecksumFlag", ctypes.c_int)]


class _Prefs(ctypes.Structure):
    _fields_ = [("frameInfo", _FrameInfo), ("compressionLevel", ctypes.c_int), ("autoFlush", ctypes.c_uint),
                ("favorDecSpeed", ctypes.c_uint), ("reserved", ctypes.c_uint * 3)]


class LZ4F:
    def __init__(self, path: str):
        self.lib = lib = ctypes.CDLL(path)
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        lib.LZ4F_isError.argtypes = [sz]
        lib.LZ4F_isError.restype = ctypes.c_uint
        lib.LZ4F_compressFrameBound.argtypes = [sz, vp]
        lib.LZ4F_compressFrameBound.restype = sz
        lib.LZ4F_compressFrame.argtypes = [vp, sz, vp, sz, vp]
        lib.LZ4F_compressFrame.restype = sz
        lib.LZ4F_createCompressionContext.argtypes = [ctypes.POINTER(vp), ctypes.c_uint]
        lib.LZ4F_freeCompressionContext.argtypes = [vp]
        lib.LZ4F_compressBound.argtypes = [sz, vp]
        lib.LZ4F_compressBound.restype = sz
        for name in ("LZ4F_compressBegin",):
            getattr(lib, name).argtypes = [vp, vp, sz, vp]
            getattr(lib, name).restype = sz
        for name in ("LZ4F_compressUpdate", "LZ4F_uncompressedUpdate"):
            getattr(lib, name).argtypes = [vp, vp, sz, vp, sz, vp]
            getattr(lib, name).restype = sz
        for name in ("LZ4F_flush", "LZ4F_compressEnd"):
            getattr(lib, name).argtypes = [vp, vp, sz, vp]
            getattr(lib, name).restype = sz
        lib.LZ4F_createDecompressionContext.argtypes = [ctypes.POINTER(vp), ctypes.c_uint]
        lib.LZ4F_freeDecompressionContext.argtypes = [vp]
        lib.LZ4F_decompress.argtypes = [vp, vp, ctypes.POINTER(sz), vp, ctypes.POINTER(sz), vp]
        lib.LZ4F_decompress.restype = sz

    @staticmethod
    def prefs(code, independent, bc, cs, cc, n, dict_id=0, auto_flush=0):
        p = _Prefs()
        p.frameInfo.blockSizeID = code
        p.frameInfo.blockMode = 1 if independent else 0
        p.frameInfo.contentChecksumFlag = 1 if cc else 0
        p.frameInfo.contentSize = n if cs else 0
        p.frameInfo.dictID = dict_id
        p.frameInfo.blockChecksumFlag = 1 if bc else 0
        p.autoFlush = auto_flush
        return p

    def compress_frame(self, data: bytes, p: _Prefs) -> bytes:
        cap = self.lib.LZ4F_compressFrameBound(len(data), ctypes.byref(p))
        dst = ctypes.create_string_buffer(cap)
        r = self.lib.LZ4F_compressFrame(dst, cap, data, len(data), ctypes.byref(p))
        assert not self.lib.LZ4F_isError(r)
        return dst.raw[:r]

    def compress_pieces(self, pieces, p: _Prefs, flush: bool, stored: bool = False) -> bytes:
        """compressBegin, one update per piece (LZ4F_uncompressedUpdate if stored) followed by LZ4F_flush if flush, End"""
        ctx = ctypes.c_void_p()
        assert self.lib.LZ4F_createCompressionContext(ctypes.byref(ctx), 100) == 0
        cap = 64 + self.lib.LZ4F_compressBound(max([len(x) for x in pieces] + [1]), ctypes.byref(p)) + 4 * (1 << 22)
        dst = ctypes.create_string_buffer(cap)
        out = []

        def take(r):
            assert not self.lib.LZ4F_isError(r), r
            out.append(dst.raw[:r])
        take(self.lib.LZ4F_compressBegin(ctx, dst, cap, ctypes.byref(p)))
        for x in pieces:
            upd = self.lib.LZ4F_uncompressedUpdate if stored else self.lib.LZ4F_compressUpdate
            take(upd(ctx, dst, cap, x, len(x), None))
            if flush:
                take(self.lib.LZ4F_flush(ctx, dst, cap, None))
        take(self.lib.LZ4F_compressEnd(ctx, dst, cap, None))
        self.lib.LZ4F_freeCompressionContext(ctx)
        return b"".join(out)

    def decompress(self, blob: bytes, expect: int):
        """(accepted, content) of LZ4F_decompress over the whole range"""
        ctx = ctypes.c_void_p()
        assert self.lib.LZ4F_createDecompressionContext(ctypes.byref(ctx), 100) == 0
        cap = expect + (8 << 20)
        dst = ctypes.create_string_buffer(cap)
        src = ctypes.create_string_buffer(blob, len(blob) + 1)
        got, at, ok, hint = [], 0, True, 1
        while True:
            dn, sn = ctypes.c_size_t(cap), ctypes.c_size_t(len(blob) - at)
            hint = self.lib.LZ4F_decompress(ctx, dst, ctypes.byref(dn), ctypes.byref(src, at), ctypes.byref(sn), None)
            if self.lib.LZ4F_isError(hint):
                ok = False
                break
            got.append(dst.raw[:dn.value])
            at += sn.value
            if hint == 0 or (sn.value == 0 and dn.value == 0):
                break
        self.lib.LZ4F_freeDecompressionContext(ctx)
        accepted = ok and hint == 0 and at == len(blob)
        return accepted, b"".join(got)


def content(kind: str, seed: int, length: int) -> bytes:
    from streamly_lz4_b200 import datagen
    return datagen.make(kind, seed, length).tobytes() if length else b""


def xxh32_short(data: bytes) -> int:
    from streamly_lz4_b200.api import _xxh32_short
    return _xxh32_short(data)


def header_code(blob: bytes) -> str:
    """The class a frame reader reports for this header: frame (structure) or checksum (HC), "ok" if it passes"""
    if len(blob) < 7 or int.from_bytes(blob[:4], "little") != 0x184D2204:
        return "frame"
    flg, bd = blob[4], blob[5]
    if (flg >> 6) != 1 or flg & 0x02 or bd & 0x8F or flg & 0x01 or ((bd >> 4) & 7) < 4:
        return "frame"
    at = 14 if flg & 0x08 else 6
    if len(blob) <= at:
        return "frame"
    return "ok" if blob[at] == (xxh32_short(blob[4:at]) >> 8) & 0xFF else "checksum"


def rehc(blob: bytearray) -> bytearray:
    at = 14 if blob[4] & 0x08 else 6
    blob[at] = (xxh32_short(bytes(blob[4:at])) >> 8) & 0xFF
    return blob


def boundaries(blob: bytes):
    """offsets where a frame's structures end: header fields, each block size / data / checksum, end mark"""
    flg = blob[4]
    at = 14 if flg & 0x08 else 6
    out = [4, 5, 6, at, at + 1]
    at += 1
    while True:
        size = int.from_bytes(blob[at:at + 4], "little")
        at += 4
        out.append(at)
        if size & 0x7FFFFFFF == 0:
            break
        at += size & 0x7FFFFFFF
        out.append(at)
        if flg & 0x10:
            at += 4
            out.append(at)
    return sorted(set(x for x in out if 0 < x < len(blob))) + [len(blob) - 1]


def main(path: str) -> None:
    up = LZ4F(path)
    os.makedirs(OUT, exist_ok=True)
    for f in os.listdir(OUT):
        os.remove(os.path.join(OUT, f))
    records = []

    def add(name, blob, kind, seed, length, code="ok"):
        data = content(kind, seed, length)
        acc, got = up.decompress(blob, length)
        if code == "ok":
            assert acc and got == data, name
        with open(os.path.join(OUT, name + ".lz4"), "wb") as fh:
            fh.write(blob)
        records.append({"file": name + ".lz4", "kind": kind, "seed": seed, "length": length,
                        "sha256": hashlib.sha256(data).hexdigest(), "upstream": "accept" if acc else "reject", "code": code})

    # every block maximum x independent / linked x block checksum x content size x content checksum
    seed = 100
    for code, (kind, length) in {4: ("records", 100_000), 5: ("zero", (256 << 10) + 1), 6: ("zero", (1 << 20) + 1),
                                 7: ("zero", (4 << 20) + 1)}.items():
        for ind in (False, True):
            for combo in (range(8) if code < 7 else (0, 7)):
                bc, cs, cc = bool(combo & 4), bool(combo & 2), bool(combo & 1)
                data = content(kind, seed, length)
                blob = up.compress_frame(data, LZ4F.prefs(code, ind, bc, cs, cc, len(data)))
                add(f"b{code}_{'ind' if ind else 'lnk'}_{combo}", blob, kind, seed, length)
                seed += 1
    # empty and 1-byte content, exactly the block maximum
    for code in (4, 7):
        for n in (0, 1, BMAX[code]):
            for ind in (False, True):
                kind = "zero" if n > 1 else "text"
                data = content(kind, seed, n)
                blob = up.compress_frame(data, LZ4F.prefs(code, ind, True, True, True, n))
                add(f"n{n}_b{code}_{'ind' if ind else 'lnk'}", blob, kind, seed, n)
                seed += 1
    # stored blocks: incompressible data, and LZ4F_uncompressedUpdate (independent blocks only in 1.9.4)
    for ind in (False, True):
        data = content("random", seed, 70_000)
        add(f"stored_random_{'ind' if ind else 'lnk'}", up.compress_frame(data, LZ4F.prefs(4, ind, True, True, True, len(data))),
            "random", seed, len(data))
        seed += 1
    data = content("text", seed, 30_000)
    blob = up.compress_pieces([data[:20_000], data[20_000:]], LZ4F.prefs(4, True, True, False, True, 0), flush=False, stored=True)
    add("stored_update_ind", blob, "text", seed, len(data))
    seed += 1
    # linked frames flushed after small updates: short blocks whose matches reach across several earlier blocks
    for piece, count, kind in ((3000, 10, "text"), (700, 40, "records"), (20_000, 4, "records")):
        data = content(kind, seed, piece * count)
        blob = up.compress_pieces([data[k:k + piece] for k in range(0, len(data), piece)],
                                  LZ4F.prefs(4, False, True, True, True, len(data)), flush=True)
        add(f"flushed_{piece}x{count}", blob, kind, seed, len(data))
        seed += 1

    # corrupted copies
    kind, length = "zero", 140_000
    base_seed = seed
    data = content(kind, base_seed, length)
    full = up.compress_frame(data, LZ4F.prefs(4, False, True, True, True, length))
    for byte in (0, 4, 5):
        for bit in range(8):
            b = bytearray(full)
            b[byte] ^= 1 << bit
            add(f"bad_hdr_{byte}_{bit}", bytes(b), kind, base_seed, length, header_code(bytes(b)))
    b = bytearray(full)
    b[14] ^= 0x5A
    add("bad_hc", bytes(b), kind, base_seed, length, "checksum")
    for name, at, bit in (("bad_reserved_flg", 4, 0x02), ("bad_reserved_bd7", 5, 0x80), ("bad_reserved_bd0", 5, 0x01)):
        b = bytearray(full)
        b[at] |= bit
        add(name, bytes(rehc(b)), kind, base_seed, length, "frame")
    b = bytearray(full)
    b[6:14] = (length + 1).to_bytes(8, "little")
    add("bad_content_size", bytes(rehc(b)), kind, base_seed, length, "frame")
    first = 15
    size = int.from_bytes(full[first:first + 4], "little") & 0x7FFFFFFF
    b = bytearray(full)
    b[first:first + 4] = ((64 << 10) + 1).to_bytes(4, "little")
    add("bad_block_above_max", bytes(b), kind, base_seed, length, "frame")
    b = bytearray(full)
    b[first + 4 + size] ^= 0x01
    add("bad_block_checksum", bytes(b), kind, base_seed, length, "checksum")
    b = bytearray(full)
    b[-1] ^= 0x80
    add("bad_content_checksum", bytes(b), kind, base_seed, length, "checksum")
    for k, cut in enumerate(boundaries(full)):
        add(f"bad_trunc_{k:02d}_{cut}", full[:cut], kind, base_seed, length, "frame")
    plain = up.compress_frame(data, LZ4F.prefs(4, False, False, False, False, length))
    add("bad_no_end_mark", plain[:-4], kind, base_seed, length, "frame")
    # a compressed block cut by one byte (no checksums): the decoder itself rejects it
    size = int.from_bytes(plain[7:11], "little")
    assert not size >> 31
    b = bytearray(plain[:11 + size - 1] + plain[11 + size:])
    b[7:11] = (size - 1).to_bytes(4, "little")
    add("bad_block_cut", bytes(b), kind, base_seed, length, "block")
    add("bad_dict_id", up.compress_frame(data, LZ4F.prefs(4, False, False, False, False, 0, dict_id=7)), kind, base_seed, length,
        "frame")
    with open(os.path.join(OUT, "frames.json"), "w") as fh:
        json.dump({"generator": "tests/golden/frame_golden.py", "library": os.path.basename(path), "frames": records}, fh, indent=0)
    total = sum(os.path.getsize(os.path.join(OUT, r["file"])) for r in records)
    print(f"{len(records)} frames, {total} bytes")


def window(path: str) -> None:
    """Upstream's verdict on the hand-built window cases (the frames are rebuilt from window_cases.py, not stored)"""
    sys.path.insert(0, HERE)
    import window_cases
    up = LZ4F(path)
    checks = {}
    for c in window_cases.cases():
        acc, got = up.decompress(c.blob, len(c.plain) if c.plain is not None else c.block_max)
        if c.plain is not None:
            assert acc and got == c.plain, c.id
        checks[c.id] = {"upstream": "accept" if acc else "reject", "sha256": hashlib.sha256(got).hexdigest() if acc else None}
    v = up.lib.LZ4_versionNumber()
    with open(os.path.join(OUT, "window_checks.json"), "w") as fh:
        json.dump({"generator": "tests/golden/frame_golden.py window", "library": f"{os.path.basename(path)} "
                   f"({v // 10000}.{v // 100 % 100}.{v % 100})", "cases": checks}, fh, indent=0)
    print(f"{len(checks)} window cases, {sum(r['upstream'] == 'reject' for r in checks.values())} rejected")


if __name__ == "__main__":
    args = sys.argv[1:]
    sub = args.pop(0) if args and args[0] == "window" else None
    lib = args[0] if args else ctypes.util.find_library("lz4")
    assert lib, "no liblz4 found: name one, frame_golden.py [window] /path/to/liblz4.so"
    (window if sub else main)(lib)
