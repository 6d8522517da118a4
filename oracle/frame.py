"""LZ4 FRAME format (v1.6.x) restated for the checker (TEST INFRASTRUCTURE ONLY).

The reference's frame support is a stub (src/Streamly/Internal/LZ4.hs:590-651: magic, FLG, BD, any header-checksum byte;
every optional feature dies with "not yet supported"; benchmark/Main.hs:92-118 writes a header with HC = 0).  The frame
library of LZ4 is not part of the reference tree, so what follows restates the published frame specification
(lz4_Frame_format.md), with the block codec taken from the oracle:

    magic 0x184D2204 (LE) | FLG | BD | [content size LE64] | [dict id LE32] | HC
        FLG: bits 7-6 version = 01, bit 5 block independence, bit 4 block checksum, bit 3 content size,
             bit 2 content checksum, bit 1 reserved (0), bit 0 dict id
        BD : bits 6-4 block maximum (4: 64 KiB, 5: 256 KiB, 6: 1 MiB, 7: 4 MiB), other bits reserved (0)
        HC : (XXH32(FLG .. last descriptor byte, seed 0) >> 8) & 0xFF
    blocks: [size LE32: bit 31 set = stored uncompressed][data][XXH32(data) LE32 iff block checksum]
    end mark 0x00000000 | [XXH32(whole content) LE32 iff content checksum]
    linked blocks (independence flag clear) may reference the previous 64 KiB of DECODED data, across block boundaries.

Known answers pinned in tests/test_oracle.py: descriptors 60 40 -> HC 82, 64 40 -> A7, 64 70 -> B9 (the headers the
stock `lz4` tool writes for -B4 / -B4 --content-checksum / -B7 --content-checksum streams).
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

MAGIC = 0x184D2204
BD_SIZES = {4: 64 << 10, 5: 256 << 10, 6: 1 << 20, 7: 4 << 20}

E_NOMEM, E_BLOCK, E_FRAME, E_CHECKSUM = -3, -4, -5, -6      # B200LZ4_E_* (include/b200lz4.h)
WINDOW = 65536

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


class _DStream(ctypes.Structure):         # struct ora_dstream (lz4_oracle.c)
    _fields_ = [("prev_out", ctypes.c_void_p), ("prev_len", ctypes.c_size_t)]


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(os.path.join(_HERE, "liboracle.so"))
        lib.ora_xxh32.restype = ctypes.c_uint32
        lib.ora_xxh32.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32]
        lib.ora_dstream_create.restype = ctypes.POINTER(_DStream)
        lib.ora_dstream_free.argtypes = [ctypes.POINTER(_DStream)]
        lib.ora_decompress_continue.argtypes = [ctypes.POINTER(_DStream), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                                ctypes.c_int]
        lib.ora_decompress_continue.restype = ctypes.c_int
        _lib = lib
    return _lib


def xxh32(data: bytes, seed: int = 0) -> int:
    return int(_load().ora_xxh32(bytes(data), len(data), seed))


def decode_block(payload: bytes, cap: int, dictionary: bytes = b"") -> Optional[bytes]:
    """LZ4_decompress_safe_usingDict(payload, cap, dictionary) through the restatement (a decode record whose previous
    output is `dictionary`, as dict_golden.Port sets it up): the block's output, or None when the block is rejected."""
    lib = _load()
    dbuf = ctypes.create_string_buffer(bytes(dictionary), len(dictionary) + 1)
    src = ctypes.create_string_buffer(bytes(payload), len(payload) + 1)
    dst = ctypes.create_string_buffer(cap + 1)
    s = lib.ora_dstream_create()
    s.contents.prev_out = ctypes.addressof(dbuf) if dictionary else None
    s.contents.prev_len = len(dictionary)
    r = lib.ora_decompress_continue(s, src, dst, len(payload), cap)
    lib.ora_dstream_free(s)
    return None if r < 0 else dst.raw[:r]


def header(bd_code: int, independent: bool = False, block_checksum: bool = False, content_size: Optional[int] = None,
           content_checksum: bool = False) -> bytes:
    flg = 0x40 | (0x20 if independent else 0) | (0x10 if block_checksum else 0) | (0x08 if content_size is not None else 0) \
        | (0x04 if content_checksum else 0)
    desc = bytes([flg, bd_code << 4]) + (content_size.to_bytes(8, "little") if content_size is not None else b"")
    return MAGIC.to_bytes(4, "little") + desc + bytes([(xxh32(desc) >> 8) & 0xFF])


def encode(oracle, arrays: Sequence[bytes], bd_code: int, accel: int = 1, independent: bool = False, block_checksum: bool = False,
           content_size: bool = False, content_checksum: bool = False, store_incompressible: bool = True) -> bytes:
    """A frame as a stock writer would produce it from `arrays` (each at most the block maximum): oracle blocks, stored
    uncompressed when compression does not shrink them (what LZ4F does), checksums as flagged."""
    assert all(len(a) <= BD_SIZES[bd_code] for a in arrays)
    framed = oracle.compress_chunks(list(arrays), accel, block_size={4: "BlockMax64KB", 5: "BlockMax256KB", 6: "BlockMax1MB", 7: "BlockMax4MB"}[bd_code],
                                    linked=not independent)
    out = [header(bd_code, independent, block_checksum, sum(len(a) for a in arrays) if content_size else None, content_checksum)]
    for a, f in zip(arrays, framed):
        payload = f[4:]
        if store_incompressible and len(payload) >= len(a):
            data, size = bytes(a), len(a) | 0x80000000
        else:
            data, size = payload, len(payload)
        out.append(size.to_bytes(4, "little") + data)
        if block_checksum:
            out.append(xxh32(data).to_bytes(4, "little"))
    out.append(b"\0\0\0\0")
    if content_checksum:
        out.append(xxh32(b"".join(bytes(a) for a in arrays)).to_bytes(4, "little"))
    return b"".join(out)


def parse(blob: bytes) -> Tuple[dict, List[Tuple[bool, bytes]], Optional[int]]:
    """Split a frame into (descriptor, [(stored_uncompressed, block data)], content checksum); verifies HC, block
    checksums, reserved bits; raises ValueError like a stock reader would."""
    if int.from_bytes(blob[0:4], "little") != MAGIC:
        raise ValueError("bad magic")
    flg, bd = blob[4], blob[5]
    if (flg >> 6) != 1:
        raise ValueError("version is not 01")
    if flg & 0x02 or bd & 0x8F:
        raise ValueError("reserved bits set")
    code = (bd >> 4) & 7
    if code not in BD_SIZES:
        raise ValueError("unknown block maximum")
    at = 6
    d = {"independent": bool(flg & 0x20), "block_checksum": bool(flg & 0x10), "content_checksum": bool(flg & 0x04),
         "content_size": None, "dict_id": None, "bd_code": code, "block_max": BD_SIZES[code]}
    if flg & 0x08:
        d["content_size"] = int.from_bytes(blob[at:at + 8], "little"); at += 8
    if flg & 0x01:
        d["dict_id"] = int.from_bytes(blob[at:at + 4], "little"); at += 4
    if blob[at] != (xxh32(blob[4:at]) >> 8) & 0xFF:
        raise ValueError("header checksum mismatch")
    at += 1
    blocks = []
    while True:
        size = int.from_bytes(blob[at:at + 4], "little"); at += 4
        if size == 0:
            break
        stored, n = bool(size >> 31), size & 0x7FFFFFFF
        if n > d["block_max"]:
            raise ValueError("block larger than the block maximum")
        data = blob[at:at + n]; at += n
        if len(data) != n:
            raise ValueError("truncated block")
        if d["block_checksum"]:
            if int.from_bytes(blob[at:at + 4], "little") != xxh32(data):
                raise ValueError("block checksum mismatch")
            at += 4
        blocks.append((stored, data))
    cc = None
    if d["content_checksum"]:
        cc = int.from_bytes(blob[at:at + 4], "little"); at += 4
    d["frame_bytes"] = at
    return d, blocks, cc


def _walk(blob: bytes, dict_id_ok: bool):
    """The frame's structure as frame_walk_kernel reads it: (descriptor, [(stored, block data, block checksum or None)],
    content checksum or None), or the error code of the first structural fault (FRAME; CHECKSUM for the header checksum).
    dict_id_ok: a dictionary id is read rather than refused."""
    L = len(blob)
    flg, bd = (blob[4], blob[5]) if L >= 6 else (0, 0)
    if L < 7 or int.from_bytes(blob[0:4], "little") != MAGIC or (flg >> 6) != 1 or flg & 0x02 or bd & 0x8F \
            or (flg & 0x01 and not dict_id_ok) or (bd >> 4) & 7 < 4:
        return E_FRAME
    at = 6 + (8 if flg & 0x08 else 0) + (4 if flg & 0x01 else 0)
    if L <= at:
        return E_FRAME
    if blob[at] != (xxh32(blob[4:at]) >> 8) & 0xFF:
        return E_CHECKSUM
    d = {"independent": bool(flg & 0x20), "block_checksum": bool(flg & 0x10), "content_checksum": bool(flg & 0x04),
         "content_size": int.from_bytes(blob[6:14], "little") if flg & 0x08 else None, "bd_code": (bd >> 4) & 7,
         "block_max": BD_SIZES[(bd >> 4) & 7]}
    at += 1
    blocks = []
    while True:
        if L - at < 4:
            return E_FRAME                                   # truncated before a block size or the end mark
        size = int.from_bytes(blob[at:at + 4], "little"); at += 4
        n = size & 0x7FFFFFFF
        if n == 0:
            break                                            # the end mark (read without its stored bit, as upstream does)
        bc = 4 if d["block_checksum"] else 0
        if n > d["block_max"] or L - at < n + bc:
            return E_FRAME
        blocks.append((bool(size >> 31), blob[at:at + n], int.from_bytes(blob[at + n:at + n + 4], "little") if bc else None))
        at += n + bc
    cc = None
    if d["content_checksum"]:
        if L - at < 4:
            return E_FRAME
        cc = int.from_bytes(blob[at:at + 4], "little"); at += 4
    if at != L:
        return E_FRAME                                       # one frame per range: nothing may follow it
    return d, blocks, cc


def decode_result(blob: bytes, cap: Optional[int], dictionary: bytes, dict_id_ok: bool, codec=None):
    """(code, content): code is the content length or the first fault in stream order -- the structure, then per block its
    checksum before its decode, then the content size, the capacity (cap; None: any) and the content checksum.
    codec: decodes the blocks that see no earlier bytes (oracle.Oracle, or None: the restatement); a block with a window
    goes through the restatement's dictionary decode (decode_block)."""
    w = _walk(blob, dict_id_ok)
    if isinstance(w, int):
        return w, None
    d, blocks, cc = w
    out = bytearray()
    for stored, data, csum in blocks:
        if csum is not None and csum != xxh32(data):
            return E_CHECKSUM, None
        if stored:
            out += data
            continue
        # linked blocks see the last 64 KiB of the dictionary followed by everything decoded so far (LZ4F_decompress)
        window = dictionary[-WINDOW:] if d["independent"] else (dictionary[-WINDOW:] + bytes(out[-WINDOW:]))[-WINDOW:]
        if window or codec is None:
            got = decode_block(data, d["block_max"], window)
        else:
            try:
                name = {4: "BlockMax64KB", 5: "BlockMax256KB", 6: "BlockMax1MB", 7: "BlockMax4MB"}[d["bd_code"]]
                (got,) = codec.decompress_chunks_raw([len(data).to_bytes(4, "little") + data], block_size=name, linked=False)
            except RuntimeError:
                got = None
        if got is None:
            return E_BLOCK, None
        out += got
    if d["content_size"] is not None and d["content_size"] != len(out):
        return E_FRAME, None
    if cap is not None and len(out) > cap:
        return E_NOMEM, None
    if cc is not None and cc != xxh32(out):
        return E_CHECKSUM, bytes(out)
    return len(out), bytes(out)


def verdict(blob: bytes, cap: int) -> int:
    """What b200lz4_frame_decompress_batch reports for one frame given dst_cap = cap: the content length, or the code of
    the frame's first fault (frame_walk_kernel's structural checks, then frame_settle_kernel's order)."""
    return decode_result(blob, cap, b"", False)[0]


def decode(oracle, blob: bytes, dictionary: bytes = b"") -> bytes:
    """Stock frame decode (LZ4F_decompress, LZ4F_decompress_usingDict with a dictionary) over the whole range: a linked
    block sees the last 64 KiB of the dictionary and the content decoded before it, across any number of blocks; every
    block of an independent frame sees the dictionary alone.  `oracle` decodes the blocks that see no earlier bytes (see
    decode_result).  Raises ValueError like a stock reader would."""
    code, out = decode_result(blob, None, bytes(dictionary), True, oracle)
    if code < 0:
        raise ValueError(f"frame rejected ({code})")
    return out


def literal_block(raw: bytes) -> bytes:
    """The LZ4 block that decodes to `raw` using literals only: token, length bytes, the literals."""
    n = len(raw)
    if n < 15:
        return bytes([n << 4]) + raw
    rest, ext = n - 15, bytearray()
    while rest >= 255:
        ext.append(255); rest -= 255
    ext.append(rest)
    return bytes([0xF0]) + bytes(ext) + raw
