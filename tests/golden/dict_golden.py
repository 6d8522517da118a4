#!/usr/bin/env python
"""Shared dictionaries (LZ4_loadDict / LZ4_setStreamDecode / LZ4_decompress_safe_usingDict): the inputs the dictionary
tests use, two CPU codecs that follow upstream's dictionary semantics, and the generator of their stored outputs.

  python tests/golden/dict_golden.py [LIB]  -> dict_checks.json from upstream LZ4 LIB (default: the system liblz4, 1.9.x):
                                               framed digests of LZ4_loadDict + LZ4_compress_fast_continue on every
                                               generator, dictionary length and configuration, the verdicts of
                                               LZ4_decompress_safe_usingDict on corrupted and hand-built boundary blocks,
                                               and two LZ4F_compressFrame_usingCDict frames with a dictionary id

Codecs (same methods: compress_chunks / decompress_chunks_raw with a `dictionary`, framed as [compLen][uncompLen][block]):
  Upstream(path)  any upstream LZ4 shared library through ctypes (the system liblz4, or the reference build oracle/_ref);
  Port()          the restatement oracle/lz4_oracle.c (liboracle.so), its stream records set up by load_dict_table below --
                  a restatement of LZ4_loadDict -- and by LZ4_setStreamDecode's rule (the dictionary is the previous
                  output, all of its bytes count for the offset check).  The tests check Port against the stored digests
                  before they trust it.
The tests import this module for the inputs, so generator and tests cannot drift apart.
"""
import base64
import ctypes
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import frame  # noqa: E402
from oracle.oracle import _PATHS, available, build  # noqa: E402
from streamly_lz4_b200 import datagen  # noqa: E402

KINDS = ["text", "random", "sparse01", "records", "mixed", "bits01", "biased01", "zero"]


def sha(chunks) -> str:
    return hashlib.sha256(b"".join(chunks)).hexdigest()


def load() -> dict:
    with open(os.path.join(HERE, "dict_checks.json")) as f:
        return json.load(f)


DICT_LENS = [0, 1, 7, 8, 9, 100, 4096, 65535, 65536, 65537, 1 << 20]
DICT_TINY = list(range(14))                      # arrays of 0 .. 13 bytes
DICT_GAPS = [5000, 0, 3000, 0, 0, 70000, 13]     # empty arrays in the middle of a stream
DICT_CONFIGS = [  # name, array sizes, accel, linked
    ("tiny_indep", DICT_TINY, 1, False), ("tiny_linked", DICT_TINY, 1, True),
    ("4k_indep_a1", [4096] * 16, 1, False), ("4k_linked_a12", [4096] * 16, 12, True),
    ("64k_indep_a400", [65536] * 4, 400, False), ("64k_linked_a1", [65536] * 4, 1, True),
    ("640000_indep_a65537", [640000] * 2, 65537, False), ("640000_linked_a1", [640000] * 2, 1, True),
    ("gaps_linked_a1", DICT_GAPS, 1, True),
]
DICT_PREFIX = 1 << 20                            # the dictionary is the DICT_LENS[i] bytes right before the body


def dict_inputs(kind: str, sizes):
    """(dictionary of the largest length, body arrays): one generator stream, dictionary first, body right after it."""
    d = datagen.make(kind, 31, DICT_PREFIX + sum(sizes)).tobytes()
    arrays, at = [], DICT_PREFIX
    for n in sizes:
        arrays.append(d[at:at + n]); at += n
    return d[:DICT_PREFIX], arrays


def dict_of(prefix: bytes, n: int) -> bytes:
    return prefix[len(prefix) - n:] if n else b""


def dict_decoder_cases(ora):
    """(dictionary, framed block with an 8-byte header) pairs for the decoder's verdicts: a text block compressed (by
    `ora`, whose bytes dict_checks.json pins) against dictionaries of 100 bytes and 64 KiB, truncated and bit-flipped; and
    hand-built blocks whose match reaches exactly to the dictionary's first byte or one byte further, at dictionary
    lengths 5, 100 and 65535."""
    prefix, (body,) = dict_inputs("text", [30000])
    cases = []
    rng = np.random.default_rng(17)
    for dl in (100, 65536):
        dic = dict_of(prefix, dl)
        payload = ora.compress_chunks([body], 1, linked=False, dictionary=dic)[0][8:]
        variants = [payload] + [payload[:k] for k in (1, 2, 10, len(payload) // 2, len(payload) - 1)]
        for _ in range(100):
            b = bytearray(payload)
            at = int(rng.integers(0, len(b)))
            b[at] ^= 1 << int(rng.integers(0, 8))
            variants.append(bytes(b))
        cases += [(dic, len(v).to_bytes(4, "little") + len(body).to_bytes(4, "little") + v) for v in variants]
    for dl in (5, 100, 65535):
        dic = dict_of(prefix, dl)
        for lit, off in ((0, dl), (0, dl + 1), (2, dl + 2), (2, dl + 3), (7, dl + 7), (7, dl + 8)):
            if off > 65535:
                continue
            lit_bytes = b"xyzuvwq"[:lit]
            # match of 5, then 5 last literals; a capacity of 64 keeps the end-of-block rules out of the way
            blk = bytes([(lit << 4) | 1]) + lit_bytes + off.to_bytes(2, "little") + bytes([0x50]) + b"12345"
            cases.append((dic, len(blk).to_bytes(4, "little") + (64).to_bytes(4, "little") + blk))
    return cases




def _framed(r: int, n: int, payload: bytes) -> bytes:
    return r.to_bytes(4, "little") + n.to_bytes(4, "little") + payload


def _unframe(f: bytes, meta: int, max_block: int):
    """(payload, capacity) of one framed block, or None when its header is unusable (decompressChunk's checks)"""
    if len(f) < meta:
        return None
    comp = int.from_bytes(f[0:4], "little", signed=True) if meta >= 4 else len(f)
    cap = int.from_bytes(f[4:8], "little", signed=True) if meta == 8 else max_block
    if comp <= 0 or comp > len(f) - meta or cap < 0:
        return None
    return f[meta:meta + comp], cap


class Upstream:
    """An upstream LZ4 shared library's dictionary calls through ctypes.  Each array, output and the dictionary live in
    buffers of their own (one spare byte each), so upstream never switches to prefix mode."""

    def __init__(self, path: str):
        self.lib = lib = ctypes.CDLL(path)
        vp, ip = ctypes.c_void_p, ctypes.c_int
        lib.LZ4_createStream.restype = vp
        lib.LZ4_freeStream.argtypes = [vp]
        lib.LZ4_loadDict.argtypes = [vp, vp, ip]
        lib.LZ4_compress_fast_continue.argtypes = [vp, vp, vp, ip, ip, ip]
        lib.LZ4_createStreamDecode.restype = vp
        lib.LZ4_freeStreamDecode.argtypes = [vp]
        lib.LZ4_setStreamDecode.argtypes = [vp, vp, ip]
        lib.LZ4_decompress_safe_continue.argtypes = [vp, vp, vp, ip, ip]
        lib.LZ4_decompress_safe_usingDict.argtypes = [vp, vp, ip, ip, vp, ip]
        self.path = path

    def compress_chunks(self, arrays, accel: int = 1, linked: bool = True, dictionary: bytes = b""):
        lib, dic = self.lib, dictionary
        keep = [ctypes.create_string_buffer(dic, len(dic) + 1)]
        out, s = [], None
        for a in arrays:
            if s is None or not linked:
                if s is not None:
                    lib.LZ4_freeStream(s)
                s = lib.LZ4_createStream()
                lib.LZ4_loadDict(s, keep[0], len(dic))
            src = ctypes.create_string_buffer(a, len(a) + 1)
            keep.append(src)
            cap = len(a) + len(a) // 255 + 16
            dst = ctypes.create_string_buffer(cap)
            r = lib.LZ4_compress_fast_continue(s, src, dst, len(a), cap, accel)
            if r <= 0:
                raise RuntimeError("LZ4_compress_fast_continue failed")
            out.append(_framed(r, len(a), dst.raw[:r]))
        if s is not None:
            lib.LZ4_freeStream(s)
        return out

    def decompress_chunks_raw(self, framed, linked: bool = True, dictionary: bytes = b"", meta: int = 8, max_block: int = 0):
        lib, dic = self.lib, dictionary
        keep = [ctypes.create_string_buffer(dic, len(dic) + 1)]
        out, s = [], None
        for f in framed:
            if s is None or not linked:
                if s is not None:
                    lib.LZ4_freeStreamDecode(s)
                s = lib.LZ4_createStreamDecode()
                lib.LZ4_setStreamDecode(s, keep[0], len(dic))
            u = _unframe(f, meta, max_block)
            if u is None:
                raise RuntimeError("bad block header")
            payload, cap = u
            src = ctypes.create_string_buffer(payload, len(payload) + 1)
            dst = ctypes.create_string_buffer(cap + 1)
            keep += [src, dst]
            r = lib.LZ4_decompress_safe_continue(s, src, dst, len(payload), cap)
            if r < 0:
                raise RuntimeError("LZ4_decompress_safe_continue failed")
            out.append(dst.raw[:r])
        if s is not None:
            lib.LZ4_freeStreamDecode(s)
        return out

    def decode_verdict(self, dic: bytes, framed: bytes):
        """LZ4_decompress_safe_usingDict on one block: None when rejected, else the output's SHA-256"""
        n, cap = int.from_bytes(framed[0:4], "little"), int.from_bytes(framed[4:8], "little")
        src = ctypes.create_string_buffer(framed[8:], len(framed) - 8 + 1)
        d = ctypes.create_string_buffer(dic, len(dic) + 1)
        dst = ctypes.create_string_buffer(cap + 1)
        r = self.lib.LZ4_decompress_safe_usingDict(src, dst, n, cap, d, len(dic))
        return None if r < 0 else sha([dst.raw[:r]])

class UpstreamFrames(Upstream):
    """Upstream LZ4's frame library with a CDict (what the stored frames were written with)."""

    def frame(self, dic: bytes, data: bytes, independent: bool, dict_id: int) -> bytes:
        """LZ4F_compressFrame_usingCDict: 64 KiB blocks, content checksum, the dictionary id in the descriptor."""
        ct, lib = ctypes, self.lib

        class Prefs(ct.Structure):
            _fields_ = [("blockSizeID", ct.c_int), ("blockMode", ct.c_int), ("contentChecksumFlag", ct.c_int),
                        ("frameType", ct.c_int), ("contentSize", ct.c_ulonglong), ("dictID", ct.c_uint),
                        ("blockChecksumFlag", ct.c_int), ("compressionLevel", ct.c_int), ("autoFlush", ct.c_uint),
                        ("favorDecSpeed", ct.c_uint), ("reserved", ct.c_uint * 3)]
        lib.LZ4F_createCDict.restype = ct.c_void_p
        lib.LZ4F_createCDict.argtypes = [ct.c_void_p, ct.c_size_t]
        lib.LZ4F_freeCDict.argtypes = [ct.c_void_p]
        lib.LZ4F_createCompressionContext.argtypes = [ct.POINTER(ct.c_void_p), ct.c_uint]
        lib.LZ4F_freeCompressionContext.argtypes = [ct.c_void_p]
        lib.LZ4F_compressFrame_usingCDict.restype = ct.c_size_t
        lib.LZ4F_compressFrame_usingCDict.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_size_t, ct.c_void_p, ct.c_size_t,
                                                      ct.c_void_p, ct.POINTER(Prefs)]
        lib.LZ4F_isError.argtypes = [ct.c_size_t]
        d = ct.create_string_buffer(dic, len(dic) + 1)
        cd = lib.LZ4F_createCDict(d, len(dic))
        cctx = ct.c_void_p()
        assert lib.LZ4F_createCompressionContext(ct.byref(cctx), 100) == 0
        p = Prefs(blockSizeID=4, blockMode=1 if independent else 0, contentChecksumFlag=1, dictID=dict_id)
        cap = len(data) + len(data) // 255 + 4096
        dst = ct.create_string_buffer(cap)
        r = lib.LZ4F_compressFrame_usingCDict(cctx, dst, cap, data, len(data), cd, ct.byref(p))
        assert not lib.LZ4F_isError(r)
        lib.LZ4F_freeCompressionContext(cctx)
        lib.LZ4F_freeCDict(cd)
        return dst.raw[:r]

    def frame_decode(self, dic: bytes, blob: bytes, out_len: int) -> bytes:
        ct, lib = ctypes, self.lib
        lib.LZ4F_createDecompressionContext.argtypes = [ct.POINTER(ct.c_void_p), ct.c_uint]
        lib.LZ4F_freeDecompressionContext.argtypes = [ct.c_void_p]
        lib.LZ4F_decompress_usingDict.restype = ct.c_size_t
        lib.LZ4F_decompress_usingDict.argtypes = [ct.c_void_p, ct.c_void_p, ct.POINTER(ct.c_size_t), ct.c_void_p,
                                                  ct.POINTER(ct.c_size_t), ct.c_void_p, ct.c_size_t, ct.c_void_p]
        dctx = ct.c_void_p()
        assert lib.LZ4F_createDecompressionContext(ct.byref(dctx), 100) == 0
        dst = ct.create_string_buffer(out_len + 1)
        dn, sn = ct.c_size_t(out_len + 1), ct.c_size_t(len(blob))
        r = lib.LZ4F_decompress_usingDict(dctx, dst, ct.byref(dn), blob, ct.byref(sn), dic, len(dic), None)
        lib.LZ4F_freeDecompressionContext(dctx)
        assert r == 0 and sn.value == len(blob), "frame did not decode in one call"
        return dst.raw[:dn.value]



_OFFSET0 = 65536        # LZ4_loadDict's currentOffset


def hash5(buf: np.ndarray, pos: np.ndarray) -> np.ndarray:
    """LZ4_hash5 of the 5 bytes at each position (x86-64 little-endian variant)"""
    five = np.zeros(len(pos), dtype=np.uint64)
    for k in range(5):
        five |= buf[pos + k].astype(np.uint64) << np.uint64(8 * k)
    return (((five << np.uint64(24)) * np.uint64(889523592379)) >> np.uint64(52)).astype(np.int64)


def load_dict_table(dic: bytes):
    """LZ4_loadDict restated: (table, dictSize).  Below HASH_UNIT (8) bytes the table stays empty and dictSize is 0;
    otherwise the last min(len, 64 KiB) bytes are the dictionary, positions p = 0, 3, ... with p + 8 <= dictSize are
    inserted with index 65536 - (dictSize - p), and when several positions hash to one bucket the last one stays."""
    table = np.zeros(4096, dtype=np.uint32)
    if len(dic) < 8:
        return table, 0
    kept = min(len(dic), 65536)
    buf = np.frombuffer(dic[len(dic) - kept:], dtype=np.uint8)
    pos = np.arange(0, kept - 7, 3, dtype=np.int64)
    h = hash5(buf, pos)
    rev_h = h[::-1]
    buckets, first_rev = np.unique(rev_h, return_index=True)       # first in reverse order = last writer
    table[buckets] = (_OFFSET0 - (kept - pos[::-1][first_rev])).astype(np.uint32)
    return table, kept


class _OraC(ctypes.Structure):     # struct ora_cstream (oracle/lz4_oracle.c)
    _fields_ = [("table", ctypes.c_uint32 * 4096), ("offset", ctypes.c_uint32), ("dict", ctypes.c_void_p),
                ("dict_len", ctypes.c_uint32)]


class _OraD(ctypes.Structure):     # struct ora_dstream
    _fields_ = [("prev_out", ctypes.c_void_p), ("prev_len", ctypes.c_size_t)]


class Port:
    """The restatement (oracle/liboracle.so) given a dictionary: a fresh stream record is overwritten with what
    LZ4_loadDict leaves in it (load_dict_table), a decode record with the dictionary as the previous output."""

    def __init__(self):
        if not available("port"):
            build()
        self.lib = lib = ctypes.CDLL(_PATHS["port"])
        vp, ip = ctypes.c_void_p, ctypes.c_int
        lib.ora_cstream_create.restype = ctypes.POINTER(_OraC)
        lib.ora_cstream_free.argtypes = [ctypes.POINTER(_OraC)]
        lib.ora_dstream_create.restype = ctypes.POINTER(_OraD)
        lib.ora_dstream_free.argtypes = [ctypes.POINTER(_OraD)]
        lib.ora_compress_continue.argtypes = [ctypes.POINTER(_OraC), vp, vp, ip, ip, ip]
        lib.ora_compress_continue.restype = ip
        lib.ora_decompress_continue.argtypes = [ctypes.POINTER(_OraD), vp, vp, ip, ip]
        lib.ora_decompress_continue.restype = ip
        self._tables = {}
        self.path = _PATHS["port"]

    def _loaded(self, s, dbuf, dic: bytes):
        key = hashlib.sha256(dic).digest()
        if key not in self._tables:
            self._tables[key] = load_dict_table(dic)
        table, kept = self._tables[key]
        ctypes.memmove(s.contents.table, table.ctypes.data, 4 * 4096)
        s.contents.offset = _OFFSET0
        s.contents.dict = ctypes.addressof(dbuf) + (len(dic) - kept) if kept else None
        s.contents.dict_len = kept

    def compress_chunks(self, arrays, accel: int = 1, linked: bool = True, dictionary: bytes = b""):
        lib, dic = self.lib, dictionary
        dbuf = ctypes.create_string_buffer(dic, len(dic) + 1)
        keep, out, s = [dbuf], [], None
        for a in arrays:
            if s is None or not linked:
                if s is not None:
                    lib.ora_cstream_free(s)
                s = lib.ora_cstream_create()
                self._loaded(s, dbuf, dic)
            src = ctypes.create_string_buffer(a, len(a) + 1)
            keep.append(src)
            cap = len(a) + len(a) // 255 + 16
            dst = ctypes.create_string_buffer(cap)
            r = lib.ora_compress_continue(s, src, dst, len(a), cap, accel)
            if r <= 0:
                raise RuntimeError("ora_compress_continue failed")
            out.append(_framed(r, len(a), dst.raw[:r]))
        if s is not None:
            lib.ora_cstream_free(s)
        return out

    def decompress_chunks_raw(self, framed, linked: bool = True, dictionary: bytes = b"", meta: int = 8, max_block: int = 0):
        lib, dic = self.lib, dictionary
        dbuf = ctypes.create_string_buffer(dic, len(dic) + 1)
        keep, out, s = [dbuf], [], None
        for f in framed:
            if s is None or not linked:
                if s is not None:
                    lib.ora_dstream_free(s)
                s = lib.ora_dstream_create()
                s.contents.prev_out = ctypes.addressof(dbuf) if dic else None      # LZ4_setStreamDecode
                s.contents.prev_len = len(dic)
            u = _unframe(f, meta, max_block)
            if u is None:
                raise RuntimeError("bad block header")
            payload, cap = u
            src = ctypes.create_string_buffer(payload, len(payload) + 1)
            dst = ctypes.create_string_buffer(cap + 1)
            keep += [src, dst]
            r = lib.ora_decompress_continue(s, src, dst, len(payload), cap)
            if r < 0:
                raise RuntimeError("ora_decompress_continue failed")
            out.append(dst.raw[:r])
        if s is not None:
            lib.ora_dstream_free(s)
        return out

    def decode_verdict(self, dic: bytes, framed: bytes):
        try:
            return sha(self.decompress_chunks_raw([framed], linked=False, dictionary=dic))
        except RuntimeError:
            return None


def codecs():
    """the CPU codecs the tests check: the restatement, and the reference build where oracle/Makefile could make it"""
    return [Port()] + ([Upstream(_PATHS["reference"])] if available("reference") else [])


def frame_decode(codec, blob: bytes, dictionary: bytes = b"") -> bytes:
    """A stock frame reader given `dictionary` (LZ4F_decompress_usingDict): every block of an independent frame, the first
    of a linked one, starts from it; linked blocks see the previous block (every block but the last is 64 KiB in the
    frames the tests use).  Raises ValueError / RuntimeError like a reader would."""
    d, blocks, cc = frame.parse(blob)
    framed = []
    for stored, data in blocks:
        if stored:
            data = frame.literal_block(data)
        framed.append(len(data).to_bytes(4, "little") + data)
    out = b"".join(codec.decompress_chunks_raw(framed, linked=not d["independent"], dictionary=dictionary, meta=4,
                                               max_block=d["block_max"]))
    if cc is not None and cc != frame.xxh32(out):
        raise ValueError("content checksum mismatch")
    return out

DICT_FRAMES = [  # name, independent, dict id; text, 64 KiB dictionary, a full 64 KiB block and a short one
    ("frame_indep", True, 0x1234ABCD), ("frame_linked", False, 7)]
DICT_FRAME_SIZES = [65536, 3000]


def make_dict(up: "UpstreamFrames"):
    v = up.lib.LZ4_versionNumber()
    digests = {}
    for kind in KINDS:
        for name, sizes, accel, linked in DICT_CONFIGS:
            prefix, arrays = dict_inputs(kind, sizes)
            for dl in DICT_LENS:
                digests[f"{kind}/{name}/{dl}"] = sha(up.compress_chunks(arrays, accel, linked, dict_of(prefix, dl)))
    cases = dict_decoder_cases(up)
    verdicts = [up.decode_verdict(dic, framed) for dic, framed in cases]
    frames = {}
    prefix, arrays = dict_inputs("text", DICT_FRAME_SIZES)
    data = b"".join(arrays)
    for name, indep, did in DICT_FRAMES:
        blob = up.frame(dict_of(prefix, 65536), data, indep, did)
        assert up.frame_decode(dict_of(prefix, 65536), blob, len(data)) == data
        frames[name] = {"independent": indep, "dict_id": did, "input_sha256": sha([data]),
                        "frame_b64": base64.b64encode(blob).decode()}
    print("dict: digests", len(digests), "decoder cases", len(verdicts), "rejected", verdicts.count(None), "frames", len(frames))
    return {"generator": "tests/golden/dict_golden.py",
            "codec": f"LZ4 {v // 10000}.{v // 100 % 100}.{v % 100} ({os.path.basename(up.path)}, LZ4_loadDict + "
                     "LZ4_compress_fast_continue, LZ4_decompress_safe_usingDict, LZ4F_compressFrame_usingCDict through ctypes)",
            "digests": digests, "decoder_verdicts": verdicts, "frames": frames}


def main():
    import ctypes.util
    path = sys.argv[1] if len(sys.argv) > 1 else ctypes.util.find_library("lz4")
    assert path, "no liblz4 found: name one, dict_golden.py /path/to/liblz4.so"
    out = make_dict(UpstreamFrames(path))
    with open(os.path.join(HERE, "dict_checks.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
