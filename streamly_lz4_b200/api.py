"""Host-side mirror of the reference's public API over the C ABI.

Names, argument meaning and error behaviour follow `Streamly.LZ4`
(src/Streamly/LZ4.hs:40-122) and `Streamly.Internal.LZ4`
(src/Streamly/Internal/LZ4.hs:342-567):

    compress_chunks(cfg, speed, chunks)      compressChunks   LZ4.hs:94-100   / Internal/LZ4.hs:353-394
    decompress_chunks(cfg, chunks)           decompressChunks LZ4.hs:114-122  (= resize then raw decode)
    decompress_chunks_raw(cfg, chunks)       decompressChunksRawD  Internal/LZ4.hs:539-567
    resize_chunks(cfg, frame_cfg, chunks)    resizeChunksD    Internal/LZ4.hs:432-523
    BlockConfig / BlockSize / FrameConfig    Internal/LZ4/Config.hs:41-161

A "stream" is any Python iterable of bytes-like arrays.  Where the reference
calls the codec once per array, this mirror gathers arrays into a pinned host
batch and makes ONE call into libb200lz4.so per batch (the behaviour the
patched Haskell shim in INTEGRATION.md has); results are yielded in order, one
output array per input array, with the reference's block header layout.

All codec work happens in the CUDA library; there is no CPU path here.
"""
from __future__ import annotations

import ctypes
import enum
import threading
from dataclasses import dataclass, replace
from typing import Iterable, Iterator, List, Optional, Sequence

import numpy as np

from . import _lib

LZ4_MAX_INPUT_SIZE = 0x7E000000


class BlockSize(enum.Enum):                 # Config.hs:104-119
    BlockHasSize = 0
    BlockMax64KB = 64 * 1024
    BlockMax256KB = 256 * 1024
    BlockMax1MB = 1024 * 1024
    BlockMax4MB = 4 * 1024 * 1024


@dataclass(frozen=True)
class BlockConfig:                           # Config.hs:121-134
    block_size: BlockSize = BlockSize.BlockHasSize
    independent: bool = False                # setBlockIndependence (a stub in the reference, Config.hs:142-146)

    @property
    def meta_size(self) -> int:              # metaSize, Internal/LZ4.hs:177-181
        return 8 if self.block_size is BlockSize.BlockHasSize else 4

    @property
    def max_block_size(self) -> int:         # Internal/LZ4.hs:275-281
        return LZ4_MAX_INPUT_SIZE if self.block_size is BlockSize.BlockHasSize else self.block_size.value


@dataclass(frozen=True)
class FrameConfig:                           # Config.hs:41-48
    has_end_mark: bool = False


default_block_config = BlockConfig()
default_frame_config = FrameConfig()


def set_block_max_size(bs: BlockSize):       # setBlockMaxSize, Config.hs:136-140
    return lambda cfg: replace(cfg, block_size=bs)


def set_block_independence(flag: bool):      # setBlockIndependence, Config.hs:142-146 (implemented here)
    return lambda cfg: replace(cfg, independent=flag)


def set_frame_end_mark(flag: bool):          # setFrameEndMark, Config.hs:60-63
    return lambda cfg: replace(cfg, has_end_mark=flag)


class LZ4Error(RuntimeError):
    pass


class Context:
    """One b200lz4_ctx (device + CUDA stream + staging arenas) with pinned batch buffers."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = ctypes.c_void_p()
        rc = self.lib.b200lz4_ctx_create(device, ctypes.byref(h))
        if rc != 0:
            raise LZ4Error(f"b200lz4_ctx_create({device}) failed ({rc}): {_lib.last_error()}")
        self.handle = h
        self.device = device
        self._pins = {}

    def close(self):
        if self.handle:
            for p, _ in self._pins.values():
                self.lib.b200lz4_host_free(p)
            self._pins = {}
            self.lib.b200lz4_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def pinned(self, name: str, nbytes: int, write_combined: bool = False) -> np.ndarray:
        """A reusable page-locked uint8 buffer of at least nbytes (write_combined: for input the host only writes)."""
        cur = self._pins.get(name)
        if cur is None or cur[1].size < nbytes:
            if cur is not None:
                self.lib.b200lz4_host_free(cur[0])
            cap = max(int(nbytes * 1.25) + 4096, 1 << 16)
            p = self.lib.b200lz4_host_alloc_wc(cap) if write_combined else self.lib.b200lz4_ctx_host_alloc(self.handle, cap)
            if not p:
                raise LZ4Error("b200lz4_host_alloc failed: " + _lib.last_error())
            arr = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(cap,))
            self._pins[name] = cur = (p, arr)
        return cur[1]

    def timing(self):
        a, b, c = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
        self.lib.b200lz4_last_timing(self.handle, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        return {"h2d_ms": a.value, "kernel_ms": b.value, "d2h_ms": c.value}

    def launch_count(self) -> int:
        return int(self.lib.b200lz4_launch_count(self.handle))

    def last_error(self) -> str:
        return self.lib.b200lz4_ctx_last_error(self.handle).decode("utf-8", "replace")

    def xxh32(self, buf: np.ndarray, offs: np.ndarray, lens: np.ndarray, seed: int = 0) -> np.ndarray:
        """XXH32 of n byte ranges of `buf`, computed on the device (b200lz4_xxh32_batch)."""
        offs = np.ascontiguousarray(offs, dtype=np.int64); lens = np.ascontiguousarray(lens, dtype=np.int32)
        out = np.zeros(len(lens), dtype=np.uint32)
        rc = self.lib.b200lz4_xxh32_batch(self.handle, buf.ctypes.data, buf.size, offs.ctypes.data, lens.ctypes.data, len(lens), seed,
                                          out.ctypes.data)
        if rc != 0:
            raise LZ4Error("b200lz4_xxh32_batch: " + _lib.last_error())
        return out

    def copy_probe(self, h_src: np.ndarray, h2d_bytes: int, h_dst: np.ndarray, d2h_bytes: int, check: bool = False) -> int:
        """One plain H2D + D2H copy pair on the ctx's copy streams (measurement aid, no kernels)."""
        rc = self.lib.b200lz4_copy_probe(self.handle, h_src.ctypes.data, h2d_bytes, h_dst.ctypes.data, d2h_bytes)
        if check and rc != 0:
            raise LZ4Error("b200lz4_copy_probe: " + _lib.last_error())
        return rc

    def dictionary(self, data) -> "Dictionary":
        """Load `data` as a shared dictionary on this ctx's device (LZ4_loadDict / LZ4_setStreamDecode semantics)."""
        return Dictionary(self, data)

    # ---- raw batch calls on numpy buffers --------------------------------
    def compress_batch(self, src: np.ndarray, src_off: np.ndarray, src_len: np.ndarray,
                       accel: int, header: int, dst: np.ndarray,
                       stream_first: Optional[np.ndarray] = None, streams: Optional[Sequence] = None,
                       dictionary: Optional["Dictionary"] = None):
        """dictionary: every stream without a persistent handle starts from it (b200lz4_compress_batch_dict)."""
        n = len(src_len)
        dst_off = np.zeros(n + 1, dtype=np.int64)
        out_len = np.zeros(n, dtype=np.int32)
        sf = None if stream_first is None else np.ascontiguousarray(stream_first, dtype=np.int32)
        ns = 0 if sf is None else len(sf) - 1
        sh = None
        if streams is not None:
            sh = (ctypes.c_void_p * ns)(*[s.handle for s in streams])
        args = (self.handle, src.ctypes.data, src.size, src_off.ctypes.data, src_len.ctypes.data, n,
                None if sf is None else sf.ctypes.data, ns, sh, accel, header,
                dst.ctypes.data, dst.size, dst_off.ctypes.data, out_len.ctypes.data)
        if dictionary is None:
            rc = self.lib.b200lz4_compress_batch(*args)
        else:
            rc = self.lib.b200lz4_compress_batch_dict(*args, dictionary.handle)
        return rc, dst_off, out_len

    def decompress_batch(self, src: np.ndarray, src_off: np.ndarray, src_len: np.ndarray,
                         header: int, max_block: int, dst: np.ndarray,
                         stream_first: Optional[np.ndarray] = None, streams: Optional[Sequence] = None,
                         dictionary: Optional["Dictionary"] = None):
        """dictionary: every stream without a persistent handle starts from it (b200lz4_decompress_batch_dict)."""
        n = len(src_len)
        dst_off = np.zeros(n + 1, dtype=np.int64)
        out_len = np.zeros(n, dtype=np.int32)
        sf = None if stream_first is None else np.ascontiguousarray(stream_first, dtype=np.int32)
        ns = 0 if sf is None else len(sf) - 1
        sh = None
        if streams is not None:
            sh = (ctypes.c_void_p * ns)(*[s.handle for s in streams])
        args = (self.handle, src.ctypes.data, src.size, src_off.ctypes.data, src_len.ctypes.data, n,
                None if sf is None else sf.ctypes.data, ns, sh, header, max_block,
                dst.ctypes.data, dst.size, dst_off.ctypes.data, out_len.ctypes.data)
        if dictionary is None:
            rc = self.lib.b200lz4_decompress_batch(*args)
        else:
            rc = self.lib.b200lz4_decompress_batch_dict(*args, dictionary.handle)
        return rc, dst_off, out_len


class Dictionary:
    """A dictionary loaded on one Context's device (b200lz4_dict).  Only the last 64 KiB reach the codec; `len(d)` is the
    full length, which the decoder's offset check uses."""

    def __init__(self, ctx: Context, data):
        self.ctx = ctx
        self.data = bytes(data)
        h = ctypes.c_void_p()
        rc = ctx.lib.b200lz4_dict_create(ctx.handle, self.data, len(self.data), ctypes.byref(h))
        if rc != 0:
            raise LZ4Error("b200lz4_dict_create: " + _lib.last_error())
        self.handle = h

    def __len__(self) -> int:
        return len(self.data)

    def free(self):
        if self.handle:
            self.ctx.lib.b200lz4_dict_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.free()
        except Exception:
            pass


class CompressStream:
    """Device-resident LZ4_stream_t (c_createStream / c_freeStream, Internal/LZ4.hs:105-110)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = ctypes.c_void_p()
        rc = ctx.lib.b200lz4_cstream_create(ctx.handle, ctypes.byref(h))
        if rc != 0:
            raise LZ4Error("b200lz4_cstream_create: " + _lib.last_error())
        self.handle = h

    def peek(self):
        table = np.zeros(4096, dtype=np.uint32)
        off = ctypes.c_uint32()
        rc = self.ctx.lib.b200lz4_cstream_peek(self.handle, table.ctypes.data, ctypes.addressof(off))
        if rc != 0:
            raise LZ4Error(_lib.last_error())
        return table, off.value

    def load_dict(self, d: Dictionary):
        """LZ4_loadDict on this stream: the next array is compressed with `d` as its dictionary."""
        if self.ctx.lib.b200lz4_cstream_load_dict(self.handle, d.handle) != 0:
            raise LZ4Error("b200lz4_cstream_load_dict: " + _lib.last_error())

    def free(self):
        if self.handle:
            self.ctx.lib.b200lz4_cstream_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.free()
        except Exception:
            pass


class DecompressStream:
    """Device-resident LZ4_streamDecode_t (c_createStreamDecode, Internal/LZ4.hs:113-118)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = ctypes.c_void_p()
        rc = ctx.lib.b200lz4_dstream_create(ctx.handle, ctypes.byref(h))
        if rc != 0:
            raise LZ4Error("b200lz4_dstream_create: " + _lib.last_error())
        self.handle = h

    def set_dict(self, d: Dictionary):
        """LZ4_setStreamDecode(d): the next block is decoded with `d` as the previous output."""
        if self.ctx.lib.b200lz4_dstream_set_dict(self.handle, d.handle) != 0:
            raise LZ4Error("b200lz4_dstream_set_dict: " + _lib.last_error())

    def free(self):
        if self.handle:
            self.ctx.lib.b200lz4_dstream_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.free()
        except Exception:
            pass


class MultiContext:
    """b200lz4_mctx: one batch striped over several GPUs of the box by one process (host thread + ctx per device)."""

    def __init__(self, devices: Optional[Sequence[int]] = None, n: int = 0):
        self.lib = _lib.load()
        h = ctypes.c_void_p()
        if devices is not None:
            arr = (ctypes.c_int * len(devices))(*devices)
            rc = self.lib.b200lz4_mctx_create(arr, len(devices), ctypes.byref(h))
        else:
            rc = self.lib.b200lz4_mctx_create(None, n, ctypes.byref(h))
        if rc != 0:
            raise LZ4Error(f"b200lz4_mctx_create failed ({rc}): {_lib.last_error()}")
        self.handle = h
        self.size = int(self.lib.b200lz4_mctx_size(h))

    def close(self):
        if self.handle:
            self.lib.b200lz4_mctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def last_error(self) -> str:
        return self.lib.b200lz4_mctx_last_error(self.handle).decode("utf-8", "replace")

    def timing(self, i: int):
        a, b, c = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
        self.lib.b200lz4_last_timing(self.lib.b200lz4_mctx_ctx(self.handle, i), ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        return {"h2d_ms": a.value, "kernel_ms": b.value, "d2h_ms": c.value}

    def launch_count(self) -> int:
        return sum(int(self.lib.b200lz4_launch_count(self.lib.b200lz4_mctx_ctx(self.handle, i))) for i in range(self.size))

    def compress_batch(self, src, src_off, src_len, accel, header, dst, stream_first=None):
        n = len(src_len)
        dst_off = np.zeros(n + 1, dtype=np.int64)
        out_len = np.zeros(n, dtype=np.int32)
        sf = None if stream_first is None else np.ascontiguousarray(stream_first, dtype=np.int32)
        rc = self.lib.b200lz4_compress_batch_multi(
            self.handle, src.ctypes.data, src.size, src_off.ctypes.data, src_len.ctypes.data, n,
            None if sf is None else sf.ctypes.data, 0 if sf is None else len(sf) - 1, accel, header,
            dst.ctypes.data, dst.size, dst_off.ctypes.data, out_len.ctypes.data)
        return rc, dst_off, out_len

    def decompress_batch(self, src, src_off, src_len, header, max_block, dst, stream_first=None):
        n = len(src_len)
        dst_off = np.zeros(n + 1, dtype=np.int64)
        out_len = np.zeros(n, dtype=np.int32)
        sf = None if stream_first is None else np.ascontiguousarray(stream_first, dtype=np.int32)
        rc = self.lib.b200lz4_decompress_batch_multi(
            self.handle, src.ctypes.data, src.size, src_off.ctypes.data, src_len.ctypes.data, n,
            None if sf is None else sf.ctypes.data, 0 if sf is None else len(sf) - 1, header, max_block,
            dst.ctypes.data, dst.size, dst_off.ctypes.data, out_len.ctypes.data)
        return rc, dst_off, out_len


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def _batches(chunks: Iterable, batch_arrays: int, batch_bytes: int):
    group: List[bytes] = []
    size = 0
    for c in chunks:
        b = c if isinstance(c, (bytes, bytearray, memoryview)) else np.ascontiguousarray(c, dtype=np.uint8).reshape(-1)
        group.append(b)
        size += len(b)
        if len(group) >= batch_arrays or size >= batch_bytes:
            yield group
            group, size = [], 0
    if group:
        yield group


def _gather(ctx: Context, name: str, arrays: Sequence):
    """Lay the arrays of one batch out in a page-locked buffer (b200lz4_gather_host: parallel memcpy in the library)."""
    n = len(arrays)
    views = [a if isinstance(a, np.ndarray) else np.frombuffer(a, dtype=np.uint8) for a in arrays]
    lens = np.fromiter((v.size for v in views), dtype=np.int32, count=n)
    offs = np.zeros(n, dtype=np.int64)
    # 16-byte aligned starts; a gap keeps consecutive arrays non-adjacent like separate Haskell arrays
    strides = (lens.astype(np.int64) + 16 + 15) // 16 * 16
    if n > 1:
        offs[1:] = np.cumsum(strides[:-1])
    total = int(strides.sum())
    buf = ctx.pinned(name, total)
    ptrs = np.fromiter((v.ctypes.data for v in views), dtype=np.uint64, count=n)
    rc = ctx.lib.b200lz4_gather_host(buf.ctypes.data, ptrs.ctypes.data, offs.ctypes.data, lens.ctypes.data, n, 0)
    if rc != 0:
        raise LZ4Error("b200lz4_gather_host: " + _lib.last_error())
    return buf[:total], offs, lens


def _staged(ctx: Context, name: str, groups):
    """Yield (group, src, offs, lens) with the gather of the NEXT group running on a helper thread while the caller
    works on the current one (two alternating pinned buffers; ctypes releases the GIL inside the library)."""
    it = iter(groups)
    slot = 0
    box = {}

    def stage(g, k):
        try:
            box["out"] = (g,) + _gather(ctx, f"{name}{k}", g)
        except BaseException as e:      # re-raised on the consumer side
            box["err"] = e

    def start():
        nonlocal slot
        g = next(it, None)
        if g is None:
            return None
        t = threading.Thread(target=stage, args=(g, slot))
        slot ^= 1
        t.start()
        return t

    t = start()
    while t is not None:
        t.join()
        if "err" in box:
            raise box.pop("err")
        cur = box.pop("out")
        t = start()
        yield cur


def compress_chunks(cfg: BlockConfig, speed: int, chunks: Iterable, *, ctx: Optional[Context] = None,
                    batch_arrays: int = 4096, batch_bytes: int = 256 << 20, copy: bool = True,
                    dictionary: Optional[Dictionary] = None) -> Iterator[bytes]:
    """compressChunks cfg speed (LZ4.hs:94-100): each input array becomes one framed LZ4 block.

    Linked mode (default, like the reference): one device stream state for the whole
    stream, arrays strictly in order.  cfg.independent: fresh state per array.
    dictionary: a Dictionary of the same ctx; every array (independent) or the first one (linked) is compressed as after
    LZ4_loadDict.
    copy=False yields numpy views into the pinned result buffer instead of bytes objects (what the Haskell shim does
    with array slices); a view stays valid until the batch after the next one has been produced.
    """
    ctx = ctx or (dictionary.ctx if dictionary is not None else default_context())
    speed = max(int(speed), 0)                                   # Internal/LZ4.hs:364
    header = cfg.meta_size
    stream = None if cfg.independent else CompressStream(ctx)    # CompressInit, Internal/LZ4.hs:367-376
    if stream is not None and dictionary is not None:
        stream.load_dict(dictionary)

    def checked(groups):
        for group in groups:
            for a in group:
                if len(a) >= 2 * 1024 * 1024 * 1024:             # Internal/LZ4.hs:384-385
                    raise LZ4Error("compressChunksD: Array element > 2 GB encountered")
                if len(a) > cfg.max_block_size:                  # Internal/LZ4.hs:237-241
                    raise LZ4Error(f"compressChunk: Source array length {len(a)} exceeds the maximum block size "
                                   f"of {cfg.max_block_size}")
            yield group
    try:
        k = 0
        for group, src, offs, lens in _staged(ctx, "c_src", checked(_batches(chunks, batch_arrays, batch_bytes))):
            cap = int((lens.astype(np.int64) + lens // 255 + 16 + header).sum())
            dst = ctx.pinned(f"c_dst{k}", cap)
            k ^= 1
            sf = None if stream is None else np.array([0, len(group)], dtype=np.int32)
            rc, dst_off, out_len = ctx.compress_batch(src, offs, lens, speed, header, dst, sf,
                                                      None if stream is None else [stream],
                                                      dictionary if stream is None else None)
            if rc != 0:                                          # Internal/LZ4.hs:257-260
                raise LZ4Error(f"compressChunk: c_compressFastContinue failed ({rc}): {ctx.last_error()}")
            for i in range(len(group)):
                blk = dst[dst_off[i]:dst_off[i + 1]]
                yield blk.tobytes() if copy else blk
    finally:
        if stream is not None:
            stream.free()                                        # CompressDone, Internal/LZ4.hs:393-394


def _decode_batches(chunks: Iterable, batch_arrays: int, batch_bytes: int, cap_of, out_budget: int):
    """Group framed arrays so that neither the compressed bytes nor the WORST-CASE output of a batch exceed their
    budgets (BlockMax* headers carry no size: every block may expand to the configured maximum)."""
    group: List = []
    size = out = 0
    for c in chunks:
        b = c if isinstance(c, (bytes, bytearray, memoryview)) else np.ascontiguousarray(c, dtype=np.uint8).reshape(-1)
        cap = cap_of(b)
        if group and (out + cap > out_budget):
            yield group
            group, size, out = [], 0, 0
        group.append(b)
        size += len(b)
        out += cap
        if len(group) >= batch_arrays or size >= batch_bytes:
            yield group
            group, size, out = [], 0, 0
    if group:
        yield group


def decompress_chunks_raw(cfg: BlockConfig, chunks: Iterable, *, ctx: Optional[Context] = None,
                          batch_arrays: int = 4096, batch_bytes: int = 256 << 20, out_budget: int = 1 << 30,
                          copy: bool = True, dictionary: Optional[Dictionary] = None) -> Iterator[bytes]:
    """decompressChunksRawD (Internal/LZ4.hs:539-567): every input array is exactly one framed block.
    A batch is flushed as soon as its worst-case output would exceed out_budget bytes (1 GiB).
    dictionary: every block (independent) or the first one (linked) is decoded as LZ4_decompress_safe_usingDict would."""
    ctx = ctx or (dictionary.ctx if dictionary is not None else default_context())
    header = cfg.meta_size
    max_block = 0 if cfg.block_size is BlockSize.BlockHasSize else cfg.block_size.value
    stream = None if cfg.independent else DecompressStream(ctx)
    if stream is not None and dictionary is not None:
        stream.set_dict(dictionary)

    def cap_of(a) -> int:
        if header == 8:
            return max(int.from_bytes(bytes(a[4:8]), "little", signed=True), 0) if len(a) >= 8 else 0
        return max_block + 16
    try:
        k = 0
        for group, src, offs, lens in _staged(ctx, "d_src", _decode_batches(chunks, batch_arrays, batch_bytes // 2, cap_of, out_budget)):
            cap = sum(cap_of(a) for a in group)
            dst = ctx.pinned(f"d_dst{k}", cap + 64)
            k ^= 1
            sf = None if stream is None else np.array([0, len(group)], dtype=np.int32)
            rc, dst_off, out_len = ctx.decompress_batch(src, offs, lens, header, max_block, dst, sf,
                                                        None if stream is None else [stream],
                                                        dictionary if stream is None else None)
            if rc != 0:                                          # Internal/LZ4.hs:309-330
                raise LZ4Error(f"decompressChunk: c_decompressSafeContinue failed ({rc}): {ctx.last_error()}")
            for i in range(len(group)):
                blk = dst[dst_off[i]:dst_off[i] + out_len[i]]
                yield blk.tobytes() if copy else blk
    finally:
        if stream is not None:
            stream.free()


def resize_chunks(cfg: BlockConfig, frame_cfg: FrameConfig, chunks: Iterable) -> Iterator[bytes]:
    """resizeChunksD (Internal/LZ4.hs:432-523): re-frame an arbitrarily fragmented compressed
    stream into one array per [header][block].  The header walk runs in b200lz4_reframe."""
    lib = _lib.load()
    header = cfg.meta_size
    buf = bytearray()
    max_blocks = 1 << 16
    off = np.zeros(max_blocks, dtype=np.int64)
    ln = np.zeros(max_blocks, dtype=np.int32)
    nf, used, ended = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()

    def drain():
        while True:
            raw = (ctypes.c_char * len(buf)).from_buffer(buf) if buf else None
            rc = lib.b200lz4_reframe(raw, len(buf), header, int(frame_cfg.has_end_mark),
                                     off.ctypes.data, ln.ctypes.data, max_blocks,
                                     ctypes.byref(nf), ctypes.byref(used), ctypes.byref(ended))
            del raw
            if rc != 0:
                raise LZ4Error("resizeChunksD: " + _lib.last_error())
            out = [bytes(buf[off[k]:off[k] + ln[k]]) for k in range(nf.value)]
            del buf[:used.value]
            yield from out
            if ended.value or nf.value < max_blocks:
                return

    for c in chunks:
        buf += bytes(c)
        yield from drain()
        if ended.value:
            return                                               # RFooter -> Stop, Internal/LZ4.hs:506-522
    if buf:
        raise LZ4Error("resizeChunksD: Incomplete block")        # RAccumulate + Stop, Internal/LZ4.hs:505
    if frame_cfg.has_end_mark:
        raise LZ4Error("resizeChunksD: No end mark found")       # RInit + Stop, Internal/LZ4.hs:493-496


def decompress_chunks(cfg: BlockConfig, chunks: Iterable, *, ctx: Optional[Context] = None, **kw) -> Iterator[bytes]:
    """decompressChunks (LZ4.hs:114-122) = decompressChunksRawD . resizeChunksD."""
    return decompress_chunks_raw(cfg, resize_chunks(cfg, default_frame_config, chunks), ctx=ctx, **kw)


# ---------------------------------------------------------------------------------------------------------------
# LZ4 frame format.  First the reference's own stub (Internal/LZ4.hs:569-651; SURVEY.md section 8f rank 3), mirrored as
# it is; then the complete reader / writer the stub stands in for (header checksum, content size, block independence,
# XXH32 block and content checksums, stored blocks), which is what interoperates with the stock `lz4` tool.

FRAME_MAGIC = 407708164                       # 0x184D2204, little endian on the stream (Internal/LZ4.hs:610)
_BD_CODES = {4: BlockSize.BlockMax64KB, 5: BlockSize.BlockMax256KB, 6: BlockSize.BlockMax1MB, 7: BlockSize.BlockMax4MB}


def _xxh32_short(data: bytes, seed: int = 0) -> int:
    """XXH32 of fewer than 16 bytes (the frame descriptor is 2 .. 14 bytes): only the tail rounds and the avalanche of the
    published definition apply.  Payload checksums are computed on the device (Context.xxh32)."""
    assert len(data) < 16
    m = 0xFFFFFFFF
    rotl = lambda x, r: ((x << r) | (x >> (32 - r))) & m
    h = (seed + 374761393 + len(data)) & m
    at = 0
    while at + 4 <= len(data):
        h = (rotl((h + int.from_bytes(data[at:at + 4], "little") * 3266489917) & m, 17) * 668265263) & m
        at += 4
    for b in data[at:]:
        h = (rotl((h + b * 374761393) & m, 11) * 2654435761) & m
    h ^= h >> 15; h = (h * 2246822519) & m
    h ^= h >> 13; h = (h * 3266489917) & m
    return h ^ (h >> 16)


@dataclass(frozen=True)
class FrameInfo:
    """What a complete frame descriptor says beyond BlockConfig / FrameConfig."""
    block_checksum: bool = False
    content_checksum: bool = False
    content_size: Optional[int] = None
    header_len: int = 7
    dict_id: Optional[int] = None


def simple_frame_parser(header: bytes, *, allow_independent: bool = False):
    """simpleFrameParserD (Internal/LZ4.hs:590-651) over the 7 header bytes [magic LE32][FLG][BD][HC]:
    returns (BlockConfig, FrameConfig) with hasEndMark = True; same rejections, same messages.
    allow_independent: accept the block-independence flag (the reference dies on it, :631-632; this codec supports it)."""
    if len(header) < 7:
        raise LZ4Error("simpleFrameParserD: input ended inside the frame header")
    magic = int.from_bytes(header[0:4], "little")
    if magic != FRAME_MAGIC:                                                    # :604-620
        raise LZ4Error(f"The parsed magic {magic} does not match {FRAME_MAGIC}")
    flg = header[4]
    if not (not (flg >> 7) & 1 and (flg >> 6) & 1):                            # :624
        raise LZ4Error("Version is not 01")
    independent = bool((flg >> 5) & 1)
    if independent and not allow_independent:
        raise LZ4Error("Block independence is not yet supported")               # :631-632
    if (flg >> 4) & 1:
        raise LZ4Error("Block checksum is not yet supported")
    if (flg >> 3) & 1:
        raise LZ4Error("Content size is not yet supported")
    if (flg >> 2) & 1:
        raise LZ4Error("Content checksum is not yet supported")
    if flg & 1:
        raise LZ4Error("Dict is not yet supported")
    bs = _BD_CODES.get(header[5] >> 4)                                           # :643-650
    if bs is None:
        raise LZ4Error("parseBD: Unknown block max size")
    return BlockConfig(block_size=bs, independent=independent), FrameConfig(has_end_mark=True)   # header checksum: any byte, :602


def frame_header(block_size: BlockSize, *, independent: bool = False, block_checksum: bool = False,
                 content_size: Optional[int] = None, content_checksum: bool = False, checksum: bool = True,
                 dict_id: Optional[int] = None) -> bytes:
    """A frame header [magic][FLG][BD][content size?][dict id?][HC].  checksum=False writes HC = 0 like
    benchmark/Main.hs:92-100 (which only the reference's own stub parser accepts); the default is the real
    (XXH32(descriptor) >> 8) & 0xFF."""
    code = {v: k for k, v in _BD_CODES.items()}[block_size]
    flg = 0x40 | (0x20 if independent else 0) | (0x10 if block_checksum else 0) | (0x08 if content_size is not None else 0) \
        | (0x04 if content_checksum else 0) | (0x01 if dict_id is not None else 0)
    desc = bytes([flg, code << 4]) + (b"" if content_size is None else int(content_size).to_bytes(8, "little")) \
        + (b"" if dict_id is None else int(dict_id).to_bytes(4, "little"))
    hc = (_xxh32_short(desc) >> 8) & 0xFF if checksum else 0
    return FRAME_MAGIC.to_bytes(4, "little") + desc + bytes([hc])


def parse_frame_header(head: bytes, allow_dict_id: bool = False):
    """The complete descriptor parser: (BlockConfig, FrameConfig, FrameInfo).  Verifies the version, the reserved bits and
    the header checksum.  A dictionary id is rejected unless allow_dict_id (then FrameInfo.dict_id holds it).  `head` must
    hold at least 19 bytes or the whole header."""
    if len(head) < 7:
        raise LZ4Error("frame: input ended inside the frame header")
    magic = int.from_bytes(head[0:4], "little")
    if magic != FRAME_MAGIC:
        raise LZ4Error(f"The parsed magic {magic} does not match {FRAME_MAGIC}")
    flg, bd = head[4], head[5]
    if (flg >> 6) != 1:
        raise LZ4Error("Version is not 01")
    if flg & 0x02 or bd & 0x8F:
        raise LZ4Error("frame: reserved bits are set")
    if flg & 0x01 and not allow_dict_id:
        raise LZ4Error("Dict is not yet supported")
    bs = _BD_CODES.get(bd >> 4)
    if bs is None:
        raise LZ4Error("parseBD: Unknown block max size")
    at, size, dict_id = 6, None, None
    if flg & 0x08:
        if len(head) < 15:
            raise LZ4Error("frame: input ended inside the frame header")
        size = int.from_bytes(head[6:14], "little"); at = 14
    if flg & 0x01:
        if len(head) < at + 5:
            raise LZ4Error("frame: input ended inside the frame header")
        dict_id = int.from_bytes(head[at:at + 4], "little"); at += 4
    if head[at] != (_xxh32_short(bytes(head[4:at])) >> 8) & 0xFF:
        raise LZ4Error("frame: header checksum mismatch")
    info = FrameInfo(block_checksum=bool(flg & 0x10), content_checksum=bool(flg & 0x04), content_size=size, header_len=at + 1,
                     dict_id=dict_id)
    return BlockConfig(block_size=bs, independent=bool(flg & 0x20)), FrameConfig(has_end_mark=True), info


def compress_chunks_frame(cfg: BlockConfig, frame_cfg: FrameConfig, speed: int, chunks: Iterable, **kw) -> Iterator[bytes]:
    """compressChunksFrame of benchmark/Main.hs:105-118: compressChunksD, then the 4-byte end mark if the frame has one."""
    yield from compress_chunks(cfg, speed, chunks, **kw)
    if frame_cfg.has_end_mark:
        yield b"\x00\x00\x00\x00"


def decompress_chunks_with(parser, chunks: Iterable, *, ctx: Optional[Context] = None, **kw) -> Iterator[bytes]:
    """decompressChunksWithD (Internal/LZ4.hs:569-577): run `parser` over the first 7 bytes of the stream, then
    decompressChunksRawD cfg . resizeChunksD cfg frameCfg on what follows."""
    it = iter(chunks)
    head = b""
    rest = None
    for c in it:
        head += bytes(c)
        if len(head) >= 7:
            rest = head[7:]
            break
    cfg, frame_cfg = parser(head[:7])

    def tail():
        if rest:
            yield rest
        yield from it
    return decompress_chunks_raw(cfg, resize_chunks(cfg, frame_cfg, tail()), ctx=ctx, **kw)


def write_frame(block_size: BlockSize, speed: int, chunks: Iterable, *, independent: bool = False, block_checksum: bool = False,
                content_checksum: bool = False, content_size: Optional[int] = None, ctx: Optional[Context] = None,
                dictionary: Optional[Dictionary] = None, dict_id: Optional[int] = None, **kw) -> Iterator[bytes]:
    """A complete LZ4 frame (what the stock `lz4` tool reads): header with its real checksum, one block per input array
    ([size LE32][LZ4 block][XXH32 of the block iff block_checksum]), end mark, XXH32 of the content iff content_checksum.
    Arrays must not exceed the block maximum.  Linked blocks use the previous ARRAY as dictionary (the reference's
    semantics), which every frame decoder accepts.  Checksums are computed on the device; the content checksum needs the
    whole content in one page-locked buffer.
    dictionary: every block (independent) or the first one (linked) is compressed against it (`lz4 -D`); dict_id: the
    descriptor's dictionary id (FLG bit 0), which tells a reader which dictionary to load."""
    ctx = ctx or (dictionary.ctx if dictionary is not None else default_context())
    if dictionary is not None:
        kw["dictionary"] = dictionary
    cfg = BlockConfig(block_size=block_size, independent=independent)
    yield frame_header(block_size, independent=independent, block_checksum=block_checksum, content_size=content_size,
                       content_checksum=content_checksum, dict_id=dict_id)
    import collections
    kept: List[bytes] = []
    raws = collections.deque()

    def tee(src):
        for c in src:
            b = bytes(c)
            raws.append(b)
            if content_checksum:
                kept.append(b)
            yield b

    def blocks():
        # a block that did not shrink is STORED: size field with bit 31 set, then the raw bytes (what every frame writer does;
        # a compressed block may not exceed the block maximum)
        for blk in compress_chunks(cfg, speed, tee(chunks), ctx=ctx, **kw):
            raw = raws.popleft()
            if len(blk) - 4 >= len(raw) and len(raw):
                yield (len(raw) | 0x80000000).to_bytes(4, "little") + raw
            else:
                yield bytes(blk)
    pending: List[bytes] = []
    for blk in blocks():
        if not block_checksum:
            yield blk
            continue
        pending.append(blk)
        if len(pending) >= 1024:
            yield from _with_block_checksums(ctx, pending)
            pending = []
    if pending:
        yield from _with_block_checksums(ctx, pending)
    yield b"\x00\x00\x00\x00"
    if content_checksum:
        whole = b"".join(kept)
        buf = ctx.pinned("f_content", max(len(whole), 1))
        buf[:len(whole)] = np.frombuffer(whole, dtype=np.uint8)
        yield int(ctx.xxh32(buf[:max(len(whole), 1)], [0], [len(whole)])[0]).to_bytes(4, "little")


def _with_block_checksums(ctx: Context, blocks: Sequence[bytes]) -> Iterator[bytes]:
    src, offs, lens = _gather(ctx, "f_blocks", blocks)
    sums = ctx.xxh32(src, offs + 4, lens - 4)                    # the checksum covers the block data, not its size field
    for b, h in zip(blocks, sums):
        yield b + int(h).to_bytes(4, "little")


def read_frame(chunks: Iterable, *, ctx: Optional[Context] = None, verify: bool = True,
               dictionary: Optional[Dictionary] = None, **kw) -> Iterator[bytes]:
    """Decode one complete LZ4 frame from an arbitrarily fragmented byte stream: header (checksum verified), blocks
    (stored blocks pass through as literal-only LZ4 blocks, so a linked chain stays intact), block checksums, end
    mark, content size and content checksum.  Yields one array per block.
    dictionary: the blocks are decoded as LZ4F_decompress_usingDict does (every block of an independent frame, the first
    of a linked one).  A frame with a dictionary id is refused without one; the id itself is not checked (it names the
    dictionary the writer used, and only the caller knows which one that is)."""
    ctx = ctx or (dictionary.ctx if dictionary is not None else default_context())
    data = b"".join(bytes(c) for c in chunks)
    cfg, _, info = parse_frame_header(data[:19], allow_dict_id=dictionary is not None)
    if dictionary is not None:
        kw["dictionary"] = dictionary
    at = info.header_len
    framed: List[bytes] = []
    check_off, check_len, check_want = [], [], []
    while True:
        if at + 4 > len(data):
            raise LZ4Error("resizeChunksD: No end mark found")
        size = int.from_bytes(data[at:at + 4], "little")
        at += 4
        if size == 0:
            break
        stored, n = bool(size >> 31), size & 0x7FFFFFFF
        if n > cfg.max_block_size or at + n > len(data):
            raise LZ4Error("resizeChunksD: Incomplete block")
        body = data[at:at + n]
        if info.block_checksum:
            check_off.append(at); check_len.append(n); check_want.append(int.from_bytes(data[at + n:at + n + 4], "little"))
            at += 4
        at += n
        if stored:                                               # token, length bytes, literals: decodes to `body` itself
            m = len(body)
            if m < 15:
                body = bytes([m << 4]) + body
            else:
                q, r = divmod(m - 15, 255)
                body = b"\xf0" + b"\xff" * q + bytes([r]) + body
        framed.append(len(body).to_bytes(4, "little") + body)
    if verify and check_want:
        buf = ctx.pinned("f_in", len(data))
        buf[:len(data)] = np.frombuffer(data, dtype=np.uint8)
        got = ctx.xxh32(buf[:len(data)], check_off, check_len)
        bad = np.nonzero(got != np.array(check_want, dtype=np.uint32))[0]
        if len(bad):
            raise LZ4Error(f"frame: block checksum mismatch in block {int(bad[0])}")
    total, outs = 0, []
    for a in decompress_chunks_raw(cfg, framed, ctx=ctx, **kw):
        total += len(a)
        if info.content_checksum and verify:
            outs.append(a)
        yield a
    if info.content_size is not None and info.content_size != total:
        raise LZ4Error(f"frame: content size {total} does not match the header's {info.content_size}")
    if info.content_checksum and verify:
        want = int.from_bytes(data[at:at + 4], "little")
        whole = b"".join(outs)
        buf = ctx.pinned("f_content", max(len(whole), 1))
        buf[:len(whole)] = np.frombuffer(whole, dtype=np.uint8)
        if int(ctx.xxh32(buf[:max(len(whole), 1)], [0], [len(whole)])[0]) != want:
            raise LZ4Error("frame: content checksum mismatch")
