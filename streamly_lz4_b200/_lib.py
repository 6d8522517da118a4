"""ctypes loader for libb200lz4.so (the C ABI in include/b200lz4.h).

The library is the product; this module only declares its prototypes.  It fails
loudly when the shared object is missing -- there is no Python or CPU fallback.
"""
from __future__ import annotations

import ctypes
import os

# The streamed host calls want the copy streams and the kernel streams on separate hardware work queues (csrc/api.cu:
# probe_stream_aliasing); CUDA reads this when the context is created, so ask before anything initialises CUDA.  The
# library's own load-time constructor does the same for non-Python hosts.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200LZ4_LIB") or os.path.join(_HERE, "libb200lz4.so")   # override: A/B builds of the same ABI

c_int, c_i64, c_vp, c_sz = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_size_t

# name -> (restype, argtypes); every symbol include/b200lz4.h declares
PROTOTYPES = {
    "b200lz4_compress_bound": (c_int, [c_int]),
    "b200lz4_version": (c_int, []),
    "b200lz4_last_error": (ctypes.c_char_p, []),
    "b200lz4_device_count": (c_int, []),
    "b200lz4_ctx_create": (c_int, [c_int, ctypes.POINTER(c_vp)]),
    "b200lz4_ctx_destroy": (None, [c_vp]),
    "b200lz4_host_alloc": (c_vp, [c_sz]),
    "b200lz4_ctx_host_alloc": (c_vp, [c_vp, c_sz]),
    "b200lz4_host_alloc_wc": (c_vp, [c_sz]),
    "b200lz4_host_free": (None, [c_vp]),
    "b200lz4_last_timing": (c_int, [c_vp, ctypes.POINTER(ctypes.c_float)] + [ctypes.POINTER(ctypes.c_float)] * 2),
    "b200lz4_launch_count": (c_i64, [c_vp]),
    "b200lz4_ctx_last_error": (ctypes.c_char_p, [c_vp]),
    "b200lz4_gather_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int]),
    "b200lz4_copy_probe": (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64]),
    "b200lz4_mctx_create": (c_int, [c_vp, c_int, ctypes.POINTER(c_vp)]),
    "b200lz4_mctx_destroy": (None, [c_vp]),
    "b200lz4_mctx_size": (c_int, [c_vp]),
    "b200lz4_mctx_ctx": (c_vp, [c_vp, c_int]),
    "b200lz4_mctx_last_error": (ctypes.c_char_p, [c_vp]),
    "b200lz4_compress_batch_multi": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int,
                                             c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "b200lz4_decompress_batch_multi": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int,
                                               c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "b200lz4_cstream_create": (c_int, [c_vp, ctypes.POINTER(c_vp)]),
    "b200lz4_cstream_free": (None, [c_vp]),
    "b200lz4_dstream_create": (c_int, [c_vp, ctypes.POINTER(c_vp)]),
    "b200lz4_dstream_free": (None, [c_vp]),
    "b200lz4_cstream_peek": (c_int, [c_vp, c_vp, c_vp]),
    "b200lz4_compress_batch": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp,
                                       c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "b200lz4_decompress_batch": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp,
                                         c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "b200lz4_dict_create": (c_int, [c_vp, c_vp, c_i64, ctypes.POINTER(c_vp)]),
    "b200lz4_dict_free": (None, [c_vp]),
    "b200lz4_cstream_load_dict": (c_int, [c_vp, c_vp]),
    "b200lz4_dstream_set_dict": (c_int, [c_vp, c_vp]),
    "b200lz4_compress_batch_dict": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp,
                                            c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "b200lz4_decompress_batch_dict": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_int, c_vp,
                                              c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "b200lz4_cstate_bytes": (c_sz, []),
    "b200lz4_dstate_bytes": (c_sz, []),
    "b200lz4_scratch_bytes": (c_sz, []),
    "b200lz4_cstate_set_dict": (c_int, [c_vp, c_vp, ctypes.c_uint32, c_vp]),
    "b200lz4_compress_dev": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                                     c_int, c_int, c_vp, c_vp]),
    "b200lz4_decompress_dev": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                                       c_int, c_int, c_vp, c_vp]),
    "b200lz4_dict_load_dev": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp]),
    "b200lz4_compress_dev_dict": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                          c_int, c_int, c_vp, c_vp]),
    "b200lz4_decompress_dev_dict": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                            c_int, c_int, c_vp, c_vp]),
    "b200lz4_compact_dev": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "b200lz4_reframe": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64,
                                ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), ctypes.POINTER(c_int)]),
    "b200lz4_reframe_dev": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "b200lz4_xxh32_dev": (c_int, [c_vp, c_vp, c_vp, c_int, ctypes.c_uint32, c_vp, c_vp]),
    "b200lz4_xxh32_batch": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_int, ctypes.c_uint32, c_vp]),
    # legacy aliases of the reference's 7 foreign imports (src/Streamly/Internal/LZ4.hs:105-140)
    "LZ4_createStream": (c_vp, []),
    "LZ4_freeStream": (c_int, [c_vp]),
    "LZ4_createStreamDecode": (c_vp, []),
    "LZ4_freeStreamDecode": (c_int, [c_vp]),
    "LZ4_compressBound": (c_int, [c_int]),
    "LZ4_compress_fast_continue": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int]),
    "LZ4_decompress_safe_continue": (c_int, [c_vp, c_vp, c_vp, c_int, c_int]),
    "LZ4_loadDict": (c_int, [c_vp, c_vp, c_int]),
    "LZ4_setStreamDecode": (c_int, [c_vp, c_vp, c_int]),
}

_LIB = None


def load() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
                "streamly_lz4_b200 has no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)          # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _LIB = lib
    return _LIB


def last_error() -> str:
    return load().b200lz4_last_error().decode("utf-8", "replace")
