"""streamly_lz4_b200 -- B200-native LZ4 block codec behind streamly-lz4's API.

The product is the C-ABI CUDA library `libb200lz4.so` (include/b200lz4.h);
this package is the host-side mirror of the reference's `Streamly.LZ4` interface
plus the ctypes binding used by tests and bench.  No CPU codec lives here.
"""
from .api import (BlockConfig, BlockSize, FrameConfig, Context, MultiContext, CompressStream, DecompressStream, LZ4Error,
                  Dictionary, compress_chunks, decompress_chunks, decompress_chunks_raw, resize_chunks,
                  default_block_config, default_frame_config, set_block_max_size,
                  set_block_independence, set_frame_end_mark,
                  simple_frame_parser, frame_header, compress_chunks_frame, decompress_chunks_with,
                  parse_frame_header, write_frame, read_frame, FrameInfo, frame_bound, frame_info)

__all__ = ["BlockConfig", "BlockSize", "FrameConfig", "Context", "MultiContext", "CompressStream", "DecompressStream", "LZ4Error",
           "Dictionary", "compress_chunks", "decompress_chunks", "decompress_chunks_raw", "resize_chunks",
           "default_block_config", "default_frame_config", "set_block_max_size",
           "set_block_independence", "set_frame_end_mark",
           "simple_frame_parser", "frame_header", "compress_chunks_frame", "decompress_chunks_with",
           "parse_frame_header", "write_frame", "read_frame", "FrameInfo", "frame_bound", "frame_info"]
