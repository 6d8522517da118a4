"""The compressor has three kernels (wide: one stream per SM; classic dense; compact-table dense) chosen by the number of
streams in a launch.  The library reads its A/B switches once per process, so this test re-runs the byte-parity fuzz
files in child processes with each kernel forced, and checks which kernel actually ran."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUBSET = ["tests/test_gpu_fuzz.py", "tests/test_gpu_parity.py", "tests/test_gpu_device_abi.py", "-k",
          "random_round_trips or echoing or split_over or generators or edge_sizes or acceleration_sweep or linked_state or "
          "(device_abi and not decompress_dev and not compact_dev)"]


DECODE_SUBSET = ["tests/test_gpu_fuzz.py", "tests/test_gpu_parity.py", "tests/test_gpu_configs.py", "tests/test_gpu_device_abi.py",
                 "tests/test_gpu_decode_geometry.py", "-k",
                 "handbuilt or corrupted or random_round_trips or echoing or split_over or generators or edge_sizes or "
                 "empty_and_tiny or block_max or large_blocks or linked_state or malformed or fragmented or "
                 "config3 or config4 or (device_abi and (decompress_dev or scratch_shared)) or decode_geometry"]       # config 3: 1 678 one-block streams = several streams per CTA in the wide kernel


@pytest.mark.parametrize("env", [{"B200LZ4_DWIDE": "0"},        # every decode through the narrow kernel (parser + copier warp per stream)
                                 {"B200LZ4_DWIDE": "1"}],       # every decode through the wide kernel (8 parsers + 7 copiers per stream)
                         ids=["narrow", "wide"])
def test_decoder_parity_with_forced_kernel(ctx, env):
    """The decoder has two kernels chosen by the number of streams in a launch; both must make the reference's
    accept/reject decisions and produce its bytes on every fuzz and edge case."""
    e = dict(os.environ, **env)
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", *DECODE_SUBSET], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert out.returncode == 0, out.stdout[-3000:]
    assert " passed" in out.stdout


@pytest.mark.parametrize("env", [{"B200LZ4_NO_WIDE": "1", "B200LZ4_COMPACT": "1"},      # everything through the compact-table kernel
                                 {"B200LZ4_NO_WIDE": "1", "B200LZ4_COMPACT": "0"}],     # everything through the classic dense kernel
                         ids=["compact", "classic"])
def test_parity_with_forced_kernel(ctx, env):
    e = dict(os.environ, **env)
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", *SUBSET], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:]
    assert " passed" in out.stdout


def test_decoder_bounds_checked_build_on_malformed_input(ctx):
    """compute-sanitizer is not available on the GPU pool, so memory safety of the decoders on hostile input is shown with
    a debug build (make bounds: -DB200LZ4_BOUNDS_CHECK) that checks every destination range against the block capacity
    and traps on a violation: the hand-built, corrupted and malformed-block tests and the copy-path geometry cases run
    through it, narrow and wide."""
    lib = os.path.join(ROOT, "streamly_lz4_b200", "libb200lz4_bounds.so")
    if not os.path.exists(lib):
        pytest.skip("libb200lz4_bounds.so not built (make bounds)")
    for wide in ("0", "1"):
        e = dict(os.environ, B200LZ4_LIB=lib, B200LZ4_DWIDE=wide)
        out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "tests/test_gpu_fuzz.py", "tests/test_gpu_parity.py",
                              "tests/test_gpu_device_abi.py", "tests/test_gpu_decode_geometry.py",
                              "-k", "handbuilt or corrupted or malformed or edge_sizes or echoing or (device_abi and decompress_dev) or "
                              "decode_geometry"],
                             cwd=ROOT, env=e,
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
        assert out.returncode == 0, out.stdout[-3000:]
        assert " passed" in out.stdout
