"""Streamed host call (csrc/api.cu: compress_host_streamed, schedule in csrc/host_plan.h; compress.cu: kStreamed): a batch of equally long independent
blocks at a constant pitch is sent to the device segment by segment in deadline order, and the finders run while their
blocks are still arriving.  The bytes must be the reference's whatever the order of arrival: every schedule extreme
(plain block order, segment-major, the tuned default), each way of raising the arrival flags and of sending the decoded
output home, host pitches with gaps, a short last block, and the SAME device
addresses reused by consecutive calls with different data (a 32-byte L1 sector read before it has landed would show up
as the previous call's bytes)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _batch(ctx, kind, seed, n_blocks, block, pitch, last):
    """n_blocks blocks of `block` bytes (the last one `last` bytes) at host pitch `pitch` in one pinned buffer"""
    from streamly_lz4_b200 import datagen
    lens = np.full(n_blocks, block, dtype=np.int32)
    lens[-1] = last
    offs = (np.arange(n_blocks, dtype=np.int64) * pitch)
    buf = ctx.pinned("s_src", int(offs[-1]) + block + 64)[:int(offs[-1]) + block + 64]
    buf[:] = 0xEE
    data = datagen.make(kind, seed, n_blocks * block)
    rows = np.lib.stride_tricks.as_strided(buf, shape=(n_blocks, block), strides=(pitch, 1))
    rows[:, :] = data.reshape(n_blocks, block)
    return buf, offs, lens, data


def _check(ctx, ref, kind, seed, n_blocks, block, pitch, last, accel):
    buf, offs, lens, data = _batch(ctx, kind, seed, n_blocks, block, pitch, last)
    bound = int(sum(int(l) + int(l) // 255 + 16 + 8 + 32 for l in lens))
    dst = ctx.pinned("s_dst", bound)
    rc, doff, olen = ctx.compress_batch(buf, offs, lens, accel, 8, dst)
    assert rc == 0, ctx.last_error()
    assert (olen > 0).all()
    arrays = [data[i * block:i * block + int(lens[i])].tobytes() for i in range(n_blocks)]
    want = ref.compress_chunks(arrays, accel, linked=False, threads=os.cpu_count() or 8)
    bad = [i for i in range(n_blocks) if dst[int(doff[i]):int(doff[i]) + 8 + int(olen[i])].tobytes() != want[i]]
    assert not bad, f"{len(bad)} of {n_blocks} blocks differ from the reference ({kind}, accel {accel}): {bad[:20]}"
    # the whole stream decodes back
    back = ctx.pinned("s_back", int(lens.astype(np.int64).sum()) + 64)
    c_off = doff[:-1].copy()
    c_len = (olen + 8).astype(np.int32)
    rc2, boff, blen = ctx.decompress_batch(dst, c_off, c_len, 8, 0, back)
    assert rc2 == 0, ctx.last_error()
    assert (blen == lens).all()
    for i in range(n_blocks):
        assert np.array_equal(back[int(boff[i]):int(boff[i]) + int(lens[i])], data[i * block:i * block + int(lens[i])]), i


BODY = r"""
import sys, numpy as np
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(root)r + "/tests")
import streamly_lz4_b200 as lz
from oracle.oracle import Oracle
from test_gpu_streamed import _check
ctx = lz.Context(0)
ref = Oracle("auto")
n = 170
# three consecutive calls on one ctx: same shapes and device addresses, different data and schedules tuned by the
# previous call's measurements
_check(ctx, ref, "mixed", 11, n, 640000, 640000, 640000, 400)
_check(ctx, ref, "text", 12, n, 640000, 640000, 123457, 1)
_check(ctx, ref, "mixed", 13, n, 640000, 640016, 5, 400)
_check(ctx, ref, "sparse01", 14, n, 640000, 650000, 640000, 7)
_check(ctx, ref, "random", 15, n, 640000, 640000, 639999, 400)
_check(ctx, ref, "zero", 16, n, 640000, 640000, 640000, 1)
# other block sizes: not a multiple of 128, and 4 MiB
_check(ctx, ref, "records", 17, 1100, 100003, 100003, 77, 3)
_check(ctx, ref, "mixed", 18, 97, 4194304, 4194304, 4194304, 400)
print("launches", ctx.launch_count())
ctx.close()
print("streamed ok")
"""


@pytest.mark.parametrize("env", [{}, {"B200LZ4_STREAM_W": "0"}, {"B200LZ4_STREAM_W": "1000"},
                                 {"B200LZ4_STREAM_W": "0.7", "B200LZ4_STREAM_G": "5", "B200LZ4_STREAM_S": "13"},
                                 {"B200LZ4_STREAM_FLAG": "copy", "B200LZ4_DECODE_OUT": "mirror"},
                                 {"B200LZ4_STREAM_FLAG": "kernel", "B200LZ4_DECODE_OUT": "copy"},
                                 {"B200LZ4_NO_STREAMED": "1"}],
                         ids=["tuned", "block-order", "segment-major", "odd-geometry", "flag-copies+mirror", "flag-kernels+copy", "plain-pipeline"])
def test_streamed_call_is_byte_identical(ctx, ref, env):
    e = dict(os.environ, B200LZ4_DEBUG="1", **env)
    out = subprocess.run([sys.executable, "-c", BODY % {"root": ROOT}], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "streamed ok" in out.stdout
    took_streamed_path = "[b200lz4] streamed:" in out.stdout
    if "B200LZ4_NO_STREAMED" not in env and not took_streamed_path:
        import re
        m = re.search(r"hardware queues: (\d+) of", out.stdout)
        if m and int(m.group(1)) < 2:       # measured by the library at ctx creation (api.cu: probe_stream_aliasing)
            pytest.skip("this platform gave the library fewer than two kernel queues independent of the copy queues: "
                        "streamed calls are off by design; the bytes above were verified through the plain pipeline")
    assert took_streamed_path == ("B200LZ4_NO_STREAMED" not in env), out.stdout[-2000:]
    assert "gave up" not in out.stdout, "finders timed out waiting for their input: the call fell back to the plain pipeline"
