"""The dense finder's one-literal restart (compress.cu retest_run): after a re-test miss at p, probe 0 of the next search
run at p+1 is taken inside the re-test loop, with its one-byte catch-up, and a miss there hands the run to the probe
windows at probe 1.  Blocks are checked byte for byte against the reference, in the classic kernel (compress_dev with
more streams than SMs) and in the streamed kernel (a streamed host batch whose finders wait for every segment).

The inputs are records: a template of R bytes repeated with mutations at drifting offsets.  A record whose mutation
sits at the offset of the previous one's is a re-test miss at the mutated byte followed by a hit at the next byte (the
previous record inserted that position); two adjacent mutations make a miss on both probes, so the run goes on in the
probe windows at probe 1; a mutated byte equal to its left neighbour in the template gives the restart a one-byte
catch-up; a record without mutations is a match of R bytes (32+ when R >= 32).  Gaps of filler push candidates below
the 512-byte ring, and a copy of the block's head 65 536 bytes later offers a candidate just out of reach.  Runs of
restarts leave the queue at varying fill levels, and blocks cut at every length from 2000 to 2063 end runs at every offset
before mflimit and matchlimit.  datagen's records and sparse01 are run at sizes from 1 byte to 4 MiB."""
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

from test_gpu_device_abi import bound, dev, framed, kernel_streams, place, ref_compress  # noqa: F401  (dev: fixture)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ACCELS = [1, 2, 17, 400, 65537]


def restart_records(rng, n, far=False):
    """n bytes of mutated records (see the module docstring)."""
    R = int(rng.choice([int(rng.integers(12, 32)), int(rng.integers(32, 90))]))
    rec = bytearray(rng.integers(0, 256, size=R, dtype=np.uint8).tobytes())
    out = bytearray(rng.integers(0, 256, size=int(rng.integers(8, 300)), dtype=np.uint8).tobytes())
    k = int(rng.integers(1, R - 2))
    while len(out) < n:
        new = bytearray(rec)
        r = rng.random()
        offs = [k] if r < 0.6 else [k, k + 1] if r < 0.8 else [] if r < 0.9 else [k, int(rng.integers(1, R - 1))]
        for j in offs:
            new[j] = new[j - 1] if rng.random() < 0.3 else int(rng.integers(0, 256))
        out += new
        if rng.random() < 0.15:
            k = min(max(1, k + int(rng.integers(-1, 2))), R - 3)
        if rng.random() < 0.5:
            rec = new
        if far and rng.random() < 0.02:
            out += rng.integers(0, 256, size=int(rng.integers(600, 2000)), dtype=np.uint8).tobytes()
    if n > 65536 + 600 and far:          # the head again, 65 536 bytes on: its candidates are one byte out of reach
        out[65536:65536 + 512] = out[0:512]
    return bytes(out[:n])


def hand_built(rng, count):
    out = []
    for i in range(count):
        if i % 3 == 0:
            n = 2000 + (i // 3) % 64
        elif i % 7 == 1:
            n = int(rng.integers(66000, 140000))
        else:
            n = int(rng.integers(3000, 30000))
        out.append(restart_records(rng, n, far=bool(i & 2)))
    return out


def check_classic(dev, ref, arrays, accel):  # noqa: F811
    n = len(arrays)
    rng = np.random.default_rng(n)
    src, src_off, lens = place(arrays, "aligned", rng)
    caps = np.array([bound(len(a)) for a in arrays], dtype=np.int32)
    dst_off = np.zeros(n, dtype=np.int64)
    dst_off[1:] = np.cumsum((caps[:-1].astype(np.int64) + 15) // 16 * 16)
    out = dev.zeros(int(dst_off[-1]) + int(caps[-1]) + 64)
    out_len = dev.zeros(n, dev.torch.int32)
    dev.compress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), None, out_len, 0, accel=accel)
    dev.sync_and_check_scratch()
    want = ref_compress(ref, arrays, np.arange(n + 1, dtype=np.int32), accel=accel)
    got_len, got = dev.get(out_len), dev.get(out)
    for i, w in enumerate(want):
        o = int(dst_off[i])
        assert got_len[i] == len(w), f"block {i} (n={len(arrays[i])}, accel {accel}): out_len {got_len[i]}, reference {len(w)}"
        assert got[o:o + len(w)].tobytes() == framed(w, len(arrays[i]), 0), f"block {i} (n={len(arrays[i])}, accel {accel})"


@pytest.mark.parametrize("accel", ACCELS)
def test_restarts_in_classic_kernel_match_reference(dev, ref, accel):  # noqa: F811
    rng = np.random.default_rng(zlib.crc32(f"restart {accel}".encode()))
    check_classic(dev, ref, hand_built(rng, kernel_streams(dev, "classic")), accel)


@pytest.mark.parametrize("accel", [1, 400])
@pytest.mark.parametrize("kind", ["records", "sparse01"])
def test_generated_blocks_of_every_size_match_reference(dev, ref, kind, accel):  # noqa: F811
    from streamly_lz4_b200 import datagen
    sizes = [1, 5, 12, 13, 64, 127, 128, 129, 1000, 2047, 4096, 65535, 65536, 65537, 100003, 640000, 4 << 20]
    arrays = [datagen.make(kind, 50 + i, s).tobytes() for i, s in enumerate(sizes)]
    count = kernel_streams(dev, "classic")
    arrays = (arrays * (count // len(arrays) + 1))[:count]
    check_classic(dev, ref, arrays, accel)


STREAMED_BODY = r"""
import sys
import numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import streamly_lz4_b200 as lz
from oracle.oracle import Oracle
from test_gpu_retest_exits import restart_records
ctx = lz.Context(0)
ref = Oracle("auto")
L, n = 640000, 160
rng = np.random.default_rng(7)
distinct = [restart_records(rng, L, far=bool(i & 1)) for i in range(16)]
arrays = [distinct[i %% 16] for i in range(n - 1)] + [distinct[3][:%(last)d]]
buf = ctx.pinned("s_src", n * L + 64)[:n * L + 64]
buf[:] = 0xEE
for i, a in enumerate(arrays):
    buf[i * L:i * L + len(a)] = np.frombuffer(a, dtype=np.uint8)
offs = np.arange(n, dtype=np.int64) * L
lens = np.array([len(a) for a in arrays], dtype=np.int32)
dst = ctx.pinned("s_dst", int(sum(l + l // 255 + 16 + 8 + 32 for l in lens)))
for accel in %(accels)r:
    rc, doff, olen = ctx.compress_batch(buf, offs, lens, accel, 8, dst)
    assert rc == 0, ctx.last_error()
    want = ref.compress_chunks(arrays, accel, linked=False, threads=8)
    bad = [i for i in range(n) if dst[int(doff[i]):int(doff[i]) + 8 + int(olen[i])].tobytes() != want[i]]
    print("@@ accel", accel, "differs on", len(bad), "of", n, "blocks", bad[:20], flush=True)
ctx.close()
"""


def test_restarts_in_streamed_kernel_match_reference():
    """Segment-major arrival in 16 segments: every finder waits at every segment boundary."""
    e = dict(os.environ, B200LZ4_DEBUG="1", B200LZ4_STREAM_W="1000", B200LZ4_STREAM_S="16")
    accels = [1, 17, 400, 65537]
    out = subprocess.run([sys.executable, "-c", STREAMED_BODY % {"root": ROOT, "last": 2031, "accels": accels}],
                         cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    log = out.stdout
    if "[b200lz4] streamed: G" not in log:
        m = re.search(r"hardware queues: (\d+) of", log)
        if m and int(m.group(1)) < 2:
            pytest.skip("this platform gave the library fewer than two kernel queues independent of the copy queues: "
                        "streamed calls are off by design")
    assert out.returncode == 0, log[-4000:]
    assert "gave up" not in log, "finders timed out waiting for their input"
    assert len(re.findall(r"\[b200lz4\] streamed: G", log)) == len(accels), log[-4000:]
    for a in accels:
        assert f"@@ accel {a} differs on 0 of 160 blocks" in log, log[-4000:]
