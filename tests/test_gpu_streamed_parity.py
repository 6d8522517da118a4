"""Streamed host calls checked on EVERY block (csrc/api.cu: compress_host_streamed / decompress_host_streamed).

Compress.  The streamed kernel is the only one that reads its input while DMA is still writing it; a wrong arrival gate
(compress.cu: wait_for / count_ahead) gives a valid but different parse -- a missed or shortened match -- that a round trip
cannot see.  So every block of every call below is compared byte for byte with the reference (the `ref` fixture), and with
a dictionary against the restatement that reproduces upstream's dictionary output (tests/golden/dict_golden.py: Port).
Each schedule runs in a child process: it starts from a fresh ctx, and its consecutive calls on that ctx tune each other.

  schedule (env)              calls: kind, block length L, host pitch, last-block length, acceleration
  tuned                       mixed   640 000  pitch L    last L      accel 1
                              text    640 000  pitch L+5  last L-1    accel 2
                              mixed   640 000  pitch L    last L      accel 400    with a 64 KiB dictionary (retest_probe)
  block order (W=0)           sparse01 100 003 pitch L    last 129    accel 400
                              zero    65 536   pitch L+5  last 128    accel 1
  segment-major (W=1000 S=16) random  640 000  pitch L    last 127    accel 65537
                              bits01  640 000  pitch L+5  last 13     accel 1
                              records 100 003  pitch L    last 12     accel 2
                              text    640 000  pitch L    last 1      accel 1      with a 64 KiB dictionary
  one group, one segment      mixed   65 536   pitch L    last 1      accel 400
    (G=1 S=1)                 text    640 000  pitch L    last L      accel 1
  odd geometry (G=16 S=13)    bits01  100 003  pitch L+5  last L      accel 1
                              mixed   4 MiB    pitch L    last L-1    accel 2
  flags by inline copies      records 640 000  pitch L    last 129    accel 1
  flags by kernels            sparse01 65 536  pitch L+5  last 1      accel 65537

Segment-major with 16 segments starves every finder at every segment boundary (all finders together consume faster than
the link delivers); fast data (zero, sparse01, random at high acceleration) reaches the arrival front soonest.  Every call
must have taken the streamed path and no finder may have given up waiting; the cases are skipped only where the library
measured fewer than two kernel queues independent of the copy queues (streamed calls are off by design there).

Decompress.  A failing block never aborts a batch: it reports out_len < 0 and the call B200LZ4_E_BLOCK.  Batches in the
streamed shape (120 blocks of 1 MiB, header mode 8, the same uncompLen everywhere) with blocks the reference rejects (bit
flips) and blocks that decode to fewer than L bytes, at block 0, the last block, both sides of group boundaries and
filling one whole group, go through each output route: pieces (decompress_host_streamed, whose copier must still raise
every segment flag of a block that ended early), mirror, copy and the plain pipeline."""
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from test_gpu_dict import dref  # noqa: F401  (the restatement, once it has reproduced upstream's dictionary output)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THREADS = os.cpu_count() or 8
E_BLOCK = -4
MiB = 1 << 20

# kind, seed, blocks, L, pitch, last-block length, acceleration, with a dictionary
SCHEDULES = {
    "tuned": ({}, [
        ("mixed", 31, 170, 640000, 640000, 640000, 1, False),
        ("text", 32, 170, 640000, 640005, 639999, 2, False),
        ("mixed", 33, 170, 640000, 640000, 640000, 400, True)]),
    "block-order": ({"B200LZ4_STREAM_W": "0"}, [
        ("sparse01", 34, 1007, 100003, 100003, 129, 400, False),
        ("zero", 35, 1536, 65536, 65541, 128, 1, False)]),
    "segment-major": ({"B200LZ4_STREAM_W": "1000", "B200LZ4_STREAM_S": "16"}, [
        ("random", 36, 170, 640000, 640000, 127, 65537, False),
        ("bits01", 37, 170, 640000, 640005, 13, 1, False),
        ("records", 38, 1007, 100003, 100003, 12, 2, False),
        ("text", 39, 170, 640000, 640000, 1, 1, True)]),
    "one-group-one-segment": ({"B200LZ4_STREAM_G": "1", "B200LZ4_STREAM_S": "1"}, [
        ("mixed", 40, 1536, 65536, 65536, 1, 400, False),
        ("text", 41, 170, 640000, 640000, 640000, 1, False)]),
    "odd-geometry": ({"B200LZ4_STREAM_G": "16", "B200LZ4_STREAM_S": "13"}, [
        ("bits01", 42, 1007, 100003, 100008, 100003, 1, False),
        ("mixed", 43, 96, 4 * MiB, 4 * MiB, 4 * MiB - 1, 2, False)]),
    "flag-copies": ({"B200LZ4_STREAM_FLAG": "copy"}, [
        ("records", 44, 170, 640000, 640000, 129, 1, False)]),
    "flag-kernels": ({"B200LZ4_STREAM_FLAG": "kernel"}, [
        ("sparse01", 45, 1536, 65536, 65541, 1, 65537, False)]),
}


def compress_every_block(ctx, ref, dref, kind, seed, n, L, pitch, last, accel, with_dict):
    """One streamed-shape batch through ctx.compress_batch; returns the indices of blocks whose framed bytes differ from
    the reference's (with_dict: a 64 KiB dictionary, checked against dref)."""
    from test_gpu_streamed import _batch
    import dict_golden as mg
    buf, offs, lens, data = _batch(ctx, kind, seed, n, L, pitch, last)
    bound = int(sum(int(l) + int(l) // 255 + 16 + 8 + 32 for l in lens))
    dst = ctx.pinned("s_dst", bound)
    arrays = [data[i * L:i * L + int(lens[i])].tobytes() for i in range(n)]
    if with_dict:
        dic = mg.dict_of(mg.dict_inputs(kind, [1])[0], 65536)
        d = ctx.dictionary(dic)
        rc, doff, olen = ctx.compress_batch(buf, offs, lens, accel, 8, dst, None, None, d)
        want = dref.compress_chunks(arrays, accel, linked=False, dictionary=dic)
    else:
        rc, doff, olen = ctx.compress_batch(buf, offs, lens, accel, 8, dst)
        want = ref.compress_chunks(arrays, accel, linked=False, threads=THREADS)
    assert rc == 0, ctx.last_error()
    return [i for i in range(n) if dst[int(doff[i]):int(doff[i]) + 8 + int(olen[i])].tobytes() != want[i]]


COMPRESS_BODY = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests"); sys.path.insert(0, %(root)r + "/tests/golden")
import streamly_lz4_b200 as lz
import dict_golden as mg
from oracle.oracle import Oracle
from test_gpu_streamed_parity import compress_every_block
ctx = lz.Context(0)
ref, dref = Oracle("auto"), mg.Port()
for k, call in enumerate(%(calls)r):
    print("@@ call", k, call, file=sys.stderr, flush=True)
    bad = compress_every_block(ctx, ref, dref, *call)
    print("@@ call", k, "differs on", len(bad), "of", call[2], "blocks", bad[:20], file=sys.stderr, flush=True)
ctx.close()
"""


def _queues_skip(log):
    m = re.search(r"hardware queues: (\d+) of", log)
    if m and int(m.group(1)) < 2:       # measured by the library at ctx creation (api.cu: probe_stream_aliasing)
        pytest.skip("this platform gave the library fewer than two kernel queues independent of the copy queues: "
                    "streamed calls are off by design")


@pytest.mark.parametrize("schedule", list(SCHEDULES))
def test_streamed_compress_every_block_is_the_reference(ctx, ref, dref, schedule):  # noqa: F811
    env, calls = SCHEDULES[schedule]
    e = dict(os.environ, B200LZ4_DEBUG="1", **env)
    out = subprocess.run([sys.executable, "-c", COMPRESS_BODY % {"root": ROOT, "calls": calls}], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    log = out.stdout
    if "[b200lz4] streamed: G" not in log:
        _queues_skip(log)
    assert out.returncode == 0, log[-4000:]
    assert "gave up" not in log, "finders timed out waiting for their input: the call fell back to the plain pipeline"
    parts = log.split("@@ call ")[1:]
    assert len(parts) == 2 * len(calls), log[-4000:]
    for k, call in enumerate(calls):
        during, verdict = parts[2 * k], parts[2 * k + 1]
        assert f"differs on 0 of {call[2]} blocks" in verdict, f"{schedule} call {k} {call}: {verdict.strip()}"
        m = re.findall(r"\[b200lz4\] streamed: G (\d+) S (\d+) seg \d+ w ([\d.]+)", during)
        assert len(m) == 1, f"{schedule} call {k} {call} did not take the streamed path:\n{during[-2000:]}"
        G, S, w = int(m[0][0]), int(m[0][1]), float(m[0][2])
        if "B200LZ4_STREAM_G" in env:
            assert G == int(env["B200LZ4_STREAM_G"]), during
        if "B200LZ4_STREAM_S" in env:
            assert S == int(env["B200LZ4_STREAM_S"]), during
        if "B200LZ4_STREAM_W" in env:
            assert w == pytest.approx(min(float(env["B200LZ4_STREAM_W"]), G), abs=1e-3), during


# ---- decompress: failing blocks in streamed-shape batches --------------------------------------------------------------

DEC_N, DEC_L = 120, MiB          # 12 groups of 10 blocks (host_plan.h: decompress_geometry)
# block -> "flip" (payload bits flipped until the reference rejects it) or a length: a block that compresses only that many
# bytes under a header that still says L
DEC_LAYOUTS = {
    "ends-flipped": {0: "flip", 9: DEC_L - 1, 10: "flip", 29: "flip", 30: 4096, 89: 1, 90: "flip", 119: "flip",
                     **{i: "flip" for i in range(50, 60)}},
    "ends-short": {0: DEC_L // 2 + 3, 19: "flip", 20: DEC_L - 1, 119: 1,
                   **{i: ("flip" if i % 2 else 777) for i in range(70, 80)}},
}


def _verdict(ref, framed):
    """the reference's verdict on one framed block: its output, or None when it rejects the block"""
    try:
        return ref.decompress_chunks_raw([framed], linked=False)[0]
    except RuntimeError:
        return None


def _failing_batch(ref, layout, seed):
    from streamly_lz4_b200 import datagen
    rng = np.random.default_rng(seed)
    data = datagen.make("mixed", seed, DEC_N * DEC_L)
    arrays = [data[i * DEC_L:(i + 1) * DEC_L].tobytes() for i in range(DEC_N)]
    framed = ref.compress_chunks(arrays, 1, linked=False, threads=THREADS)
    want = ref.decompress_chunks_raw(framed, linked=False, threads=THREADS)
    assert want == arrays
    want = list(want)
    for i, what in DEC_LAYOUTS[layout].items():
        if what == "flip":
            for _ in range(200):
                b = bytearray(framed[i])
                for at in rng.integers(8, len(b), 4):
                    b[int(at)] ^= 1 << int(rng.integers(0, 8))
                if _verdict(ref, bytes(b)) is None:
                    break
            else:
                pytest.fail(f"no bit flip of block {i} that the reference rejects")
            framed[i], want[i] = bytes(b), None
        else:
            payload = ref.compress_chunks([arrays[i][:what]], 1, linked=False)[0][8:]
            framed[i] = len(payload).to_bytes(4, "little") + DEC_L.to_bytes(4, "little") + payload
            want[i] = _verdict(ref, framed[i])
            assert want[i] is not None and len(want[i]) == what
    blob = np.frombuffer(b"".join(framed), dtype=np.uint8)
    clen = np.array([len(f) for f in framed], dtype=np.int32)
    coff = np.zeros(DEC_N, dtype=np.int64)
    coff[1:] = np.cumsum(clen[:-1].astype(np.int64))
    want_len = np.array([-1 if w is None else len(w) for w in want], dtype=np.int32)
    want_sha = np.frombuffer(b"".join(bytes(32) if w is None else hashlib.sha256(w).digest() for w in want),
                             dtype=np.uint8).reshape(-1, 32)
    return blob, coff, clen, want_len, want_sha


@pytest.fixture(scope="module")
def failing_batches(ref, tmp_path_factory):
    """the batches and the reference's per-block verdicts (length, SHA-256 of the output), saved for the child processes"""
    d = tmp_path_factory.mktemp("failing_batches")
    paths = {}
    for k, layout in enumerate(DEC_LAYOUTS):
        blob, coff, clen, want_len, want_sha = _failing_batch(ref, layout, 60 + k)
        paths[layout] = str(d / f"{layout}.npz")
        np.savez(paths[layout], blob=blob, coff=coff, clen=clen, want_len=want_len, want_sha=want_sha)
    return paths


DECODE_BODY = r"""
import hashlib, sys
import numpy as np
sys.path.insert(0, %(root)r)
import streamly_lz4_b200 as lz
ctx = lz.Context(0)
for layout, path in %(paths)r.items():
    z = np.load(path)
    blob, coff, clen, want_len, want_sha = z["blob"], z["coff"], z["clen"], z["want_len"], z["want_sha"]
    src = ctx.pinned("d_src", blob.size); src[:blob.size] = blob
    back = ctx.pinned("d_back", len(clen) * %(L)d + 64)
    print("@@", layout, file=sys.stderr, flush=True)
    rc, boff, blen = ctx.decompress_batch(src[:blob.size], coff, clen, 8, 0, back)
    assert rc == %(E_BLOCK)d, (layout, rc, ctx.last_error())
    for i in range(len(clen)):
        assert (blen[i] < 0) == (want_len[i] < 0), (layout, i, int(blen[i]), int(want_len[i]))
        if want_len[i] >= 0:
            assert blen[i] == want_len[i], (layout, i, int(blen[i]), int(want_len[i]))
            got = back[int(boff[i]):int(boff[i]) + int(blen[i])]
            assert hashlib.sha256(got.tobytes()).digest() == want_sha[i].tobytes(), (layout, i, "output differs from the reference's")
ctx.close()
print("failing blocks ok")
"""

ROUTES = {"pieces": ({}, "[b200lz4] streamed decompress: G"),
          "mirror": ({"B200LZ4_DECODE_OUT": "mirror"}, "[b200lz4] decompress: mirror output"),
          "copy": ({"B200LZ4_DECODE_OUT": "copy"}, "[b200lz4] decompress: copy output"),
          "plain-pipeline": ({"B200LZ4_NO_STREAMED": "1"}, "[b200lz4] decompress: copy output")}


@pytest.mark.parametrize("route", list(ROUTES))
def test_failing_blocks_in_streamed_shape_decode_batches(ctx, failing_batches, route):
    """Every block gets the reference's verdict (its output, or out_len < 0) and the call B200LZ4_E_BLOCK, through each
    output route: the batch is never lost as a whole."""
    env, marker = ROUTES[route]
    e = dict(os.environ, B200LZ4_DEBUG="1", **env)
    body = DECODE_BODY % {"root": ROOT, "paths": failing_batches, "L": DEC_L, "E_BLOCK": E_BLOCK}
    out = subprocess.run([sys.executable, "-c", body], cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "failing blocks ok" in out.stdout
    for part in out.stdout.split("@@ ")[1:]:
        assert marker in part, f"{route} did not run for {part.splitlines()[0]}:\n{part[-2000:]}"
