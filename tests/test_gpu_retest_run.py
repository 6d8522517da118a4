"""The dense finder's run of re-tests (compress.cu retest_run) against the reference, byte for byte, on inputs built to
be long chains of zero-literal follow-up matches.  Each such chain leaves the finder's inner loop through one of its
exits: a queue buffer filled in the middle of a run (runs of more than 16 follow-ups), the ring window's edge (every
128 bytes), the last 32 bytes before matchlimit (block sizes that end a chain at every offset there), a candidate older
than the 512-byte ring (copies from far back), and matches of 32 bytes and more (long copies).  Every compressor kernel
runs the same inputs; only the classic and streamed ones take retest_run, the others check that the inputs mean the same
thing to them."""
import zlib

import numpy as np
import pytest

from test_gpu_device_abi import bound, dev, framed, kernel_streams, place, ref_compress  # noqa: F401  (dev: fixture)

pytestmark = pytest.mark.gpu


def segments(rng, n, short, far):
    """n bytes: a random head, then copies of earlier bytes, lengths 4..31 (short) or 32..300, taken from within the last
    120 bytes (in the ring) or from 600..4000 bytes back (older than the ring)."""
    head = int(rng.integers(64, 700))
    out = bytearray(rng.integers(0, 256, size=head, dtype=np.uint8).tobytes())
    while len(out) < n:
        length = int(rng.integers(4, 32)) if short else int(rng.integers(32, 301))
        lo, hi = (600, 4000) if far else (length, 120 + length)
        dist = int(rng.integers(min(lo, len(out)), min(hi, len(out)) + 1))
        start = len(out) - dist
        out += out[start:start + length]
    return bytes(out[:n])


def arrays_for(rng, count):
    """Chains of every flavour; every third block is cut at 2000 + k (k = 0..63), so that chains end at every offset
    before matchlimit."""
    out = []
    for i in range(count):
        short, far = bool(i & 1), bool(i & 2)
        n = 2000 + (i // 4) % 64 if i % 3 == 0 else int(rng.integers(3000, 20000))
        out.append(segments(rng, n, short, far))
    return out


@pytest.mark.parametrize("accel", [1, 400])
@pytest.mark.parametrize("kernel", ["classic", "compact", "wide"])
def test_follow_up_chains_match_reference(dev, ref, kernel, accel):  # noqa: F811
    rng = np.random.default_rng(zlib.crc32(f"retest {kernel} {accel}".encode()))
    arrays = arrays_for(rng, kernel_streams(dev, kernel))
    n = len(arrays)
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
    ratio = sum(len(a) for a in arrays) / sum(len(w) for w in want)
    if accel == 1:                         # (at 400 the search skips most copies: chains follow the few it finds)
        assert ratio > 2, f"the inputs are meant to be chains of matches (ratio {ratio:.2f})"
    for i, w in enumerate(want):
        o = int(dst_off[i])
        assert got_len[i] == len(w), f"block {i} (n={len(arrays[i])}): out_len {got_len[i]}, reference {len(w)}"
        assert got[o:o + len(w)].tobytes() == framed(w, len(arrays[i]), 0), f"block {i} (n={len(arrays[i])})"
