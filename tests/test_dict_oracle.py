"""Shared dictionaries on the CPU: the restatement given a dictionary (tests/golden/dict_golden.py: Port, i.e.
oracle/lz4_oracle.c with its stream records set up by a restatement of LZ4_loadDict / LZ4_setStreamDecode) reproduces
what upstream LZ4 stored in tests/golden/dict_checks.json -- LZ4_loadDict compression digests, the verdicts of
LZ4_decompress_safe_usingDict on corrupted and boundary blocks, and two LZ4F frames with a dictionary id.  The reference
build (oracle/_ref) is checked the same way where it exists."""
import base64
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

import dict_golden as dg  # noqa: E402
from oracle import frame  # noqa: E402

CHECKS = dg.load()


@pytest.fixture(scope="module", params=range(len(dg.codecs())), ids=lambda i: ["port", "reference"][i])
def codec(request, built):
    return dg.codecs()[request.param]


@pytest.mark.parametrize("cfg", dg.DICT_CONFIGS, ids=[c[0] for c in dg.DICT_CONFIGS])
def test_dict_compress_digests(codec, cfg):
    name, sizes, accel, linked = cfg
    for kind in dg.KINDS:
        prefix, arrays = dg.dict_inputs(kind, sizes)
        for dl in dg.DICT_LENS:
            dic = dg.dict_of(prefix, dl)
            framed = codec.compress_chunks(arrays, accel, linked=linked, dictionary=dic)
            assert dg.sha(framed) == CHECKS["digests"][f"{kind}/{name}/{dl}"], (kind, name, dl)
            assert codec.decompress_chunks_raw(framed, linked=linked, dictionary=dic) == arrays, (kind, name, dl)


def test_dict_decoder_verdicts(codec):
    cases = dg.dict_decoder_cases(codec)
    assert len(cases) == len(CHECKS["decoder_verdicts"])
    for i, ((dic, framed), want) in enumerate(zip(cases, CHECKS["decoder_verdicts"])):
        assert codec.decode_verdict(dic, framed) == want, f"case {i}"


@pytest.mark.parametrize("name", [f[0] for f in dg.DICT_FRAMES])
def test_dict_stock_frames(codec, name):
    f = CHECKS["frames"][name]
    prefix, arrays = dg.dict_inputs("text", dg.DICT_FRAME_SIZES)
    assert dg.sha(arrays) == f["input_sha256"]
    blob = base64.b64decode(f["frame_b64"])
    d, _, _ = frame.parse(blob)
    assert d["dict_id"] == f["dict_id"] and d["independent"] == f["independent"]
    assert dg.frame_decode(codec, blob, dg.dict_of(prefix, 65536)) == b"".join(arrays)
    with pytest.raises((ValueError, RuntimeError)):     # without the dictionary: a match reaches before the output, or the checksum fails
        dg.frame_decode(codec, blob)


def test_load_dict_table_rules():
    """LZ4_loadDict's rules as restated: nothing below 8 bytes, only the last 64 KiB, every third position that has 8
    bytes behind it, index 65536 - distance to the end, the last position of a bucket stays."""
    t, n = dg.load_dict_table(b"abcdefg")
    assert n == 0 and not t.any()
    t, n = dg.load_dict_table(b"abcdefgh")
    assert n == 8 and np.count_nonzero(t) == 1 and t.max() == 65536 - 8
    rng = np.random.default_rng(3)
    big = rng.integers(0, 256, 70000, dtype=np.uint8).tobytes()
    t1, n1 = dg.load_dict_table(big)
    t2, n2 = dg.load_dict_table(big[-65536:])
    assert n1 == n2 == 65536 and np.array_equal(t1, t2)
    # a plain loop in position order, last writer wins
    tail = np.frombuffer(big[-65536:], dtype=np.uint8)
    want = np.zeros(4096, dtype=np.uint32)
    pos = np.arange(0, 65536 - 7, 3)
    for p, h in zip(pos, dg.hash5(tail, pos)):
        want[h] = 65536 - (65536 - p)
    assert np.array_equal(t1, want)
