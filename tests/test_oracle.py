"""CPU tests: pin the oracle.

1. The restatement (oracle/lz4_oracle.c) must reproduce the committed golden vectors, which
   are outputs of the reference's codec (tests/golden/make_golden.py).
2. On fresh seeded inputs, including the hash-table-dependent linked mode and the decoder's
   accept/reject decisions on corrupted blocks, the restatement must equal the reference's codec:
   its stored digests (tests/golden/reference_checks.json), and byte for byte a live reference
   build wherever one is present (oracle/_ref/libreflz4.so).
3. The Haskell-level logic restated in Python (resize, headers) must satisfy the properties
   of test/Main.hs:189-245.
"""
import hashlib
import importlib.util
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(golden)
GOLDEN = golden.load("golden.json")
CHECKS = golden.load("reference_checks.json")


def live_reference():
    from oracle.oracle import Oracle, available
    return Oracle("reference") if available("reference") else None


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=[c["name"] for c in GOLDEN["cases"]])
def test_port_matches_golden(port, case):
    golden.check_golden_case(port, case)


def test_reference_matches_golden_when_present(built):
    ref = live_reference()
    if ref is None:
        pytest.skip("reference build not present on this box")
    for case in GOLDEN["cases"]:
        framed = ref.compress_chunks(golden.arrays_of(case), case["accel"], block_size=case["block_size"], linked=case["linked"])
        assert golden.sha(framed) == case["framed_sha256"], case["name"]


@pytest.mark.parametrize("kind", golden.KINDS)
def test_port_equals_reference(built, port, kind):
    ref = live_reference()
    stored = CHECKS["configs"][kind]
    assert [(c["block"], c["accel"], c["linked"]) for c in stored] == golden.CONFIGS
    for want in stored:
        bs, accel, linked = want["block"], want["accel"], want["linked"]
        arrays = golden.config_arrays(kind, bs)
        assert golden.sha(arrays) == want["input_sha256"], "data generator drifted"
        b = port.compress_chunks(arrays, accel, linked=linked)
        assert golden.sha(b) == want["framed_sha256"], (kind, bs, accel, linked)
        assert port.decompress_chunks_raw(b, linked=linked) == arrays
        if ref is not None:
            a = ref.compress_chunks(arrays, accel, linked=linked)
            assert a == b, (kind, bs, accel, linked)
            assert ref.decompress_chunks_raw(b, linked=linked) == arrays


def test_port_equals_reference_edge_sizes(built, port):
    ref = live_reference()
    trials = golden.edge_size_trials()
    assert len(trials) == len(CHECKS["edge_size_trials"])
    for (arrays, accel), want in zip(trials, CHECKS["edge_size_trials"]):
        b = port.compress_chunks(arrays, accel, linked=True)
        assert golden.sha(b) == want, ([len(a) for a in arrays], accel)
        if ref is not None:
            assert ref.compress_chunks(arrays, accel, linked=True) == b, ([len(a) for a in arrays], accel)
        assert port.decompress_chunks_raw(b, linked=True) == arrays


def test_acceleration_clamp(port):
    """cbits/lz4.c:1577-1578: -5,-1,0,1 coincide; 65537, 65538, 10**6 coincide (SURVEY.md section 0.5)."""
    from streamly_lz4_b200 import datagen
    d = datagen.make("mixed", 3, 1 << 20)
    arrays = [d[i:i + 100000].tobytes() for i in range(0, d.size, 100000)]
    low = [port.compress_chunks(arrays, a) for a in (-5, -1, 0, 1)]
    assert all(x == low[0] for x in low)
    high = [port.compress_chunks(arrays, a) for a in (65537, 65538, 10 ** 6)]
    assert all(x == high[0] for x in high)
    assert low[0] != high[0]


def test_decoder_accept_reject_agrees_with_reference(built, port):
    ref = live_reference()
    d = golden.decoder_input()
    payload = port.compress_chunks([d], 1, linked=False)[0][8:]
    assert hashlib.sha256(payload).hexdigest() == CHECKS["decoder"]["payload_sha256"]
    blocks = golden.corrupted_blocks(payload, len(d))
    want = CHECKS["decoder"]["verdicts"]
    assert len(blocks) == len(want) and want.count(None) > 0
    for i, (arr, w) in enumerate(zip(blocks, want)):
        got = golden.decode_verdict(port, arr)
        assert got == w, f"corrupted block {i}: restatement {'rejects' if got is None else 'accepts'} it, the reference did not"
        if ref is not None:
            assert golden.decode_verdict(ref, arr) == got, f"corrupted block {i}"


@pytest.mark.parametrize("section", ["single", "linked"])
def test_port_limited_output_agrees_with_reference(built, port, section):
    """LZ4_compress_fast_continue with dstCapacity r - 1 and r (r = the size at the bound), on inputs shaped at each of the
    three limitedOutput guards: the restatement must give upstream's sizes, verdicts and bytes and never write past
    dstCapacity.  Only the first capacity-limited call of a stream is pinned: after a failure lz4.h leaves the state
    undefined."""
    want = CHECKS["limited"]
    pairs = ([(None, a) for a in golden.limited_inputs()] if section == "single" else golden.limited_linked_inputs())
    rows, digest = golden.limited_results(port, pairs)
    assert len(rows) == len(want[section])
    for i, (got, w) in enumerate(zip(rows, want[section])):
        assert got == w, f"{section} input {i}: restatement {got}, upstream {w} ([r, at r - 1, at r])"
    assert digest == want[f"{section}_payload_sha256"]
    assert all(r1 == 0 and rr == r for r, r1, rr in rows)      # success exactly when the payload fits
    ref = live_reference()
    if ref is not None:
        assert golden.limited_results(ref, pairs) == (rows, digest)


# ---- resizeChunksD restatement (pure Python) --------------------------------------------------

def _framed(port, n_arrays=20, bs=5000):
    from streamly_lz4_b200 import datagen
    d = datagen.make("biased01", 2, n_arrays * bs)
    arrays = [d[i:i + bs].tobytes() for i in range(0, d.size, bs)]
    return arrays, port.compress_chunks(arrays, 1)


@pytest.mark.parametrize("bufsize", [1, 7, 512, 4000, 32 * 1024, 256 * 1024])
def test_resize_restatement_refragments(port, bufsize):
    from oracle.oracle import resize_chunks
    arrays, framed = _framed(port)
    blob = b"".join(framed)
    chunks = [blob[i:i + bufsize] for i in range(0, len(blob), bufsize)]
    assert resize_chunks(chunks) == framed
    assert resize_chunks(resize_chunks(chunks)) == framed            # idempotent, test/Main.hs:189-201


def test_resize_restatement_end_mark_and_errors(port):
    from oracle.oracle import resize_chunks
    arrays, framed = _framed(port, 5, 1000)
    blob = b"".join(framed)
    with_mark = blob + b"\0\0\0\0" + b"trailing garbage is ignored"
    assert resize_chunks([with_mark], has_end_mark=True) == framed   # test/Main.hs:234-243
    with pytest.raises(RuntimeError, match="No end mark"):
        resize_chunks([blob], has_end_mark=True)
    with pytest.raises(RuntimeError, match="Incomplete block"):
        resize_chunks([blob[:-3]])
    assert resize_chunks([]) == []


def test_xxh32_known_answers(built):
    """XXH32 restated in oracle/lz4_oracle.c against published known answers, and the frame-header checksum bytes of the
    headers the stock `lz4` tool writes (04 22 4D 18 60 40 82 / 64 40 A7 / 64 70 B9)."""
    from oracle import frame
    assert frame.xxh32(b"") == 0x02CC5D05
    assert frame.xxh32(b"a") == 0x550D7456
    assert frame.xxh32(b"abc") == 0x32D153FF
    assert frame.xxh32(b"Nobody inspects the spammish repetition") == 0xE2293B2F
    for desc, hc in ((b"\x60\x40", 0x82), (b"\x64\x40", 0xA7), (b"\x64\x70", 0xB9)):
        assert (frame.xxh32(desc) >> 8) & 0xFF == hc
    assert frame.header(4, independent=True, content_checksum=True).hex() == "04224d186440a7"


def test_frame_restatement_round_trips(built):
    """oracle/frame.py: encode -> parse -> decode over every flag combination, stored (incompressible) blocks included;
    corrupted checksums are rejected."""
    import numpy as np
    from oracle import frame
    from oracle.oracle import Oracle
    from streamly_lz4_b200 import datagen
    ora = Oracle("auto")
    data = datagen.make("mixed", 17, 5 * 65536 + 1234).tobytes()
    arrays = [data[i:i + 65536] for i in range(0, len(data), 65536)]
    for ind in (False, True):
        for bc in (False, True):
            for cs in (False, True):
                for cc in (False, True):
                    blob = frame.encode(ora, arrays, 4, 1, ind, bc, cs, cc)
                    d, blocks, _ = frame.parse(blob)
                    assert d["frame_bytes"] == len(blob) and len(blocks) == len(arrays)
                    assert any(stored for stored, _ in blocks)              # the random segment is stored uncompressed
                    assert frame.decode(ora, blob) == data
    blob = bytearray(frame.encode(ora, arrays, 4, 1, False, True, False, True))
    blob[40] ^= 1
    with pytest.raises(ValueError):
        frame.decode(ora, bytes(blob))
