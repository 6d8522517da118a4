"""The golden LZ4 frames of tests/golden/frames (written and judged by upstream LZ4F, tests/golden/frame_golden.py): their
stored content digests match the data generator, and the frame checker oracle/frame.py gives upstream's verdict on every
frame it can express (CPU only)."""
import hashlib
import json
import os

import pytest

from streamly_lz4_b200 import datagen

HERE = os.path.dirname(os.path.abspath(__file__))
FRAMES = os.path.join(HERE, "golden", "frames")


def records():
    with open(os.path.join(FRAMES, "frames.json")) as fh:
        return json.load(fh)["frames"]


def test_golden_set_covers_the_cases():
    recs = records()
    names = {r["file"] for r in recs}
    assert sum(os.path.getsize(os.path.join(FRAMES, n)) for n in names) < (1 << 20)
    for code in (4, 5, 6, 7):
        for mode in ("ind", "lnk"):
            assert any(n.startswith(f"b{code}_{mode}_") for n in names)
    assert {r["code"] for r in recs} == {"ok", "frame", "checksum", "block"}
    assert any(r["upstream"] == "accept" and r["length"] == 0 for r in recs)
    assert any(n.startswith("flushed_") for n in names) and any(n.startswith("stored_") for n in names)


@pytest.mark.parametrize("rec", records(), ids=lambda r: r["file"])
def test_golden_content_digest(rec):
    data = datagen.make(rec["kind"], rec["seed"], rec["length"]).tobytes() if rec["length"] else b""
    assert hashlib.sha256(data).hexdigest() == rec["sha256"]


CODE = {"ok": None, "frame": -5, "checksum": -6, "block": -4}     # B200LZ4_E_FRAME, _CHECKSUM, _BLOCK


def test_oracle_agrees_with_upstream():
    """Every golden frame, the flushed ones (short linked blocks reached across by matches) included: the window reference
    accepts what upstream accepts with the same content, and its verdict is the code the C ABI must report."""
    from oracle import frame
    from oracle.oracle import Oracle
    ora = Oracle("auto")
    for rec in records():
        with open(os.path.join(FRAMES, rec["file"]), "rb") as fh:
            blob = fh.read()
        try:
            out = frame.decode(ora, blob)
        except ValueError:
            out = None
        assert (out is not None) == (rec["upstream"] == "accept"), rec["file"]
        if out is not None:
            assert hashlib.sha256(out).hexdigest() == rec["sha256"], rec["file"]
        want = CODE[rec["code"]]
        assert frame.verdict(blob, max(rec["length"], 1)) == (rec["length"] if want is None else want), rec["file"]


def test_window_reference_reproduces_upstream():
    """The hand-built window cases (tests/golden/window_cases.py): the window reference gives upstream's stored verdict on
    every one, its content has upstream's digest and equals the builder's model, and the verdict is the content length
    or BLOCK (every rejected case fails inside a block)."""
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import window_cases
    from oracle import frame
    from oracle.oracle import Oracle
    ora = Oracle("auto")
    with open(os.path.join(FRAMES, "window_checks.json")) as fh:
        checks = json.load(fh)["cases"]
    cases = window_cases.cases()
    assert sorted(c.id for c in cases) == sorted(checks)
    for c in cases:
        want = checks[c.id]
        assert (c.plain is not None) == (want["upstream"] == "accept"), c.id
        code = frame.verdict(c.blob, c.block_max * 8)
        if c.plain is None:
            assert code == frame.E_BLOCK, c.id
            with pytest.raises(ValueError):
                frame.decode(ora, c.blob)
            continue
        out = frame.decode(ora, c.blob)
        assert code == len(out) and out == c.plain, c.id
        assert hashlib.sha256(out).hexdigest() == want["sha256"], c.id
