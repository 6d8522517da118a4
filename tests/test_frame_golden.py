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


def test_oracle_agrees_with_upstream():
    from oracle import frame
    from oracle.oracle import Oracle
    ora = Oracle("auto")
    checked = 0
    for rec in records():
        # the checker's linked decoder takes the previous BLOCK as dictionary, not the last 64 KiB: frames whose blocks
        # are shorter than that (LZ4F_flush) are beyond what it can express
        if rec["file"].startswith("flushed_"):
            continue
        with open(os.path.join(FRAMES, rec["file"]), "rb") as fh:
            blob = fh.read()
        try:
            out = frame.decode(ora, blob)
            d = frame.parse(blob)[0]
            ok = d["frame_bytes"] == len(blob)
        except Exception:
            ok, out = False, None
        assert ok == (rec["upstream"] == "accept"), rec["file"]
        if ok:
            assert hashlib.sha256(out).hexdigest() == rec["sha256"], rec["file"]
        checked += 1
    assert checked > 100
