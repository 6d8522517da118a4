#!/usr/bin/env python
"""Stored outputs of the reference's codec, and the one definition of the inputs they were computed on.

  python tests/golden/make_golden.py           -> golden.json: per case the generator parameters, every block's
                                                  compressed length, the SHA-256 of the framed stream and, for the small
                                                  cases, the framed bytes themselves (hex)
  python tests/golden/make_golden.py checks    -> reference_checks.json: what tests/test_oracle.py compares the
                                                  restatement with (compress digests on every generator and
                                                  configuration, random edge sizes, the decoder's accept/reject verdict
                                                  and output digest on truncated and bit-flipped blocks, and the
                                                  compressor's size and verdict at dstCapacity r - 1 and r)
  python tests/golden/make_golden.py limited [LIB] -> only the `limited` section of reference_checks.json, from the
                                                  upstream LZ4 shared library LIB (default: the system liblz4)

Both need the reference build, oracle/_ref/libreflz4.so: oracle/ref_driver.c compiled with -DDRV_USE_REFERENCE against
an LZ4 (oracle/Makefile builds it from the reference's own cbits/lz4.c when REF points at its tree).  The reference
ships no golden vectors of its own (SURVEY.md section 8c), so these outputs are the pin; each file records the LZ4
version that made it.  The tests import this module for the inputs, so generator and tests cannot drift apart.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.oracle import Oracle, available  # noqa: E402
from streamly_lz4_b200 import datagen  # noqa: E402

CASES = [
    # name, kind, seed, total bytes, block size, accel, linked, block_size config
    ("text_64k_linked_a1", "text", 101, 1 << 20, 65536, 1, True, "BlockHasSize"),
    ("text_64k_indep_a1", "text", 101, 1 << 20, 65536, 1, False, "BlockHasSize"),
    ("mixed_640000_indep_a400", "mixed", 2, 4 * 640000, 640000, 400, False, "BlockHasSize"),
    ("mixed_640000_indep_a1", "mixed", 2, 4 * 640000, 640000, 1, False, "BlockHasSize"),
    ("mixed_64k_linked_a1", "mixed", 7, 1 << 20, 65536, 1, True, "BlockHasSize"),
    ("records_4k_linked_a5", "records", 9, 1 << 18, 4096, 5, True, "BlockHasSize"),
    ("sparse_100000_linked_a12", "sparse01", 4, 1 << 20, 100000, 12, True, "BlockHasSize"),
    ("bits01_10k_linked_a-1", "bits01", 5, 200000, 10000, -1, True, "BlockHasSize"),
    ("biased01_100k_linked_a100", "biased01", 6, 500000, 100000, 100, True, "BlockHasSize"),
    ("random_64k_indep_a1", "random", 8, 1 << 18, 65536, 1, False, "BlockHasSize"),
    ("mixed_256k_max256_a1", "mixed", 12, 1 << 20, 200000, 1, True, "BlockMax256KB"),
    ("text_65547_edge", "text", 13, 65547 * 2, 65547, 1, False, "BlockHasSize"),
    ("mixed_a65537", "mixed", 14, 2 * 640000, 640000, 65537, False, "BlockHasSize"),
    ("tiny_text_300", "text", 15, 300, 300, 1, False, "BlockHasSize"),
    ("tiny_bits_1000_b100", "bits01", 16, 1000, 100, 1, True, "BlockHasSize"),
    ("tiny_sizes", "text", 17, 0, 0, 1, True, "BlockHasSize"),        # special: explicit size list
]
TINY_SIZES = [0, 1, 4, 12, 13, 14, 0, 3, 64, 2, 500, 0, 15, 31]

# inputs of the restatement-vs-reference checks (tests/test_oracle.py)
KINDS = ["text", "random", "sparse01", "records", "mixed", "bits01", "biased01", "zero"]
CONFIGS = [(65536, 1, True), (65536, 1, False), (640000, 400, False), (100000, 5, True), (4096, 1, True),
           (1000, 12, True), (333, 0, True), (3 << 20, 1, False), (50000, 65537, True)]     # block, accel, linked


def sha(chunks) -> str:
    return hashlib.sha256(b"".join(chunks)).hexdigest()


def load(name: str) -> dict:
    with open(os.path.join(HERE, name)) as f:
        return json.load(f)


def arrays_of(case: dict):
    if case["name"] == "tiny_sizes":
        d = datagen.make(case["kind"], case["seed"], 4096)
        out, at = [], 0
        for n in TINY_SIZES:
            out.append(d[at:at + n].tobytes()); at += n
        return out
    d = datagen.make(case["kind"], case["seed"], case["total"])
    return [d[i:i + case["block"]].tobytes() for i in range(0, case["total"], case["block"])]


def check_golden_case(ora, case: dict) -> None:
    """`ora` reproduces the stored framed stream of `case` and decodes it back to the input."""
    arrays = arrays_of(case)
    assert sha(arrays) == case["input_sha256"], "data generator drifted"
    framed = ora.compress_chunks(arrays, case["accel"], block_size=case["block_size"], linked=case["linked"])
    assert [len(f) for f in framed] == case["framed_lens"], case["name"]
    assert sha(framed) == case["framed_sha256"], case["name"]
    if "framed_hex" in case:
        assert b"".join(framed).hex() == case["framed_hex"], case["name"]
    assert ora.decompress_chunks_raw(framed, block_size=case["block_size"], linked=case["linked"]) == arrays, case["name"]


def config_arrays(kind: str, block: int):
    d = datagen.make(kind, 4242, 3 << 20)
    return [d[i:i + block].tobytes() for i in range(0, min(d.size, 200 * block), block)]


def edge_size_trials():
    """30 linked streams of 12 arrays with sizes around the format's thresholds, each with its acceleration."""
    rng = np.random.default_rng(1)
    d = datagen.make("text", 1, 400000)
    trials = []
    for _ in range(30):
        sizes = [int(x) for x in rng.choice([0, 1, 2, 3, 4, 5, 11, 12, 13, 14, 15, 16, 17, 100, 255, 270, 4096, 65535, 65536, 65547],
                                            size=12)]
        arrays, at = [], 0
        for n in sizes:
            at = (at + 997) % (d.size - n - 1)
            arrays.append(d[at:at + n].tobytes())
        trials.append((arrays, int(rng.integers(-1, 13))))
    return trials


def decoder_input():
    return datagen.make("text", 13, 100000).tobytes()


def corrupted_blocks(payload: bytes, n_plain: int):
    """Framed single blocks (8-byte header) whose payload is truncated or has one bit flipped."""
    rng = np.random.default_rng(7)
    cases = [payload[:k] for k in (1, 2, 10, len(payload) // 2, len(payload) - 1)]
    for _ in range(300):
        b = bytearray(payload)
        at = int(rng.integers(0, len(b)))
        b[at] ^= 1 << int(rng.integers(0, 8))
        cases.append(bytes(b))
    return [len(c).to_bytes(4, "little") + n_plain.to_bytes(4, "little") + c for c in cases]


def decode_verdict(ora, framed: bytes):
    """The decoder's decision on one independent framed block: None when rejected, else the output's SHA-256."""
    try:
        return sha(ora.decompress_chunks_raw([framed], linked=False))
    except RuntimeError:
        return None


def codec_name(ora) -> str:
    v = ora.lib.LZ4_versionNumber()
    return f"LZ4 {v // 10000}.{v // 100 % 100}.{v % 100} through oracle/ref_driver.c"


# ---- capacity-limited compression (LZ4_compress_fast_continue with dstCapacity below the bound) ----------------------

def _nonzero(rng, n: int) -> bytes:
    return rng.integers(1, 256, size=n, dtype=np.uint8).tobytes()


def limited_inputs():
    """Single arrays for the limitedOutput checks: every generator, the edge sizes, and two families shaped at the three
    guards of LZ4_compress_generic (cbits/lz4.c:1024-1027 literals, :1097-1121 match length, :1207-1217 last literals):
      tail  -- zeros then t non-zero random bytes: one match, then a last literal run of exactly t bytes;
      match -- L random bytes repeated up to the end: one literal run of L, one match that stops at matchlimit (a last
               run of exactly 5) with its length code around the 15 / 270 limits."""
    rng = np.random.default_rng(11)
    out = []
    for kind in KINDS:
        for n in (300, 5000, 70000):
            out.append(datagen.make(kind, 7, n).tobytes())
    for kind in ("text", "random", "zero"):
        d = datagen.make(kind, 3, 65547).tobytes()
        for n in (0, 1, 2, 3, 4, 5, 11, 12, 13, 14, 15, 16, 17, 31, 32, 33, 64, 255, 256, 270, 271, 300, 4096, 65535, 65547):
            out.append(d[:n])
    for t in list(range(5, 21)) + list(range(265, 276)) + [524, 525, 526]:
        for p in (64, 300):
            out.append(bytes(p) + _nonzero(rng, t))
    for lit in list(range(1, 21)) + list(range(250, 275)):
        r = _nonzero(rng, lit)
        for m in (12, 13, 20, 23, 24, 25, 36, 270, 273, 274, 275, 290):
            out.append((r * (m // lit + 2))[:lit + m])
    return out


def limited_linked_inputs():
    """(dictionary, array) pairs: the array is compressed, capacity-limited, right after the dictionary on one stream."""
    rng = np.random.default_rng(12)
    pairs = []
    for kind in ("text", "records", "mixed"):
        d = datagen.make(kind, 19, 140000).tobytes()
        for n in (20, 300, 5000, 70000):
            a = d[70000:70000 + n]
            pairs.append((d[:70000], a))
            pairs.append((d[70000 - n // 2:70000 + n // 2], a))
    for lit in (14, 15, 16, 255, 269, 270):
        r = _nonzero(rng, lit)
        pairs.append((r * 3, r[:7] + _nonzero(rng, lit)))
    return pairs


def limited_results(ora, pairs):
    """For each (dictionary or None, array): [r, result at dstCapacity r - 1, result at r], r = the size at the bound,
    each call on a fresh stream that first compressed the dictionary; and the SHA-256 of the payloads at capacity r.
    A write past dstCapacity is an error."""
    rows, payloads = [], []
    for dic, a in pairs:
        keep = [np.frombuffer(x, dtype=np.uint8).copy() if x else np.zeros(1, np.uint8) for x in (dic or b"", a)]
        src = keep[1]
        bound = ora.bound(len(a))
        row = []
        for cap in (None, "r-1", "r"):
            c = bound if cap is None else row[0] - (cap == "r-1")
            dst = np.full(bound + 64, 0xA5, dtype=np.uint8)
            s = ora.ccreate()
            if dic is not None:
                scratch = np.zeros(ora.bound(len(dic)), dtype=np.uint8)
                assert ora.ccont(s, keep[0].ctypes.data, scratch.ctypes.data, len(dic), scratch.size, 1) > 0
            got = ora.ccont(s, src.ctypes.data, dst.ctypes.data, len(a), c, 1)
            ora.cfree(s)
            assert (dst[max(c, 0):] == 0xA5).all(), "write past dstCapacity"
            row.append(int(got))
            if cap == "r":
                payloads.append(dst[:max(got, 0)].tobytes())
        rows.append(row)
    return rows, sha(payloads)


class UpstreamLz4:
    """The streaming compressor of an upstream LZ4 shared library (system liblz4 or oracle/_ref) through ctypes, with the
    names Oracle uses (ccreate / cfree / ccont / bound)."""

    def __init__(self, path: str):
        import ctypes
        self.lib = lib = ctypes.CDLL(path)
        vp, ip = ctypes.c_void_p, ctypes.c_int
        self.ccreate = lib.LZ4_createStream; self.ccreate.restype = vp; self.ccreate.argtypes = []
        self.cfree = lib.LZ4_freeStream; self.cfree.argtypes = [vp]
        self.bound = lib.LZ4_compressBound; self.bound.restype = ip; self.bound.argtypes = [ip]
        self.ccont = lib.LZ4_compress_fast_continue; self.ccont.restype = ip
        self.ccont.argtypes = [vp, vp, vp, ip, ip, ip]
        self.path = path


def make_limited(up: UpstreamLz4):
    single, single_sha = limited_results(up, [(None, a) for a in limited_inputs()])
    linked, linked_sha = limited_results(up, limited_linked_inputs())
    v = up.lib.LZ4_versionNumber()
    print("limited: single", len(single), "linked", len(linked))
    return {"codec": f"LZ4 {v // 10000}.{v // 100 % 100}.{v % 100} ({os.path.basename(up.path)}, "
                     "LZ4_compress_fast_continue through ctypes)",
            "single": single, "single_payload_sha256": single_sha, "linked": linked, "linked_payload_sha256": linked_sha}


def make_golden(ref):
    out = {"generator": "tests/golden/make_golden.py", "codec": codec_name(ref), "cases": []}
    for name, kind, seed, total, bs, accel, linked, cfg in CASES:
        case = {"name": name, "kind": kind, "seed": seed, "total": total, "block": bs}
        arrays = arrays_of(case)
        framed = ref.compress_chunks(arrays, accel, block_size=cfg, linked=linked)
        blob = b"".join(framed)
        entry = dict(case, accel=accel, linked=linked, block_size=cfg, input_sha256=sha(arrays),
                     framed_lens=[len(f) for f in framed], framed_sha256=sha(framed))
        if len(blob) <= 4096:
            entry["framed_hex"] = blob.hex()
            entry["input_hex"] = b"".join(arrays).hex()
        out["cases"].append(entry)
        print(name, len(arrays), "blocks", len(blob), "bytes")
    return out


def make_checks(ref):
    configs = {}
    for kind in KINDS:
        configs[kind] = []
        for block, accel, linked in CONFIGS:
            arrays = config_arrays(kind, block)
            framed = ref.compress_chunks(arrays, accel, linked=linked)
            assert ref.decompress_chunks_raw(framed, linked=linked) == arrays
            configs[kind].append({"block": block, "accel": accel, "linked": linked, "input_sha256": sha(arrays),
                                  "framed_sha256": sha(framed)})
    edges = [sha(ref.compress_chunks(arrays, accel, linked=True)) for arrays, accel in edge_size_trials()]
    d = decoder_input()
    payload = ref.compress_chunks([d], 1, linked=False)[0][8:]
    verdicts = [decode_verdict(ref, c) for c in corrupted_blocks(payload, len(d))]
    print("configs", sum(map(len, configs.values())), "edge trials", len(edges), "corrupted blocks", len(verdicts),
          "rejected", verdicts.count(None))
    return {"generator": "tests/golden/make_golden.py checks", "codec": codec_name(ref),
            "configs": configs, "edge_size_trials": edges,
            "decoder": {"payload_sha256": hashlib.sha256(payload).hexdigest(), "verdicts": verdicts},
            "limited": make_limited(UpstreamLz4(ref.lib._name))}


def main():
    if sys.argv[1:2] == ["limited"]:
        # only the `limited` section of reference_checks.json, from any upstream LZ4 build (default: the system liblz4)
        import ctypes.util
        path = sys.argv[2] if len(sys.argv) > 2 else ctypes.util.find_library("lz4")
        assert path, "no liblz4 found: name one, make_golden.py limited /path/to/liblz4.so"
        out = load("reference_checks.json")
        out["limited"] = make_limited(UpstreamLz4(path))
        with open(os.path.join(HERE, "reference_checks.json"), "w") as f:
            json.dump(out, f, indent=1)
        return
    assert available("reference"), "needs the reference build oracle/_ref/libreflz4.so"
    ref = Oracle("reference")
    if sys.argv[1:] == ["checks"]:
        name, out = "reference_checks.json", make_checks(ref)
    else:
        name, out = "golden.json", make_golden(ref)
    with open(os.path.join(HERE, name), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
