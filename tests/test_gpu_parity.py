"""GPU parity tests (run on the B200 box): the CUDA path through the C ABI vs the CPU oracle.

Bar: compressed bytes identical to the reference block for block and per acceleration value;
decompression bit-exact; cross round-trips in both directions (SURVEY.md section 8c).
Re-states the properties of test/Main.hs:203-306 with the same generators and speeds.
"""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def split(data: np.ndarray, bs: int):
    return [data[i:i + bs].tobytes() for i in range(0, data.size, bs)]


def first_diff(a: bytes, b: bytes) -> str:
    n = min(len(a), len(b))
    x = np.frombuffer(a[:n], dtype=np.uint8) != np.frombuffer(b[:n], dtype=np.uint8)
    at = int(np.argmax(x)) if x.any() else n
    return f"len {len(a)} vs {len(b)}, first difference at byte {at}"


def check_compress(lz, ctx, ref, arrays, accel, linked, block_size="BlockHasSize"):
    cfg = lz.BlockConfig(block_size=lz.BlockSize[block_size], independent=not linked)
    got = list(lz.compress_chunks(cfg, accel, arrays, ctx=ctx))
    want = ref.compress_chunks(arrays, accel, block_size=block_size, linked=linked)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, f"block {i} (n={len(arrays[i])}, accel={accel}, linked={linked}): {first_diff(g, w)}"
    return cfg, want


def check_roundtrip(lz, ctx, ref, arrays, accel, linked, block_size="BlockHasSize"):
    cfg, framed = check_compress(lz, ctx, ref, arrays, accel, linked, block_size)
    # GPU decode of reference bytes
    back = list(lz.decompress_chunks_raw(cfg, framed, ctx=ctx))
    if block_size == "BlockHasSize":
        assert back == arrays
    else:
        assert b"".join(back) == b"".join(arrays) and [len(b) for b in back] == [len(a) for a in arrays]
    # reference decode of GPU bytes (== framed, asserted above) closes the loop
    assert ref.decompress_chunks_raw(framed, block_size=block_size, linked=linked) == arrays


@pytest.mark.parametrize("kind", ["text", "random", "sparse01", "records", "mixed", "bits01", "biased01", "zero"])
@pytest.mark.parametrize("bs,accel,linked", [(65536, 1, False), (65536, 1, True), (640000, 400, False),
                                               (100000, 5, True), (4096, 12, True), (1000, 1, False)])
def test_generators(ctx, ref, kind, bs, accel, linked):
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    data = datagen.make(kind, 11, 1 << 20)
    check_roundtrip(lz, ctx, ref, split(data, bs), accel, linked)


@pytest.mark.parametrize("accel", [-1, 0, 1, 2, 5, 10, 12, 100, 400, 1000, 65537, 65538])
def test_acceleration_sweep(ctx, ref, accel):
    """config 5(ii): bytes identical to the oracle per value (cbits/lz4.c:1577-1578 clamp)."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    data = datagen.make("mixed", 5, 4 * 640000)
    check_roundtrip(lz, ctx, ref, split(data, 640000), accel, False)
    check_roundtrip(lz, ctx, ref, split(data[:1 << 20], 65536), accel, True)


@pytest.mark.parametrize("n", [0, 1, 4, 5, 11, 12, 13, 14, 15, 16, 17, 31, 32, 33, 64, 255, 256, 270, 271, 300,
                               4095, 4096, 65535, 65536, 65546, 65547, 65548, 131072 + 7])
def test_edge_sizes(ctx, ref, n):
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    for kind in ("text", "bits01", "random", "zero"):
        data = datagen.make(kind, 3, max(n, 1))[:n]
        check_roundtrip(lz, ctx, ref, [data.tobytes()], 1, False)


def test_empty_and_tiny_arrays_midstream(ctx, ref):
    """Quirk 3 of SURVEY.md section 5: empty arrays reset the dictionary, 1-3 byte dictionaries are dropped."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("text", 9, 200000)
    arrays = [d[:50000].tobytes(), b"", d[50000:50003].tobytes(), d[40000:90000].tobytes(), d[90000:90001].tobytes(),
              d[60000:120000].tobytes(), b"", b"", d[100000:100012].tobytes(), d[100000:200000].tobytes()]
    for accel in (1, 7):
        check_roundtrip(lz, ctx, ref, arrays, accel, True)
        check_roundtrip(lz, ctx, ref, arrays, accel, False)


def test_quickcheck_like_lists(ctx, ref):
    """test/Main.hs:33-52: lists of {0,1} arrays incl. empty ones; 50-100 arrays of 10-100 KiB."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    rng = np.random.default_rng(42)
    for trial in range(3):
        k = int(rng.integers(50, 101))
        arrays = []
        for i in range(k):
            n = int(rng.integers(0, 100 * 1024)) if i % 7 else int(rng.integers(0, 20))
            kind = "biased01" if trial else "bits01"
            arrays.append(datagen.make(kind, 1000 * trial + i, max(n, 1))[:n].tobytes())
        for accel in (-1, 5, 12, 100):
            check_roundtrip(lz, ctx, ref, arrays, accel, True)


def test_block_max_configs(ctx, ref):
    """test/Main.hs:225-229: 4-byte header variant with fixed destination capacity."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("mixed", 21, 1 << 20)
    check_roundtrip(lz, ctx, ref, split(d, 65536), 1, True, "BlockMax64KB")
    check_roundtrip(lz, ctx, ref, split(d, 200000), 3, True, "BlockMax256KB")
    cfg = lz.BlockConfig(block_size=lz.BlockSize.BlockMax64KB)
    with pytest.raises(lz.LZ4Error):
        list(lz.compress_chunks(cfg, 1, [bytes(65537)], ctx=ctx))


def test_large_blocks_4mib(ctx, ref):
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("mixed", 8, 3 * (4 << 20) + 777)
    check_roundtrip(lz, ctx, ref, split(d, 4 << 20), 1, False)
    check_roundtrip(lz, ctx, ref, split(d, 4 << 20), 1, True)


def test_linked_state_persists_across_batches(ctx, ref, port):
    """One Haskell stream == one LZ4_stream_t across ALL arrays (Internal/LZ4.hs:367-394): splitting the
    stream into several library calls must not change a byte, and the device hash table must equal the
    oracle's after every call (SURVEY.md section 0.5: the table is observable state)."""
    import ctypes
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("text", 77, 40 * 30000)
    arrays = split(d, 30000)
    want = ref.compress_chunks(arrays, 1, linked=True)
    for batch_arrays in (1, 3, 7):
        got = list(lz.compress_chunks(lz.BlockConfig(), 1, arrays, ctx=ctx, batch_arrays=batch_arrays))
        assert got == want, f"batch_arrays={batch_arrays}"
        back = list(lz.decompress_chunks_raw(lz.BlockConfig(), want, ctx=ctx, batch_arrays=batch_arrays))
        assert back == arrays

    # the state itself: drive one device stream and one oracle stream (the restatement exposes its table) call by
    # call and compare currentOffset and every table entry that can still produce a candidate (within 65535 of it)
    lib = port.lib
    lib.ora_cstream_table.restype = ctypes.POINTER(ctypes.c_uint32); lib.ora_cstream_table.argtypes = [ctypes.c_void_p]
    lib.ora_cstream_offset.restype = ctypes.c_uint32; lib.ora_cstream_offset.argtypes = [ctypes.c_void_p]
    arena, ptrs, lens = port.lay_out(arrays)
    ocs = port.ccreate()
    cs = lz.CompressStream(ctx)
    dstbuf = np.zeros(40000, dtype=np.uint8)
    per_call = 3
    try:
        for c0 in range(0, len(arrays), per_call):
            group = arrays[c0:c0 + per_call]
            src, offs, glens = lz.api._gather(ctx, "t_src", group)
            dst = ctx.pinned("t_dst", int((glens.astype(np.int64) + glens // 255 + 24).sum()))
            rc, doff, olen = ctx.compress_batch(src, offs, glens, 1, 8, dst, np.array([0, len(group)], dtype=np.int32), [cs])
            assert rc == 0
            for i in range(c0, c0 + len(group)):
                r = port.ccont(ocs, int(ptrs[i]), dstbuf.ctypes.data, int(lens[i]), dstbuf.size, 1)
                assert r > 0 and dst[doff[i - c0] + 8:doff[i - c0 + 1]].tobytes() == dstbuf[:r].tobytes()
            table, off = cs.peek()
            want_off = int(lib.ora_cstream_offset(ocs))
            want_table = np.ctypeslib.as_array(lib.ora_cstream_table(ocs), shape=(4096,)).copy()
            assert off == want_off
            live = (want_table.astype(np.int64) + 65535 >= want_off) | (table.astype(np.int64) + 65535 >= off)
            assert np.array_equal(table[live], want_table[live]), f"device table differs from the oracle's after array {c0 + len(group)}"
            assert live.sum() > 1000
    finally:
        cs.free()
        port.cfree(ocs)


def test_fragmented_stream_decompress(ctx, ref):
    """test/Main.hs:91-103, :217-224: write the stream, re-read with bufsize in {1,512,32K,256K}, decompressChunks."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("biased01", 5, 600000)
    arrays = split(d, 40000)
    for accel in (-1, 5, 12, 100):
        blob = b"".join(lz.compress_chunks(lz.BlockConfig(), accel, arrays, ctx=ctx))
        for bufsize in (1, 512, 32 * 1024, 256 * 1024):
            if bufsize == 1 and accel != 5:
                continue
            chunks = [blob[i:i + bufsize] for i in range(0, len(blob), bufsize)]
            assert list(lz.decompress_chunks(lz.BlockConfig(), chunks, ctx=ctx)) == arrays


def test_malformed_input_is_rejected_safely(ctx, ref):
    """Decoder must stay memory-safe and report < 0 (cbits/lz4.c:2162-2163); accept/reject must agree
    with the oracle on truncated and bit-flipped blocks."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("text", 13, 100000).tobytes()
    framed = ref.compress_chunks([d], 1, linked=False)[0]
    payload = framed[8:]
    rng = np.random.default_rng(7)
    cases = [payload[:k] for k in (1, 2, 10, len(payload) // 2, len(payload) - 1)]
    for _ in range(40):
        b = bytearray(payload)
        at = int(rng.integers(0, len(b)))
        b[at] ^= 1 << int(rng.integers(0, 8))
        cases.append(bytes(b))
    cfg = lz.BlockConfig(independent=True)
    for c in cases:
        arr = len(c).to_bytes(4, "little") + len(d).to_bytes(4, "little") + c
        try:
            want = ref.decompress_chunks_raw([arr], linked=False)
        except RuntimeError:
            want = None
        try:
            got = list(lz.decompress_chunks_raw(cfg, [arr], ctx=ctx))
        except lz.LZ4Error:
            got = None
        assert got == want


def test_legacy_aliases(ctx, ref):
    """The unmodified reference's 7 foreign imports, called the way compressChunk/decompressChunk do."""
    import ctypes
    from streamly_lz4_b200 import _lib, datagen
    lib = _lib.load()
    d = datagen.make("text", 31, 150000)
    arrays = split(d, 50000)
    want = ref.compress_chunks(arrays, 2, linked=True)
    cs, ds = lib.LZ4_createStream(), lib.LZ4_createStreamDecode()
    assert cs and ds
    keep = []
    for a, w in zip(arrays, want):
        bound = lib.LZ4_compressBound(len(a))
        dst = ctypes.create_string_buffer(bound)
        n = lib.LZ4_compress_fast_continue(cs, a, dst, len(a), bound, 2)
        assert n > 0 and dst.raw[:n] == w[8:]
        out = ctypes.create_string_buffer(len(a))
        m = lib.LZ4_decompress_safe_continue(ds, dst.raw[:n], out, n, len(a))
        assert m == len(a) and out.raw == a
        keep.append(out)
    # limitedOutput: a destination that is too small returns 0 (cbits/lz4.c:1026,1120,1216)
    cs2 = lib.LZ4_createStream()
    small = ctypes.create_string_buffer(100)
    rnd = datagen.make("random", 1, 5000).tobytes()
    assert lib.LZ4_compress_fast_continue(cs2, rnd, small, len(rnd), 100, 1) == 0
    lib.LZ4_freeStream(cs); lib.LZ4_freeStream(cs2); lib.LZ4_freeStreamDecode(ds)


def test_full_size_config2_checksum(ctx, ref):
    """BASELINE config 2 at full size through size-independent properties: 1 GiB mixed stream, 640000-byte
    independent blocks, accel 400: GPU round trip is the identity (checksum of checksums), and every one of the 1 678
    blocks is byte-identical to the oracle."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    total, bs = 1 << 30, 640000
    data = datagen.make("mixed", 2, total)
    offs = np.arange(0, total, bs, dtype=np.int64)
    lens = np.minimum(bs, total - offs).astype(np.int32)
    cap = int((lens.astype(np.int64) + lens // 255 + 16 + 8).sum())
    dst = ctx.pinned("t_dst", cap)
    rc, dst_off, out_len = ctx.compress_batch(data, offs, lens, 400, 8, dst)
    assert rc == 0 and (out_len > 0).all()
    bad = []
    for b0 in range(0, len(offs), 256):         # the reference in slices of 256 blocks: host memory stays bounded
        b1 = min(len(offs), b0 + 256)
        want = ref.compress_chunks([data[offs[i]:offs[i] + lens[i]].tobytes() for i in range(b0, b1)], 400, linked=False,
                                   threads=os.cpu_count() or 8)
        bad += [i for i in range(b0, b1) if dst[dst_off[i]:dst_off[i + 1]].tobytes() != want[i - b0]]
    assert not bad, f"{len(bad)} of {len(offs)} blocks differ from the reference: {bad[:20]}"
    comp = dst[:dst_off[-1]]
    back = ctx.pinned("t_back", total + 64)
    rc, boff, blen = ctx.decompress_batch(comp, dst_off[:-1].copy(), np.diff(dst_off).astype(np.int32), 8, 0, back)
    assert rc == 0 and (blen == lens).all()
    h0 = hashlib.sha256(data.tobytes()).hexdigest()
    h1 = hashlib.sha256(back[:total].tobytes()).hexdigest()
    assert h0 == h1


def test_c_example_links_and_round_trips(ctx):
    """examples/c_roundtrip.c: the C ABI from plain C (gcc, include/b200lz4.h only): batched and legacy interfaces."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "c_roundtrip")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    lib_dir = os.path.join(root, "streamly_lz4_b200")
    subprocess.check_call(["gcc", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "examples", "c_roundtrip.c"),
                           "-L" + lib_dir, "-lb200lz4", "-Wl,-rpath," + lib_dir, "-o", exe])
    out = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert out.returncode == 0, out.stdout
    assert "batched : " in out.stdout and "legacy  : " in out.stdout


def test_haskell_shim_call_sequences_replayed_in_c(ctx):
    """examples/ffi_replay.c: the foreign-call sequences of haskell/Streamly/Internal/LZ4/B200.hs (which cannot be compiled
    here: no GHC) with the shim's exact argument marshalling -- compressChunksD, resizeChunksD over b200lz4_reframe,
    decompressChunksRawD; linked (persistent stream handles across batches) and independent (NULL stream table)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "ffi_replay")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    lib_dir = os.path.join(root, "streamly_lz4_b200")
    subprocess.check_call(["gcc", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "examples", "ffi_replay.c"),
                           "-L" + lib_dir, "-lb200lz4", "-Wl,-rpath," + lib_dir, "-o", exe])
    out = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert out.returncode == 0, out.stdout
    assert "linked     : 37 arrays" in out.stdout and "independent: 37 arrays" in out.stdout


def test_framed_stream_with_header_and_end_mark(ctx, ref):
    """benchmark/Main.hs:85-118 + decompressChunksWithD (Internal/LZ4.hs:569-577): 7-byte frame header, BlockMax64KB blocks
    (4-byte block headers), 4-byte end mark, junk after it; re-read at several buffer sizes."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    d = datagen.make("text", 91, 1 << 20)
    arrays = split(d, 65536)
    hdr = lz.frame_header(lz.BlockSize.BlockMax64KB, checksum=False)          # HC = 0, as benchmark/Main.hs:92-100 writes it
    cfg, fc = lz.simple_frame_parser(hdr)
    body = list(lz.compress_chunks_frame(cfg, fc, 65537, arrays, ctx=ctx))
    assert body[-1] == b"\0\0\0\0"
    assert body[:-1] == ref.compress_chunks(arrays, 65537, block_size="BlockMax64KB", linked=True)
    blob = hdr + b"".join(body) + b"trailing bytes after the end mark"
    for bufsize in (5, 7, 512, 65536, 1 << 20):
        chunks = [blob[i:i + bufsize] for i in range(0, len(blob), bufsize)]
        out = b"".join(lz.decompress_chunks_with(lz.simple_frame_parser, chunks, ctx=ctx))
        assert out == d.tobytes(), f"bufsize {bufsize}"
