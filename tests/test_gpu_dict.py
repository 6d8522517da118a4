"""Shared dictionaries on the GPU (LZ4_loadDict / LZ4_decompress_safe_usingDict semantics): byte parity with what upstream
LZ4 stored in tests/golden/dict_checks.json through every entry point that takes a dictionary -- host batch calls
(plain and streamed pipelines), persistent streams, device entry points with output capacities, the legacy
LZ4_loadDict / LZ4_setStreamDecode aliases, LZ4 frames with a dictionary id -- accept/reject verdicts on corrupted and
boundary blocks, every compressor and decoder kernel forced in turn, and the argument checks of the new C entry points."""
import base64
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

import dict_golden as mg  # noqa: E402

CHECKS = mg.load()
E_ARG = -2


@pytest.fixture(scope="module")
def dref(built):
    """The CPU restatement given a dictionary (tests/golden/dict_golden.py: Port), once it has reproduced every upstream
    digest and verdict of dict_checks.json (tests that need bytes beyond the stored digests take them from it)."""
    ora = mg.Port()
    for name, sizes, accel, linked in mg.DICT_CONFIGS:
        for kind in mg.KINDS:
            prefix, arrays = mg.dict_inputs(kind, sizes)
            for dl in mg.DICT_LENS:
                got = mg.sha(ora.compress_chunks(arrays, accel, linked=linked, dictionary=mg.dict_of(prefix, dl)))
                if got != CHECKS["digests"][f"{kind}/{name}/{dl}"]:
                    pytest.fail(f"the oracle no longer reproduces upstream's dictionary output ({kind}/{name}/{dl})")
    for i, ((dic, framed), want) in enumerate(zip(mg.dict_decoder_cases(ora), CHECKS["decoder_verdicts"])):
        try:
            got = mg.sha(ora.decompress_chunks_raw([framed], linked=False, dictionary=dic))
        except RuntimeError:
            got = None
        if got != want:
            pytest.fail(f"the oracle no longer reproduces upstream's verdict on dictionary decoder case {i}")
    return ora


def _layout(arrays, gap=16):
    """arrays in one buffer, 16-byte aligned starts with a gap (never address-adjacent)"""
    lens = np.array([len(a) for a in arrays], dtype=np.int32)
    strides = (lens.astype(np.int64) + gap + 15) // 16 * 16
    offs = np.zeros(len(arrays), dtype=np.int64)
    if len(arrays) > 1:
        offs[1:] = np.cumsum(strides[:-1])
    buf = np.zeros(int(strides.sum()) + 64, dtype=np.uint8)
    for a, o in zip(arrays, offs):
        buf[o:o + len(a)] = np.frombuffer(a, dtype=np.uint8)
    return buf, offs, lens


def batch_compress(ctx, arrays, accel, linked, d, header=8):
    buf, offs, lens = _layout(arrays)
    dst = np.zeros(int((lens.astype(np.int64) + lens // 255 + 16 + header + 16).sum()) + 64, dtype=np.uint8)
    sf = np.array([0, len(arrays)], dtype=np.int32) if linked else None
    rc, doff, olen = ctx.compress_batch(buf, offs, lens, accel, header, dst, sf, None, d)
    assert rc == 0, ctx.last_error()
    return [dst[int(doff[i]):int(doff[i + 1])].tobytes() for i in range(len(arrays))]


def batch_decompress(ctx, framed, linked, d):
    """per block: the output, or None when the block was rejected"""
    buf, offs, lens = _layout(framed)
    caps = [max(int.from_bytes(f[4:8], "little", signed=True), 0) if len(f) >= 8 else 0 for f in framed]
    dst = np.zeros(sum(caps) + 64, dtype=np.uint8)
    sf = np.array([0, len(framed)], dtype=np.int32) if linked else None
    rc, doff, olen = ctx.decompress_batch(buf, offs, lens, 8, 0, dst, sf, None, d)
    assert rc in (0, -4), ctx.last_error()
    return [None if olen[i] < 0 else dst[int(doff[i]):int(doff[i]) + int(olen[i])].tobytes() for i in range(len(framed))]


@pytest.mark.parametrize("cfg", mg.DICT_CONFIGS, ids=[c[0] for c in mg.DICT_CONFIGS])
def test_batch_dict_parity(ctx, cfg):
    """b200lz4_compress_batch_dict reproduces upstream's bytes on every generator and dictionary length, and
    b200lz4_decompress_batch_dict decodes them back; compress_chunks / decompress_chunks_raw (linked: a persistent stream
    given the dictionary by b200lz4_cstream_load_dict / b200lz4_dstream_set_dict) do the same."""
    import streamly_lz4_b200 as lz
    name, sizes, accel, linked = cfg
    bc = lz.BlockConfig(independent=not linked)
    for kind in mg.KINDS:
        prefix, arrays = mg.dict_inputs(kind, sizes)
        for dl in mg.DICT_LENS:
            want = CHECKS["digests"][f"{kind}/{name}/{dl}"]
            d = ctx.dictionary(mg.dict_of(prefix, dl))
            framed = batch_compress(ctx, arrays, accel, linked, d)
            assert mg.sha(framed) == want, (kind, name, dl, "batch")
            assert batch_decompress(ctx, framed, linked, d) == arrays, (kind, name, dl, "batch decode")
            framed2 = list(lz.compress_chunks(bc, accel, arrays, ctx=ctx, dictionary=d))
            assert mg.sha(framed2) == want, (kind, name, dl, "compress_chunks")
            assert list(lz.decompress_chunks_raw(bc, framed, ctx=ctx, dictionary=d)) == arrays, (kind, name, dl)
            d.free()


def test_dict_without_dictionary_is_unchanged(ctx, ref):
    """A dictionary of length 0 changes nothing on the decode side; on the compress side it still moves currentOffset to
    64 KiB (upstream's behaviour), which the digests above pin.  And the plain calls are unaffected by dictionaries used
    before them on the same ctx."""
    prefix, arrays = mg.dict_inputs("text", [4096] * 8)
    d = ctx.dictionary(mg.dict_of(prefix, 65536))
    batch_compress(ctx, arrays, 1, False, d)
    plain = batch_compress(ctx, arrays, 1, False, None)
    assert plain == ref.compress_chunks(arrays, 1, linked=False)
    assert batch_decompress(ctx, plain, False, ctx.dictionary(b"")) == arrays


def test_decoder_verdicts_match_upstream(ctx, dref):
    """LZ4_decompress_safe_usingDict's accept/reject decision and output on truncated and bit-flipped blocks and on
    hand-built blocks whose match reaches exactly to the dictionary's first byte or one byte further."""
    cases = mg.dict_decoder_cases(dref)
    want = CHECKS["decoder_verdicts"]
    by_dict = {}
    for i, (dic, framed) in enumerate(cases):
        by_dict.setdefault(dic, []).append(i)
    for dic, idx in by_dict.items():
        d = ctx.dictionary(dic)
        for linked in (False, True):        # linked: one block per stream, the dictionary through stream_first
            if linked:
                got = []
                for i in idx:
                    got += batch_decompress(ctx, [cases[i][1]], True, d)
            else:
                got = batch_decompress(ctx, [cases[i][1] for i in idx], False, d)
            for k, i in enumerate(idx):
                g = None if got[k] is None else mg.sha([got[k]])
                assert g == want[i], f"case {i} (dictionary of {len(dic)} bytes, linked={linked})"


class _Dev:
    def __init__(self):
        import torch
        from streamly_lz4_b200 import _lib
        self.torch, self.lib = torch, _lib.load()
        self.dev = torch.device("cuda", 0)
        self.scratch = self.zeros(self.lib.b200lz4_scratch_bytes())

    def zeros(self, n, dtype=None):
        return self.torch.zeros(int(n), dtype=dtype or self.torch.uint8, device=self.dev)

    def put(self, a):
        """a device copy; the caller keeps the tensor alive until the work using it has finished (a temporary would go
        back to the allocator while queued kernels still read it)"""
        return self.torch.from_numpy(np.array(a, copy=True)).to(self.dev)

    def stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("kind,name,dl", [("text", "4k_indep_a1", 65536), ("mixed", "64k_linked_a1", 100),
                                          ("text", "tiny_linked", 7), ("records", "640000_indep_a65537", 1 << 20),
                                          ("text", "gaps_linked_a1", 65537), ("mixed", "4k_linked_a12", 0)])
def test_dev_dict_parity_and_capacity(ctx, dref, kind, name, dl):
    """b200lz4_dict_load_dev + b200lz4_compress_dev_dict / b200lz4_decompress_dev_dict on device buffers: upstream's bytes,
    a slot capacity of exactly header + payload succeeds and one byte less fails, the decoder gets the arrays back."""
    torch = pytest.importorskip("torch")
    dev = _Dev()
    lib = dev.lib
    _, sizes, accel, linked = next(c for c in mg.DICT_CONFIGS if c[0] == name)
    prefix, arrays = mg.dict_inputs(kind, sizes)
    dic = mg.dict_of(prefix, dl)
    want = dref.compress_chunks(arrays, accel, linked=linked, dictionary=dic)
    assert mg.sha(want) == CHECKS["digests"][f"{kind}/{name}/{dl}"]
    n = len(arrays)
    d_dict = dev.put(np.frombuffer(dic + b"\0" * 16, dtype=np.uint8))
    cs = dev.zeros(lib.b200lz4_cstate_bytes())
    ds = dev.zeros(lib.b200lz4_dstate_bytes())
    assert lib.b200lz4_dict_load_dev(d_dict.data_ptr(), len(dic), cs.data_ptr(), ds.data_ptr(), dev.stream()) == 0
    buf, offs, lens = _layout(arrays)
    d_src, d_off, d_len = dev.put(buf), dev.put(offs), dev.put(lens)
    sf = dev.put(np.array([0, n], dtype=np.int32)) if linked else None
    caps = np.array([len(w) for w in want], dtype=np.int32)                    # header + payload: exactly what upstream wrote
    slot = ((caps.astype(np.int64) + 8 + 63) // 64) * 64 + 64
    doff = np.zeros(n, dtype=np.int64)
    doff[1:] = np.cumsum(slot[:-1])
    d_doff = dev.put(doff)
    for delta, ok in ((None, True), (0, True), (-1, False)):
        d_dst = dev.zeros(int(slot.sum()) + 64)
        olen = dev.zeros(n, torch.int32)
        d_cap = None if delta is None else dev.put(caps + delta)
        rc = lib.b200lz4_compress_dev_dict(d_src.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), n,
                                           None if sf is None else sf.data_ptr(), 1 if linked else 0, None, cs.data_ptr(),
                                           d_dst.data_ptr(), d_doff.data_ptr(), None if d_cap is None else d_cap.data_ptr(),
                                           olen.data_ptr(), accel, 8, dev.scratch.data_ptr(), dev.stream())
        assert rc == 0, lib.b200lz4_last_error()
        torch.cuda.synchronize()
        out, ol = d_dst.cpu().numpy(), olen.cpu().numpy()
        if ok:
            got = [out[doff[i]:doff[i] + 8 + ol[i]].tobytes() for i in range(n)]
            assert got == want, (kind, name, dl, delta)
        elif linked:
            assert ol[0] == 0                      # later blocks of the stream: whatever upstream does after a failed block
        else:
            assert (ol == 0).all()
    # decode the oracle's bytes on the device
    fbuf, foffs, flens = _layout(want)
    cap = np.array([len(a) for a in arrays], dtype=np.int32)
    ooff = np.zeros(n, dtype=np.int64)
    ooff[1:] = np.cumsum((cap[:-1].astype(np.int64) + 63) // 64 * 64 + 64)
    d_out = dev.zeros(int(ooff[-1]) + int(cap[-1]) + 128)
    olen = dev.zeros(n, torch.int32)
    d_fbuf, d_foffs, d_flens, d_ooff, d_cap = dev.put(fbuf), dev.put(foffs), dev.put(flens), dev.put(ooff), dev.put(cap)
    rc = lib.b200lz4_decompress_dev_dict(d_fbuf.data_ptr(), d_foffs.data_ptr(), d_flens.data_ptr(), n,
                                         None if sf is None else sf.data_ptr(), 1 if linked else 0, None, ds.data_ptr(),
                                         d_out.data_ptr(), d_ooff.data_ptr(), d_cap.data_ptr(), olen.data_ptr(),
                                         8, 0, dev.scratch.data_ptr(), dev.stream())
    assert rc == 0, lib.b200lz4_last_error()
    torch.cuda.synchronize()
    out, ol = d_out.cpu().numpy(), olen.cpu().numpy()
    assert [out[ooff[i]:ooff[i] + ol[i]].tobytes() for i in range(n)] == arrays


def test_legacy_load_dict_and_set_stream_decode(built, dref):
    """LZ4_loadDict / LZ4_setStreamDecode with upstream's signatures and return values, then the _continue calls."""
    from streamly_lz4_b200 import _lib
    lib = _lib.load()
    prefix, arrays = mg.dict_inputs("text", [3000, 5000, 13])
    for dl in (0, 7, 8, 100, 65536, 70000):
        dic = mg.dict_of(prefix, dl)
        want = dref.compress_chunks(arrays, 1, linked=True, dictionary=dic)
        s = lib.LZ4_createStream()
        assert s
        assert lib.LZ4_loadDict(s, dic, len(dic)) == (0 if dl < 8 else min(dl, 65536))
        keep = [ctypes.create_string_buffer(a, len(a) + 1) for a in arrays]
        got = []
        for a, k in zip(arrays, keep):
            cap = len(a) + len(a) // 255 + 16
            out = ctypes.create_string_buffer(cap)
            r = lib.LZ4_compress_fast_continue(s, k, out, len(a), cap, 1)
            assert r > 0
            got.append(out.raw[:r])
        lib.LZ4_freeStream(s)
        assert got == [w[8:] for w in want], dl
        ds = lib.LZ4_createStreamDecode()
        assert lib.LZ4_setStreamDecode(ds, dic, len(dic)) == 1
        outs = [ctypes.create_string_buffer(len(a) + 16) for a in arrays]
        for blk, a, o in zip(got, arrays, outs):
            assert lib.LZ4_decompress_safe_continue(ds, blk, o, len(blk), len(a)) == len(a)
            assert o.raw[:len(a)] == a
        lib.LZ4_freeStreamDecode(ds)


@pytest.mark.parametrize("name", [f[0] for f in mg.DICT_FRAMES])
def test_stock_frames_with_dict_id(ctx, name):
    """Frames written by LZ4F_compressFrame_usingCDict decode through read_frame(dictionary=...); without a dictionary
    the dictionary id is refused as before, with the wrong one the frame fails."""
    import streamly_lz4_b200 as lz
    f = CHECKS["frames"][name]
    prefix, arrays = mg.dict_inputs("text", mg.DICT_FRAME_SIZES)
    blob = base64.b64decode(f["frame_b64"])
    _, _, info = lz.parse_frame_header(blob[:19], allow_dict_id=True)
    assert info.dict_id == f["dict_id"]
    d = ctx.dictionary(mg.dict_of(prefix, 65536))
    assert b"".join(lz.read_frame([blob], ctx=ctx, dictionary=d)) == b"".join(arrays)
    with pytest.raises(lz.LZ4Error, match="Dict is not yet supported"):
        list(lz.read_frame([blob], ctx=ctx))
    with pytest.raises(lz.LZ4Error, match="Dict is not yet supported"):
        lz.parse_frame_header(blob[:19])
    wrong = ctx.dictionary(mg.dict_of(mg.dict_inputs("mixed", [1])[0], 65536))
    with pytest.raises(lz.LZ4Error):
        list(lz.read_frame([blob], ctx=ctx, dictionary=wrong))


@pytest.mark.parametrize("independent", [True, False], ids=["independent", "linked"])
def test_write_frame_with_dictionary(ctx, dref, independent):
    """write_frame(dictionary=, dict_id=) output: FLG bit 0 and the id in the descriptor, decodable by the frame
    restatement given the same dictionary."""
    import streamly_lz4_b200 as lz
    from oracle import frame
    prefix, arrays = mg.dict_inputs("text", [65536, 65536, 777])
    dic = mg.dict_of(prefix, 65536)
    d = ctx.dictionary(dic)
    blob = b"".join(lz.write_frame(lz.BlockSize.BlockMax64KB, 1, arrays, independent=independent, content_checksum=True,
                                   ctx=ctx, dictionary=d, dict_id=0xC0FFEE))
    desc, _, _ = frame.parse(blob)      # (the frame restatement reads the dictionary id; decoding goes through dref)
    assert desc["dict_id"] == 0xC0FFEE and desc["independent"] == independent
    assert mg.frame_decode(dref, blob, dic) == b"".join(arrays)
    assert b"".join(lz.read_frame([blob], ctx=ctx, dictionary=d)) == b"".join(arrays)


STREAMED = r"""
import sys, numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests"); sys.path.insert(0, %(root)r + "/tests/golden")
import streamly_lz4_b200 as lz
import dict_golden as mg
from test_gpu_streamed import _batch
ctx = lz.Context(0)
ref = mg.Port()
n, block = 170, 640000
buf, offs, lens, data = _batch(ctx, "mixed", 21, n, block, block, 640000)
dic = mg.dict_of(mg.dict_inputs("mixed", [1])[0], 65536)
d = ctx.dictionary(dic)
dst = ctx.pinned("s_dst", n * (block + block // 255 + 16 + 8 + 32))
rc, doff, olen = ctx.compress_batch(buf, offs, lens, 400, 8, dst, None, None, d)
assert rc == 0, ctx.last_error()
want = ref.compress_chunks([data[i * block:(i + 1) * block].tobytes() for i in range(n)], 400, linked=False, dictionary=dic)
bad = [i for i in range(n) if dst[int(doff[i]):int(doff[i]) + 8 + int(olen[i])].tobytes() != want[i]]
assert not bad, bad[:20]
back = ctx.pinned("s_back", n * block + 64)
rc, boff, blen = ctx.decompress_batch(dst, doff[:-1].copy(), (olen + 8).astype(np.int32), 8, 0, back, None, None, d)
assert rc == 0, ctx.last_error()
assert (blen == lens).all()
for i in range(n):
    assert np.array_equal(back[int(boff[i]):int(boff[i]) + block], data[i * block:(i + 1) * block]), i
ctx.close()
print("streamed dict ok")
"""


@pytest.mark.parametrize("env", [{}, {"B200LZ4_NO_STREAMED": "1"}], ids=["streamed", "plain-pipeline"])
def test_streamed_shape_batch_with_dictionary(ctx, dref, env):
    """A batch the plan sends through the streamed pipelines (equal independent blocks at a constant pitch) gives the same
    bytes with a dictionary whether it takes them or the plain pipeline."""
    e = dict(os.environ, B200LZ4_DEBUG="1", **env)
    out = subprocess.run([sys.executable, "-c", STREAMED % {"root": ROOT}], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "streamed dict ok" in out.stdout
    took = "[b200lz4] streamed:" in out.stdout
    if not env and not took:
        m = re.search(r"hardware queues: (\d+) of", out.stdout)
        if m and int(m.group(1)) < 2:
            pytest.skip("fewer than two kernel queues independent of the copy queues on this platform: no streamed calls")
    assert took == (not env), out.stdout[-2000:]


SUBSET = ["tests/test_gpu_dict.py", "-k", "batch_dict_parity or dev_dict or verdicts or without_dictionary"]


@pytest.mark.parametrize("env", [{"B200LZ4_NO_WIDE": "1", "B200LZ4_COMPACT": "1"}, {"B200LZ4_NO_WIDE": "1", "B200LZ4_COMPACT": "0"},
                                 {"B200LZ4_DWIDE": "0"}, {"B200LZ4_DWIDE": "1"}],
                         ids=["compact", "classic", "narrow-decoder", "wide-decoder"])
def test_dictionary_with_forced_kernel(ctx, env):
    """The library reads its kernel switches once per process: every compressor kernel and both decoders, each forced
    in a child process, on the parity, capacity and verdict cases above."""
    e = dict(os.environ, **env)
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", *SUBSET], cwd=ROOT, env=e,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert out.returncode == 0, out.stdout[-3000:]
    assert " passed" in out.stdout


def test_bounds_checked_decoders_on_dictionary_blocks(ctx):
    """The bounds-checked build (make bounds) traps on any write outside a block's capacity: the corrupted and boundary
    dictionary blocks through it, narrow and wide."""
    lib = os.path.join(ROOT, "streamly_lz4_b200", "libb200lz4_bounds.so")
    if not os.path.exists(lib):
        pytest.skip("libb200lz4_bounds.so not built (make bounds)")
    for wide in ("0", "1"):
        e = dict(os.environ, B200LZ4_LIB=lib, B200LZ4_DWIDE=wide)
        out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "tests/test_gpu_dict.py", "-k", "verdicts"],
                             cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
        assert out.returncode == 0, out.stdout[-3000:]
        assert " passed" in out.stdout


def test_dictionary_argument_checks(ctx):
    """A dictionary of another ctx, a dictionary together with persistent streams, a NULL dictionary or a negative
    length are B200LZ4_E_ARG; so is a device dictionary call given stream records."""
    import streamly_lz4_b200 as lz
    lib = ctx.lib
    other = lz.Context(0)
    try:
        d_other = other.dictionary(b"x" * 100)
        buf, offs, lens = _layout([b"abc" * 100])
        dst = np.zeros(4096, dtype=np.uint8)
        rc, _, _ = ctx.compress_batch(buf, offs, lens, 1, 8, dst, None, None, d_other)
        assert rc == E_ARG
        rc, _, _ = ctx.decompress_batch(buf, offs, lens, 8, 0, dst, None, None, d_other)
        assert rc == E_ARG
        s, ds = lz.CompressStream(ctx), lz.DecompressStream(ctx)
        with pytest.raises(lz.LZ4Error, match="another ctx"):
            s.load_dict(d_other)
        with pytest.raises(lz.LZ4Error, match="another ctx"):
            ds.set_dict(d_other)
        d = ctx.dictionary(b"y" * 100)
        sf = np.array([0, 1], dtype=np.int32)
        rc, _, _ = ctx.compress_batch(buf, offs, lens, 1, 8, dst, sf, [s], d)
        assert rc == E_ARG
        rc, _, _ = ctx.decompress_batch(buf, offs, lens, 8, 0, dst, sf, [ds], d)
        assert rc == E_ARG
        args = (ctx.handle, buf.ctypes.data, buf.size, offs.ctypes.data, lens.ctypes.data, 1, None, 0, None, 1, 8,
                dst.ctypes.data, dst.size, np.zeros(2, np.int64).ctypes.data, np.zeros(1, np.int32).ctypes.data, None)
        assert lib.b200lz4_compress_batch_dict(*args) == E_ARG
        h = ctypes.c_void_p()
        assert lib.b200lz4_dict_create(ctx.handle, None, 10, ctypes.byref(h)) == E_ARG
        assert lib.b200lz4_dict_create(ctx.handle, b"abc", -1, ctypes.byref(h)) == E_ARG
        assert lib.b200lz4_dict_create(None, b"abc", 3, ctypes.byref(h)) == E_ARG
        assert lib.b200lz4_dict_load_dev(None, 5, None, None, None) == E_ARG
        assert lib.b200lz4_dict_load_dev(None, -1, None, None, None) == E_ARG
        states = (ctypes.c_void_p * 1)(1)
        assert lib.b200lz4_compress_dev_dict(None, None, None, 1, None, 0, states, ctypes.c_void_p(16), None, None, None, None,
                                             1, 8, None, None) == E_ARG
        assert lib.b200lz4_decompress_dev_dict(None, None, None, 1, None, 0, None, None, None, None, None, None,
                                               8, 0, None, None) == E_ARG
        s.free(); ds.free(); d.free(); d_other.free()
    finally:
        other.close()
