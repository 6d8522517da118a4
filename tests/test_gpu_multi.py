"""One batch striped over every visible GPU by ONE process (b200lz4_mctx, SURVEY.md section 8e / section 7 step 7):
the concatenated result must be byte-identical to the single-GPU result and, block by block, to the reference."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BLOCK = 640000
THREADS = os.cpu_count() or 8


def _blocks(total, block):
    offs = np.arange(0, total, block, dtype=np.int64)
    lens = np.minimum(block, total - offs).astype(np.int32)
    return offs, lens


@pytest.fixture(scope="module")
def mctx(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import streamly_lz4_b200 as lz
    m = lz.MultiContext()
    assert m.size == torch.cuda.device_count()
    yield m
    m.close()


@pytest.mark.parametrize("accel", [400, 1])
def test_config2_batch_striped_over_all_gpus(ctx, mctx, ref, accel):
    """BASELINE configs[1] shape (640000-byte independent blocks, mixed data), one batch, all visible devices."""
    from streamly_lz4_b200 import datagen
    total = 256 << 20
    data = datagen.make("mixed", 2, total)
    offs, lens = _blocks(total, BLOCK)
    n = len(lens)
    cap = int((lens.astype(np.int64) + lens // 255 + 24).sum())
    src = ctx.pinned("m_src", total); src[:total] = data
    one = ctx.pinned("m_one", cap); many = ctx.pinned("m_many", cap)
    rc, off1, len1 = ctx.compress_batch(src[:total], offs, lens, accel, 8, one)
    assert rc == 0
    rc, offm, lenm = mctx.compress_batch(src[:total], offs, lens, accel, 8, many)
    assert rc == 0, mctx.last_error()
    assert np.array_equal(len1, lenm)
    assert all(offm[i] + 8 + lenm[i] <= offm[i + 1] for i in range(n))          # in order, gaps only between devices
    cat_one = one[:off1[-1]].tobytes()
    cat_many = b"".join(many[offm[i]:offm[i] + 8 + lenm[i]].tobytes() for i in range(n))
    assert cat_one == cat_many
    want = ref.compress_chunks([data[offs[i]:offs[i] + lens[i]].tobytes() for i in range(n)], accel, linked=False,
                               threads=THREADS)
    bad = [i for i in range(n) if many[offm[i]:offm[i] + 8 + lenm[i]].tobytes() != want[i]]
    assert not bad, f"{len(bad)} of {n} blocks differ from the reference: {bad[:20]}"
    # decode the concatenated stream on all devices again
    blob = np.frombuffer(cat_many, dtype=np.uint8)
    csrc = ctx.pinned("m_csrc", blob.size); csrc[:blob.size] = blob
    coff = np.zeros(n, dtype=np.int64); coff[1:] = np.cumsum(lenm[:-1].astype(np.int64) + 8)
    clen = (lenm + 8).astype(np.int32)
    back = ctx.pinned("m_back", total + 64)
    rc, boff, blen = mctx.decompress_batch(csrc[:blob.size], coff, clen, 8, 0, back)
    assert rc == 0, mctx.last_error()
    assert np.array_equal(blen, lens) and np.array_equal(boff[:-1], offs)
    assert back[:total].tobytes() == data.tobytes()


def test_linked_streams_striped_over_all_gpus(ctx, mctx, ref):
    """Whole streams per device (BASELINE configs[3] shape, shortened): bytes equal the single-GPU call and the oracle."""
    from streamly_lz4_b200 import datagen
    ns, per, bs = 12, 1 << 20, 65536
    total = ns * per
    data = datagen.make("mixed", 4, total)
    offs, lens = _blocks(total, bs)
    n = len(lens)
    sf = (np.arange(ns + 1) * (per // bs)).astype(np.int32)
    cap = int((lens.astype(np.int64) + lens // 255 + 24).sum())
    src = ctx.pinned("m_src", total); src[:total] = data
    one = ctx.pinned("m_one", cap); many = ctx.pinned("m_many", cap)
    rc, off1, len1 = ctx.compress_batch(src[:total], offs, lens, 1, 8, one, stream_first=sf)
    assert rc == 0
    rc, offm, lenm = mctx.compress_batch(src[:total], offs, lens, 1, 8, many, stream_first=sf)
    assert rc == 0, mctx.last_error()
    assert np.array_equal(len1, lenm)
    blocks = [many[offm[i]:offm[i] + 8 + lenm[i]].tobytes() for i in range(n)]
    assert b"".join(blocks) == one[:off1[-1]].tobytes()
    want = ref.compress_chunks([data[o:o + bs].tobytes() for o in offs], 1, linked=True, stream_first=sf, threads=THREADS)
    bad = [s for s in range(ns) if blocks[sf[s]:sf[s + 1]] != want[sf[s]:sf[s + 1]]]
    assert not bad, f"streams {bad} of {ns} differ from the reference"
    blob = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    csrc = ctx.pinned("m_csrc", blob.size); csrc[:blob.size] = blob
    coff = np.zeros(n, dtype=np.int64); coff[1:] = np.cumsum(lenm[:-1].astype(np.int64) + 8)
    back = ctx.pinned("m_back", total + 64)
    rc, boff, blen = mctx.decompress_batch(csrc[:blob.size], coff, (lenm + 8).astype(np.int32), 8, 0, back, stream_first=sf)
    assert rc == 0, mctx.last_error()
    assert back[:total].tobytes() == data.tobytes()


def test_staged_array_api_matches_reference(ctx, ref):
    """compress_chunks from separately allocated pageable arrays (gather one batch ahead on a helper thread, zero-copy
    outputs) yields the reference's bytes; several batches so both pinned buffers of each pair are used."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    data = datagen.make("mixed", 9, 23 * 300000 + 17)
    arrays = [data[i:i + 300000].copy() for i in range(0, data.size, 300000)]
    want = ref.compress_chunks([a.tobytes() for a in arrays], 7, linked=True)
    got = [bytes(v) for v in lz.compress_chunks(lz.BlockConfig(), 7, arrays, ctx=ctx, batch_arrays=4, copy=False)]
    assert got == want
    back = [bytes(v) for v in lz.decompress_chunks_raw(lz.BlockConfig(), want, ctx=ctx, batch_arrays=5, copy=False)]
    assert back == [a.tobytes() for a in arrays]


def test_blockmax_decode_batches_are_bounded(ctx, ref):
    """BlockMax4MB headers carry no size: the decoder must budget 4 MiB per block, so many small blocks have to be cut
    into several device batches instead of one 16 GiB allocation (out_budget)."""
    import streamly_lz4_b200 as lz
    from streamly_lz4_b200 import datagen
    cfg = lz.BlockConfig(block_size=lz.BlockSize.BlockMax4MB)
    data = datagen.make("text", 3, 40 * 5000)
    arrays = [data[i:i + 5000].tobytes() for i in range(0, data.size, 5000)]
    framed = ref.compress_chunks(arrays, 1, block_size="BlockMax4MB", linked=True)
    l0 = ctx.launch_count()
    back = list(lz.decompress_chunks_raw(cfg, framed, ctx=ctx, out_budget=64 << 20))      # 15 blocks of 4 MiB + 16 per batch
    assert back == arrays
    assert ctx.launch_count() - l0 >= 3 * 3                                               # at least three batches
