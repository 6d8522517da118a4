"""The device-pointer entry points (b200lz4_compress_dev, _compact_dev, _decompress_dev, _cstate_set_dict), byte for byte
against the reference, on layouts the host batch calls never produce.

The host calls always place arrays and output slots at 16-byte strides with gaps and size every compress slot at the
bound, so here:
  - arrays start at every residue mod 16, or back to back (neighbours adjacent: a stray read changes the output);
  - output slots are tight (slot i ends where slot i + 1 starts) in a buffer pre-filled with a sentinel, with capacities
    around the reference's own size r, so the three limitedOutput guards decide and any write outside a slot shows;
  - stream state records, dictionary buffers and scratch belong to the caller and cross calls;
  - compaction is checked against numpy on lengths, headers and alignments the host path never hands it.
The expected value is always the `ref` fixture called on separately laid-out arrays: by the canonical semantics
(SURVEY.md section 5 quirk 1) a linked stream packed back to back gives the same bytes as separate arrays.

Stream counts are chosen per kernel by the rule of launch_compress (at most one stream per SM: wide; up to 12 per SM:
classic; more: compact); tests/test_gpu_modes.py re-runs this file with each kernel forced."""
import ctypes
import zlib

import numpy as np
import pytest

from test_gpu_fuzz import _echo_arrays, _has_zero_offset, build_block

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
SCRATCH_HEADER = 256                  # sizeof(Scratch): the work counters every kernel leaves at zero
EDGE_SIZES = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 31, 32, 33, 64, 255, 256, 270, 271, 300,
              4095, 4096, 65535, 65536, 65546, 65547, 65548]
KINDS = ["text", "random", "sparse01", "records", "mixed", "bits01", "biased01", "zero"]
LAYOUTS = ["aligned", "odd", "packed"]


def bound(n):
    return n + n // 255 + 16


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class Dev:
    """Device buffers and the four entry points, called on one CUDA stream."""

    def __init__(self, torch, lib):
        self.torch, self.lib = torch, lib
        self.dev = torch.device("cuda", 0)
        self.sm = torch.cuda.get_device_properties(0).multi_processor_count
        self.stream = torch.cuda.current_stream()
        self.sh = ctypes.c_void_p(self.stream.cuda_stream)
        self.scratch = self.zeros(lib.b200lz4_scratch_bytes())

    def zeros(self, n, dtype=None):
        return self.torch.zeros(int(n), dtype=dtype or self.torch.uint8, device=self.dev)

    def put(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev) if a is not None else None

    def get(self, t):
        return t.cpu().numpy()

    def sync_and_check_scratch(self, scratch=None):
        self.torch.cuda.synchronize()
        s = self.get((self.scratch if scratch is None else scratch)[:SCRATCH_HEADER])
        assert not s.any(), f"scratch header not zero after the launch: {s[:16]}"

    def compress(self, src, src_off, src_len, dst, dst_off, dst_cap, out_len, header, sf=None, states=None, accel=1,
                 scratch=None):
        n = len(src_len) if not hasattr(src_len, "numel") else src_len.numel()
        ns = 0 if sf is None else sf.numel() - 1
        rc = self.lib.b200lz4_compress_dev(_p(src), _p(src_off), _p(src_len), n, _p(sf), ns, _p(states), _p(dst),
                                           _p(dst_off), _p(dst_cap), _p(out_len), accel, header,
                                           _p(self.scratch if scratch is None else scratch), self.sh)
        assert rc == 0, rc

    def decompress(self, src, src_off, src_len, dst, dst_off, dst_cap, out_len, header, max_block, sf=None, states=None,
                   scratch=None):
        ns = 0 if sf is None else sf.numel() - 1
        rc = self.lib.b200lz4_decompress_dev(_p(src), _p(src_off), _p(src_len), src_len.numel(), _p(sf), ns, _p(states),
                                             _p(dst), _p(dst_off), _p(dst_cap), _p(out_len), header, max_block,
                                             _p(self.scratch if scratch is None else scratch), self.sh)
        assert rc == 0, rc

    def compact(self, slots, slot_off, lens, header, out, out_off, scratch=None):
        rc = self.lib.b200lz4_compact_dev(_p(slots), _p(slot_off), _p(lens), lens.numel(), header, _p(out), _p(out_off),
                                          _p(self.scratch if scratch is None else scratch), self.sh)
        assert rc == 0, rc


@pytest.fixture(scope="module")
def dev(ctx):
    import torch
    from streamly_lz4_b200 import _lib
    return Dev(torch, _lib.load())


# ---- layouts -------------------------------------------------------------------------------------------------------------

def starts(sizes, layout, rng, base=0):
    """Start offsets of consecutive regions of `sizes` bytes: aligned (16-byte starts, >= 16 bytes apart), odd (every
    residue mod 16, chosen per region), packed (back to back) or tight (back to back from a start at residue `base`)."""
    offs, at = [], base
    for i, n in enumerate(sizes):
        if layout == "aligned":
            at = (at + 15) // 16 * 16
        elif layout == "odd":
            at = (at + 15) // 16 * 16 + (i * 7 + int(rng.integers(0, 16))) % 16
        offs.append(at)
        at += int(n) + (16 if layout == "aligned" else 0)
    return np.array(offs, dtype=np.int64), at


def place(arrays, layout, rng):
    """One buffer holding `arrays` in `layout`; gaps hold random bytes, the end is padded to the next 16-byte boundary
    plus 64 bytes.  Returns (host buffer, offsets, lengths)."""
    lens = np.array([len(a) for a in arrays], dtype=np.int32)
    offs, end = starts(lens, layout, rng)
    buf = rng.integers(0, 256, size=(end + 15) // 16 * 16 + 64, dtype=np.uint8)
    for a, o in zip(arrays, offs):
        buf[o:o + len(a)] = np.frombuffer(a, dtype=np.uint8)
    return buf, offs, lens


def ref_compress(ref, arrays, sf, caps=None, accel=1):
    """Per array: the reference's LZ4 payload (None = the call returned 0), one fresh stream per stream of `sf`, arrays laid
    out apart from each other, dstCapacity caps[i] (default: the bound)."""
    arena, ptrs, lens = ref.lay_out(arrays)
    out = []
    for s in range(len(sf) - 1):
        st = ref.ccreate()
        for i in range(sf[s], sf[s + 1]):
            n = int(lens[i])
            cap = bound(n) if caps is None else int(caps[i])
            buf = np.zeros(max(cap, bound(n)) + 64, dtype=np.uint8)
            r = ref.ccont(st, int(ptrs[i]), buf.ctypes.data, n, cap, accel) if cap >= 0 else 0
            out.append(buf[:r].tobytes() if r > 0 else None)
        ref.cfree(st)
    return out


def framed(payload, n, header):
    """[header][payload] as LZ4.hs writes it (compLen, then uncompLen when the header has 8 bytes)."""
    h = b""
    if header >= 4:
        h += len(payload).to_bytes(4, "little")
    if header == 8:
        h += n.to_bytes(4, "little")
    return h + payload


def stream_firsts(counts):
    sf = np.zeros(len(counts) + 1, dtype=np.int32)
    sf[1:] = np.cumsum(counts)
    return sf


# ---- data -----------------------------------------------------------------------------------------------------------------

def mixed_arrays(rng, count, max_len):
    """Generator data of every kind at random sizes up to max_len, every fourth array at one of the edge sizes."""
    from streamly_lz4_b200 import datagen
    out = []
    for i in range(count):
        pick = i % 4
        if pick == 0:
            n = EDGE_SIZES[int(rng.integers(0, len(EDGE_SIZES)))]
        else:
            n = int(rng.integers(0, max_len + 1))
        kind = KINDS[int(rng.integers(0, len(KINDS)))]
        out.append(datagen.make(kind, int(rng.integers(0, 1 << 30)), max(n, 1))[:n].tobytes())
    return out


def kernel_streams(dev, kernel):
    """A stream count that lands on `kernel` by launch_compress's rule."""
    return {"wide": min(dev.sm, 24), "classic": dev.sm + 40, "compact": 12 * dev.sm + 60}[kernel]


def workload(dev, rng, kernel, linked):
    """(arrays, stream_first) for one compress_dev launch on `kernel`."""
    ns = kernel_streams(dev, kernel)
    if linked:
        if kernel == "wide":
            streams = [_echo_arrays(rng, int(rng.integers(2, 6))) for _ in range(ns - 4)]
            streams += [[b"", e, e[:3], e] for e in mixed_arrays(rng, 4, 3000)]       # empty and 1-3 byte dictionaries
        else:
            streams = [[a for a in mixed_arrays(rng, int(rng.integers(1, 4)), 3000)] for _ in range(ns - 8)]
            streams += [[a[:int(rng.integers(0, 1500))] for a in _echo_arrays(rng, 3)] for _ in range(8)]
        arrays = [a for s in streams for a in s]
        return arrays, stream_firsts([len(s) for s in streams])
    arrays = mixed_arrays(rng, ns, 70000 if kernel == "wide" else 2500)
    if kernel == "wide":
        arrays[:6] = _echo_arrays(rng, 6)
    return arrays, np.arange(len(arrays) + 1, dtype=np.int32)


# ---- 1. compress_dev parity ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("linked", [False, True], ids=["independent", "linked"])
@pytest.mark.parametrize("header", [0, 4, 8])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("kernel", ["wide", "classic", "compact"])
def test_compress_dev_matches_reference(dev, ref, kernel, layout, header, linked):
    rng = np.random.default_rng(zlib.crc32(f"{kernel} {layout} {header} {linked}".encode()))
    arrays, sf = workload(dev, rng, kernel, linked)
    n = len(arrays)
    src, src_off, lens = place(arrays, layout, rng)
    caps = np.array([header + bound(len(a)) for a in arrays], dtype=np.int32)
    dst_off, end = starts(caps, layout if layout != "packed" else "tight", rng, base=int(rng.integers(0, 16)))
    out = dev.put(np.full(end + 64, SENTINEL, dtype=np.uint8))
    out_len = dev.zeros(n, dev.torch.int32)
    use_cap = bool(rng.integers(0, 2))                 # d_dst_cap NULL means the same capacities
    dev.compress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), dev.put(caps) if use_cap else None,
                 out_len, header, sf=dev.put(sf) if linked else None)
    dev.sync_and_check_scratch()
    want = ref_compress(ref, arrays, sf)
    got_len, got = dev.get(out_len), dev.get(out)
    for i, w in enumerate(want):
        assert w is not None
        f = framed(w, len(arrays[i]), header)
        o = int(dst_off[i])
        assert got_len[i] == len(w), f"block {i} (n={len(arrays[i])}): out_len {got_len[i]}, reference {len(w)}"
        assert got[o:o + len(f)].tobytes() == f, f"block {i} (n={len(arrays[i])}, start {src_off[i]} mod 16 = {src_off[i] % 16})"
        assert (got[o + len(f):o + caps[i]] == SENTINEL).all(), f"block {i} wrote past its framed length"
    assert (got[:dst_off[0]] == SENTINEL).all() and (got[dst_off[-1] + caps[-1]:] == SENTINEL).all()


# ---- 2. output capacity ----------------------------------------------------------------------------------------------------

def capacity_inputs(rng):
    """Arrays shaped at the limitedOutput guards (tests/golden/make_golden.py), generator data and edge sizes."""
    from test_oracle import golden
    shaped = golden.limited_inputs()
    pick = rng.choice(len(shaped), size=160, replace=False)
    return [shaped[i] for i in sorted(pick)] + mixed_arrays(rng, 40, 20000)


def cap_variants(r, header):
    """Slot capacities (header included) around the reference's payload size r."""
    caps = {header + r - 1, header + r, header + r + 1, header + r // 2, header + 1}
    if header:
        caps |= {0, 1, header - 1, header}
    return sorted(caps)


def check_slots(got, got_len, dst_off, caps, header, arrays, want, pinned):
    """Verdict and bytes where pinned; everywhere: nothing outside a block's slot changed, a successful block wrote
    nothing past [header][payload], a failed block reports 0 and a slot too small for the header is untouched."""
    for i in range(len(arrays)):
        o, c, n = int(dst_off[i]), int(caps[i]), len(arrays[i])
        slot = got[o:o + c]
        note = f"block {i} (n={n}, cap {c}, header {header})"
        if pinned[i]:
            w = want[i]
            if w is None:
                assert got_len[i] == 0, f"{note}: out_len {got_len[i]}, the reference fails"
            else:
                assert got_len[i] == len(w), f"{note}: out_len {got_len[i]}, reference {len(w)}"
                assert slot[:header + len(w)].tobytes() == framed(w, n, header), note
        if got_len[i] > 0:
            assert (slot[header + got_len[i]:] == SENTINEL).all(), f"{note}: wrote past its framed length"
        elif c < header:
            assert (slot == SENTINEL).all(), f"{note}: a slot smaller than its header was written"
        elif header:
            assert slot[:header].tobytes() == framed(b"", n, header), f"{note}: header of a failed block"
    assert (got[:dst_off[0]] == SENTINEL).all(), "bytes before the first slot changed"
    assert (got[int(dst_off[-1] + caps[-1]):] == SENTINEL).all(), "bytes after the last slot changed"


@pytest.mark.parametrize("header", [0, 4, 8])
@pytest.mark.parametrize("many", [False, True], ids=["few", "many"])
def test_compress_dev_capacity(dev, ref, header, many):
    """Capacities header + {r-1, r, r+1, r/2, 1} (and 0, 1, header-1, header): a block succeeds exactly where the
    reference does at capacity - header, which is exactly where r fits.  Failing and fitting blocks alternate, so with
    many blocks each finder/emitter pair handles failed blocks followed by good ones."""
    rng = np.random.default_rng(100 + header + 10 * many)
    base = capacity_inputs(rng)
    fresh = ref_compress(ref, base, np.arange(len(base) + 1))
    fit, fail = [], []
    for a, w in zip(base, fresh):
        r = len(w)
        for c in cap_variants(r, header):
            (fit if c - header >= r else fail).append((a, c, r))
    order_fit, order_fail = rng.permutation(len(fit)), rng.permutation(len(fail))
    fit, fail = [fit[i] for i in order_fit], [fail[i] for i in order_fail]
    entries = [e for pair in zip(fit, fail) for e in pair] + fit[len(fail):] + fail[len(fit):]
    if not many:
        entries = entries[:min(dev.sm, 100)]
    else:
        while len(entries) < 2 * 16 * dev.sm:             # more blocks than the compact kernel has pairs, twice over
            entries = entries + entries
    arrays = [a for a, _, _ in entries]
    caps = np.array([c for _, c, _ in entries], dtype=np.int32)
    n = len(arrays)
    want = ref_compress(ref, arrays, np.arange(n + 1), caps=caps - header)
    assert any(w is None for w in want) and any(w is not None for w in want)
    for (a, c, r), w in zip(entries, want):               # LZ4's guards: success exactly when the payload fits
        assert (w is not None) == (c - header >= r), (len(a), c, r)
    src, src_off, lens = place(arrays, "odd", rng)
    dst_off, end = starts(caps, "tight", rng, base=int(rng.integers(0, 16)))
    out = dev.put(np.full(end + 64, SENTINEL, dtype=np.uint8))
    out_len = dev.put(np.full(n, -7, dtype=np.int32))
    dev.compress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), dev.put(caps), out_len, header)
    dev.sync_and_check_scratch()
    check_slots(dev.get(out), dev.get(out_len), dst_off, caps, header, arrays, want, [True] * n)


@pytest.mark.parametrize("header", [0, 8])
def test_compress_dev_capacity_linked(dev, ref, header):
    """Linked streams with limited slots: verdict and bytes are pinned up to and including each stream's first failing
    block (after a failure lz4.h leaves the stream state undefined); later blocks must still stay inside their slots."""
    rng = np.random.default_rng(200 + header)
    streams = [_echo_arrays(rng, int(rng.integers(2, 6))) for _ in range(12)]
    streams += [mixed_arrays(rng, 3, 4000) for _ in range(dev.sm + 20)]
    sf = stream_firsts([len(s) for s in streams])
    arrays = [a for s in streams for a in s]
    full = ref_compress(ref, arrays, sf)
    caps = []
    for a, w in zip(arrays, full):
        r = len(w)
        caps.append(header + int(rng.choice([r - 1, r, r + 1, r // 2, r, r + 5])))
    caps = np.array(caps, dtype=np.int32)
    want = ref_compress(ref, arrays, sf, caps=caps - header)
    pinned = []
    for s in range(len(streams)):
        ok = True
        for i in range(sf[s], sf[s + 1]):
            pinned.append(ok)
            ok = ok and want[i] is not None
    assert any(w is None for w in want)
    for layout in ("odd", "packed"):
        src, src_off, lens = place(arrays, layout, rng)
        dst_off, end = starts(caps, "tight", rng, base=int(rng.integers(0, 16)))
        out = dev.put(np.full(end + 64, SENTINEL, dtype=np.uint8))
        out_len = dev.zeros(len(arrays), dev.torch.int32)
        dev.compress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), dev.put(caps), out_len, header,
                     sf=dev.put(sf))
        dev.sync_and_check_scratch()
        check_slots(dev.get(out), dev.get(out_len), dst_off, caps, header, arrays, want, pinned)


def test_legacy_compress_capacity_boundary(dev, ref):
    """LZ4_compress_fast_continue (the legacy alias) with dstCapacity r - 1 and r on a fresh stream per input: 0 and the
    reference's bytes, and nothing written past dstCapacity."""
    lib = dev.lib
    rng = np.random.default_rng(300)
    from test_oracle import golden
    shaped = golden.limited_inputs()
    inputs = [shaped[i] for i in sorted(rng.choice(len(shaped), size=40, replace=False))]
    for a, w in zip(inputs, ref_compress(ref, inputs, np.arange(len(inputs) + 1))):
        r = len(w)
        for cap in (r - 1, r):
            cs = lib.LZ4_createStream()
            dst = ctypes.create_string_buffer(r + 64)
            ctypes.memset(dst, SENTINEL, r + 64)
            got = lib.LZ4_compress_fast_continue(cs, a, dst, len(a), cap, 1)
            lib.LZ4_freeStream(cs)
            assert got == (r if cap == r else 0), f"n={len(a)} r={r} cap={cap}: {got}"
            if got:
                assert dst.raw[:r] == w
            assert dst.raw[cap:] == bytes([SENTINEL]) * (r + 64 - cap), f"n={len(a)} cap={cap}: wrote past dstCapacity"


# ---- 3. caller-owned stream state -------------------------------------------------------------------------------------------

def cut_calls(n_max, calls, rng):
    """Cut points splitting each stream's arrays over `calls` calls."""
    if calls == 1:
        return [0, n_max]
    inner = sorted(int(x) for x in rng.integers(0, n_max + 1, size=calls - 1))
    return [0] + inner + [n_max]


@pytest.mark.parametrize("n_streams", [1, 7, "classic"])
def test_compress_dev_caller_state_across_calls(dev, ref, n_streams):
    """Zero-filled b200lz4_cstate_bytes() records with dictionary buffers attached by b200lz4_cstate_set_dict (sized to each
    stream's largest array): one or several streams pushed through compress_dev in 1, 3 and k calls equal the
    reference's single pass."""
    torch = dev.torch
    rng = np.random.default_rng(400 + (n_streams if isinstance(n_streams, int) else 99))
    ns = dev.sm + 12 if n_streams == "classic" else n_streams
    per = 10 if ns < 10 else 3
    streams = [(_echo_arrays(rng, per) if s < 8 else mixed_arrays(rng, per, 3000)) for s in range(ns)]
    for s in streams[:min(2, ns)]:
        s[1:1] = [b"", s[0][:2]]                               # an empty array and a 2-byte (dropped) dictionary
    counts = [len(s) for s in streams]
    arrays = [a for s in streams for a in s]
    sf_all = stream_firsts(counts)
    want = ref_compress(ref, arrays, sf_all)
    sb = dev.lib.b200lz4_cstate_bytes()
    for calls in (1, 3, max(counts)):
        states = dev.zeros(ns * sb)
        dict_caps = [max(len(a) for a in s) for s in streams]
        dict_offs = np.cumsum([0] + [(c + 31) // 16 * 16 for c in dict_caps])
        dicts = dev.zeros(int(dict_offs[-1]) + 64)
        for s in range(ns):
            rc = dev.lib.b200lz4_cstate_set_dict(ctypes.c_void_p(states.data_ptr() + s * sb),
                                                 ctypes.c_void_p(dicts.data_ptr() + int(dict_offs[s])), dict_caps[s], dev.sh)
            assert rc == 0
        ptrs = dev.put(np.array([states.data_ptr() + s * sb for s in range(ns)], dtype=np.uint64).view(np.int64))
        cuts = [cut_calls(c, calls, rng) for c in counts]
        got = [None] * len(arrays)
        for k in range(calls):
            idx = [int(sf_all[s]) + j for s in range(ns) for j in range(cuts[s][k], cuts[s][k + 1])]
            if not idx:
                continue
            part = [arrays[i] for i in idx]
            sf = stream_firsts([cuts[s][k + 1] - cuts[s][k] for s in range(ns)])
            src, src_off, lens = place(part, "odd", rng)
            caps = np.array([8 + bound(len(a)) for a in part], dtype=np.int32)
            dst_off, end = starts(caps, "tight", rng, base=3)
            out = dev.zeros(end + 64)
            out_len = dev.zeros(len(part), torch.int32)
            dev.compress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), None, out_len, 8,
                         sf=dev.put(sf), states=ptrs)
            dev.sync_and_check_scratch()
            o, ol = dev.get(out), dev.get(out_len)
            for j, i in enumerate(idx):
                got[i] = o[dst_off[j] + 8:dst_off[j] + 8 + ol[j]].tobytes()
        for i, w in enumerate(want):
            assert got[i] == w, f"{calls} calls: array {i} (n={len(arrays[i])}) differs from the reference's single pass"


@pytest.mark.parametrize("header", [8, 4])
@pytest.mark.parametrize("many", [False, True], ids=["wide_decoder", "narrow_decoder"])
def test_decompress_dev_caller_state_across_calls(dev, ref, header, many):
    """Zero-filled b200lz4_dstate_bytes() records: linked streams decoded in 1, 3 and k calls of decompress_dev give back
    the arrays, with few streams (the wide decoder) and with more than two per SM (the narrow one)."""
    torch = dev.torch
    rng = np.random.default_rng(500 + header + many)
    ns = 2 * dev.sm + 30 if many else 5
    max_block = 65536
    streams = [[a[:max_block] for a in (_echo_arrays(rng, 8) if s < 5 else mixed_arrays(rng, 3, 3000))] for s in range(ns)]
    counts = [len(s) for s in streams]
    arrays = [a for s in streams for a in s]
    sf_all = stream_firsts(counts)
    payloads = ref_compress(ref, arrays, sf_all)
    frames = [framed(w, len(a), header) for w, a in zip(payloads, arrays)]
    sb = dev.lib.b200lz4_dstate_bytes()
    for calls in (1, 3, max(counts)):
        states = dev.zeros(ns * sb)
        ptrs = dev.put(np.array([states.data_ptr() + s * sb for s in range(ns)], dtype=np.uint64).view(np.int64))
        cuts = [cut_calls(c, calls, rng) for c in counts]
        got = [None] * len(arrays)
        for k in range(calls):
            idx = [int(sf_all[s]) + j for s in range(ns) for j in range(cuts[s][k], cuts[s][k + 1])]
            if not idx:
                continue
            part = [frames[i] for i in idx]
            sf = stream_firsts([cuts[s][k + 1] - cuts[s][k] for s in range(ns)])
            src, src_off, lens = place(part, "odd", rng)
            caps = np.array([len(arrays[i]) if header == 8 else max_block for i in idx], dtype=np.int32)
            dst_off, end = starts(caps, "tight", rng, base=5)
            out = dev.zeros(end + 64)
            out_len = dev.zeros(len(part), torch.int32)
            dev.decompress(dev.put(src), dev.put(src_off), dev.put(lens), out, dev.put(dst_off), dev.put(caps), out_len,
                           header, max_block if header != 8 else 0, sf=dev.put(sf), states=ptrs)
            dev.sync_and_check_scratch()
            o, ol = dev.get(out), dev.get(out_len)
            for j, i in enumerate(idx):
                assert ol[j] == len(arrays[i]), f"{calls} calls: array {i}: out_len {ol[j]}, want {len(arrays[i])}"
                got[i] = o[dst_off[j]:dst_off[j] + ol[j]].tobytes()
        for i, a in enumerate(arrays):
            assert got[i] == a, f"{calls} calls: array {i} (n={len(a)}) decoded wrong"


# ---- 4. decompress_dev capacities and failures -----------------------------------------------------------------------------

def decode_cases(ref, rng):
    """(payload, plaintext length) of encoder-made and hand-built blocks, intact, truncated, bit-flipped and empty."""
    from streamly_lz4_b200 import datagen
    out = []
    arrays = mixed_arrays(rng, 30, 60000)
    for a, w in zip(arrays, ref_compress(ref, arrays, np.arange(len(arrays) + 1))):
        out.append((w, len(a)))
    for target in (64, 300, 5000, 60000):
        out.append(build_block(rng, target, 0))
    d = datagen.make("text", 13, 50000).tobytes()
    p = ref_compress(ref, [d], [0, 1])[0]
    for _ in range(40):
        b = bytearray(p)
        if rng.integers(0, 2):
            b = b[:int(rng.integers(1, len(b)))]
        else:
            at = int(rng.integers(0, len(b))); b[at] ^= 1 << int(rng.integers(0, 8))
        out.append((bytes(b), len(d)))
    out.append((b"\x00", 0))                                   # the one valid block of an empty array
    return [(w, n) for w, n in out if w and not _has_zero_offset(w)]


def ref_decode(ref, payload, cap):
    """LZ4_decompress_safe_continue on a fresh stream: the output, or None when rejected."""
    src = np.frombuffer(payload, dtype=np.uint8).copy()
    dst = np.zeros(max(cap, 1) + 64, dtype=np.uint8)
    ds = ref.dcreate()
    r = ref.dcont(ds, src.ctypes.data, dst.ctypes.data, len(payload), cap)
    ref.dfree(ds)
    return dst[:r].tobytes() if r >= 0 else None


@pytest.mark.parametrize("header", [0, 4, 8])
def test_decompress_dev_capacity_then_compact(dev, ref, header):
    """Per block: the declared capacity (header 8: uncompLen, else max_block) against a slot of d_dst_cap bytes just below
    or equal to it.  Verdict = the block fits its slot AND the reference accepts it at that capacity, with the
    reference's bytes, nothing written outside the slot.  Then compact_dev (header 0) over the result, failed and empty
    blocks included, as the host call does for headers 4 and 0."""
    torch = dev.torch
    rng = np.random.default_rng(600 + header)
    cases = decode_cases(ref, rng)
    max_block = 65536
    blocks, caps, want = [], [], []
    for w, n in cases:
        declared = n if rng.integers(0, 4) else max(0, n + int(rng.integers(-20, 20)))
        cap_decl = declared if header == 8 else max_block
        for slot in (cap_decl - 1, cap_decl):
            if slot < 0:
                continue
            blocks.append(framed(w, declared, header) if header == 8 else framed(w, n, header))
            caps.append(slot)
            want.append(ref_decode(ref, w, cap_decl) if cap_decl <= slot else None)
    order = rng.permutation(len(blocks))
    blocks = [blocks[i] for i in order]; caps = np.array([caps[i] for i in order], dtype=np.int32)
    want = [want[i] for i in order]
    assert any(w is None for w in want) and any(w is not None for w in want)
    for layout, sf in (("odd", None), ("packed", None), ("odd", "linked")):
        src, src_off, lens = place(blocks, layout, rng)
        dst_off, end = starts(caps, "tight", rng, base=int(rng.integers(0, 16)))
        out = dev.put(np.full(end + 64, SENTINEL, dtype=np.uint8))
        out_len = dev.zeros(len(blocks), torch.int32)
        d_sf = None
        if sf == "linked":                                    # one-block streams: the same verdicts through the linked path
            d_sf = dev.put(np.arange(len(blocks) + 1, dtype=np.int32))
        d_dst_off = dev.put(dst_off)
        dev.decompress(dev.put(src), dev.put(src_off), dev.put(lens), out, d_dst_off, dev.put(caps), out_len, header,
                       max_block if header != 8 else 0, sf=d_sf)
        dev.sync_and_check_scratch()
        got, got_len = dev.get(out), dev.get(out_len)
        for i, w in enumerate(want):
            note = f"block {i} (slot {caps[i]}, header {header}, {layout}, {sf or 'independent'})"
            if w is None:
                assert got_len[i] < 0, f"{note}: out_len {got_len[i]}, expected a failure"
            else:
                assert got_len[i] == len(w), f"{note}: out_len {got_len[i]}, reference {len(w)}"
                assert got[dst_off[i]:dst_off[i] + len(w)].tobytes() == w, note
        assert (got[:dst_off[0]] == SENTINEL).all() and (got[int(dst_off[-1] + caps[-1]):] == SENTINEL).all()
        # compaction of the decoded slots: only successful, non-empty blocks contribute
        d_cout = dev.put(np.full(int(caps.astype(np.int64).sum()) + 64, SENTINEL, dtype=np.uint8))
        d_coff = dev.zeros(len(blocks) + 1, torch.int64)
        dev.compact(out, d_dst_off, out_len, 0, d_cout, d_coff)
        dev.sync_and_check_scratch()
        sizes = np.maximum(got_len.astype(np.int64), 0)
        assert (dev.get(d_coff) == np.concatenate([[0], np.cumsum(sizes)])).all()
        joined = b"".join(w for w in want if w)
        cout = dev.get(d_cout)
        assert cout[:len(joined)].tobytes() == joined
        assert (cout[len(joined):] == SENTINEL).all()


# ---- 5. compact_dev against numpy -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("header", [0, 4, 8])
@pytest.mark.parametrize("n", [0, 1, 2, 31, 1023, 1024, 1025, 4097, 100000])
def test_compact_dev_matches_numpy(dev, n, header):
    torch = dev.torch
    rng = np.random.default_rng(700 + n + header)
    choices = np.array([-5, 0] + list(range(1, 18)) + [100], dtype=np.int32)
    lens = choices[rng.integers(0, len(choices), size=n)]
    if n:
        lens[rng.integers(0, n, size=max(1, min(4, n // 8)))] = 70000      # a few long blocks: the vector paths
    slot_bytes = np.where(lens > 0, lens.astype(np.int64) + header, 0) + 3
    slot_off, end = starts(slot_bytes, "odd", rng)
    slots = rng.integers(0, 256, size=end + 64, dtype=np.uint8)
    size = np.where(lens > 0, lens.astype(np.int64) + header, 0)
    want_off = np.concatenate([[0], np.cumsum(size)]).astype(np.int64)
    total = int(want_off[-1])
    idx = np.repeat(slot_off - want_off[:-1], size) + np.arange(total) if total else np.zeros(0, dtype=np.int64)
    want = slots[idx]
    d_slots, d_soff, d_len = dev.put(slots), dev.put(slot_off), dev.put(lens)
    for shift in (0, 1, 7, 15):
        d_out = dev.put(np.full(total + 96 + 70016, SENTINEL, dtype=np.uint8))      # room for one stray block past the end
        d_off = dev.put(np.full(n + 1, -1, dtype=np.int64))
        dev.compact(d_slots, d_soff, d_len, header, d_out[shift:], d_off)
        dev.sync_and_check_scratch()
        assert (dev.get(d_off) == want_off).all(), f"n={n} header={header}: out_off differs"
        got = dev.get(d_out)
        assert (got[:shift] == SENTINEL).all()
        if total:
            bad = np.flatnonzero(got[shift:shift + total] != want)
            assert not bad.size, f"n={n} header={header} shift={shift}: first wrong byte at {bad[0]} of {total}"
        assert (got[shift + total:] == SENTINEL).all(), f"n={n} header={header} shift={shift}: wrote past out_off[n]"


# ---- 6. one scratch shared by back-to-back launches -----------------------------------------------------------------------

def test_scratch_shared_by_back_to_back_launches(dev, ref):
    """compress -> compact -> decompress -> compress on one CUDA stream with one scratch block and no host sync in between
    gives what the same launches give with a sync after each; the scratch header is zero again at the end."""
    torch = dev.torch
    rng = np.random.default_rng(800)
    arrays = mixed_arrays(rng, 3 * dev.sm, 30000)              # classic kernel: several CTAs share the work counter
    n = len(arrays)
    src, src_off, lens = place(arrays, "odd", rng)
    d_src, d_soff, d_len = dev.put(src), dev.put(src_off), dev.put(lens)
    caps = np.array([8 + bound(len(a)) for a in arrays], dtype=np.int32)
    slot_off, end = starts(caps, "odd", rng)
    d_slot_off = dev.put(slot_off)
    back_off, back_end = starts(lens, "aligned", rng)
    d_back_off, d_back_cap = dev.put(back_off), dev.put(lens)

    def run(sync):
        b = {"slots": dev.zeros(end + 64), "olen": dev.zeros(n, torch.int32), "out": dev.zeros(end + 64),
             "ooff": dev.zeros(n + 1, torch.int64), "back": dev.zeros(back_end + 64), "blen": dev.zeros(n, torch.int32),
             "slots2": dev.zeros(end + 64), "olen2": dev.zeros(n, torch.int32)}
        step = dev.sync_and_check_scratch if sync else (lambda: None)
        dev.compress(d_src, d_soff, d_len, b["slots"], d_slot_off, None, b["olen"], 8)
        step()
        dev.compact(b["slots"], d_slot_off, b["olen"], 8, b["out"], b["ooff"])
        step()
        c_off = b["ooff"][:-1]
        c_len = (b["ooff"][1:] - b["ooff"][:-1]).to(torch.int32)
        dev.decompress(b["out"], c_off, c_len, b["back"], d_back_off, d_back_cap, b["blen"], 8, 0)
        step()
        dev.compress(d_src, d_soff, d_len, b["slots2"], d_slot_off, None, b["olen2"], 8)
        dev.sync_and_check_scratch()
        return {k: dev.get(v) for k, v in b.items()}

    synced, queued = run(True), run(False)
    for k in synced:
        assert np.array_equal(synced[k], queued[k]), f"{k} differs without host syncs"
    want = ref_compress(ref, arrays, np.arange(n + 1))
    assert synced["olen"].tolist() == [len(w) for w in want]
    assert (synced["blen"] == lens).all()
    for i, a in enumerate(arrays):
        assert synced["back"][back_off[i]:back_off[i] + len(a)].tobytes() == a
