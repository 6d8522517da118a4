#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 LZ4 block codec (contract: DESIGN.md section "Measurement").

Headline workload (BASELINE.json configs[1]): 1 GiB synthetic mixed-entropy stream per GPU, strategy
`c+400+640000` of the reference's benchmark (benchmark/Main.hs:189-207: compress, acceleration 400,
640000-byte arrays -> 1678 blocks), independent blocks.  A step = one pass of the compress path (codec kernel +
compaction pass) over that batch.

  value        uncompressed GB/s, inputs resident in HBM, CUDA-event timed on the launching stream
  e2e          same metric through b200lz4_compress_batch with PINNED host buffers (H2D + kernels + D2H inside)
  e2e_staged   same through the public array API (compress_chunks) from PAGEABLE per-array buffers: includes the
               gather into page-locked memory that the Haskell shim / api.py perform before every call
  copy_ceiling plain cudaMemcpyAsync of the same H2D + D2H bytes on all ranks at once (what the box can move)
  roofline     dominant kernel (compress_kernel): (U + C) bytes / its own event-timed duration vs measured HBM peak
  extra        other operating points, each device-timed with its own roofline: d+640000, c+1 / d on mixed and text
               at 64 KiB / 640000 / 4 MiB blocks, config 4 (128 linked streams), config 3 (8 GiB / N, N > 1)
  cpu_baseline / --impl reference: the reference's own cbits/lz4.c (oracle/_ref) on the box's host cores; the
               output arena is allocated and touched ONCE and reused by every step (no first-touch page faults
               inside the timed call).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")     # before CUDA is initialised (see streamly_lz4_b200/_lib.py)

BLOCK = 640000
ACCEL = 400
HEADER = 8
METRIC = "LZ4 compress GB/s (uncompressed), c+400+640000 independent blocks"
UNIT = "GB/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_blocks(total: int, block: int = BLOCK):
    offs = np.arange(0, total, block, dtype=np.int64)
    lens = np.minimum(block, total - offs).astype(np.int32)
    return offs, lens


# --------------------------------------------------------------------------- reference (CPU) arm

class CpuRef:
    """The reference's lz4.c driven like compressChunk / decompressChunk (oracle/ref_driver.c), `threads` pthreads.
    All buffers are allocated and TOUCHED once in the constructor and reused by every timed call."""

    def __init__(self, data: np.ndarray, offs, lens, threads: int, accel: int, stream_first=None):
        from oracle.oracle import Oracle
        self.ora = Oracle("auto")
        self.kind = "reference" if self.ora.kind == "reference" else "port"
        self.data, self.offs, self.lens, self.threads, self.accel = data, offs, lens, threads, accel
        n = len(lens)
        self.n = n
        self.bytes = int(lens.astype(np.int64).sum())
        if stream_first is not None:
            # linked streams: the reference's arrays are separate allocations; address-adjacent arrays would switch
            # lz4.c into prefix mode (SURVEY.md section 5 quirk 1), so re-lay the blocks out with a gap (setup, untimed)
            stride = (int(lens.max()) + 64 + 63) // 64 * 64
            arena = np.zeros(n * stride + 64, dtype=np.uint8)
            if len(set(lens.tolist())) == 1:
                arena[:n * stride].reshape(n, stride)[:, :int(lens[0])] = data[:n * int(lens[0])].reshape(n, int(lens[0]))
            else:
                for i in range(n):
                    arena[i * stride:i * stride + lens[i]] = data[offs[i]:offs[i] + lens[i]]
            self.data = data = arena
            self.offs = offs = np.arange(n, dtype=np.int64) * stride
        self.ptrs = (data.ctypes.data + offs).astype(np.uint64)
        self.caps = (lens.astype(np.int64) + lens // 255 + 16 + HEADER).astype(np.int32)
        self.arena, self.dptrs, self.doffs = self.ora.slots(self.caps)
        self.arena[::4096] = 1                                  # first touch: every page mapped before any timing
        self.out_len = np.zeros(n, dtype=np.int32)
        self.sf = np.arange(n + 1, dtype=np.int32) if stream_first is None else np.ascontiguousarray(stream_first, dtype=np.int32)
        self.bytes = int(lens.astype(np.int64).sum())
        self.back = None

    def compress(self) -> float:
        t0 = time.perf_counter()
        rc = self.ora.compress_ptrs(self.ptrs, self.lens, self.dptrs, self.caps, self.out_len, self.accel, HEADER,
                                    self.sf, 0, self.threads)
        dt = time.perf_counter() - t0
        assert rc == 0, rc
        return dt

    def decompress(self) -> float:
        """Decode what compress() left in the arena (d+bufsize of the same stream)."""
        if self.back is None:
            self.dcaps = self.lens.copy()
            self.back, self.bptrs, _ = self.ora.slots(self.dcaps)
            self.back[::4096] = 1
            self.bout = np.zeros(self.n, dtype=np.int32)
        fptrs = (self.arena.ctypes.data + self.doffs[:-1]).astype(np.uint64)
        flens = (self.out_len + HEADER).astype(np.int32)
        t0 = time.perf_counter()
        rc = self.ora.decompress_ptrs(fptrs, flens, self.bptrs, self.dcaps, self.bout, HEADER, self.sf, 0, self.threads)
        dt = time.perf_counter() - t0
        assert rc == 0, rc
        return dt

    @property
    def comp_bytes(self) -> int:
        return int(self.out_len.astype(np.int64).sum())


def host_threads() -> int:
    return min(os.cpu_count() or 1, 256)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from streamly_lz4_b200 import datagen
    total = args.size_mib << 20
    data = datagen.make("mixed", 2, total)
    offs, lens = make_blocks(total)
    threads = host_threads()
    ref = CpuRef(data, offs, lens, threads, ACCEL)
    for _ in range(max(args.warmup, 1)):
        ref.compress()
    t = [ref.compress() for _ in range(args.steps)]
    ms = 1e3 * sum(t) / len(t)
    val = total / (ms / 1e3) / 1e9
    best = total / min(t) / 1e9
    extra = {}
    if not args.no_extras:
        td = min(ref.decompress() for _ in range(3))
        extra["d+640000"] = {"value": total / td / 1e9, "unit": UNIT, "what": "decode of the stream above, best of 3"}
        one = CpuRef(data, offs[:210], lens[:210], 1, ACCEL)
        one.compress()
        extra["single_thread"] = {"value": one.bytes / one.compress() / 1e9, "unit": UNIT, "what": "c+400+640000, first 210 blocks, 1 thread"}
        # the reference's own mode: linked blocks (one LZ4_stream_t per stream), config-4 shape scaled to this buffer
        ns, bs = 128, 65536
        o4, l4 = make_blocks(total, bs)
        sf = (np.arange(ns + 1, dtype=np.int64) * (len(l4) // ns)).astype(np.int32)
        sf[-1] = len(l4)
        lk = CpuRef(data, o4, l4, threads, 1, stream_first=sf)
        lk.compress()
        tc = min(lk.compress() for _ in range(2))
        tdl = min(lk.decompress() for _ in range(2))
        extra["config4_linked"] = {"compress": total / tc / 1e9, "decompress": total / tdl / 1e9, "unit": UNIT,
                                   "what": f"{ns} linked streams x {total // ns >> 20} MiB, 64 KiB blocks, accel 1, one stream per pthread"}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "best_value": best, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[1]: {args.size_mib} MiB mixed-entropy stream, c+{ACCEL}+{BLOCK}, "
                                   f"independent blocks ({len(lens)} blocks), BlockHasSize headers",
                       "note": "reference cbits/lz4.c (LZ4 1.9.3) on the host cores; always ONE stripe of the weak-scaling "
                               "workload (the GPU arm runs one such stripe per GPU); output arena allocated and touched once",
                       "ratio": total / ref.comp_bytes},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": ref.kind,
                             "sample": f"whole {args.size_mib} MiB batch per step, {threads} pthreads, one block range per thread; "
                                       f"mean of {args.steps} steps (best step {best:.2f} GB/s)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "extra": extra}
    emit(line)


# --------------------------------------------------------------------------- GPU arm

class DevBatch:
    """Device-resident buffers for kernel-resident probes over one source buffer (block partition chosen per probe)."""

    def __init__(self, lib, torch, dev, stream, total: int):
        self.lib, self.torch, self.dev, self.stream, self.total = lib, torch, dev, stream, total
        self.sh = ctypes.c_void_p(stream.cuda_stream)
        cap = total + total // 255 + (total // 4096 + 4) * 64 + (1 << 20)          # slots of >= 4 KiB blocks
        self.d_slots = torch.empty(cap, dtype=torch.uint8, device=dev)
        self.d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
        self.d_back = torch.empty(total + 64, dtype=torch.uint8, device=dev)
        self.scratch = torch.zeros(lib.b200lz4_scratch_bytes(), dtype=torch.uint8, device=dev)

    @staticmethod
    def p(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    def layout(self, block: int, n_streams: int = 0):
        torch = self.torch
        offs, lens = make_blocks(self.total, block)
        n = len(lens)
        bound = lens.astype(np.int64) + lens // 255 + 16
        ss = (bound + HEADER + 16 + 15) // 16 * 16
        so = np.zeros(n, dtype=np.int64); so[1:] = np.cumsum(ss[:-1])
        assert int(ss.sum()) <= self.d_slots.numel()
        L = {"n": n, "offs": offs, "lens": lens, "so": so,
             "d_off": torch.from_numpy(offs).to(self.dev), "d_len": torch.from_numpy(lens).to(self.dev),
             "d_so": torch.from_numpy(so).to(self.dev),
             "d_olen": torch.zeros(n, dtype=torch.int32, device=self.dev),
             "d_ooff": torch.zeros(n + 1, dtype=torch.int64, device=self.dev),
             "d_blen": torch.zeros(n, dtype=torch.int32, device=self.dev), "ns": 0, "d_sf": None}
        if n_streams:
            per = n // n_streams
            sf = (np.arange(n_streams + 1, dtype=np.int64) * per).astype(np.int32)
            sf[-1] = n
            L["ns"] = n_streams; L["d_sf"] = torch.from_numpy(sf).to(self.dev); L["sf"] = sf
        return L

    def compress(self, d_src, L, accel):
        p = self.p
        rc = self.lib.b200lz4_compress_dev(p(d_src), p(L["d_off"]), p(L["d_len"]), L["n"], p(L["d_sf"]), L["ns"], None,
                                           p(self.d_slots), p(L["d_so"]), None, p(L["d_olen"]), accel, HEADER,
                                           p(self.scratch), self.sh)
        assert rc == 0

    def compact(self, L):
        p = self.p
        rc = self.lib.b200lz4_compact_dev(p(self.d_slots), p(L["d_so"]), p(L["d_olen"]), L["n"], HEADER, p(self.d_out),
                                          p(L["d_ooff"]), p(self.scratch), self.sh)
        assert rc == 0

    def decompress(self, L, c_off, c_len):
        p = self.p
        rc = self.lib.b200lz4_decompress_dev(p(self.d_out), p(c_off), p(c_len), L["n"], p(L["d_sf"]), L["ns"], None,
                                             p(self.d_back), p(L["d_off"]), p(L["d_len"]), p(L["d_blen"]), HEADER, 0,
                                             p(self.scratch), self.sh)
        assert rc == 0

    def timed(self, fn, steps, warmup):
        torch = self.torch
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def probe(self, d_src, block, accel, peak, steps=3, warmup=1, n_streams=0, label=""):
        """c+accel+block then d+block of its output, kernel-resident; returns the extra-line dict."""
        torch = self.torch
        L = self.layout(block, n_streams)
        cms = self.timed(lambda: self.compress(d_src, L, accel), steps, warmup)
        self.compact(L)
        torch.cuda.synchronize()
        ctot = int(L["d_ooff"][-1].item())
        failed = int((L["d_olen"] <= 0).sum().item())
        c_off = L["d_ooff"][:-1].contiguous()
        c_len = (L["d_ooff"][1:] - L["d_ooff"][:-1]).to(torch.int32).contiguous()
        dms = self.timed(lambda: self.decompress(L, c_off, c_len), steps, warmup)
        ok = bool(torch.equal(self.d_back[:self.total], d_src)) and failed == 0
        algo = self.total + ctot

        def one(ms, kernel):
            ach = algo / ms / 1e6
            return {"value": self.total / ms / 1e6, "unit": UNIT, "ms_per_step": ms,
                    "roofline": {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s",
                                 "frac": ach / peak, "algorithmic_bytes_per_launch": algo}}
        mode = f"{n_streams} linked streams" if n_streams else "independent blocks"
        return {"what": f"{label}: {L['n']} blocks of {block} B, {mode}, acceleration {accel}, {self.total >> 20} MiB per GPU, "
                        f"kernel-resident, {steps} steps", "ratio": self.total / ctot, "round_trip_identical": ok,
                f"c+{accel}+{block}": one(cms, "compress_kernel*"), f"d+{block}": one(dms, "decompress_kernel*")}


DUMP_SAMPLE_BLOCKS = 8


def dump_outputs(out_dir, d_out, d_ooff, d_olen):
    """Write what the last timed step hands its caller, so that two builds can be compared output for output: every
    block's offset in the compacted stream, its compressed length and the CRC-32 of its framed bytes (float64), and the
    framed bytes (header included) of a fixed, seeded sample of blocks, one byte per float32 element.  The whole stream
    (~0.6 GB at the default size) is not written; the sample stays under 21 MB at any size, as the blocks are 640000
    bytes."""
    os.makedirs(out_dir, exist_ok=True)
    ooff = d_ooff.cpu().numpy()
    n = ooff.size - 1
    out = d_out[:int(ooff[-1])].cpu().numpy()
    blocks = [out[int(ooff[i]):int(ooff[i + 1])] for i in range(n)]
    pick = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SAMPLE_BLOCKS), replace=False))
    np.save(os.path.join(out_dir, "block_offsets.npy"), ooff.astype(np.float64))
    np.save(os.path.join(out_dir, "block_lengths.npy"), d_olen.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "block_crc32.npy"), np.array([zlib.crc32(b) for b in blocks], dtype=np.float64))
    np.save(os.path.join(out_dir, "sample_block_index.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "sample_block_bytes.npy"), np.concatenate([blocks[i] for i in pick]).astype(np.float32))
    log(f"outputs of the last timed step written to {out_dir}")


def copy_ceiling(ctx, pin_src, total, pin_dst, comp_total, reps, barrier):
    """Plain cudaMemcpyAsync of one step's H2D and D2H bytes on two streams at once (b200lz4_copy_probe: no kernels),
    all ranks together; wall-clock per repetition."""
    ctx.copy_probe(pin_src, total, pin_dst, comp_total, True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        ctx.copy_probe(pin_src, total, pin_dst, comp_total, True)
    barrier()
    both = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        ctx.copy_probe(pin_src, total, pin_dst, 0, True)
    barrier()
    h2d = (time.perf_counter() - t0) / reps
    return {"h2d_and_d2h_overlapped_ms": 1e3 * both, "h2d_alone_ms": 1e3 * h2d}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from streamly_lz4_b200 import _lib, datagen
    import streamly_lz4_b200 as lz

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback")
    from streamly_lz4_b200 import stripe
    numa = stripe.bind_host_to_device(local)               # pinned staging buffers next to this rank's GPU
    log(f"[rank {rank}] host binding: {numa}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    stream = torch.cuda.current_stream()
    peak, peak_src = measured_peak()

    total = args.size_mib << 20
    t0 = time.time()
    host = datagen.make("mixed", 2 + rank, total)          # every rank its own stripe of the stream (weak scaling)
    offs, lens = make_blocks(total)
    n = len(lens)
    log(f"[rank {rank}] generated {total >> 20} MiB in {time.time() - t0:.1f}s, {n} blocks")

    B = DevBatch(lib, torch, dev, stream, total)
    p = B.p
    d_src = torch.from_numpy(host).to(dev)
    L = B.layout(BLOCK)
    bound = lens.astype(np.int64) + lens // 255 + 16

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        B.compress(d_src, L, ACCEL); B.compact(L)
    torch.cuda.synchronize()
    comp_total = int(L["d_ooff"][-1].item())
    assert int((L["d_olen"] <= 0).sum().item()) == 0, "a block failed to compress"

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # ---- timed region: exactly K steps, device-timed, barrier + synchronize on both sides
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    barrier()
    ev[0].record(stream)
    for k in range(args.steps):
        B.compress(d_src, L, ACCEL)
        ev[2 * k + 1].record(stream)
        B.compact(L)
        ev[2 * k + 2].record(stream)
    barrier()
    total_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = [ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(args.steps)]
    compact_ms = [ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(args.steps)]
    gpu_launches = args.steps * 3
    if args.dump_outputs and rank == 0:                    # before the probes below reuse B's buffers
        dump_outputs(args.dump_outputs, B.d_out, L["d_ooff"], L["d_olen"])

    # ---- e2e: the C-ABI host call with pinned host buffers (H2D + kernels + D2H + sync inside)
    ctx = lz.Context(local)
    pin_src = ctx.pinned("b_src", total, write_combined=bool(os.environ.get("B200LZ4_BENCH_WC")))
    pin_src[:total] = host
    pin_dst = ctx.pinned("b_dst", int((bound + HEADER).sum()))
    src_view = pin_src[:total]
    for _ in range(min(args.warmup, 2)):
        rc, doff, olen = ctx.compress_batch(src_view, offs, lens, ACCEL, HEADER, pin_dst)
        assert rc == 0, _lib.last_error()
    split = {"h2d_ms": [], "kernel_ms": [], "d2h_ms": []}
    barrier()
    launches0 = ctx.launch_count()
    t_all0 = time.perf_counter()
    for _ in range(args.steps):
        rc, doff, olen = ctx.compress_batch(src_view, offs, lens, ACCEL, HEADER, pin_dst)
        tm = ctx.timing()
        for k in split:
            split[k].append(tm[k])
    barrier()
    e2e_wall = time.perf_counter() - t_all0
    e2e_launches = ctx.launch_count() - launches0          # counted by the library: chunks x (codec + scan + gather)
    assert rc == 0 and int(doff[-1]) == comp_total
    # the same call through the plain chunk pipeline (whole blocks land before their kernel starts), for comparison
    prev_env = os.environ.get("B200LZ4_NO_STREAMED")
    os.environ["B200LZ4_NO_STREAMED"] = "1"
    ctx.compress_batch(src_view, offs, lens, ACCEL, HEADER, pin_dst)
    barrier()
    t_p0 = time.perf_counter()
    for _ in range(min(args.steps, 4)):
        rc, doff, olen = ctx.compress_batch(src_view, offs, lens, ACCEL, HEADER, pin_dst)
    barrier()
    e2e_plain_wall = (time.perf_counter() - t_p0) / min(args.steps, 4)
    if prev_env is None:
        del os.environ["B200LZ4_NO_STREAMED"]
    assert rc == 0 and int(doff[-1]) == comp_total
    clocks = sampler.stop() if rank == 0 else None
    ceiling = copy_ceiling(ctx, pin_src, total, ctx.pinned("b_probe", comp_total), comp_total, 5, barrier)

    # ---- e2e_staged: the public array API from pageable per-array buffers (gather into pinned memory inside)
    staged = None
    if not args.no_extras:
        arrays = [host[o:o + l].copy() for o, l in zip(offs, lens)]         # separately allocated pageable arrays
        cfg = lz.BlockConfig(independent=True)
        sizes = 0
        for a in lz.compress_chunks(cfg, ACCEL, arrays, ctx=ctx, copy=False, batch_bytes=512 << 20):
            sizes += len(a)
        assert sizes == comp_total, (sizes, comp_total)
        reps = max(2, min(args.steps, 5))
        barrier()
        l0 = ctx.launch_count()
        t_s0 = time.perf_counter()
        for _ in range(reps):
            for a in lz.compress_chunks(cfg, ACCEL, arrays, ctx=ctx, copy=False, batch_bytes=512 << 20):
                pass
        barrier()
        staged_wall = (time.perf_counter() - t_s0) / reps
        staged = {"wall_ms_per_step": 1e3 * rmax(staged_wall), "launches": ctx.launch_count() - l0,
                  "api": "streamly_lz4_b200.compress_chunks(copy=False, batch_bytes=512 MiB) over 1678 pageable numpy arrays: multi-threaded gather "
                         "into pinned memory (b200lz4_gather_host) one batch ahead of b200lz4_compress_batch; outputs are "
                         "slices of the pinned result"}
        del arrays

    # ---- extras (kernel-resident, each with its own roofline)
    extra = {}
    gpu_launches_extra = 0
    if not args.no_extras:
        c_off = L["d_ooff"][:-1].contiguous()
        c_len = (L["d_ooff"][1:] - L["d_ooff"][:-1]).to(torch.int32).contiguous()
        barrier()
        d_ms = rmax(B.timed(lambda: B.decompress(L, c_off, c_len), args.steps, args.warmup))
        same = bool(torch.equal(B.d_back[:total], d_src)) and bool((L["d_blen"] == L["d_len"]).all().item())
        algo = total + comp_total
        extra["d+640000"] = {"what": "decode of the headline's compressed stream (strategy d+640000), kernel-resident",
                             "ms_per_step": d_ms, "value": world * total / (d_ms / 1e3) / 1e9, "unit": UNIT,
                             "round_trip_identical": same,
                             "roofline": {"bound": "hbm", "kernel": "decompress_kernel", "achieved": algo / d_ms / 1e6,
                                          "peak": peak, "unit": "GB/s", "frac": algo / d_ms / 1e6 / peak}}
        gpu_launches_extra += args.steps
        # the same through b200lz4_decompress_batch (pinned host in / out)
        comp_host = pin_dst[:comp_total]
        pin_back = ctx.pinned("b_back", total + 64)
        c_off_h = np.ascontiguousarray(doff[:-1]); c_len_h = np.diff(doff).astype(np.int32)
        for _ in range(2):
            rc2, boff, blen = ctx.decompress_batch(comp_host, c_off_h, c_len_h, HEADER, 0, pin_back)
            assert rc2 == 0, _lib.last_error()
        barrier()
        l0 = ctx.launch_count()
        t_d0 = time.perf_counter()
        for _ in range(args.steps):
            rc2, boff, blen = ctx.decompress_batch(comp_host, c_off_h, c_len_h, HEADER, 0, pin_back)
        barrier()
        d_e2e = rmax((time.perf_counter() - t_d0) / args.steps)
        tmd = ctx.timing()
        extra["d+640000"]["e2e"] = {"wall_ms_per_step": 1e3 * d_e2e, "value": world * total / d_e2e / 1e9, "unit": UNIT,
                                    "h2d_ms": tmd["h2d_ms"], "kernel_ms": tmd["kernel_ms"], "d2h_ms": tmd["d2h_ms"],
                                    "identical": bool((pin_back[:total] == host).all())}
        gpu_launches_extra += ctx.launch_count() - l0
        if rank == 0 and not args.quick:
            steps_x = 3
            extra["mixed_accel1"] = B.probe(d_src, BLOCK, 1, peak, steps_x, 1, label="config 2 data at acceleration 1")
            extra["mixed_64k"] = B.probe(d_src, 65536, 1, peak, steps_x, 1, label="config 2 data in 64 KiB arrays")
            extra["mixed_4m"] = B.probe(d_src, 4 << 20, 1, peak, steps_x, 1, label="config 2 data in 4 MiB arrays (full-wave batch)")
            extra["config4_linked"] = B.probe(d_src, 65536, 1, peak, 2, 1, n_streams=128,
                                              label="BASELINE configs[3] shape per GPU, streams shortened to fit the 1 GiB buffer")
            text = torch.from_numpy(datagen.make("text", 7, total)).to(dev)
            extra["text_64k"] = B.probe(text, 65536, 1, peak, steps_x, 1, label="text-like data (configs[0] generator), 64 KiB arrays")
            extra["text_640000"] = B.probe(text, BLOCK, 1, peak, steps_x, 1, label="text-like data, 640000-byte arrays")
            B1 = DevBatch(lib, torch, dev, stream, 16 << 20)
            extra["config1_single_linked_stream"] = B1.probe(text[:16 << 20].clone(), 65536, 1, peak, 2, 1, n_streams=1,
                                                            label="BASELINE configs[0] on the GPU: ONE linked 16 MiB text stream")
            del B1
            del text
            gpu_launches_extra += 5 * 2 * (steps_x + 1) + 2 * 2 * 3 + 7
    # ---- one batch striped over all N GPUs by ONE process (b200lz4_mctx): rank 0 drives every device, the other ranks wait
    if world > 1 and not args.no_extras:
        barrier()
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                m = lz.MultiContext(list(range(world)))
                many = ctx.pinned("b_many", int((bound + HEADER).sum()))
                rc, offm, lenm = m.compress_batch(src_view, offs, lens, ACCEL, HEADER, many)
                assert rc == 0, m.last_error()
                t_m = []
                for _ in range(3):
                    t1 = time.perf_counter()
                    rc, offm, lenm = m.compress_batch(src_view, offs, lens, ACCEL, HEADER, many)
                    t_m.append(time.perf_counter() - t1)
                same = bool(np.array_equal(lenm, olen)) and all(
                    many[offm[i]:offm[i] + HEADER + lenm[i]].tobytes() == pin_dst[doff[i]:doff[i + 1]].tobytes() for i in (0, n // 2, n - 1))
                extra["mctx_one_process"] = {
                    "what": f"b200lz4_compress_batch_multi: ONE {args.size_mib} MiB batch (rank 0's stripe) cut into {world} block ranges, one host "
                            f"thread + ctx per GPU, pinned host in/out; strong scaling of the end-to-end call",
                    "value": total / min(t_m) / 1e9, "unit": UNIT, "wall_ms": 1e3 * min(t_m), "identical_to_single_gpu": same,
                    "per_device_ms": [m.timing(i) for i in range(m.size)]}
                gpu_launches_extra += 3 * 4 * world
                m.close()
            except Exception as e:                  # reported, never fatal for the headline
                extra["mctx_one_process"] = {"error": repr(e)}
            store.set("b200lz4_mctx_done", "1")
        else:
            store.wait(["b200lz4_mctx_done"])       # on the CPU: an NCCL barrier would park a kernel on this rank's SMs
        barrier()
    # ---- config 3 (strong scaling, N > 1 or --config3): d+640000 of an 8 GiB pre-compressed stream, 8 GiB / N per rank
    if (world > 1 or args.config3) and not args.no_extras:
        extra["config3_strong"] = run_config3(args, torch, dist, lib, lz, ctx, dev, stream, rank, world, peak, barrier, rmax)

    total_ms = rmax(total_ms)
    e2e_wall = rmax(e2e_wall)
    e2e_plain_max = rmax(e2e_plain_wall)
    ms_per_step = total_ms / args.steps
    value = world * total / (ms_per_step / 1e3) / 1e9
    e2e_value = world * total / (e2e_wall / args.steps) / 1e9
    ceil_ms = rmax(ceiling["h2d_and_d2h_overlapped_ms"])
    h2d_ms_alone = rmax(ceiling["h2d_alone_ms"])

    if rank == 0:
        k_ms = statistics.mean(kern_ms)
        algo = total + comp_total                      # U + C per launch (SURVEY.md section 8d)
        achieved = algo / (k_ms / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": "compress_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo, "kernel_ms": k_ms, "compact_ms": statistics.mean(compact_ms),
                "kernel_share_of_step": k_ms / ms_per_step}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("size_mib") == args.size_mib:
                    roof["traffic"] = tj.get("compress_kernel_dram_bytes")
                    if "d+640000" in extra:
                        extra["d+640000"]["roofline"]["traffic"] = tj.get("decompress_kernel_dram_bytes")
            except Exception:
                pass
        cpu = None
        parity = None
        if not args.no_cpu:
            # ---- cpu_baseline leg: the only place of this arm that touches oracle/ (timing + a parity spot check)
            threads = host_threads()
            ref = CpuRef(host, offs, lens, threads, ACCEL)
            ref.compress()
            ts = [ref.compress() for _ in range(3)]
            if not args.no_check:
                idx = sorted(set([0, n // 2, n - 1]))
                ok = True
                for i in idx:
                    want = ref.arena[ref.doffs[i]:ref.doffs[i] + HEADER + ref.out_len[i]].tobytes()
                    ok &= pin_dst[doff[i]:doff[i + 1]].tobytes() == want
                parity = {"blocks_checked": idx, "byte_identical_to_oracle": bool(ok), "oracle": ref.kind}
            one = CpuRef(host, offs[:210], lens[:210], 1, ACCEL)
            one.compress()
            one_gbps = one.bytes / one.compress() / 1e9
            cpu = {"value": total / statistics.mean(ts) / 1e9, "best_value": total / min(ts) / 1e9, "unit": UNIT,
                   "cores": threads, "kind": ref.kind,
                   "sample": f"all {n} blocks ({total >> 20} MiB) per call, mean of 3 calls after a warm-up, {threads} pthreads, "
                             f"arena touched once; single thread on the first 210 blocks: {one_gbps:.3f} GB/s",
                   "single_thread_value": one_gbps}
        ceiling_gbps = world * total / (ceil_ms / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[1]: {args.size_mib} MiB mixed-entropy stream per GPU, c+{ACCEL}+{BLOCK}, "
                                   f"independent blocks ({n} blocks/GPU), BlockHasSize headers; step = codec kernel + compaction",
                       "ratio": total / comp_total, "l2": "inputs_exceed_l2 (1 GiB in, 0.6+ GiB out per step)",
                       "parallelism": f"block stripes over {world} GPU(s), no collective", "host_numa": numa},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": total + 20 * n,
                    "d2h_bytes_per_step": comp_total + 12 * n + 8,
                    "api": "b200lz4_compress_batch (pinned host in/out; streamed call: blocks reach the device segment by segment in "
                           "deadline order while their finders run, see DESIGN.md section 5)",
                    "h2d_ms": statistics.mean(split["h2d_ms"]), "kernel_ms": statistics.mean(split["kernel_ms"]),
                    "d2h_ms": statistics.mean(split["d2h_ms"]), "wall_ms_per_step": 1e3 * e2e_wall / args.steps,
                    "copy_ceiling": {"value": ceiling_gbps, "unit": UNIT, "ms": ceil_ms, "h2d_alone_ms": h2d_ms_alone,
                                     "what": "plain cudaMemcpyAsync of the same H2D and D2H bytes on two streams, all ranks at once, "
                                             "max over ranks"},
                    "frac_of_copy_ceiling": e2e_value / ceiling_gbps,
                    "plain_pipeline": {"value": world * total / e2e_plain_max / 1e9, "unit": UNIT, "wall_ms_per_step": 1e3 * e2e_plain_max,
                                       "what": "same call with B200LZ4_NO_STREAMED=1: six chunks, each kernel starts when its whole chunk has landed"}},
            "e2e_staged": None if staged is None else dict(staged, value=world * total / (staged["wall_ms_per_step"] / 1e3) / 1e9, unit=UNIT),
            "gpu_launches": gpu_launches + e2e_launches + gpu_launches_extra + (staged["launches"] * max(2, min(args.steps, 5)) if staged else 0),
            "gpu_launches_detail": {"timed_value_region": gpu_launches, "e2e_region": e2e_launches,
                                    "per_step": "compress_kernel + scan_kernel + gather_kernel (e2e: per block group, plus one flag kernel per copied piece)"},
            "roofline": roof, "cpu_baseline": cpu, "clocks": clocks, "parity": parity,
            "extra": {k: v for k, v in extra.items() if v is not None},
        }
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_config3(args, torch, dist, lib, lz, ctx, dev, stream, rank, world, peak, barrier, rmax):
    """BASELINE configs[2]: d+640000 of an 8 GiB pre-compressed stream, blocks striped over the ranks (STRONG scaling:
    8 GiB / N per rank).  The stream is produced on the GPU at acceleration 1 (byte-identical to the reference's
    output, which is what the parity suite establishes), consumed as one framed byte stream: device re-frame
    (resizeChunksD) + decode, kernel-resident; and from pinned host memory through host re-frame +
    b200lz4_decompress_batch for the end-to-end figure."""
    from streamly_lz4_b200 import datagen
    whole = (args.config3_gib << 30)
    piece = 1 << 30
    per_rank = whole // world
    n_pieces = max(per_rank // piece, 1)
    piece = per_rank // n_pieces
    B = DevBatch(lib, torch, dev, stream, piece)
    L = B.layout(BLOCK)
    p = B.p
    pin_in = ctx.pinned("c3_in", piece + (piece >> 6))
    pin_out = ctx.pinned("c3_out", piece + 64)
    d_stream = torch.empty(piece + (piece >> 6), dtype=torch.uint8, device=dev)
    nmax = L["n"] + 8
    d_boff = torch.zeros(nmax, dtype=torch.int64, device=dev); d_blen = torch.zeros(nmax, dtype=torch.int32, device=dev)
    d_res = torch.zeros(4, dtype=torch.int64, device=dev)
    boff = np.zeros(nmax, dtype=np.int64); blen = np.zeros(nmax, dtype=np.int32)
    found, used, ended = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()
    kern_ms, e2e_s, ubytes, cbytes, ok = 0.0, 0.0, 0, 0, True
    for k in range(n_pieces):
        host = datagen.make("mixed", 300 + rank * 64 + k, piece)
        d_src = torch.from_numpy(host).to(dev)
        B.compress(d_src, L, 1); B.compact(L)
        torch.cuda.synchronize()
        ctot = int(L["d_ooff"][-1].item())
        d_stream[:ctot] = B.d_out[:ctot]
        pin_in[:ctot] = d_stream[:ctot].cpu().numpy()
        # kernel-resident: device re-frame of the framed stream, then decode
        def dev_pass():
            rc = lib.b200lz4_reframe_dev(p(d_stream), ctot, HEADER, 0, p(d_boff), p(d_blen), nmax, p(d_res), B.sh)
            assert rc == 0
            rc = lib.b200lz4_decompress_dev(p(d_stream), p(d_boff), p(d_blen), L["n"], None, 0, None, p(B.d_back), p(L["d_off"]),
                                            p(L["d_len"]), p(L["d_blen"]), HEADER, 0, p(B.scratch), B.sh)
            assert rc == 0
        barrier()
        kern_ms += B.timed(dev_pass, 2, 1)
        ok &= bool(torch.equal(B.d_back[:piece], d_src)) and int(d_res[0].item()) == L["n"]
        # end to end: pinned host stream -> host re-frame -> decompress_batch -> pinned host output
        best = None
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            rc = lib.b200lz4_reframe(pin_in.ctypes.data, ctot, HEADER, 0, boff.ctypes.data, blen.ctypes.data, nmax,
                                     ctypes.byref(found), ctypes.byref(used), ctypes.byref(ended))
            assert rc == 0 and found.value == L["n"]
            rc, _, _ = ctx.decompress_batch(pin_in[:ctot], boff[:L["n"]].copy(), blen[:L["n"]].copy(), HEADER, 0, pin_out)
            assert rc == 0
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        ok &= bool((pin_out[:piece] == host).all())
        e2e_s += best
        ubytes += piece; cbytes += ctot
        del d_src
    kern_ms = rmax(kern_ms); e2e_s = rmax(e2e_s)
    algo = (ubytes + cbytes)
    return {"what": f"BASELINE configs[2]: d+640000 of a {args.config3_gib} GiB pre-compressed stream (acceleration 1, ratio "
                    f"{ubytes / cbytes:.2f}), block stripes over {world} GPU(s): {per_rank >> 20} MiB per rank, in {n_pieces} batch(es)",
            "scaling": "strong", "identical": bool(ok),
            "kernel_resident": {"value": whole / (kern_ms / 1e3) / 1e9, "unit": UNIT, "ms": kern_ms,
                                "what": "b200lz4_reframe_dev + b200lz4_decompress_dev on the stream resident in HBM",
                                "roofline": {"bound": "hbm", "kernel": "decompress_kernel", "achieved": algo / kern_ms / 1e6, "peak": peak,
                                             "unit": "GB/s", "frac": algo / kern_ms / 1e6 / peak}},
            "e2e": {"value": whole / e2e_s / 1e9, "unit": UNIT, "ms": 1e3 * e2e_s,
                    "what": "pinned host stream -> b200lz4_reframe (host header walk) -> b200lz4_decompress_batch -> pinned host output"}}


_REAL_STDOUT = None


def quiet_stdout():
    """Point file descriptor 1 at stderr while the benchmark runs (NCCL prints a version banner to stdout); emit() writes
    the one JSON line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size-mib", type=int, default=1024, help="stream size per GPU (default: the 1 GiB of configs[1])")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip every extra (decompress, staged e2e, other operating points)")
    ap.add_argument("--quick", action="store_true", help="keep d+640000 and e2e_staged, skip the other operating points")
    ap.add_argument("--no-check", action="store_true", help="skip the in-bench parity spot check")
    ap.add_argument("--config3", action="store_true", help="run config 3 (8 GiB pre-compressed stream) at N = 1 as well")
    ap.add_argument("--config3-gib", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's stripe) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    import __graft_entry__ as ge
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        ge.build_cpu_side()
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
