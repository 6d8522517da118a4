"""Rates of the LZ4 frame calls on 1 GiB of data, each next to what the same data costs through the plain block calls.

  python tools/frame_probe.py [--gib 1] [--reps 5] [--out results.json]

Workloads:
  msgs    16 384 independent frames of 64 KiB with content checksum (message-sized objects)
  tool    256 frames of one 4 MiB block each with content checksum (the `lz4` tool's defaults)
  linked  128 linked frames of 64 KiB-max blocks flushed every 16 KiB (short blocks: the decoder's window mode)
Per workload: kernel-resident time of the frame calls (device pointers, CUDA events around the call's kernels), the
same blocks through b200lz4_{de,}compress_batch (their kernel span), end-to-end time of the frame calls from pinned host
memory, and upstream LZ4F on every host core (ctypes, one frame per task) where the system liblz4 exists.  Also the rate
of one XXH32 chain (one 1 GiB range through b200lz4_xxh32_dev).  Prints the card and its power limit with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes
import ctypes.util
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import streamly_lz4_b200 as lz  # noqa: E402
from streamly_lz4_b200 import api, datagen  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def best(fn, reps):
    out = []
    for _ in range(reps):
        out.append(fn())
    return min(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    total = int(args.gib * (1 << 30))
    ctx = lz.Context(0)
    res = {"card": card(), "bytes": total, "workloads": {}}
    print("card, power limit:", res["card"])
    data = datagen.make("mixed", 7, total)

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()

    shapes = {"msgs": (16384, 65536, api.FRAME_INDEPENDENT | api.FRAME_CONTENT_CHECKSUM),
              "tool": (256, 4 << 20, api.FRAME_CONTENT_CHECKSUM),
              "linked": (128, 65536, 0)}
    for name, (n, bmax, flags) in shapes.items():
        L = total // n
        off = (np.arange(n, dtype=np.int64) * L)
        ln = np.full(n, L, dtype=np.int32)
        d_src = t(data[:n * L])
        if name == "linked":
            # blocks of 16 KiB compressed as linked streams (previous block as dictionary, a valid window-mode frame),
            # wrapped as frames: [header][compLen][payload]...[end mark]
            per = L // 16384
            boff = np.arange(n * per, dtype=np.int64) * 16384
            blen = np.full(n * per, 16384, dtype=np.int32)
            first = (np.arange(n + 1) * per).astype(np.int32)
            out = np.zeros(n * per * 16500 + 64, dtype=np.uint8)
            rc, doff, olen = ctx.compress_batch(data, boff, blen, 1, 4, out, stream_first=first)
            assert rc == 0, ctx.last_error()
            hdr = api.frame_header(api.BlockSize.BlockMax64KB)
            frames = [hdr + out[doff[f * per]:doff[(f + 1) * per]].tobytes() + b"\0\0\0\0" for f in range(n)]
            buf = np.frombuffer(b"".join(frames), dtype=np.uint8).copy()
            foff = np.concatenate([[0], np.cumsum([len(x) for x in frames])[:-1]]).astype(np.int64)
            flen = np.array([len(x) for x in frames], dtype=np.int32)
            blocks = (out, doff, first, 16384)
        else:
            cap = sum(api.frame_bound(L, bmax, flags) for _ in range(n))
            d_dst = torch.zeros(cap, dtype=torch.uint8, device="cuda")

            def comp_dev():
                torch.cuda.synchronize()
                rc, _, fo, fl = ctx.frame_compress_batch(d_src, t(off - off[0]), t(ln), bmax, flags, 1, dst=d_dst)
                assert rc == 0, ctx.last_error()
                return ctx.timing()["kernel_ms"], fo, fl
            comp_dev()
            kms = best(lambda: comp_dev()[0], args.reps)
            _, fo, fl = comp_dev()
            buf = d_dst[:int(fo[-1])].cpu().numpy()
            foff, flen = fo[:-1].copy(), fl.copy()
            res["workloads"].setdefault(name, {})["frame_compress_kernel_GBps"] = total / kms / 1e6
            # the same blocks through the plain block call (kernel span of the host call)
            bl = np.minimum(bmax, L)
            nb = n * ((L + bmax - 1) // bmax)
            boff = np.arange(nb, dtype=np.int64) * bl
            blen = np.full(nb, bl, dtype=np.int32)
            sf = None if flags & api.FRAME_INDEPENDENT else (np.arange(n + 1) * (nb // n)).astype(np.int32)
            outb = np.zeros(int(nb * (bl + bl // 255 + 32)), dtype=np.uint8)

            def comp_block():
                rc, _, _ = ctx.compress_batch(data, boff, blen, 1, 4, outb, stream_first=sf)
                assert rc == 0
                return ctx.timing()["kernel_ms"]
            comp_block()
            res["workloads"][name]["block_compress_kernel_GBps"] = total / best(comp_block, args.reps) / 1e6
            _, bdoff, _ = ctx.compress_batch(data, boff, blen, 1, 4, outb, stream_first=sf)
            blocks = (outb, bdoff, sf, int(bl))
            # end to end from pinned host memory
            h_src = ctx.pinned("probe_src", n * L)
            h_src[:n * L] = data[:n * L]
            h_dst = ctx.pinned("probe_dst", cap)

            def comp_e2e():
                t0 = time.perf_counter()
                rc, _, _, _ = ctx.frame_compress_batch(h_src[:n * L], off - off[0], ln, bmax, flags, 1, dst=h_dst[:cap])
                assert rc == 0
                return (time.perf_counter() - t0) * 1e3
            comp_e2e()
            res["workloads"][name]["frame_compress_e2e_GBps"] = total / best(comp_e2e, args.reps) / 1e6
        w = res["workloads"].setdefault(name, {})
        w["compressed_bytes"] = int(buf.size)
        d_buf = t(buf)
        caps = np.full(n, L, dtype=np.int32)
        dofs = (np.arange(n, dtype=np.int64) * L)
        d_out = torch.zeros(n * L, dtype=torch.uint8, device="cuda")

        def dec_dev():
            rc, ol = ctx.frame_decompress_batch(d_buf, t(foff), t(flen), d_out, t(dofs), t(caps))
            assert rc == 0 and (ol == L).all(), (rc, ctx.last_error())
            return ctx.timing()["kernel_ms"]
        dec_dev()
        assert torch.equal(d_out.cpu(), torch.from_numpy(data[:n * L])) if name != "linked" else True
        w["frame_decompress_kernel_GBps"] = total / best(dec_dev, args.reps) / 1e6
        # the same blocks through the plain block call (kernel span of the host call)
        bsrc, bdoff, bsf, bl = blocks
        boffs, blens = bdoff[:-1].copy(), np.diff(bdoff).astype(np.int32)
        bout = np.zeros(len(blens) * bl + 64, dtype=np.uint8)

        def dec_block():
            rc, _, _ = ctx.decompress_batch(bsrc, boffs, blens, 4, 65536 if bl <= 65536 else bl, bout, stream_first=bsf)
            assert rc == 0, ctx.last_error()
            return ctx.timing()["kernel_ms"]
        dec_block()
        w["block_decompress_kernel_GBps"] = total / best(dec_block, args.reps) / 1e6
        h_in = ctx.pinned("probe_in", buf.size)
        h_in[:buf.size] = buf
        h_out = ctx.pinned("probe_out", n * L)

        def dec_e2e():
            t0 = time.perf_counter()
            rc, _ = ctx.frame_decompress_batch(h_in[:buf.size], foff, flen, h_out[:n * L], dofs, caps)
            assert rc == 0
            return (time.perf_counter() - t0) * 1e3
        dec_e2e()
        w["frame_decompress_e2e_GBps"] = total / best(dec_e2e, args.reps) / 1e6
        # upstream LZ4F on every host core
        path = ctypes.util.find_library("lz4")
        if path:
            from frame_golden import LZ4F
            lib = LZ4F(path).lib
            cores = os.cpu_count()
            parts = np.array_split(np.arange(n), cores)

            def worker(idx):        # one decompression context and one output buffer per thread, one call per frame
                dctx = ctypes.c_void_p()
                assert lib.LZ4F_createDecompressionContext(ctypes.byref(dctx), 100) == 0
                dst = ctypes.create_string_buffer(L)
                ok = True
                for i in idx:
                    dn, sn = ctypes.c_size_t(L), ctypes.c_size_t(int(flen[i]))
                    r = lib.LZ4F_decompress(dctx, dst, ctypes.byref(dn), ctypes.c_void_p(buf.ctypes.data + int(foff[i])),
                                            ctypes.byref(sn), None)
                    ok = ok and r == 0 and dn.value == L
                lib.LZ4F_freeDecompressionContext(dctx)
                return ok
            with ThreadPoolExecutor(cores) as ex:
                t0 = time.perf_counter()
                ok = list(ex.map(worker, parts))
                w["upstream_lz4f_decompress_GBps"] = total / (time.perf_counter() - t0) / 1e9
            assert all(ok)
            w["host_cores"] = cores
        print(name, json.dumps(w))

    # one XXH32 chain
    lib = ctx.lib
    d_all = t(data)
    o = t(np.zeros(1, dtype=np.int64)); l1 = t(np.array([min(total, 0x7FFFFFFF)], dtype=np.int32))
    h = torch.zeros(1, dtype=torch.int32, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream().cuda_stream
    lib.b200lz4_xxh32_dev(d_all.data_ptr(), o.data_ptr(), l1.data_ptr(), 1, 0, h.data_ptr(), stream)
    e0.record()
    lib.b200lz4_xxh32_dev(d_all.data_ptr(), o.data_ptr(), l1.data_ptr(), 1, 0, h.data_ptr(), stream)
    e1.record()
    torch.cuda.synchronize()
    res["xxh32_one_chain_GBps"] = min(total, 0x7FFFFFFF) / e0.elapsed_time(e1) / 1e6
    print("xxh32 one chain GB/s", res["xxh32_one_chain_GBps"])
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
