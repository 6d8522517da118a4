#!/usr/bin/env python
"""A/B timing of compress_kernel between two builds of the library, in one process on one GPU.

    python tools/compress_ab.py A.so B.so [--mib 1024] [--rounds 5] [--reps 3]

Workloads (independent 640 000-byte blocks, the geometry of bench.py's headline): sparse01, records and mixed at
acceleration 400, mixed at acceleration 1 -- 1 GiB each, resident in HBM (more than L2 holds).  Every round times each
workload with both libraries, alternating which goes first; a time is the mean of --reps calls of
b200lz4_compress_dev between CUDA events on the launching stream, after one warm-up call.  Such a call is one launch
(launch_compress: no memset, no copy), and 1 678 streams land on compress_kernel, so the time is that kernel's.  The
two builds' block sizes and slot bytes are compared once per workload.  The card's name and power limit are read in the
same run."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = (("sparse01", 400), ("records", 400), ("mixed", 400), ("mixed", 1))
BLOCK = 640000


def open_lib(path):
    from streamly_lz4_b200._lib import PROTOTYPES
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs=2)
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    from streamly_lz4_b200 import datagen
    libs = [open_lib(p) for p in args.libs]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    sh = ctypes.c_void_p(stream.cuda_stream)
    print(f"card: {card()}  (torch: {torch.cuda.get_device_name(0)})")
    print(f"A = {args.libs[0]}\nB = {args.libs[1]}")
    scratch = [torch.zeros(lib.b200lz4_scratch_bytes(), dtype=torch.uint8, device=dev) for lib in libs]

    def p(t):
        return ctypes.c_void_p(t.data_ptr())

    total = args.mib << 20
    offs = np.arange(0, total, BLOCK, dtype=np.int64)
    lens = np.minimum(BLOCK, total - offs).astype(np.int32)
    n = len(lens)
    ss = (lens.astype(np.int64) + lens // 255 + 16 + 8 + 16 + 15) // 16 * 16
    so = np.zeros(n, dtype=np.int64); so[1:] = np.cumsum(ss[:-1])
    d_off, d_len, d_so = (torch.from_numpy(x).to(dev) for x in (offs, lens, so))
    d_slots = [torch.zeros(int(ss.sum()) + 64, dtype=torch.uint8, device=dev) for _ in libs]
    d_olen = [torch.zeros(n, dtype=torch.int32, device=dev) for _ in libs]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    times = {w: ([], []) for w in WORKLOADS}
    for kind in dict.fromkeys(k for k, _ in WORKLOADS):
        d_src = torch.from_numpy(datagen.make(kind, 2, total)).to(dev)
        for w in (w for w in WORKLOADS if w[0] == kind):
            accel = w[1]

            def comp(i):
                rc = libs[i].b200lz4_compress_dev(p(d_src), p(d_off), p(d_len), n, None, 0, None, p(d_slots[i]), p(d_so),
                                                  None, p(d_olen[i]), accel, 8, p(scratch[i]), sh)
                assert rc == 0, libs[i].b200lz4_last_error()
            for i in (0, 1):
                comp(i)
            torch.cuda.synchronize()
            same = bool(torch.equal(d_olen[0], d_olen[1]) and torch.equal(d_slots[0], d_slots[1]))
            for r in range(args.rounds):
                for i in ((0, 1) if r % 2 == 0 else (1, 0)):
                    comp(i)
                    ev[0].record(stream)
                    for _ in range(args.reps):
                        comp(i)
                    ev[1].record(stream)
                    torch.cuda.synchronize()
                    times[w][i].append(ev[0].elapsed_time(ev[1]) / args.reps)
            a, b = times[w]
            print(f"{kind:9s} accel {accel:3d}: A {statistics.median(a):7.3f} ms [{min(a):.3f}-{max(a):.3f}]  "
                  f"B {statistics.median(b):7.3f} ms [{min(b):.3f}-{max(b):.3f}]  "
                  f"B/A time {statistics.median(b) / statistics.median(a):.4f}  "
                  f"A {total / statistics.median(a) / 1e6:6.1f} GB/s  B {total / statistics.median(b) / 1e6:6.1f} GB/s  "
                  f"bytes {'identical' if same else 'DIFFER'}", flush=True)
        del d_src
    print(f"card: {card()}")


if __name__ == "__main__":
    main()
