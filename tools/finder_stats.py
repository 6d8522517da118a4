#!/usr/bin/env python
"""Where the dense compress finder's cycles go, per region and per exit of its re-test loop (the stats build's finder
cycle account, compress.cu FinderStat).

    make stats
    python tools/finder_stats.py build/libb200lz4_stats.so [more stats builds ...] [--mib 1024]

Workloads: independent 640 000-byte blocks (bench.py's headline geometry, 1 678 blocks per GiB: one wave of
compress_kernel) of records, sparse01 and mixed at acceleration 400, and mixed at acceleration 1.  For each library and
workload, one warm-up call, then one call with the counters zeroed.  Cycles are clock64() intervals summed over all
finders; regions nest (move_window inside the loop, a queue wait inside whatever pushed), and every cycle is charged to
exactly one region.  The clock reads sit at region changes only, never inside the loop, but they do slow the build a
little: compare shares and counts, not absolute times, with the product."""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = (("records", 400), ("sparse01", 400), ("mixed", 400), ("mixed", 1))
BLOCK = 640000
REGIONS = ["other (set-up, pushes, tail, re-tests near matchlimit)", "re-test loop (retest_run)", "move_window",
           "scalar first probe + verify_count", "probe windows", "long counts + window catch-up", "queue flush waits"]
COUNTS = ["sequences stored by the loop", "loop exits: re-test miss", "loop exits: re-test match of 32+ bytes (left the loop)",
          "loop exits: window edge / matchlimit", "loop exits: full queue", "scalar first probes", "scalar first-probe hits",
          "probe windows", "search runs after a re-test miss that hit at probe 0", "descriptors pushed outside the loop",
          "one-literal restarts that hit in the loop", "one-literal restarts that missed (run goes on at probe 1)",
          "one-literal restarts with a match of 31+ bytes (left the loop)",
          "matches of 31/32+ bytes settled in the loop by a second ballot"]
SLOTS = 22          # kFsSlots_: regions 0-7 (7 unused), counts 8-21


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
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--mib", type=int, default=1024)
    args = ap.parse_args()
    import torch
    from streamly_lz4_b200 import datagen
    libs = [open_lib(p) for p in args.libs]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    sh = ctypes.c_void_p(stream.cuda_stream)
    print(f"card: {card()}")

    def p(t):
        return ctypes.c_void_p(t.data_ptr())

    total = args.mib << 20
    offs = np.arange(0, total, BLOCK, dtype=np.int64)
    lens = np.minimum(BLOCK, total - offs).astype(np.int32)
    n = len(lens)
    ss = (lens.astype(np.int64) + lens // 255 + 16 + 8 + 16 + 15) // 16 * 16
    so = np.zeros(n, dtype=np.int64); so[1:] = np.cumsum(ss[:-1])
    d_off, d_len, d_so = (torch.from_numpy(x).to(dev) for x in (offs, lens, so))
    d_slots = torch.zeros(int(ss.sum()) + 64, dtype=torch.uint8, device=dev)
    d_olen = torch.zeros(n, dtype=torch.int32, device=dev)
    for kind in dict.fromkeys(k for k, _ in WORKLOADS):
        d_src = torch.from_numpy(datagen.make(kind, 2, total)).to(dev)
        for accel in (a for k, a in WORKLOADS if k == kind):
            for path, lib in zip(args.libs, libs):
                scratch = torch.zeros(lib.b200lz4_scratch_bytes(), dtype=torch.uint8, device=dev)

                def comp():
                    rc = lib.b200lz4_compress_dev(p(d_src), p(d_off), p(d_len), n, None, 0, None, p(d_slots), p(d_so),
                                                  None, p(d_olen), accel, 8, p(scratch), sh)
                    assert rc == 0, lib.b200lz4_last_error()
                comp(); torch.cuda.synchronize()
                scratch.zero_()
                comp(); torch.cuda.synchronize()
                v = scratch[16:16 + 8 * SLOTS].cpu().numpy().view(np.uint64).astype(np.float64)
                ratio = total / float(d_olen.sum().item())
                cyc = v[:len(REGIONS)]
                seqs = v[8] + v[17]
                print(f"\n== {kind} accel {accel}  ({os.path.basename(os.path.dirname(os.path.abspath(path)))}/"
                      f"{os.path.basename(path)}; ratio {ratio:.3f}; {int(seqs)} descriptors, "
                      f"{cyc.sum() / max(seqs, 1):.0f} finder cycles per descriptor)")
                for name, c in zip(REGIONS, cyc):
                    print(f"   {name:55s} {c / 1e9:9.3f} Gcycles  {100 * c / cyc.sum():5.1f} %  "
                          f"{c / max(seqs, 1):7.1f} per descriptor")
                for name, c in zip(COUNTS, v[8:SLOTS]):
                    print(f"   {name:55s} {int(c):12d}")
        del d_src
    print(f"\ncard: {card()}")


if __name__ == "__main__":
    main()
