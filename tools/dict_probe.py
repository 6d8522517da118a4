#!/usr/bin/env python
"""Kernel-resident cost of a shared dictionary: compress and decompress 1 GiB of independent blocks already in HBM
(b200lz4_compress_dev / _dev_dict, b200lz4_decompress_dev / _dev_dict; CUDA events around each call, best of --reps
after one warm-up), without and with a 64 KiB dictionary, and the compression ratio.  Every block restores the 16 KiB
table of the dictionary's state record, which is the cost to watch at small blocks.  Rates are uncompressed bytes per
second.  Needs a GPU; prints the card's name and power limit first.

    python tools/dict_probe.py [--mib 1024] [--reps 3] [--kinds text,mixed] [--blocks 4096,65536]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kinds", default="text,mixed")
    ap.add_argument("--blocks", default="4096,65536")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("dict_probe: no CUDA device")
    from streamly_lz4_b200 import _lib, datagen
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(json.dumps({"card": torch.cuda.get_device_name(0), "power_limit": power}), flush=True)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    scratch = torch.zeros(lib.b200lz4_scratch_bytes(), dtype=torch.uint8, device=dev)
    total = args.mib << 20

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        best = None
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            best = a.elapsed_time(b) if best is None else min(best, a.elapsed_time(b))
        return best

    for kind in args.kinds.split(","):
        host = datagen.make(kind, 5, total + 65536)
        dic = torch.from_numpy(host[:65536].copy()).to(dev)
        src = torch.from_numpy(host[65536:]).to(dev)
        cs = torch.zeros(lib.b200lz4_cstate_bytes(), dtype=torch.uint8, device=dev)
        ds = torch.zeros(lib.b200lz4_dstate_bytes(), dtype=torch.uint8, device=dev)
        assert lib.b200lz4_dict_load_dev(dic.data_ptr(), 65536, cs.data_ptr(), ds.data_ptr(), stream) == 0
        for block in (int(b) for b in args.blocks.split(",")):
            n = total // block
            s_off = torch.arange(n, dtype=torch.int64, device=dev) * block
            s_len = torch.full((n,), block, dtype=torch.int32, device=dev)
            slot = (block + block // 255 + 16 + 8 + 15) // 16 * 16
            c_off = torch.arange(n, dtype=torch.int64, device=dev) * slot
            comp = torch.zeros(n * slot + 64, dtype=torch.uint8, device=dev)
            olen = torch.zeros(n, dtype=torch.int32, device=dev)
            back = torch.zeros(total + 64, dtype=torch.uint8, device=dev)
            blen = torch.zeros(n, dtype=torch.int32, device=dev)
            cap = torch.full((n,), block, dtype=torch.int32, device=dev)
            for with_dict in (False, True):
                def compress():
                    if with_dict:
                        rc = lib.b200lz4_compress_dev_dict(src.data_ptr(), s_off.data_ptr(), s_len.data_ptr(), n, None, 0, None,
                                                           cs.data_ptr(), comp.data_ptr(), c_off.data_ptr(), None, olen.data_ptr(),
                                                           1, 8, scratch.data_ptr(), stream)
                    else:
                        rc = lib.b200lz4_compress_dev(src.data_ptr(), s_off.data_ptr(), s_len.data_ptr(), n, None, 0, None,
                                                      comp.data_ptr(), c_off.data_ptr(), None, olen.data_ptr(), 1, 8,
                                                      scratch.data_ptr(), stream)
                    assert rc == 0, lib.b200lz4_last_error()
                t_c = timed(compress)
                d_len = (olen + 8).to(torch.int32)
                assert int(olen.min()) > 0

                def decompress():
                    if with_dict:
                        rc = lib.b200lz4_decompress_dev_dict(comp.data_ptr(), c_off.data_ptr(), d_len.data_ptr(), n, None, 0, None,
                                                             ds.data_ptr(), back.data_ptr(), s_off.data_ptr(), cap.data_ptr(),
                                                             blen.data_ptr(), 8, 0, scratch.data_ptr(), stream)
                    else:
                        rc = lib.b200lz4_decompress_dev(comp.data_ptr(), c_off.data_ptr(), d_len.data_ptr(), n, None, 0, None,
                                                        back.data_ptr(), s_off.data_ptr(), cap.data_ptr(), blen.data_ptr(), 8, 0,
                                                        scratch.data_ptr(), stream)
                    assert rc == 0, lib.b200lz4_last_error()
                t_d = timed(decompress)
                assert bool((blen == block).all()) and torch.equal(back[:total], src[:total]), "round trip failed"
                ratio = total / float((olen.to(torch.int64) + 8).sum())
                print(json.dumps({"kind": kind, "block": block, "dictionary": 65536 if with_dict else 0,
                                  "compress_ms": round(t_c, 3), "compress_GBps": round(total / t_c / 1e6, 2),
                                  "decompress_ms": round(t_d, 3), "decompress_GBps": round(total / t_d / 1e6, 2),
                                  "ratio": round(ratio, 3)}), flush=True)
            del comp, back


if __name__ == "__main__":
    main()
