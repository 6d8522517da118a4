#!/usr/bin/env python
"""Sequence mix of the reference's LZ4 blocks, on the CPU: datagen's bytes compressed by the oracle restatement
(oracle/), each block parsed back into its sequences.

    python tools/sequence_mix.py [--kinds sparse01,records,mixed] [--block 640000] [--blocks 1] [--accel 400] [--seed 2]

Per kind: sequences per block, and how many have 0, 1 and 15+ literals and a match longer than 32 bytes, plus the
compression ratio.  The GPU compressor's output is byte-identical to the restatement, so these are the sequences the
finder produces.  Divide a kernel time by them to get cycles per sequence."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def sequences(block):
    """(literal length, match length) of every sequence of an LZ4 block; the last one has match length 0."""
    out, i, n = [], 0, len(block)
    while i < n:
        tok = block[i]; i += 1
        lit = tok >> 4
        if lit == 15:
            while True:
                b = block[i]; i += 1; lit += b
                if b != 255:
                    break
        i += lit
        if i >= n:
            out.append((lit, 0))
            break
        i += 2
        ml = tok & 15
        if ml == 15:
            while True:
                b = block[i]; i += 1; ml += b
                if b != 255:
                    break
        out.append((lit, ml + 4))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kinds", default="sparse01,records,mixed")
    ap.add_argument("--block", type=int, default=640000)
    ap.add_argument("--blocks", type=int, default=1, help="blocks per kind (counts are per block)")
    ap.add_argument("--accel", type=int, default=400)
    ap.add_argument("--seed", type=int, default=2)
    args = ap.parse_args()
    from streamly_lz4_b200 import datagen
    from oracle.oracle import Oracle
    ref = Oracle("auto")
    print(f"oracle: {ref.kind}; {args.blocks} block(s) of {args.block} bytes, acceleration {args.accel}, seed {args.seed}")
    print(f"{'kind':10s} {'sequences':>10s} {'0 lit':>8s} {'1 lit':>8s} {'15+ lit':>8s} {'match>32':>9s} {'ratio':>6s}")
    for kind in args.kinds.split(","):
        data = datagen.make(kind, args.seed, args.block * args.blocks).tobytes()
        arrays = [data[i:i + args.block] for i in range(0, len(data), args.block)]
        blocks = ref.compress_chunks(arrays, args.accel, linked=False)
        c = [0] * 5
        for b in blocks:
            seqs = [s for s in sequences(b[8:]) if s[1]]     # (8-byte LZ4.hs header; the final literals are no sequence)
            c[0] += len(seqs)
            c[1] += sum(1 for l, _ in seqs if l == 0)
            c[2] += sum(1 for l, _ in seqs if l == 1)
            c[3] += sum(1 for l, _ in seqs if l >= 15)
            c[4] += sum(1 for _, m in seqs if m > 32)
        k = len(blocks)
        ratio = len(data) / sum(len(b) - 8 for b in blocks)
        print(f"{kind:10s} {c[0] / k:10.0f} {c[1] / k:8.0f} {c[2] / k:8.0f} {c[3] / k:8.0f} {c[4] / k:9.0f} {ratio:6.2f}")


if __name__ == "__main__":
    main()
