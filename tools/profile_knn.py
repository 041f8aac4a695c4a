#!/usr/bin/env python3
"""Time the fused Hamming kNN sweep on one GPU.

    python tools/profile_knn.py --n 262144
Used under ncu for the profiles committed in profiles/ (small --n).
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=262144)
    ap.add_argument("--length", type=int, default=256)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dist", default="uniform")
    args = ap.parse_args()
    from prograph_b200.engine import get_engine
    from bench import make_tokens
    eng = get_engine()
    X = make_tokens(args.n, args.length, args.dist)
    tab = eng.pack(X)
    eng.hamming_knn(tab, 0, args.n, tab, args.k, drop=1)      # warm-up
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.hamming_knn(tab, 0, args.n, tab, args.k, drop=1)
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    print(f"{best:.2f} ms  {args.n * args.n / best / 1e6:.1f} Gpairs/s", flush=True)


if __name__ == "__main__":
    main()
