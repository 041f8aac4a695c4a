#!/usr/bin/env python3
"""A/B timing of the symmetric sweeps' schedule knobs in ONE process (the library reads its
environment at every call): L2 band size, bootstrap columns, emulated ranks.

    python tools/sym_variants.py --n 1000000 --band 0,24,40 [--eps 1] [--world 8 --rank -1] [--stats]
"""
import argparse
import itertools
import json
import operator
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--length", type=int, default=256)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--dist", default="uniform")
    ap.add_argument("--delay", default="0", help=argparse.SUPPRESS)
    ap.add_argument("--band", default="0,24")
    ap.add_argument("--boot", default="8192")
    ap.add_argument("--eps", type=int, default=0)
    ap.add_argument("--world", type=int, default=1, help="emulate one rank of a `world`-GPU build")
    ap.add_argument("--rank", type=int, default=0, help="-1: every rank of `world` in turn")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--stats", action="store_true")
    args = ap.parse_args()
    from bench import make_tokens, make_gb1_library
    from prograph_b200 import graph
    from prograph_b200.engine import get_engine
    eng = get_engine()
    X = make_gb1_library() if args.dist == "gb1" else make_tokens(args.n, args.length, args.dist)
    n = X.shape[0]
    tab = eng.pack(X)
    lut = graph.distance_lut(tab.words * 32, operator.le, args.eps, False) if args.eps else None
    if args.stats:
        os.environ["PG_SYM_STATS"] = "1"
    ranks = list(range(args.world)) if args.rank < 0 else [args.rank]
    for delay, band, boot, rank in itertools.product(args.delay.split(","), args.band.split(","), args.boot.split(","),
                                                     ranks):
        args.rank = rank
        os.environ["PG_SYM_BAND_MB"], os.environ["PG_SYM_BOOT"] = band, boot
        os.environ["PG_SYM_DELAY"] = delay
        best = None
        for _ in range(args.reps):
            eng.time_sweeps(True)
            eng.sweep_times(reset=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if args.eps:
                if args.world > 1:
                    eng.hamming_eps_sym(tab, lut, args.rank, args.world, mode=1, capacity=int(120 * n / args.world) + (4 << 20))
                else:
                    graph.hamming_eps_graph(eng, tab, lut, False, 0, 1, None)
            elif args.world > 1:
                bt = graph.sym_boot_rows(n)
                seed = eng.hamming_knn_boot(tab, 0, n, bt, args.k + 1)
                eng.hamming_knn_sym(tab, args.k + 1, args.rank, args.world, lists=seed, boot_rows=bt, mode=1)
                eng.sym_check()
            else:
                graph.hamming_knn_graph(eng, tab, args.k, False, 0, 1, None)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b)
            sw = eng.sweep_times(reset=True)
            eng.time_sweeps(False)
            if best is None or ms < best[0]:
                best = (ms, sw)
        print(json.dumps({"n": n, "dist": args.dist, "eps": args.eps, "world": args.world, "rank": args.rank,
                          "delay": delay, "band_mb": band, "boot": boot, "build_ms": round(best[0], 2),
                          "sweeps_ms": [round(v, 2) for v in best[1]],
                          "gpairs_n2": round(n * n / best[0] / 1e6, 1)}), flush=True)


if __name__ == "__main__":
    main()
