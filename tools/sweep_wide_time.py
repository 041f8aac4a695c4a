"""Rate of the fused Hamming sweep on long rows (pg_sweep_long.cuh), against the element-wise kernel.

Widths: 5 bit planes at L = 1792 (whole rows in the ring, the anchor) and 2048 .. 32768 (chunked
ring); 8 bit planes at L = 512, 1024, 4096 (chunked).  Every width sweeps a mutational library
(tokens 1..20 at 5 planes, 1..40 at 8; up to 8 substitutions per row, every 37th row a copy of the
one before) whose packed table is about 256 MB -- twice the 126 MB L2 -- so the stream table comes
from HBM on every pass: 240 000 rows at L = 1792, 13 100 at L = 32768.  Modes: kNN k = 16 (drop 1)
and the epsilon count (d <= 3) of 2 x 256 own rows per SM (one wave of two CTAs per SM, or every row
of smaller tables) against the whole table, and the int64 distance tile of 1024 query rows.  CUDA
events around back-to-back calls after a warm-up call, over a window of at least one second.  The
element-wise kernel (pg_hamming_values_tile on int64 rows, what the library ran at these widths
before) runs on 64 query rows of the same data.  Reported per case: Gpairs/s, residue comparisons/s
(pairs x L) and the ratio to the element-wise rate.  Every timed output is checked bit for bit
against the element-wise kernel on sampled rows.

usage: python tools/sweep_wide_time.py [--out LOG] [--cases 5:1792,5:2048,...] [--table-mb 256]
"""
import argparse
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

CASES = "5:1792,5:2048,5:4096,5:8192,5:16384,5:32768,8:512,8:1024,8:4096"


def log(fh, msg):
    print(msg, flush=True)
    if fh:
        fh.write(msg + "\n")
        fh.flush()


def device_tokens(n, L, alphabet, seed):
    """Mutational library on the device: a wild type, 1..8 substitutions per row, every 37th row a copy."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    wt = torch.randint(1, alphabet + 1, (L,), generator=g, device="cuda", dtype=torch.uint8)
    X = wt.repeat(n, 1)
    rows = torch.arange(n, device="cuda")
    for s in range(8):
        pos = torch.randint(0, L, (n,), generator=g, device="cuda")
        tok = torch.randint(1, alphabet + 1, (n,), generator=g, device="cuda", dtype=torch.uint8)
        keep = torch.randint(0, 8, (n,), generator=g, device="cuda") >= s      # 1..8 substitutions
        X[rows[keep], pos[keep]] = tok[keep]
    X[37::37] = X[36::37][: X[37::37].shape[0]]
    return X


def timed(fn, window=1.0):
    """(seconds per call, calls) over back-to-back calls between CUDA events, after one warm-up call."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    one = a.elapsed_time(b) * 1e-3
    reps = max(3, math.ceil(window / max(one, 1e-6)))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3 / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cases", default=CASES)
    ap.add_argument("--table-mb", type=float, default=256.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sweep_wide_time.py needs a CUDA device")
    from prograph_b200.engine import get_engine
    from prograph_b200.graph import distance_lut
    import operator
    eng = get_engine()
    fh = open(args.out, "w") if args.out else None
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log(fh, f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi}")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ok = True
    for case in args.cases.split(","):
        P, L = (int(v) for v in case.split(":"))
        t0 = time.time()
        words = eng.packed_words(L)
        N = int(args.table_mb * 1e6 / (P * words * 4))
        X = device_tokens(N, L, 20 if P == 5 else 40, L + P)
        tx = eng.pack(X, planes=P)
        assert (tx.planes, tx.words) == (P, words)
        X64 = X.to(torch.int64)
        kind = "whole rows" if P == 5 and words <= 56 else "chunked"
        log(fh, f"-- P={P} L={L} (W={words}, {kind}): {N} rows, packed table {N * P * words * 4 / 1e6:.0f} MB "
                f"({time.time() - t0:.1f} s set-up)")
        M = min(N, 2 * 256 * sms)
        sample = torch.tensor(sorted({0, 1, 36, 37, M // 2, M - 2, M - 1}), device="cuda")
        ref = eng.hamming_values_tile(X64, X64[sample], 0, len(sample))            # (samples, N) int64
        lut = distance_lut(words * 32, operator.le, 3, similarity=False, guard=False)
        qt = eng.gather_packed(tx, np.arange(1024))
        rates = {}
        for mode in ("knn", "count", "tile"):
            if mode == "knn":
                def run():
                    return eng.hamming_knn(tx, 0, M, tx, 16, drop=1)
                pairs_call = M * N
            elif mode == "count":
                def run():
                    return eng.hamming_eps_degrees(tx, 0, M, tx, lut)
                pairs_call = M * N
            else:
                def run():
                    return eng.hamming_tile(tx, qt)
                pairs_call = 1024 * N
            sec, reps = timed(run)
            out = run()
            if mode == "knn":
                r = ref.cpu().numpy()
                order = np.argsort(r, axis=1, kind="stable")[:, 1:17]
                good = np.array_equal(out[0][sample].cpu().numpy(), order) and \
                    np.array_equal(out[1][sample].cpu().numpy(), np.take_along_axis(r, order, axis=1))
            elif mode == "count":
                good = torch.equal(out[sample], (ref <= 3).sum(dim=1))
            else:
                qs = sample[sample < 1024]
                good = torch.equal(out[qs], ref[: len(qs)])
            ok &= bool(good)
            pairs = pairs_call / sec
            name = {"knn": "kNN k=16", "count": "eps count", "tile": "tile i64"}[mode]
            rows = f"{1024 if mode == 'tile' else M}x{N}"
            log(fh, f"P={P} L={L:5d} {name:9s} {rows:>13s}: {sec * 1e3:9.2f} ms/call ({reps:4d} calls), "
                    f"{pairs / 1e9:7.2f} Gpairs/s, {pairs * L / 1e12:6.1f} T residue comparisons/s; "
                    f"check {'ok' if good else 'MISMATCH'}")
            rates[mode] = pairs
            del out
        Qe = X64[:64]
        sec, reps = timed(lambda: eng.hamming_values_tile(X64, Qe, 0, 64))
        pe = 64 * N / sec
        log(fh, f"P={P} L={L:5d} element-wise  64x{N}: {sec * 1e3:9.2f} ms/call ({reps:4d} calls), {pe / 1e9:7.2f} "
                f"Gpairs/s, {pe * L / 1e12:6.1f} T residue comparisons/s")
        log(fh, f"P={P} L={L:5d} fused / element-wise: " +
            ", ".join(f"{m} {rates[m] / pe:.1f}x" for m in ("knn", "count", "tile")))
        del X, X64, tx, ref, qt
        torch.cuda.empty_cache()
    log(fh, "all checks ok" if ok else "CHECK FAILED")
    if fh:
        fh.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
