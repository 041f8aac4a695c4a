"""Rate of the Minkowski p=2 GEMM (pg_gemm.cu) on wide integer rows, against the element-wise kernel.

For K in {256 (resident A tiles), 512, 1184, 5376 (K-chunked ring)}: a 262 144-row mutational
library (tokens 1..20, fp16 chain, about 4 substitutions per row; 67 MB .. 1.4 GB of int8 operands,
so the dataset does not stay in the 126 MB L2 beyond K = 256) is timed as a materialised tile and as
fused kNN with k = 1 and k = 16 (256 query rows per SM), with CUDA events around back-to-back calls after a warm-up call, over
a window of at least one second.  The element-wise kernel (pg_minkowski_tile) runs on 64 query rows of
the same data.  Reported: Gpairs/s, int8 operations/s (2 K per pair), the share of the int8 MMA rate
measured by eng.i8_mma_peak() in the same run, and the L2 operand traffic (bytes streamed per pair:
K / 256 with resident A tiles, 3 K / 256 chunked) against the ~5.8 TB/s the resident kernel was
measured to pull (DESIGN.md 4.1b).  Every timed output is checked bit for bit against the element-wise
kernel on sampled query rows.

usage: python tools/gemm_wide_time.py [--out LOG] [--widths 256,512,1184,5376] [--rows 262144]
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

L2_STREAM = 5.8e12      # bytes/s the resident kernel pulled out of L2 (profiles/r1_ncu_notes.md)


def log(fh, msg):
    print(msg, flush=True)
    if fh:
        fh.write(msg + "\n")
        fh.flush()


def device_tokens(n, L, seed):
    """Mutational library on the device: a wild type, ~4 substitutions per row, every 37th row a copy."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    wt = torch.randint(1, 21, (L,), generator=g, device="cuda", dtype=torch.uint8)
    X = wt.repeat(n, 1)
    for _ in range(4):
        pos = torch.randint(0, L, (n,), generator=g, device="cuda")
        X[torch.arange(n, device="cuda"), pos] = torch.randint(1, 21, (n,), generator=g, device="cuda",
                                                               dtype=torch.uint8)
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
    ap.add_argument("--widths", default="256,512,1184,5376")
    ap.add_argument("--rows", type=int, default=262144)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("gemm_wide_time.py needs a CUDA device")
    from prograph_b200.engine import get_engine
    eng = get_engine()
    fh = open(args.out, "w") if args.out else None
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log(fh, f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi}")
    peak, _ = eng.i8_mma_peak()
    log(fh, f"measured int8 MMA peak (eng.i8_mma_peak): {peak / 1e15:.3f} POPS")
    N = args.rows
    ok = True
    for K in (int(w) for w in args.widths.split(",")):
        t0 = time.time()
        X = device_tokens(N, K, K)
        g = eng.gemm_pack(X, max_token=31)
        Xh = X.to(torch.float16)
        bpp = (K / 256) * (1 if K <= 256 else 3)          # L2 operand bytes per pair
        log(fh, f"-- K = {K}: {N} rows, {N * K / 1e6:.0f} MB of operands ({time.time() - t0:.1f} s set-up)")
        # kNN: one CTA of 256 query rows per SM (a smaller M leaves SMs idle); the tile launcher splits
        # the dataset over gridDim.y itself when there are few query rows
        mk = 256 * torch.cuda.get_device_properties(0).multi_processor_count
        for mode, k, M in (("tile", 0, 4096), ("knn", 1, mk), ("knn", 16, mk)):
            q = eng.gemm_pack(X[:M], max_token=31, K=g.K)
            rows = sorted({0, 1, 36, 37, 1000, M // 2, M - 2, M - 1})   # sampled query rows (the first M dataset rows)
            assert 0 <= rows[0] and rows[-1] < M <= N
            sample = torch.tensor(rows, device="cuda")
            if mode == "tile":
                def run():
                    return eng.minkowski2_gemm_tile(g, q, 0)
            else:
                def run(k=k):
                    return eng.minkowski2_gemm_knn(g, q, k, 0, 0)
            sec, reps = timed(run)
            pairs = M * N / sec
            ops = 2 * K * pairs
            frac = ops / peak
            l2 = pairs * bpp
            bound = "L2" if l2 / L2_STREAM > frac else "tensor"
            # check: sampled query rows against the element-wise kernel, bit for bit
            out = run()
            ref = eng.minkowski_tile(Xh, Xh[sample], 0, len(sample))
            if mode == "tile":
                good = torch.equal(out[sample].view(torch.int16), ref.view(torch.int16))
            else:
                refs = np.stack([np.argsort(r, kind="stable")[:k] for r in ref.float().cpu().numpy()])
                good = np.array_equal(out[0][sample].cpu().numpy(), refs) and torch.equal(
                    out[1][sample].view(torch.int16), torch.gather(ref, 1, torch.as_tensor(refs, device="cuda")).view(torch.int16))
            ok &= bool(good)
            name = "tile fp16" if mode == "tile" else f"kNN k={k}"
            log(fh, f"K={K:5d} {name:9s} {M}x{N}: {sec * 1e3:8.2f} ms/call ({reps} calls), {pairs / 1e9:7.1f} Gpairs/s, "
                    f"{ops / 1e12:7.1f} int8 TOPS = {100 * frac:5.1f} % of measured peak, L2 {l2 / 1e12:5.2f} TB/s "
                    f"-> {bound}-bound; check {'ok' if good else 'MISMATCH'}")
            del q, out
        Qe = Xh[:64]
        sec, reps = timed(lambda: eng.minkowski_tile(Xh, Qe, 0, 64))
        pairs_e = 64 * N / sec
        log(fh, f"K={K:5d} element-wise fp16 64x{N}: {sec * 1e3:8.2f} ms/call ({reps} calls), {pairs_e / 1e9:7.2f} Gpairs/s")
        del X, g, Xh
        torch.cuda.empty_cache()
    log(fh, "all checks ok" if ok else "CHECK FAILED")
    if fh:
        fh.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
