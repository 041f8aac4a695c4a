"""Time of extend_neighbours against the rebuild it replaces, on a C4-M library grown by M rows.

Library: 1 M rows x 256 residues (tokens 1..20, a wild type with 1..8 substitutions per row, every
37th row a copy of the one before), whose 160 MB packed table is larger than the 126 MB L2.  The
M in {1 000, 10 000, 100 000} new rows are more mutants of the same wild type.  The rows live on the
device as uint8 tokens; the previous graph (kNN k = 16, epsilon d <= 1) is a host table, as
build_neighbours returns it.  Per case:
  * extension: extend_neighbours(prev, A, B) end to end (pack, sweeps, upload of the previous table,
    merge / append, copy of the grown graph to the host), against the rebuild
    build_neighbours(A over B) -- both with CUDA events around calls after a warm-up call;
  * Gpairs/s of the 2NM + M^2 pairs the extension evaluates;
  * bytes/s of pg_knn_extend_merge / pg_csr_append on the case's own inputs (bytes read + written),
    against a device-to-device copy of the same bytes measured in the same run.
Every extension is compared with the rebuild bit for bit; a mismatch exits non-zero.

usage: python tools/extend_time.py [--out LOG] [--n 1000000] [--m 1000,10000,100000]
"""
import argparse
import operator
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

L_RES = 256


def log(fh, msg):
    print(msg, flush=True)
    if fh:
        fh.write(msg + "\n")
        fh.flush()


def mutants(n, wt, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = wt.repeat(n, 1)
    rows = torch.arange(n, device="cuda")
    for s in range(8):
        pos = torch.randint(0, wt.numel(), (n,), generator=g, device="cuda")
        tok = torch.randint(1, 21, (n,), generator=g, device="cuda", dtype=torch.uint8)
        keep = torch.randint(0, 8, (n,), generator=g, device="cuda") >= s
        X[rows[keep], pos[keep]] = tok[keep]
    X[37::37] = X[36::37][: X[37::37].shape[0]]
    return X


def timed(fn, reps):
    """(seconds per call) between CUDA events over `reps` back-to-back calls, after a warm-up call."""
    out = fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3 / reps, out


def same(x, y):
    names = ("indptr", "idx", "w") if hasattr(y, "indptr") else ("idx", "w")
    return all(getattr(x, n).dtype == getattr(y, n).dtype and np.array_equal(getattr(x, n), getattr(y, n))
               for n in names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", default="1000,10000,100000")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("extend_time.py needs a CUDA device")
    from prograph_b200 import build_neighbours, extend_neighbours
    from prograph_b200.engine import get_engine
    from prograph_b200.graph import distance_lut, informative_table
    eng = get_engine()
    fh = open(args.out, "w") if args.out else None
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log(fh, f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi}")
    N = args.n
    g = torch.Generator(device="cuda").manual_seed(1)
    wt = torch.randint(1, 21, (L_RES,), generator=g, device="cuda", dtype=torch.uint8)
    A = mutants(N, wt, 2)
    ok = True
    for mode, kw in (("kNN k=16", dict(k=16)), ("eps d<=1", dict(eps=1))):
        prev = build_neighbours(A, **kw)
        log(fh, f"-- {mode}: previous graph of {N} x {L_RES} built")
        for m in (int(v) for v in args.m.split(",")):
            B = mutants(m, wt, 3 + m)
            C = torch.cat([A, B])
            t_ext, ext = timed(lambda: extend_neighbours(prev, A, B, **kw), 3)
            t_re, re = timed(lambda: build_neighbours(C, **kw), 2)
            good = same(ext, re)
            ok &= good
            pairs = 2 * N * m + m * m
            # the new kernel of this mode on the case's own inputs, against a device copy of the same bytes
            packed = informative_table(eng, eng.pack(C))
            fresh = eng.gather_packed(packed, np.arange(N, N + m))
            if "k" in kw:
                ci, cw = eng.hamming_knn(packed, 0, N, fresh, 16, drop=0)
                pi, pw = (torch.from_numpy(a).cuda() for a in (prev.idx, prev.w))
                t_k, _ = timed(lambda: eng.knn_extend_merge(pi, pw, ci, cw, N, 16), 20)
                nbytes = N * (16 + 16 + 16) * 16
                kname = "pg_knn_extend_merge"
            else:
                add = eng.hamming_eps(packed, 0, N, fresh, distance_lut(packed.words * 32, operator.le, 1, False))
                old = tuple(torch.from_numpy(a).cuda() for a in (prev.indptr, prev.idx, prev.w))
                t_k, _ = timed(lambda: eng.csr_append(old, add, N), 20)
                nnz = old[1].numel() + add[1].numel()
                nbytes = 2 * nnz * 16 + 3 * (N + 1) * 8
                kname = "pg_csr_append"
            src = torch.empty(nbytes // 2, dtype=torch.uint8, device="cuda")
            dst = torch.empty_like(src)
            t_c, _ = timed(lambda: dst.copy_(src), 20)
            log(fh, f"{mode} N={N} M={m:6d}: extension {t_ext * 1e3:8.2f} ms, rebuild {t_re * 1e3:8.2f} ms "
                    f"({t_re / t_ext:5.1f}x); {pairs / t_ext / 1e9:7.1f} Gpairs/s of 2NM+M^2 = {pairs:.3e} pairs; "
                    f"{kname} {t_k * 1e3:6.3f} ms = {nbytes / t_k / 1e9:6.0f} GB/s vs device copy "
                    f"{nbytes / t_c / 1e9:6.0f} GB/s; result {'identical to the rebuild' if good else 'MISMATCH'}")
            del B, C, ext, re, packed, fresh, src, dst
            torch.cuda.empty_cache()
    log(fh, "all results identical to the rebuild" if ok else "CHECK FAILED")
    if fh:
        fh.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
