#!/usr/bin/env python3
"""Headline benchmark: Gpairs/s of the Hamming all-pairs + kNN (k=16) graph build on a
synthetic library of N=1M sequences, L=256 (BASELINE.json configs[3]), at 1/2/4/8 B200, with the
threshold (epsilon) graphs of the same path as a second block of the same JSON line.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 3 --warmup 3
    python bench.py --impl reference --steps 3 --warmup 1      # CPU arm (oracle port)
    python bench.py --steps 3 --warmup 3 --dump-outputs bench_outputs   # + the last step's kNN lists as .npy

A step = one full graph build: pack the token table into bit planes, build the kNN lists of
all N rows with the fused Hamming+top-k sweeps, finalise, exchange.  The build is the symmetric
one (prograph_b200/csrc/pg_sweep_sym.cuh): d(i,j) == d(j,i), so after a one-sided bootstrap pass
over the first 8192 columns every unordered pair is evaluated ONCE and offered to both rows'
lists.  The metric still counts all N^2 ordered pairs -- what the reference evaluates and what
`--one-sided` (the previous kernel) evaluates -- while the roofline is computed on the pair
evaluations actually issued (`pairs_evaluated`).  `value` times the build with the uint8 token
table resident in HBM and the whole graph left on every GPU; `e2e` times the public API call
(prograph_b200.build_neighbours) on a pinned HOST token table: H2D of every rank's rows + the
same sweeps + D2H of the neighbour lists (with several ranks: output="sharded", every rank copies
the rows of its own block, so the graph reaches host memory exactly once).  Ranks own bands of
stream rows of the triangle holding equal numbers of pair evaluations (total work fixed ->
"strong" scaling); the exchange is an all-to-all of candidate lists + an all-gather of merged
keys.  Times are CUDA-event times, max over ranks.  One JSON line is printed by rank 0.

After the timed regions (never inside them) the run checks itself and exits non-zero on a
mismatch: the whole symmetric result against the one-sided sweep on the device, sampled rows
(band and bootstrap edges, block edges, last row, random rows) against the CPU oracle, every
rank against rank 0 (`parity`).  The `eps` block does the same for the threshold graphs:
C4-M (mutational library, N=1M) eps=1 as a CSR, eps=2 as a degree census (its CSR would hold
1.6e10 edges = 250 GB), and the GB1-style 160 000 x 56 library (C3) with its known answers.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Gpairs/s Hamming all-pairs + kNN graph build, N=1M L=256"
UNIT = "Gpairs/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000, help="sequences (default: the headline 1M)")
    ap.add_argument("--length", type=int, default=256)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--dist", default="uniform", choices=["uniform", "mutational"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eps", action="store_true", help="skip the threshold-graph block")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run parity checks")
    ap.add_argument("--no-queries", action="store_true", help="skip the distance-to-dataset query block (C5)")
    ap.add_argument("--one-sided", action="store_true",
                    help="evaluate all N^2 ordered pairs with the one-sided sweep (no symmetry)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the kNN lists of the last one as DIR/knn_{rows,idx,w}.npy "
                         "(float64; a fixed, seeded sample of rows on large tables)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU build computed: it needs --impl b200")
    return args


def make_tokens(n, L, kind, seed=0):
    """SURVEY.md §8(d) C4: U = iid uniform residues (adversarial ties), M = mutational library.
    `seed` != 0 draws another set of rows around the SAME wild type (the query set of C5)."""
    rng = np.random.default_rng(0)
    if kind == "uniform":
        return np.random.default_rng(seed).integers(1, 21, size=(n, L), dtype=np.uint8)
    wt = rng.integers(1, 21, size=L, dtype=np.uint8)
    if seed != 0:
        rng = np.random.default_rng(seed)
    X = np.tile(wt, (n, 1))
    m = rng.integers(1, 9, size=n)
    for j in range(8):
        rows = np.nonzero(m > j)[0]
        pos = rng.integers(0, L, size=len(rows))
        X[rows, pos] = (X[rows, pos] - 1 + rng.integers(1, 20, size=len(rows))) % 20 + 1
    return X


GB1 = "MTYKLILNGKTLKGETTTEAVDAATAEKVFKQYANDNGVDGEWTYDDATKTFTVTE"
GB1_SITES = (38, 39, 40, 53)
ALPHABET = "ACDEFGHIKLMNPQRSTVWY"


def make_gb1_library():
    """SURVEY.md §8(d) C3: every combination of the 20 residues at 4 sites of the 56-residue GB1 domain,
    in itertools.product order -> (160 000, 56) uint8 tokens 1..20."""
    tok = {a: i + 1 for i, a in enumerate(ALPHABET)}
    wt = np.array([tok[c] for c in GB1], dtype=np.uint8)
    X = np.tile(wt, (20 ** 4, 1))
    idx = np.indices((20, 20, 20, 20)).reshape(4, -1)
    for s, site in enumerate(GB1_SITES):
        X[:, site] = idx[s] + 1
    return X


def config_of(args, world):
    return {
        "workload": f"C4-{'U' if args.dist == 'uniform' else 'M'}: synthetic {args.n} sequences, L={args.length}, "
                    f"Hamming kNN k={args.k}, N^2 ordered pairs counted, "
                    + ("one-sided sweep, rows" if args.one_sided else "symmetric sweep (each unordered pair evaluated "
                       "once), bands of the triangle") + f" sharded over {world} GPU(s)",
        "n_sequences": args.n, "seq_len": args.length, "k": args.k, "distribution": args.dist,
        "parallelism": (f"row-block x{world}" if args.one_sided else f"triangle bands x{world}"),
        "l2": "inputs exceed L2 (126 MB): 160 MB packed table + 136 MB of per-row lists + 8 MB of filter words are "
              "re-read every step",
    }


emit = None      # set by main(): writes the one JSON line to the real stdout


# ----------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm restated with torch CPU ops (oracle port)
# ----------------------------------------------------------------------------------------
def cpu_reference_batches(tokens_u8, k, n_batches, budget_s=None):
    """hamming.py:34 + prograph.py:726,756-762 on the host: fp16 staging, batches of 8 query
    rows against all N, full sort per row.  Returns (pairs, seconds, batches done)."""
    import torch
    from oracle import prograph_oracle as O
    X = torch.from_numpy(tokens_u8).to(torch.float16)
    n = X.shape[0]
    t0 = time.perf_counter()
    done = 0
    for b in range(n_batches):
        batch = X[(8 * b) % n:(8 * b) % n + 8]
        O.reference_knn_batch_torch(X, batch, k)
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done * 8 * n, dt, done


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    tokens = make_tokens(args.n, args.length, args.dist)
    per_step = 2            # batches of 8 query rows per step: a bounded sample of the build
    for _ in range(args.warmup):
        cpu_reference_batches(tokens, args.k, 1)
    t0 = time.perf_counter()
    pairs = 0
    for _ in range(args.steps):
        p, _, _ = cpu_reference_batches(tokens, args.k, per_step)
        pairs += p
    dt = time.perf_counter() - t0
    val = pairs / dt / 1e9
    sample = f"{per_step * 8} query rows x all {args.n} columns per step (reference batches of 8), torch CPU fp16"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "fp16 compare -> int64", "data": "synthetic",
        "config": config_of(args, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def ncu_traffic_bytes(n, world, capture):
    """dram__bytes_read.sum + dram__bytes_write.sum of the sweep kernel, per launch, from the
    committed ncu capture of this exact configuration (profiles/); None otherwise.  ncu is the only
    source of DRAM counters, so this figure cannot be measured inside an un-profiled run."""
    if n != 1_000_000 or world != 1:
        return None
    path = os.path.join(ROOT, "profiles", capture)
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total = 0.0
    try:
        for line in open(path):
            parts = [p.strip().strip('"') for p in line.split(",")]
            if len(parts) == 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                total += float(parts[2]) * scale.get(parts[1], 1.0)
    except OSError:
        return None
    return total or None


def triangle_pairs(n, boot, band):
    """Pair evaluations of the symmetric sweep inside the stream-row band [band[0], band[1]): every
    256-row block sweeps the stream rows from its own block on (bootstrap blocks: from `boot` on)."""
    total = 0.0
    for rb in range(0, -(-n // 256)):
        a, b = rb * 256, min(n, rb * 256 + 256)
        lo = max(boot if a < boot else a, band[0])
        total += float(b - a) * max(0, band[1] - lo)
    return total


# ----------------------------------------------------------------------------------------
# parity helpers (run after the timed regions)
# ----------------------------------------------------------------------------------------
def sample_rows(n, world, eng, words, boot, count=256, seed=7):
    """Rows whose lists meet every seam of the build: bootstrap edge, row-block and tile edges, the
    band edges of every rank, the row-block shard edges, first / last row -- plus random rows."""
    from prograph_b200 import shard
    rows = {0, 1, 255, 256, 511, 512, n - 1, n - 2, n // 2}
    if boot:
        rows |= {boot - 1, boot, boot + 1, boot + 255, boot + 256}
    for r in range(world):
        if world > 1:
            a, b = eng.sym_band(n, words, boot, r, world)
            rows |= {a - 1, a, a + 1, b - 1, b}
        r0, rr = shard.row_range(n, r, world)
        rows |= {r0 - 1, r0, r0 + rr - 1}
    rows = {r for r in rows if 0 <= r < n}
    rng = np.random.default_rng(seed)
    while len(rows) < min(count, n):
        rows.add(int(rng.integers(0, n)))
    return np.array(sorted(rows), dtype=np.int64)


DUMP_BYTES = 32 << 20     # idx + w written by --dump-outputs (the row list adds at most 1/(2k) of that)


def dump_knn(out_dir, idx, w):
    """--dump-outputs: the (idx, w) lists of a kNN build -- what build_neighbours hands its caller -- as
    float64 .npy files (exact for every index and integer distance).  Tables whose lists exceed
    DUMP_BYTES are written for a fixed, seeded sample of rows; knn_rows.npy lists the rows written."""
    import torch
    n, kk = idx.shape
    cap = max(1, DUMP_BYTES // (16 * max(1, kk)))
    rows = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, size=cap, replace=False))
    sel = torch.from_numpy(rows).to(idx.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("rows", rows), ("idx", idx[sel].cpu().numpy()), ("w", w[sel].cpu().numpy())):
        np.save(os.path.join(out_dir, f"knn_{name}.npy"), a.astype(np.float64))


def all_true(flag, world, device):
    import torch
    import torch.distributed as dist
    t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(int(t.item()))


def same_on_all_ranks(tensors, rank, world):
    """Every rank holds bit-identical copies of `tensors` (compared with rank 0's)."""
    import torch
    import torch.distributed as dist
    if world <= 1:
        return True
    ok = True
    for t in tensors:
        ref = t.clone()
        dist.broadcast(ref, src=0)
        ok &= bool(torch.equal(ref, t))
        del ref
    return all_true(ok, world, tensors[0].device)


# ----------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.one_sided:
        os.environ["PG_KNN_SYM"] = "0"
    from prograph_b200 import build_neighbours
    from prograph_b200 import graph, shard, trace
    from prograph_b200.engine import get_engine
    eng = get_engine()
    n, L, k = args.n, args.length, args.k
    cores = len(os.sched_getaffinity(0))

    tokens = make_tokens(n, L, args.dist)
    host = torch.from_numpy(tokens).pin_memory()
    dev = host.to(eng.device)
    row0, rows = shard.row_range(n, rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=eng.device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def max_over_ranks(d):
        """{phase: ms} -> max over ranks per phase (rank 0's key set)."""
        keys = sorted(d)
        t = torch.tensor([d[key] for key in keys], device=eng.device, dtype=torch.float64)
        if world > 1 and len(keys):
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {key: float(v) for key, v in zip(keys, t.tolist())}

    last = {}

    def step_resident():
        with trace.phase("pack"):
            tab = eng.pack(dev)
        last["knn"] = graph.hamming_knn_graph(eng, tab, k, False, rank, world, None)[:2]

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.launch_count(reset=True)
    eng.time_sweeps(True)
    eng.sweep_time(reset=True)
    trace.enable_timing(True)
    ms_total = timed(step_resident, args.steps)
    phases = max_over_ranks({key: v / args.steps for key, v in trace.phases().items()})
    trace.enable_timing(False)
    sweep_list = eng.sweep_times(reset=True)
    eng.time_sweeps(False)
    launches = eng.launch_count(reset=True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_knn(args.dump_outputs, *last["knn"])
    pairs = float(n) * float(n)
    value = pairs * args.steps / (ms_total * 1e-3) / 1e9

    # ---- end to end through the public API, host buffers in, host arrays out -------------
    e2e = None
    if not args.no_e2e:
        out_mode = "sharded" if world > 1 else "replicated"
        got = {}

        def step_e2e():
            got["t"] = build_neighbours(host, k=k, output=out_mode)
        step_e2e()
        step_e2e()          # two warm-ups: the pinned result buffers of two consecutive builds alternate
        e2e_steps = max(1, min(args.steps, 3))
        trace.enable_timing(True)
        e2e_ms = timed(step_e2e, e2e_steps)
        e2e_phases = max_over_ranks({key: v / e2e_steps for key, v in trace.phases().items()})
        trace.enable_timing(False)
        kk = min(k, n - 1)
        e2e = {"value": pairs * e2e_steps / (e2e_ms * 1e-3) / 1e9, "unit": UNIT,
               # every rank uploads only its own rows and reads back only its own rows: one copy of the
               # token table in, one copy of the graph out, summed over the ranks
               "h2d_bytes_per_step": int(host.numel()), "d2h_bytes_per_step": int(n * kk * 16),
               "ms_per_step": e2e_ms / e2e_steps, "phases_ms": e2e_phases,
               "api": f"prograph_b200.build_neighbours(pinned uint8 tokens, k={k}, output='{out_mode}') -> numpy "
                      "idx/weights" + (" of this rank's row block (the graph reaches host memory once)"
                                       if world > 1 else "")}
        # the API result of the last step must be what the resident build produced
        if not args.no_parity:
            t = got["t"]
            gi, gw = last["knn"]
            e2e["matches_resident"] = all_true(
                bool(np.array_equal(t.idx, gi[t.row0:t.row0 + t.n_rows].cpu().numpy())
                     and np.array_equal(t.w, gw[t.row0:t.row0 + t.n_rows].cpu().numpy())), world, eng.device)
        del got

    # ---- parity of the timed result (outside every timed region) --------------------------------
    words = eng.packed_words(L)
    symmetric = (not args.one_sided) and len(sweep_list) == 2 * args.steps
    boot = graph.sym_boot_rows(n) if symmetric else 0
    parity = None
    if not args.no_parity:
        gi, gw = last["knn"]
        tab = eng.pack(dev)
        # (a) every entry of this rank's row block against the one-sided sweep (all rows at N=1)
        oi, ow = eng.hamming_knn(tab, row0, rows, tab, min(k, n - 1), drop=1)
        full = all_true(bool(torch.equal(oi, gi[row0:row0 + rows]) and torch.equal(ow, gw[row0:row0 + rows])),
                        world, eng.device)
        del oi, ow
        # (b) all ranks hold the same graph
        ident = same_on_all_ranks([gi, gw], rank, world)
        # (c) sampled rows against the CPU oracle (rank 0; C restatement, pinned by tests/ to the numpy
        #     oracle, which is pinned to fixtures generated from the unmodified reference)
        ok_oracle, n_oracle = True, 0
        if rank == 0:
            from oracle import c_oracle as CO
            srows = sample_rows(n, world, eng, words, boot)
            planes = CO.pack(tokens)
            ri, rd = CO.hamming_knn_rows(planes, L, srows, min(k, n - 1), threads=cores)
            sel = torch.from_numpy(srows).to(eng.device)
            ok_oracle = bool(np.array_equal(gi[sel].cpu().numpy(), ri) and np.array_equal(gw[sel].cpu().numpy(), rd))
            n_oracle = len(srows)
            del planes
        ok_oracle = all_true(ok_oracle, world, eng.device)
        parity = {"rows_vs_oracle": n_oracle, "oracle_ok": ok_oracle, "full_vs_onesided": full,
                  "ranks_identical": ident, "ok": bool(ok_oracle and full and ident),
                  "how": "one-sided sweep (pg_hamming_knn) over every row of each rank's block; rows sampled at "
                         "band / bootstrap / block edges + random ones against oracle/hamming_knn_cpu.c; "
                         "broadcast of rank 0's idx/w compared on every rank"}
        if e2e is not None and "matches_resident" in e2e:
            parity["ok"] = bool(parity["ok"] and e2e["matches_resident"])
        del tab
    last.clear()

    # ---- threshold graphs: the second headline ----------------------------------------------------
    eps_block = None
    if not args.no_eps and not args.one_sided:
        del dev, host
        torch.cuda.empty_cache()
        eps_block = run_eps_block(args, eng, rank, world, timed, max_over_ranks, cores)
        if parity is not None and eps_block is not None:
            parity["eps_ok"] = bool(all(c.get("parity", {}).get("ok", True) for c in eps_block["cases"]))
            parity["ok"] = bool(parity["ok"] and parity["eps_ok"])

    # ---- distance-to-dataset queries (BASELINE.json configs[4]) -----------------------------------
    query_block = None
    if not args.no_queries and not args.one_sided:
        query_block = run_query_block(args, eng, rank, world, timed, cores)
        if parity is not None and query_block is not None:
            parity["queries_ok"] = bool(query_block.get("parity_ok", True))
            parity["ok"] = bool(parity["ok"] and parity["queries_ok"])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if parity is not None and not parity["ok"]:
            sys.exit(1)
        return

    # ---- roofline of the dominant kernel, on the pair evaluations it actually issued ---------
    lane_ops_per_pair = 7 * words                       # 5 LOP3 + 1 POPC + 1 IADD per 32 residues
    if symmetric:
        # rank 0's share: bootstrap rectangle + its piece of the triangle (one GPU: everything;
        # several: the band of stream rows the library's planner gives rank 0)
        boot_pairs = float(shard.row_range(n, 0, world)[1]) * boot
        band = (0, n) if world == 1 else eng.sym_band(n, words, boot, 0, world)
        tri_pairs = triangle_pairs(n, boot, band)
        kernel_ms = sum(sweep_list[1::2]) / args.steps
        boot_ms = sum(sweep_list[0::2]) / args.steps
        pairs_per_launch, kernel_name = tri_pairs, "pg::sweep_sym_kernel<5,8,KNN>"
        capture = "r2_ncu_sym_1m_dram.csv"
    else:
        boot_pairs, boot_ms = 0.0, 0.0
        kernel_ms = sum(sweep_list) / max(1, len(sweep_list))
        pairs_per_launch, kernel_name = float(rows) * float(n), "pg::sweep_kernel<5,8,KNN>"
        capture = "r1_ncu_sweep_r1d.csv"
    mix_ops, _ = eng.int_peak(mix=0, iters=2048)
    lop_ops, _ = eng.int_peak(mix=1, iters=2048)
    popc_ops, _ = eng.int_peak(mix=2, iters=2048)
    roofline = None
    if sweep_list:
        achieved = lane_ops_per_pair * pairs_per_launch / (kernel_ms * 1e-3)
        # the binding pipe is the ALU pipe's LOP3 rate: 5 of the 7 lane-ops of a word-pair are LOP3s, so
        # a kernel that keeps that pipe full runs at 7/5 of the measured LOP3 rate
        peak_ops = lop_ops * 7.0 / 5.0
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        packed_bytes = float(n) * 5 * words * 4
        hbm_algo = packed_bytes + float(n) * (k + 1) * 8     # table read once + lists written once
        traffic = ncu_traffic_bytes(n, world, capture)
        roofline = {
            "bound": "int-alu", "kernel": kernel_name, "achieved": achieved / 1e12,
            "peak": peak_ops / 1e12, "unit": "Tlane-op/s", "frac": achieved / peak_ops,
            "peak_source": "measured live, conservative: 7/5 x the LOP3-only rate of pg_measure_int_peak (a register-only "
                           "kernel); 5 of the 7 lane-ops per 32 residues and pair are LOP3s on the ALU pipe",
            "frac_of_mix_probe": achieved / mix_ops, "mix_probe_tlops": mix_ops / 1e12,
            "lane_ops_per_pair": lane_ops_per_pair, "pairs_evaluated_per_launch": pairs_per_launch,
            "ordered_pairs_counted_per_step": float(n) * float(n),
            "kernel_ms": kernel_ms, "kernel_launches": args.steps,
            "kernel_share_of_step": kernel_ms * args.steps / ms_total,
            "gpairs_evaluated_per_s_kernel": pairs_per_launch / (kernel_ms * 1e-3) / 1e9,
            "bootstrap": ({"rows": boot, "pairs_evaluated": boot_pairs, "kernel": "pg::sweep_kernel<5,8,KNN>",
                           "kernel_ms": boot_ms} if symmetric else None),
            "lop3_peak_tlops": lop_ops / 1e12, "popc_peak_tlops": popc_ops / 1e12,
            "traffic": traffic,
            "traffic_source": (f"profiles/{capture} (ncu dram__bytes_read.sum + dram__bytes_write.sum of this kernel at "
                               "this size; DRAM counters exist only under ncu)" if traffic else None),
            "hbm": {"algorithmic_bytes_per_launch": hbm_algo, "achieved_gbs": hbm_algo / (kernel_ms * 1e-3) / 1e9,
                    "peak_gbs": peaks.get("hbm_gbs", 6650.0),
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                    "note": "compute-bound kernel: the HBM roofline is not the binding one"},
        }

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(cores)
        cpu_reference_batches(tokens, k, 1)
        p, dt, done = cpu_reference_batches(tokens, k, 16, budget_s=20.0)
        # second, best-effort CPU number (SURVEY.md §8d): uint8 compare + partial selection on all
        # cores, so that the reported baseline is not handicapped by fp16-on-CPU and the full sort
        best = None
        try:
            from oracle import prograph_oracle as O
            O.knn_batch_uint8(tokens, tokens[:8], k, threads=cores)
            t0, nb = time.perf_counter(), 0
            while nb < 16 and time.perf_counter() - t0 < 8.0:
                O.knn_batch_uint8(tokens, tokens[8 * nb:8 * nb + 8], k, threads=cores)
                nb += 1
            bt = time.perf_counter() - t0
            best = {"value": nb * 8 * n / bt / 1e9, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"{nb * 8} query rows x all {n} columns (numpy uint8 compare in column chunks on "
                              f"{cores} threads, partial selection of the k+1 smallest (distance, index) keys)"}
        except Exception as exc:            # a reported extra, never a reason to lose the bench line
            best = {"error": repr(exc)}
        # third: the C restatement (oracle/hamming_knn_cpu.c: bit planes + popcount + sorted k+1 lists on
        # all cores), timed in a child process so that nothing it does can cost the bench line
        best_c = None
        try:
            out = subprocess.run([sys.executable, "-m", "oracle.c_oracle", "--n", str(n), "--length", str(L), "--k", str(k),
                                  "--rows", "512", "--threads", str(cores), "--dist", args.dist], cwd=ROOT,
                                 capture_output=True, text=True, timeout=180)
            lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
            best_c = json.loads(lines[-1]) if lines else {"error": (out.stderr or "no output")[-300:]}
        except Exception as exc:
            best_c = {"error": repr(exc)}
        cpu = {"value": p / dt / 1e9, "unit": UNIT, "cores": cores, "kind": "port", "best_effort": best,
               "best_effort_c": best_c,
               "sample": f"{done * 8} query rows x all {n} columns (reference batches of 8, fp16 compare + full "
                         f"sort per row, torch CPU with {cores} threads); extrapolated full build "
                         f"{pairs / (p / dt) / 3600:.1f} h"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8 tokens -> 5 bit planes, int32 popcount distances", "data": "synthetic",
        "config": config_of(args, world), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "phases_ms": phases, "parity": parity, "roofline": roofline, "eps": eps_block, "queries": query_block,
        "cpu_baseline": cpu,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.exit(1)


# ----------------------------------------------------------------------------------------
# threshold (epsilon) graphs: C4-M eps=1 (CSR), eps=2 (degree census), C3 eps=1 / eps=2
# ----------------------------------------------------------------------------------------
def run_eps_block(args, eng, rank, world, timed, max_over_ranks, cores):
    import operator
    import torch
    import torch.distributed as dist
    from prograph_b200 import build_neighbours, graph, shard, trace
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    lop_ops, _ = eng.int_peak(mix=1, iters=2048)
    int_peak = lop_ops * 7.0 / 5.0
    steps = max(1, min(args.steps, 3))
    cases = []

    def run_case(name, tokens, eps, mode, known_degree=None, oracle_rows=48):
        """mode 'csr': the public graph build (symmetric sweep -> edge keys -> radix sort -> CSR, or the
        one-sided count / fill passes for dense graphs), CSR left on every rank; 'census': degrees only."""
        n, L = tokens.shape
        words = eng.packed_words(L)
        host = torch.from_numpy(tokens).pin_memory()
        dev = host.to(eng.device)
        row0, rows = shard.row_range(n, rank, world)
        lut = graph.distance_lut(words * 32, operator.le, eps, False)
        # what the build sweeps: the residue positions that are not constant over the library
        # (graph.informative_table); the rooflines below count the lane-ops of THAT width
        swept = graph.informative_table(eng, eng.pack(dev))
        words_swept, cols_swept = swept.words, swept.L
        del swept
        res = {}

        def step():
            with trace.phase("pack"):
                tab = eng.pack(dev)
            if mode == "csr":
                res["csr"] = graph.hamming_eps_graph(eng, tab, lut, False, rank, world, None)
            else:
                with trace.phase("sweep"):
                    part = eng.hamming_eps_degrees(tab, row0, rows, tab, lut)
                with trace.phase("gather"):
                    res["deg"] = shard.gather_rows((part,), n, rank, world, None, eng)[0]

        step()
        if mode == "csr":
            step()
        reps = steps if mode == "csr" else min(steps, 2)      # the census sweeps all N^2 ordered pairs: 3 s a step
        eng.time_sweeps(True)
        eng.sweep_times(reset=True)
        trace.enable_timing(True)
        ms = timed(step, reps) / reps
        ph = max_over_ranks({key: v / reps for key, v in trace.phases().items()})
        trace.enable_timing(False)
        sw = eng.sweep_times(reset=True)
        eng.time_sweeps(False)
        # sweep launches per step: [degree sample, symmetric sweep] or [sample, count(, fill)] or [count]
        per = max(1, len(sw) // reps)
        main_ms = max(sum(sw[i::per]) / reps for i in range(per)) if sw else None
        case = {"name": name, "n": n, "L": L, "columns_swept": cols_swept, "eps": eps, "mode": mode, "ms_per_build": ms,
                "gpairs_per_s": float(n) * n / (ms * 1e-3) / 1e9, "phases_ms": ph}
        if mode == "csr":
            indptr, idx, w = res["csr"]
            nnz = int(indptr[-1].item())
            deg = indptr[1:] - indptr[:-1]
            symmetric = "csr" in ph                       # the key-sort phase only exists on the symmetric path
            if symmetric:
                band = (0, n) if world == 1 else eng.sym_band(n, words_swept, 0, 0, world)
                evaluated = triangle_pairs(n, 0, band)
            else:
                evaluated = float(shard.row_range(n, 0, world)[1]) * n          # per launch (count, and fill if it ran)
            csr_bytes = nnz * 16.0 + (n + 1) * 8.0
            csr_ms = ph.get("csr") if symmetric else None
            case.update({"nnz": nnz, "path": "symmetric sweep + key sort" if symmetric else "one-sided count / fill",
                         "roofline_sweep": ({"bound": "int-alu", "achieved": 7.0 * words_swept * evaluated / (main_ms * 1e-3) / 1e12,
                                             "peak": int_peak / 1e12, "unit": "Tlane-op/s",
                                             "frac": 7.0 * words_swept * evaluated / (main_ms * 1e-3) / int_peak,
                                             "kernel_ms": main_ms, "pairs_evaluated_per_launch": evaluated}
                                            if main_ms else None),
                         "roofline_csr": ({"bound": "hbm", "achieved": csr_bytes / (csr_ms * 1e-3) / 1e9, "peak": hbm_peak,
                                           "unit": "GB/s", "frac": csr_bytes / (csr_ms * 1e-3) / 1e9 / hbm_peak,
                                           "algorithmic_bytes": csr_bytes, "ms": csr_ms,
                                           "note": "radix sort of the 8-byte edge keys + decode; algorithmic bytes = the "
                                                   "CSR written (nnz*16 + (N+1)*8), the sort's own passes are overhead"}
                                          if csr_ms else None)})
        else:
            deg = res["deg"]
            nnz = int(deg.sum().item())
            evaluated = float(shard.row_range(n, 0, world)[1]) * n
            case.update({"nnz": nnz, "path": "one-sided count sweep (degrees only)",
                         "csr_bytes_if_materialised": nnz * 16.0 + (n + 1) * 8.0,
                         "why_census": "the CSR of this graph (int64 index + int64 weight per edge) exceeds the 180 GB of "
                                       "one B200; the reference would exhaust host memory on it as well",
                         "roofline_sweep": ({"bound": "int-alu", "achieved": 7.0 * words * evaluated / (main_ms * 1e-3) / 1e12,
                                             "peak": int_peak / 1e12, "unit": "Tlane-op/s",
                                             "frac": 7.0 * words * evaluated / (main_ms * 1e-3) / int_peak,
                                             "kernel_ms": main_ms, "pairs_evaluated_per_launch": evaluated}
                                            if main_ms else None)})
        # ---- parity (outside the timed region) ----
        if not args.no_parity:
            ok, ident = True, True
            how = []
            if known_degree is not None:
                ok &= bool(torch.all(deg == known_degree).item()) and nnz == known_degree * n
                how.append(f"known answer: every degree == {known_degree}")
            if mode == "csr":
                # degrees of this rank's row block against the one-sided count sweep (every row at N=1)
                tab = eng.pack(dev)
                cnt = eng.hamming_eps_degrees(tab, row0, rows, tab, lut)
                ok &= bool(torch.equal(cnt, deg[row0:row0 + rows]))
                how.append("degrees of every row vs the one-sided count sweep")
                ident = same_on_all_ranks([indptr, idx, w], rank, world)
                del tab, cnt
            else:
                ident = same_on_all_ranks([deg], rank, world)
            n_rows = 0
            if rank == 0:
                from oracle import c_oracle as CO
                srows = sample_rows(n, world, eng, words_swept, 0, count=oracle_rows, seed=11)
                D = CO.hamming_rows(CO.pack(tokens), L, srows, threads=cores)
                keep = (D <= eps) & (D > 0)                          # prograph.py:736
                if mode == "csr":
                    ip = indptr.cpu().numpy()
                    for i, r in enumerate(srows):
                        cols = np.nonzero(keep[i])[0]
                        a, b = ip[r], ip[r + 1]
                        ok &= bool(b - a == len(cols) and np.array_equal(idx[a:b].cpu().numpy(), cols)
                                   and np.array_equal(w[a:b].cpu().numpy(), D[i, cols]))
                else:
                    ok &= bool(np.array_equal(deg[torch.from_numpy(srows).to(deg.device)].cpu().numpy(), keep.sum(1)))
                n_rows = len(srows)
                how.append(f"{n_rows} sampled rows (index lists and weights) vs oracle/hamming_knn_cpu.c distances")
            ok = all_true(ok, world, eng.device)
            case["parity"] = {"ok": bool(ok and ident), "rows_vs_oracle": n_rows, "ranks_identical": ident,
                              "how": "; ".join(how)}
        res.clear()
        # ---- end to end: public API, host tokens in, host CSR out (every rank its own rows) ----
        if mode == "csr" and not args.no_e2e:
            out_mode = "sharded" if world > 1 else "replicated"
            build_neighbours(host, eps=eps, output=out_mode)
            e_ms = timed(lambda: build_neighbours(host, eps=eps, output=out_mode), 1)
            case["e2e"] = {"ms_per_build": e_ms, "gpairs_per_s": float(n) * n / (e_ms * 1e-3) / 1e9,
                           "h2d_bytes": int(host.numel()), "d2h_bytes": int(nnz * 16 + (n + world) * 8),
                           "api": f"prograph_b200.build_neighbours(pinned uint8 tokens, eps={eps}, output='{out_mode}')"}
        del dev, host
        torch.cuda.empty_cache()
        cases.append(case)

    M = make_tokens(args.n, args.length, "mutational")
    run_case("C4-M eps=1", M, 1, "csr")
    run_case("C4-M eps=2", M, 2, "census")
    del M
    G = make_gb1_library()
    run_case("C3 GB1 20^4 eps=1", G, 1, "csr", known_degree=76)
    run_case("C3 GB1 20^4 eps=2", G, 2, "csr", known_degree=2242)
    if world > 1:
        dist.barrier()
    return {"metric": "threshold (epsilon) Hamming graphs, N^2 ordered pairs counted per build", "unit": "Gpairs/s",
            "steps": steps, "int_peak_tlops": int_peak / 1e12, "hbm_peak_gbs": hbm_peak, "cases": cases}


# ----------------------------------------------------------------------------------------
# distance-to-dataset queries: 100k queries x 1M library, every metric of prograph/distance (C5)
# ----------------------------------------------------------------------------------------
def run_query_block(args, eng, rank, world, timed, cores):
    import functools
    import operator
    import torch
    from prograph_b200 import minkowski, query
    n, L = args.n, args.length
    m = max(1024, n // 10)
    X = make_tokens(n, L, "mutational")
    Qh = make_tokens(m, L, "mutational", seed=1)
    Q = torch.from_numpy(Qh).to(eng.device)          # queries resident in HBM, like the library
    lib = query.Library(X)
    lib.packed()
    lib.gemm(255)
    torch.cuda.synchronize()
    out = {}
    cases = []

    def run(name, fn, pairs, reps=3):
        fn()
        each = [timed(fn, 1) for _ in range(reps)]          # every repetition on its own: shows the spread
        ms = sorted(each)[len(each) // 2]                   # median: one slow first repetition does not decide
        cases.append({"name": name, "ms": ms, "gpairs_per_s": pairs / (ms * 1e-3) / 1e9, "ms_each": each,
                      "ms_is": "median of ms_each"})

    def hn():
        out["hn"] = query.nearest(lib, Q)

    def hc():
        out["hc"] = query.count_within(lib, Q, 3)

    def mn():
        out["mn"] = query.nearest(lib, Q, distance=minkowski)

    run(f"hamming argmin/min, {m} queries x {n}", hn, float(m) * n)
    run(f"hamming count(d <= 3), {m} queries x {n}", hc, float(m) * n)
    run(f"minkowski p=2 argmin/min (integer tokens -> float32), {m} queries x {n}", mn, float(m) * n)
    run(f"hamming (1024, {n}) int64 tile", lambda: query.tile(lib, Q, 0, 1024), 1024.0 * n)
    run(f"hamming similarity (1024, {n}) float32 tile", lambda: query.tile(lib, Q, 0, 1024, similarity=True), 1024.0 * n)
    run(f"minkowski p=2 (1024, {n}) float32 tile", lambda: query.tile(lib, Q, 0, 1024, distance=minkowski), 1024.0 * n)
    run(f"minkowski p=2 similarity (1024, {n}) float32 tile",
        lambda: query.tile(lib, Q, 0, 1024, distance=minkowski, similarity=True), 1024.0 * n)
    sub = min(1000, m)
    for p in (1, 3):
        how = "rank-1 tile: sum(x) - sum(y), no abs in the reference" if p == 1 else "element-wise kernel, no-abs quirk"
        run(f"minkowski p={p} ({sub}, {n}) float32 tile ({how})",
            lambda p=p: query.tile(lib, Q, 0, sub, distance=functools.partial(minkowski, p=p)), float(sub) * n, reps=1)
    block = {"workload": f"C5: {m} queries (mutational, default_rng(1)) x {n}-row mutational library, L={L}; query rows "
                         f"sharded over {world} GPU(s), library layouts resident", "cases": cases}
    if not args.no_parity:
        ok = True
        if rank == 0:
            from oracle import c_oracle as CO
            sample = np.sort(np.random.default_rng(2).choice(m, size=16, replace=False))
            D = CO.hamming_rows(CO.pack(np.concatenate([X, Qh[sample]])), L, n + np.arange(len(sample)), threads=cores)[:, :n]
            D = D.astype(np.int64)
            sel = torch.from_numpy(sample).to(eng.device)
            ok &= bool(np.array_equal(out["hn"][0][sel].cpu().numpy(), D.argmin(axis=1))
                       and np.array_equal(out["hn"][1][sel].cpu().numpy(), D.min(axis=1))
                       and np.array_equal(out["hc"][sel].cpu().numpy(), (D <= 3).sum(axis=1)))
            few = sample[:4]
            S2 = np.stack([((X.astype(np.int32) - Qh[q].astype(np.int32)) ** 2).sum(axis=1, dtype=np.int64) for q in few])
            fsel = torch.from_numpy(few).to(eng.device)
            ok &= bool(np.array_equal(out["mn"][0][fsel].cpu().numpy(), S2.argmin(axis=1))
                       and np.array_equal(out["mn"][1][fsel].cpu().numpy(),
                                          np.sqrt(S2.min(axis=1).astype(np.float32)).astype(np.float32)))
        block["parity_ok"] = all_true(ok, world, eng.device)
        block["parity_how"] = "16 sampled queries: argmin / min / count against oracle/hamming_knn_cpu.c distance rows; 4 sampled " \
                              "queries: Minkowski argmin / float32 root against exact integer sums (numpy)"
    out.clear()
    return block


def main():
    args = parse_args()
    # stdout must carry exactly one JSON line: park the real stdout, let everything libraries
    # write to fd 1 (NCCL prints its version banner there) go to stderr, and hand the JSON line
    # to the parked descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global emit
    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
