"""Graph construction on the device: threshold (epsilon) and k-nearest-neighbour adjacency.

Host-side mirror of ``Prograph.build_graph`` (prograph/prograph.py:656-765) and of the
row batching / per-row list assembly around it (get_every_n :617-624, prod_neighbours
:626-654, merge/fill :743-753).  The reference loops over batches of 8 query rows,
materialises an (8, N, L) temporary per batch, sorts or scans it and copies every batch
back to the host; here one fused sweep per build produces CSR arrays on the device and the
per-row tuples the reference returns are O(N) views into them.

Dispatch (SURVEY.md §8b):
  * ``distance is prograph_b200.distance.hamming`` and the representation is integer tokens
    -> fused bit-plane sweeps (pg_hamming_knn / pg_hamming_eps_*), the N x N matrix never
    exists;
  * ``minkowski`` (or hamming on non-token values) -> element-wise tile kernels per row
    block + the tile consumers (pg_tile_topk / pg_tile_threshold_*);
  * any other callable honouring the ``fn(X, Y, similarity=...) -> (M, N)`` protocol is
    called per row block exactly as the reference calls it and its device tile goes
    through the same consumers.
The work is sharded across the ranks of an initialised torch.distributed group (shard.py);
by default every rank ends up with the whole graph, ``output="sharded"`` leaves every rank with
the rows of its own block (``row0`` of the returned table) and skips the final all-gather.
Phases are wrapped in NVTX ranges (trace.py).  Off the kernel path torch is used for plumbing
only: allocation, copies, collectives, concatenation of shards and the prefix sum / gather of
the user-callable tile path.
"""
import functools
import operator
import os

import numpy as np
import torch

from . import _lib as L
from . import shard as _shard
from .distance.hamming import hamming, value_dtype
from .distance.minkowski import minkowski, staged_dtype
from .engine import get_engine, sweep_covers
from .trace import phase

_CMP_CODES = {operator.lt: L.LT, operator.le: L.LE, operator.eq: L.EQ,
              operator.ne: L.NE, operator.ge: L.GE, operator.gt: L.GT}

TILE_BUDGET_BYTES = 512 << 20   # materialised tile slab for the non-fused metrics


# ---------------------------------------------------------------------------------
# results
# ---------------------------------------------------------------------------------
class NeighbourTable:
    """Adjacency in CSR form on the host: row r owns idx[indptr[r]:indptr[r+1]] (int64,
    ascending for epsilon graphs, (distance, index) order for kNN) and the matching w."""

    def __init__(self, indptr, idx, w, row0=0):
        self.indptr, self.idx, self.w = indptr, idx, w
        self.row0 = row0            # first row of this table in the whole graph (output="sharded")

    @property
    def n_rows(self):
        return len(self.indptr) - 1

    def degrees(self):
        return np.diff(self.indptr)

    def as_list(self):
        """The reference's return value: a list of (indices, weights) tuples, one per row
        (prograph.py:753,764).  Rows without neighbours carry two empty *int* arrays even for
        float metrics (prograph.py:753)."""
        ip, idx, w = self.indptr, self.idx, self.w
        empty = (np.array([], dtype=int), np.array([], dtype=int))
        out = [None] * self.n_rows
        for r in range(self.n_rows):
            a, b = ip[r], ip[r + 1]
            out[r] = (idx[a:b], w[a:b]) if b > a else empty
        return out


class KnnTable:
    """Fixed-degree kNN result: idx (N, k) int64 and w (N, k)."""

    def __init__(self, idx, w, row0=0):
        self.idx, self.w = idx, w
        self.row0 = row0            # first row of this table in the whole graph (output="sharded")

    @property
    def n_rows(self):
        return self.idx.shape[0]

    def as_list(self):
        return list(zip(self.idx, self.w))      # row views, prograph.py:764

    def to_csr(self):
        n, k = self.idx.shape
        return NeighbourTable(np.arange(0, (n + 1) * k, k, dtype=np.int64), self.idx.reshape(-1), self.w.reshape(-1))


def row_sums_f32(indptr, w):
    """float32 sum of every CSR row's weights, bit for bit what the reference's per-row
    ``np.sum(weights.astype(np.float32))`` returns (prograph.py:819-821) without a Python loop over
    the rows: rows of equal length are summed as one 2-D array, whose contiguous-axis reduction is
    numpy's same pairwise routine."""
    indptr = np.asarray(indptr)
    w32 = np.asarray(w).astype(np.float32)
    deg = np.diff(indptr)
    out = np.zeros(len(deg), dtype=np.float32)
    for d in np.unique(deg):
        if d == 0:
            continue
        rows = np.nonzero(deg == d)[0]
        out[rows] = w32[indptr[rows][:, None] + np.arange(d)].sum(axis=1, dtype=np.float32)
    return out


# ---------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------
def as_matrix(rep):
    """A representation column (pandas Series of row arrays, list of rows, 2-D array or
    tensor) as one 2-D array."""
    if isinstance(rep, torch.Tensor):
        return rep
    if hasattr(rep, "to_numpy") and not isinstance(rep, np.ndarray):
        rep = rep.to_numpy()
    if isinstance(rep, np.ndarray) and rep.dtype != object:
        out = rep
    else:
        out = np.stack([np.asarray(r) for r in rep])
    if out.ndim == 1:
        out = out.reshape(-1, 1)
    return out


def validate(eps, k):
    """Argument checks of prograph.py:714-718 (truthiness: eps=0 and k=0 are rejected)."""
    if operator.xor(bool(eps), bool(k)) is False:
        raise ValueError("Epsilon or K must be provided, but both cannot be as they are different "
                         "methods of graph construction.")
    if k is not None and not isinstance(k, int):
        raise TypeError("K must be provided as an integer.")


def distance_lut(max_d, comp, eps, similarity, guard=True):
    """Truth table over d = 0..max_d of the reference's edge test, evaluated with the same
    torch expressions the reference applies to the distance tensor:
        comp(d, eps) & (d > 0)                         prograph.py:736
        comp(eps, s) & (s < 1),  s = 1/(1+d)           prograph.py:734 (similarity)
    ``guard=False`` drops the second factor (calc_neighbours, prograph.py:544).  Returned as
    uint32 words, bit d of the table = edge."""
    d = torch.arange(max_d + 1, dtype=torch.int64)
    if similarity:
        s = 1 / (1 + d)
        keep = comp(eps, s)
        if guard:
            keep = keep & (s < 1)
    else:
        keep = comp(d, eps)
        if guard:
            keep = keep & (d > 0)
    keep = torch.as_tensor(keep)
    if keep.shape != d.shape:
        raise TypeError("comp must be an element-wise comparison such as operator.le")
    bits = keep.to(torch.bool).numpy()
    words = np.zeros((max_d + 1 + 31) // 32, dtype=np.uint32)
    for i in np.nonzero(bits)[0]:
        words[i >> 5] |= np.uint32(1) << np.uint32(i & 31)
    return words


def _metric_kind(distance):
    """('hamming'|'minkowski'|'callable', p)"""
    fn, p = distance, 2
    if isinstance(distance, functools.partial):
        fn = distance.func
        p = distance.keywords.get("p", distance.args[0] if distance.args else 2)
        if len(distance.args) > 1 or set(distance.keywords) - {"p"}:
            return "callable", None
    if fn is hamming:
        return "hamming", None
    if fn is minkowski:
        return "minkowski", p
    return "callable", None


def _to_host(t):
    """Device tensor -> numpy.  Large results go through pinned memory from torch's caching host
    allocator (a pageable copy of the 256 MB of a 1 M x 16 kNN graph costs several times the
    PCIe time); the numpy array keeps the pinned block alive and hands it back when it dies."""
    if not isinstance(t, torch.Tensor):
        return np.asarray(t)
    if not t.is_cuda:
        return t.numpy()
    if t.numel() * t.element_size() < (1 << 20):
        return t.cpu().numpy()
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return host.numpy()


# ---------------------------------------------------------------------------------
# fused Hamming path
# ---------------------------------------------------------------------------------
def pack_table(eng, X, rank, world, group):
    """Bit-plane table of the whole representation on this rank's GPU.

    Single rank: one pack of the whole matrix.  Several ranks with tile-aligned row blocks:
    every rank uploads and packs only its own rows and the packed shards are all-gathered
    (NCCL over NVLink) straight into one table -- 160 B per sequence instead of each rank
    pushing the whole token matrix through its PCIe link."""
    n = X.shape[0]
    if world <= 1 or n < world or not _shard.is_tile_aligned(n, world) or not eng.sharded_pack:
        return eng.pack(X)
    row0, rows = _shard.row_range(n, rank, world)
    per = _shard.rows_per_rank(n, world)
    mine = eng.to_device(X[row0:row0 + rows])
    # the ranks must agree on the plane count: take it from the global token range
    lim = torch.stack([mine.max().to(torch.float64), -(mine.min().to(torch.float64))])
    torch.distributed.all_reduce(lim, op=torch.distributed.ReduceOp.MAX, group=group)
    hi, lo = float(lim[0]), -float(lim[1])
    if lo < 0 or hi >= 256:
        raise OverflowError("values are not integer tokens in [0, 256)")
    planes = 5 if hi < 32 else 8
    # a shard may be unpackable on its own (fractional values on one rank only): the decision to
    # leave the bit-plane path is taken by all ranks together, before the all-gather below
    part, code = None, _shard.OK
    try:
        part = eng.pack(mine, planes=planes)
    except OverflowError:
        code = _shard.UNPACKABLE
    if _shard.agree(code, world, group, mine.device) != _shard.OK:
        raise OverflowError("values are not integer tokens in [0, 256) on some rank")
    words = part.words
    shard_buf = torch.zeros((per, planes, words), dtype=torch.int32, device=part.data.device)
    shard_buf[: min(per, part.data.shape[0])] = part.data[:per]
    full = torch.empty((world * per, planes, words), dtype=torch.int32, device=part.data.device)
    torch.distributed.all_gather_into_tensor(full, shard_buf, group=group)
    from .engine import PackedTable
    return PackedTable(full, n, part.L, planes, words)



COMPACT_MIN_ROWS = 4096     # smaller tables: the look at the columns costs more than it can save


def informative_table(eng, packed):
    """The table a graph build sweeps: `packed` itself, or its restriction to the residue positions
    that are not constant over the rows when that is a narrower kernel instantiation.  A position
    where every row carries the same token adds 0 to every pairwise Hamming distance
    (hamming.py:34), so distances, neighbours and edges are bit for bit the same; libraries built
    around one wild type (a 4-site combinatorial library of 56-residue sequences) are exactly the
    tables prograph is used on.  Every rank holds the whole table and takes the same decision."""
    done = packed.informative     # None: not looked at yet; False: nothing to drop
    if done is not None:
        return packed if done is False else done
    out = False
    if packed.rows >= COMPACT_MIN_ROWS:
        cols = eng.varying_columns(packed)
        if eng.packed_words(max(1, len(cols))) < packed.words:
            out = eng.compact_columns(packed, cols)
            out.informative = False
    packed.informative = out        # looked at once per table (the Prograph mirror keeps its table)
    return packed if out is False else out


def hamming_knn_device(eng, own, stream, k, similarity, row0, rows):
    """kNN rows [row0,row0+rows) of `own` against `stream` (both PackedTable)."""
    kk = min(k, stream.rows - 1)          # [:, 1:k+1] of a row of N entries
    if kk <= 0:
        wdt = torch.float32 if similarity else torch.int64
        return eng.empty((rows, 0), torch.int64), eng.empty((rows, 0), wdt)
    try:
        return eng.hamming_knn(own, row0, rows, stream, kk, drop=1, similarity=similarity)
    except L.Unsupported:
        return hamming_knn_tiles(eng, own, stream, k, similarity, row0, rows)


# ---------------------------------------------------------------------------------
# symmetric kNN build: every unordered pair once (pg_sweep_sym.cuh)
# ---------------------------------------------------------------------------------
SYM_MIN_ROWS = 65536      # below this the one-sided sweep is as fast (bootstrap + merge overheads)
SYM_BOOT_ROWS = 8192      # bootstrap columns: tight filters from the first tile on
SYM_BOOT_DIV = 8          # ... but at most 1/8 of the table


def _sym_enabled(eng, packed, k1, world):
    force = os.environ.get("PG_KNN_SYM")
    if force is not None:
        return force not in ("0", "")
    return SYM_MIN_ROWS <= packed.rows < (1 << 31) and k1 <= eng.SYM_MAX_LIST


def sym_boot_rows(n):
    """Bootstrap columns for a table of n rows: a multiple of the 512-row packed tile
    (PG_SYM_BOOT overrides the default of 8192 for experiments)."""
    want = int(os.environ.get("PG_SYM_BOOT", SYM_BOOT_ROWS))
    return max(0, min(want, n // SYM_BOOT_DIV) // _shard.ROW_ALIGN * _shard.ROW_ALIGN)


def hamming_knn_graph(eng, packed, k, similarity, rank, world, group, output="replicated"):
    """kNN lists of EVERY row of `packed` against itself (prograph.py:755-765): (idx, w, row0).
    ``output="replicated"``: all rows on every rank (row0 = 0); ``"sharded"``: this rank's row block.

    Large tables take the symmetric sweep: d(i,j) == d(j,i), so each unordered pair is evaluated
    once and offered to both rows' lists.  Ranks own bands of stream rows of the triangle (equal
    numbers of pair evaluations); the exchange step of this path is an all-to-all of the per-rank
    candidate lists (every rank receives all ranks' lists of its own rows and merges them),
    followed by the all-gather of the merged keys.  Small tables and long lists take the one-sided
    sweep on this rank's row block followed by the all-gather of the result rows."""
    n = packed.rows
    kk = min(k, n - 1)
    with phase("columns"):
        packed = informative_table(eng, packed)
    if kk > 0 and _sym_enabled(eng, packed, kk + 1, world):
        try:
            return _hamming_knn_sym(eng, packed, kk, similarity, rank, world, group, output)
        except L.Unsupported:
            pass
    row0, rows = _shard.row_range(n, rank, world)
    with phase("sweep"):
        part = hamming_knn_device(eng, packed, packed, k, similarity, row0, rows) if rows else None
    if output == "sharded":
        return part + (row0,)
    with phase("gather"):
        return _shard.gather_rows(part, n, rank, world, group, eng) + (0,)


def _hamming_knn_sym(eng, packed, kk, similarity, rank, world, group, output):
    n, k1 = packed.rows, kk + 1
    sharded = world > 1 and n >= world
    if not sharded:
        rank, world = 0, 1
    boot = sym_boot_rows(n)
    seed = None
    row0, rows = _shard.row_range(n, rank, world)
    if boot:
        with phase("boot"):
            seed = eng.hamming_knn_boot(packed, row0, rows, boot, k1)
        with phase("boot_gather"):
            seed = _shard.gather_rows((seed,), n, rank, world, group, eng)[0].contiguous()
    # several ranks: column bands (mode 1) -- all column-side candidates of a row meet on one rank,
    # so its filter tightens as fast as on a single GPU
    with phase("sweep"):
        lists = eng.hamming_knn_sym(packed, k1, rank, world, lists=seed, boot_rows=boot, mode=1 if sharded else 0)
    if not sharded:
        with phase("finalize"):
            out = eng.knn_lists_finalize(lists, 0, n, kk, 1, similarity)
        eng.sym_check()
        return out + (0,)
    with phase("exchange"):
        mine = _shard.exchange_lists(lists, n, rank, world, group)        # (world, rows, k1): my rows, every rank's view
    with phase("merge"):
        keys = eng.knn_lists_merge(mine, kk, drop=1)                      # (rows, kk) merged keys
    if output == "sharded":
        with phase("finalize"):
            out = eng.knn_lists_finalize(keys, 0, rows, kk, 0, similarity)
        eng.sym_check()
        return out + (row0,)
    with phase("gather"):
        keys = _shard.gather_rows((keys,), n, rank, world, group, eng)[0].contiguous()
    with phase("finalize"):
        out = eng.knn_lists_finalize(keys, 0, n, kk, 0, similarity)
    eng.sym_check()
    return out + (0,)


def hamming_knn_tiles(eng, own, stream, k, similarity, row0, rows, drop=1):
    """Same result through materialised int64 tiles + the tile top-k: used when k is too large
    for the in-shared-memory lists of the fused sweep.  Ascending distance with index ties is
    the same order as descending similarity, so the sort always runs on the distances."""
    kk = min(k, stream.rows - drop)
    step = max(512, (TILE_BUDGET_BYTES // (8 * stream.rows)) // 512 * 512)
    idxs, ws = [], []
    a0 = row0 // 512 * 512
    for q0 in range(a0, row0 + rows, step):
        qn = min(step, own.rows - q0)
        tile = eng.hamming_tile(stream, own, q0, qn, weight=L.W_I64)
        lo, hi = max(row0, q0) - q0, min(row0 + rows, q0 + qn) - q0
        i, d = eng.tile_topk(tile[lo:hi], kk, drop=drop, descending=False)
        idxs.append(i)
        ws.append(1 / (1 + d) if similarity else d)        # hamming.py:38, on the device
    return torch.cat(idxs), torch.cat(ws)


def hamming_eps_device(eng, own, stream, lut, similarity, row0, rows, capture=None):
    return eng.hamming_eps(own, row0, rows, stream, lut, similarity=similarity, capture=capture)


SYM_EPS_MIN_ROWS = 32768    # smaller epsilon graphs: count + capture with the one-sided sweep
SYM_EPS_MAX_DEGREE = 384    # denser graphs are bound by writing their edges: one-sided count / fill


def _eps_sample(n):
    """(first row, rows) of the row sample that estimates the mean degree."""
    rows = min(n, max(512, min(2048, n // 128 // _shard.ROW_ALIGN * _shard.ROW_ALIGN)))
    row0 = (n // 2) // _shard.ROW_ALIGN * _shard.ROW_ALIGN
    return (row0, rows) if row0 + rows <= n else (0, rows)


def _raise_code(code, exc=None):
    """Raise on every rank what some rank ran into (its own exception where it has one)."""
    if exc is not None:
        raise exc
    if code == _shard.NO_MEMORY:
        raise MemoryError("the requested graph does not fit in device memory on some rank; lower eps or build a "
                          "kNN graph")
    if code == _shard.UNPACKABLE:
        raise OverflowError("values are not integer tokens on some rank")


def hamming_eps_graph(eng, packed, lut, similarity, rank, world, group):
    """Epsilon graph (CSR of every row) of `packed` against itself, on every rank
    (prograph.py:731-753).  Large, sparse graphs whose edge test is one contiguous distance range
    take the symmetric sweep: one pass over the triangle of unordered pairs appends both directed
    edges of every passing pair as packed keys, a radix sort by (row, column) turns them into the
    CSR.  A one-sided count over a small row sample estimates the mean degree first: it sizes the
    key buffer and sends dense graphs (bound by writing their edges, not by distances) to the
    count / fill passes.  Ranks sweep bands of the triangle and all-gather their key buffers.
    Everything else: count / fill with the one-sided sweep on this rank's row block, then the CSR
    all-gather.  Rank-local failures (edge budget) are agreed on before every collective."""
    n = packed.rows
    dev = eng.device
    sharded = world > 1 and n >= world
    capture = None
    with phase("columns"):
        packed = informative_table(eng, packed)
    force = os.environ.get("PG_EPS_SYM")
    use_sym = n >= SYM_EPS_MIN_ROWS if force is None else force not in ("0", "")
    if use_sym:
        # the ranks split the sample rows and add their counts up -> the same degree, capacity and
        # branch on all of them
        parts = world if sharded else 1
        with phase("sample"):
            s0, srows = _eps_sample(n)
            if sharded and srows >= 2 * world:
                a, b = s0 + rank * srows // world, s0 + (rank + 1) * srows // world
                deg = eng.hamming_eps_degrees(packed, a, b - a, packed, lut)
                total, top = deg.sum().reshape(1), deg.max().reshape(1)
                torch.distributed.all_reduce(total, group=group)
                torch.distributed.all_reduce(top, op=torch.distributed.ReduceOp.MAX, group=group)
                degree, top_degree = float(total.item()) / srows, int(top.item())
            else:
                degree, top_degree = eng.hamming_eps_mean_degree(packed, s0, srows, packed, lut)
        capacity = int(1.5 * degree * n / parts) + (4 << 20)
        if (degree > SYM_EPS_MAX_DEGREE and force is None) or capacity * parts >= (1 << 31):
            use_sym = False        # dense graph, or more keys than one radix sort takes
            # ... whose count pass keeps every hit (room for 1.25 x the largest sampled degree per row;
            # rows beyond that get the fill sweep), so that the fill pass is one copy, not a second sweep
            capture = int(1.25 * top_degree) + 64
    if use_sym:
        code, keys, edges, exc = _shard.OK, None, 0, None
        try:
            with phase("sweep"):
                keys, edges = eng.hamming_eps_sym(packed, lut, rank if sharded else 0, parts, mode=1 if sharded else 0,
                                                  capacity=capacity)
        except L.Unsupported:
            code = _shard.UNSUPPORTED          # shape / predicate: the same on every rank
        except MemoryError as e:
            code, exc = _shard.NO_MEMORY, e
        code = _shard.agree(code, world, group, dev) if sharded else code
        _raise_code(code, exc)
        if code == _shard.OK:
            if sharded:
                with phase("exchange"):
                    keys, edges = _shard.gather_edge_keys(keys, edges, world, group)
            code = _shard.OK
            try:
                eng.check_edge_budget(edges)
            except MemoryError as e:
                code, exc = _shard.NO_MEMORY, e
            _raise_code(_shard.agree(code, world, group, dev) if sharded else code, exc)
            with phase("csr"):
                return eng.edge_keys_to_csr(keys, n, packed.words, edges, similarity)
    row0, rows = _shard.row_range(n, rank, world)
    code, part, exc = _shard.OK, None, None
    try:
        with phase("sweep"):
            part = hamming_eps_device(eng, packed, packed, lut, similarity, row0, rows, capture) if rows else None
    except MemoryError as e:
        code, exc = _shard.NO_MEMORY, e
    _raise_code(_shard.agree(code, world, group, dev) if sharded else code, exc)
    with phase("gather"):
        return _shard.gather_csr(part, n, rank, world, group, eng)


# ---------------------------------------------------------------------------------
# Minkowski p=2 on integer tokens: the edge test as a range of the exact integer sum S
# ---------------------------------------------------------------------------------
def minkowski_s_range(s_max, comp, eps, similarity):
    """The fp16 rounding chain of minkowski.py:36-40 maps the exact integer
    S = sum (x - y)^2 to d = fp16(sqrt(fp16(S))) (and to 1/(1+d) for similarity), monotonically.
    Evaluate the reference's edge test (prograph.py:734-736) for every S in [0, s_max] and return
    it as an inclusive range (lo, hi), (1, 0) when nothing passes, or None when the passing set is
    not one interval (operator.ne)."""
    S = np.arange(s_max + 1, dtype=np.int64)
    with np.errstate(over="ignore"):
        s16 = S.astype(np.float32).astype(np.float16)
        d = np.sqrt(s16.astype(np.float32)).astype(np.float16)
        if similarity:
            one_plus = (np.float32(1.0) + d.astype(np.float32)).astype(np.float16)
            d = (np.float32(1.0) / one_plus.astype(np.float32)).astype(np.float16)
    t = torch.from_numpy(d)
    keep = (comp(eps, t) & (t < 1)) if similarity else (comp(t, eps) & (t > 0))
    keep = torch.as_tensor(keep).numpy().astype(bool)
    hits = np.nonzero(keep)[0]
    if len(hits) == 0:
        return 1, 0
    lo, hi = int(hits[0]), int(hits[-1])
    if hi - lo + 1 != len(hits):
        return None
    return lo, hi


# ---------------------------------------------------------------------------------
# tile path (minkowski, hamming on values, user callables)
# ---------------------------------------------------------------------------------
def _tile_rows(n_cols, itemsize, batch_size):
    rows = max(1, TILE_BUDGET_BYTES // max(1, n_cols * itemsize))
    return int(max(batch_size, min(rows, 4096)))


def _tiles(eng, X, kind, p, distance, similarity, batch_size, row0, rows, gemm=None):
    """Yield (b0, tile) with tile = distance(X, X[b0:b1]) on the device, (b1-b0, N)."""
    n = X.shape[0]
    if kind == "callable":
        step = batch_size                  # the reference's own batching, prograph.py:731
    else:
        step = _tile_rows(n, 8, batch_size)
    for b0 in range(row0, row0 + rows, step):
        b1 = min(b0 + step, row0 + rows)
        if gemm is not None:
            q = eng.gemm_pack(X[b0:b1], max_token=gemm.max_token, K=gemm.K)
            tile = eng.minkowski2_gemm_tile(gemm, q, 0, similarity=similarity)
        elif kind == "minkowski":
            tile = eng.minkowski_tile(X, X, b0, b1 - b0, p=p, similarity=similarity)
        elif kind == "hamming":
            tile = eng.hamming_values_tile(X, X, b0, b1 - b0, similarity=similarity)
        else:
            tile = torch.as_tensor(distance(X, X[b0:b1], similarity=similarity))
            if not tile.is_cuda:
                tile = tile.to(eng.device)
            tile = tile.contiguous()
            if tile.dtype == torch.bfloat16:
                tile = tile.to(torch.float32)
        yield b0, tile


def _tile_knn(eng, tiles, k, similarity, n):
    kk = min(k, n - 1)
    idxs, ws = [], []
    for _, tile in tiles:
        if kk <= 0:
            idxs.append(eng.empty((tile.shape[0], 0), torch.int64))
            ws.append(eng.empty((tile.shape[0], 0), tile.dtype))
            continue
        i, w = eng.tile_topk(tile, kk, drop=1, descending=similarity)
        idxs.append(i)
        ws.append(w)
    return torch.cat(idxs), torch.cat(ws)


def _tile_eps(eng, tiles, eps, comp, similarity):
    code = _CMP_CODES.get(comp)
    counts, idxs, ws = [], [], []
    for _, tile in tiles:
        if code is not None:
            ip, i, w = eng.tile_threshold(tile, code, eps, swap=similarity, guard=2 if similarity else 1)
        else:
            # arbitrary comparison callables are evaluated on the device tile by torch exactly as
            # the reference does (prograph.py:734-736); the compaction is ours
            mask = (comp(eps, tile) & (tile < 1)) if similarity else (comp(tile, eps) & (tile > 0))
            ip, i, _ = eng.tile_threshold(mask.to(torch.uint8).contiguous(), L.NE, 0.0, values=False)
            rows_of = torch.repeat_interleave(torch.arange(tile.shape[0], device=tile.device), ip[1:] - ip[:-1])
            w = tile[rows_of, i]
        counts.append(ip[1:] - ip[:-1])
        idxs.append(i)
        ws.append(w)
    counts = torch.cat(counts)
    indptr = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=counts.device)
    torch.cumsum(counts, 0, out=indptr[1:])
    return indptr, torch.cat(idxs), torch.cat(ws)


# ---------------------------------------------------------------------------------
# public entry
# ---------------------------------------------------------------------------------
def _shard_csr(csr, n, rank, world):
    """Rows of this rank's block out of a whole-graph CSR on the device: (indptr, idx, w, row0)."""
    indptr, idx, w = csr
    row0, rows = _shard.row_range(n, rank, world)
    a, b = (int(v) for v in indptr[[row0, row0 + rows]].tolist())
    return indptr[row0:row0 + rows + 1] - a, idx[a:b], w[a:b], row0


def build_neighbours(rep, eps=None, k=None, similarity=False, distance=hamming, comp=operator.le,
                     batch_size=8, idxs=None, engine=None, group=None, packed=None, output="replicated"):
    """Device implementation of ``Prograph.build_graph`` (prograph.py:656-765) on a
    representation matrix.  Returns a NeighbourTable (epsilon) or KnnTable (k) of host arrays.

    output : "replicated" (default) -- the whole graph on every rank of the process group, what a
        drop-in ``build_graph`` returns; "sharded" -- every rank keeps and copies to the host only
        the rows of its own block (``table.row0``, ``shard.row_range``): the graph then exists once
        across the job's host memory and the final all-gather is skipped."""
    validate(eps, k)
    if output not in ("replicated", "sharded"):
        raise ValueError("output must be 'replicated' or 'sharded'")
    if similarity and eps:
        eps = 1 / (1 + eps)                                   # prograph.py:720-721
    eng = engine if engine is not None else get_engine()
    X = as_matrix(rep)
    if idxs is not None:
        X = X[idxs, :] if not isinstance(idxs, type(Ellipsis)) else X   # indices relative to the subset
    if X.shape[0] == 0:
        raise ValueError("empty representation")
    n = X.shape[0]
    kind, p = _metric_kind(distance)
    rank, world = _shard.rank_world(group)
    row0, rows = _shard.row_range(n, rank, world)

    if packed is not None and (kind != "hamming" or idxs is not None or packed.rows != n):
        packed = None
    if kind == "hamming" and packed is None:
        try:
            with phase("pack"):
                packed = pack_table(eng, X, rank, world, group)
        except OverflowError:
            packed = None
    if packed is not None:
        with phase("columns"):
            packed = informative_table(eng, packed)     # may bring a wide table back into range
    if packed is not None and not sweep_covers(packed.planes, packed.words):
        packed = None          # wider than the fused sweeps: element-wise tiles below

    if packed is not None:
        if eps:
            lut = distance_lut(packed.words * 32, comp, eps, similarity)
            csr = hamming_eps_graph(eng, packed, lut, similarity, rank, world, group)
            shard0 = 0
            if output == "sharded":
                *csr, shard0 = _shard_csr(csr, n, rank, world)
            with phase("d2h"):
                return NeighbourTable(*(_to_host(t) for t in csr), row0=shard0)
        else:
            idx, w, shard0 = hamming_knn_graph(eng, packed, k, similarity, rank, world, group, output)
            with phase("d2h"):
                return KnnTable(_to_host(idx), _to_host(w), row0=shard0)
    else:
        # prograph.py:726: every representation is rounded to fp16 before the metric sees it
        Xh = eng.to_device(X).to(torch.float16)
        gemm = None
        if kind == "minkowski" and float(p) == 2.0 and Xh.shape[1] <= eng.GEMM_MAX_WIDTH:
            # integer tokens <= 31: the fp16 chain is a function of the exact integer
            # |x|^2 + |y|^2 - 2 x.y  ->  int8 tensor-core contraction (pg_gemm.cu)
            try:
                gemm = eng.gemm_pack(Xh, max_token=31)
            except (OverflowError, L.Unsupported):
                gemm = None
        part = None
        if gemm is not None and not eps and rows:
            kk = min(k, n - 1)
            if kk > 0:
                try:
                    q = gemm if (row0 == 0 and rows == n) else eng.gemm_pack(Xh[row0:row0 + rows], max_token=31, K=gemm.K)
                    part = eng.minkowski2_gemm_knn(gemm, q, kk, 1, 0, similarity=similarity)
                except L.Unsupported:
                    part = None
        if gemm is not None and eps and rows and comp in _CMP_CODES:
            rng = minkowski_s_range(gemm.K * gemm.max_token * gemm.max_token, comp, eps, similarity)
            if rng is not None:
                lo, hi = rng
                if lo > hi:
                    part = (torch.zeros(rows + 1, dtype=torch.int64, device=eng.device),
                            eng.empty((0,), torch.int64), eng.empty((0,), torch.float16))
                else:
                    q = gemm if (row0 == 0 and rows == n) else eng.gemm_pack(Xh[row0:row0 + rows], max_token=31, K=gemm.K)
                    part = eng.minkowski2_gemm_eps(gemm, q, lo, hi, 0, similarity=similarity)
        if part is None:
            tiles = _tiles(eng, Xh, kind, p, distance, similarity, batch_size, row0, rows, gemm=gemm)
            if eps:
                part = _tile_eps(eng, tiles, eps, comp, similarity) if rows else None
            else:
                part = _tile_knn(eng, tiles, k, similarity, n) if rows else None

    sharded_out = output == "sharded"
    if eps:
        indptr, idx, w = part if sharded_out else _shard.gather_csr(part, n, rank, world, group, eng)
        return NeighbourTable(_to_host(indptr), _to_host(idx), _to_host(w), row0=row0 if sharded_out else 0)
    idx, w = part if sharded_out else _shard.gather_rows(part, n, rank, world, group, eng)
    return KnnTable(_to_host(idx), _to_host(w), row0=row0 if sharded_out else 0)


# ---------------------------------------------------------------------------------
# growing a built graph by new rows
# ---------------------------------------------------------------------------------
def stack_rows(A, B):
    """`A` over `B`, the narrower side right-padded with token 0 (the clean_input rule,
    distance/utils.py): a position padded in both rows of a pair adds nothing to their distance."""
    width = max(A.shape[1], B.shape[1])
    if isinstance(A, torch.Tensor) or isinstance(B, torch.Tensor):
        dev = A.device if isinstance(A, torch.Tensor) else B.device
        A, B = (torch.as_tensor(t).to(dev) for t in (A, B))
        return torch.cat([torch.nn.functional.pad(t, (0, width - t.shape[1])) for t in (A, B)])
    return np.concatenate([np.pad(t, ((0, 0), (0, width - t.shape[1]))) for t in (A, B)])


def _check_previous(table, n_old, eps, k):
    if eps and not isinstance(table, NeighbourTable):
        raise ValueError("an epsilon graph is extended from the NeighbourTable its build returned")
    if not eps and not isinstance(table, KnnTable):
        raise ValueError("a kNN graph is extended from the KnnTable its build returned")
    if table.row0 != 0 or table.n_rows != n_old:
        raise ValueError(f"table must hold the whole graph of rep ({n_old} rows from row 0), not rows "
                         f"[{table.row0}, {table.row0 + table.n_rows}): gather a sharded build first")
    if not eps and table.idx.shape[1] != min(k, n_old - 1):
        raise ValueError(f"table has {table.idx.shape[1]} neighbours per row, a build of {n_old} rows with "
                         f"k={k} has {min(k, n_old - 1)}")


def _upload(eng, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(eng.device)


def _extend_knn_rows(eng, table, packed, fresh, kk, similarity, a, b, col_base):
    """kNN lists of old rows [a, b) in the grown graph: the stored lists merged with the rows'
    candidates among the new rows.  Position 0 of an old row is itself or a lower-indexed duplicate,
    never a new row (indices >= col_base), so the stored positions 1..k and the new candidates hold
    the grown row's positions 1..kk."""
    kc = min(kk, fresh.rows)
    try:
        ci, cw = eng.hamming_knn(packed, a, b - a, fresh, kc, drop=0, similarity=similarity)
    except L.Unsupported:
        ci, cw = hamming_knn_tiles(eng, packed, fresh, kc, similarity, a, b - a, drop=0)
    with phase("upload"):
        pi, pw = _upload(eng, table.idx[a:b]), _upload(eng, table.w[a:b])
    with phase("merge"):
        return eng.knn_extend_merge(pi, pw, ci, cw, col_base, kk, similarity)


def _extend_eps_rows(eng, table, packed, fresh, lut, similarity, a, b, col_base):
    """Epsilon rows [a, b) in the grown graph: the stored rows followed by their edges to the new
    rows, which all have larger indices."""
    add = hamming_eps_device(eng, packed, fresh, lut, similarity, a, b - a)
    with phase("upload"):
        ip = table.indptr[a:b + 1]
        lo, hi = int(ip[0]), int(ip[-1])
        old = (_upload(eng, ip), _upload(eng, table.idx[lo:hi]), _upload(eng, table.w[lo:hi]))
    with phase("merge"):
        return eng.csr_append(old, add, col_base, similarity)


def _cat_csr(parts):
    if len(parts) == 1:
        return parts[0]
    (ip0, i0, w0), (ip1, i1, w1) = parts
    return torch.cat([ip0, ip1[1:] - ip1[0] + ip0[-1]]), torch.cat([i0, i1]), torch.cat([w0, w1])


def extend_neighbours(table, rep, new, eps=None, k=None, similarity=False, distance=hamming, comp=operator.le,
                      engine=None, group=None, output="replicated"):
    """The graph of `rep` stacked over `new` from `table`, the graph ``build_neighbours(rep, eps|k,
    similarity, distance, comp)`` returned (whole: row0 0, one row per row of rep), without sweeping
    the old x old pairs again.  The result is bit for bit ``build_neighbours(concat, ...)`` with
    the same arguments and `output`, where `concat` is rep over new with the narrower side
    right-padded with token 0 (as clean_input pads): CSR arrays or kNN lists, dtypes and tie order.

    Hamming on integer tokens within the fused sweeps: each old row is swept against the new rows
    only and joined with its stored row (pg_knn_extend_merge / pg_csr_append); the new rows are
    swept against the whole grown table, 2NM + M^2 pair evaluations instead of (N+M)^2.  The ranks
    of a process group split the grown rows as a build does.  Every other metric or value type is
    a rebuild of the concatenation."""
    validate(eps, k)
    if output not in ("replicated", "sharded"):
        raise ValueError("output must be 'replicated' or 'sharded'")
    A, B = as_matrix(rep), as_matrix(new)
    n_old, m = A.shape[0], B.shape[0]
    if m == 0:
        raise ValueError("no new rows to add")
    if n_old == 0:
        raise ValueError("empty representation")
    _check_previous(table, n_old, eps, k)
    X = stack_rows(A, B)
    n = n_old + m
    eng = engine if engine is not None else get_engine()
    rank, world = _shard.rank_world(group)
    packed = None
    if _metric_kind(distance)[0] == "hamming":
        try:
            with phase("pack"):
                packed = pack_table(eng, X, rank, world, group)
        except OverflowError:
            packed = None
    if packed is not None:
        with phase("columns"):
            # over the grown table: a position constant over the old rows may vary over the new ones
            packed = informative_table(eng, packed)
    if packed is None or not sweep_covers(packed.planes, packed.words):
        return build_neighbours(X, eps=eps, k=k, similarity=similarity, distance=distance, comp=comp, engine=eng,
                                group=group, output=output)
    wdt = np.dtype(np.float32 if similarity else np.int64)
    if np.asarray(table.w).dtype != wdt:
        raise ValueError(f"table weights are {np.asarray(table.w).dtype}; a build with similarity={similarity} "
                         f"gives {wdt}")
    with phase("columns"):
        fresh = eng.gather_packed(packed, np.arange(n_old, n))      # the new rows, same columns
    row0, rows = _shard.row_range(n, rank, world)
    old_rows = (row0, min(row0 + rows, n_old))                      # this rank's rows of each part
    new_rows = (max(row0, n_old), row0 + rows)
    sharded = world > 1 and n >= world
    if eps:
        lut = distance_lut(packed.words * 32, comp, 1 / (1 + eps) if similarity else eps, similarity)
        code, exc, parts = _shard.OK, None, []
        try:
            with phase("sweep"):
                if old_rows[1] > old_rows[0]:
                    parts.append(_extend_eps_rows(eng, table, packed, fresh, lut, similarity, *old_rows, n_old))
                if new_rows[1] > new_rows[0]:
                    a, b = new_rows
                    parts.append(hamming_eps_device(eng, packed, packed, lut, similarity, a, b - a))
        except MemoryError as e:
            code, exc = _shard.NO_MEMORY, e
        _raise_code(_shard.agree(code, world, group, eng.device) if sharded else code, exc)
        part = _cat_csr(parts)
        if output != "sharded":
            with phase("gather"):
                part = _shard.gather_csr(part, n, rank, world, group, eng)
            row0 = 0
        with phase("d2h"):
            return NeighbourTable(*(_to_host(t) for t in part), row0=row0)
    kk = min(k, n - 1)
    parts = []
    with phase("sweep"):
        if old_rows[1] > old_rows[0]:
            parts.append(_extend_knn_rows(eng, table, packed, fresh, kk, similarity, *old_rows, n_old))
        if new_rows[1] > new_rows[0]:
            a, b = new_rows
            parts.append(hamming_knn_device(eng, packed, packed, k, similarity, a, b - a))
    part = tuple(torch.cat(t) for t in zip(*parts))
    if output != "sharded":
        with phase("gather"):
            part = _shard.gather_rows(part, n, rank, world, group, eng)
        row0 = 0
    with phase("d2h"):
        return KnnTable(_to_host(part[0]), _to_host(part[1]), row0=row0)
