"""Distance-to-dataset queries fused with their consumers (SURVEY.md §8 a8).

The reference answers a query by materialising ``distance(self.tokenized, rows)`` -- an (M, N)
matrix -- and reducing it on the host: ``np.argmin / np.min`` (nearest_neighbour,
prograph.py:567-569), ``np.where(comp(d, eps))`` (calc_neighbours, :544), ``d <= eps``
(neighbourhood, :587).  At the size of BASELINE.json's configs[4] (100 000 queries against a
1 000 000-row library) that matrix would hold 10^11 entries; here every consumer runs inside the
sweep that produces the distances and only its result leaves the kernel:

    nearest(lib, Q)                 argmin / min per query          pg_hamming_knn(k=1, drop=0) /
                                                                    pg_minkowski2_gemm_knn / tile + pg_tile_topk
    count_within(lib, Q, eps, comp) |{n : comp(d(q, n), eps)}|      pg_hamming_eps_count (truth table of comp)
    tile(lib, Q, q0, rows)          the (rows, N) slice itself      pg_hamming_tile / pg_minkowski2_gemm_tile / ...

``Library`` keeps the dataset resident in the layouts the kernels read (bit planes for Hamming,
K-major uint8 core matrices for the tensor-core Minkowski kernel), so a stream of query batches
pays for the conversion once.  Query rows are sharded over the ranks of an initialised
torch.distributed group; every rank ends up with all results.
"""
import operator

import torch

from . import _lib as L
from . import shard as _shard
from .distance.hamming import hamming
from .distance.minkowski import gemm_value_kind, staged_dtype
from .engine import get_engine, sweep_covers
from .graph import TILE_BUDGET_BYTES, _metric_kind, as_matrix, distance_lut
from .trace import phase


class Library:
    """A dataset matrix (N, L) resident on the device for repeated queries."""

    def __init__(self, data, engine=None):
        self.eng = engine if engine is not None else get_engine()
        self.data = as_matrix(data)
        self.n, self.L = int(self.data.shape[0]), int(self.data.shape[1])
        if self.n == 0:
            raise ValueError("empty dataset")                     # distance/utils.py:29-30
        self._packed = None
        self._gemm = {}
        self._dev = {}

    def packed(self):
        """Bit planes of the dataset (raises OverflowError / Unsupported when it is not tokens)."""
        if self._packed is None:
            tab = self.eng.pack(self.data)
            if not sweep_covers(tab.planes, tab.words):
                raise L.Unsupported("rows longer than 32768 residues take the element-wise kernels")
            self._packed = tab
        return self._packed

    def gemm(self, max_token):
        if max_token not in self._gemm:
            self._gemm[max_token] = self.eng.gemm_pack(self.data, max_token=max_token)
        return self._gemm[max_token]

    def device(self, dtype):
        if dtype not in self._dev:
            self._dev[dtype] = self.eng.to_device(self.data, dtype)
        return self._dev[dtype]


def _probe(a):
    """A zero-size CPU tensor with the dtype of `a` (numpy array or tensor on any device): what the
    dtype-promotion helpers of the distance modules need to see."""
    if isinstance(a, torch.Tensor):
        return torch.empty(0, dtype=a.dtype)
    return torch.as_tensor(a[:0])


def _as_library(lib):
    return lib if isinstance(lib, Library) else Library(lib)


def _gather(part, m, rank, world, group, eng):
    return _shard.gather_rows(part, m, rank, world, group, eng)


def nearest(lib, queries, distance=hamming, group=None):
    """Closest dataset row of every query row: ``(idx int64 (M,), value (M,))`` =
    ``(np.argmin(d, axis=1), np.min(d, axis=1))`` of ``d = distance(dataset, queries)`` -- the first
    index on ties, like numpy's argmin (prograph.py:567-569).  Device tensors."""
    lib = _as_library(lib)
    eng = lib.eng
    Q = as_matrix(queries)
    m = int(Q.shape[0])
    if m == 0:
        raise ValueError("empty query set")
    kind, p = _metric_kind(distance)
    rank, world = _shard.rank_world(group)
    r0, rows = _shard.row_range(m, rank, world)
    Qr = Q[r0:r0 + rows]
    part = None
    if kind == "hamming":
        try:
            tab = lib.packed()
            q = eng.pack(Qr, planes=tab.planes, words=tab.words)
            with phase("query_sweep"):
                idx, d = eng.hamming_knn(q, 0, rows, tab, 1, drop=0)
            part = (idx[:, 0].contiguous(), d[:, 0].contiguous())
        except (OverflowError, L.Unsupported):
            part = None
    elif kind == "minkowski" and float(p) == 2.0 and lib.L <= eng.GEMM_MAX_WIDTH:
        vk, max_token = gemm_value_kind(staged_dtype(_probe(lib.data), _probe(Qr), p), lib.L)
        if vk is not None:
            try:
                g = lib.gemm(max_token)
                q = eng.gemm_pack(Qr, max_token=max_token, K=g.K)
                with phase("query_sweep"):
                    idx, v = eng.minkowski2_gemm_knn(g, q, 1, 0, vk)
                part = (idx[:, 0].contiguous(), v[:, 0].contiguous())
            except (OverflowError, L.Unsupported):
                part = None
    if part is None:
        idxs, vals = [], []
        for _, t in _tiles(lib, Qr, distance, kind, p, False):
            i, v = eng.tile_topk(t, 1, drop=0, descending=False)
            idxs.append(i[:, 0])
            vals.append(v[:, 0])
        part = (torch.cat(idxs), torch.cat(vals))
    return _gather(part, m, rank, world, group, eng)


def count_within(lib, queries, eps, comp=operator.le, distance=hamming, group=None):
    """Number of dataset rows n with ``comp(distance(n, q), eps)`` for every query row q: the
    size of what calc_neighbours (prograph.py:544; no ``d > 0`` filter) returns.  (M,) int64."""
    lib = _as_library(lib)
    eng = lib.eng
    Q = as_matrix(queries)
    m = int(Q.shape[0])
    kind, p = _metric_kind(distance)
    rank, world = _shard.rank_world(group)
    r0, rows = _shard.row_range(m, rank, world)
    Qr = Q[r0:r0 + rows]
    part = None
    if kind == "hamming":
        try:
            tab = lib.packed()
            q = eng.pack(Qr, planes=tab.planes, words=tab.words)
            lut = distance_lut(tab.words * 32, comp, eps, similarity=False, guard=False)
            with phase("query_sweep"):
                part = (eng.hamming_eps_degrees(q, 0, rows, tab, lut),)
        except (OverflowError, L.Unsupported):
            part = None
    if part is None:
        counts = []
        for _, t in _tiles(lib, Qr, distance, kind, p, False):
            code = {operator.lt: L.LT, operator.le: L.LE, operator.eq: L.EQ, operator.ne: L.NE, operator.ge: L.GE,
                    operator.gt: L.GT}.get(comp)
            if code is None:
                raise TypeError("comp must be one of operator.{lt,le,eq,ne,ge,gt} for non-Hamming metrics")
            counts.append(eng.tile_threshold_counts(t, code, eps))
        part = (torch.cat(counts),)
    return _gather(part, m, rank, world, group, eng)[0]


def tile(lib, queries, q0=0, rows=None, distance=hamming, similarity=False):
    """The materialised (rows, N) slice ``distance(dataset, queries[q0:q0+rows], similarity)`` on the
    device (hamming.py:34-38 / minkowski.py:36-40 semantics and dtypes)."""
    lib = _as_library(lib)
    Q = as_matrix(queries)
    rows = int(Q.shape[0]) - q0 if rows is None else rows
    kind, p = _metric_kind(distance)
    out = [t for _, t in _tiles(lib, Q[q0:q0 + rows], distance, kind, p, similarity, whole=True)]
    return out[0] if len(out) == 1 else torch.cat(out)


def _tiles(lib, Q, distance, kind, p, similarity, whole=False):
    """Yield (first query row, (rows, N) device tile) over the query rows Q."""
    eng = lib.eng
    m = int(Q.shape[0])
    step = m if whole else max(1, min(4096, TILE_BUDGET_BYTES // max(1, lib.n * 8)))
    for b0 in range(0, m, step):
        Qb = Q[b0:b0 + step]
        if kind == "hamming":
            try:
                tab = lib.packed()
                q = eng.pack(Qb, planes=tab.planes, words=tab.words)
                yield b0, eng.hamming_tile(tab, q, 0, q.rows, weight=L.W_SIM_F32 if similarity else L.W_I64)
                continue
            except (OverflowError, L.Unsupported):
                pass
            from .distance.hamming import value_dtype
            dt = value_dtype(torch.result_type(_probe(lib.data), _probe(Qb)))
            yield b0, eng.hamming_values_tile(lib.device(dt), eng.to_device(Qb, dt), 0, Qb.shape[0], similarity=similarity)
        elif kind == "minkowski":
            dt = staged_dtype(_probe(lib.data), _probe(Qb), p)
            vk, max_token = gemm_value_kind(dt, lib.L)
            if float(p) == 2.0 and vk is not None and lib.L <= eng.GEMM_MAX_WIDTH:
                try:
                    g = lib.gemm(max_token)
                    yield b0, eng.minkowski2_gemm_tile(g, eng.gemm_pack(Qb, max_token=max_token, K=g.K), vk,
                                                       similarity=similarity)
                    continue
                except (OverflowError, L.Unsupported):
                    pass
            yield b0, eng.minkowski_tile(lib.device(dt), eng.to_device(Qb, dt), 0, Qb.shape[0], p=p, similarity=similarity)
        else:
            t = torch.as_tensor(distance(lib.data, Qb, similarity=similarity))
            yield b0, (t if t.is_cuda else t.to(eng.device)).contiguous()
