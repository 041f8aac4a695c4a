"""CPU-side checks of extend_neighbours: the similarity order its kNN merge relies on, its argument
checks, and its sharded host logic over gloo with an oracle-backed engine.  No kernel is launched."""
import operator
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _cpu_engine import CheckerEngine, _Packed  # noqa: E402


class ExtendEngine(CheckerEngine):
    """The checker engine plus the engine calls extend_neighbours adds, answered in numpy."""

    def gather_packed(self, table, rows):
        return _Packed(table.tokens[np.asarray(rows)])

    def knn_extend_merge(self, prev_idx, prev_w, cand_idx, cand_w, col_base, k, similarity=False):
        self.merged = getattr(self, "merged", 0) + prev_idx.shape[0]
        wdt = np.float32 if similarity else np.int64
        pi, pw, ci, cw = (t.numpy() for t in (prev_idx, prev_w, cand_idx, cand_w))
        idx = np.full((pi.shape[0], k), -1, dtype=np.int64)
        w = np.zeros((pi.shape[0], k), dtype=wdt)
        for r in range(pi.shape[0]):
            ent = [(wdt(x), int(i)) for x, i in zip(pw[r], pi[r]) if i >= 0]
            ent += [(wdt(x), int(i) + col_base) for x, i in zip(cw[r], ci[r]) if i >= 0]
            ent = sorted(ent, key=lambda e: (-e[0] if similarity else e[0], e[1]))[:k]
            for j, (x, i) in enumerate(ent):
                idx[r, j], w[r, j] = i, x
        return torch.from_numpy(idx), torch.from_numpy(w)

    def csr_append(self, old, add, col_base, similarity=False):
        (oip, oi, ow), (aip, ai, aw) = ([t.numpy() for t in part] for part in (old, add))
        oip, aip = oip - oip[0], aip - aip[0]
        idx, w = [], []
        for r in range(len(oip) - 1):
            idx += [oi[oip[r]:oip[r + 1]], ai[aip[r]:aip[r + 1]] + col_base]
            w += [ow[oip[r]:oip[r + 1]], aw[aip[r]:aip[r + 1]]]
        wdt = np.float32 if similarity else np.int64
        return (torch.from_numpy(oip + aip), torch.from_numpy(np.concatenate(idx).astype(np.int64)),
                torch.from_numpy(np.concatenate(w).astype(wdt)))


def test_similarity_is_strictly_decreasing_in_the_distance():
    """The kNN merge orders similarities (desc, index) and takes that for the (distance, index)
    order: float32 1/(1+d) must be strictly decreasing over every distance a sweep returns, and the
    same number on the tile path (torch) as in the kernels (a correctly rounded float32 divide)."""
    d = np.arange(32769, dtype=np.int64)
    s = np.float32(1) / (1 + d).astype(np.float32)
    assert s.dtype == np.float32 and np.all(np.diff(s) < 0)
    t = (1 / (1 + torch.from_numpy(d))).numpy()
    assert t.dtype == np.float32 and np.array_equal(t.view(np.uint32), s.view(np.uint32))


def _tables(eng):
    from prograph_b200.graph import build_neighbours
    rng = np.random.default_rng(1)
    X = rng.integers(1, 4, size=(20, 10)).astype(np.int64)
    return X, build_neighbours(X, k=4, engine=eng), build_neighbours(X, eps=2, engine=eng)


def test_argument_errors():
    from prograph_b200.graph import KnnTable, NeighbourTable, extend_neighbours
    eng = ExtendEngine()
    X, knn, eps = _tables(eng)
    new = X[:3] + 1
    with pytest.raises(ValueError, match="no new rows"):
        extend_neighbours(knn, X, X[:0], k=4, engine=eng)
    with pytest.raises(ValueError):
        extend_neighbours(knn, X, new, engine=eng)                     # neither eps nor k
    with pytest.raises(ValueError):
        extend_neighbours(knn, X, new, eps=1, k=4, engine=eng)
    with pytest.raises(TypeError):
        extend_neighbours(knn, X, new, k=2.5, engine=eng)
    with pytest.raises(ValueError, match="output"):
        extend_neighbours(knn, X, new, k=4, engine=eng, output="local")
    with pytest.raises(ValueError, match="KnnTable"):
        extend_neighbours(eps, X, new, k=4, engine=eng)
    with pytest.raises(ValueError, match="NeighbourTable"):
        extend_neighbours(knn, X, new, eps=2, engine=eng)
    with pytest.raises(ValueError, match="neighbours per row"):
        extend_neighbours(knn, X, new, k=5, engine=eng)
    with pytest.raises(ValueError, match="whole graph"):               # a shard of another rank
        extend_neighbours(KnnTable(knn.idx[10:], knn.w[10:], row0=10), X[10:], new, k=4, engine=eng)
    with pytest.raises(ValueError, match="whole graph"):               # rows missing
        extend_neighbours(KnnTable(knn.idx[:10], knn.w[:10]), X, new, k=4, engine=eng)
    with pytest.raises(ValueError, match="whole graph"):
        part = NeighbourTable(eps.indptr[:11], eps.idx[:eps.indptr[10]], eps.w[:eps.indptr[10]])
        extend_neighbours(part, X, new, eps=2, engine=eng)
    with pytest.raises(ValueError, match="weights"):                   # a distance table, similarity asked
        extend_neighbours(knn, X, new, k=4, similarity=True, engine=eng)
    with pytest.raises(ValueError, match="weights"):
        extend_neighbours(eps, X, new, eps=2, similarity=True, engine=eng)


def _cases(eng, group=None, output="replicated"):
    """(extended, rebuilt) pairs of a few growths; new rows longer than the old ones, duplicates."""
    from prograph_b200.graph import build_neighbours, extend_neighbours
    rng = np.random.default_rng(7)
    out = []
    for n_old, m in ((30, 13), (5, 40), (1, 3)):
        A = rng.integers(1, 4, size=(n_old, 10)).astype(np.int64)
        B = rng.integers(1, 4, size=(m, 12)).astype(np.int64)
        B[0, :10], B[0, 10:] = A[0], 0                                 # a duplicate of old row 0
        B[1] = B[0]
        C = np.concatenate([np.pad(A, ((0, 0), (0, 2))), B])
        for args in (dict(k=4), dict(k=50), dict(k=6, similarity=True), dict(eps=2), dict(eps=1, similarity=True),
                     dict(eps=2, comp=operator.ne)):
            prev = build_neighbours(A, engine=eng, group=group, **args)
            got = extend_neighbours(prev, A, B, engine=eng, group=group, output=output, **args)
            want = build_neighbours(C, engine=eng, group=group, output=output, **args)
            out.append((got, want, C, args))
    return out


def _assert_same(got, want):
    assert type(got) is type(want) and got.row0 == want.row0
    names = ("indptr", "idx", "w") if hasattr(want, "indptr") else ("idx", "w")
    for name in names:
        a, b = getattr(got, name), getattr(want, name)
        assert a.dtype == b.dtype and np.array_equal(a, b), name


def test_extension_equals_the_rebuild_on_one_rank():
    from oracle import prograph_oracle as O
    eng = ExtendEngine()
    for got, want, C, args in _cases(eng):
        _assert_same(got, want)
        if "k" in args:
            ri, rw = O.knn_from_distances(O.hamming(C, C, similarity=args.get("similarity", False)),
                                          min(args["k"], len(C) - 1), descending=args.get("similarity", False))
            assert np.array_equal(got.idx, ri) and np.array_equal(got.w, rw)
    assert eng.merged > 0


def _gloo_worker(rank, world, port, tmpdir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    eng = ExtendEngine()
    arrays = {}
    for output in ("replicated", "sharded"):
        for c, (got, want, _, _) in enumerate(_cases(eng, output=output)):
            for name in ("indptr", "idx", "w"):
                if hasattr(want, name):
                    arrays[f"{output}{c}{name}"] = getattr(got, name)
                    arrays[f"{output}{c}{name}_want"] = getattr(want, name)
            arrays[f"{output}{c}row0"] = np.array([got.row0, want.row0])
    np.savez(os.path.join(tmpdir, f"r{rank}.npz"), rows=np.array(eng.rows_seen), **arrays)
    dist.destroy_process_group()


def test_sharded_extension_over_gloo(tmp_path):
    """world_size 2 on CPU: each rank extends the rows of its block of the grown table (old rows
    through the merge / append, new rows through the one-sided sweep) and the all-gathers, or the
    sharded output, match a rebuild of the concatenation on the same ranks."""
    import torch.multiprocessing as mp
    world = 2
    port = 29400 + os.getpid() % 150
    mp.spawn(_gloo_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        z = np.load(tmp_path / f"r{r}.npz")
        keys = [key for key in z.files if key.endswith("_want")]
        assert len(keys) >= 36
        for key in keys:
            got, want = z[key[:-5]], z[key]
            assert got.dtype == want.dtype and np.array_equal(got, want), (r, key)
        for key in (f for f in z.files if f.endswith("row0")):
            assert z[key][0] == z[key][1], (r, key)
