"""extend_neighbours on the B200: every extension equals build_neighbours on the concatenation bit for
bit (CSR arrays or kNN lists, dtypes, tie order), sampled rows equal the oracle, and the two new
kernels (pg_knn_extend_merge, pg_csr_append) equal a numpy merge on random lists."""
import operator

import numpy as np
import pytest
import torch

from oracle import prograph_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from prograph_b200.engine import get_engine
    return get_engine()


def _library(rng, n, L=40, sites=8, letters=3, wt=None):
    """Mutants of one wild type at a few sites: many duplicates and distance ties."""
    wt = rng.integers(1, 21, size=L) if wt is None else wt
    X = np.tile(wt, (n, 1)).astype(np.int64)
    pos = rng.choice(L, size=sites, replace=False)
    X[:, pos] = rng.integers(1, letters + 1, size=(n, sites))
    return X


def _same(got, want):
    assert type(got) is type(want) and got.row0 == want.row0
    for name in ("indptr", "idx", "w"):
        if hasattr(want, name):
            a, b = getattr(got, name), getattr(want, name)
            assert a.dtype == b.dtype, (name, a.dtype, b.dtype)
            np.testing.assert_array_equal(a, b, err_msg=name)


def _oracle_rows(got, C, args, rng, count=12, extra=()):
    """Sampled rows (and the rows `extra`) of the extension against the CPU oracle."""
    sim = args.get("similarity", False)
    rows = np.unique(np.concatenate([rng.integers(0, len(C), size=count), [0, len(C) - 1], list(extra)]).astype(int))
    D = O.hamming(C, C[rows], similarity=sim)
    if "k" in args:
        ri, rw = O.knn_from_distances(D, min(args["k"], len(C) - 1), descending=sim)
        np.testing.assert_array_equal(got.idx[rows], ri)
        np.testing.assert_array_equal(got.w[rows], rw)
        return
    Dd = O.hamming(C, C[rows])
    eps, comp = args["eps"], args.get("comp", operator.le)
    for j, r in enumerate(rows):
        if sim:
            s = torch.from_numpy(D[j])
            keep = (comp(1 / (1 + eps), s) & (s < 1)).numpy()
        else:
            d = torch.from_numpy(Dd[j])
            keep = (comp(d, eps) & (d > 0)).numpy()
        a, b = got.indptr[r], got.indptr[r + 1]
        np.testing.assert_array_equal(got.idx[a:b], np.nonzero(keep)[0])
        np.testing.assert_array_equal(got.w[a:b], D[j][keep])


def _check(eng, A, B, rng=None, oracle=True, extra=(), **args):
    from prograph_b200 import build_neighbours, extend_neighbours
    from prograph_b200.graph import stack_rows
    prev = build_neighbours(A, engine=eng, **args)
    got = extend_neighbours(prev, A, B, engine=eng, **args)
    C = stack_rows(A, B)
    _same(got, build_neighbours(C, engine=eng, **args))
    if oracle:
        _oracle_rows(got, C, args, rng if rng is not None else np.random.default_rng(0), extra=extra)
    return got


# ---- kNN --------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 16, 32, 77, 100])
@pytest.mark.parametrize("similarity", [False, True])
def test_knn_extension(eng, k, similarity):
    """N in {1, 2, 511, 512, 513, 5000} x M in {1, 7, 512, 3N}; k >= N+M-1 truncates and widens the
    stored lists; k = 100 takes the tile top-k for the candidates and the new rows."""
    rng = np.random.default_rng(k + 1000 * similarity)
    for n in (1, 2, 511, 512, 513, 5000):
        wt = rng.integers(1, 21, size=40)
        for m in sorted({1, 7, 512, 3 * n}):
            X = _library(rng, n + m, wt=wt)
            _check(eng, X[:n], X[n:], rng, k=k, similarity=similarity)


def test_knn_ties_and_duplicates(eng):
    """New rows duplicating old rows and each other; old row 7 duplicates old row 3, so its sorted
    position 0 is row 3 and row 7 itself is a neighbour at d = 0 ahead of every new duplicate."""
    rng = np.random.default_rng(5)
    A = _library(rng, 300, L=20, sites=6, letters=20)
    A[7] = A[3]
    B = np.concatenate([A[[3, 3, 7, 0, 150]], _library(rng, 40, L=20, sites=3, letters=2, wt=A[0])])
    for k in (1, 3, 16, 40, 90):
        for sim in (False, True):
            got = _check(eng, A, B, rng, extra=(3, 7, 300, 301, 302, 303), k=k, similarity=sim)
            if k == 3 and not sim and (A == A[3]).all(1).sum() == 2:
                assert got.idx[7].tolist() == [7, 300, 301]        # position 0 of row 7 is row 3
    # a library of few variants: most rows have duplicates, old and new
    A = _library(rng, 300, L=20, sites=3, letters=2)
    B = _library(rng, 60, L=20, sites=3, letters=2, wt=A[0])
    for k in (1, 16, 90):
        _check(eng, A, B, rng, extra=range(0, 360, 7), k=k)


# ---- epsilon ----------------------------------------------------------------------------------
@pytest.mark.parametrize("comp", [operator.le, operator.lt, operator.eq, operator.ne, lambda a, b: a <= b],
                         ids=["le", "lt", "eq", "ne", "lambda"])
@pytest.mark.parametrize("similarity", [False, True])
def test_eps_extension(eng, comp, similarity):
    rng = np.random.default_rng(11)
    for n, m in ((1, 1), (2, 7), (513, 512), (5000, 700)):
        X = _library(rng, n + m)
        for eps in (1, 2):
            _check(eng, X[:n], X[n:], rng, oracle=n <= 513, eps=eps, comp=comp, similarity=similarity)


def test_eps_rows_without_edges_and_dense(eng):
    from prograph_b200 import build_neighbours, extend_neighbours
    rng = np.random.default_rng(12)
    A = rng.integers(1, 21, size=(300, 64))           # random rows: no pair within distance 1
    B = np.concatenate([A[:1], rng.integers(1, 21, size=(30, 64))])
    B[0, 0] = A[0, 0] % 20 + 1                        # new row 300 at distance 1 from old row 0
    got = _check(eng, A, B, rng, eps=1)
    lst = got.as_list()
    assert len(lst[5][0]) == 0 and lst[5][0].dtype == np.dtype(int) and lst[5][1].dtype == np.dtype(int)
    assert lst[0][0].tolist() == [300] and lst[300][0].tolist() == [0]
    X = _library(rng, 900, L=30, sites=6, letters=2)  # every pair within 6: a dense graph
    got = _check(eng, X[:600], X[600:], rng, eps=6)
    assert got.indptr[-1] > 0.5 * 900 * 899
    prev = build_neighbours(X[:600], eps=6, similarity=True)
    _same(extend_neighbours(prev, X[:600], X[600:], eps=6, similarity=True),
          build_neighbours(X, eps=6, similarity=True))


# ---- shapes -----------------------------------------------------------------------------------
def test_planes_widths_and_columns(eng):
    from prograph_b200.engine import get_engine
    from prograph_b200.graph import informative_table, stack_rows
    rng = np.random.default_rng(13)
    # 5 -> 8 planes through the new rows
    X = _library(rng, 700, L=50)
    B = X[500:].copy()
    B[::7, 3] = 40
    for args in (dict(k=16), dict(k=16, similarity=True), dict(eps=2)):
        _check(eng, X[:500], B, rng, **args)
    assert get_engine().pack(stack_rows(X[:500], B)).planes == 8
    # new rows longer than the old ones (old rows padded with token 0), and the other way round
    A, B = _library(rng, 400, L=40), _library(rng, 60, L=70)
    for args in (dict(k=16), dict(eps=3), dict(k=5, similarity=True)):
        _check(eng, A, B, rng, **args)
        _check(eng, B, A, rng, **args)
    # L = 2048: the chunked sweep
    X = _library(rng, 1200, L=2048, sites=40, letters=4)
    for args in (dict(k=16), dict(eps=20), dict(k=8, similarity=True)):
        _check(eng, X[:1000], X[1000:], rng, **args)
    # a position constant over the old rows and varying over the new ones: the informative columns
    # of the grown table, not of the old one
    X = _library(rng, 6000, L=200, sites=10, letters=3)
    free = np.setdiff1d(np.arange(200), np.nonzero((X != X[0]).any(0))[0])[0]
    B = X[5000:].copy()
    B[::3, free] = (X[0, free] % 20) + 1
    C = stack_rows(X[:5000], B)
    assert informative_table(eng, eng.pack(C)).words < eng.pack(C).words
    for args in (dict(k=16), dict(eps=2), dict(k=16, similarity=True), dict(eps=1, similarity=True)):
        _check(eng, X[:5000], B, rng, **args)


def test_previous_tables_from_the_symmetric_builds(eng):
    """kNN tables of N >= 65 536 rows and epsilon tables of N >= 32 768 come from the symmetric sweeps."""
    rng = np.random.default_rng(17)
    X = _library(rng, 66000, L=56, sites=12, letters=4)
    _check(eng, X[:65536], X[65536:], rng, k=16)
    _check(eng, X[:65536], X[65536:], rng, k=16, similarity=True)
    X = _library(rng, 33500, L=56, sites=12, letters=4)
    _check(eng, X[:32768], X[32768:], rng, eps=2)
    _check(eng, X[:32768], X[32768:], rng, eps=1, similarity=True)


# ---- kernels ----------------------------------------------------------------------------------
def _sorted_lists(rng, rows, width, idx_lo, idx_hi, sim, dmax=6):
    d = np.sort(rng.integers(0, dmax, size=(rows, width)), axis=1)
    # ascending indices beside ascending distances: (distance, index) order
    idx = np.stack([np.sort(rng.choice(np.arange(idx_lo, idx_hi), size=width, replace=False)) for _ in range(rows)])
    cut = rng.integers(0, width + 1, size=rows)          # -1 tails, some rows empty
    cut[::5] = width
    live = np.arange(width)[None, :] < cut[:, None]
    idx = np.where(live, idx, -1)
    w = (np.float32(1) / (1 + d).astype(np.float32)) if sim else d
    return idx, np.where(live, w, 0).astype(np.float32 if sim else np.int64), d


@pytest.mark.parametrize("ka,kb,k", [(0, 5, 3), (16, 16, 16), (15, 16, 16), (77, 20, 78), (100, 100, 150),
                                     (500, 300, 600)])
@pytest.mark.parametrize("similarity", [False, True])
def test_knn_extend_merge_kernel(eng, ka, kb, k, similarity):
    rng = np.random.default_rng(ka * 7 + kb + similarity)
    rows, base = 700, 10_000
    pi, pw, pd = _sorted_lists(rng, rows, ka, 0, 20_000, similarity)
    ci, cw, cd = _sorted_lists(rng, rows, kb, 0, 20_000, similarity)   # overlapping ranges: ties by index
    gi, gw = eng.knn_extend_merge(*(torch.from_numpy(a).cuda() for a in (pi, pw, ci, cw)), base, k, similarity)
    wi = np.full((rows, k), -1, dtype=np.int64)
    ww = np.zeros((rows, k), dtype=np.float32 if similarity else np.int64)
    for r in range(rows):
        ent = [(pd[r, j], pi[r, j], pw[r, j]) for j in range(ka) if pi[r, j] >= 0]
        ent += [(cd[r, j], ci[r, j] + base, cw[r, j]) for j in range(kb) if ci[r, j] >= 0]
        ent = sorted(ent, key=lambda e: (e[0], e[1]))[:k]
        for j, (_, i, x) in enumerate(ent):
            wi[r, j], ww[r, j] = i, x
    np.testing.assert_array_equal(gi.cpu().numpy(), wi)
    assert gw.dtype == (torch.float32 if similarity else torch.int64)
    np.testing.assert_array_equal(gw.cpu().numpy(), ww)


@pytest.mark.parametrize("similarity", [False, True])
@pytest.mark.parametrize("rows", [1, 33, 5000])
def test_csr_append_kernel(eng, rows, similarity):
    rng = np.random.default_rng(rows + similarity)
    wdt = np.float32 if similarity else np.int64

    def csr(max_deg, offset):
        deg = rng.integers(0, max_deg + 1, size=rows)
        deg[::4] = 0
        ip = np.concatenate([[0], np.cumsum(deg)]) + offset            # a row slice of a larger CSR
        return ip, rng.integers(0, 9999, size=ip[-1] - offset), rng.random(ip[-1] - offset).astype(wdt) * 100

    (oip, oi, ow), (aip, ai, aw) = csr(90, 17), csr(40, 0)
    gp, gi, gw = eng.csr_append(tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (oip, oi, ow)),
                                tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (aip, ai, aw)),
                                50_000, similarity)
    o, a = oip - oip[0], aip
    wi = np.concatenate([np.concatenate([oi[o[r]:o[r + 1]], ai[a[r]:a[r + 1]] + 50_000]) for r in range(rows)])
    ww = np.concatenate([np.concatenate([ow[o[r]:o[r + 1]], aw[a[r]:a[r + 1]]]) for r in range(rows)])
    np.testing.assert_array_equal(gp.cpu().numpy(), o + a)
    np.testing.assert_array_equal(gi.cpu().numpy(), wi)
    np.testing.assert_array_equal(gw.cpu().numpy(), ww)


# ---- errors and fallback ----------------------------------------------------------------------
def test_errors_and_rebuild_fallback(eng):
    from prograph_b200 import KnnTable, build_neighbours, extend_neighbours, minkowski
    rng = np.random.default_rng(19)
    X = _library(rng, 400)
    A, B = X[:300], X[300:]
    knn = build_neighbours(A, k=8)
    eps = build_neighbours(A, eps=2)
    for bad, kwargs in ((knn, dict(k=8, similarity=True)), (eps, dict(k=8)), (knn, dict(eps=2)),
                        (knn, dict(k=9)), (KnnTable(knn.idx[:100], knn.w[:100]), dict(k=8)),
                        (KnnTable(knn.idx, knn.w, row0=5), dict(k=8)), (eps, dict(eps=2, similarity=True))):
        with pytest.raises(ValueError):
            extend_neighbours(bad, A, B, **kwargs)
    with pytest.raises(ValueError):
        extend_neighbours(knn, A, B[:0], k=8)
    # Minkowski and Hamming on non-token values take the rebuild of the concatenation
    for args in (dict(k=8, distance=minkowski), dict(eps=3.0, distance=minkowski), dict(k=8, similarity=True,
                                                                                      distance=minkowski)):
        _check(eng, A, B, oracle=False, **args)
    V = X.astype(np.float64) + 0.5
    _check(eng, V[:300], V[300:], oracle=False, k=8)
