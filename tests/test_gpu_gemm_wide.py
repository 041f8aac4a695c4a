"""The K-chunked mode of the tcgen05 Minkowski p=2 GEMM (pg_gemm.cu, rows of 257 .. 8192 tokens).

Rows wider than 256 tokens do not leave room for two resident A tiles, so every ring stage carries
one 128-wide K-chunk of A tile 0, A tile 1 and the B tile, and the MMA issuers accumulate the chunks
of a B tile into one TMEM accumulator.  Every case compares bit for bit (fp16 as uint16) with the
element-wise kernel (eng.minkowski_tile) on the same device data, with oracle/prograph_oracle.py on a
sample of rows, and for kNN lists with a stable sort.  Inputs are seeded and tie-heavy: mutational
libraries with duplicated rows, and one-hot rows, where S = 2 * Hamming.

Code path -> test:
  chunk loop, partial last chunk, descriptors, accumulate flag   test_chunked_widths
  S up to 255^2 * 8192 (int32 epilogue sums, eps range bound)    test_chunked_integer_range
  L = 8193: Unsupported, public calls take the element-wise path  test_width_limit
  kNN lists on the chunked ring, 42 / 43 limit, 1 or 2 issuers     test_chunked_knn_list_lengths
  epsilon count / fill for every comparison, similarity on / off  test_chunked_eps_comparisons
  M / N edges, -1 / 0 tails, dataset split, ld > N stores          test_chunked_row_and_column_edges
  public API on wide rows, GEMM dispatch proven                    test_public_* (minkowski_tile raises)
"""
import operator

import numpy as np
import pytest
import torch

from oracle import prograph_oracle as O

pytestmark = pytest.mark.gpu

# largest k + drop of the chunked mode: 256 lists of 12-byte entries next to a 2-stage ring of
# 3 x 16 KB stages, the norm ring and the barriers (gemm_smem_bytes <= 227 KB): 42 at every K > 256
CHUNKED_MAX_K1 = 42
WIDTHS = [288, 320, 352, 384, 416, 512, 640, 1184, 2048, 5376, 8192]


@pytest.fixture(scope="module")
def eng():
    from prograph_b200.engine import get_engine
    return get_engine()


def unsupported():
    from prograph_b200._lib import Unsupported
    return Unsupported


def np_(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def same(got, want):
    """Bit-exact comparison (fp16 as uint16), dtypes included."""
    got, want = np_(got), np_(want)
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    if got.dtype == np.float16:
        got, want = got.view(np.uint16), want.view(np.uint16)
    np.testing.assert_array_equal(got, want)


def library(rng, n, L, alphabet=20, max_mut=6, dup_every=37):
    """Mutational library: a random wild type, 1..max_mut substitutions per row (tokens
    1..alphabet), every dup_every-th row a copy of the row before it (distance-0 ties)."""
    wt = rng.integers(1, alphabet + 1, size=L)
    X = np.tile(wt, (n, 1))
    for i in range(1, n):
        pos = rng.choice(L, size=min(int(rng.integers(1, max_mut + 1)), L), replace=False)
        X[i, pos] = (X[i, pos] - 1 + rng.integers(1, alphabet, size=len(pos))) % alphabet + 1
    for i in range(dup_every, n, dup_every):
        X[i] = X[i - 1]
    return X.astype(np.int64)


def one_hot(tokens, alphabet=21):
    """(n, L) tokens in [0, alphabet) -> (n, L * alphabet) 0/1 rows."""
    n, L = tokens.shape
    out = np.zeros((n, L, alphabet), dtype=np.int64)
    np.put_along_axis(out, tokens[:, :, None], 1, axis=2)
    return out.reshape(n, L * alphabet)


def staged(eng, X, kind):
    return eng.to_device(np.ascontiguousarray(X)).to(torch.float16 if kind == 0 else torch.int64)


def elem(eng, X, Q, kind, sim=False):
    """The element-wise kernel's (M, N) matrix of queries Q against dataset X."""
    Xd, Qd = staged(eng, X, kind), staged(eng, Q, kind)
    return eng.minkowski_tile(Xd, Qd, 0, Qd.shape[0], p=2, similarity=sim)


def oracle_rows(X, Q, kind, rows):
    dt = np.float16 if kind == 0 else np.int64
    return np.concatenate([O.minkowski(X.astype(dt), Q[r:r + 1].astype(dt)) for r in rows])


def sq_sums(X, Q):
    X, Q = X.astype(np.int64), Q.astype(np.int64)
    return (X * X).sum(1)[None, :] + (Q * Q).sum(1)[:, None] - 2 * (Q @ X.T)


def tables(eng, X, Q, kind):
    tx = eng.gemm_pack(X, max_token=31 if kind == 0 else 255)
    return tx, eng.gemm_pack(Q, max_token=tx.max_token, K=tx.K)


def knn_ref(D, k, drop, descending=False):
    order = np.argsort(-D if descending else D, axis=1, kind="stable")[:, drop:drop + k]
    idx = np.full((D.shape[0], k), -1, dtype=np.int64)
    w = np.zeros((D.shape[0], k), dtype=D.dtype)
    idx[:, :order.shape[1]] = order
    w[:, :order.shape[1]] = np.take_along_axis(D, order, axis=1)
    return idx, w


def check_tile(eng, tx, tq, X, Q, kind):
    for sim in (False, True):
        same(eng.minkowski2_gemm_tile(tx, tq, kind, similarity=sim), elem(eng, X, Q, kind, sim))


def check_knn(eng, tx, tq, X, Q, kind, k, drop):
    for sim in (False, True):
        D = np_(elem(eng, X, Q, kind, sim))
        idx, w = eng.minkowski2_gemm_knn(tx, tq, k, drop, kind, similarity=sim)
        ri, rw = knn_ref(D, k, drop, descending=sim)
        same(idx, ri)
        same(w, rw)


def check_eps(eng, tx, tq, X, Q, kind, lo, hi):
    keep = (sq_sums(X, Q) >= lo) & (sq_sums(X, Q) <= hi)
    rows, cols = np.nonzero(keep)
    for sim in (False, True):
        D = np_(elem(eng, X, Q, kind, sim))
        indptr, idx, w = eng.minkowski2_gemm_eps(tx, tq, lo, hi, kind, similarity=sim)
        same(indptr, np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64))
        same(idx, cols.astype(np.int64))
        same(w, D[rows, cols])


@pytest.fixture
def gemm_only(eng, monkeypatch):
    """The element-wise Minkowski kernel raises: whatever answers came from the GEMM.  References
    are computed before the fixture is requested, or with `ref_elem` (the unpatched kernel)."""
    real = eng.minkowski_tile

    def boom(*a, **k):
        raise AssertionError("the element-wise kernel was called")

    monkeypatch.setattr(eng, "minkowski_tile", boom)
    return real


# ------------------------------------------------------------------ engine level
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("K", WIDTHS)
def test_chunked_widths(eng, K, kind):
    """L = K and L = K - 5 (the pack pads to K; K - 5 leaves zero columns in the last chunk), tiles
    with and without similarity, kNN and an epsilon graph.  Chunks of 128: the last chunk of K = 288 /
    416 / 1184 is 32 wide (one k-step), of K = 320 64 (two), of K = 352 96 (three), and full (four)
    for K = 384, 512, 640, 2048, 5376 and 8192; K = 640 has five chunks, K = 8192 sixty-four."""
    rng = np.random.default_rng(K * 2 + kind)
    for L in (K, K - 5):
        n = 300 if K <= 2048 else 160
        if kind == 0:
            X = library(rng, n, L, alphabet=31, max_mut=12)
        else:
            X = library(rng, n, L, alphabet=256, max_mut=12) - 1
            X[5, :64], X[6, :64] = 255, 0
        Q = X[: n // 2 + 3]
        tx, tq = tables(eng, X, Q, kind)
        assert tx.K == K
        check_tile(eng, tx, tq, X, Q, kind)
        same(eng.minkowski2_gemm_tile(tx, tq, kind)[:3], oracle_rows(X, Q, kind, range(3)))
        check_knn(eng, tx, tq, X, Q, kind, 9, 1)
        hi = 6 * 31 * 31 if kind == 0 else 6 * 255 * 255
        check_eps(eng, tx, tq, X, Q, kind, 1, hi)


def test_chunked_integer_range(eng):
    """K = 8192, tokens 0 / 255: rows all 0 against all 255 give S = 255^2 * 8192 = 532 684 800, the
    largest sum of the path; neighbours one token away give S - 509 and 509."""
    K = 8192
    rng = np.random.default_rng(8192)
    X = rng.integers(0, 256, size=(200, K))
    X[0], X[1], X[2], X[3] = 0, 255, 255, 0
    X[2, 17], X[3, 4000] = 254, 1
    X[4] = X[1]
    Q = X[:40]
    tx, tq = tables(eng, X, Q, 1)
    S = sq_sums(X, Q)
    assert S.max() == 255 * 255 * K
    check_tile(eng, tx, tq, X, Q, 1)
    same(eng.minkowski2_gemm_tile(tx, tq, 1)[:4], oracle_rows(X, Q, 1, range(4)))
    check_knn(eng, tx, tq, X, Q, 1, 5, 0)
    check_knn(eng, tx, tq, X, Q, 1, 12, 1)
    check_eps(eng, tx, tq, X, Q, 1, 1, 255 * 255 * K)
    check_eps(eng, tx, tq, X, Q, 1, 255 * 255 * K - 509, 255 * 255 * K - 1)


@pytest.mark.parametrize("issuers", [None, "1", "2"])
def test_chunked_knn_list_lengths(eng, monkeypatch, issuers):
    """k + drop in {1, 2, 4, 5 (issuer switch), 17, 42}; 43 raises Unsupported (found by calling).
    PG_GEMM_ISSUERS forces one or two MMA-issuing warps."""
    if issuers is not None:
        monkeypatch.setenv("PG_GEMM_ISSUERS", issuers)
    rng = np.random.default_rng(1184 + (0 if issuers is None else int(issuers)))
    X = library(rng, 500, 1184, alphabet=6, max_mut=8)
    tabs = {kind: eng.gemm_pack(X, max_token=31 if kind == 0 else 255) for kind in (0, 1)}

    def fits(k1):
        try:
            eng.minkowski2_gemm_knn(tabs[0], tabs[0], k1, 0, 0)
            return True
        except unsupported():
            return False

    top = next(k1 for k1 in range(96, 0, -1) if fits(k1))
    assert top == CHUNKED_MAX_K1
    with pytest.raises(unsupported()):
        eng.minkowski2_gemm_knn(tabs[1], tabs[1], top, 1, 1)
    for kind in (0, 1):
        for k1 in (1, 2, 4, 5, 17, top):
            check_knn(eng, tabs[kind], tabs[kind], X, X, kind, k1, 0)
            if k1 > 1:
                check_knn(eng, tabs[kind], tabs[kind], X, X, kind, k1 - 1, 1)
    check_tile(eng, tabs[1], tabs[1], X, X, 1)


@pytest.mark.parametrize("comp", [operator.lt, operator.le, operator.eq, operator.ge, operator.gt])
@pytest.mark.parametrize("sim", [False, True])
def test_chunked_eps_comparisons(eng, comp, sim):
    """build_neighbours(eps) on 1 176-column one-hot rows takes the fused count / fill passes; the
    reference is the threshold compaction (eng.tile_threshold) of the element-wise tile, the path
    such rows took before.  eps = 2 hits S = 4 exactly (Hamming 2)."""
    from prograph_b200 import build_neighbours, minkowski
    from prograph_b200 import _lib as L
    rng = np.random.default_rng(56)
    X = one_hot(library(rng, 400, 56, alphabet=20, max_mut=4) % 21)
    eps = 2.0
    e = 1 / (1 + eps) if sim else eps
    Xd = eng.to_device(X).to(torch.float16)
    tile = eng.minkowski_tile(Xd, Xd, 0, len(X), p=2, similarity=sim)
    code = {operator.lt: L.LT, operator.le: L.LE, operator.eq: L.EQ, operator.ge: L.GE, operator.gt: L.GT}[comp]
    ip, i, w = eng.tile_threshold(tile, code, e, swap=sim, guard=2 if sim else 1)
    mp = pytest.MonkeyPatch()
    mp.setattr(eng, "minkowski_tile", lambda *a, **k: (_ for _ in ()).throw(AssertionError("element-wise")))
    try:
        got = build_neighbours(X, eps=eps, comp=comp, similarity=sim, distance=minkowski)
    finally:
        mp.undo()
    same(got.indptr, ip)
    same(got.idx, i)
    same(got.w, w)


@pytest.mark.parametrize("M", [1, 255, 256, 257])
def test_chunked_row_and_column_edges(eng, M):
    """Query rows around the two A tiles of a CTA against datasets of 1, 127, 128 and 129 rows at
    K = 416 (three full chunks and one of 32): tiles (odd N: scalar stores), kNN with k + drop > N
    (-1 / 0 tails) and the epsilon graph; a tile with ld > N through the C entry point."""
    from prograph_b200 import _lib as L
    from prograph_b200.engine import _ptr
    rng = np.random.default_rng(M + 416)
    pool = library(rng, 600, 411, alphabet=20, max_mut=8)
    Q = pool[-M:]
    for N in (1, 127, 128, 129):
        X = pool[:N]
        for kind in (0, 1):
            tx, tq = tables(eng, X, Q, kind)
            check_tile(eng, tx, tq, X, Q, kind)
            check_knn(eng, tx, tq, X, Q, kind, 3, 1)
            check_knn(eng, tx, tq, X, Q, kind, 5, 0)
            check_eps(eng, tx, tq, X, Q, kind, 1, 2000)
            for ld in (N + 3, N + 8 - N % 8):
                dt = torch.float16 if kind == 0 else torch.float32
                out = torch.full((M, ld), -7.0, dtype=dt, device=eng.device)
                L.check(eng.lib.pg_minkowski2_gemm_tile(_ptr(tq.data), _ptr(tq.norms), tq.rows, _ptr(tx.data),
                                                        _ptr(tx.norms), tx.rows, tx.K, kind, 0, _ptr(out), ld,
                                                        eng._stream()))
                same(out[:, :N], elem(eng, X, Q, kind))
                assert bool((out[:, N:] == -7.0).all())


def test_chunked_tile_split_dataset(eng):
    """100 queries x 4 097 rows at K = 1 184: the tile kernel splits the dataset across gridDim.y
    and the odd row length makes every store take the scalar path."""
    rng = np.random.default_rng(4097)
    X = library(rng, 4097, 1184, alphabet=20, max_mut=10)
    Q = library(rng, 100, 1184, alphabet=20, max_mut=10)
    for kind in (0, 1):
        tx, tq = tables(eng, X, Q, kind)
        check_tile(eng, tx, tq, X, Q, kind)


# ------------------------------------------------------------------ public API
def test_width_limit(eng):
    """L = 8193 is one token past the GEMM: gemm_pack raises Unsupported, and minkowski,
    build_neighbours and the query entry points answer as the element-wise kernel does."""
    from prograph_b200 import build_neighbours, minkowski, query
    rng = np.random.default_rng(8193)
    X = library(rng, 90, 8193, alphabet=20, max_mut=30)
    Q = X[:7]
    with pytest.raises(unsupported()):
        eng.gemm_pack(X)
    for kind, dt in ((1, np.int64), (0, np.float16)):
        same(minkowski(X.astype(dt), Q.astype(dt)), elem(eng, X, Q, kind))
    D16 = np_(elem(eng, X, X, 0))
    got = build_neighbours(X, k=4, distance=minkowski)
    ri, rw = knn_ref(D16, 4, 1)
    same(got.idx, ri)
    same(got.w, rw)
    lib = query.Library(X)
    D = np_(elem(eng, X, Q, 1))
    mi, mv = query.nearest(lib, Q, distance=minkowski)
    same(mi, D.argmin(axis=1))
    same(mv, D.min(axis=1))
    same(query.tile(lib, Q, distance=minkowski), D)
    same(query.count_within(lib, Q, 8.0, distance=minkowski), (D <= 8.0).sum(axis=1).astype(np.int64))


@pytest.mark.parametrize("L", [300, 1176, 8192])
def test_public_minkowski_wide_rows(eng, gemm_only, L):
    """minkowski(X, Y) on wide int64 and fp16 rows answers through the GEMM, bit for bit with the
    element-wise kernel; float32 rows take it while L * max_token^2 <= 2^24 and fall back above."""
    from prograph_b200 import minkowski
    rng = np.random.default_rng(L)
    X = library(rng, 150, L, alphabet=31, max_mut=20)
    Y = X[:33]
    ref = {kind: gemm_only(staged(eng, X, kind), staged(eng, Y, kind), 0, len(Y)) for kind in (0, 1)}
    same(minkowski(X, Y), ref[1])
    same(minkowski(X.astype(np.float16), Y.astype(np.float16)), ref[0])
    same(minkowski(X, Y, similarity=True),
         gemm_only(staged(eng, X, 1), staged(eng, Y, 1), 0, len(Y), similarity=True))
    # float32 rows of tokens <= 31: 961 * L <= 2^24 for every L here
    X32, Y32 = X.astype(np.float32), Y.astype(np.float32)
    same(minkowski(X32, Y32), gemm_only(eng.to_device(X32), eng.to_device(Y32), 0, len(Y)))


def test_public_float32_token_cap(eng, monkeypatch):
    """float32 rows of 1 184 columns: tokens <= 119 (1184 * 119^2 <= 2^24) take the GEMM, a token of
    120 sends the call to the element-wise kernel, which sums in float32."""
    from prograph_b200 import minkowski
    rng = np.random.default_rng(119)
    X = rng.integers(0, 120, size=(80, 1184)).astype(np.float32)
    X[1] = 119
    X[2] = 0
    Y = X[:9].copy()
    ref = eng.minkowski_tile(eng.to_device(X), eng.to_device(Y), 0, len(Y))
    calls = []
    real = eng.minkowski_tile
    monkeypatch.setattr(eng, "minkowski_tile", lambda *a, **k: calls.append(1) or real(*a, **k))
    same(minkowski(X, Y), ref)
    assert not calls
    X[3, 7] = 120
    ref = real(eng.to_device(X), eng.to_device(Y), 0, len(Y))
    same(minkowski(X, Y), ref)
    assert calls


def test_public_build_graph_one_hot(eng, gemm_only):
    """build_neighbours(distance=minkowski) kNN and epsilon graphs on one-hot rows of 56 x 21 = 1 176
    columns (the GB1 library's shape) through the GEMM, against the reference's graph."""
    from prograph_b200 import build_neighbours, minkowski
    rng = np.random.default_rng(1176)
    X = one_hot(library(rng, 160, 56, alphabet=20, max_mut=4))
    assert X.shape[1] == 1176
    for k in (1, 8, 41):
        got = build_neighbours(X, k=k, distance=minkowski).to_csr()
        for g, r in zip((got.indptr, got.idx, got.w), O.to_csr(O.build_graph(X, k=k, distance=O.minkowski))):
            same(g, r)
    for eps, sim in ((2.0, False), (3.0, False), (2.0, True)):
        got = build_neighbours(X, eps=eps, distance=minkowski, similarity=sim)
        want = O.build_graph(X, eps=eps, distance=O.minkowski, similarity=sim)
        for g, r in zip((got.indptr, got.idx, got.w), O.to_csr(want)):
            same(g, r)


def test_public_prograph_build_graph_representation(eng, gemm_only, tmp_path):
    """Prograph.build_graph(representation=...) with a one-hot column of 1 176 entries per row."""
    import pandas as pd
    import prograph_b200 as pgb
    rng = np.random.default_rng(21)
    tok = library(rng, 120, 56, alphabet=20, max_mut=4)
    aa = np.array(list(O.AMINO_ACIDS))
    seqs = ["".join(aa[t - 1]) for t in tok]
    path = tmp_path / "lib.csv"
    pd.DataFrame({"Sequence": seqs, "Fitness": rng.normal(size=len(seqs)),
                  "Neighbours": ["[]"] * len(seqs)}).to_csv(path)
    pg = pgb.Prograph(file=str(path))
    X = one_hot(tok)
    pg.graph["OneHot"] = list(X)
    for kw in ({"k": 6}, {"eps": 2.0}):
        got = pg.build_graph(representation="OneHot", distance=pgb.minkowski, **kw)
        want = O.build_graph(X, distance=O.minkowski, **kw)
        assert len(got) == len(want)
        for (gi, gw), (ri, rw) in zip(got, want):
            same(gi, ri)
            same(gw, rw)


def test_public_query_wide_library(eng, gemm_only):
    """query.nearest, query.tile and query.count_within on a library of 2 048-token rows."""
    from prograph_b200 import minkowski, query
    rng = np.random.default_rng(2048)
    X = library(rng, 700, 2048, alphabet=20, max_mut=12)
    Q = library(rng, 300, 2048, alphabet=20, max_mut=12)
    Q[:5] = X[10:15]
    D = np_(gemm_only(staged(eng, X, 1), staged(eng, Q, 1), 0, len(Q)))
    lib = query.Library(X)
    mi, mv = query.nearest(lib, Q, distance=minkowski)
    same(mi, D.argmin(axis=1))
    same(mv, D.min(axis=1))
    same(query.tile(lib, Q, distance=minkowski), D)
    same(query.tile(lib, Q, 7, 30, distance=minkowski, similarity=True),
         np_(gemm_only(staged(eng, X, 1), staged(eng, Q[7:37], 1), 0, 30, similarity=True)))
    for eps, comp in ((10.0, operator.le), (12.0, operator.lt), (0.0, operator.eq)):
        same(query.count_within(lib, Q, eps, comp, distance=minkowski), comp(D, eps).sum(axis=1).astype(np.int64))
