"""Boundary cases of the two fused kernel families, bit for bit against the numpy oracle.

The fused Hamming sweeps (pg_sweep.cu, pg_sweep.cuh, pg_sweep_long.cu) and the tcgen05 int8
Minkowski GEMM (pg_gemm.cu) pick their code paths from the bit-plane count, the row width, the list
length (rounds of 32 entries against a shared-memory budget), the split count, the ring-stage count,
the number of MMA-issuing warps and the output alignment.  Every case here sits on one side of such
a boundary and compares the kernel with oracle/prograph_oracle.py: a stable sort of the oracle
matrix for kNN lists, the oracle's edge test for epsilon graphs, the oracle matrix itself for tiles.
Inputs are seeded and full of ties (small alphabets, duplicated rows, mutational libraries), so a
wrong tie order fails as surely as a wrong distance.

Code path -> test:
  8 bit planes, kNN / count / fill / capture / flags epilogues   test_sweep_planes_widths_epilogues
  long rows (words 40, 48, 56), range and LUT predicates          test_sweep_planes_widths_epilogues
  list rounds of knn_insert_coop, 78 / 79 limit, 32-row merge     test_sweep_list_length_boundaries
  multi-split merge, fill split prefix, overflow-row fill sweep   test_sweep_forced_splits
  stream_rows edges, -1 tails and their weight, long-row pad rows  test_sweep_stream_edges
  list rounds of knn_insert_coop_s, ring stages 4 -> 2            test_gemm_list_length_boundaries
  M / N edges, fast and scalar tile stores                        test_gemm_row_and_column_edges
  instruction / smem descriptors for K = 32 .. 256, value kinds   test_gemm_every_width
  one or two MMA issuers at short and long lists                  test_gemm_forced_issuers
  tile-mode dataset split (gridDim.y > 1) with odd N              test_gemm_tile_split_dataset_odd_rows
  fp16 chain overflow to inf, inf ties                            test_gemm_fp16_overflow_ties
  pad columns of the last B tile when N < k + drop                test_gemm_knn_short_dataset_has_empty_tail
"""
import operator

import numpy as np
import pytest
import torch

from oracle import prograph_oracle as O

pytestmark = pytest.mark.gpu


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
    got, want = np_(got), np.asarray(want)
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


def knn_ref(D, k, drop, descending=False):
    """Sorted positions [drop, drop+k) of every row of D in (value, index) order -- torch's stable
    sort of prograph.py:757-762.  Positions past the end of a row: index -1, weight 0."""
    order = np.argsort(-D if descending else D, axis=1, kind="stable")[:, drop:drop + k]
    idx = np.full((D.shape[0], k), -1, dtype=np.int64)
    w = np.zeros((D.shape[0], k), dtype=D.dtype)
    idx[:, :order.shape[1]] = order
    w[:, :order.shape[1]] = np.take_along_axis(D, order, axis=1)
    return idx, w


def csr_ref(W, keep):
    rows, cols = np.nonzero(keep)
    return np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64), cols.astype(np.int64), W[rows, cols]


def check_knn(got, D, k, drop, descending=False):
    ri, rw = knn_ref(D, k, drop, descending)
    same(got[0], ri)
    same(got[1], rw)


def check_csr(got, W, keep):
    for g, r in zip(got, csr_ref(W, keep)):
        same(g, r)


# ------------------------------------------------------------------ fused Hamming sweeps
def hamming_eps_keep(D, comp, eps):
    return comp(D, eps) & (D > 0)                      # prograph.py:736


@pytest.mark.parametrize("Lw,alphabet", [(7, 200), (33, 200), (100, 200), (256, 200),
                                         (1200, 20), (1500, 20), (1792, 20)])
def test_sweep_planes_widths_epilogues(eng, Lw, alphabet):
    """8 bit planes at words 1, 2, 4, 8 and long rows at words 40, 48, 56: kNN (drop 0 / 1, both
    weight kinds), epsilon graphs with a range (le) and a LUT (ne) predicate, with the default
    capture and with one that holds every hit, membership flags, and queries of another table
    starting at a row that is not a multiple of 256."""
    from prograph_b200.graph import distance_lut
    rng = np.random.default_rng(Lw * 7 + alphabet)
    n = 1000 if Lw <= 512 else 700
    X = library(rng, n, Lw, alphabet=alphabet, max_mut=min(6, Lw))
    tab = eng.pack(X)
    assert tab.planes == (8 if alphabet > 31 else 5)
    assert tab.words == eng.packed_words(Lw)
    D = O.hamming(X, X)
    S = O._similarity(D)
    for k, drop in ((9, 1), (12, 0)):
        check_knn(eng.hamming_knn(tab, 0, n, tab, k, drop=drop), D, k, drop)
        check_knn(eng.hamming_knn(tab, 0, n, tab, k, drop=drop, similarity=True), S, k, drop, descending=True)
    # le: range test, sparse; ne: LUT test, dense (every row overflows the default 128-hit capture)
    for comp, eps in ((operator.le, 3), (operator.ne, 2)):
        lut = distance_lut(tab.words * 32, comp, eps, False)
        for capture in (None, n):
            check_csr(eng.hamming_eps(tab, 0, n, tab, lut, capture=capture), D, hamming_eps_keep(D, comp, eps))
    e = 1 / (1 + 3)
    lut = distance_lut(tab.words * 32, operator.le, e, True)
    check_csr(eng.hamming_eps(tab, 0, n, tab, lut, similarity=True), S, (np.float32(e) <= S) & (S < 1))
    same(eng.hamming_flags(tab, tab, n, 1, 3), ((D >= 1) & (D <= 3)).astype(np.uint8))
    # queries: another table (700 rows near the library), rows [37, 537) against all n rows
    Q = X[rng.permutation(n)[:700]].copy()
    Q[::3, rng.integers(0, Lw)] = alphabet
    tq = eng.pack(Q, planes=tab.planes, words=tab.words)
    Dq = O.hamming(X, Q)[37:537]
    check_knn(eng.hamming_knn(tq, 37, 500, tab, 5, drop=0), Dq, 5, 0)
    lut = distance_lut(tab.words * 32, operator.le, 2, False)
    check_csr(eng.hamming_eps(tq, 37, 500, tab, lut), Dq, hamming_eps_keep(Dq, operator.le, 2))


@pytest.mark.parametrize("Lw,alphabet", [(20, 4), (100, 200), (256, 4)])
def test_sweep_list_length_boundaries(eng, Lw, alphabet):
    """k1 = k + drop across the insertion rounds of knn_insert_coop (32 | 33, 64 | 65, 78) and the
    merge kernel's switch to 32-row blocks (k = 32 | 33); k1 = 79 does not fit the shared-memory
    lists and raises Unsupported.  Uniform tokens from a small alphabet: every list ends in a tie."""
    rng = np.random.default_rng(Lw + alphabet)
    n = 1500
    X = rng.integers(1, alphabet + 1, size=(n, Lw)).astype(np.int64)
    X[50::50] = X[49:-1:50]
    tab = eng.pack(X)
    D = O.hamming(X, X)
    for k1 in (32, 33, 64, 65, 78):
        for drop in (0, 1):
            check_knn(eng.hamming_knn(tab, 0, n, tab, k1 - drop, drop=drop), D, k1 - drop, drop)
    check_knn(eng.hamming_knn(tab, 0, n, tab, 77, drop=1, similarity=True), O._similarity(D), 77, 1, descending=True)
    with pytest.raises(unsupported()):
        eng.hamming_knn(tab, 0, n, tab, 78, drop=1)
    with pytest.raises(unsupported()):
        eng.hamming_knn(tab, 0, n, tab, 79, drop=0)


def test_sweep_list_boundary_public_build_graph():
    """build_graph(k=77) runs in the fused sweep (k1 = 78), build_graph(k=78) falls back to the
    tiles; both are the reference's graph."""
    from prograph_b200 import build_neighbours
    rng = np.random.default_rng(78)
    X = rng.integers(1, 5, size=(1100, 20)).astype(np.int64)
    for k in (77, 78):
        got = build_neighbours(X, k=k).to_csr()
        for g, r in zip((got.indptr, got.idx, got.w), O.to_csr(O.build_graph(X, k=k))):
            same(g, r)


def tile_count(n, words):
    """Ring tiles of a stream of n rows: 512 / words rows per tile, 32 for long rows."""
    return -(-n // (512 // words if words <= 16 else 32))


@pytest.mark.parametrize("splits", ["2", "3", "tiles"])
@pytest.mark.parametrize("Lw", [256, 1200])
def test_sweep_forced_splits(eng, monkeypatch, Lw, splits):
    """PG_SWEEP_SPLITS: the stream cut into 2, 3 or one split per tile.  kNN merges the split lists
    (k1 <= 32 and > 32); the epsilon fill starts every split at its prefix, and the rows whose
    capture overflowed in some split (here: rows near the wild type, more than 128 hits in a split)
    get the second sweep over the overflow rows while the others are copied from the captures."""
    from prograph_b200.graph import distance_lut
    rng = np.random.default_rng(Lw + len(splits))
    n = 1000
    X = library(rng, n, Lw, max_mut=4)
    tab = eng.pack(X)
    monkeypatch.setenv("PG_SWEEP_SPLITS", str(tile_count(n, tab.words)) if splits == "tiles" else splits)
    D = O.hamming(X, X)
    for k, drop in ((16, 1), (40, 1), (33, 0)):
        check_knn(eng.hamming_knn(tab, 0, n, tab, k, drop=drop), D, k, drop)
    check_knn(eng.hamming_knn(tab, 0, n, tab, 40, drop=1, similarity=True), O._similarity(D), 40, 1, descending=True)
    keep = hamming_eps_keep(D, operator.le, 3)
    deg = keep.sum(1)
    assert deg.max() > 3 * 128 and deg.min() < 128     # some rows overflow a split's capture, some do not
    for comp, eps in ((operator.le, 3), (operator.ne, 4)):
        lut = distance_lut(tab.words * 32, comp, eps, False)
        check_csr(eng.hamming_eps(tab, 0, n, tab, lut), D, hamming_eps_keep(D, comp, eps))
    lut = distance_lut(tab.words * 32, operator.le, 0.25, True)
    S = O._similarity(D)
    check_csr(eng.hamming_eps(tab, 0, n, tab, lut, similarity=True), S, (np.float32(0.25) <= S) & (S < 1))


@pytest.mark.parametrize("Lw", [20, 256, 1500])
def test_sweep_stream_edges(eng, Lw):
    """Stream tables of 1 row, one tile minus / exactly / plus one row (512 / words rows; 32 for
    long rows) and k1 - 1 rows: when stream_rows < k + drop the tail is index -1 with weight 0
    (0.0 in similarity mode), never one of the zero pad rows that fill the last ring tile."""
    from prograph_b200.graph import distance_lut
    rng = np.random.default_rng(Lw)
    n = 1000
    X = library(rng, n, Lw)
    tab = eng.pack(X)
    words = tab.words
    tile = 512 // words if words <= 16 else 32
    k, drop = 20, 1
    for s in sorted({1, tile - 1, tile, tile + 1, k + drop - 1}):
        st = eng.pack(X[300:300 + s], planes=tab.planes, words=words)
        D = O.hamming(X[300:300 + s], X)
        check_knn(eng.hamming_knn(tab, 0, n, st, k, drop=drop), D, k, drop)
        check_knn(eng.hamming_knn(tab, 0, n, st, k, drop=drop, similarity=True), O._similarity(D), k, drop,
                  descending=True)
        lut = distance_lut(words * 32, operator.le, 3, False)
        check_csr(eng.hamming_eps(tab, 0, n, st, lut), D, hamming_eps_keep(D, operator.le, 3))
        same(eng.hamming_flags(st, tab, n, 0, 2), (D <= 2).astype(np.uint8))


# ------------------------------------------------------------------ tcgen05 Minkowski p=2
def mink(X, Y, kind, chunk=32):
    """Oracle Minkowski p=2 matrix of queries Y against dataset X, (M, N): the fp16 chain of the
    fp16-staged representation (value_kind 0, prograph.py:726) or int64 tokens with a float32 root
    (value_kind 1)."""
    dt = np.float16 if kind == 0 else np.int64
    Xs, Ys = X.astype(dt), Y.astype(dt)
    return np.concatenate([O.minkowski(Xs, Ys[m:m + chunk]) for m in range(0, len(Ys), chunk)])


def sq_sums(X, Y):
    """Exact integer S = sum (x - y)^2 of queries Y against dataset X, (M, N): the quantity the
    epsilon edge test of the GEMM is defined on."""
    X, Y = X.astype(np.int64), Y.astype(np.int64)
    return (X * X).sum(1)[None, :] + (Y * Y).sum(1)[:, None] - 2 * (Y @ X.T)


def gemm_tables(eng, X, Q, kind):
    tx = eng.gemm_pack(X, max_token=31 if kind == 0 else 255)
    return tx, eng.gemm_pack(Q, max_token=tx.max_token, K=tx.K)


def check_gemm_knn(eng, tx, tq, D, kind, k, drop):
    for sim, M in ((False, D), (True, O._similarity(D))):
        check_knn(eng.minkowski2_gemm_knn(tx, tq, k, drop, kind, similarity=sim), M, k, drop, descending=sim)


def check_gemm_eps(eng, tx, tq, D, S, kind, lo, hi):
    keep = (S >= lo) & (S <= hi)
    for sim, M in ((False, D), (True, O._similarity(D))):
        check_csr(eng.minkowski2_gemm_eps(tx, tq, lo, hi, kind, similarity=sim), M, keep)


def check_gemm_tile(eng, tx, tq, D, kind):
    for sim, M in ((False, D), (True, O._similarity(D))):
        same(eng.minkowski2_gemm_tile(tx, tq, kind, similarity=sim), M)


# largest k + drop whose lists fit next to a 2-stage ring (gemm_smem_bytes <= 227 KB):
# 68 needs the third insertion round, 63 and 36 the second, 31 the first
GEMM_MAX_K1 = {32: 68, 64: 63, 224: 36, 256: 31}


@pytest.mark.parametrize("K", sorted(GEMM_MAX_K1))
def test_gemm_list_length_boundaries(eng, K):
    """k1 in {4 | 5 (issuer switch), 33, the largest k1 that fits} against the oracle's stable sort;
    one more raises Unsupported.  The boundary is found by calling."""
    rng = np.random.default_rng(K)
    n = 700
    X = library(rng, n, K - 5, alphabet=6, max_mut=5)
    tabs = {kind: eng.gemm_pack(X, max_token=31 if kind == 0 else 255) for kind in (0, 1)}
    assert tabs[0].K == K

    def fits(k1):
        try:
            eng.minkowski2_gemm_knn(tabs[0], tabs[0], k1, 0, 0)
            return True
        except unsupported():
            return False

    top = next(k1 for k1 in range(96, 0, -1) if fits(k1))
    assert top == GEMM_MAX_K1[K]
    with pytest.raises(unsupported()):
        eng.minkowski2_gemm_knn(tabs[1], tabs[1], top, 1, 1)
    for kind in (0, 1):
        D = mink(X, X, kind)
        for k1 in sorted({4, 5, 33, top}):
            if k1 <= top:
                check_gemm_knn(eng, tabs[kind], tabs[kind], D, kind, k1 - 1, 1)
        check_gemm_knn(eng, tabs[kind], tabs[kind], D, kind, top, 0)


@pytest.mark.parametrize("K", [32, 256])
def test_gemm_list_boundary_public_build_graph(eng, K):
    """build_graph(distance=minkowski) one below and at the largest k that fits the fused lists
    (the second call falls back to the tiles), against the reference's graph."""
    from prograph_b200 import build_neighbours, minkowski
    rng = np.random.default_rng(K + 1)
    X = library(rng, 600, K - 5, alphabet=6, max_mut=5)
    top = GEMM_MAX_K1[K]
    for k in (top - 1, top):
        got = build_neighbours(X, k=k, distance=minkowski).to_csr()
        for g, r in zip((got.indptr, got.idx, got.w), O.to_csr(O.build_graph(X, k=k, distance=O.minkowski))):
            same(g, r)


@pytest.mark.parametrize("M", [1, 127, 128, 129, 255, 256, 257])
def test_gemm_row_and_column_edges(eng, M):
    """Query rows around the two 128-row A tiles of a CTA (M <= 128: the second tile is all padding)
    against datasets of 1, 127, 128, 129 and 700 rows: tiles of both value kinds (odd N takes the
    scalar store path), kNN at k1 = 4 (two issuers) and 5 (one; N = 1 leaves a -1 tail) and the
    epsilon graph."""
    rng = np.random.default_rng(M)
    pool = library(rng, 1000, 59, alphabet=20, max_mut=4)
    Q = pool[-M:]
    for N in (1, 127, 128, 129, 700):
        X = pool[:N]
        S = sq_sums(X, Q)
        for kind in (0, 1):
            tx, tq = gemm_tables(eng, X, Q, kind)
            D = mink(X, Q, kind)
            check_gemm_tile(eng, tx, tq, D, kind)
            check_gemm_knn(eng, tx, tq, D, kind, 3, 1)
            check_gemm_knn(eng, tx, tq, D, kind, 5, 0)
            check_gemm_eps(eng, tx, tq, D, S, kind, 1, 400)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("Lw", [K - 5 for K in range(32, 257, 32)])
def test_gemm_every_width(eng, Lw, kind):
    """kNN and epsilon graphs at every K from 32 to 256 (instruction and shared-memory descriptors
    depend on K).  value_kind 1 draws its tokens from 0..255 (unsigned int8 operands)."""
    rng = np.random.default_rng(Lw * 2 + kind)
    n = 600
    if kind == 0:
        X = library(rng, n, Lw, alphabet=20)
    else:
        X = library(rng, n, Lw, alphabet=256) - 1
        X[5, :4], X[6, :4] = 255, 0
    tx, _ = gemm_tables(eng, X, X, kind)
    assert tx.K == Lw + 5
    D = mink(X, X, kind)
    check_gemm_knn(eng, tx, tx, D, kind, 10, 1)
    hi = 3 * 361 if kind == 0 else 3 * 255 * 255
    check_gemm_eps(eng, tx, tx, D, sq_sums(X, X), kind, 1, hi)


@pytest.mark.parametrize("issuers", ["1", "2"])
def test_gemm_forced_issuers(eng, monkeypatch, issuers):
    """PG_GEMM_ISSUERS forces one or two MMA-issuing warps at short (k1 = 4, 5) and long (33) lists,
    and for the tile and epsilon modes."""
    monkeypatch.setenv("PG_GEMM_ISSUERS", issuers)
    rng = np.random.default_rng(int(issuers))
    X = library(rng, 900, 120, alphabet=20)
    S = sq_sums(X, X)
    for kind in (0, 1):
        tx, _ = gemm_tables(eng, X, X, kind)
        D = mink(X, X, kind)
        for k1 in (4, 5, 33):
            check_gemm_knn(eng, tx, tx, D, kind, k1 - 1, 1)
        check_gemm_tile(eng, tx, tx, D, kind)
        check_gemm_eps(eng, tx, tx, D, S, kind, 1, 700)


def test_gemm_tile_split_dataset_odd_rows(eng):
    """200 queries x 4 097 rows: the tile kernel splits the dataset across gridDim.y (few query
    rows) and the odd row length makes every store take the scalar path; both value kinds."""
    rng = np.random.default_rng(4097)
    X = library(rng, 4097, 91, alphabet=20)
    Q = library(rng, 200, 91, alphabet=20)
    for kind in (0, 1):
        tx, tq = gemm_tables(eng, X, Q, kind)
        check_gemm_tile(eng, tx, tq, mink(X, Q, kind), kind)


def test_gemm_fp16_overflow_ties(eng):
    """Tokens in {0, 31} at K = 128: S = 961 x (positions that differ) spans 64 387 .. 69 192, so the
    fp16 chain gives finite values up to S = 65 348 and inf from S = 66 309 on.  kNN lists then run
    into ties at inf (similarity: at 0), which order by index like torch's stable sort."""
    from prograph_b200.graph import minkowski_s_range
    rng = np.random.default_rng(31)
    Lw, n = 123, 600
    base = rng.choice([0, 31], size=Lw)
    flips = rng.choice([67, 68, 69, 70, 72], size=n, p=[0.03, 0.04, 0.5, 0.33, 0.1])
    X = np.tile(base, (n, 1))
    for i in range(n):
        pos = rng.choice(Lw, size=flips[i], replace=False)
        X[i, pos] = 31 - X[i, pos]
    Q = np.concatenate([base[None, :], X[:40]])
    tx, tq = gemm_tables(eng, X, Q, 0)
    D = mink(X, Q, 0)
    assert np.isinf(D).any() and (np.isfinite(D) & (D > 250)).any()
    check_gemm_tile(eng, tx, tq, D, 0)
    check_gemm_knn(eng, tx, tq, D, 0, 50, 0)
    check_gemm_knn(eng, tx, tq, D, 0, 49, 1)
    lo, hi = minkowski_s_range(tx.K * 31 * 31, operator.le, 256.0, False)
    assert hi == 65519                                  # the last S whose fp16 chain stays finite
    check_gemm_eps(eng, tx, tq, D, sq_sums(X, Q), 0, lo, hi)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("N", [1, 3, 8])
def test_gemm_knn_short_dataset_has_empty_tail(eng, N, kind):
    """N < k + drop: the pad columns of the last B tile are not dataset rows; the missing list
    positions are index -1 with value 0, as in the Hamming sweep."""
    rng = np.random.default_rng(N)
    pool = library(rng, 400, 40, alphabet=20)
    X, Q = pool[:N], pool[N:]
    tx, tq = gemm_tables(eng, X, Q, kind)
    D = mink(X, Q, kind)
    check_gemm_knn(eng, tx, tq, D, kind, 8, 1)
    check_gemm_knn(eng, tx, tq, D, kind, 12, 0)
