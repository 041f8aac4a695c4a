"""The chunked mode of the long-row Hamming sweep (pg_sweep_long.cuh, pg_sweep_wide.cu): rows of more
than 1792 residues at 5 bit planes and more than 256 at 8, up to 32768.

A ring stage carries one 32-word chunk (1024 residues) of 32 stream rows; the accumulators stay in
registers across the chunks of a tile and the epilogues run after the last chunk.  Every case compares
bit for bit with oracle/prograph_oracle.py: kNN lists with a stable sort, CSR graphs with the oracle's
edge test, tiles with the matrix.  Inputs are seeded and tie-heavy: mutational libraries with
duplicated rows, small alphabets, and rows that differ everywhere.

Code path -> test:
  chunk loop, every last-chunk width (8, 16, 24, 32 words), 1 / many chunks   test_chunk_widths
  kNN drop 0 / 1 x int64 / similarity weights, own rows of another table       test_knn_epilogue
  count / fill with a range and LUT predicates over more than 64 words,
    default capture (overflow fill sweep) and a capture that holds every hit   test_eps_long_truth_tables
  flags tile, tile as int64 / float32 similarity / int32                       test_tile_epilogues
  k + drop = 77, 78 work, 79 raises, narrowest / widest width of both P        test_knn_list_limit
  build_neighbours(k = 77 / 78): fused lists / tile fallback, same graph       test_build_knn_list_limit
  PG_SWEEP_SPLITS = 2, 3: split merge, fill prefix, overflow-row fill          test_splits
  stream tables of 1, 31, 32, 33, k1 - 1 rows: pad rows, -1 / 0 tails          test_stream_edges
  d = 32768 in kNN keys, int32 tiles and eps ranges                            test_value_range
  L = 32769: Unsupported, public calls take the element-wise path              test_width_limit
  distance census / column census / column compaction beyond 48 KB of
    shared memory (Prograph construction, informative tables of long rows)    test_long_row_helpers_*
  public API with the element-wise kernel patched to raise                     test_public_*
"""
import operator

import numpy as np
import pytest
import torch

from oracle import prograph_oracle as O

pytestmark = pytest.mark.gpu

ALPHABET = {5: 20, 8: 40}       # 8 planes: alphabets of 32..255 tokens


@pytest.fixture(scope="module")
def eng():
    from prograph_b200.engine import get_engine
    return get_engine()


def L_():
    from prograph_b200 import _lib
    return _lib


def np_(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def same(got, want):
    got, want = np_(got), np_(want)
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    np.testing.assert_array_equal(got, want)


def library(rng, n, L, alphabet=20, max_mut=40, dup_every=29, random_every=0):
    """Mutational library: a random wild type, 1..max_mut substitutions per row, every dup_every-th
    row a copy of the row before it, every random_every-th row uniform random (distances near L)."""
    wt = rng.integers(1, alphabet + 1, size=L)
    X = np.tile(wt, (n, 1))
    for i in range(1, n):
        pos = rng.choice(L, size=min(int(rng.integers(1, max_mut + 1)), L), replace=False)
        X[i, pos] = (X[i, pos] - 1 + rng.integers(1, alphabet, size=len(pos))) % alphabet + 1
    if random_every:
        X[::random_every] = rng.integers(1, alphabet + 1, size=X[::random_every].shape)
    for i in range(dup_every, n, dup_every):
        X[i] = X[i - 1]
    return X.astype(np.int64)


def ref(X, Q):
    """The oracle's (len(Q), len(X)) Hamming matrix, in query chunks of bounded memory."""
    return O.hamming(X, Q, chunk=max(1, (1 << 27) // (len(X) * X.shape[1])))


def knn_ref(D, k, drop, descending=False):
    order = np.argsort(-D if descending else D, axis=1, kind="stable")[:, drop:drop + k]
    idx = np.full((D.shape[0], k), -1, dtype=np.int64)
    w = np.zeros((D.shape[0], k), dtype=D.dtype)
    idx[:, :order.shape[1]] = order
    w[:, :order.shape[1]] = np.take_along_axis(D, order, axis=1)
    return idx, w


def csr_ref(D, keep, w=None):
    rows, cols = np.nonzero(keep)
    indptr = np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64)
    return indptr, cols.astype(np.int64), (D if w is None else w)[rows, cols]


def sim32(D):
    return np.float32(1) / (np.float32(1) + D.astype(np.float32))


def pack(eng, X, Q, planes):
    tx = eng.pack(X, planes=planes)
    return tx, eng.pack(Q, planes=planes, words=tx.words)


def lut(words, comp, eps, guard=True):
    from prograph_b200.graph import distance_lut
    return distance_lut(words * 32, comp, eps, similarity=False, guard=guard)


def check_eps(eng, tx, tq, D, comp, eps, capture=None, guard=True):
    """eng.hamming_eps of the rows of tq against tx vs comp(D, eps) (& D > 0 with the guard)."""
    keep = np.asarray(comp(torch.as_tensor(D), eps)) & ((D > 0) if guard else True)
    indptr, idx, w = eng.hamming_eps(tq, 0, tq.rows, tx, lut(tx.words, comp, eps, guard), capture=capture)
    for g, r in zip((indptr, idx, w), csr_ref(D, keep)):
        same(g, r)
    return int(keep.sum())


WIDTHS = [(5, 2048, 64), (5, 2049, 72), (5, 2500, 80), (5, 2800, 88), (5, 32768, 1024),
          (8, 512, 16), (8, 768, 24), (8, 1024, 32), (8, 1280, 40), (8, 4096, 128)]


@pytest.mark.parametrize("planes,L,words", WIDTHS)
def test_chunk_widths(eng, planes, L, words):
    rng = np.random.default_rng(L + planes)
    n = 120 if L > 8192 else 300
    X = library(rng, n, L, alphabet=ALPHABET[planes], max_mut=60)
    tx = eng.pack(X, planes=planes)
    assert (tx.planes, tx.words) == (planes, words)
    D = ref(X, X)
    same(eng.hamming_tile(tx, tx), D)
    ri, rw = knn_ref(D, 9, 1)
    idx, w = eng.hamming_knn(tx, 0, n, tx, 9, drop=1)
    same(idx, ri)
    same(w, rw)
    check_eps(eng, tx, tx, D, operator.le, 40)


@pytest.mark.parametrize("planes,L", [(5, 2049), (8, 1280)])
def test_knn_epilogue(eng, planes, L):
    """drop 0 / 1 with int64 and similarity weights; own rows [37, 37 + 150) of a query table."""
    rng = np.random.default_rng(7 * L)
    X = library(rng, 260, L, alphabet=ALPHABET[planes])
    Q = library(rng, 200, L, alphabet=ALPHABET[planes])
    Q[40:45] = X[3:8]
    tx, tq = pack(eng, X, Q, planes)
    D = ref(X, Q[37:187])
    for drop in (0, 1):
        for sim in (False, True):
            idx, w = eng.hamming_knn(tq, 37, 150, tx, 12, drop=drop, similarity=sim)
            ri, rw = knn_ref(D, 12, drop)
            same(idx, ri)
            same(w, sim32(rw) if sim else rw)


@pytest.mark.parametrize("planes,L", [(5, 2500), (8, 2500)])
def test_eps_long_truth_tables(eng, planes, L):
    """Truth tables of 79 words (d up to 2500 > 2047): a range (le / ge), the non-contiguous ne and a
    user comparison (device copy of the table), with the default capture of 128 hits per (split, row)
    -- dense predicates overflow it -- and with a capture that holds every hit."""
    rng = np.random.default_rng(L * planes)
    X = library(rng, 280, L, alphabet=ALPHABET[planes], max_mut=30, random_every=3)
    tx = eng.pack(X, planes=planes)
    assert tx.words + 1 > 64
    D = ref(X, X)
    d_far = int(np.median(D[D > 1000]))
    preds = [(operator.le, 20), (operator.ge, d_far), (operator.ne, d_far),
             (lambda d, e: (d % e == 0) | (d > 2400), 3)]
    for comp, eps in preds:
        hits = check_eps(eng, tx, tx, D, comp, eps)
        check_eps(eng, tx, tx, D, comp, eps, capture=len(X))
        assert hits > 0
    # without the d > 0 guard (count_within / calc_neighbours semantics)
    counts = eng.hamming_eps_degrees(tx, 0, tx.rows, tx, lut(tx.words, operator.ne, d_far, guard=False))
    same(counts, (D != d_far).sum(axis=1).astype(np.int64))


@pytest.mark.parametrize("planes,L", [(5, 3000), (8, 700)])
def test_tile_epilogues(eng, planes, L):
    lib = L_()
    rng = np.random.default_rng(L)
    X = library(rng, 333, L, alphabet=ALPHABET[planes], random_every=5)
    Q = library(rng, 70, L, alphabet=ALPHABET[planes], random_every=5)
    tx, tq = pack(eng, X, Q, planes)
    D = ref(X, Q)
    same(eng.hamming_tile(tx, tq), D)
    same(eng.hamming_tile(tx, tq, weight=lib.W_I32), D.astype(np.int32))
    same(eng.hamming_tile(tx, tq, weight=lib.W_SIM_F32), sim32(D))
    for lo, hi in ((0, 30), (1, 1), (L // 2, L), (5, 4)):
        same(eng.hamming_flags(tx, tq, len(Q), lo, hi), ((D >= lo) & (D <= hi)).astype(np.uint8))


@pytest.mark.parametrize("planes,L", [(5, 2048), (5, 32768), (8, 512), (8, 32768)])
def test_knn_list_limit(eng, planes, L):
    rng = np.random.default_rng(L + 78)
    n = 100 if L > 8192 else 200
    X = library(rng, n, L, alphabet=ALPHABET[planes], max_mut=20)
    tx = eng.pack(X, planes=planes)
    D = ref(X, X)
    for k, drop in ((76, 1), (77, 1), (78, 0)):
        idx, w = eng.hamming_knn(tx, 0, n, tx, k, drop=drop)
        ri, rw = knn_ref(D, k, drop)
        same(idx, ri)
        same(w, rw)
    for k, drop in ((78, 1), (79, 0)):
        with pytest.raises(L_().Unsupported):
            eng.hamming_knn(tx, 0, n, tx, k, drop=drop)


def record(monkeypatch, eng, name, seen):
    real = getattr(eng, name)

    def wrapped(*a, **k):
        t = a[0]
        seen.append((name, t.planes, t.words))
        return real(*a, **k)
    monkeypatch.setattr(eng, name, wrapped)


@pytest.mark.parametrize("planes,L,words", [(5, 2100, 72), (8, 600, 24)])
def test_build_knn_list_limit(eng, monkeypatch, planes, L, words):
    """build_neighbours(k=77): k + drop = 78 on the fused sweep; k=78 is one entry too many and takes
    the tile top-k; both give the reference's graph."""
    from prograph_b200 import build_neighbours
    rng = np.random.default_rng(words)
    X = library(rng, 180, L, alphabet=ALPHABET[planes], max_mut=20)
    if planes == 8:
        X[0, 0] = 40                     # tokens beyond 31: 8 planes
    D = ref(X, X)
    seen = []
    record(monkeypatch, eng, "hamming_knn", seen)
    for k in (77, 78):
        got = build_neighbours(X, k=k)
        ri, rw = knn_ref(D, k, 1)
        same(got.idx, ri)
        same(got.w, rw)
    assert seen and all(s == ("hamming_knn", planes, words) for s in seen), seen


@pytest.mark.parametrize("splits", ["2", "3"])
@pytest.mark.parametrize("planes,L", [(5, 2049), (8, 1280)])
def test_splits(eng, monkeypatch, planes, L, splits):
    monkeypatch.setenv("PG_SWEEP_SPLITS", splits)
    rng = np.random.default_rng(int(splits) * L)
    X = library(rng, 400, L, alphabet=ALPHABET[planes], max_mut=20)
    tx = eng.pack(X, planes=planes)
    D = ref(X, X)
    for k, drop in ((9, 1), (40, 0)):
        idx, w = eng.hamming_knn(tx, 0, len(X), tx, k, drop=drop)
        ri, rw = knn_ref(D, k, drop)
        same(idx, ri)
        same(w, rw)
    check_eps(eng, tx, tx, D, operator.le, 30)          # sparse: every row from its captures
    check_eps(eng, tx, tx, D, operator.ne, 17)          # dense: overflow rows take the fill sweep
    check_eps(eng, tx, tx, D, operator.ne, 17, capture=len(X))


@pytest.mark.parametrize("planes,L", [(5, 2049), (8, 1000)])
def test_stream_edges(eng, planes, L):
    rng = np.random.default_rng(L - planes)
    X = library(rng, 300, L, alphabet=ALPHABET[planes], max_mut=20)
    tx = eng.pack(X, planes=planes)
    k, drop = 8, 1
    for s in (1, 31, 32, 33, k + drop - 1):
        ts = eng.pack(X[:s], planes=planes, words=tx.words)
        D = ref(X[:s], X)
        idx, w = eng.hamming_knn(tx, 0, len(X), ts, k, drop=drop)
        ri, rw = knn_ref(D, k, drop)
        same(idx, ri)
        same(w, rw)
        check_eps(eng, ts, tx, D, operator.le, 25)
        same(eng.hamming_tile(tx, ts), D.T)


def test_value_range(eng):
    """Rows of 32768 residues that differ everywhere: d = 32768 in kNN keys, int32 tiles, eps ranges."""
    lib = L_()
    L = 32768
    X = np.repeat(np.arange(1, 21, dtype=np.int64)[:, None], L, axis=1)      # row i = all token i + 1
    X = np.concatenate([X, X])                                                # duplicates: d = 0
    X[5, :100] = 1                                                            # d(5, 0) = L - 100
    Xp = X
    for planes in (5, 8):
        tx = eng.pack(Xp, planes=planes)
        assert tx.words == 1024
        D = ref(Xp, Xp)
        assert D.max() == L
        idx, w = eng.hamming_knn(tx, 0, len(Xp), tx, 30, drop=0)
        ri, rw = knn_ref(D, 30, 0)
        same(idx, ri)
        same(w, rw)
        same(eng.hamming_tile(tx, tx, weight=lib.W_I32), D.astype(np.int32))
        for comp, eps in ((operator.ge, L), (operator.eq, L), (operator.gt, L - 101), (operator.ne, L),
                          (lambda d, e: (d == e) | (d == e - 100), L)):       # bits 32668 and 32768 of 1025 words
            check_eps(eng, tx, tx, D, comp, eps)
        same(eng.hamming_flags(tx, tx, len(Xp), L, L), (D == L).astype(np.uint8))


def test_width_limit(eng, tmp_path):
    """32769 residues: the sweep raises Unsupported; hamming, build_neighbours, query.* and
    Prograph.nearest_neighbour answer through the element-wise kernel."""
    from prograph_b200 import build_neighbours, hamming, query
    rng = np.random.default_rng(32769)
    L = 32769
    X = library(rng, 60, L, alphabet=20, max_mut=30)
    Q = X[[3, 10, 11, 50]].copy()
    Q[1, :7] = 4
    tx = eng.pack(X)
    assert tx.words == 1032
    with pytest.raises(L_().Unsupported):
        eng.hamming_knn(tx, 0, tx.rows, tx, 3, drop=1)
    D = ref(X, X)
    DQ = ref(X, Q)
    same(hamming(X, Q), DQ)
    got = build_neighbours(X, k=5)
    ri, rw = knn_ref(D, 5, 1)
    same(got.idx, ri)
    same(got.w, rw)
    got = build_neighbours(X, eps=25)
    for g, r in zip((got.indptr, got.idx, got.w), csr_ref(D, (D <= 25) & (D > 0))):
        same(g, r)
    lib = query.Library(X)
    mi, mv = query.nearest(lib, Q)
    same(mi, DQ.argmin(axis=1))
    same(mv, DQ.min(axis=1))
    same(query.count_within(lib, Q, 20), (DQ <= 20).sum(axis=1).astype(np.int64))
    same(query.tile(lib, Q), DQ)
    pg = prograph_from(tmp_path, X, O.AMINO_ACIDS)
    rows, dmin = pg.nearest_neighbour(list(pg.graph["Sequence"].iloc[[3, 10, 11, 50]]))
    ni, nd = O.nearest_neighbour(pg.tokenized, pg.tokenized[[3, 10, 11, 50]])
    same(np.asarray(rows.index), np.asarray(pg.graph.index[ni]))
    assert dmin == nd == 0


@pytest.mark.parametrize("words", [384, 392, 1024, 1032, 2048])
def test_long_row_helpers_distance_hist(eng, words):
    """Distance census of mutation masks (Prograph.__str__): 32 * words + 1 bins in shared memory up to
    227 KB (more than the default 48 KB above 384 words), counted in global memory beyond (2048 words)."""
    g = torch.Generator(device=eng.device).manual_seed(words)
    mut = torch.randint(-(1 << 31), 1 << 31, (700, words), generator=g, device=eng.device, dtype=torch.int64)
    mut = mut.to(torch.int32)
    keep = torch.rand((700, words), generator=g, device=eng.device) < 0.3
    mut = torch.where(keep, mut, torch.zeros_like(mut))
    mut[:5] = 0
    mut[5] = -1                                                  # d = 32 * words
    d = np.unpackbits(np.ascontiguousarray(mut.cpu().numpy()).view(np.uint8), axis=1).sum(axis=1)
    same(eng.distance_hist(mut), np.bincount(d, minlength=32 * words + 1).astype(np.int64))


def test_long_row_helpers_columns(eng):
    """Column census and compaction of long rows: a 4096-row library of 32768 residues whose 20000
    varying positions compact to 632 words (an 80 KB column map), and the census of 8-plane rows of
    65536 residues (a 64 KB accumulator)."""
    rng = np.random.default_rng(632)
    n, L = 4096, 32768
    X = np.tile(rng.integers(1, 21, size=L, dtype=np.uint8), (n, 1))
    cols = np.sort(rng.choice(L, size=20000, replace=False))
    X[:, cols] = rng.integers(1, 21, size=(n, len(cols)), dtype=np.uint8)
    X[1:, cols[0]] = X[0, cols[0]] % 20 + 1                      # varies in row 0 only
    tx = eng.pack(X, planes=5)
    same(eng.varying_columns(tx), cols.astype(np.int32))
    small = eng.compact_columns(tx, cols)
    assert small.words == 632
    same(small.data, eng.pack(X[:, cols], planes=5, words=632).data)
    Y = rng.integers(1, 41, size=(64, 65536), dtype=np.uint8)
    Y[:, ::3] = Y[0, ::3]
    ty = eng.pack(Y, planes=8)
    assert ty.words == 2048
    same(eng.varying_columns(ty), np.nonzero((Y != Y[0]).any(axis=0))[0].astype(np.int32))


# ---- public API, fused path proven: the element-wise Hamming kernel raises ------------------

@pytest.fixture
def no_elem(eng, monkeypatch):
    def boom(*a, **k):
        raise AssertionError("element-wise Hamming kernel called")
    monkeypatch.setattr(eng, "hamming_values_tile", boom)
    return eng


def wide_library(rng, n, L, alphabet):
    """More varying positions than the older kernels cover (1792 at 5 planes, 256 at 8)."""
    return library(rng, n, L, alphabet=alphabet, max_mut=L // 4, dup_every=17)


@pytest.mark.parametrize("planes,L", [(5, 2300), (8, 900)])
def test_public_hamming_and_query(no_elem, planes, L):
    from prograph_b200 import hamming, query
    rng = np.random.default_rng(L + 1)
    X = wide_library(rng, 240, L, ALPHABET[planes])
    Q = wide_library(rng, 50, L, ALPHABET[planes])
    Q[:4] = X[20:24]
    DQ = ref(X, Q)
    same(hamming(X, Q), DQ)
    same(hamming(X, Q, similarity=True), sim32(DQ))
    lib = query.Library(X)
    assert (lib.packed().planes, lib.packed().words) == (planes, (L + 255) // 256 * 8)
    mi, mv = query.nearest(lib, Q)
    same(mi, DQ.argmin(axis=1))
    same(mv, DQ.min(axis=1))
    for comp, eps in ((operator.le, L // 2), (operator.ne, int(DQ[5, 7])), (operator.eq, 0)):
        same(query.count_within(lib, Q, eps, comp), np.asarray(comp(torch.as_tensor(DQ), eps)).sum(axis=1))
    same(query.tile(lib, Q), DQ)
    same(query.tile(lib, Q, 7, 30, similarity=True), sim32(DQ[7:37]))


@pytest.mark.parametrize("eps_sym", [None, "1"])
@pytest.mark.parametrize("planes,L", [(5, 2300), (8, 900)])
def test_public_build_neighbours(no_elem, monkeypatch, planes, L, eps_sym):
    """kNN and epsilon graphs; PG_EPS_SYM=1 sends the epsilon graph to the symmetric sweep, which does
    not take these widths, so it samples degrees and builds with count / fill."""
    from prograph_b200 import build_neighbours
    if eps_sym:
        monkeypatch.setenv("PG_EPS_SYM", eps_sym)
    rng = np.random.default_rng(L + 2)
    X = wide_library(rng, 300, L, ALPHABET[planes])
    D = ref(X, X)
    seen = []
    for name in ("hamming_knn", "hamming_eps", "hamming_eps_degrees"):
        record(monkeypatch, no_elem, name, seen)
    for k in (1, 16):
        got = build_neighbours(X, k=k)
        ri, rw = knn_ref(D, k, 1)
        same(got.idx, ri)
        same(got.w, rw)
    med = int(np.median(D))
    for comp, eps in ((operator.le, med), (operator.ne, med)):
        got = build_neighbours(X, eps=eps, comp=comp)
        want = O.to_csr(O.build_graph(X, eps=eps, comp=comp))
        for g, r in zip((got.indptr, got.idx, got.w), want):
            same(g, r)
    words = (L + 255) // 256 * 8
    assert seen and all(s[1:] == (planes, words) for s in seen), seen
    if eps_sym:
        assert any(s[0] == "hamming_eps_degrees" for s in seen)


def prograph_from(tmp_path, tok, alphabet):
    import pandas as pd
    import prograph_b200 as pgb
    aa = np.array(list(alphabet))
    seqs = ["".join(aa[t - 1]) for t in tok]
    path = tmp_path / "lib.csv"
    pd.DataFrame({"Sequence": seqs, "Fitness": np.arange(len(seqs), dtype=float)}).to_csv(path)
    return pgb.Prograph(file=str(path), amino_acids=alphabet)


@pytest.mark.parametrize("planes,L", [(5, 2300), (8, 900)])
def test_public_prograph(no_elem, monkeypatch, tmp_path, planes, L):
    """Prograph from a CSV of long sequences: the default eps=1 graph, calc_neighbours,
    nearest_neighbour and neighbourhood_clustering, all on the fused sweeps."""
    alphabet = O.AMINO_ACIDS if planes == 5 else O.AMINO_ACIDS + "abcdefghijklmnopqrst"
    rng = np.random.default_rng(L + 3)
    tok = library(rng, 200, L, alphabet=len(alphabet), max_mut=3, dup_every=13)
    tok[100:] = wide_library(rng, 100, L, len(alphabet))
    seen = []
    for name in ("hamming_eps", "hamming_knn", "hamming_flags"):
        record(monkeypatch, no_elem, name, seen)
    pg = prograph_from(tmp_path, tok, alphabet)
    assert (pg._device_tokens().planes, pg._device_tokens().words) == (planes, (L + 255) // 256 * 8)
    D = ref(tok, tok)
    want = O.build_graph(tok, eps=1)
    assert len(pg.graph["Neighbours"]) == len(want)
    for (gi, gw), (ri, rw) in zip(pg.graph["Neighbours"], want):
        same(gi, ri)
        same(np.asarray(gw, dtype=np.int64), np.asarray(rw, dtype=np.int64))
    seq = pg.graph["Sequence"].iloc[5]
    same(np.asarray(pg.calc_neighbours(seq, eps=2, comp=operator.le), dtype=np.int64),
         np.nonzero(D[5] <= 2)[0])
    queries = list(pg.graph["Sequence"].iloc[[7, 150, 199]])
    rows, dmin = pg.nearest_neighbour(queries)
    ni, nd = O.nearest_neighbour(tok, tok[[7, 150, 199]])
    same(np.asarray(rows.index), np.asarray(pg.graph.index[ni]))
    assert dmin == nd
    eps = 3
    clusters = pg.neighbourhood_clustering(eps)
    covered = np.zeros(len(tok), dtype=bool)
    want = {}
    for s in range(len(tok)):
        if not covered[s]:
            members = np.nonzero(D[s] <= eps)[0]
            want[s] = members
            covered[members] = True
    assert sorted(clusters) == sorted(want)
    for s, members in want.items():
        same(np.asarray(clusters[s].index), np.asarray(pg.graph.index[members]))
    words = (L + 255) // 256 * 8
    assert {s[0] for s in seen} >= {"hamming_eps", "hamming_knn", "hamming_flags"}
    assert all(s[1:] == (planes, words) for s in seen), seen
