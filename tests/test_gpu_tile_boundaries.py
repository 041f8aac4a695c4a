"""Boundary cases of the tile kernels and the selection masks, against the numpy oracle.

Much of the public API ends in the element-wise tiles of pg_tile.cu (Minkowski with p != 2 or wide
rows, Hamming on values, "Embedded" representations, user callables, long kNN lists) and in its two
tile consumers, the top-k and the threshold -> CSR compaction.  The selection kernels of pg_masks.cu
answer indexing / get_mutated_positions / calc_neighbours.  Every case here sits on one side of a
block, staging, dispatch or size limit of these kernels and compares with oracle/prograph_oracle.py
(the literal torch expression on CPU tensors for the threshold tests): bit for bit (fp16 as uint16)
wherever every partial sum is order independent -- integers, multiples of 1/8 in [-8, 8], sums of at
most two terms -- and within the bounds DESIGN.md states for powf exponents otherwise.  NaN positions
always agree.  Inputs are seeded and full of ties.

Code path -> test:
  elem_tile_kernel 128 x 64 blocks, 16-component staging, q0 offset   test_elem_block_and_staging_edges
  launch_elem instantiations, I64 branch, fp16 exponent cast            test_elem_exponent_dispatch
  METRIC 1 on NaN, +-0, +-inf, subnormals, int64 beyond 2^53            test_hamming_values_special
  rank-1 p = 1 path: 255 | 256, fraction / NaN / inf flag, D and qrows
    limits, row sums from q0                                            test_minkowski_p1_rank1_limits
  more than 65 535 query blocks (chunked launch)                        test_elem_beyond_65535_query_blocks
  top-k shared-memory / two-sort switch at k + drop = 4096 | 4097       test_topk_path_edges
  top-k N edges, -1 / 0 tails on both paths, ld > N                     test_topk_row_length_edges
  top-k keys of NaN, +-0, +-inf, fp16 +-65504, INT32/INT64 MIN/MAX      test_topk_special_values
  top-k sort path row_bits (rows 1 .. 1025)                             test_topk_row_counts
  threshold count / fill: dtypes x cmp x swap x guard x N, ld > N       test_threshold_grid
  eps rounding per tile dtype, int vs float eps on integer tiles        test_threshold_eps_rounding
  count_within on the fused and the tile path                          test_count_within_float_eps_fused_vs_tile
  build_graph on "Embedded" floats with a float eps                     test_build_graph_embedded_float_eps
  pg_select_rows / pg_distance_hist / pg_mutant_any / pg_flag_indices
    on 1 .. 157 mask words (by-value and buffered masks)                test_selection_masks_wide_rows
"""
import operator

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import prograph_oracle as O

pytestmark = pytest.mark.gpu

CMPS = {"lt": operator.lt, "le": operator.le, "eq": operator.eq, "ne": operator.ne, "ge": operator.ge,
        "gt": operator.gt}


@pytest.fixture(scope="module")
def eng():
    from prograph_b200.engine import get_engine
    return get_engine()


def np_(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _bits(a):
    """Float arrays as their bit patterns (NaN payloads and the sign of zero count)."""
    if a.dtype.kind == "f":
        return a.view({2: np.uint16, 4: np.uint32, 8: np.uint64}[a.itemsize])
    return a


def same(got, want):
    """Bit-exact comparison, dtypes included; NaN in the same positions (its payload is whatever
    the arithmetic that made it produces)."""
    got, want = np_(got), np.asarray(want)
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    assert got.shape == want.shape, (got.shape, want.shape)
    if got.dtype.kind == "f":
        nan = np.isnan(want)
        np.testing.assert_array_equal(np.isnan(got), nan)
        got, want = got[~nan], want[~nan]
    np.testing.assert_array_equal(_bits(got), _bits(want))


def within_ulps(got, want, ulps):
    """Equal NaN and inf positions; finite values at most `ulps` units in the last place apart."""
    got, want = np_(got), np.asarray(want)
    assert got.dtype == want.dtype and got.shape == want.shape
    gn, wn = np.isnan(got), np.isnan(want)
    np.testing.assert_array_equal(gn, wn)
    g, w = got[~wn], want[~wn]
    inf = np.isinf(g) | np.isinf(w)
    np.testing.assert_array_equal(g[inf], w[inf])
    g, w = g[~inf], w[~inf]
    it = {2: np.int16, 4: np.int32, 8: np.int64}[g.itemsize]
    mag = np.int64(np.iinfo(it).max)

    def key(a):
        b = a.view(it).astype(np.int64)
        return np.where(b < 0, -(b & mag), b)          # ordered: -0 and +0 both 0
    diff = np.abs(key(g) - key(w))
    assert diff.size == 0 or diff.max() <= ulps, f"{diff.max()} ulps apart (bound {ulps})"


def order_ref(T, descending):
    """torch.sort(stable=True) order of every row: NaN last ascending and first descending,
    -0 == +0, ties by index."""
    if T.dtype.kind == "f":
        v = T.astype(np.float64)
        nan = np.isnan(v)
        v = np.where(nan, 0.0, v)
        return np.lexsort((-v, ~nan) if descending else (v, nan), axis=-1)
    v = T.astype(np.int64)
    return np.argsort(~v if descending else v, axis=1, kind="stable")


def knn_ref(T, k, drop, descending=False, order=None):
    """Sorted positions [drop, drop+k) of every row of T; past the end of a row index -1, value 0."""
    order = order_ref(T, descending) if order is None else order
    sel = order[:, drop:drop + k]
    idx = np.full((T.shape[0], k), -1, dtype=np.int64)
    val = np.zeros((T.shape[0], k), dtype=T.dtype)
    idx[:, :sel.shape[1]] = sel
    val[:, :sel.shape[1]] = np.take_along_axis(T, sel, axis=1)
    return idx, val


def csr_ref(W, keep):
    rows, cols = np.nonzero(keep)
    return np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64), cols.astype(np.int64), W[rows, cols]


def on_device(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def wide_slice(a, extra=7):
    """`a` as the first columns of a wider device tile: ld > N."""
    rows, n = a.shape
    pad = np.zeros((rows, n + extra), dtype=a.dtype)
    pad[:, :n] = a
    return on_device(pad)[:, :n]


def eighths(rng, shape, lo=-8, hi=8):
    """Multiples of 1/8 in [lo, hi]: differences are exact in every float dtype and every term of a
    sum of squares / cubes a multiple of 1/64 / 1/512, so fp32 sums are order independent."""
    return rng.integers(lo * 8, hi * 8 + 1, size=shape) / 8.0


# ------------------------------------------------------------------ element-wise tiles
ELEM_DTYPES = {"f16": np.float16, "f32": np.float32, "f64": np.float64, "i64": np.int64}


def elem_data(rng, dt, shape):
    if dt == np.int64:
        return rng.integers(-8, 9, size=shape).astype(np.int64)
    return eighths(rng, shape).astype(dt)


@pytest.mark.parametrize("dtype", list(ELEM_DTYPES))
def test_elem_block_and_staging_edges(eng, dtype):
    """N around the 128-row dataset block, qrows around the 64-row query block, q0 = 0 / 37 and D
    around the 16-component staging chunk, with and without similarity; p = 2 (fp16: the half2
    path).  Data are multiples of 1/8 (integers for int64): bit-exact."""
    dt = ELEM_DTYPES[dtype]
    rng = np.random.default_rng(len(dtype) * 100 + dt().itemsize)
    Ns, Qs = (1, 127, 128, 129, 515), (1, 63, 64, 65, 130)
    for D in (1, 15, 16, 17, 48, 257):
        Y = elem_data(rng, dt, (37 + 130, D))
        for N in Ns:
            X = elem_data(rng, dt, (N, D))
            X[N // 2] = Y[40]                                  # a zero distance
            ref = O.minkowski(X, Y)
            ref_s = O._similarity(ref)
            Xd, Yd = on_device(X), on_device(Y)
            for i, qrows in enumerate(Qs):
                q0 = (0, 37)[(i + N) % 2]
                same(eng.minkowski_tile(Xd, Yd, q0, qrows), ref[q0:q0 + qrows])
                same(eng.minkowski_tile(Xd, Yd, q0, qrows, similarity=True), ref_s[q0:q0 + qrows])


@pytest.mark.parametrize("dtype", list(ELEM_DTYPES))
def test_elem_exponent_dispatch(eng, dtype):
    """Every instantiation launch_elem picks: (2, sqrt), (1, 1), (3, general), (sqrt, 2), general;
    for fp16 p in {1, 2, 3} is the half2 path, the others the scalar one.  p in {1, 2}: bit-exact;
    p = 3 sums exactly and is held to the powf bound (1 fp16 / 4 fp32 or fp64 ulp) through its root.
    The other exponents run on D <= 2 (order-independent sums): NaN / inf positions agree on
    differences of both signs, values are held to the powf bound where all differences are positive
    (signed terms of p = -1 cancel, and no ulp bound survives a cancelling sum).  int64 takes p in
    {1, 2, 3, 4} and refuses a non-integer or negative p; fp16 casts p = 2.0001 to 2."""
    dt = ELEM_DTYPES[dtype]
    rng = np.random.default_rng(7 + dt().itemsize)
    ulps = 1 if dt == np.float16 else 4
    ps = (1, 2, 3, 4) if dt == np.int64 else (1, 2, 3, 0.5, 1.5, 4, -1)
    for p in ps:
        general = p not in (1, 2, 3) and dt != np.int64
        for D in ((1, 2) if general else (17, 2)):
            if dt == np.int64:
                X, Y = rng.integers(-3, 4, size=(129, D)), rng.integers(-3, 4, size=(70, D))
            else:
                X, Y = eighths(rng, (129, D), -2, 2).astype(dt), eighths(rng, (70, D), -2, 2).astype(dt)
            X[5] = Y[3]
            Xd, Yd = on_device(X), on_device(Y)
            for sim in (False, True):
                got = eng.minkowski_tile(Xd, Yd, 3, 65, p=p, similarity=sim)
                want = O.minkowski(X, Y[3:68], p=p, similarity=sim)
                if p in (1, 2):
                    same(got, want)
                elif not general:
                    within_ulps(got, want, ulps)
                else:
                    got = np_(got)
                    np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
                    np.testing.assert_array_equal(np.isposinf(got), np.isposinf(want))
                    np.testing.assert_array_equal(np.isneginf(got), np.isneginf(want))
            if general:                                    # x - y in [1/8, 4]
                X = (rng.integers(1, 17, size=(129, D)) / 8).astype(dt)
                Y = (-rng.integers(0, 17, size=(70, D)) / 8).astype(dt)
                for sim in (False, True):
                    within_ulps(eng.minkowski_tile(on_device(X), on_device(Y), 3, 65, p=p, similarity=sim),
                                O.minkowski(X, Y[3:68], p=p, similarity=sim), ulps)
    if dt == np.int64:
        X = on_device(rng.integers(-3, 4, size=(9, 4)))
        for p in (1.5, 0.5, -1, -2):
            with pytest.raises(ValueError):
                eng.minkowski_tile(X, X, 0, 9, p=p)
    if dt == np.float16:
        X, Y = eighths(rng, (129, 17)).astype(dt), eighths(rng, (70, 17)).astype(dt)
        got = eng.minkowski_tile(on_device(X), on_device(Y), 0, 70, p=2.0001)
        same(got, O.minkowski(X, Y, p=2.0001))
        same(got, O.minkowski(X, Y, p=2))


SPECIAL = {
    "f16": [np.nan, 0.0, -0.0, np.inf, -np.inf, 1.5, -2.25, 2.0 ** -24, 2.0 ** -20, -(2.0 ** -24), 65504.0],
    "f32": [np.nan, 0.0, -0.0, np.inf, -np.inf, 1.5, -2.25, 1e-45, 1e-40, -1e-45, 3.4e38],
    "f64": [np.nan, 0.0, -0.0, np.inf, -np.inf, 1.5, -2.25, 5e-324, 1e-310, -5e-324, 1.7e308],
    "i64": [2 ** 53, 2 ** 53 + 1, -2 ** 63, 2 ** 63 - 1, 0, -1, 7],
}


@pytest.mark.parametrize("dtype", list(ELEM_DTYPES))
def test_hamming_values_special(eng, dtype):
    """Hamming on values (hamming.py:34, element-wise !=): NaN differs from everything including
    itself, +0 equals -0, infinities and subnormals compare as values, int64 2^53 and 2^53 + 1 are
    distinct.  int64 distances and float32 similarities, across block edges and from q0 = 3."""
    dt = ELEM_DTYPES[dtype]
    rng = np.random.default_rng(53 + dt().itemsize)
    pool = np.array(SPECIAL[dtype], dtype=dt)
    X = pool[rng.integers(0, len(pool), size=(129, 17))]
    Y = pool[rng.integers(0, len(pool), size=(70, 17))]
    Y[10] = X[20]                                          # equal rows: 0 unless a NaN is in them
    Y[11] = X[21]
    Y[11][Y[11] == 0] = -0.0 if dt != np.int64 else 0
    Xd, Yd = on_device(X), on_device(Y)
    same(eng.hamming_values_tile(Xd, Yd, 3, 65), O.hamming(X, Y[3:68]))
    same(eng.hamming_values_tile(Xd, Yd, 3, 65, similarity=True), O.hamming(X, Y[3:68], similarity=True))
    if dt == np.int64:
        a = np.array([[2 ** 53], [2 ** 53 + 1]], dtype=np.int64)
        same(eng.hamming_values_tile(on_device(a), on_device(a), 0, 2), np.array([[0, 1], [1, 0]]))


@pytest.mark.parametrize("dtype", ["f16", "f32", "i64"])
def test_minkowski_p1_rank1_limits(eng, dtype):
    """p = 1 has no abs in the reference: sum(x) - sum(y), a rank-1 tile when every value is an
    integer of magnitude <= 255 (float types) and D <= 32768, qrows <= 8 * 65535; otherwise the
    device flag hands the tile to the element-wise kernel.  Both sides of each limit, bit-exact."""
    dt = ELEM_DTYPES[dtype]
    rng = np.random.default_rng(255 + dt().itemsize)

    def check(X, Y, q0, qrows):
        Xd, Yd = on_device(X), on_device(Y)
        ref = O.minkowski(X, Y[q0:q0 + qrows], p=1)
        same(eng.minkowski_tile(Xd, Yd, q0, qrows, p=1), ref)
        same(eng.minkowski_tile(Xd, Yd, q0, qrows, p=1, similarity=True), O._similarity(ref))

    base_x = rng.integers(-255, 256, size=(130, 40)).astype(dt)
    base_y = rng.integers(-255, 256, size=(90, 40)).astype(dt)
    base_x[:, 0], base_y[:, 0] = 255, -255
    check(base_x, base_y, 0, 90)
    check(base_x, base_y, 17, 65)                          # row sums of Y from q0
    if dt != np.int64:
        for v in (256.0, 0.5, np.nan, np.inf):             # one value off the rank-1 path, in one row
            X = base_x.copy()
            X[77, 13] = v
            check(X, base_y, 17, 65)
            Y = base_y.copy()
            Y[30, 5] = v
            check(base_x, Y, 17, 65)
    else:
        X = base_x.copy()
        X[77, 13] = 1 << 40                                # int64 keeps the rank-1 identity
        check(X, base_y, 17, 65)
    for D in (32768, 32769):
        X = rng.integers(-255, 256, size=(3, D)).astype(dt)
        Y = rng.integers(-255, 256, size=(5, D)).astype(dt)
        X[:, :], Y[0] = 255, -255                          # the largest sums: exact in fp32
        check(X, Y, 1, 4)
    for qrows in (524280, 524281):
        X = rng.integers(-255, 256, size=(2, 1)).astype(dt)
        Y = rng.integers(-255, 256, size=(qrows + 3, 1)).astype(dt)
        check(X, Y, 3, qrows)


ELEM_ROWS_LIMIT = 65535 * 64


@pytest.mark.parametrize("M", [ELEM_ROWS_LIMIT, ELEM_ROWS_LIMIT + 1])
def test_elem_beyond_65535_query_blocks(M):
    """The element-wise kernel puts query blocks of 64 rows on gridDim.y (at most 65 535); taller
    tiles are launched in chunks.  Public minkowski / hamming and query.tile on N = 3, D = 2 float32
    non-integer values (no token path), compared with the oracle chunk by chunk (two terms: exact)."""
    from prograph_b200 import hamming, minkowski
    from prograph_b200.query import Library, tile
    rng = np.random.default_rng(M)
    X = (rng.integers(0, 3, size=(3, 2)) + 0.5).astype(np.float32)
    Y = (rng.integers(0, 3, size=(M, 2)) + 0.5).astype(np.float32)
    Y[-1] = X[2]
    lib = Library(X)
    outs = {
        "minkowski": (np_(minkowski(X, Y)), O.minkowski),
        "hamming": (np_(hamming(X, Y)), O.hamming),
        "tile minkowski": (np_(tile(lib, Y, distance=minkowski)), O.minkowski),
        "tile hamming": (np_(tile(lib, Y, distance=hamming)), O.hamming),
    }
    step = 1 << 20
    for name, (got, fn) in outs.items():
        assert got.shape == (M, 3), name
        for m0 in range(0, M, step):
            same(got[m0:m0 + step], fn(X, Y[m0:m0 + step]))


# ------------------------------------------------------------------ tile top-k
TOPK_DTYPES = {"f16": np.float16, "f32": np.float32, "f64": np.float64, "i32": np.int32, "i64": np.int64}


def tie_tile(rng, dt, rows, n, nan_every=0):
    """Values 0..39 (a tie every few entries); floats with -0 for some zeros and NaN every
    `nan_every`-th entry."""
    T = rng.integers(0, 40, size=(rows, n)).astype(dt)
    if dt().dtype.kind == "f":
        T[(T == 0) & (rng.random((rows, n)) < 0.5)] = -0.0
        if nan_every:
            T.reshape(-1)[rng.integers(0, nan_every):: nan_every] = np.nan
    return T


def check_topk(eng, T, k, drop, descending, order=None, dev=None):
    ri, rv = knn_ref(T, k, drop, descending, order)
    gi, gv = eng.tile_topk(wide_slice(T) if dev is None else dev, k, drop=drop, descending=descending)
    same(gi, ri)
    same(gv, rv)


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("dtype", list(TOPK_DTYPES))
def test_topk_path_edges(eng, dtype, descending):
    """k + drop around the bitonic sizes (2, 3 | 255, 256, 257) and the shared-memory / device-sort
    switch: 4096 is the last size the shared-memory sort holds (48 KiB with 8-byte keys), 4097 the
    first that takes the two radix sorts; drop in {0, 1, 5}; 3 rows of 9001 tie-heavy entries."""
    dt = TOPK_DTYPES[dtype]
    rng = np.random.default_rng(9001 + len(dtype))
    T = tie_tile(rng, dt, 3, 9001, nan_every=97)
    dev, order = wide_slice(T), order_ref(T, descending)
    for k1 in (1, 2, 3, 255, 256, 257, 4095, 4096, 4097):
        for drop in (0, 1, 5):
            if k1 - drop >= 1:
                check_topk(eng, T, k1 - drop, drop, descending, order, dev)


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("dtype", list(TOPK_DTYPES))
def test_topk_row_length_edges(eng, dtype, descending):
    """N around the 256-thread strides and the 4096 switch, from 1 to 9001.  N < k + drop leaves a
    tail of index -1 / value 0 on the shared-memory path (k1 <= 4096) and on the sort path
    (N = 5000, k = 6000)."""
    dt = TOPK_DTYPES[dtype]
    rng = np.random.default_rng(4097 + len(dtype))
    for N in (1, 2, 255, 256, 257, 4096, 4097, 5000, 9001):
        T = tie_tile(rng, dt, 2, N, nan_every=13)
        dev, order = wide_slice(T), order_ref(T, descending)
        for k, drop in ((3, 0), (256, 1), (4095, 1), (4097, 0), (6000, 1)):
            check_topk(eng, T, k, drop, descending, order, dev)


def special_tile(rng, dt, rows, n):
    """Tie-heavy rows with the extreme keys of each dtype: NaN, +-0, +-inf, +-65504 for fp16, the
    limits for integers (INT32_MAX's ascending key is the padding key ~0; INT32_MIN's descending)."""
    T = tie_tile(rng, dt, rows, n)
    if dt().dtype.kind == "f":
        specials = [np.nan, 0.0, -0.0, np.inf, -np.inf, -1.0]
        if dt == np.float16:
            specials += [65504.0, -65504.0]
        else:
            specials += [float(np.finfo(dt).max), float(-np.finfo(dt).max), float(np.finfo(dt).tiny)]
    else:
        info = np.iinfo(dt)
        specials = [info.min, info.max, info.min + 1, info.max - 1, 0, -1]
    s = np.array(specials, dtype=dt)
    flat = T.reshape(-1)
    at = rng.choice(flat.size, size=flat.size // 3, replace=False)
    flat[at] = s[rng.integers(0, len(s), size=len(at))]
    return T


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("dtype", list(TOPK_DTYPES))
def test_topk_special_values(eng, dtype, descending):
    """A third of the entries are extreme keys, heavily tied: both paths (k + drop = 300 and 6000),
    whole rows sorted (k = N) and a row shorter than the list."""
    dt = TOPK_DTYPES[dtype]
    rng = np.random.default_rng(65504 + len(dtype))
    for N in (300, 6000):
        T = special_tile(rng, dt, 3, N)
        dev, order = wide_slice(T), order_ref(T, descending)
        for k, drop in ((299, 1), (N, 0), (5999, 1), (4000, 5), (7000, 0)):
            check_topk(eng, T, k, drop, descending, order, dev)


@pytest.mark.parametrize("dtype", list(TOPK_DTYPES))
def test_topk_row_counts(eng, dtype):
    """Rows 1, 2, 3, 1024, 1025: the second radix sort of the sort path keys on row_bits =
    ceil(log2(rows)) bits; the shared-memory path runs one CTA per row."""
    dt = TOPK_DTYPES[dtype]
    rng = np.random.default_rng(1025 + len(dtype))
    for rows in (1, 2, 3, 1024, 1025):
        T = special_tile(rng, dt, rows, 4100)
        for descending in (False, True):
            dev, order = wide_slice(T), order_ref(T, descending)
            check_topk(eng, T, 3, 4094, descending, order, dev)     # k1 = 4097: sort path
            check_topk(eng, T, 5, 1, descending, order, dev)


# ------------------------------------------------------------------ threshold -> CSR
THRESH_DTYPES = {"u8": np.uint8, "f16": np.float16, "f32": np.float32, "f64": np.float64, "i32": np.int32,
                 "i64": np.int64}
GUARDS = {0: lambda t: torch.ones_like(t, dtype=torch.bool), 1: lambda t: t > 0, 2: lambda t: t < 1}


def torch_keep(T, cmp, eps, swap, guard):
    """The reference's literal expression on a CPU tensor (prograph.py:734-736 / :544)."""
    t = torch.from_numpy(np.ascontiguousarray(T))
    if T.dtype == np.uint8:
        return (t != 0).numpy()
    c = cmp(eps, t) if swap else cmp(t, eps)
    return (c & GUARDS[guard](t)).numpy()


def check_threshold(eng, T, cmp, eps, swap, guard):
    from prograph_b200 import _lib as L
    code = {operator.lt: L.LT, operator.le: L.LE, operator.eq: L.EQ, operator.ne: L.NE, operator.ge: L.GE,
            operator.gt: L.GT}[cmp]
    keep = torch_keep(T, cmp, eps, swap, guard)
    dev = wide_slice(T, 5)
    same(eng.tile_threshold_counts(dev, code, eps, swap=swap, guard=guard), keep.sum(1).astype(np.int64))
    ip, idx, val = eng.tile_threshold(dev, code, eps, swap=swap, guard=guard)
    rp, ri, rv = csr_ref(T, keep)
    same(ip, rp)
    same(idx, ri)
    same(val, rv)


def thresh_tile(rng, dt, n, eps):
    """Six rows: tie-heavy values around eps (NaN sprinkled in for floats), all eps, all NaN (or
    all large), all 3, all -2, and values in {0, 1} -- rows with no hits and rows with all hits for
    every comparison."""
    if dt == np.uint8:
        T = rng.integers(0, 2, size=(6, n)).astype(np.uint8)
        T[1], T[2] = 0, 1
        return T
    T = (rng.integers(-8, 17, size=(6, n)) / 4.0).astype(np.float64)
    T[1], T[2], T[3], T[4] = eps, np.nan, 3, -2
    T[5] = rng.integers(0, 2, size=n)
    if np.dtype(dt).kind == "f":
        T[0, rng.random(n) < 0.1] = np.nan
        return T.astype(dt)
    T[2] = 1 << 20
    return np.round(T[:, :]).astype(dt)


@pytest.mark.parametrize("dtype", list(THRESH_DTYPES))
def test_threshold_grid(eng, dtype):
    """Every cmp x swap x guard on every tile dtype, N around the warp ballot (32) and the 256-entry
    block prefix sum, counts-only entry and CSR; integer tiles with an int and a float eps."""
    dt = THRESH_DTYPES[dtype]
    rng = np.random.default_rng(33 + len(dtype) + np.dtype(dt).itemsize)
    kind = np.dtype(dt).kind
    eps_list = (0.5,) if kind == "f" else (1, 1.5) if kind == "i" else (0.0,)
    cmps = list(CMPS.values()) if dt != np.uint8 else [operator.ne]
    for N in (1, 31, 32, 33, 255, 256, 257, 4097):
        for eps in eps_list:
            T = thresh_tile(rng, dt, N, eps)
            for cmp in cmps:
                for swap in (False, True):
                    for guard in (0, 1, 2):
                        check_threshold(eng, T, cmp, eps, swap, guard)


@pytest.mark.parametrize("dtype", ["f16", "f32", "f64", "i32", "i64"])
def test_threshold_eps_rounding(eng, dtype):
    """A python scalar is compared as torch compares it with the tile: rounded to fp16 / float32
    for those tiles (0.1, 1.0004 -> 1, 70000 -> inf in fp16); against an integer tile exactly when
    it is an int and in float32 when it is a float (2 < 2.00000001 is false; 16777217 <= 16777216.5
    is true)."""
    dt = THRESH_DTYPES[dtype]
    if dt == np.float16:
        vals = np.array([0.0999755859375, 0.10003662109375, 0.0999145507812, 1.0, 1.0009765625, 0.99951171875,
                         65504.0, np.inf, -np.inf, np.nan], dtype=dt)
        eps_list = (0.1, 1.0004, 70000, 1, 65504)
    elif dt == np.float32:
        f = np.float32(0.1)
        vals = np.array([f, np.nextafter(f, np.float32(1)), np.nextafter(f, np.float32(0)), 0.1, 16777216.0,
                         16777218.0, np.nan], dtype=dt)
        eps_list = (0.1, 16777217, 16777216.5)
    elif dt == np.float64:
        vals = np.array([0.1, np.nextafter(0.1, 1), np.float32(0.1), 2.00000001, 2.0, np.nan], dtype=dt)
        eps_list = (0.1, 2.00000001, 2)
    else:
        vals = np.array([2, 3, 1, 16777216, 16777217, 16777218, 0, -2], dtype=dt)
        eps_list = (2.00000001, 16777216.5, 2, 16777217, 1.9999999, -1.5)
    T = np.stack([np.resize(vals, 40), np.resize(vals[::-1], 40)])
    for eps in eps_list:
        for cmp in CMPS.values():
            for swap in (False, True):
                for guard in (0, 1):
                    check_threshold(eng, T, cmp, eps, swap, guard)


def mutants(rng, n, L):
    """Tokens 1..4: a wild type and rows with 1 .. 3 substitutions, so that many pairs sit at
    distance 2."""
    wt = rng.integers(1, 5, size=L)
    X = np.tile(wt, (n, 1))
    for i in range(1, n):
        pos = rng.choice(L, size=int(rng.integers(1, 4)), replace=False)
        X[i, pos] = (X[i, pos] + rng.integers(0, 3, size=len(pos))) % 4 + 1
    return X.astype(np.int64)


def test_count_within_float_eps_fused_vs_tile():
    """query.count_within on integer tokens runs the fused sweep (its truth table comes from torch);
    the same data shifted by 0.5 have the same Hamming distances but are no tokens, so they run the
    values tile and the threshold count.  Both must be torch's ``comp(d, eps)``, also for a float
    eps just above an integer distance."""
    from prograph_b200.query import Library, count_within
    rng = np.random.default_rng(2)
    X = mutants(rng, 500, 20)
    Q = np.concatenate([X[:40], mutants(rng, 10, 20)])
    D = torch.from_numpy(O.hamming(X, Q))
    assert (D == 2).sum() > 100                            # the distance the float eps sits above
    tok, val = Library(X), Library(X + 0.5)
    for eps in (2.00000001, 2, 1.99999999, 2.5):
        for cmp in (operator.lt, operator.le, operator.eq):
            want = cmp(D, eps).sum(1).numpy()
            same(count_within(tok, Q, eps, cmp), want)
            same(count_within(val, Q + 0.5, eps, cmp), want)


def test_build_graph_embedded_float_eps():
    """build_graph on a float representation (fp16 staging, values tile, threshold fill) with a
    float eps just above an integer distance, against the oracle's graph."""
    from prograph_b200 import build_neighbours
    rng = np.random.default_rng(3)
    X = mutants(rng, 300, 20) + 0.5
    assert (O.hamming(X, X) == 2).sum() > 100
    for eps, comp in ((2.00000001, operator.lt), (2.00000001, operator.le), (2.00000001, operator.eq),
                      (1.99999999, operator.le), (2, operator.lt)):
        got = build_neighbours(X, eps=eps, comp=comp)
        for g, r in zip((got.indptr, got.idx, got.w), O.to_csr(O.build_graph(X, eps=eps, comp=comp))):
            same(g, r)


# ------------------------------------------------------------------ selection masks
def mask_library(rng, n, L):
    """Letters of a mutational library: row 0 the wild type (the seed), rows 1.. with 0 .. 3
    substitutions at a few hot positions (bit 31 of word 0, the first and last positions of the
    last word, L - 1) and every third row with up to 4 more anywhere; every 37th row a duplicate;
    rows 40 .. 42 shorter by 1 .. 3 residues (pad token 0)."""
    aa = np.array(list(O.AMINO_ACIDS))
    wt = rng.integers(0, 20, size=L)
    hot = np.array(sorted({p for p in (0, 31, 32, L // 2, 32 * ((L - 1) // 32), L - 2, L - 1) if 0 <= p < L}))
    T = np.tile(wt, (n, 1))
    k_hot = rng.integers(0, 4, size=n)
    for j in range(3):
        rows = np.nonzero(k_hot > j)[0]
        pos = hot[rng.integers(0, len(hot), size=len(rows))]
        T[rows, pos] = (wt[pos] + rng.integers(1, 20, size=len(rows))) % 20
    for j in range(4):
        rows = np.nonzero((np.arange(n) % 3 == 0) & (rng.random(n) < 0.6))[0]
        pos = rng.integers(0, L, size=len(rows))
        T[rows, pos] = (wt[pos] + rng.integers(1, 20, size=len(rows))) % 20
    T[0] = wt
    T[37::37] = T[36:-1:37]
    seqs = ["".join(aa[r]) for r in T]
    for i in (40, 41, 42):
        if i < n:
            seqs[i] = seqs[i][: L - (i % 3) - 1]
    return seqs, hot


def agree(got_fn, ref_fn):
    """The product and the oracle return the same arrays, or both refuse (AssertionError)."""
    try:
        want = ref_fn()
    except AssertionError:
        with pytest.raises(AssertionError):
            got_fn()
        return
    got = got_fn()
    if isinstance(want, tuple):
        assert isinstance(got, tuple) and len(got) == len(want)
        for g, w in zip(got, want):
            np.testing.assert_array_equal(np.asarray(g), w)
    else:
        np.testing.assert_array_equal(np.asarray(got), want)


@pytest.mark.parametrize("L,n", [(33, 1000), (64, 1000), (100, 1000), (300, 1000), (1000, 1000), (4096, 1000),
                                 (4097, 1000), (5000, 1000), (33, 1), (33, 2), (4097, 2), (300, 70000)])
def test_selection_masks_wide_rows(tmp_path, L, n):
    """Prograph.indexing (distances, positions or / and, complement, another reference row),
    get_mutated_positions, calc_mutated_positions, calc_neighbours and the distance census behind
    indexing's assert, on rows of 2 .. 157 mask words.  Up to 4096 residues (128 words) the masks
    travel as kernel parameters, beyond that through a device buffer.  70 000 rows make the flag
    compaction span many tiles."""
    import prograph_b200 as pgb
    rng = np.random.default_rng(L * 7 + n)
    seqs, hot = mask_library(rng, n, L)
    path = tmp_path / "lib.csv"
    # a stored Neighbours column: the constructor keeps it instead of building the eps = 1 graph,
    # which at 70 000 rows around one wild type is dense and not what is tested here
    pd.DataFrame({"Sequence": seqs, "Fitness": rng.normal(size=n), "Neighbours": ["[]"] * n}).to_csv(path)
    pg = pgb.Prograph(file=str(path))
    tok = O.tokenize(seqs)
    np.testing.assert_array_equal(pg.tokenized, tok)
    mp = O.calc_mutated_positions(tok, tok[0])
    np.testing.assert_array_equal(pg.calc_mutated_positions(), mp)
    np.testing.assert_array_equal(pg.mutated_positions, mp)
    refs = [0] + ([5] if n > 5 else [])
    for ref in refs:
        d = O.hamming(tok, tok[ref:ref + 1])[0]
        np.testing.assert_array_equal(pg._distance_hist(ref), np.bincount(d, minlength=L + 1)[:L + 1])
        present = np.unique(d)
        absent = [x for x in range(L + 1) if x not in set(present.tolist())][:1]
        seq = None if ref == 0 else ref
        for ds in ([int(present[0])], [int(present[-1])], [int(x) for x in present[1:4]], absent):
            if ds:
                agree(lambda: pg.indexing(reference_seq=seq, distances=ds),
                      lambda: O.indexing(tok, ref, distances=ds))
        for pos in ([31], [L - 1], [int(p) for p in hot[-3:]], [int(p) for p in hot[:3]], [int(p) for p in hot]):
            pos = [p for p in pos if p < L]
            for Bool in ("or", "and"):
                agree(lambda: pg.indexing(reference_seq=seq, positions=pos, Bool=Bool),
                      lambda: O.indexing(tok, ref, positions=pos, Bool=Bool))
                agree(lambda: pg.indexing(reference_seq=seq, positions=pos, Bool=Bool, complement=True),
                      lambda: O.indexing(tok, ref, positions=pos, Bool=Bool, complement=True))
            dd = [int(x) for x in present[:3]]
            agree(lambda: pg.indexing(reference_seq=seq, distances=dd, positions=pos, complement=True),
                  lambda: O.indexing(tok, ref, distances=dd, positions=pos, complement=True))
        for eps, comp in ((1, operator.eq), (2, operator.le), (2.5, operator.le), (3, operator.gt), (0, operator.ne)):
            np.testing.assert_array_equal(pg.calc_neighbours(ref, eps=eps, comp=comp),
                                          O.calc_neighbours(tok, ref, eps=eps, comp=comp))
    mut = O.boolean_mutant_array(tok, 0)
    hot_mut = [int(p) for p in hot if p in set(mp.tolist())]
    for positions in ([], hot_mut[:1], hot_mut[-2:], hot_mut, [int(p) for p in mp[-3:]]):
        positions = np.array(sorted(set(positions)), dtype=np.int64)
        np.testing.assert_array_equal(pg.get_mutated_positions(positions), O.get_mutated_positions(mut, mp, positions))
