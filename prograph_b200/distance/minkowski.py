"""Minkowski distance, drop-in for prograph/distance/minkowski.py:8-41."""
import math

import torch

from ..engine import get_engine
from .utils import clean_input, result_device, is_integer_dtype


def staged_dtype(X, Y, p):
    """Compute dtype as torch's type promotion picks it for
    ``pow(sum(pow(X - Y, p)), 1/p)``: fp16 stays fp16, float32/float64 stay, integers stay
    exact (int64) for positive integer p and promote to float32 otherwise."""
    dt = torch.result_type(X, Y)
    if is_integer_dtype(dt):
        return torch.int64 if (float(p) == int(p) and p > 0) else torch.float32
    if dt in (torch.float16, torch.float32, torch.float64):
        return dt
    return torch.float32


def gemm_value_kind(dt, width=0):
    """Rounding chain of the tensor-core path for a compute dtype and row width: 0 = fp16 chain
    (needs tokens <= 31 so that every squared difference is an exact fp16 integer), 1 = float32
    root of the exact integer sum (int64 and float32 inputs), None = not applicable.  float32 rows
    are summed in float32, which equals the exact sum only while it stays <= 2^24: their largest
    token is capped so that width * max_token^2 <= 2^24 (255 up to 258 columns, 45 at 8192)."""
    if dt == torch.float16:
        return 0, 31
    if dt == torch.int64:
        return 1, 255
    if dt == torch.float32:
        return 1, min(255, math.isqrt((1 << 24) // max(1, int(width))))
    return None, None


def minkowski_matrix(eng, X, Y, p=2, similarity=False):
    from .. import _lib as L
    dt = staged_dtype(X, Y, p)
    kind, max_token = gemm_value_kind(dt, X.shape[1])
    if float(p) == 2.0 and kind is not None and X.shape[1] <= eng.GEMM_MAX_WIDTH:
        # p=2 on integer-valued rows is an exact int8 contraction: tensor cores (pg_gemm.cu)
        try:
            tx = eng.gemm_pack(X, max_token=max_token)
            ty = eng.gemm_pack(Y, max_token=max_token, K=tx.K)
            return eng.minkowski2_gemm_tile(tx, ty, kind, similarity=similarity)
        except (OverflowError, L.Unsupported):
            pass
    Xd, Yd = eng.to_device(X, dt), eng.to_device(Y, dt)
    return eng.minkowski_tile(Xd, Yd, 0, Yd.shape[0], p=p, similarity=similarity)


def minkowski(X, Y, p=2, similarity=False):
    """Pairwise Minkowski "distances" between the rows of X (N, D) and Y (M, D):
    ``pow(sum(pow(X - Y[:, None, :], p), axis=2), 1/p)`` -- without an absolute value,
    exactly as the reference computes it (minkowski.py:36), so p=1 gives signed sums and
    odd p can give NaN.  Shape (M, N).  fp16 in -> fp16 out with every step rounded to
    fp16 as torch does (the dtype ``build_graph`` feeds, prograph.py:726); float32 ->
    float32; integers -> exact integer power sum, float32 root.  ``similarity`` returns
    ``1/(1+d)`` (minkowski.py:39-40).
    """
    X, Y = clean_input(X, Y)
    dev = result_device(X, Y)
    out = minkowski_matrix(get_engine(), X, Y, p, similarity)
    return out if out.device == dev else out.to(dev)
