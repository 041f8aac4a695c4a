"""Hamming distance, drop-in for prograph/distance/hamming.py:8-39."""
import torch

from .. import _lib as L
from ..engine import get_engine, sweep_covers
from .utils import clean_input, result_device, is_integer_dtype

_QBLOCK = 512           # query rows per tile call: the packed stream-tile granularity
_SLAB_BYTES = 1 << 30   # soft cap on the rows handed to one pg_hamming_tile call


def value_dtype(dt):
    """Compute dtype of the element-wise (non-token) kernels for a torch dtype."""
    if is_integer_dtype(dt):
        return torch.int64
    if dt in (torch.float16, torch.float32, torch.float64):
        return dt
    return torch.float32


def hamming_matrix(eng, X, Y, similarity=False):
    """(M, N) Hamming matrix of 2-D operands on the engine's device."""
    try:
        xp = eng.pack(X)
        yp = eng.pack(Y, planes=xp.planes, words=xp.words)
        if not sweep_covers(xp.planes, xp.words):
            raise L.Unsupported("rows longer than 32768 residues take the element-wise kernel")
    except (OverflowError, L.Unsupported):
        # arbitrary numeric values: element-wise != on the device (IEEE: NaN differs from all)
        dt = value_dtype(torch.result_type(X, Y))
        Xd, Yd = eng.to_device(X, dt), eng.to_device(Y, dt)
        return eng.hamming_values_tile(Xd, Yd, 0, Yd.shape[0], similarity=similarity)
    weight = L.W_SIM_F32 if similarity else L.W_I64
    out = eng.empty((yp.rows, xp.rows), torch.float32 if similarity else torch.int64)
    rows_per = max(_QBLOCK, (_SLAB_BYTES // (8 * xp.rows)) // _QBLOCK * _QBLOCK)
    for q0 in range(0, yp.rows, rows_per):
        qn = min(rows_per, yp.rows - q0)
        L.check(eng.lib.pg_hamming_tile(xp.data.data_ptr(), xp.rows, yp.data.data_ptr(), yp.rows, q0, qn, xp.planes,
                                        xp.words, weight, out[q0:].data_ptr(), xp.rows, eng._stream()))
    return out


def hamming(X, Y, similarity=False):
    """Pairwise Hamming distances between the rows of X (N, D) and Y (M, D).

    Returns a tensor of shape (M, N) -- rows follow Y, columns follow X, exactly like
    ``torch.sum(X != Y[:, None, :], axis=2)`` (hamming.py:34; the reference docstring says
    N x M but the code returns M x N).  int64, or float32 ``1/(1+d)`` when ``similarity``
    (hamming.py:37-38).  The result lives on the device of the inputs.

    The (M, N, D) boolean temporary of the reference is never formed: integer tokens are
    packed into bit planes and compared 32 residues per instruction (pg_hamming_tile);
    other numeric values go through pg_hamming_values_tile.
    """
    X, Y = clean_input(X, Y)
    dev = result_device(X, Y)
    out = hamming_matrix(get_engine(), X, Y, similarity)
    return out if out.device == dev else out.to(dev)
