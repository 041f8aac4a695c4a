"""prograph_b200: B200-native graph-construction path of acmater/prograph.

Drop-in surface (prograph/__init__.py:1-2, prograph/distance/__init__.py:1-3):
``Prograph``, ``Protein``, ``hamming``, ``minkowski``, ``clean_input``.  All pairwise
distance, neighbour-list and mutation-mask work runs in hand-written sm_100a CUDA kernels
behind the C ABI declared in include/prograph_b200.h; importing this package without the
built shared library, or using it without a CUDA device, raises -- there is no CPU path.
"""
from . import _lib

_lib.load()   # fail loudly at import time when libprograph_b200.so has not been built

from .distance import hamming, minkowski, clean_input  # noqa: E402
from .protein import Protein  # noqa: E402
from .prograph import Prograph  # noqa: E402
from .graph import build_neighbours, extend_neighbours, NeighbourTable, KnnTable  # noqa: E402
from .io import save  # noqa: E402
from . import query  # noqa: E402,F401  (distance-to-dataset queries fused with their consumers)

__all__ = ["Prograph", "Protein", "hamming", "minkowski", "clean_input", "build_neighbours", "extend_neighbours",
           "NeighbourTable", "KnnTable", "save", "query"]
__version__ = "0.1.0"
