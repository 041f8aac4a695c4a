"""Host-side rules of the Minkowski p=2 GEMM on wide rows (no GPU needed)."""
import torch

from prograph_b200.distance.minkowski import gemm_value_kind
from prograph_b200.engine import CudaEngine


def test_gemm_width_limit():
    assert CudaEngine.GEMM_MAX_WIDTH == 8192


def test_gemm_value_kind_float32_token_cap():
    """float32 rows are summed in float32: the largest token keeps width * max_token^2 <= 2^24, so every
    partial sum of the element-wise kernel is an exact integer and the GEMM's exact S gives the same
    root.  Up to 256 columns the cap is the full 255 it always was; int64 and fp16 do not depend on it."""
    for width in (0, 1, 32, 256, 258):
        assert gemm_value_kind(torch.float32, width) == (1, 255)
    for width in (259, 300, 1176, 1184, 5376, 8192):
        kind, mt = gemm_value_kind(torch.float32, width)
        assert kind == 1
        assert width * mt * mt <= 1 << 24 < width * (mt + 1) ** 2
    assert gemm_value_kind(torch.float32, 8192) == (1, 45)
    for width in (1, 256, 8192):
        assert gemm_value_kind(torch.int64, width) == (1, 255)
        assert gemm_value_kind(torch.float16, width) == (0, 31)
        assert gemm_value_kind(torch.float64, width) == (None, None)
