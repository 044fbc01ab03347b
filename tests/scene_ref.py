"""fp64 restatement of the whole-scene blend (nirgan_b200/scene.py) for the scene tests."""
from __future__ import annotations

import numpy as np


def blend_reference(pred, row_origins, col_origins, T, overlap, W, y0, y1):
    """out[y0:y1, :W] = sum_t w_t p_t / sum_t w_t in float64; pred [len(row_origins) * len(col_origins)][T][T] holds the
    tile at (row_origins[ky], col_origins[kx]) at index ky * len(col_origins) + kx."""
    pred = np.asarray(pred, dtype=np.float64).reshape(len(row_origins) * len(col_origins), T, T)
    i = np.arange(T)
    w1 = np.minimum(np.minimum(i + 1, T - i), overlap + 1) / (overlap + 1)
    w = np.outer(w1, w1)
    base = row_origins[0]
    num = np.zeros((row_origins[-1] + T - base, W))
    den = np.zeros_like(num)
    for ky, oy in enumerate(row_origins):
        for kx, ox in enumerate(col_origins):
            num[oy - base:oy - base + T, ox:ox + T] += w * pred[ky * len(col_origins) + kx]
            den[oy - base:oy - base + T, ox:ox + T] += w
    with np.errstate(invalid="ignore", divide="ignore"):
        out = num / den
    return out[y0 - base:y1 - base]
