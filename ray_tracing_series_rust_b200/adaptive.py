"""Adaptive sampling: the numpy reference of rt_render_adaptive (include/rtb200.h, csrc/cuda/adaptive.cu).

Round k traces samples [k*step, min((k+1)*step, max)) of the pixels still active, into the half accumulator A (even k) or B (odd k).
After every odd round, at n = (k+1)*step samples with min_samples <= n < max, `half_buffer_error` rates every active pixel from its
int64 sums and `next_active` keeps the pixels that have an unconverged pixel within Chebyshev distance `radius`.  Every decision
comes from integer sums and correctly rounded f64 operations, so this mirror reproduces the library's active sets, sample counts and
sums exactly: `adaptive_reference` over rt_render sample ranges equals rt_render_adaptive bit for bit.
"""
from __future__ import annotations

from typing import Callable, Sequence, Tuple

import numpy as np


def half_buffer_error(A: np.ndarray, B: np.ndarray, h: int) -> np.ndarray:
    """Per-pixel error [H, W] of two half accumulators [H, W, 3] of h samples each (f64, this exact order of operations):
    (((|a_r-b_r| + |a_g-b_g|) + |a_b-b_b|) / S) / sqrt(1e-4 + (((a_r+b_r) + (a_g+b_g)) + (a_b+b_b)) / (2S)),  S = h * 2^32."""
    a = np.asarray(A).astype(np.float64)
    b = np.asarray(B).astype(np.float64)
    d = (np.abs(a[..., 0] - b[..., 0]) + np.abs(a[..., 1] - b[..., 1])) + np.abs(a[..., 2] - b[..., 2])
    t = ((a[..., 0] + b[..., 0]) + (a[..., 1] + b[..., 1])) + (a[..., 2] + b[..., 2])
    S = float(h) * 4294967296.0
    return (d / S) / np.sqrt(1e-4 + t / (2.0 * S))


def _dilate(mask: np.ndarray, radius: int) -> np.ndarray:
    """Box (Chebyshev) dilation of a boolean [H, W] mask, clipped at the borders (separable: rows, then columns)."""
    if radius == 0:
        return mask.copy()
    H, W = mask.shape
    p = np.pad(mask, radius)
    rows = np.zeros((H + 2 * radius, W), dtype=bool)
    for dx in range(2 * radius + 1):
        rows |= p[:, dx:dx + W]
    out = np.zeros((H, W), dtype=bool)
    for dy in range(2 * radius + 1):
        out |= rows[dy:dy + H]
    return out


def next_active(active: np.ndarray, err: np.ndarray, tau: float, radius: int, rows: int) -> np.ndarray:
    """Active set [H, W] after a check point: U = active pixels with !(err < tau); a pixel stays iff it is active and a pixel of U
    on a rendered row (< rows) lies within Chebyshev distance `radius`."""
    active = np.asarray(active, dtype=bool)
    with np.errstate(invalid="ignore"):
        U = active & ~(np.asarray(err) < tau)
    U[rows:] = False
    return active & _dilate(U, int(radius))


def adaptive_reference(render_range: Callable[[int, int], np.ndarray], shape: Sequence[int], rows: int, spp: int, min_samples: int, step: int,
                       threshold: float, radius: int) -> Tuple[np.ndarray, np.ndarray]:
    """The adaptive render driven by full-image renders of sample ranges: `render_range(s0, s1)` -> int64 sums [H, W, 3] of samples
    [s0, s1) of every pixel (rt_render with sample_begin / sample_end).  -> (accum [H, W, 3] int64, samples [H, W] int32)."""
    if step < 1 or not (0 <= min_samples <= spp) or not (0 <= radius <= 8) or not (threshold >= 0.0):
        raise ValueError("bad adaptive request")
    H, W = int(shape[0]), int(shape[1])
    A = np.zeros((H, W, 3), dtype=np.int64)
    B = np.zeros((H, W, 3), dtype=np.int64)
    samples = np.zeros((H, W), dtype=np.int32)
    active = np.zeros((H, W), dtype=bool)
    active[:rows] = True
    k = 0
    while active.any() and k * step < spp:
        s0, s1 = k * step, min((k + 1) * step, spp)
        part = render_range(s0, s1)
        half = B if k & 1 else A
        half[active] += part[active]
        if k & 1 and min_samples <= s1 < spp:
            nxt = next_active(active, half_buffer_error(A, B, s1 // 2), threshold, radius, rows)
            samples[active & ~nxt] = s1
            active = nxt
        k += 1
    samples[active] = spp
    return A + B, samples
