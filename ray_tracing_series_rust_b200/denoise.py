"""Denoised renders: the numpy reference of rt_render_denoised's filter (include/rtb200.h, csrc/cuda/denoise.cu, DESIGN.md section 11).

The inputs are two half accumulators A (samples [0, hA)) and B (samples [hA, n)) and the first-hit feature sums of samples
[0, m) (rt_render_aov).  `filter_inputs` turns them into the mean c, the noise of the mean v and the feature means; `atrous` runs the
feature-guided a-trous passes in f64, in exactly the order of operations of the device kernels; `screen_values` quantises like
rt_render.  Only pixels on the rendered rows (< rows) take part, as outputs and as neighbours; the other rows stay 0.  The library's
result differs from this one only where the device's exp and sqrt round their last bit differently.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

S32 = 1.0 / 4294967296.0
H_KERNEL = (1.0 / 16.0, 1.0 / 4.0, 3.0 / 8.0, 1.0 / 4.0, 1.0 / 16.0)
G_BLUR = (0.25, 0.5, 0.25)


def lum(x: np.ndarray) -> np.ndarray:
    """(0.2126 r + 0.7152 g) + 0.0722 b over the last axis"""
    return (0.2126 * x[..., 0] + 0.7152 * x[..., 1]) + 0.0722 * x[..., 2]


def filter_inputs(A: np.ndarray, B: np.ndarray, hA: int, hB: int, albedo_sum: np.ndarray, normal_sum: np.ndarray, m: int, rows: int):
    """-> (c [rows, W, 3], v [rows, W], albedo mean [rows, W, 3], normal mean [rows, W, 3]) of the rendered rows:
    c = ((A+B) 2^-32)(1/n), v = (lum(A 2^-32 (1/hA)) - lum(B 2^-32 (1/hB)))^2 * (hA hB / n^2), features = sum 2^-32 / m."""
    A = np.asarray(A, dtype=np.int64)[:rows]
    B = np.asarray(B, dtype=np.int64)[:rows]
    n = hA + hB
    c = ((A + B).astype(np.float64) * S32) * (1.0 / n)
    ma = (A.astype(np.float64) * S32) * (1.0 / hA)
    mb = (B.astype(np.float64) * S32) * (1.0 / hB)
    d = lum(ma) - lum(mb)
    v = (d * d) * (float(hA * hB) / float(n * n))
    a = (np.asarray(albedo_sum, dtype=np.int64)[:rows].astype(np.float64) * S32) / float(m)
    nm = (np.asarray(normal_sum, dtype=np.int64)[:rows].astype(np.float64) * S32) / float(m)
    return c, v, a, nm


def _tap(x: np.ndarray, oy: int, ox: int) -> Tuple[np.ndarray, np.ndarray]:
    """x at (y + oy, x + ox) for every (y, x), 0 outside, and the mask of the taps inside"""
    R, W = x.shape[0], x.shape[1]
    out = np.zeros_like(x)
    ok = np.zeros((R, W), dtype=bool)
    y0, y1 = max(0, -oy), min(R, R - oy)
    x0, x1 = max(0, -ox), min(W, W - ox)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = x[y0 + oy:y1 + oy, x0 + ox:x1 + ox]
        ok[y0:y1, x0:x1] = True
    return out, ok


def blur_variance(v: np.ndarray) -> np.ndarray:
    """3x3 blur, (1/4, 1/2, 1/4) per axis, the weights of the taps inside renormalised; dy outer, dx inner"""
    s = np.zeros_like(v)
    ws = np.zeros_like(v)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            q, ok = _tap(v, dy, dx)
            w = G_BLUR[dy + 1] * G_BLUR[dx + 1]
            s = np.where(ok, s + w * q, s)
            ws = np.where(ok, ws + w, ws)
    return s / ws


def atrous_pass(c, v, a, nm, step: int, sigma_color: float, sigma_albedo: float, sigma_normal: float):
    """One pass at `step`: 25 taps, w = h(dx) h(dy) exp(-(|lum(c_p) - lum(c_q)| / (sigma_c sqrt(vbar_p) + 1e-10) + |a_p - a_q|^2 / sigma_a^2
    + |n_p - n_q|^2 / sigma_n^2)); -> (sum w c_q / sum w, sum w^2 v_q / (sum w)^2)"""
    vbar = blur_variance(v)
    lp = lum(c)
    den = sigma_color * np.sqrt(vbar) + 1e-10
    sa2, sn2 = sigma_albedo * sigma_albedo, sigma_normal * sigma_normal
    sw = np.zeros_like(v)
    sc = np.zeros_like(c)
    sv = np.zeros_like(v)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            cq, ok = _tap(c, dy * step, dx * step)
            vq, _ = _tap(v, dy * step, dx * step)
            aq, _ = _tap(a, dy * step, dx * step)
            nq, _ = _tap(nm, dy * step, dx * step)
            da_, dn_ = a - aq, nm - nq
            da = (da_[..., 0] * da_[..., 0] + da_[..., 1] * da_[..., 1]) + da_[..., 2] * da_[..., 2]
            dn = (dn_[..., 0] * dn_[..., 0] + dn_[..., 1] * dn_[..., 1]) + dn_[..., 2] * dn_[..., 2]
            with np.errstate(over="ignore", invalid="ignore"):
                e = (np.abs(lp - lum(cq)) / den + da / sa2) + dn / sn2
                w = (H_KERNEL[dx + 2] * H_KERNEL[dy + 2]) * np.exp(-e)
            sw = np.where(ok, sw + w, sw)
            sc = np.where(ok[..., None], sc + w[..., None] * cq, sc)
            sv = np.where(ok, sv + (w * w) * vq, sv)
    return sc / sw[..., None], sv / (sw * sw)


def denoise(A, B, hA: int, hB: int, albedo_sum, normal_sum, m: int, rows: int, iterations: int, sigma_color: float, sigma_albedo: float,
            sigma_normal: float) -> np.ndarray:
    """The filtered mean [H, W, 3] (rt_render_denoised's out_linear): `iterations` passes at steps 1, 2, 4, ...; rows >= rows are 0."""
    if not (1 <= iterations <= 8) or hA < 1 or hB < 1 or m < 1:
        raise ValueError("bad denoise request")
    c, v, a, nm = filter_inputs(A, B, hA, hB, albedo_sum, normal_sum, m, rows)
    for i in range(iterations):
        c, v = atrous_pass(c, v, a, nm, 1 << i, sigma_color, sigma_albedo, sigma_normal)
    out = np.zeros(np.asarray(A).shape, dtype=np.float64)
    out[:rows] = c
    return out


def screen_values(linear: np.ndarray, rows: int | None = None) -> np.ndarray:
    """rt_render's quantisation of a mean: (255.9 * clamp(sqrt(x), 0, 1)) as i32, NaN -> 0; rows >= rows are 0"""
    x = np.asarray(linear, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        c = np.sqrt(x)
        c = np.where(c < 0.0, 0.0, np.where(c > 1.0, 1.0, c))
        q = 255.9 * c
        out = np.where(np.isnan(q), 0.0, np.trunc(q))
    if rows is not None:
        out[rows:] = 0.0
    return out


def split(n: int) -> Tuple[int, int]:
    """The half renders' sample counts: hA = n // 2 ([0, hA)) and hB = n - hA ([hA, n))."""
    return n // 2, n - n // 2
