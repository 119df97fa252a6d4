"""numpy restatement of Pillow's ``Image.resize(size)`` with its default filter (BICUBIC) on 8-bit images.

Test infrastructure only: the device resize (``se_resize_u8``) and its host-side coefficient tables (``se_resize_coeffs``) are
checked against it, and it is checked against the installed Pillow byte for byte.

Each channel is resampled independently: a horizontal pass if the width changes, then a vertical pass if the height changes,
with a uint8 intermediate; the same size is a copy. Coefficients are computed in double precision in the order below (one ulp
in a weight can move its fixed-point value), normalised by a division, and rounded to 22-bit fixed point; the accumulation is
int32 starting at 2^21, and the output is ``clamp(acc >> 22, 0, 255)``.
"""
import math

import numpy as np

PRECISION_BITS = 22
_A = -0.5


def _bicubic(x):
    x = np.abs(x)
    near = ((_A + 2.0) * x - (_A + 3.0)) * x * x + 1
    far = (((x - 5) * x + 8) * x - 4) * _A
    return np.where(x < 1.0, near, np.where(x < 2.0, far, 0.0))


def coeffs(n_in, n_out):
    """Tables of one ``n_in -> n_out`` pass: (bounds int32 [n_out, 2] = (first source index, tap count),
    weights int32 [n_out, ksize] in 22-bit fixed point, zero past the tap count)."""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = 2 * int(math.ceil(support)) + 1
    center = (np.arange(n_out, dtype=np.float64) + 0.5) * scale
    xmin = np.maximum((center - support + 0.5).astype(np.int64), 0)          # astype truncates toward zero, like the C cast
    n = np.minimum((center + support + 0.5).astype(np.int64), n_in) - xmin
    taps = np.arange(ksize)
    w = _bicubic(((taps[None, :] + xmin[:, None]).astype(np.float64) - center[:, None] + 0.5) * (1.0 / fs))
    w = np.where(taps[None, :] < n[:, None], w, 0.0)
    ww = np.zeros(n_out)
    for x in range(ksize):                                                  # sequential sum, not numpy's pairwise one
        ww = ww + w[:, x]
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    fixed = np.where(w < 0, w * (1 << PRECISION_BITS) - 0.5, w * (1 << PRECISION_BITS) + 0.5)
    return np.stack([xmin, n], 1).astype(np.int32), np.trunc(fixed).astype(np.int32)


def _pass(a, bounds, weights, axis):
    """Resample uint8 array ``a`` ([H, W, C]) along ``axis`` (1: horizontal, 0: vertical)."""
    a = np.moveaxis(a, axis, 0).astype(np.int64)
    n_out, ksize = weights.shape
    idx = np.minimum(bounds[:, :1] + np.arange(ksize)[None, :], a.shape[0] - 1)    # taps past the count have weight 0
    acc = np.full((n_out,) + a.shape[1:], 1 << (PRECISION_BITS - 1), np.int64)
    for t in range(ksize):
        acc += a[idx[:, t]] * weights[:, t].astype(np.int64).reshape((n_out,) + (1,) * (a.ndim - 1))
    out = np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def resize(a, size):
    """``Image.fromarray(a).resize(size)`` as an array: ``a`` uint8 [H, W] or [H, W, C]; ``size`` = (width, height) as in PIL."""
    a = np.asarray(a, np.uint8)
    w_out, h_out = size
    x = a if a.ndim == 3 else a[:, :, None]
    h_in, w_in = x.shape[:2]
    if w_out != w_in:
        x = _pass(x, *coeffs(w_in, w_out), axis=1)
    if h_out != h_in:
        x = _pass(x, *coeffs(h_in, h_out), axis=0)
    x = np.array(x)
    return x if a.ndim == 3 else x[:, :, 0]
