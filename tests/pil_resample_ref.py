"""numpy restatement of Pillow's 8-bit BILINEAR / BICUBIC resample (libImaging/Resample.c) -- TEST-ONLY.

The oracle the CPU suite checks against Image.resize, and the reference the header (csrc/bj_resize_pil_math.cuh) and
the GPU kernel are compared with.  Coefficients are computed tap by tap in Python floats (IEEE doubles, Pillow's
operation order); the passes are exact integer arithmetic.
"""
from __future__ import annotations

import math

import numpy as np

PRECISION_BITS = 32 - 8 - 2


def bilinear(x: float) -> float:
    if x < 0.0:
        x = -x
    if x < 1.0:
        return 1.0 - x
    return 0.0


def bicubic(x: float) -> float:
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


FILTERS = {"bilinear": (bilinear, 1.0), "bicubic": (bicubic, 2.0)}


def coeffs(in_size: int, out_size: int, name: str):
    """precompute_coeffs + normalize_coeffs_8bpc for box [0, in_size): (xmin (out,), n (out,), k (out, ksize) int64)."""
    f, support0 = FILTERS[name]
    scale = float(in_size) / out_size
    filterscale = max(scale, 1.0)
    support = support0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    ss = 1.0 / filterscale
    xmins = np.zeros(out_size, np.int64)
    ns = np.zeros(out_size, np.int64)
    k = np.zeros((out_size, ksize), np.int64)
    for xx in range(out_size):
        center = 0.0 + (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        w = [f((x + xmin - center + 0.5) * ss) for x in range(xmax)]
        ww = 0.0
        for v in w:
            ww += v
        if ww != 0.0:
            w = [v / ww for v in w]
        k[xx, :xmax] = [int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
                        for v in w]
        xmins[xx], ns[xx] = xmin, xmax
    return xmins, ns, k


def clip8(s: np.ndarray) -> np.ndarray:
    return np.where(s >= (1 << PRECISION_BITS << 8), 255, np.where(s <= 0, 0, s >> PRECISION_BITS))


def resample_axis(a: np.ndarray, out_size: int, name: str, axis: int) -> np.ndarray:
    """One pass along `axis` of an integer array: clip8(2^21 + sum src * k).  Pillow skips the pass when the size is
    unchanged; the pass it would run there is the identity (the header shows why), so this always runs it."""
    xmins, ns, k = coeffs(a.shape[axis], out_size, name)
    a = np.moveaxis(a.astype(np.int64), axis, 0)
    out = np.empty((out_size,) + a.shape[1:], np.int64)
    for i in range(out_size):
        m, n = xmins[i], ns[i]
        kk = k[i, :n].reshape((-1,) + (1,) * (a.ndim - 1))
        out[i] = clip8((1 << (PRECISION_BITS - 1)) + (a[m:m + n] * kk).sum(0))
    return np.moveaxis(out, 0, axis)


def resize(img: np.ndarray, w: int, h: int, name: str) -> np.ndarray:
    """Image.fromarray(img).resize((w, h), BILINEAR | BICUBIC) for uint8 (H, W) or (H, W, C) img: the horizontal pass,
    rounded to uint8, then the vertical pass."""
    t = resample_axis(img, w, name, 1)
    return resample_axis(t, h, name, 0).astype(np.uint8)

