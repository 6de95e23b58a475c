"""Test helpers for the reduced-size decode: the fp64 evaluation of its definition (csrc/bj_scaled_math.cuh) and the
host model of the kernel (tests/hostsim/scaled_hostsim.cpp), both over a bj_image record and an MCU-major
coefficient buffer."""
import ctypes
from functools import lru_cache

import numpy as np

from hostsim import build

ZZ_NATURAL = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                       13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52,
                       45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
ERR_C, ERR_K = 3.25, 1.0          # BJ_SCALED_ERR_C / BJ_SCALED_ERR_K


@lru_cache(None)
def hostsim():
    L = build("scaled_hostsim")
    vp = ctypes.c_void_p
    L.hs_scaled_prefix.restype = ctypes.c_int
    L.hs_scaled_prefix.argtypes = [ctypes.c_int, ctypes.c_int]
    L.hs_scaled_block.restype = None
    L.hs_scaled_block.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    L.hs_scaled_image.restype = None
    L.hs_scaled_image.argtypes = [vp, vp, vp, vp, vp]
    return L


def basis(n: int) -> np.ndarray:
    """(n, n) fp64: B[x, u] = 2 sqrt 2 * C(u) / 2 * cos((2x + 1) u pi / 2n), so that f = B_y F B_x^T / 8.  The values
    that are exactly 0 or +-1 (u = 0 and the pi/4 terms) are set exactly: the sums of blocks made of such terms are
    then exact, and so are their rounding ties."""
    x = np.arange(n)[:, None]
    u = np.arange(n)[None, :]
    b = np.where(u == 0, 1.0, 2 ** 0.5 * np.cos((2 * x + 1) * u * np.pi / (2 * n)))
    for exact in (-1.0, 0.0, 1.0):
        b[np.abs(b - exact) < 1e-12] = exact
    return b


def dequant(coef_zz, q_zz) -> np.ndarray:
    """(8, 8) fp64 [v, u] of int16-wrapped products, natural order."""
    prod = (np.asarray(coef_zz, np.int64) * np.asarray(q_zz, np.int64)).astype(np.int16)
    F = np.zeros(64)
    F[ZZ_NATURAL] = prod
    return F.reshape(8, 8)


def tile_f64(coef_zz, q_zz, nx: int, ny: int):
    """(ny, nx) fp64 f of the definition, and sum |F| over the corner."""
    F = dequant(coef_zz, q_zz)[:ny, :nx]
    return basis(ny) @ F @ basis(nx).T / 8, np.abs(F).sum()


def bound(sum_abs) -> np.ndarray:
    return ERR_C * 2.0 ** -24 * (np.asarray(sum_abs) + ERR_K)


def image_f64(rec, log2s: int, coef: np.ndarray, qtabs: np.ndarray) -> np.ndarray:
    """uint8 (ceil(H/s), ceil(W/s)[, 3]) of one image by the definition in fp64 (colour with the reference's fp64
    expression)."""
    coef = np.asarray(coef).reshape(-1, 64)
    hmax, vmax, nc = int(rec["hmax"]), int(rec["vmax"]), int(rec["ncomp"])
    mx_n, my_n, bpm = int(rec["mcus_x"]), int(rec["mcus_y"]), int(rec["blocks_per_mcu"])
    mw, mh = (8 * hmax) >> log2s, (8 * vmax) >> log2s
    planes = np.zeros((nc, my_n * mh, mx_n * mw))
    b0 = int(rec["coef_block0"])
    nat = np.argsort(ZZ_NATURAL)                      # natural index -> zig-zag index
    for c in range(nc):
        hs, vs = int(rec["hs"][c]), int(rec["vs"][c])
        nx, ny = (8 * hmax // hs) >> log2s, (8 * vmax // vs) >> log2s
        q = np.asarray(qtabs[int(rec["qtab"][c])], np.int64)
        grid = planes[c].reshape(my_n, mh, mx_n, mw)
        for r in range(hs * vs):
            bx, by = r % hs, r // hs
            blk = b0 + np.arange(my_n * mx_n) * bpm + int(rec["slot0"][c]) + r
            prod = (coef[blk].astype(np.int64) * q).astype(np.int16).astype(np.float64)
            F = prod[:, nat].reshape(-1, 8, 8)[:, :ny, :nx]                     # (mcus, v, u)
            f = np.einsum("yv,mvu,xu->myx", basis(ny), F, basis(nx)) / 8
            s = (np.round(f) + 128).reshape(my_n, mx_n, ny, nx)
            grid[:, by * ny:(by + 1) * ny, :, bx * nx:(bx + 1) * nx] = s.transpose(0, 2, 1, 3)
    s_ = 1 << log2s
    H, W = -(-int(rec["height"]) // s_), -(-int(rec["width"]) // s_)
    p = planes[:, :H, :W]
    if nc == 1:
        return np.clip(p[0], 0, 255).astype(np.uint8)
    Y, cb, cr = p[0], p[1] - 128.0, p[2] - 128.0
    rgb = np.stack([Y + 1.402 * cr, Y - 0.34414 * cb - 0.71414 * cr, Y + 1.772 * cb], -1)
    return np.round(np.clip(rgb, 0, 255)).astype(np.uint8)


def image_hostsim(rec, log2s: int, coef: np.ndarray, qtabs: np.ndarray) -> np.ndarray:
    """The same image from the host model of the kernel (bit-identical fp32 arithmetic)."""
    from pyjpegdecoder_b200._native import IMAGE_DTYPE
    from pyjpegdecoder_b200.scaled import SCALED_JOB_DTYPE
    s_ = 1 << log2s
    H, W = -(-int(rec["height"]) // s_), -(-int(rec["width"]) // s_)
    ch = 3 if int(rec["ncomp"]) == 3 else 1
    im = np.zeros(1, IMAGE_DTYPE)
    im[0] = rec
    job = np.zeros(1, SCALED_JOB_DTYPE)
    job["out_pitch"], job["log2_scale"] = W * ch, log2s
    out = np.zeros(H * W * ch, np.uint8)
    c = np.ascontiguousarray(coef, dtype=np.int16)
    q = np.ascontiguousarray(qtabs, dtype=np.int16)
    hostsim().hs_scaled_image(im.ctypes.data, job.ctypes.data, c.ctypes.data, q.ctypes.data, out.ctypes.data)
    return out.reshape((H, W, 3) if ch == 3 else (H, W))
