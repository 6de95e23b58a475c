"""Reduced-size decode: scale 1/2, 1/4 or 1/8 in the DCT domain (csrc/bj_pixels_scaled.cu).

This module owns every decision the scale introduces, so the planners and the pipeline stay as they are: the numpy
mirror of bj_scaled_job, the output layout of a batch decoded at per-image scales, the "auto" rule of
decode_to_tensor and the launch that fills the output.  A scale-s image is (ceil(H/s), ceil(W/s), 3) (or without the
channel axis for greyscale); csrc/bj_scaled_math.cuh defines its samples.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native

# numpy mirror of struct bj_scaled_job (24 bytes, see include/b200jpeg.h)
SCALED_JOB_DTYPE = np.dtype([("out_offset", "<u8"), ("out_pitch", "<u4"), ("image", "<u4"), ("log2_scale", "<u4"),
                             ("reserved", "<u4")])
assert SCALED_JOB_DTYPE.itemsize == 24

SCALES = (1, 2, 4, 8)
_LOG2 = {1: 0, 2: 1, 4: 2, 8: 3}
# MCUs per CTA of bj_pixels_scaled: min(MAX_BLOCKS // blocks_per_mcu, PLANE // (ncomp * 16 * hmax * vmax))
MAX_BLOCKS = 192
PLANE = 6144


def check_scale(scale, allow_auto: bool = False):
    """The scale argument of decode_batch / decode_stream (1, 2, 4, 8) or decode_to_tensor (also "auto")."""
    if allow_auto and isinstance(scale, str) and scale == "auto":
        return scale
    if isinstance(scale, (bool, np.bool_)) or not isinstance(scale, (int, np.integer)) or int(scale) not in SCALES:
        raise ValueError(f"scale must be one of 1, 2, 4, 8{' or auto' if allow_auto else ''}, got {scale!r}")
    return int(scale)


def per_image(scales, n: int) -> np.ndarray:
    """int64 array of n scales from one scale or a sequence of them."""
    if isinstance(scales, (int, np.integer)):
        return np.full(n, check_scale(scales), dtype=np.int64)
    sc = np.asarray(scales, dtype=np.int64).reshape(-1)
    if len(sc) != n or not np.isin(sc, SCALES).all():
        raise ValueError(f"need {n} scales out of 1, 2, 4, 8")
    return sc


class OutputLayout:
    """Where each image of a batch lies in the batch's uint8 output buffer: byte offset, pitch, size, channels.
    out_offsets / out_shapes / out_bytes have the meaning of the BatchGeometry attributes of the same names."""

    def __init__(self, offsets, pitches, widths, heights, channels):
        self.offsets = np.asarray(offsets, dtype=np.int64)
        self.pitches = np.asarray(pitches, dtype=np.int64)
        self.widths = np.asarray(widths, dtype=np.int64)
        self.heights = np.asarray(heights, dtype=np.int64)
        self.channels = np.asarray(channels, dtype=np.int64)
        self.out_offsets = self.offsets.tolist()
        self.out_shapes = [(h, w, 3) if c == 3 else (h, w)
                           for h, w, c in zip(self.heights.tolist(), self.widths.tolist(), self.channels.tolist())]
        ends = self.offsets + self.heights * self.pitches
        self.out_bytes = int(ends.max()) if len(ends) else 0

    @classmethod
    def from_geometry(cls, geom) -> "OutputLayout":
        """The full-size layout bj_pixels writes from a planner's records."""
        rec = geom.images
        return cls(rec["out_offset"], rec["out_pitch"], rec["width"], rec["height"], np.where(rec["ncomp"] == 3, 3, 1))

    @classmethod
    def scaled(cls, images: np.ndarray, scales: np.ndarray) -> "OutputLayout":
        """Images of the given bj_image records at per-image scales, back to back, every start 16-byte aligned."""
        s = np.asarray(scales, dtype=np.int64)
        w = -(-images["width"].astype(np.int64) // s)
        h = -(-images["height"].astype(np.int64) // s)
        return cls.packed(w, h, np.where(images["ncomp"] == 3, 3, 1))

    @classmethod
    def packed(cls, widths, heights, channels) -> "OutputLayout":
        """Images of the given sizes back to back, rows unpadded, every start 16-byte aligned."""
        w, h = np.asarray(widths, dtype=np.int64), np.asarray(heights, dtype=np.int64)
        ch = np.asarray(channels, dtype=np.int64)
        pitch = w * ch
        padded = (h * pitch + 15) & ~15
        offsets = np.zeros(len(w), dtype=np.int64)
        if len(w) > 1:
            np.cumsum(padded[:-1], out=offsets[1:])
        return cls(offsets, pitch, w, h, ch)


def scaled_strip_mcus(images: np.ndarray) -> np.ndarray:
    """MCUs per CTA of bj_pixels_scaled per image."""
    bpm = images["blocks_per_mcu"].astype(np.int64)
    plane = images["ncomp"].astype(np.int64) * 16 * images["hmax"].astype(np.int64) * images["vmax"].astype(np.int64)
    return np.minimum(MAX_BLOCKS // bpm, PLANE // plane)


def scaled_strips(images: np.ndarray) -> np.ndarray:
    """CTAs of bj_pixels_scaled per image: mcus_y * ceil(mcus_x / MCUs per CTA)."""
    return images["mcus_y"].astype(np.int64) * -(-images["mcus_x"].astype(np.int64) // scaled_strip_mcus(images))


def auto_scales(widths, heights, roi, size) -> np.ndarray:
    """decode_to_tensor(scale="auto"): per image the largest s in (1, 2, 4, 8) whose roi box, taken on the image
    decoded at 1/s, is still at least size = (h, w): never upscale what the full decode would have downscaled (the
    rule of PIL's draft())."""
    from .tensor_out import pixel_boxes
    W = np.asarray(widths, dtype=np.int64)
    H = np.asarray(heights, dtype=np.int64)
    h, w = size
    best = np.ones(len(W), dtype=np.int64)
    for s in SCALES[1:]:
        b = pixel_boxes(roi, -(-W // s), -(-H // s), size)
        best = np.where((b[:, 2] - b[:, 0] >= w) & (b[:, 3] - b[:, 1] >= h), s, best)
    return best


_BOUND = False


def _bind():
    global _BOUND
    L = _native.lib()
    if not _BOUND:
        vp = ctypes.c_void_p
        L.bj_pixels_scaled.restype = ctypes.c_int
        L.bj_pixels_scaled.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
        if L.bj_sizeof(2) != SCALED_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_scaled_job layout mismatch between Python and libb200jpeg.so")
        _BOUND = True
    return L


def upload(a: np.ndarray, device) -> torch.Tensor:
    """Asynchronous copy of a small structured array on the current stream (the pinned block is kept by the
    allocator until the copy has completed)."""
    staged = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
    staged.numpy()[:] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    d = torch.empty(a.nbytes, dtype=torch.uint8, device=device)
    d.copy_(staged, non_blocking=True)
    return d


def launch(dg, coef: torch.Tensor, scales, stream: torch.cuda.Stream):
    """Decode the pixels of one planned batch (stages.DeviceGeometry dg, coefficient buffer coef) at per-image scales
    on `stream`: bj_pixels_scaled for the images with s > 1, and bj_pixels over a copy of the records of the images
    with s = 1 whose out_offset / out_pitch point into the same output.  Returns (output buffer, OutputLayout)."""
    L = _bind()
    g = dg.geom
    rec = g.images
    sc = per_image(scales, len(rec))
    lay = OutputLayout.scaled(rec, sc)
    big = np.nonzero(sc > 1)[0]
    one = np.nonzero(sc == 1)[0]
    with torch.cuda.device(dg.device), torch.cuda.stream(stream):
        out = torch.empty(max(lay.out_bytes, 16), dtype=torch.uint8, device=dg.device)
        if len(big):
            jobs = np.zeros(len(big), dtype=SCALED_JOB_DTYPE)
            jobs["out_offset"] = lay.offsets[big]
            jobs["out_pitch"] = lay.pitches[big]
            jobs["image"] = big
            jobs["log2_scale"] = [_LOG2[int(s)] for s in sc[big]]
            max_strips = int(scaled_strips(rec[big]).max())
            dev_jobs = upload(jobs, dg.device)
            _native.check(L.bj_pixels_scaled(dg.images.data_ptr(), dev_jobs.data_ptr(), len(big), max_strips,
                                             coef.data_ptr(), dg.qtabs.data_ptr(), out.data_ptr(), stream.cuda_stream),
                          "bj_pixels_scaled")
        if len(one):
            sub = rec[one].copy()
            sub["out_offset"] = lay.offsets[one]
            sub["out_pitch"] = lay.pitches[one]
            max_strips = int((sub["strips_per_row"].astype(np.int64) * sub["mcus_y"]).max())
            mask = 0
            for lv in np.unique(sub["layout"]):
                mask |= 1 << int(lv)
            dev_sub = upload(sub, dg.device)
            _native.check(L.bj_pixels(dev_sub.data_ptr(), len(one), max_strips, coef.data_ptr(), _native.IN_COEF,
                                      g.total_blocks, dg.qtabs.data_ptr(), dg.table.data_ptr(), out.data_ptr(),
                                      _native.OUT_RGB, mask, None, stream.cuda_stream), "bj_pixels")
    return out, lay
