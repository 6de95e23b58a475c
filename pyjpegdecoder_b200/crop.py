"""Crop decode: only the MCUs under a pixel box, at scale 1, 2, 4 or 8 (bj_pixels_crop, include/b200jpeg.h).

This module owns every decision the crop introduces, so the planners, the entropy stage and the full-image pixel
launches stay as they are: the box checks, the rule file box -> scaled box -> MCU window, the output layout of a batch
of crops, the numpy mirror of bj_crop_job and the launch.

A box (x0, y0, x1, y1) is half-open and in full-resolution pixels of the file, like PIL.Image.crop.  It is clipped to
its image; at scale s the result is the scaled pixels [x0 // s, ceil(min(x1, W) / s)) x [y0 // s, ceil(min(y1, H) / s)),
so decoding with a crop gives exactly the same-scale full decode sliced there.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native
from .scaled import OutputLayout, per_image, scaled_strip_mcus, upload

# numpy mirror of struct bj_crop_job (40 bytes, see include/b200jpeg.h)
CROP_JOB_DTYPE = np.dtype([("out_offset", "<u8"), ("out_pitch", "<u4"), ("image", "<u4"), ("log2_scale", "<u4"),
                           ("x0", "<u4"), ("y0", "<u4"), ("x1", "<u4"), ("y1", "<u4"), ("reserved", "<u4")])
assert CROP_JOB_DTYPE.itemsize == 40

CROP_SCALED = 8   # BJ_CROP_SCALED: bit of bj_pixels_crop's `kinds` for jobs at s > 1
_LOG2 = {1: 0, 2: 1, 4: 2, 8: 3}


def _is_int(v) -> bool:
    return isinstance(v, (int, np.integer)) and not isinstance(v, (bool, np.bool_))


def _check_box(box) -> tuple:
    try:
        items = list(box)
    except TypeError:
        raise ValueError(f"a crop box is (x0, y0, x1, y1) in integer pixels, got {box!r}") from None
    if len(items) != 4 or not all(_is_int(v) for v in items):
        raise ValueError(f"a crop box is (x0, y0, x1, y1) in integer pixels, got {box!r}")
    x0, y0, x1, y1 = (int(v) for v in items)
    if x0 < 0 or y0 < 0:
        raise ValueError(f"a crop box needs x0 >= 0 and y0 >= 0, got {box!r}")
    if x1 <= x0 or y1 <= y0:
        raise ValueError(f"a crop box needs x1 > x0 and y1 > y0, got {box!r}")
    return x0, y0, x1, y1


class Boxes:
    """A checked crop argument: one box for every file, or one box per file.  Called like decode_batch's scale
    functions, (bj_image records of a sub-batch, indices of its files) -> (n, 4) int64 file boxes."""

    def __init__(self, boxes: np.ndarray, per_file: bool):
        self.boxes, self.per_file = boxes, per_file

    def box(self, i: int) -> np.ndarray:
        return self.boxes[i] if self.per_file else self.boxes

    def __call__(self, images, idx) -> np.ndarray:
        if self.per_file:
            return self.boxes[np.asarray(idx, dtype=np.int64)]
        return np.broadcast_to(self.boxes, (len(idx), 4)).copy()


def check_crop(crop, n=None):
    """None, or Boxes for the crop argument of decode_batch / decode_stream / JpegDecoder.  One box is told from a list
    of boxes by its elements' type (integers: one box).  n: the number of files (None: not known, and then per-file
    boxes are an error)."""
    if crop is None:
        return None
    if isinstance(crop, np.ndarray):
        if crop.ndim == 1:
            return Boxes(np.asarray(_check_box(list(crop)), np.int64), False)
        if crop.ndim != 2 or crop.shape[1] != 4:
            raise ValueError(f"crop must be one box (x0, y0, x1, y1) or an (n, 4) array of boxes, got shape {crop.shape}")
        if crop.dtype.kind not in "iu":
            raise ValueError(f"crop boxes need an integer dtype, got {crop.dtype}")
        items = [tuple(int(v) for v in b) for b in crop]
    else:
        try:
            items = list(crop)
        except TypeError:
            raise ValueError(f"crop must be None, one box (x0, y0, x1, y1) or one box per file, got {crop!r}") from None
        if items and all(isinstance(v, (int, float, np.integer, np.floating, bool, np.bool_)) for v in items):
            return Boxes(np.asarray(_check_box(items), np.int64), False)
    if n is None:
        raise ValueError("per-file crop boxes need a sized sequence of files")
    if len(items) != n:
        raise ValueError(f"crop has {len(items)} boxes for {n} files")
    return Boxes(np.asarray([_check_box(b) for b in items], np.int64).reshape(n, 4), True)


def outside(boxes, widths, heights) -> np.ndarray:
    """Per image: the box lies entirely outside the image (x0 >= W or y0 >= H)."""
    b = np.asarray(boxes, dtype=np.int64).reshape(-1, 4)
    return (b[:, 0] >= np.asarray(widths, np.int64)) | (b[:, 1] >= np.asarray(heights, np.int64))


def outside_error(box, width: int, height: int) -> ValueError:
    x0, y0, x1, y1 = (int(v) for v in box)
    return ValueError(f"crop box ({x0}, {y0}, {x1}, {y1}) lies outside the {width} x {height} image")


def scaled_boxes(boxes, widths, heights, scales) -> np.ndarray:
    """(n, 4) boxes in pixels of the images decoded at 1/s: the file boxes clipped to their images, then
    [x0 // s, ceil(x1 / s)) x [y0 // s, ceil(y1 / s)).  Boxes outside their image raise ValueError."""
    b = np.asarray(boxes, dtype=np.int64).reshape(-1, 4)
    W, H = np.asarray(widths, np.int64), np.asarray(heights, np.int64)
    s = np.asarray(scales, dtype=np.int64)
    bad = np.nonzero(outside(b, W, H))[0]
    if len(bad):
        i = int(bad[0])
        raise outside_error(b[i], W[i], H[i])
    x1, y1 = np.minimum(b[:, 2], W), np.minimum(b[:, 3], H)
    return np.stack([b[:, 0] // s, b[:, 1] // s, -(-x1 // s), -(-y1 // s)], 1)


def windows(sboxes, hmax, vmax, scales) -> np.ndarray:
    """(n, 4) MCU windows [mx0, mx1) x [my0, my1) of scaled boxes: every MCU the box touches (an MCU is 8 hmax / s by
    8 vmax / s pixels at scale s)."""
    b = np.asarray(sboxes, dtype=np.int64).reshape(-1, 4)
    s = np.asarray(scales, dtype=np.int64)
    mw = 8 * np.asarray(hmax, np.int64) // s
    mh = 8 * np.asarray(vmax, np.int64) // s
    return np.stack([b[:, 0] // mw, b[:, 1] // mh, -(-b[:, 2] // mw), -(-b[:, 3] // mh)], 1)


def layout(images: np.ndarray, sboxes) -> OutputLayout:
    """The crops of the given bj_image records, back to back, every start 16-byte aligned."""
    b = np.asarray(sboxes, dtype=np.int64).reshape(-1, 4)
    return OutputLayout.packed(b[:, 2] - b[:, 0], b[:, 3] - b[:, 1], np.where(images["ncomp"] == 3, 3, 1))


def file_boxes(crops, images: np.ndarray) -> np.ndarray:
    """The (n, 4) file boxes of a planned batch from decode_batch_on_device's crops (an array, or a function of the
    bj_image records); a box outside its image raises ValueError."""
    b = crops(images) if callable(crops) else crops
    b = np.broadcast_to(np.asarray(b, dtype=np.int64), (len(images), 4))
    bad = np.nonzero(outside(b, images["width"], images["height"]))[0]
    if len(bad):
        i = int(bad[0])
        raise outside_error(b[i], int(images["width"][i]), int(images["height"][i]))
    return b


_BOUND = False


def _bind():
    global _BOUND
    L = _native.lib()
    if not _BOUND:
        vp = ctypes.c_void_p
        L.bj_pixels_crop.restype = ctypes.c_int
        L.bj_pixels_crop.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_uint64, vp, vp, vp,
                                     ctypes.c_uint32, vp, vp]
        if L.bj_sizeof(3) != CROP_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_crop_job layout mismatch between Python and libb200jpeg.so")
        _BOUND = True
    return L


def jobs_for(rec: np.ndarray, boxes, scales):
    """(bj_crop_job array, OutputLayout, max_strips, kinds) for file boxes of the images `rec` at per-image scales."""
    sc = np.asarray(scales, dtype=np.int64)
    sb = scaled_boxes(boxes, rec["width"], rec["height"], sc)
    lay = layout(rec, sb)
    win = windows(sb, rec["hmax"], rec["vmax"], sc)
    strip = np.where(sc == 1, rec["strip_mcus"].astype(np.int64), scaled_strip_mcus(rec))
    strips = (win[:, 3] - win[:, 1]) * -(-(win[:, 2] - win[:, 0]) // strip)
    jobs = np.zeros(len(rec), dtype=CROP_JOB_DTYPE)
    jobs["out_offset"] = lay.offsets
    jobs["out_pitch"] = lay.pitches
    jobs["image"] = np.arange(len(rec))
    jobs["log2_scale"] = [_LOG2[int(s)] for s in sc]
    jobs["x0"], jobs["y0"], jobs["x1"], jobs["y1"] = sb[:, 0], sb[:, 1], sb[:, 2], sb[:, 3]
    kinds = 0
    for lv in np.unique(rec["layout"][sc == 1]):
        kinds |= 1 << int(lv)
    if (sc > 1).any():
        kinds |= CROP_SCALED
    return jobs, lay, int(strips.max()), kinds


def launch(dg, coef: torch.Tensor, scales, boxes, stream: torch.cuda.Stream):
    """Decode the pixels under each image's file box of one planned batch (stages.DeviceGeometry dg, coefficient
    buffer coef) at per-image scales on `stream`, with one bj_pixels_crop call.  Returns (output buffer, OutputLayout)."""
    L = _bind()
    g = dg.geom
    rec = g.images
    jobs, lay, max_strips, kinds = jobs_for(rec, boxes, per_image(scales, len(rec)))
    with torch.cuda.device(dg.device), torch.cuda.stream(stream):
        out = torch.empty(max(lay.out_bytes, 16), dtype=torch.uint8, device=dg.device)
        dev_jobs = upload(jobs, dg.device)
        _native.check(L.bj_pixels_crop(dg.images.data_ptr(), dev_jobs.data_ptr(), len(jobs), max_strips,
                                       coef.data_ptr(), g.total_blocks, dg.qtabs.data_ptr(), dg.table.data_ptr(),
                                       out.data_ptr(), kinds, None, stream.cuda_stream), "bj_pixels_crop")
    return out, lay
