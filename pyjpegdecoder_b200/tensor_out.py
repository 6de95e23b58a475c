"""decode_to_tensor: decode a batch of files straight into one resized, normalised (N, 3, h, w) device tensor.

The data-loader end of the pipeline: what a training or inference loop feeds a model.  Files are decoded by the
same batch / streaming pipeline as decode_batch; each decoded sub-batch is resized by one bj_resize launch
(csrc/bj_resize.cu: antialiased bilinear, like torch's antialiased interpolate) or one bj_resize_pil launch
(csrc/bj_resize_pil.cu: Pillow's Image.resize, bit for bit) into its slots of the output tensor, after which its
full-size RGB pixels go back to the allocator.  Memory therefore stays bounded by the sub-batches in flight plus
the output, whatever the number of files.
"""
from __future__ import annotations

import ctypes
import math
from pathlib import Path
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _native

# numpy mirror of struct bj_resize_job (40 bytes, see include/b200jpeg.h)
RESIZE_JOB_DTYPE = np.dtype([
    ("src_offset", "<u8"), ("src_pitch", "<u4"), ("channels", "<u4"),
    ("x0", "<u4"), ("y0", "<u4"), ("x1", "<u4"), ("y1", "<u4"),
    ("dst_index", "<u4"), ("reserved", "<u4"),
])
assert RESIZE_JOB_DTYPE.itemsize == 40

# numpy mirror of struct bj_resize_pil_job (56 bytes, see include/b200jpeg.h)
RESIZE_PIL_JOB_DTYPE = np.dtype([
    ("src_offset", "<u8"), ("src_pitch", "<u4"), ("channels", "<u4"),
    ("x0", "<u4"), ("y0", "<u4"), ("x1", "<u4"), ("y1", "<u4"),
    ("dst_index", "<u4"), ("virt_w", "<u4"), ("virt_h", "<u4"), ("win_x", "<u4"), ("win_y", "<u4"),
    ("reserved", "<u4"),
])
assert RESIZE_PIL_JOB_DTYPE.itemsize == 56

# largest virt_w / virt_h of a bj_resize_pil_job
VIRT_MAX = 2 ** 31 - 1

# resample= of decode_to_tensor -> the filter argument of bj_resize_pil (None: bj_resize)
RESAMPLES = {"torch": None, "pil-bilinear": 0, "pil-bicubic": 1}


class ResizeParams(ctypes.Structure):
    """struct bj_resize_params"""
    _fields_ = [("out_h", ctypes.c_uint32), ("out_w", ctypes.c_uint32), ("dtype", ctypes.c_uint32),
                ("channels_last", ctypes.c_uint32), ("a", ctypes.c_float * 3), ("b", ctypes.c_float * 3)]


DTYPES = {torch.uint8: 0, torch.float16: 1, torch.bfloat16: 2, torch.float32: 3}

Source = Union[str, Path, bytes, bytearray, memoryview]


def _bind():
    L = _native.lib()
    if not getattr(L, "_resize_bound", False):
        L.bj_resize.restype = ctypes.c_int
        L.bj_resize.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                ctypes.POINTER(ResizeParams), ctypes.c_void_p]
        L.bj_resize_pil.restype = ctypes.c_int
        L.bj_resize_pil.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.POINTER(ResizeParams), ctypes.c_int, ctypes.c_void_p]
        if L.bj_sizeof(1) != RESIZE_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_resize_job layout mismatch between Python and libb200jpeg.so")
        if L.bj_sizeof(4) != RESIZE_PIL_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_resize_pil_job layout mismatch between Python and "
                                             "libb200jpeg.so")
        L._resize_bound = True
    return L


# ---- argument checks and the host-side box rule (no device involved) --------------------------------------------

def _check_size(size) -> Tuple[int, int]:
    try:
        h, w = (int(size[0]), int(size[1])) if len(size) == 2 else (None, None)
    except TypeError:
        h = w = None
    if h is None or h < 1 or w < 1 or h > 65535 or w > 65535:
        raise ValueError(f"size must be (h, w) with 1 <= h, w <= 65535, got {size!r}")
    return h, w


def _check_box(box) -> Tuple[float, float, float, float]:
    try:
        x0, y0, x1, y1 = (float(v) for v in box)
    except (TypeError, ValueError):
        raise ValueError(f"a roi box is (x0, y0, x1, y1), got {box!r}") from None
    if not (0.0 <= x0 < x1 <= 1.0 and 0.0 <= y0 < y1 <= 1.0):
        raise ValueError(f"a roi box needs 0 <= x0 < x1 <= 1 and 0 <= y0 < y1 <= 1, got {box!r}")
    return x0, y0, x1, y1


def _check_roi(roi, n: int):
    """None, "center", one (4,) float64 box, or an (n, 4) float64 array of boxes."""
    if roi is None:
        return None
    if isinstance(roi, str):
        if roi != "center":
            raise ValueError(f"roi must be None, 'center', one box or one box per file, got {roi!r}")
        return roi
    try:
        items = list(roi)
    except TypeError:
        raise ValueError(f"roi must be None, 'center', one box or one box per file, got {roi!r}") from None
    if len(items) == 4 and all(isinstance(v, (int, float, np.integer, np.floating)) for v in items):
        return np.asarray(_check_box(items), dtype=np.float64)
    if len(items) != n:
        raise ValueError(f"roi has {len(items)} boxes for {n} files")
    return np.asarray([_check_box(b) for b in items], dtype=np.float64).reshape(n, 4)


def _fold_norm(dtype, mean, std) -> Tuple[List[float], List[float]]:
    """Per-channel (a, b) with value = v * a + b for v on the 0..255 scale."""
    if dtype not in DTYPES:
        raise ValueError(f"dtype must be one of uint8, float16, bfloat16, float32, got {dtype}")
    if (mean is None) != (std is None):
        raise ValueError("mean and std go together")
    if dtype == torch.uint8:
        if mean is not None:
            raise ValueError("mean / std need a floating-point dtype")
        return [1.0] * 3, [0.0] * 3
    if mean is None:
        return [1.0 / 255.0] * 3, [0.0] * 3
    m = [float(v) for v in mean]
    s = [float(v) for v in std]
    if len(m) != 3 or len(s) != 3:
        raise ValueError("mean and std need 3 values (R, G, B)")
    if any(v == 0.0 or not math.isfinite(v) for v in s):
        raise ValueError("std values must be finite and non-zero")
    return [1.0 / (255.0 * sv) for sv in s], [-mv / sv for mv, sv in zip(m, s)]


def _check_resample(resample, resize, roi, size: Tuple[int, int]) -> Optional[int]:
    """resample / resize of decode_to_tensor: (resample, resize, roi and size checked) -> the resize= short side or
    None."""
    if not isinstance(resample, str) or resample not in RESAMPLES:
        raise ValueError(f"resample must be one of {', '.join(map(repr, RESAMPLES))}, got {resample!r}")
    if resize is None:
        return None
    if RESAMPLES[resample] is None:
        raise ValueError("resize= needs resample='pil-bilinear' or 'pil-bicubic'")
    if roi is not None:
        raise ValueError("resize= resizes the whole image; it takes roi=None")
    if isinstance(resize, bool) or not isinstance(resize, (int, np.integer)) or not 1 <= resize <= 65535:
        raise ValueError(f"resize must be an int in 1..65535, got {resize!r}")
    if resize < max(size):
        # the resized short side is `resize`, and either side of an image may be the short one
        raise ValueError(f"resize={resize} gives images smaller than size={tuple(size)}: it must be >= {max(size)}")
    return int(resize)


def resize_geometry(widths, heights, r: int, size: Tuple[int, int]):
    """torchvision's Resize(r) then CenterCrop(size) on images of the given sizes: (virt_w, virt_h, win_x, win_y) int64
    arrays.  The short side becomes r and the long side int(r * long / short) (a square image's width counts as its
    short side); the crop starts at int(round((virt - out) / 2)) with Python's round (half to even)."""
    W = np.asarray(widths, dtype=np.int64)
    H = np.asarray(heights, dtype=np.int64)
    h, w = size
    portrait = W <= H
    short, long = np.where(portrait, W, H), np.where(portrait, H, W)
    new_long = np.floor(r * long / short).astype(np.int64)    # r * long < 2^53: numpy's division is Python's
    vw = np.where(portrait, r, new_long)
    vh = np.where(portrait, new_long, r)
    return vw, vh, np.round((vw - w) / 2.0).astype(np.int64), np.round((vh - h) / 2.0).astype(np.int64)


def pixel_boxes(roi, widths, heights, size: Tuple[int, int]) -> np.ndarray:
    """(n, 4) int64 pixel boxes (px0, py0, px1, py1) of images of the given sizes for a checked roi (_check_roi)."""
    W = np.asarray(widths, dtype=np.int64)
    H = np.asarray(heights, dtype=np.int64)
    n = len(W)
    if roi is None:
        return np.stack([np.zeros(n, np.int64), np.zeros(n, np.int64), W, H], 1)
    h, w = size
    if isinstance(roi, str):                  # "center": largest centred box of the output's aspect ratio
        wide = W * h >= H * w
        bw = np.where(wide, np.maximum(1, np.floor(H * w / h + 0.5)).astype(np.int64), W)
        bh = np.where(wide, H, np.maximum(1, np.floor(W * h / w + 0.5)).astype(np.int64))
        x0, y0 = (W - bw) // 2, (H - bh) // 2
        return np.stack([x0, y0, x0 + bw, y0 + bh], 1)
    b = np.broadcast_to(roi, (n, 4))
    Wf, Hf = W.astype(np.float64), H.astype(np.float64)

    def axis(lo, hi, size_):
        p0 = np.minimum(np.floor(lo * size_ + 0.5), size_ - 1)
        p1 = np.maximum(p0 + 1, np.minimum(size_, np.floor(hi * size_ + 0.5)))
        return p0.astype(np.int64), p1.astype(np.int64)

    x0, x1 = axis(b[:, 0], b[:, 2], Wf)
    y0, y1 = axis(b[:, 1], b[:, 3], Hf)
    return np.stack([x0, y0, x1, y1], 1)


# ---- device side -------------------------------------------------------------------------------------------------

_RESIZE_STREAMS = {}


def _resize_stream(dev: torch.device) -> torch.cuda.Stream:
    """One resize stream per device, created once (the caching allocator keeps freed blocks per stream)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _RESIZE_STREAMS:
        _RESIZE_STREAMS[key] = torch.cuda.Stream(torch.device("cuda", key))
    return _RESIZE_STREAMS[key]


class _Resizer:
    """Enqueues bj_resize (filter None) or bj_resize_pil for decoded sub-batches into the slots of one output tensor, on
    the resize stream.  resize: the resize= short side (bj_resize_pil only) or None."""

    def __init__(self, out: torch.Tensor, roi, size, dtype, a, b, channels_last: bool, filter_=None, resize=None):
        self.L = _bind()
        self.out, self.roi, self.size = out, roi, size
        self.filter, self.resize_to = filter_, resize
        self.dev = out.device
        self.stream = _resize_stream(self.dev)
        self.params = ResizeParams(size[0], size[1], DTYPES[dtype], int(channels_last), (ctypes.c_float * 3)(*a),
                                   (ctypes.c_float * 3)(*b))
        # the output was allocated (and maybe zeroed) on the caller's stream
        self.stream.wait_stream(torch.cuda.current_stream(self.dev))

    def resize(self, batch, items: Sequence[Tuple[int, int]], after: torch.cuda.Stream) -> None:
        """items: (index of the image in the batch, slot in the output).  `after`: the stream the batch was decoded on
        (None: its pixels are complete already)."""
        if not items:
            return
        lay = batch.layout                               # full size or scaled: where each decoded image lies
        idx = np.fromiter((i for i, _ in items), dtype=np.int64, count=len(items))
        W, H = lay.widths[idx], lay.heights[idx]
        roi = self.roi
        if isinstance(roi, np.ndarray) and roi.ndim == 2:
            roi = roi[np.fromiter((s for _, s in items), dtype=np.int64, count=len(items))]
        boxes = pixel_boxes(roi, W, H, self.size)
        jobs = np.zeros(len(items), dtype=RESIZE_JOB_DTYPE if self.filter is None else RESIZE_PIL_JOB_DTYPE)
        jobs["src_offset"] = lay.offsets[idx]
        jobs["src_pitch"] = lay.pitches[idx]
        jobs["channels"] = lay.channels[idx]
        jobs["x0"], jobs["y0"], jobs["x1"], jobs["y1"] = boxes[:, 0], boxes[:, 1], boxes[:, 2], boxes[:, 3]
        jobs["dst_index"] = [s for _, s in items]
        if self.filter is not None:
            if self.resize_to is None:
                jobs["virt_w"], jobs["virt_h"] = self.size[1], self.size[0]
            else:
                vw, vh, wx, wy = resize_geometry(boxes[:, 2] - boxes[:, 0], boxes[:, 3] - boxes[:, 1], self.resize_to,
                                                 self.size)
                too_long = np.flatnonzero(np.maximum(vw, vh) > VIRT_MAX)
                if too_long.size:        # checked before the launch: the kernel writes nothing for such a job
                    k = int(too_long[0])
                    raise ValueError(f"resize={self.resize_to} makes the {int(boxes[k, 2] - boxes[k, 0])} x "
                                     f"{int(boxes[k, 3] - boxes[k, 1])} image {int(max(vw[k], vh[k]))} pixels long, "
                                     f"more than {VIRT_MAX}")
                jobs["virt_w"], jobs["virt_h"], jobs["win_x"], jobs["win_y"] = vw, vh, wx, wy
        staged = torch.empty(jobs.nbytes, dtype=torch.uint8, pin_memory=True)
        staged.numpy()[:] = jobs.view(np.uint8)
        s = self.stream
        with torch.cuda.device(self.dev), torch.cuda.stream(s):
            if after is not None:
                s.wait_stream(after)
            dev_jobs = torch.empty(jobs.nbytes, dtype=torch.uint8, device=self.dev)
            dev_jobs.copy_(staged, non_blocking=True)    # the pinned block is kept until this copy has completed
            if self.filter is None:
                _native.check(self.L.bj_resize(dev_jobs.data_ptr(), len(items), batch.out.data_ptr(),
                                               self.out.data_ptr(), ctypes.byref(self.params), s.cuda_stream),
                              "bj_resize")
            else:
                _native.check(self.L.bj_resize_pil(dev_jobs.data_ptr(), len(items), batch.out.data_ptr(),
                                                   self.out.data_ptr(), ctypes.byref(self.params), self.filter,
                                                   s.cuda_stream), "bj_resize_pil")
            batch.out.record_stream(s)                   # the RGB buffer may be reused only after the resize has read it

    def finish(self) -> None:
        torch.cuda.current_stream(self.dev).wait_stream(self.stream)


def decode_to_tensor(files: Sequence[Source], size=(224, 224), *, roi=None, dtype=torch.float32, mean=None, std=None,
                     channels_last: bool = False, device=None, chunk: Optional[int] = None, on_error: str = "raise",
                     scale=1, compat: str = "reference", resample: str = "torch", resize: Optional[int] = None):
    """Decode `files` (paths or bytes, like decode_batch) into ONE device tensor of shape (N, 3, h, w), (h, w) = size.

    Each image's region `roi` is resized like torch.nn.functional.interpolate(mode="bilinear", antialias=True,
    align_corners=False) (torchvision's Resize); greyscale files give three equal channels.
      roi       None (whole image), one normalised box (x0, y0, x1, y1) for every file, one box per file, or
                "center" (largest centred box with the output's aspect ratio: Resize + CenterCrop).  Boxes are
                rounded to whole pixels on the host.
      dtype     uint8, float16, bfloat16 or float32.  Float values are (v / 255 - mean[c]) / std[c], or v / 255
                without mean / std; uint8 values are the resized 0..255 values rounded to nearest even.
      channels_last  the same values in torch.channels_last memory format.
      chunk     files per decoded sub-batch (decode_batch's default when None); more than 1.5 x chunk files flow
                through decode_stream, so device memory stays bounded whatever the number of files.
      on_error  "raise", or "return": returns (tensor, errors) with errors[i] None or the exception of file i, whose
                slot is zero.
      scale     1, 2, 4 or 8: the files are decoded at 1/scale of their size in the DCT domain (decode_batch(scale=))
                and the roi is taken on the decoded image; "auto": per file the largest of these whose roi box is
                still at least (h, w), so nothing is upscaled that the full decode would have downscaled.
      compat    "reference", or "libjpeg-turbo": the resize reads libjpeg-turbo's pixels (Pillow's), scale 1 only
                (decode_batch(compat=)).
      resample  "torch" (the resize above), or "pil-bilinear" / "pil-bicubic": each image's box is resized exactly like
                PIL.Image.resize((w, h), BILINEAR | BICUBIC) of the decoded box (torchvision's resized_crop on a PIL
                image).  uint8 output holds Pillow's bytes; float outputs are v * a[c] + b[c] of those uint8 values v,
                so with compat="libjpeg-turbo" they equal ToTensor() + Normalize() up to fp32 rounding.
      resize    an int r, PIL resamples only, roi=None, r >= max(h, w): torchvision's Resize(r) then CenterCrop(size)
                -- the short side becomes r, the long side int(r * long / short), the crop starts at
                int(round((R - h) / 2)), int(round((C - w) / 2)) -- of which only the cropped window is computed.
                With scale="auto" each file uses the largest scale whose decoded short side is still >= r.
    With a roi, only each file's roi box is decoded (decode_batch(crop=)), taken at the scale the file uses; the
    resize then reads the whole decoded crop, which holds the same bytes as the box of the full decode.
    The caller's current stream is ordered after the work, so the tensor can be used right away."""
    from .decoder import BATCH_CHUNK
    from .scaled import check_scale
    if on_error not in ("raise", "return"):
        raise ValueError("on_error must be 'raise' or 'return'")
    scale = check_scale(scale, allow_auto=True)
    from .ijg import check_compat
    check_compat(compat, scale)
    h, w = _check_size(size)
    a, b = _fold_norm(dtype, mean, std)
    files = list(files)
    n = len(files)
    roi = _check_roi(roi, n)
    resize = _check_resample(resample, resize, roi, (h, w))
    chunk = BATCH_CHUNK if chunk is None else int(chunk)
    if chunk < 1:
        raise ValueError("chunk must be positive")
    scales = None if scale == 1 else scale
    if scale == "auto":
        scales = _AutoScales(roi, (h, w) if resize is None else (resize, resize))
    crops = None if roi is None else _RoiCrops(roi, (h, w), scales)

    from .stages import require_cuda
    dev = require_cuda(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    with torch.cuda.device(dev):
        out = torch.empty((n, 3, h, w), dtype=dtype, device=dev, memory_format=fmt)
        if on_error == "return":
            out.zero_()
        if n == 0:
            return (out, []) if on_error == "return" else out
        rs = _Resizer(out, None if crops is not None else roi, (h, w), dtype, a, b, channels_last, RESAMPLES[resample],
                      resize)
        cur = torch.cuda.current_stream(dev)
        # finish() also runs when a file raises part-way: resizes already enqueued may still be writing into `out`,
        # which the caller's stream must not reuse before they are done
        try:
            if on_error == "return":
                return out, _tolerant(files, rs, dev, chunk, cur, scales, crops, compat)
            if n > chunk + chunk // 2:
                from .loader import _decode_stream
                slot = 0
                for part in _decode_stream(files, chunk, dev, scales=scales, crops=crops, compat=compat):
                    # decode_stream yields a sub-batch after synchronising the stream it was decoded on
                    batch = part[0]._batch
                    rs.resize(batch, [(i, slot + i) for i in range(len(part))], None)
                    slot += len(part)
                    del part, batch                     # the sub-batch's RGB and work buffers go back to the allocator
            else:
                from .decoder import decode_batch
                part = decode_batch(files, device=dev, chunk=chunk, compat=compat, _scales=scales, _crops=crops)
                rs.resize(part[0]._batch, [(i, i) for i in range(n)], cur)
                del part
        finally:
            rs.finish()
    return out


class _AutoScales:
    """scale="auto" of decode_to_tensor as a function of a planned sub-batch: (bj_image records, indices of its files
    among decode_to_tensor's files) -> per-image scales (scaled.auto_scales).  offset: added to the indices, for
    sub-batches whose indices count from a later file."""

    def __init__(self, roi, size, offset: int = 0):
        self.roi, self.size, self.offset = roi, size, offset

    def __call__(self, images, idx):
        from .scaled import auto_scales
        roi = self.roi
        if isinstance(roi, np.ndarray) and roi.ndim == 2:
            roi = roi[np.asarray(idx, dtype=np.int64) + self.offset]
        return auto_scales(images["width"], images["height"], roi, self.size)


class _RoiCrops:
    """decode_to_tensor's roi as crop boxes of a planned sub-batch: (bj_image records, indices of its files among
    decode_to_tensor's files) -> (n, 4) file boxes.  Each is the pixel_boxes box on the image decoded at the file's
    scale s, times s, which decodes to exactly that box (crop.py's rule), so the resize sees today's box size and
    bytes.  scales: None, one scale or a function like _AutoScales; offset as for _AutoScales."""

    def __init__(self, roi, size, scales, offset: int = 0):
        self.roi, self.size, self.scales, self.offset = roi, size, scales, offset

    def __call__(self, images, idx):
        n = len(idx)
        if callable(self.scales):
            s = np.asarray(self.scales(images, idx), dtype=np.int64)
        else:
            s = np.full(n, 1 if self.scales is None else self.scales, dtype=np.int64)
        roi = self.roi
        if isinstance(roi, np.ndarray) and roi.ndim == 2:
            roi = roi[np.asarray(idx, dtype=np.int64) + self.offset]
        W, H = images["width"].astype(np.int64), images["height"].astype(np.int64)
        return pixel_boxes(roi, -(-W // s), -(-H // s), self.size) * s[:, None]


def _tolerant(files: list, rs: _Resizer, dev, chunk: int, cur, scales=None, crops=None, compat="reference") -> list:
    """on_error="return": decode_batch(on_error="return") chunk by chunk, each chunk's good images resized into their
    slots (bad slots keep the zeros the output was created with)."""
    from .decoder import decode_batch
    errors: list = [None] * len(files)
    for c0 in range(0, len(files), chunk):
        sc = _AutoScales(scales.roi, scales.size, c0) if isinstance(scales, _AutoScales) else scales
        cr = None if crops is None else _RoiCrops(crops.roi, crops.size, sc, c0)
        res = decode_batch(files[c0:c0 + chunk], device=dev, chunk=chunk, on_error="return", compat=compat, _scales=sc,
                           _crops=cr)
        groups = {}
        for k, r in enumerate(res):
            if isinstance(r, Exception):
                errors[c0 + k] = r
            else:
                groups.setdefault(id(r._batch), (r._batch, []))[1].append((r._index, c0 + k))
        for batch, items in groups.values():
            rs.resize(batch, items, cur)
        del res, groups
    return errors
