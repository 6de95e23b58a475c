"""decode_to_tensor: decode a batch of files straight into one resized, normalised (N, 3, h, w) device tensor.

The data-loader end of the pipeline: what a training or inference loop feeds a model.  Files are decoded by the
same batch / streaming pipeline as decode_batch; each decoded sub-batch is resized by one bj_resize launch
(csrc/bj_resize.cu: antialiased bilinear, like torchvision's Resize) into its slots of the output tensor, after which
its full-size RGB pixels go back to the allocator.  Memory therefore stays bounded by the sub-batches in flight plus
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
        if L.bj_sizeof(1) != RESIZE_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_resize_job layout mismatch between Python and libb200jpeg.so")
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
    """Enqueues bj_resize for decoded sub-batches into the slots of one output tensor, on the resize stream."""

    def __init__(self, out: torch.Tensor, roi, size, dtype, a, b, channels_last: bool):
        self.L = _bind()
        self.out, self.roi, self.size = out, roi, size
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
        jobs = np.zeros(len(items), dtype=RESIZE_JOB_DTYPE)
        jobs["src_offset"] = lay.offsets[idx]
        jobs["src_pitch"] = lay.pitches[idx]
        jobs["channels"] = lay.channels[idx]
        jobs["x0"], jobs["y0"], jobs["x1"], jobs["y1"] = boxes[:, 0], boxes[:, 1], boxes[:, 2], boxes[:, 3]
        jobs["dst_index"] = [s for _, s in items]
        staged = torch.empty(jobs.nbytes, dtype=torch.uint8, pin_memory=True)
        staged.numpy()[:] = jobs.view(np.uint8)
        s = self.stream
        with torch.cuda.device(self.dev), torch.cuda.stream(s):
            if after is not None:
                s.wait_stream(after)
            dev_jobs = torch.empty(jobs.nbytes, dtype=torch.uint8, device=self.dev)
            dev_jobs.copy_(staged, non_blocking=True)    # the pinned block is kept until this copy has completed
            _native.check(self.L.bj_resize(dev_jobs.data_ptr(), len(items), batch.out.data_ptr(), self.out.data_ptr(),
                                           ctypes.byref(self.params), s.cuda_stream), "bj_resize")
            batch.out.record_stream(s)                   # the RGB buffer may be reused only after the resize has read it

    def finish(self) -> None:
        torch.cuda.current_stream(self.dev).wait_stream(self.stream)


def decode_to_tensor(files: Sequence[Source], size=(224, 224), *, roi=None, dtype=torch.float32, mean=None, std=None,
                     channels_last: bool = False, device=None, chunk: Optional[int] = None, on_error: str = "raise",
                     scale=1):
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
    The caller's current stream is ordered after the work, so the tensor can be used right away."""
    from .decoder import BATCH_CHUNK
    from .scaled import check_scale
    if on_error not in ("raise", "return"):
        raise ValueError("on_error must be 'raise' or 'return'")
    scale = check_scale(scale, allow_auto=True)
    h, w = _check_size(size)
    a, b = _fold_norm(dtype, mean, std)
    files = list(files)
    n = len(files)
    roi = _check_roi(roi, n)
    chunk = BATCH_CHUNK if chunk is None else int(chunk)
    if chunk < 1:
        raise ValueError("chunk must be positive")
    scales = None if scale == 1 else scale
    if scale == "auto":
        scales = _AutoScales(roi, (h, w))

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
        rs = _Resizer(out, roi, (h, w), dtype, a, b, channels_last)
        cur = torch.cuda.current_stream(dev)
        # finish() also runs when a file raises part-way: resizes already enqueued may still be writing into `out`,
        # which the caller's stream must not reuse before they are done
        try:
            if on_error == "return":
                return out, _tolerant(files, rs, dev, chunk, cur, scales)
            if n > chunk + chunk // 2:
                from .loader import _decode_stream
                slot = 0
                for part in _decode_stream(files, chunk, dev, scales=scales):
                    # decode_stream yields a sub-batch after synchronising the stream it was decoded on
                    batch = part[0]._batch
                    rs.resize(batch, [(i, slot + i) for i in range(len(part))], None)
                    slot += len(part)
                    del part, batch                     # the sub-batch's RGB and work buffers go back to the allocator
            else:
                from .decoder import decode_batch
                part = decode_batch(files, device=dev, chunk=chunk, _scales=scales)
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


def _tolerant(files: list, rs: _Resizer, dev, chunk: int, cur, scales=None) -> list:
    """on_error="return": decode_batch(on_error="return") chunk by chunk, each chunk's good images resized into their
    slots (bad slots keep the zeros the output was created with)."""
    from .decoder import decode_batch
    errors: list = [None] * len(files)
    for c0 in range(0, len(files), chunk):
        sc = _AutoScales(scales.roi, scales.size, c0) if isinstance(scales, _AutoScales) else scales
        res = decode_batch(files[c0:c0 + chunk], device=dev, chunk=chunk, on_error="return", _scales=sc)
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
