"""Drop-in entry point: same class name, constructor and result attributes as the reference's
JpegDecoder (jpeg_decoder.py:27-110), decoding on a B200 through libb200jpeg.so.

Differences by design: never opens a GUI (the reference calls self.show() at :1389), prints nothing
unless verbose=True, accepts str / bytes / Path, and keeps the pixels on the device until
`image_array` is read.  There is no CPU fallback.
"""
from __future__ import annotations

from collections import namedtuple
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch

from .huffman import canonical_codes
from .layout import ZIGZAG_UV
from .parser import ParsedJpeg, parse_jpeg
from .pipeline import DecodedBatch, decode_batch_on_device

# containers of the reference (:24-25)
ColorComponent = namedtuple("ColorComponent", "name order vertical_sampling horizontal_sampling quantization_table_id repeat shape")
HuffmanTable = namedtuple("HuffmanTable", "dc ac")

_NAMES = ("Y", "Cb", "Cr")


def _read(file: Union[str, Path, bytes, bytearray, memoryview]) -> bytes:
    if isinstance(file, (bytes, bytearray, memoryview)):
        return bytes(file)
    with open(file, "rb") as f:
        return f.read()


class JpegDecoder:
    """JpegDecoder(file) decodes in the constructor, like the reference (:29-110).

    Result attributes mirror the reference: image_array (uint8, (width, height, 3) or (width, height)),
    image_width, image_height, scan_mode, color_components, sample_shape, huffman_tables,
    quantization_tables, restart_interval, scan_count, scan_amount, array_width/height/depth,
    file_size, file_path.  `image_tensor` is the device tensor in (H, W, 3) layout.
    """

    def __init__(self, file: Union[str, Path, bytes], device: Optional[Union[str, torch.device]] = None,
                 verbose: bool = False, parsed: Optional[ParsedJpeg] = None, _batch: Optional[DecodedBatch] = None,
                 _index: int = 0, scale: int = 1, crop=None, compat: str = "reference"):
        """scale, crop and compat as for decode_batch."""
        if isinstance(file, (bytes, bytearray, memoryview)):
            self.file_path = None
        else:
            self.file_path = file if isinstance(file, Path) else Path(file)
        if _batch is None:
            data = _read(file)
            self.file_size = len(data)
            p = parsed if parsed is not None else parse_jpeg(data)
            from .crop import check_crop
            from .ijg import check_compat
            from .scaled import check_scale
            scale, crop = check_scale(scale), check_crop(crop, 1)
            check_compat(compat, scale)
            _batch = decode_batch_on_device([data], device=device, parsed=[p], scales=None if scale == 1 else scale,
                                            crops=None if crop is None else crop(None, [0]), compat=compat)
            _index = 0
        self._batch = _batch
        self._index = _index
        self._image_array = None
        if verbose:
            print(f"Decoded {self.image_width} x {self.image_height} {self.scan_mode} image, {self.scan_count} scan(s)")

    # The descriptive attributes of the reference (image_width, scan_mode, color_components, ...) are derived from
    # the parsed headers the first time one of them is read: a batch of thousands of results should not pay for
    # thousands of attribute sets nobody may look at.
    _LAZY = frozenset(("_parsed", "scan_finished", "scan_mode", "image_width", "image_height", "color_components",
                       "sample_shape", "restart_interval", "scan_count", "scan_amount", "array_width", "array_height",
                       "array_depth", "mcu_count_h", "mcu_count_v", "mcu_count", "file_size"))

    def __getattr__(self, name):
        if name in JpegDecoder._LAZY and "_batch" in self.__dict__:
            self._fill()
            return self.__dict__[name]
        raise AttributeError(name)

    def _fill(self) -> None:
        p = self._batch.plan.parsed[self._index]
        d = self.__dict__
        d["_parsed"] = p
        d.setdefault("file_size", p.file_size)
        d["scan_finished"] = p.finished
        d["scan_mode"] = "progressive_dct" if p.progressive else "baseline_dct"
        d["image_width"] = p.width
        d["image_height"] = p.height
        d["color_components"] = {
            c.id: ColorComponent(name=_NAMES[c.order], order=c.order, vertical_sampling=c.v, horizontal_sampling=c.h,
                                 quantization_table_id=c.tq, repeat=c.h * c.v, shape=(8 * c.h, 8 * c.v))
            for c in p.components}
        d["sample_shape"] = (8 * p.hmax, 8 * p.vmax)
        d["restart_interval"] = p.restart_interval
        d["scan_count"] = len(p.scans)
        d["scan_amount"] = p.scan_amount
        d["array_width"], d["array_height"] = p.canvas_size
        d["array_depth"] = p.ncomp
        last = p.scans[-1]
        d["mcu_count_h"], d["mcu_count_v"] = last.mcus_x, last.mcus_y
        d["mcu_count"] = last.mcus_x * last.mcus_y

    # ---- pixels ----------------------------------------------------------------------------------
    @property
    def image_tensor(self) -> torch.Tensor:
        """(H, W, 3) or (H, W) uint8 tensor on the device."""
        return self._batch.images[self._index]

    @property
    def image_array(self) -> np.ndarray:
        """uint8 numpy array shaped like the reference's: (width, height, 3) or (width, height)
        (x-major, jpeg_decoder.py:626, :1373-1386); a transposed view of the (H, W, 3) buffer."""
        if self._image_array is None:
            host_image = getattr(self._batch, "host_image", None)
            host = host_image(self._index) if host_image is not None else None    # decode_batch / decode_stream(to_host=True)
            if host is None:
                host = self.image_tensor.cpu().numpy()
            self._image_array = np.swapaxes(host, 0, 1)
        return self._image_array

    # ---- hand-off to other consumers (SURVEY.md 8f rank 3: the step after the path) -------------------------
    def __dlpack__(self, stream=None):
        """DLPack capsule of the (H, W, 3) / (H, W) uint8 device tensor: zero-copy hand-off to any DLPack consumer
        (torch.from_dlpack, cupy.from_dlpack, jax, ...)."""
        t = self.image_tensor
        return t.__dlpack__(stream=stream) if stream is not None else t.__dlpack__()

    def __dlpack_device__(self):
        return self.image_tensor.__dlpack_device__()

    @property
    def __cuda_array_interface__(self):
        """Numba / CuPy view of the device pixels ((H, W, 3) or (H, W), uint8, C order)."""
        return self.image_tensor.__cuda_array_interface__

    def save(self, path: Union[str, Path, None] = None) -> Path:
        """Write the decoded image with Pillow (the reference's save(), jpeg_decoder.py:1485-1532, minus the Tk file
        dialog): default `<input stem>.png` next to the input file, never overwriting (" (1)", " (2)", ... like the
        reference), PNG when the suffix is not a format Pillow knows.  The pixels make one device->host copy through
        pinned memory.  Returns the path written."""
        from PIL import Image
        if path is None:
            if self.file_path is None:
                raise ValueError("save() needs a path when the decoder was given bytes")
            path = self.file_path.with_suffix(".png")
        path = Path(path)
        stem, count = path.stem, 1
        while path.exists():
            path = path.with_name(f"{stem} ({count}){path.suffix}")
            count += 1
        t = self.image_tensor
        host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t)
        img = Image.fromarray(host.numpy())
        try:
            img.save(path)
        except ValueError:
            path = path.with_suffix(".png")
            count = 1
            while path.exists():
                path = path.with_name(f"{stem} ({count}).png")
                count += 1
            img.save(path, format="png")
        return path

    # ---- tables, in the reference's formats --------------------------------------------------------
    @property
    def quantization_tables(self) -> Dict[int, np.ndarray]:
        """{table id: 8x8 int16 indexed [x, y]} as define_quantization_table stores them (:454-462)."""
        out = {}
        for k, q in self._parsed.qtables.items():
            t = np.zeros((8, 8), np.int16)
            for i, (u, v) in enumerate(ZIGZAG_UV):
                t[u, v] = q[i]
            out[k] = t
        return out

    @property
    def huffman_tables(self) -> Dict[int, Dict[str, int]]:
        """{Tc/Th byte: {bit string: symbol}} as define_huffman_table builds them (:366-377)."""
        out = {}
        for dest, spec in self._parsed.huff_specs.items():
            out[dest] = {bin(code)[2:].rjust(length, "0"): sym for (code, length, sym) in canonical_codes(spec)}
        return out

    def coefficient_planes(self) -> List[np.ndarray]:
        """Quantised DCT coefficients per component, (blocks_v, blocks_h, 64) int16 in zig-zag order."""
        return self._batch.coefficient_grids(self._index)


# files per sub-batch when decode_batch() pipelines a large batch (see loader.decode_stream)
BATCH_CHUNK = 512


def decode_batch(files: Sequence[Union[str, Path, bytes]], device: Optional[Union[str, torch.device]] = None,
                 chunk: Optional[int] = None, on_error: str = "raise", keep_coefficients: bool = False,
                 to_host: bool = False, scale: int = 1, crop=None, compat: str = "reference", _scales=None,
                 _crops=None) -> List[JpegDecoder]:
    """Decode many files and return one JpegDecoder-like object per file (pixels stay on the device until
    `image_array` is read).  Small batches run as ONE device pipeline (one launch sequence for all files); batches
    larger than 1.5 x `chunk` files are cut into sub-batches of `chunk` files that flow through the streaming front
    end (loader.decode_stream): a worker thread gathers, uploads and plans sub-batch k+1 while the GPU decodes
    sub-batch k, so the host work hides behind the device time.

    on_error="raise" (default): the first bad file raises, like the reference's constructor does for its one file.
    on_error="return": nothing is raised for a bad file; its position in the result holds the exception instance
    (NotJpeg / CorruptedJpeg / UnsupportedJpeg) instead of a decoder, and all other files are decoded.

    Large (sub-batched) calls keep only the pixels on the device: the coefficient planes -- as many bytes again -- are
    released as each sub-batch completes unless keep_coefficients=True (`coefficient_planes()` then works on every
    result, at twice the memory: 12.4 MB instead of 6.2 MB per 1080p image).

    to_host=True: the pixels of every sub-batch are also copied to pinned host memory, one transfer per sub-batch
    behind the decode of the next ones; `image_array` (what the reference returns: a numpy array in host memory) is
    then a view of that copy instead of one pageable device->host copy per image.

    scale=2, 4 or 8: every image is decoded at 1/scale of its size in the DCT domain, (ceil(H/s), ceil(W/s), 3), from
    the low-frequency corner of each block (csrc/bj_scaled_math.cuh); image_tensor, image_array, save() and DLPack give
    those pixels, image_width / image_height stay the file's.  _scales: per-image scales, or a function
    (bj_image records of a sub-batch, indices of its files in `files`) -> scales (decode_to_tensor(scale="auto")).

    crop=(x0, y0, x1, y1), one box for every file, or one box per file (a sequence or an (n, 4) integer array): only
    the MCUs under each box are decoded (crop.py).  Boxes are half-open, in full-resolution pixels of the file, and
    clipped to the image; at scale s the result is image_tensor[y0 // s:ceil(y1 / s), x0 // s:ceil(x1 / s)] of the
    same-scale full decode, contiguous.  A box entirely outside its image is a ValueError for that file.  _crops: a
    function like _scales that returns (n, 4) file boxes (decode_to_tensor(roi=)).

    compat="reference" (default): the reference's pixels and coefficients.  compat="libjpeg-turbo": exactly what
    libjpeg-turbo's default decompressor gives (ISLOW IDCT, fancy upsampling, its colour tables; Pillow's Image.open
    pixels), and coefficient_planes() by the T.81 refinement rule; full size only (scale=1), with any crop (ijg.py)."""
    from .crop import check_crop
    from .ijg import check_compat
    from .scaled import check_scale
    if on_error not in ("raise", "return"):
        raise ValueError("on_error must be 'raise' or 'return'")
    scale = check_scale(scale)
    check_compat(compat, scale)
    if _scales is None and scale != 1:
        _scales = scale
    files = list(files)
    if _crops is None:
        _crops = check_crop(crop, len(files))
    if not files:
        return []
    chunk = BATCH_CHUNK if chunk is None else int(chunk)
    if chunk < 1:
        raise ValueError("chunk must be positive")
    if on_error == "return":
        return _decode_batch_tolerant(files, device, chunk, _scales, _crops, compat)
    if len(files) > chunk + chunk // 2:
        from .loader import _decode_stream
        out: List[JpegDecoder] = []
        for part in _decode_stream(files, chunk, device, keep_coefficients, to_host, _scales, _crops, compat):
            out.extend(part)
        return out
    scales = _for_files(_scales, np.arange(len(files)))
    crops = _for_files(_crops, np.arange(len(files)))
    from .pipeline import FAST_PLAN_MIN_FILES
    if len(files) >= FAST_PLAN_MIN_FILES and all(isinstance(f, (str, Path)) for f in files):
        # paths: the C helper's threads read the files straight into the pinned staging buffer and walk them
        from .fastplan import plan_batch
        from .pipeline import read_files_packed, release_pinned
        raw, offs, sizes = read_files_packed(files)
        try:
            plan = plan_batch(raw, offs, sizes, walked=getattr(raw, "_bj_walk", None))
        except Exception:
            release_pinned(raw)
            raise
        batch = decode_batch_on_device(None, device=device, packed=(raw, offs), plan=plan, scales=scales, crops=crops,
                                       compat=compat)
    else:
        datas = [_read(f) for f in files]
        batch = decode_batch_on_device(datas, device=device, scales=scales, crops=crops, compat=compat)
    if to_host:
        batch.start_host_copy()
    return [JpegDecoder(f, _batch=batch, _index=i) for i, f in enumerate(files)]


def _for_files(scales, idx: np.ndarray):
    """decode_batch_on_device's scales (or crops) for a sub-batch made of files[idx]: a function of (records, file
    indices) is bound to the indices."""
    if callable(scales):
        return lambda images: scales(images, idx)
    return scales


def _decode_batch_tolerant(files: list, device, chunk: int, scales=None, crops=None, compat: str = "reference") -> list:
    """decode_batch(on_error="return"): header problems are found per file on the host (the same parser and plan
    checks the batch path runs), entropy-data problems come back as the per-image device error words.  A crop box
    outside its image is that file's ValueError."""
    from .crop import Boxes, outside, outside_error
    from .errors import JpegError
    from .pipeline import BatchPlan, error_for
    results: list = [None] * len(files)
    good: List[int] = []
    datas = {}
    for i, f in enumerate(files):
        try:
            d = _read(f)
            p = parse_jpeg(d)
            BatchPlan([p], [0], len(d))                      # header, scan script and size checks of one file
        except JpegError as e:
            results[i] = e
            continue
        if isinstance(crops, Boxes) and outside(crops.box(i), p.width, p.height)[0]:
            results[i] = outside_error(crops.box(i), p.width, p.height)
            continue
        datas[i] = d
        good.append(i)
    for a in range(0, len(good), chunk):
        idx = good[a:a + chunk]
        batch = decode_batch_on_device([datas[i] for i in idx], device=device, check=False,
                                       scales=_for_files(scales, np.asarray(idx)), crops=_for_files(crops, np.asarray(idx)),
                                       compat=compat)
        pipe = batch.stats["_pipe"]
        err = pipe.err.cpu().numpy()                          # synchronises
        for k, i in enumerate(idx):
            e = error_for(err[k], i)
            results[i] = e if e is not None else JpegDecoder(files[i], _batch=batch, _index=k)
    return results
