"""libjpeg-turbo-exact decode: compat="libjpeg-turbo" (bj_pixels_ijg, include/b200jpeg.h; csrc/bj_ijg_math.cuh).

compat="reference" (the default everywhere) decodes like the reference, PyJpegDecoder.  compat="libjpeg-turbo" gives
exactly what libjpeg-turbo's default jpeg_read_scanlines writes -- Pillow's Image.open(f), torchvision's CPU decode and
OpenCV -- so a data pipeline that switches to this library keeps its input distribution.  This module owns what the
mode introduces: the compat check, the jobs (one per image: its crop box, or the whole image), the MCU window with
the halo the fancy upsampling reads, the workspace layout and the launch.  The entropy stage only changes its AC
refinement rule (BJ_PHASE_T81_REFINE, pipeline.py).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native
from .crop import CROP_JOB_DTYPE, layout
from .scaled import upload

COMPATS = ("reference", "libjpeg-turbo")
PHASE_T81_REFINE = 16    # BJ_PHASE_T81_REFINE of bj_entropy_decode
IJG_ALL = 3              # BJ_IJG_ALL: both launches of bj_pixels_ijg
WS_ALIGN = 256           # a job's workspace offset is stored in bj_crop_job.reserved in these units


def check_compat(compat, scale=1) -> str:
    """The compat argument of decode_batch / decode_stream / JpegDecoder / decode_to_tensor.  libjpeg-turbo's reduced
    sizes (jidctred.c, PIL's draft()) are a different contract, so compat="libjpeg-turbo" takes scale 1 only."""
    if not isinstance(compat, str) or compat not in COMPATS:
        raise ValueError(f"compat must be 'reference' or 'libjpeg-turbo', got {compat!r}")
    if compat == "libjpeg-turbo" and not (isinstance(scale, (int, np.integer)) and not isinstance(scale, bool)
                                          and int(scale) == 1):
        raise ValueError(f"compat='libjpeg-turbo' decodes at full size only (scale=1), got scale={scale!r}")
    return compat


def _need(p0, p1, n):
    """Samples [lo, hi] that a ratio-2 fancy upsampling reads for pixels [p0, p1) of a component with n real samples
    (bj::ijg_need)."""
    j0, j1 = p0 >> 1, (p1 - 1) >> 1
    lo = np.where(((p0 & 1) == 0) & (j0 > 0), j0 - 1, j0)
    hi = np.where((((p1 - 1) & 1) == 1) & (j1 < n - 1), j1 + 1, j1)
    return lo, hi


def windows(rec: np.ndarray, boxes) -> np.ndarray:
    """(n, 4) MCU windows [mx0, mx1) x [my0, my1) of full-size boxes (n, 4) of the images `rec`: the MCUs the box
    touches, grown to every MCU holding a sample the fancy upsampling reads for a box pixel (bj::ijg_window)."""
    b = np.asarray(boxes, dtype=np.int64).reshape(-1, 4)
    hmax, vmax = rec["hmax"].astype(np.int64), rec["vmax"].astype(np.int64)
    W, H = rec["width"].astype(np.int64), rec["height"].astype(np.int64)
    mw, mh = 8 * hmax, 8 * vmax
    mx0, my0 = b[:, 0] // mw, b[:, 1] // mh
    mx1, my1 = -(-b[:, 2] // mw), -(-b[:, 3] // mh)
    for c in range(3):
        has = rec["ncomp"] > c
        hs = np.where(has, rec["hs"][:, c], 1).astype(np.int64)
        vs = np.where(has, rec["vs"][:, c], 1).astype(np.int64)
        rh, rv = hmax // hs, vmax // vs
        dw, dh = -(-W * hs // hmax), -(-H * vs // vmax)
        fh = has & (rh == 2) & (dw > 2)
        fv = has & (rv == 2) & ((rh == 1) | (dw > 2))
        lo, hi = _need(b[:, 0], b[:, 2], dw)
        mx0 = np.where(fh, np.minimum(mx0, lo // (8 * hs)), mx0)
        mx1 = np.where(fh, np.maximum(mx1, hi // (8 * hs) + 1), mx1)
        lo, hi = _need(b[:, 1], b[:, 3], dh)
        my0 = np.where(fv, np.minimum(my0, lo // (8 * vs)), my0)
        my1 = np.where(fv, np.maximum(my1, hi // (8 * vs) + 1), my1)
    return np.stack([mx0, my0, mx1, my1], 1)


def workspace_layout(rec: np.ndarray, win: np.ndarray):
    """(per-job byte offsets, total bytes) of the sample planes: per job, plane c has (mx1 - mx0) 8 h_c columns and
    (my1 - my0) 8 v_c rows, components back to back; jobs start on WS_ALIGN bytes."""
    nx, ny = win[:, 2] - win[:, 0], win[:, 3] - win[:, 1]
    per = np.zeros(len(rec), dtype=np.int64)
    for c in range(3):
        has = rec["ncomp"] > c
        per += np.where(has, nx * 8 * rec["hs"][:, c].astype(np.int64) * ny * 8 * rec["vs"][:, c].astype(np.int64), 0)
    padded = (per + WS_ALIGN - 1) // WS_ALIGN * WS_ALIGN
    offs = np.zeros(len(rec), dtype=np.int64)
    if len(rec) > 1:
        np.cumsum(padded[:-1], out=offs[1:])
    return offs, int(padded.sum())


def jobs_for(rec: np.ndarray, boxes=None):
    """(bj_crop_job array, OutputLayout or None, max_strips, workspace bytes) for the images `rec`: with boxes=None one
    job per image over the whole image at its planner out_offset / out_pitch (layout None: the planner's), else the
    file boxes (n, 4) clipped to their images and packed like crop.py's output."""
    n = len(rec)
    W, H = rec["width"].astype(np.int64), rec["height"].astype(np.int64)
    jobs = np.zeros(n, dtype=CROP_JOB_DTYPE)
    jobs["image"] = np.arange(n)
    if boxes is None:
        sb = np.stack([np.zeros(n, np.int64), np.zeros(n, np.int64), W, H], 1)
        lay = None
        jobs["out_offset"] = rec["out_offset"]
        jobs["out_pitch"] = rec["out_pitch"]
    else:
        from .crop import scaled_boxes
        sb = scaled_boxes(boxes, W, H, np.ones(n, np.int64))
        lay = layout(rec, sb)
        jobs["out_offset"] = lay.offsets
        jobs["out_pitch"] = lay.pitches
    jobs["x0"], jobs["y0"], jobs["x1"], jobs["y1"] = sb[:, 0], sb[:, 1], sb[:, 2], sb[:, 3]
    win = windows(rec, sb)
    offs, ws_bytes = workspace_layout(rec, win)
    jobs["reserved"] = offs // WS_ALIGN
    return jobs, lay, int((win[:, 3] - win[:, 1]).max()), ws_bytes


_BOUND = False


def _bind():
    global _BOUND
    L = _native.lib()
    if not _BOUND:
        vp = ctypes.c_void_p
        L.bj_pixels_ijg.restype = ctypes.c_int
        L.bj_pixels_ijg.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, ctypes.c_uint32, vp]
        if L.bj_sizeof(3) != CROP_JOB_DTYPE.itemsize:
            raise _native.NativeLibraryError("struct bj_crop_job layout mismatch between Python and libb200jpeg.so")
        _BOUND = True
    return L


def launch(dg, coef: torch.Tensor, boxes, stream: torch.cuda.Stream, out=None, kinds: int = IJG_ALL):
    """libjpeg-turbo-exact pixels of one planned batch (stages.DeviceGeometry dg, coefficient buffer coef with T.81
    refinement) on `stream`, with one bj_pixels_ijg call.  boxes: None (whole images, at the planner's layout) or
    (n, 4) file boxes.  out: an output buffer to reuse (whole images only).  Returns (output buffer, OutputLayout or
    None)."""
    L = _bind()
    g = dg.geom
    jobs, lay, max_strips, ws_bytes = jobs_for(g.images, boxes)
    out_bytes = g.out_bytes if lay is None else lay.out_bytes
    with torch.cuda.device(dg.device), torch.cuda.stream(stream):
        if out is None or out.numel() < out_bytes:
            out = torch.empty(max(out_bytes, 16), dtype=torch.uint8, device=dg.device)
        ws = torch.empty(max(ws_bytes, WS_ALIGN), dtype=torch.uint8, device=dg.device)
        dev_jobs = upload(jobs, dg.device)
        _native.check(L.bj_pixels_ijg(dg.images.data_ptr(), dev_jobs.data_ptr(), len(jobs), max_strips, coef.data_ptr(),
                                      dg.qtabs.data_ptr(), ws.data_ptr(), out.data_ptr(), kinds, stream.cuda_stream),
                      "bj_pixels_ijg")
    return out, lay
