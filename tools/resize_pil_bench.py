#!/usr/bin/env python3
"""Pillow-exact resize (bj_resize_pil, decode_to_tensor(resample="pil-*")) on the flagship workload (synthetic 1080p
4:2:0 files of bench.make_files):  python tools/resize_pil_bench.py

Prints one JSON line per measurement:
  card           GPU name and power limit (nvidia-smi), read in the same run
  resize_kernel  bj_resize, bj_resize_pil bilinear and bj_resize_pil bicubic over the same 512 resident decoded 1080p
                 images -> 224 x 224 fp16 NCHW with ImageNet mean / std; CUDA events around 10 launches, 30 rounds,
                 variants alternated within each round, medians.  The source (3.2 GB) is far larger than L2.
  call           wall clock of decode_to_tensor(4096 files, 224 x 224, roi="center", fp16, compat="libjpeg-turbo")
                 with resample="pil-bilinear" against resample="torch", alternated, 5 reps after 2 warm-ups, medians
  parity         the timed pil-bilinear call's first 32 images in uint8 against Pillow (crop + resize), max abs diff
  pillow         torchvision's PIL pipeline on one core (Image.open, convert("RGB"), Resize(256), CenterCrop(224),
                 ToTensor, Normalize) over 64 distinct files, 2 passes, images/s
"""
import ctypes
import io
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import bench  # noqa: E402
from tensor_bench import MEAN, SIZE, STD, card, emit  # noqa: E402

LJT = "libjpeg-turbo"


def resize_kernel(files, torch) -> None:
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.tensor_out import (DTYPES, RESIZE_JOB_DTYPE, RESIZE_PIL_JOB_DTYPE, ResizeParams, _bind,
                                               _fold_norm)
    n = 512
    res = decode_batch([files[i % len(files)] for i in range(n)], device="cuda:0")
    batch = res[0]._batch
    rec = batch.plan.geom.images
    L = _bind()
    s = torch.cuda.current_stream()
    a, b = _fold_norm(torch.float16, MEAN, STD)
    p = ResizeParams(SIZE[0], SIZE[1], DTYPES[torch.float16], 0, (ctypes.c_float * 3)(*a), (ctypes.c_float * 3)(*b))
    outs = {}

    def jobs_of(dtype):
        j = np.zeros(n, dtype=dtype)
        j["src_offset"], j["src_pitch"], j["channels"] = rec["out_offset"], rec["out_pitch"], 3
        j["x1"], j["y1"] = rec["width"], rec["height"]
        j["dst_index"] = np.arange(n)
        if dtype is RESIZE_PIL_JOB_DTYPE:
            j["virt_w"], j["virt_h"] = SIZE[1], SIZE[0]
        return torch.from_numpy(j.view(np.uint8).copy()).cuda()

    jr, jp = jobs_of(RESIZE_JOB_DTYPE), jobs_of(RESIZE_PIL_JOB_DTYPE)

    def variant(name, fn):
        outs[name] = torch.empty((n, 3) + SIZE, dtype=torch.float16, device="cuda:0")
        o = outs[name]
        return lambda: fn(o)

    variants = {
        "bj_resize": variant("bj_resize", lambda o: L.bj_resize(jr.data_ptr(), n, batch.out.data_ptr(), o.data_ptr(),
                                                                 ctypes.byref(p), s.cuda_stream)),
        "bj_resize_pil_bilinear": variant("bil", lambda o: L.bj_resize_pil(jp.data_ptr(), n, batch.out.data_ptr(),
                                                                           o.data_ptr(), ctypes.byref(p), 0,
                                                                           s.cuda_stream)),
        "bj_resize_pil_bicubic": variant("bic", lambda o: L.bj_resize_pil(jp.data_ptr(), n, batch.out.data_ptr(),
                                                                          o.data_ptr(), ctypes.byref(p), 1,
                                                                          s.cuda_stream)),
    }
    for fn in variants.values():
        for _ in range(3):
            assert fn() == 0
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(30):
        for k, fn in variants.items():
            e0.record()
            for _ in range(10):
                fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / 10)
    med = {k: float(np.median(v)) for k, v in times.items()}
    src_bytes = int(rec["width"].astype(np.int64) @ rec["height"].astype(np.int64)) * 3
    out_bytes = n * 3 * SIZE[0] * SIZE[1] * 2
    diff = (outs["bil"].float() - outs["bj_resize"].float()).abs().max().item()
    for k in variants:
        emit("resize_kernel", kernel=k, images=n, src="1920x1080 RGB", out="224x224 fp16 NCHW", median_ms=round(med[k], 4),
             min_ms=round(min(times[k]), 4), max_ms=round(max(times[k]), 4),
             ratio_to_bj_resize=round(med[k] / med["bj_resize"], 3),
             gbs=round((src_bytes + out_bytes) / med[k] / 1e6, 1))
    emit("resize_kernel_outputs", bilinear_vs_bj_resize_max_abs_diff=round(diff, 4))
    del res, batch


def main():
    import torch
    from PIL import Image
    from pyjpegdecoder_b200 import decode_to_tensor
    emit("card", **card())
    files = bench.make_files(64)
    resize_kernel(files, torch)

    n = 4096
    datas = [files[i % len(files)] for i in range(n)]

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        del r
        return dt * 1e3

    def call(resample, dtype=torch.float16, k=n):
        mean, std = (MEAN, STD) if dtype != torch.uint8 else (None, None)
        return lambda: decode_to_tensor(datas[:k], SIZE, roi="center", dtype=dtype, mean=mean, std=std, compat=LJT,
                                        resample=resample, device="cuda:0")

    for _ in range(2):
        timed(call("pil-bilinear"))
        timed(call("torch"))
    t_pil, t_torch = [], []
    for _ in range(5):
        t_pil.append(timed(call("pil-bilinear")))
        t_torch.append(timed(call("torch")))
    emit("call", files=n, size=list(SIZE), roi="center", dtype="float16", compat=LJT,
         pil_bilinear_ms=[round(x, 1) for x in t_pil], torch_ms=[round(x, 1) for x in t_torch],
         median_ratio=round(float(np.median(t_pil) / np.median(t_torch)), 3))

    from pyjpegdecoder_b200.tensor_out import pixel_boxes
    got = call("pil-bilinear", torch.uint8, 32)().cpu()
    worst = 0
    for i in range(32):
        im = Image.open(io.BytesIO(datas[i])).convert("RGB")
        box = pixel_boxes("center", [im.width], [im.height], SIZE)[0]
        want = np.asarray(im.crop(tuple(int(v) for v in box)).resize((SIZE[1], SIZE[0]), Image.BILINEAR))
        worst = max(worst, int(np.abs(got[i].permute(1, 2, 0).numpy().astype(int) - want).max()))
    emit("parity", images=32, pil_bilinear_uint8_max_abs_diff_to_pillow=worst)

    from torchvision import transforms as T
    torch.set_num_threads(1)
    tf = T.Compose([T.Resize(256), T.CenterCrop(224), T.ToTensor(), T.Normalize(MEAN, STD)])
    t0 = time.perf_counter()
    for _ in range(2):
        for f in files:
            tf(Image.open(io.BytesIO(f)).convert("RGB"))
    dt = time.perf_counter() - t0
    emit("pillow", images=2 * len(files), pipeline="torchvision PIL Resize(256)+CenterCrop(224)+ToTensor+Normalize",
         threads=1, images_per_s=round(2 * len(files) / dt, 1))


if __name__ == "__main__":
    main()
