#!/usr/bin/env python3
"""decode_to_tensor on the flagship workload (synthetic 1080p files of bench.make_files):  python tools/tensor_bench.py

Prints one JSON line per measurement:
  card          GPU name and power limit (nvidia-smi), read in the same run
  resize_kernel bj_resize alone over a resident batch of 512 decoded 1080p images -> 224 x 224 fp16 NCHW (CUDA events
                over 50 launches), GB/s on algorithmic bytes (source boxes once + output), next to a device-to-device
                copy of a 2.5 GB buffer timed in the same run (read + write bytes), and the tile re-read factor
  call          wall clock of decode_to_tensor(4096 files, 224 x 224 fp16, ImageNet mean / std) alternated with
                decode_batch(4096 files), 5 reps each, and the user's way today: decode_batch + per-image
                F.interpolate(antialias=True) + normalise + torch.stack
  memory        peak torch.cuda.max_memory_allocated of decode_to_tensor(16384 files) against decode_batch(4096 files)
"""
import ctypes
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402

MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)
SIZE = (224, 224)
TILE = 32        # output tile of csrc/bj_resize.cu


def windows(n: int, m: int):
    """lo / hi of every output of an n -> m axis, in fp32 like csrc/bj_resize_math.cuh."""
    f = np.float32
    scale = f(n) / f(m)
    support = scale if scale >= 1 else f(1)
    c = scale * (np.arange(m, dtype=f) + f(0.5))
    lo = np.maximum((c - support + f(0.5)).astype(np.int64), 0)
    hi = np.minimum((c + support + f(0.5)).astype(np.int64), n)
    return lo, hi


def reread(n: int, m: int) -> float:
    """Source pixels the tiles of one axis read, over the axis length."""
    lo, hi = windows(n, m)
    firsts = np.arange(0, m, TILE)
    lasts = np.minimum(firsts + TILE, m) - 1
    return float((hi[lasts] - lo[firsts]).sum() / n)


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"gpu": "unknown", "error": str(e)}


def emit(what: str, **kw) -> None:
    print(json.dumps({"what": what, **kw}), flush=True)


def resize_kernel(files, torch) -> None:
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.tensor_out import (DTYPES, RESIZE_JOB_DTYPE, ResizeParams, _bind, _fold_norm,
                                               pixel_boxes)
    n = 512
    res = decode_batch([files[i % len(files)] for i in range(n)], device="cuda:0")
    batch = res[0]._batch
    g = batch.plan.geom
    rec = g.images
    boxes = pixel_boxes(None, rec["width"], rec["height"], SIZE)
    jobs = np.zeros(n, dtype=RESIZE_JOB_DTYPE)
    jobs["src_offset"], jobs["src_pitch"], jobs["channels"] = rec["out_offset"], rec["out_pitch"], 3
    jobs["x0"], jobs["y0"], jobs["x1"], jobs["y1"] = boxes.T
    jobs["dst_index"] = np.arange(n)
    dev_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).cuda()
    out = torch.empty((n, 3) + SIZE, dtype=torch.float16, device="cuda:0")
    a, b = _fold_norm(torch.float16, MEAN, STD)
    p = ResizeParams(SIZE[0], SIZE[1], DTYPES[torch.float16], 0, (ctypes.c_float * 3)(*a), (ctypes.c_float * 3)(*b))
    L = _bind()
    s = torch.cuda.current_stream()

    def launch():
        assert L.bj_resize(dev_jobs.data_ptr(), n, batch.out.data_ptr(), out.data_ptr(), ctypes.byref(p),
                           s.cuda_stream) == 0

    reps = 50
    for _ in range(5):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    src_bytes = int((boxes[:, 2] - boxes[:, 0]).astype(np.int64) @ (boxes[:, 3] - boxes[:, 1]).astype(np.int64)) * 3
    out_bytes = out.numel() * out.element_size()
    # device-to-device copy of a buffer far larger than L2, same run
    big = torch.empty(2560 << 20, dtype=torch.uint8, device="cuda:0")
    dst = torch.empty_like(big)
    for _ in range(3):
        dst.copy_(big)
    e0.record()
    for _ in range(10):
        dst.copy_(big)
    e1.record()
    torch.cuda.synchronize()
    copy_ms = e0.elapsed_time(e1) / 10
    copy_gbs = 2 * big.numel() / copy_ms / 1e6
    gbs = (src_bytes + out_bytes) / ms / 1e6
    emit("resize_kernel", images=n, src="1920x1080 RGB", out="224x224 fp16 NCHW", launches=reps, ms=round(ms, 4),
         algorithmic_bytes=src_bytes + out_bytes, gbs=round(gbs, 1), d2d_copy_gbs=round(copy_gbs, 1),
         share_of_copy=round(gbs / copy_gbs, 3), tile_reread=round(reread(1920, 224) * reread(1080, 224), 4),
         tile_reread_x=round(reread(1920, 224), 4), tile_reread_y=round(reread(1080, 224), 4))
    del big, dst, res, batch


def user_way(datas, torch):
    import torch.nn.functional as F
    from pyjpegdecoder_b200 import decode_batch
    m = torch.tensor(MEAN, device="cuda:0").view(3, 1, 1)
    s = torch.tensor(STD, device="cuda:0").view(3, 1, 1)
    res = decode_batch(datas, device="cuda:0")
    out = []
    for d in res:
        x = d.image_tensor.permute(2, 0, 1)[None].float()
        x = F.interpolate(x, SIZE, mode="bilinear", antialias=True, align_corners=False)[0]
        out.append(((x / 255 - m) / s).half())
    return torch.stack(out)


def main():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
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

    tensor_call = lambda: decode_to_tensor(datas, SIZE, dtype=torch.float16, mean=MEAN, std=STD, device="cuda:0")  # noqa: E731
    batch_call = lambda: decode_batch(datas, device="cuda:0")  # noqa: E731
    for _ in range(2):
        timed(tensor_call)
        timed(batch_call)
    t_tensor, t_batch = [], []
    for _ in range(5):
        t_tensor.append(timed(tensor_call))
        t_batch.append(timed(batch_call))
    timed(lambda: user_way(datas[:256], torch))
    t_user = [timed(lambda: user_way(datas, torch)) for _ in range(3)]
    ref = user_way(datas[:64], torch).float()
    got = decode_to_tensor(datas[:64], SIZE, dtype=torch.float16, mean=MEAN, std=STD, device="cuda:0").float()
    emit("call", files=n, decode_to_tensor_ms=[round(x, 1) for x in t_tensor], decode_batch_ms=[round(x, 1) for x in t_batch],
         median_ratio=round(float(np.median(t_tensor) / np.median(t_batch)), 3),
         user_way_ms=[round(x, 1) for x in t_user], user_way_max_abs_diff=round((got - ref).abs().max().item(), 4))

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        r = fn()
        torch.cuda.synchronize()
        p = torch.cuda.max_memory_allocated() - base
        del r
        return p

    big = [files[i % len(files)] for i in range(16384)]
    p_tensor = peak(lambda: decode_to_tensor(big, SIZE, dtype=torch.float16, mean=MEAN, std=STD, device="cuda:0"))
    p_batch = peak(batch_call)
    emit("memory", decode_to_tensor_16384_gb=round(p_tensor / 1e9, 2), output_gb=round(16384 * 3 * 224 * 224 * 2 / 1e9, 2),
         decode_batch_4096_gb=round(p_batch / 1e9, 2))


if __name__ == "__main__":
    main()
