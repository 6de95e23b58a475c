#!/usr/bin/env python3
"""Reduced-size decode on the flagship workload (synthetic 1080p 4:2:0 files of bench.make_files):
python tools/scaled_bench.py

Prints one JSON line per measurement:
  card          GPU name and power limit (nvidia-smi), read in the same run
  pixel_kernel  bj_pixels_scaled at s = 2, 4, 8 and bj_pixels on the same 512 resident images (CUDA events around each
                launch, 50 rounds, the four kernels alternated), GB/s on algorithmic bytes -- the 32-byte sectors of
                each block's needed zig-zag prefix (all 128 bytes for bj_pixels) plus the output bytes -- next to a
                device-to-device copy of a 2.5 GB buffer timed in the same run (read + write bytes)
  call          wall clock of decode_batch(4096 files) at scale 1 and 4, and of decode_to_tensor(4096 files, 224 x 224,
                roi="center", fp16, ImageNet mean / std) at scale 1 and "auto", alternated, 5 reps, medians
  memory        peak torch.cuda.max_memory_allocated of each of the four calls
"""
import json
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import bench  # noqa: E402
from tensor_bench import card, emit  # noqa: E402

MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)
SIZE = (224, 224)


def sector_bytes(rec, log2s: int) -> int:
    """Bytes of the 32-byte sectors of the zig-zag prefix every block of the image needs at 1/2^log2s."""
    zz = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,
                   6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45,
                   38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
    total = 0
    mcus = int(rec["mcus_x"]) * int(rec["mcus_y"])
    for c in range(int(rec["ncomp"])):
        hs, vs = int(rec["hs"][c]), int(rec["vs"][c])
        nx, ny = (8 * int(rec["hmax"]) // hs) >> log2s, (8 * int(rec["vmax"]) // vs) >> log2s
        prefix = 1 + max(k for k in range(64) if zz[k] % 8 < nx and zz[k] // 8 < ny)
        total += mcus * hs * vs * 32 * -(-2 * prefix // 32)
    return total


def pixel_kernel(files, torch) -> None:
    from pyjpegdecoder_b200 import _native, decode_batch
    from pyjpegdecoder_b200.scaled import SCALED_JOB_DTYPE, OutputLayout, _bind, scaled_strips
    from pyjpegdecoder_b200.stages import run_pixels
    n = 512
    res = decode_batch([files[i % len(files)] for i in range(n)], device="cuda:0")
    batch = res[0]._batch
    pipe = batch.stats["_pipe"]
    dg, coef, rec = pipe.dg, pipe.coef, pipe.dg.geom.images
    L = _bind()
    s = torch.cuda.current_stream()
    full_out = torch.empty_like(batch.out)
    variants = {"bj_pixels": (lambda: run_pixels(dg, coef, _native.IN_COEF, _native.OUT_RGB, out=full_out, stream=s),
                              128 * dg.geom.total_blocks + dg.geom.out_bytes)}
    for l in (1, 2, 3):
        lay = OutputLayout.scaled(rec, np.full(n, 1 << l))
        jobs = np.zeros(n, SCALED_JOB_DTYPE)
        jobs["out_offset"], jobs["out_pitch"], jobs["image"], jobs["log2_scale"] = lay.offsets, lay.pitches, np.arange(n), l
        dev_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).cuda()
        out = torch.empty(lay.out_bytes, dtype=torch.uint8, device="cuda:0")
        strips = int(scaled_strips(rec).max())

        def launch(dev_jobs=dev_jobs, out=out, strips=strips):
            assert L.bj_pixels_scaled(dg.images.data_ptr(), dev_jobs.data_ptr(), n, strips, coef.data_ptr(),
                                      dg.qtabs.data_ptr(), out.data_ptr(), s.cuda_stream) == 0
        alg = sum(sector_bytes(r, l) for r in rec) + int((lay.heights * lay.pitches).sum())
        variants[f"s{1 << l}"] = (launch, alg)
    for fn, _ in variants.values():
        for _ in range(3):
            fn()
    times = {k: 0.0 for k in variants}
    for _ in range(50):
        for k, (fn, _) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[k] += e0.elapsed_time(e1)
    big = torch.empty(2560 << 20, dtype=torch.uint8, device="cuda:0")
    dst = torch.empty_like(big)
    for _ in range(3):
        dst.copy_(big)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(big)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 2 * big.numel() / (e0.elapsed_time(e1) / 10) / 1e6
    ms_full = times["bj_pixels"] / 50
    for k, (_, alg) in variants.items():
        ms = times[k] / 50
        gbs = alg / ms / 1e6
        emit("pixel_kernel", kernel=k, images=n, src="1920x1080 4:2:0", launches=50, ms=round(ms, 4),
             algorithmic_bytes=alg, gbs=round(gbs, 1), d2d_copy_gbs=round(copy_gbs, 1),
             share_of_copy=round(gbs / copy_gbs, 3), speedup_vs_bj_pixels=round(ms_full / ms, 2))
    del big, dst, res, batch, pipe


def main():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    emit("card", **card())
    files = bench.make_files(64)
    pixel_kernel(files, torch)

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

    calls = {
        "decode_batch_s1": lambda: decode_batch(datas, device="cuda:0"),
        "decode_batch_s4": lambda: decode_batch(datas, device="cuda:0", scale=4),
        "decode_to_tensor_s1": lambda: decode_to_tensor(datas, SIZE, roi="center", dtype=torch.float16, mean=MEAN,
                                                        std=STD, device="cuda:0"),
        "decode_to_tensor_auto": lambda: decode_to_tensor(datas, SIZE, roi="center", dtype=torch.float16, mean=MEAN,
                                                          std=STD, device="cuda:0", scale="auto"),
    }
    for _ in range(2):
        for fn in calls.values():
            timed(fn)
    t = {k: [] for k in calls}
    for _ in range(5):
        for k, fn in calls.items():
            t[k].append(timed(fn))
    med = {k: float(np.median(v)) for k, v in t.items()}
    emit("call", files=n, **{f"{k}_ms": [round(x, 1) for x in v] for k, v in t.items()},
         **{f"{k}_median_ms": round(v, 1) for k, v in med.items()},
         tensor_auto_over_batch_s1=round(med["decode_to_tensor_auto"] / med["decode_batch_s1"], 3),
         tensor_s1_over_batch_s1=round(med["decode_to_tensor_s1"] / med["decode_batch_s1"], 3),
         batch_s4_over_batch_s1=round(med["decode_batch_s4"] / med["decode_batch_s1"], 3))

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

    emit("memory", files=n, **{f"{k}_gb": round(peak(fn) / 1e9, 2) for k, fn in calls.items()})


if __name__ == "__main__":
    main()
