#!/usr/bin/env python3
"""Crop decode on the flagship workload (synthetic 1080p 4:2:0 files of bench.make_files):
python tools/crop_bench.py

Prints one JSON line per measurement:
  card          GPU name and power limit (nvidia-smi), read in the same run
  pixel_kernel  bj_pixels_crop against bj_pixels (s = 1) and bj_pixels_scaled (s = 4) on the same 512 resident images,
                for three boxes: the whole frame, a centred 960 x 540 box (60 x 35 of 120 x 68 MCUs) and seeded
                RandomResizedCrop boxes (area 0.08..1, ratio 3/4..4/3); CUDA events around each launch, 50 rounds, all
                variants alternated, medians; algorithmic bytes 128 * blocks in the windows + channels * box pixels
  call          wall clock of decode_batch(4096) with and without crop=centre box, and of decode_to_tensor(4096, 224 x 224,
                fp16, ImageNet mean / std) with roi=None, roi="center" + scale="auto" and the random boxes at scale 1,
                alternated, 5 reps, medians, each as a ratio to decode_batch(4096)
  memory        peak torch.cuda.max_memory_allocated of decode_batch(4096) with and without crop=centre box
"""
import math
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import bench  # noqa: E402
from scaled_bench import sector_bytes  # noqa: E402
from tensor_bench import card, emit  # noqa: E402

MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)
SIZE = (224, 224)
W, H = 1920, 1080
CENTRE = (480, 270, 1440, 810)


def random_resized_crops(n: int, seed: int = 0) -> np.ndarray:
    """torchvision RandomResizedCrop's box sampling (area 0.08..1 of the image, log-uniform ratio 3/4..4/3, ten tries
    then the whole image), in numpy."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        box = (0, 0, W, H)
        for _ in range(10):
            area = W * H * rng.uniform(0.08, 1.0)
            ratio = math.exp(rng.uniform(math.log(3 / 4), math.log(4 / 3)))
            w, h = int(round(math.sqrt(area * ratio))), int(round(math.sqrt(area / ratio)))
            if 0 < w <= W and 0 < h <= H:
                x0, y0 = int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
                box = (x0, y0, x0 + w, y0 + h)
                break
        out.append(box)
    return np.asarray(out, np.int64)


def pixel_kernel(files, torch) -> None:
    from pyjpegdecoder_b200 import _native, crop, decode_batch
    from pyjpegdecoder_b200.scaled import SCALED_JOB_DTYPE, OutputLayout, _bind, scaled_strips
    from pyjpegdecoder_b200.stages import run_pixels
    n = 512
    res = decode_batch([files[i % len(files)] for i in range(n)], device="cuda:0")
    batch = res[0]._batch
    pipe = batch.stats["_pipe"]
    dg, coef, rec = pipe.dg, pipe.coef, pipe.dg.geom.images
    Ls, Lc = _bind(), crop._bind()
    s = torch.cuda.current_stream()
    full_out = torch.empty_like(batch.out)
    variants = {"bj_pixels": (lambda: run_pixels(dg, coef, _native.IN_COEF, _native.OUT_RGB, out=full_out, stream=s),
                              128 * dg.geom.total_blocks + dg.geom.out_bytes)}
    lay4 = OutputLayout.scaled(rec, np.full(n, 4))
    jobs4 = np.zeros(n, SCALED_JOB_DTYPE)
    jobs4["out_offset"], jobs4["out_pitch"], jobs4["image"], jobs4["log2_scale"] = lay4.offsets, lay4.pitches, np.arange(n), 2
    dev4 = torch.from_numpy(jobs4.view(np.uint8).copy()).cuda()
    out4 = torch.empty(lay4.out_bytes, dtype=torch.uint8, device="cuda:0")
    strips4 = int(scaled_strips(rec).max())
    variants["bj_pixels_scaled_s4"] = (
        lambda: _native.check(Ls.bj_pixels_scaled(dg.images.data_ptr(), dev4.data_ptr(), n, strips4, coef.data_ptr(),
                                                  dg.qtabs.data_ptr(), out4.data_ptr(), s.cuda_stream), "bj_pixels_scaled"),
        int((lay4.heights * lay4.pitches).sum()) + sum(sector_bytes(r, 2) for r in rec))
    boxes = {"whole": np.tile((0, 0, W, H), (n, 1)), "centre": np.tile(CENTRE, (n, 1)),
             "random": random_resized_crops(n)}
    for sc in (1, 4):
        for name, b in boxes.items():
            jobs, lay, strips, kinds = crop.jobs_for(rec, b, np.full(n, sc))
            dev_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).cuda()
            out = torch.empty(max(lay.out_bytes, 16), dtype=torch.uint8, device="cuda:0")
            win = crop.windows(crop.scaled_boxes(b, rec["width"], rec["height"], np.full(n, sc)), rec["hmax"],
                               rec["vmax"], np.full(n, sc))
            blocks = int(((win[:, 2] - win[:, 0]) * (win[:, 3] - win[:, 1]) * rec["blocks_per_mcu"]).sum())

            def launch(dev_jobs=dev_jobs, out=out, strips=strips, kinds=kinds):
                _native.check(Lc.bj_pixels_crop(dg.images.data_ptr(), dev_jobs.data_ptr(), n, strips, coef.data_ptr(),
                                                dg.geom.total_blocks, dg.qtabs.data_ptr(), dg.table.data_ptr(),
                                                out.data_ptr(), kinds, None, s.cuda_stream), "bj_pixels_crop")
            variants[f"crop_s{sc}_{name}"] = (launch, 128 * blocks + int((lay.heights * lay.pitches).sum()))
    for fn, _ in variants.values():
        for _ in range(3):
            fn()
    times = {k: [] for k in variants}
    for _ in range(50):
        for k, (fn, _) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in times.items()}
    for k, (_, alg) in variants.items():
        base = "bj_pixels_scaled_s4" if k.startswith("crop_s4") else "bj_pixels"
        emit("pixel_kernel", kernel=k, images=n, src="1920x1080 4:2:0", launches=50, median_ms=round(med[k], 4),
             algorithmic_bytes=alg, gbs=round(alg / med[k] / 1e6, 1),
             **({} if not k.startswith("crop") else {f"over_{base}": round(med[k] / med[base], 3)}))
    del res, batch, pipe


def main():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    emit("card", **card())
    files = bench.make_files(64)
    pixel_kernel(files, torch)

    n = 4096
    datas = [files[i % len(files)] for i in range(n)]
    rand = random_resized_crops(n, seed=1)
    rois = [(x0 / W, y0 / H, x1 / W, y1 / H) for x0, y0, x1, y1 in rand.tolist()]

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        del r
        return dt * 1e3

    calls = {
        "decode_batch": lambda: decode_batch(datas, device="cuda:0"),
        "decode_batch_crop_centre": lambda: decode_batch(datas, device="cuda:0", crop=CENTRE),
        "tensor_roi_none": lambda: decode_to_tensor(datas, SIZE, dtype=torch.float16, mean=MEAN, std=STD,
                                                    device="cuda:0"),
        "tensor_center_auto": lambda: decode_to_tensor(datas, SIZE, roi="center", dtype=torch.float16, mean=MEAN,
                                                       std=STD, device="cuda:0", scale="auto"),
        "tensor_random_s1": lambda: decode_to_tensor(datas, SIZE, roi=rois, dtype=torch.float16, mean=MEAN, std=STD,
                                                     device="cuda:0"),
    }
    for _ in range(2):
        for fn in calls.values():
            timed(fn)
    t = {k: [] for k in calls}
    for _ in range(5):
        for k, fn in calls.items():
            t[k].append(timed(fn))
    med = {k: float(np.median(v)) for k, v in t.items()}
    emit("call", files=n, **{f"{k}_median_ms": round(v, 1) for k, v in med.items()},
         **{f"{k}_over_decode_batch": round(v / med["decode_batch"], 3) for k, v in med.items() if k != "decode_batch"})

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

    emit("memory", files=n, **{f"{k}_gb": round(peak(calls[k]) / 1e9, 2)
                               for k in ("decode_batch", "decode_batch_crop_centre")})


if __name__ == "__main__":
    main()
