#!/usr/bin/env python3
"""compat="libjpeg-turbo" on the flagship workload (synthetic 1080p 4:2:0 files of bench.make_files):
python tools/ijg_bench.py

Prints one JSON line per measurement:
  card          GPU name and power limit (nvidia-smi), read in the same run
  pixel_kernel  bj_pixels_ijg (both launches, and each alone) against bj_pixels on the same 512 resident images; CUDA
                events around each launch, 50 rounds, variants alternated, medians; algorithmic bytes per image:
                bj_pixels 128 * blocks + RGB (12.5 MB), bj_pixels_ijg 128 * blocks + 2 * planes + RGB (18.5 MB)
  call          wall clock of decode_batch(4096) with compat="reference" and compat="libjpeg-turbo", alternated, 5 reps,
                medians
  pillow        Pillow's single-core Image.open + load of the same files (64 distinct files, 3 passes), megapixels/s
"""
import io
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import bench  # noqa: E402
from tensor_bench import card, emit  # noqa: E402


def pixel_kernel(files, torch) -> None:
    from pyjpegdecoder_b200 import _native, decode_batch, ijg
    from pyjpegdecoder_b200.scaled import upload
    from pyjpegdecoder_b200.stages import run_pixels
    n = 512
    res = decode_batch([files[i % len(files)] for i in range(n)], device="cuda:0")
    batch = res[0]._batch
    pipe = batch.stats["_pipe"]
    dg, coef, rec = pipe.dg, pipe.coef, pipe.dg.geom.images
    s = torch.cuda.current_stream()
    full_out = torch.empty_like(batch.out)
    out = torch.empty_like(batch.out)
    jobs, _, strips, ws_bytes = ijg.jobs_for(rec)
    dev_jobs = upload(jobs, "cuda:0")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda:0")
    L = ijg._bind()

    def ijg_launch(kinds):
        return lambda: _native.check(L.bj_pixels_ijg(dg.images.data_ptr(), dev_jobs.data_ptr(), n, strips, coef.data_ptr(),
                                                     dg.qtabs.data_ptr(), ws.data_ptr(), out.data_ptr(), kinds,
                                                     s.cuda_stream), "bj_pixels_ijg")
    coef_bytes = 128 * dg.geom.total_blocks
    rgb = dg.geom.out_bytes
    variants = {"bj_pixels": (lambda: run_pixels(dg, coef, _native.IN_COEF, _native.OUT_RGB, out=full_out, stream=s),
                              coef_bytes + rgb),
                "bj_pixels_ijg": (ijg_launch(3), coef_bytes + 2 * ws_bytes + rgb),
                "bj_pixels_ijg_idct": (ijg_launch(1), coef_bytes + ws_bytes),
                "bj_pixels_ijg_colour": (ijg_launch(2), ws_bytes + rgb)}
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
        emit("pixel_kernel", kernel=k, images=n, src="1920x1080 4:2:0", launches=50, median_ms=round(med[k], 4),
             algorithmic_bytes=alg, gbs=round(alg / med[k] / 1e6, 1), over_bj_pixels=round(med[k] / med["bj_pixels"], 3))
    del res, batch, pipe


def main():
    import torch
    from PIL import Image
    from pyjpegdecoder_b200 import decode_batch
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

    calls = {"reference": lambda: decode_batch(datas, device="cuda:0"),
             "libjpeg_turbo": lambda: decode_batch(datas, device="cuda:0", compat="libjpeg-turbo")}
    for _ in range(2):
        for fn in calls.values():
            timed(fn)
    t = {k: [] for k in calls}
    for _ in range(5):
        for k, fn in calls.items():
            t[k].append(timed(fn))
    med = {k: float(np.median(v)) for k, v in t.items()}
    emit("call", files=n, **{f"{k}_median_ms": round(v, 1) for k, v in med.items()},
         libjpeg_turbo_over_reference=round(med["libjpeg_turbo"] / med["reference"], 3))

    t0 = time.perf_counter()
    px = 0
    for _ in range(3):
        for d in files:
            im = Image.open(io.BytesIO(d))
            im.load()
            px += im.size[0] * im.size[1]
    dt = time.perf_counter() - t0
    emit("pillow", files=3 * len(files), threads=1, mpix_per_s=round(px / dt / 1e6, 1),
         gpu_libjpeg_turbo_mpix_per_s=round(n * 1920 * 1080 / med["libjpeg_turbo"] / 1e3, 1))


if __name__ == "__main__":
    main()
