#!/usr/bin/env python3
"""bench.py -- decoded MP/s of the B200 JPEG decode path on the BASELINE.json workload.

Workload (BASELINE.json configs[3], the configuration the metric is quoted on): a batch of 4096
1920x1080 baseline 4:2:0 JPEGs per GPU, Pillow-encoded synthetic content (SURVEY.md 8d generator,
quality 75, no restart markers).  A "step" = one pass of the hot path over the whole batch:
device un-stuffing -> speculative Huffman decode -> fix-up/prefix -> coefficient write -> fused
IDCT/upsample/colour.  Images are independent: with N GPUs every rank decodes its own batch (weak
scaling, no collective on the data path; torch.distributed is only used for the timing barrier).

  value  whole-job MP/s with the compressed files already resident in HBM
  e2e    the same through the public pipeline object with the files in PINNED HOST memory: every step
         copies them host->device, runs all kernels, and reads the per-image status words back
  roofline / stages  per-kernel CUDA-event times, algorithmic bytes and GB/s against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (oracle/, a C port of the reference's algorithm) on one host core

`--impl reference` times the reference's algorithm on the host cores instead (oracle port, all threads).
"""
import argparse
import io
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

W, H = 1920, 1080


def synth_image(seed: int, w: int = W, h: int = H) -> np.ndarray:
    """SURVEY.md 8(d): img = 128 + 100*(sin, cos, sin) + N(0, 12^2), seed = image index."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.stack([128 + 100 * np.sin(x / 37 + y / 91), 128 + 100 * np.cos(x / 53 - y / 29),
                    128 + 100 * np.sin((x + y) / 71)], -1)
    img = img + rng.normal(0, 12, img.shape).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def encode_one(seed: int) -> bytes:
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(synth_image(seed)).save(b, "JPEG", quality=75, subsampling=2)
    return b.getvalue()


def make_files(n_distinct: int, seed0: int = 0):
    from multiprocessing import get_context
    workers = min(n_distinct, os.cpu_count() or 1, 16)
    if workers > 1:
        with get_context("fork").Pool(workers) as pool:
            return pool.map(encode_one, range(seed0, seed0 + n_distinct))
    return [encode_one(s) for s in range(seed0, seed0 + n_distinct)]


def synth_jpeg(w: int, h: int, seed: int, mode: str = "RGB", **save_kw) -> bytes:
    """One Pillow-encoded synthetic image of the SURVEY 8(d) generator (quality 75 unless overridden)."""
    from PIL import Image
    img = synth_image(seed, w, h)
    im = Image.fromarray(img[..., 1] if mode == "L" else img)
    b = io.BytesIO()
    save_kw.setdefault("quality", 75)
    im.save(b, "JPEG", **save_kw)
    return b.getvalue()


def _scan_bytes(data: bytes) -> int:
    from pyjpegdecoder_b200.parser import parse_jpeg
    return sum(sc.data_end - sc.data_start for sc in parse_jpeg(data).scans)


def bench_configs(dev) -> dict:
    """The other shapes BASELINE.json names (configs 0, 1, 2, 4), each through the product's own entry points:
    latency of one decode and MP/s / bitstream GB/s, measured with wall clock around synchronised calls."""
    import tempfile
    import torch
    from pyjpegdecoder_b200 import JpegDecoder
    from pyjpegdecoder_b200.pipeline import decode_batch_on_device
    out = {}

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts))

    def entry(datas, sec, what, **extra):
        from pyjpegdecoder_b200.parser import parse_jpeg
        mp = sum(p.width * p.height for p in map(parse_jpeg, datas)) / 1e6
        sb = sum(_scan_bytes(d) for d in datas)
        e = {"images": len(datas), "megapixels": mp, "ms": sec * 1e3, "mp_s": mp / sec, "bitstream_gbs": sb / sec / 1e9, "what": what}
        e.update(extra)
        return e

    # C1: the reference's own CPU-runnable case, through the literal drop-in call JpegDecoder(path).image_array
    c1 = synth_jpeg(512, 512, 0, subsampling=2)
    with tempfile.TemporaryDirectory() as td:
        path = Path(td) / "c1.jpg"
        path.write_bytes(c1)
        sec = timed(lambda: JpegDecoder(path, device=dev).image_array, reps=20, warm=3)
    out["c1_single_512"] = entry([c1], sec, "JpegDecoder(Path).image_array: file read + parse + H2D + kernels + D2H of the pixels "
                                 "(jpeg_decoder.py:29-110), median of 20")
    # C2: 3840x2160 with restart intervals (one MCU row / 16 MCUs per interval), one image per decode
    for key, kw in (("c2_4k_dri_rows1", dict(restart_marker_rows=1)), ("c2_4k_dri_blocks16", dict(restart_marker_blocks=16))):
        d = synth_jpeg(3840, 2160, 1, subsampling=2, **kw)
        sec = timed(lambda: decode_batch_on_device([d], device=dev), reps=10)
        out[key] = entry([d], sec, "decode_batch_on_device([bytes]): parse + H2D + kernels + status, pixels stay on the device, median of 10")
    # C3: progressive, 10 scans with successive approximation: the reference's own example file (DRI) and a synthetic one (no DRI)
    base = ROOT / "tests" / "golden" / "base_image.jpg"
    c3 = [("c3_progressive_reference_file", base.read_bytes())] if base.exists() else []
    c3.append(("c3_progressive_synthetic_no_dri", synth_jpeg(4160, 2340, 7, subsampling=2, progressive=True)))
    for key, d in c3:
        sec = timed(lambda: decode_batch_on_device([d], device=dev), reps=5)
        out[key] = entry([d], sec, "decode_batch_on_device([bytes]), one 4160x2340 progressive image, median of 5")
    # C5: mixed-subsampling 8192x8192 batch, baseline + progressive (grey, 4:2:2, 4:4:4), one batch of 6
    c5 = []
    for prog in (False, True):
        c5.append(synth_jpeg(8192, 8192, 11, mode="L", progressive=prog))
        c5.append(synth_jpeg(8192, 8192, 12, subsampling=1, progressive=prog))
        c5.append(synth_jpeg(8192, 8192, 13, subsampling=0, progressive=prog))
    sec = timed(lambda: decode_batch_on_device(c5[:3], device=dev), reps=3, warm=1)
    out["c5_mixed_8192_baseline"] = entry(c5[:3], sec, "decode_batch_on_device: grey + 4:2:2 + 4:4:4 baseline 8192x8192 in one batch, median of 3")
    sec = timed(lambda: decode_batch_on_device(c5, device=dev), reps=3, warm=1)
    out["c5_mixed_8192_baseline_and_progressive"] = entry(c5, sec, "the same three plus their progressive encodings (6 images), median of 3")
    torch.cuda.empty_cache()
    return out


def python_reference_c1() -> dict:
    """The UNMODIFIED reference (baseline/_ref/jpeg_decoder.py, copied there by __graft_entry__.build()) on the C1 file,
    one host core (BASELINE.md section 3).  Its GUI call is patched out, its progress prints are discarded."""
    ref_dir = ROOT / "baseline" / "_ref"
    if not (ref_dir / "jpeg_decoder.py").exists():
        return {"unavailable": "baseline/_ref/jpeg_decoder.py is missing (run __graft_entry__.build() where /root/reference exists)"}
    import contextlib
    import tempfile
    sys.path.insert(0, str(ref_dir))
    try:
        import jpeg_decoder as ref
        ref.JpegDecoder.show = lambda self: None
        data = synth_jpeg(512, 512, 0, subsampling=2)
        with tempfile.TemporaryDirectory() as td:
            path = Path(td) / "c1.jpg"
            path.write_bytes(data)
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                d = ref.JpegDecoder(path)
            dt = time.perf_counter() - t0
        assert d.image_array.shape == (512, 512, 3)
        return {"value": 512 * 512 / 1e6 / dt, "unit": "MP/s", "cores": 1, "kind": "reference", "seconds": dt,
                "sample": "one 512x512 4:2:0 q75 file (BASELINE.json configs[0]) through the unmodified jpeg_decoder.JpegDecoder(Path)"}
    except Exception as e:  # noqa: BLE001 -- the baseline must never take the bench down
        return {"unavailable": f"{type(e).__name__}: {e}"}
    finally:
        sys.path.remove(str(ref_dir))


def measured_traffic() -> dict:
    """DRAM bytes (read + write) per image and kernel from the latest `ncu --set full` capture of this build, written by
    tools/ncu_traffic.py into profiles/; absent -> traffic is reported as null."""
    p = ROOT / "profiles" / "r2_traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text())
        except Exception:
            pass
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _gather_sample(bufs, segments, n, rng):
    """float32 values at n seeded positions of the concatenation of `segments`, each (buffer index, start, length)
    of a flat device tensor in `bufs`; positions are in ascending order of the concatenation."""
    import torch
    seg_buf = np.array([s[0] for s in segments], np.int64)
    seg_start = np.array([s[1] for s in segments], np.int64)
    cum = np.concatenate([[0], np.cumsum([s[2] for s in segments], dtype=np.int64)])
    idx = np.sort(rng.integers(0, cum[-1], n, dtype=np.int64))
    seg = np.searchsorted(cum, idx, side="right") - 1
    pos = seg_start[seg] + (idx - cum[seg])
    parts = []
    for b, buf in enumerate(bufs):
        sel = pos[seg_buf[seg] == b]
        if len(sel):
            ix = torch.from_numpy(sel).to(buf.device)
            parts.append(buf.reshape(-1).index_select(0, ix).float().cpu().numpy())
    return np.concatenate(parts)


def dump_outputs(out_dir: Path, pipes, seed: int = 0) -> None:
    """Write what the last step of the timed path left in the sub-batch buffers, as float32 .npy files (48 MiB in all):
      pixels.npy        2^23 values of the uint8 RGB output of the whole batch (images in batch order, each (H, W, 3)
                        row-major, concatenated), at seeded random positions in ascending order
      coefficients.npy  2^22 values of the int16 quantised coefficients (device order, sub-batches concatenated), the same way
      errors.npy        every image's device error word
    The positions depend only on `seed` and the batch, so two builds run with the same arguments compare value for value."""
    out_dir.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(seed)
    outs = [p.out for p in pipes]
    images = [(c, off, int(np.prod(shape))) for c, p in enumerate(pipes)
              for off, shape in zip(p.plan.geom.out_offsets, p.plan.geom.out_shapes)]
    np.save(out_dir / "pixels.npy", _gather_sample(outs, images, 1 << 23, rng))
    coefs = [p.coef for p in pipes]
    np.save(out_dir / "coefficients.npy", _gather_sample(coefs, [(c, 0, t.numel()) for c, t in enumerate(coefs)], 1 << 22, rng))
    np.save(out_dir / "errors.npy", np.concatenate([p.err.cpu().numpy() for p in pipes]).astype(np.float32))


def run_reference(args):
    """The reference's algorithm on the host cores: the CPU oracle (C port, oracle/) over all threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.lib()
    cores = os.cpu_count() or 1
    files = make_files(min(args.distinct, 2 * cores))
    per_step = max(cores, len(files))
    jobs = [files[i % len(files)] for i in range(per_step)]

    def one(d):
        return oracle.decode(d, want=("rgb",)).rgb.shape

    with ThreadPoolExecutor(cores) as ex:
        for _ in range(args.warmup):
            list(ex.map(one, jobs))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            list(ex.map(one, jobs))
        dt = time.perf_counter() - t0
    mp = per_step * args.steps * W * H / 1e6
    val = mp / dt
    line = {
        "impl": "reference", "metric": "decoded MP/s (1080p 4:2:0 batch)", "value": val, "unit": "MP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "1920x1080 baseline 4:2:0 q75 JPEGs, no restart markers (BASELINE.json configs[3])",
                   "images_per_step": per_step},
        "cpu_baseline": {"value": val, "unit": "MP/s", "cores": cores, "kind": "port",
                         "sample": f"{per_step} images/step x {args.steps} steps, oracle C port, {cores} threads"},
        "e2e": {"value": val, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--images", type=int, default=4096, help="images per GPU per step")
    ap.add_argument("--chunks", type=int, default=8, help="sub-batches per GPU, one CUDA stream each")
    ap.add_argument("--distinct", type=int, default=64, help="distinct synthetic images (cycled to --images)")
    ap.add_argument("--cpu-sample", type=int, default=48, help="images decoded by the 1-core CPU baseline")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-shape `configs` measurements and the Python-reference timing")
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help="after the timed steps, write a seeded sample of what the last one computed (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.dump_outputs is not None:
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # synthetic files first (fork pool before CUDA is touched); every rank gets its own seeds
    t_gen = time.perf_counter()
    files = make_files(args.distinct, seed0=rank * args.distinct)
    t_gen = time.perf_counter() - t_gen

    import torch
    import torch.distributed as dist
    from pyjpegdecoder_b200.parser import parse_jpeg
    from pyjpegdecoder_b200.pipeline import BatchPlan, DevicePipeline, pack_files, raise_for_errors

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_img = args.images
    n_chunks = max(1, min(args.chunks, n_img))
    parsed_d = [parse_jpeg(d) for d in files]
    # the batch is processed as n_chunks sub-batches, each with its own stream and buffers, so that the
    # host->device copy of one sub-batch and the latency-bound kernels of another overlap
    bounds = [round(i * n_img / n_chunks) for i in range(n_chunks + 1)]
    pipes, raws = [], []
    for c in range(n_chunks):
        idx = range(bounds[c], bounds[c + 1])
        datas = [files[i % len(files)] for i in idx]
        parsed = [parsed_d[i % len(files)] for i in idx]
        raw_host, offsets = pack_files(datas, pin=True)
        plan = BatchPlan(parsed, offsets, raw_host.numel())
        pipes.append(DevicePipeline(plan, dev, torch.cuda.Stream(dev)))
        raws.append(raw_host)
    main = torch.cuda.Stream(dev)
    scan_bytes = int(sum(int(p.plan.scans["raw_len"].sum()) for p in pipes))
    nblk = sum(p.plan.geom.total_blocks for p in pipes)
    n_sub = sum(int(p.plan.n_sub) for p in pipes)
    raw_bytes = sum(int(r.numel()) for r in raws)
    out_bytes = n_img * W * H * 3
    mp_per_step = n_img * W * H / 1e6

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(n_steps, body):
        """Run n_steps x body(pipe index) on the sub-batch streams, timed with CUDA events on `main`:
        every stream starts after e0 and e1 is recorded after all of them have finished."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        e0.record(main)
        for p in pipes:
            p.stream.wait_event(e0)
        for _ in range(n_steps):
            for c in range(len(pipes)):
                body(c)
        for p in pipes:
            ev = torch.cuda.Event()
            ev.record(p.stream)
            main.wait_event(ev)
        e1.record(main)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3 / n_steps
        return max(e0.elapsed_time(e1) / n_steps, 0.0), wall

    # ---- warm-up + correctness of the run ------------------------------------------------------------
    for p, r in zip(pipes, raws):
        p.upload(r)
    for _ in range(args.warmup):
        for p in pipes:
            p.launch()
    barrier()
    for p in pipes:
        raise_for_errors(p.err.cpu().numpy())

    # ---- per-stage times: sub-batches one after another, CUDA events around every stage --------------
    events = {}
    for _ in range(max(1, min(args.steps, 2))):
        for p in pipes:
            p.launch(events=events)
            p.stream.synchronize()
    stage_ms = {k: float(np.sum([a.elapsed_time(b) for (a, b) in v])) / max(1, min(args.steps, 2)) for k, v in events.items()}

    # ---- device-resident throughput (value): all sub-batch streams concurrently -----------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_dev, _ = timed_steps(args.steps, lambda c: pipes[c].launch())
    ms_dev = max_over_ranks(ms_dev)

    # ---- end to end: pinned host bytes -> device -> kernels -> status words back ---------------------
    err_hosts = [torch.empty(len(p.plan.parsed), dtype=torch.int32, pin_memory=True) for p in pipes]

    def e2e_body(c):
        pipes[c].upload(raws[c])
        pipes[c].launch()
        with torch.cuda.stream(pipes[c].stream):
            err_hosts[c].copy_(pipes[c].err, non_blocking=True)

    timed_steps(max(1, args.warmup // 2), e2e_body)
    ms_ev, ms_wall = timed_steps(args.steps, e2e_body)
    ms_e2e = max_over_ranks(max(ms_ev, ms_wall))
    clocks = sampler.stop()
    assert all(int(e.abs().sum()) == 0 for e in err_hosts), "device reported decode errors"
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, pipes)
    launches_per_step = sum(p.kernel_launches_per_step for p in pipes)
    device_bytes = sum(p.device_bytes() for p in pipes)

    # ---- the PUBLIC batch entry point on every rank (the product's own multi-GPU shape: one process per GPU, each
    #      decoding its shard; bytes in, planning INSIDE the timed region).  weak: n_img files per GPU; strong: ONE
    #      batch of n_img files split across the ranks.  Wall clock between barriers, max over ranks. ---------------
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.multigpu import shard_range
    del pipes[:]
    torch.cuda.empty_cache()
    datas_api = [files[i % len(files)] for i in range(n_img)]
    lo, hi = shard_range(n_img, world, rank)

    def api_time(datas, reps=3, warm=3):
        def once():
            res = decode_batch(datas, device=dev)
            torch.cuda.synchronize(dev)
            del res
        for _ in range(warm):        # pinned pool and caching allocator reach their steady state after two calls
            once()
        ts = []
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            once()
            ts.append(max_over_ranks(time.perf_counter() - t0))
        return float(np.median(ts))

    dt_weak = api_time(datas_api)
    dt_strong = api_time(datas_api[lo:hi]) if world > 1 else dt_weak
    what = ("pyjpegdecoder_b200.decode_batch(list of bytes) -> list of JpegDecoder objects, pixels on the device: gather into "
            "pinned memory + marker walk + plan on the host, H2D, all kernels, status read-back; sub-batches of 512 files "
            "pipelined; one process per GPU, no collective; median of 3, max over ranks")
    api = {"value": world * n_img * W * H / 1e6 / dt_weak, "unit": "MP/s", "images": world * n_img, "ms": dt_weak * 1e3,
           "scaling": "weak", "what": what,
           "strong": {"value": n_img * W * H / 1e6 / dt_strong, "unit": "MP/s", "images": n_img, "ms": dt_strong * 1e3,
                      "what": f"ONE batch of {n_img} files split across {world} rank(s)"},
           "host_threads_per_rank": int(os.environ.get("BJ_HOST_THREADS", "0")) or None}

    # ---- the same public call on PATHS (the reference's entry point takes a Path): the distinct files are written
    #      to a temporary directory once (they stay in the page cache), the list of n_img paths cycles through them;
    #      file reads go straight into the pinned staging buffer.  N = 1 only. ------------------------------------
    api_paths = None
    if world == 1 and not args.no_configs:
        import shutil
        import tempfile
        tmpdir = Path(tempfile.mkdtemp(prefix="bj_bench_"))
        try:
            fpaths = []
            for i, fdata in enumerate(files):
                fp = tmpdir / f"img{i:04d}.jpg"
                fp.write_bytes(fdata)
                fpaths.append(fp)
            paths_api = [fpaths[i % len(fpaths)] for i in range(n_img)]
            dt_paths = api_time(paths_api)
            api_paths = {"value": n_img * W * H / 1e6 / dt_paths, "unit": "MP/s", "images": n_img, "ms": dt_paths * 1e3,
                         "what": "decode_batch(list of pathlib.Path), files in the page cache: read straight into pinned memory, "
                                 "marker walk + plan, H2D, all kernels, status read-back; median of 3"}
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)

    # ---- the reference's actual return type at batch scale: numpy arrays in HOST memory.  decode_batch(to_host=True)
    #      sends the pixels of every sub-batch back in one pinned transfer behind the decode of the next ones; the
    #      figure is bound by PCIe (3 bytes per pixel out against ~0.19 in).  N = 1 only, 1024 files (6.4 GB of
    #      pinned host memory). ------------------------------------------------------------------------------------
    host_px = None
    if world == 1 and n_img >= 1024 and not args.no_configs:
        n_host = 1024

        def host_once():
            res = decode_batch(datas_api[:n_host], device=dev, to_host=True)
            checksum = 0
            for d in res:
                a = d.image_array                      # (W, H, 3) numpy view of the pinned copy; waits for its transfer
                checksum += int(a[0, 0, 0])
            return checksum
        for _ in range(2):
            host_once()
        ts = []
        for _ in range(3):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            host_once()
            ts.append(time.perf_counter() - t0)
        dt = float(np.median(ts))
        host_px = {"value": n_host * W * H / 1e6 / dt, "unit": "MP/s", "images": n_host, "ms": dt * 1e3,
                   "d2h_gbs": n_host * W * H * 3 / dt / 1e9,
                   "what": "decode_batch(list of bytes, to_host=True) and image_array of every result: pixels as numpy arrays "
                           "in (pinned) host memory, like the reference returns them; one device->host transfer per "
                           "sub-batch, overlapped with the decode of the following ones; median of 3"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline accounting (SURVEY.md 8d: algorithmic bytes) -------------------------------------
    peak, peak_src = measured_peak_gbs()
    alg = {
        "unstuff": 2 * scan_bytes,                       # read stuffed bytes, write compacted words
        "spec": scan_bytes + 32 * n_sub,                 # bitstream + entry/exit/count records
        "fix": 64 * n_sub,                               # records in, records + prefix out
        "write": scan_bytes + 128 * nblk,                # bitstream in, one 128-byte line per block out
        "pixels": 128 * nblk + out_bytes,                # coefficients in, RGB out (fused I+C)
    }
    stages = {}
    for k, ms in stage_ms.items():
        if k in alg and ms > 0:
            gbs = alg[k] / (ms * 1e-3) / 1e9
            stages[k] = {"ms": ms, "algorithmic_bytes": alg[k], "gbs": gbs, "frac_of_peak": gbs / peak,
                         "share_of_step": ms / sum(stage_ms.values())}
        else:
            stages[k] = {"ms": ms, "share_of_step": ms / sum(stage_ms.values())}
    dom = max((k for k in stages if "gbs" in stages[k]), key=lambda k: stages[k]["ms"])
    # dram__bytes_read.sum + dram__bytes_write.sum per image, from the ncu --set full capture of THIS build that
    # tools/ncu_traffic.py summarised into profiles/r2_traffic.json (null when that file is absent)
    traffic = measured_traffic()
    ncu_traffic_per_image = traffic.get("bytes_per_image", {})
    img_per_launch = n_img / n_chunks
    names = {"unstuff": "unstuff_count/scan_tiles/unstuff_scatter", "spec": "spec_kernel", "fix": "fix_local_kernel + chain_kernel",
             "write": "write_kernel", "pixels": "bj_pixels_420_kernel (fused dezigzag+dequant+IDCT+upsample+colour)"}

    def roof(k):
        st = stages.get(k, {})
        tr = ncu_traffic_per_image.get(k)
        return {"kernel": names[k], "bound": "hbm", "achieved": st.get("gbs"), "peak": peak, "unit": "GB/s",
                "frac": st.get("frac_of_peak"), "traffic": (tr * img_per_launch) if tr else None,
                "traffic_source": traffic.get("source") if tr else None,
                "peak_source": peak_src, "launches_per_step": n_chunks,
                "algorithmic_bytes_per_launch": alg[k] / n_chunks, "ms_per_launch": st.get("ms", 0.0) / n_chunks,
                "share_of_step": st.get("share_of_step")}
    roofline = roof(dom)
    roofline_pixels = roof("pixels")

    # ---- the PUBLIC batch entry point, everything included (python bytes -> pinned pack, C marker walk +
    #      plan on the host, H2D, all kernels, status read-back); smaller batch, reported for information --
    # ---- CPU baseline: oracle port, one core, bounded sample ------------------------------------------
    cpu = None
    if world == 1:
        import oracle
        oracle.lib()
        sample = [files[i % len(files)] for i in range(args.cpu_sample)]
        t0 = time.perf_counter()
        for d in sample:
            oracle.decode(d, want=("rgb",))
        dt = time.perf_counter() - t0
        cpu = {"value": len(sample) * W * H / 1e6 / dt, "unit": "MP/s", "cores": 1, "kind": "port",
               "sample": f"{len(sample)} of the same 1080p files, oracle C port (oracle/jpeg_oracle.c), 1 thread, {dt:.1f} s"}

    configs = bench_configs(dev) if (world == 1 and not args.no_configs) else None
    cpu_python = python_reference_c1() if (world == 1 and not args.no_configs) else None

    line = {
        "metric": "decoded MP/s (1080p 4:2:0 batch)", "value": mp_per_step * world / (ms_dev * 1e-3), "unit": "MP/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int16 (fp32 IDCT, fp64 tie-break)",
        "data": f"synthetic: {len(files)} distinct Pillow-encoded 1080p images per GPU cycled to {n_img}",
        "config": {"workload": "batch of 4096 1920x1080 baseline 4:2:0 q75 JPEGs per GPU, no restart markers "
                               "(BASELINE.json configs[3])",
                   "images_per_gpu": n_img, "sub_batches": n_chunks,
                   "streams": "one CUDA stream per sub-batch; stage times measured with the sub-batches run one after another",
                   "l2": "inputs larger than L2 (bitstream %.2f GB, coefficients %.1f GB per step)"
                         % (scan_bytes / 1e9, nblk * 128 / 1e9),
                   "host_parse": "marker parsing and descriptor build happen before the timed region"},
        "e2e": {"value": mp_per_step * world / (ms_e2e * 1e-3), "unit": "MP/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": raw_bytes, "d2h_bytes_per_step": 4 * n_img},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
        "roofline": roofline, "roofline_pixels": roofline_pixels, "stages": stages,
        "bitstream_gbs": {k: scan_bytes / (stage_ms[k] * 1e-3) / 1e9 for k in ("unstuff", "spec", "write") if k in stage_ms},
        "cpu_baseline": cpu, "cpu_baseline_python": cpu_python, "public_api_e2e": api, "public_api_paths_e2e": api_paths, "host_pixels_e2e": host_px, "configs": configs,
        "device_bytes": device_bytes, "gen_seconds": t_gen,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
