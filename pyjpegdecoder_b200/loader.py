"""Streaming front end for very large inputs (SURVEY.md section 8f, rank 2: the step before the hot path).

`decode_stream(files, chunk=512)` yields the decoded images chunk by chunk.  File reading, the threaded gather
into pinned memory and the host-side planning of chunk k+1 run on a worker thread while the GPU decodes chunk k
(the C helpers and numpy release the GIL), so the host work disappears behind the device time for all but the
first chunk.  Two pinned staging buffers alternate; a chunk's buffer is reused only after that chunk has been
synchronised (its status words were read back).  No CPU decode path: the worker only prepares inputs."""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Iterable, Iterator, List, Optional, Sequence, Union

import numpy as np
import torch

from .decoder import JpegDecoder, _read
from .parser import parse_jpeg
from .pipeline import FAST_PLAN_MIN_FILES, BatchPlan, decode_batch_on_device, pack_files, raise_for_errors
from .stages import require_cuda

Source = Union[str, Path, bytes, bytearray, memoryview]


def _ramp(n: int) -> List[int]:
    """Sizes of the first sub-batches when the full size is n: n/2, then growing by a quarter per step.  Nothing can
    run on the GPU until the first sub-batch has been gathered, uploaded and planned, so a shorter one cuts the
    start-up latency; the host prepares files ~1.4x faster than the GPU decodes them, so growing faster than that
    would leave the GPU waiting for the second and third sub-batch instead."""
    if n < 128 or os.environ.get("BJ_STREAM_RAMP", "1") == "0":
        return []
    out, c = [], n // 2
    while c < n:
        out.append(c)
        c += max(1, c // 4)
    return out


def _chunks(files: Iterable[Source], n: int, ramp: bool = True) -> Iterator[List[Source]]:
    """Cut the input into sub-batches of at most n files, in order; with ramp=True the first ones are smaller."""
    sizes = _ramp(n) if ramp else []
    buf: List[Source] = []
    for f in files:
        buf.append(f)
        if len(buf) == (sizes[0] if sizes else n):
            yield buf
            buf = []
            if sizes:
                sizes.pop(0)
    if buf:
        yield buf


_N_STREAMS = max(2, int(os.environ.get("BJ_STREAM_DEPTH", "3")))   # sub-batches in flight on the GPU, each on its own stream
_N_SLOTS = _N_STREAMS + 1


_STREAM_POOL = {}


def _device_streams(dev: torch.device):
    """The copy stream and the compute streams of the streaming front end, created once per device: PyTorch's caching
    allocator keeps freed blocks per stream, so fresh streams on every call would never get to reuse the tens of GB a
    large batch allocates (and sooner or later trigger a full cache flush in the middle of a decode)."""
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    if key not in _STREAM_POOL:
        with torch.cuda.device(dev):
            _STREAM_POOL[key] = (torch.cuda.Stream(dev), [torch.cuda.Stream(dev) for _ in range(_N_STREAMS)],
                                 torch.cuda.Stream(dev), torch.cuda.Stream(dev))
    return _STREAM_POOL[key]


class _Uploader:
    """Pinned staging buffers + a copy stream: the upload of chunk k+1 runs while chunk k is being decoded.  The
    buffers come from the process-wide pool of pipeline.pack_files (pinning memory costs ~0.5 ms per MB, so they
    are reused from call to call) and go back to it once the copy that reads them has completed."""

    def __init__(self, device):
        self.dev = require_cuda(device)
        self.stream = _device_streams(self.dev)[0]
        # the (small) descriptor uploads have their own stream: behind the file bytes of the NEXT sub-batch, which the
        # other worker may already have enqueued, they would hold their sub-batch back for a whole upload
        self.desc_stream = _device_streams(self.dev)[2]
        # pack_stage and plan_stage each own their lists (they may run on different threads)
        self.inflight: List = []          # pack_stage: (file-copy event, pinned file buffer)
        self.inflight_desc: List = []     # plan_stage: (descriptor-copy event, pinned descriptor buffer)
        self.desc_free: List[torch.Tensor] = []

    def _reclaim(self, block: bool) -> None:
        """Give pinned file buffers whose upload has completed back to the pool; with block=True wait for the oldest
        upload while _N_SLOTS buffers are out (called by pack_stage only)."""
        from .pipeline import release_pinned
        while self.inflight and (block and len(self.inflight) >= _N_SLOTS or self.inflight[0][0].query()):
            ev, buf = self.inflight.pop(0)
            ev.synchronize()
            release_pinned(buf)

    def _reclaim_desc(self) -> None:
        """Pinned descriptor staging buffers whose upload has completed (called by plan_stage only)."""
        while self.inflight_desc and self.inflight_desc[0][0].query():
            self.desc_free.append(self.inflight_desc.pop(0)[1])

    def pack_stage(self, files: Sequence[Source], read_threads: int = 16):
        """First half of the host side of a sub-batch (C code / file I/O, releases the GIL): get the file bytes into a
        pinned buffer and start their H2D copy.  Paths are read straight into the pinned buffer; bytes objects are
        gathered into it."""
        from .pipeline import read_files_packed
        self._reclaim(block=True)
        datas = None
        if len(files) >= FAST_PLAN_MIN_FILES and all(isinstance(f, (str, Path)) for f in files):
            raw_host, offsets, sizes = read_files_packed(files)
            packed = (raw_host, offsets)
        else:
            if any(not isinstance(f, (bytes, bytearray, memoryview)) for f in files) and len(files) > 1:
                with ThreadPoolExecutor(min(read_threads, len(files))) as ex:
                    datas = list(ex.map(_read, files))
            else:
                datas = [_read(f) for f in files]
            packed = pack_files(datas, pin=True, reuse_slot="checkout", walk=len(datas) >= FAST_PLAN_MIN_FILES)
            raw_host = packed[0]
            sizes = [len(d) for d in datas]
        with torch.cuda.device(self.dev), torch.cuda.stream(self.stream):
            raw_dev = torch.empty(raw_host.numel(), dtype=torch.uint8, device=self.dev)
            raw_dev.copy_(raw_host, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self.inflight.append((ev, raw_host))
        return list(files), datas, sizes, packed, raw_dev, ev

    def plan_stage(self, packed_stage):
        """Second half (numpy / Python, holds the GIL): plan the sub-batch and upload its descriptors.
        packed_stage: pack_stage's result or its future."""
        from .pipeline import upload_descriptors
        if hasattr(packed_stage, "result"):
            packed_stage = packed_stage.result()
        files, datas, sizes, packed, raw_dev, ev = packed_stage
        raw_host, offsets = packed
        if len(sizes) >= FAST_PLAN_MIN_FILES:
            from .fastplan import plan_batch
            plan = plan_batch(raw_host, offsets, sizes, walked=getattr(raw_host, "_bj_walk", None))
        else:
            plan = BatchPlan([parse_jpeg(d) for d in datas], offsets, raw_host.numel())
        self._reclaim_desc()
        dbuf = self.desc_free.pop() if self.desc_free else None
        desc_blob, layout, dbuf = upload_descriptors(plan, self.dev, self.desc_stream, dbuf)
        dev_ = torch.cuda.Event()
        with torch.cuda.device(self.dev):
            dev_.record(self.desc_stream)
        self.inflight_desc.append((dev_, dbuf))
        return files, packed, plan, raw_dev, (ev, dev_), (desc_blob, layout)

    def prepare(self, files: Sequence[Source], k: int = 0, read_threads: int = 8):
        """Host side of one sub-batch, both halves on the calling thread."""
        return self.plan_stage(self.pack_stage(files, read_threads))

    def close(self) -> None:
        from .pipeline import release_pinned
        for ev, buf in self.inflight:
            ev.synchronize()
            release_pinned(buf)
        for ev, _ in self.inflight_desc:
            ev.synchronize()
        self.inflight, self.inflight_desc = [], []


def _check(batch) -> None:
    pipe = batch.stats["_pipe"]
    pipe.stream.synchronize()                 # the chunk ran on its own stream: everything it produced is complete now
    raise_for_errors(pipe.err.cpu().numpy())


def decode_stream(files: Iterable[Source], chunk: int = 512, device: Optional[Union[str, torch.device]] = None,
                  keep_coefficients: bool = False, to_host: bool = False, scale: int = 1) -> Iterator[List[JpegDecoder]]:
    """Decode an arbitrarily long sequence of files in sub-batches of at most `chunk` files (the first two are
    smaller, see _chunks); yields one list of JpegDecoder objects per sub-batch, in order.  Errors of a file (NotJpeg, CorruptedJpeg, ...) are raised when its chunk is reached.
    Three things overlap: the worker thread prepares and uploads the chunks ahead, the GPU decodes up to three chunks
    on alternating streams (a chunk is checked only when two later ones have been enqueued), and the caller consumes
    the oldest finished chunk.  scale=2, 4 or 8: reduced-size decode, as in decode_batch."""
    from .scaled import check_scale
    if chunk < 1:
        raise ValueError("chunk must be positive")
    scale = check_scale(scale)
    yield from _decode_stream(files, chunk, device, keep_coefficients, to_host, None if scale == 1 else scale)


def _decode_stream(files, chunk, device, keep_coefficients=False, to_host=False, scales=None):
    """decode_stream with scales: None, one scale, or a function (bj_image records of a sub-batch, indices of its files
    in `files`) -> per-image scales, called once the sub-batch is planned."""
    up = _Uploader(device)
    it = _chunks(files, chunk)
    depth = _N_SLOTS - 1                     # chunks prepared ahead of the one being enqueued
    try:
        yield from _stream(up, it, depth, device, keep_coefficients, to_host, scales)
    finally:
        up.close()


def _stream(up, it, depth, device, keep_coefficients=False, to_host=False, scales=None):
    # consecutive chunks run on alternating streams: the latency-bound tail of chunk k (a few long-running CTAs, the
    # one-CTA-per-scan prefix kernel) overlaps the start of chunk k+1 instead of leaving the GPU half empty
    streams = _device_streams(up.dev)[1]
    d2h = _device_streams(up.dev)[3]          # to_host=True: the pixels of finished sub-batches go back on their own stream
    n_done = 0
    n_files = 0
    # ONE worker thread prepares the sub-batches.  Two were tried, both as two whole-task workers and as a gather
    # thread feeding a planning thread: the gathers fight for host memory bandwidth, the Python halves for the GIL, and
    # the run-to-run spread (61..73 ms per 4096 files) ate the 1-2 ms the overlap gained.
    with ThreadPoolExecutor(1) as worker:
        queue = []

        def refill():
            while len(queue) < depth:
                nxt = next(it, None)
                if nxt is None:
                    return
                queue.append(worker.submit(up.prepare, nxt))

        refill()
        pending = []          # enqueued, not yet checked: up to _N_STREAMS - 1 chunks run ahead of the one being consumed
        while queue:
            chunk_files, packed, plan, raw_dev, (ev, ev_desc), desc = queue.pop(0).result()
            refill()
            st = streams[n_done % _N_STREAMS]
            n_done += 1
            raw_dev.record_stream(st)
            desc[0].record_stream(st)
            st.wait_event(ev_desc)
            sc = scales
            if callable(scales):                  # the images' sizes are known only now that the sub-batch is planned
                sc = scales(plan.geom.images, np.arange(n_files, n_files + len(chunk_files)))
            n_files += len(chunk_files)
            batch = decode_batch_on_device(None, device=device, packed=packed, plan=plan, check=False,
                                           raw_dev=raw_dev, raw_ready=ev, desc=desc, stream=st, scales=sc)
            pending.append((batch, chunk_files))
            if len(pending) >= _N_STREAMS:
                b, fl = pending.pop(0)
                _check(b)
                b.release_work_buffers(keep_coefficients)
                if to_host:
                    b.start_host_copy(d2h, None)
                yield [JpegDecoder(f, _batch=b, _index=i) for i, f in enumerate(fl)]
        while pending:
            b, fl = pending.pop(0)
            _check(b)
            b.release_work_buffers(keep_coefficients)
            if to_host:
                b.start_host_copy(d2h, None)
            yield [JpegDecoder(f, _batch=b, _index=i) for i, f in enumerate(fl)]
