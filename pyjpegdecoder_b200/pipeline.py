"""Device pipeline for a batch of JPEG files on ONE GPU.

host parse (parser.py)  ->  H2D of the file bytes  ->  bj_unstuff  ->  bj_entropy_plan  ->
bj_entropy_decode per wave/mode  ->  bj_pixels  ->  per-image (H, W, 3) uint8 views.

This is the launch site that replaces the reference's start_of_scan -> baseline_dct_scan /
progressive_dct_scan -> end_of_image chain (jpeg_decoder.py:640-650, :1368-1388): the host records a
scan descriptor per SOS and defers; the whole batch then runs as a handful of kernel launches.
torch tensors are used as device buffers only; all compute is in libb200jpeg.so.
"""
from __future__ import annotations

import ctypes
import os
import threading
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native
from .errors import CorruptedJpeg, NativeLibraryError
from .huffman import build_scan_blob
from .layout import slot0_of
from .parser import ParsedJpeg, Scan, parse_jpeg
from .plan import BatchGeometry, scan_levels
from .stages import DeviceGeometry, require_cuda, run_pixels, to_device



def _subseq_bits() -> int:
    """BJ_SUBSEQ_BITS of the built library (bj_sizeof_entropy(3)); 1024 when the library is absent (planning only)."""
    try:
        L = _native.lib()
        L.bj_sizeof_entropy.restype = ctypes.c_int
        L.bj_sizeof_entropy.argtypes = [ctypes.c_int]
        v = int(L.bj_sizeof_entropy(3))
        return v if v > 0 else 1024
    except NativeLibraryError:
        return 1024


SUBSEQ_BITS = _subseq_bits()
ENTROPY_THREADS = 128
UNSTUFF_TILE = 4096
MAX_SLOTS = 10

# batches of at least this many files are planned by fastplan.py (C marker walk + templates)
FAST_PLAN_MIN_FILES = 4

MODES = {"baseline": 0, "dc_first": 1, "dc_refine": 2, "ac_first": 3, "ac_refine": 4}

# numpy mirror of struct bj_scan (144 bytes, see include/b200jpeg.h)
SCAN_DTYPE = np.dtype({
    "names": ["raw_off", "coef_block0", "raw_len", "image", "stream0", "n_streams", "ri", "n_mcu", "mcus_x",
              "sub0", "n_sub_max", "lut_off", "lut_len", "tile0", "frame_mcus_x", "frame_bpm", "nslots", "mode",
              "ss", "se", "ah", "al", "interleaved", "comp_h", "comp_v", "comp_slot0", "ncomp_scan",
              "slot_frame", "slot_comp", "slot_dc", "slot_ac", "pad0", "reserved"],
    "formats": ["<u8", "<u8", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4",
                "<u2", "u1", "u1", "u1", "u1", "u1", "u1", "u1", "u1", "u1", "u1", "u1", "u1",
                ("u1", (MAX_SLOTS,)), ("u1", (MAX_SLOTS,)), ("<u2", (MAX_SLOTS,)), ("<u2", (MAX_SLOTS,)), "<u2", "<u4"],
    "offsets": [0, 8, 16, 20, 24, 28, 32, 36, 40, 44, 48, 52, 56, 60, 64, 66, 67, 68, 69, 70, 71, 72, 73, 74, 75,
                76, 77, 78, 88, 98, 118, 138, 140],
    "itemsize": 144,
})


class EntropyBuffers(ctypes.Structure):
    """struct bj_entropy_buffers"""
    _fields_ = [("words", ctypes.c_void_p), ("words_len", ctypes.c_uint64),
                ("stream_start", ctypes.c_void_p), ("stream_end", ctypes.c_void_p), ("stream_sub", ctypes.c_void_p),
                ("sub_entry", ctypes.c_void_p), ("sub_exit", ctypes.c_void_p),
                ("sub_count", ctypes.c_void_p), ("sub_prefix", ctypes.c_void_p),
                ("lut", ctypes.c_void_p), ("coef", ctypes.c_void_p), ("err", ctypes.c_void_p),
                ("sync_changes", ctypes.c_void_p), ("blk_pos", ctypes.c_void_p)]


_BOUND = False


def _bind():
    global _BOUND
    L = _native.lib()
    if not _BOUND:
        vp, ci, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32
        L.bj_sizeof_entropy.restype = ci
        L.bj_sizeof_entropy.argtypes = [ci]
        L.bj_unstuff.restype = ci
        L.bj_unstuff.argtypes = [vp, vp, ci, vp, ci, vp, vp, vp, vp, ci, vp]
        L.bj_entropy_plan.restype = ci
        L.bj_entropy_plan.argtypes = [vp, ci, ci, vp, ctypes.POINTER(EntropyBuffers), vp]
        L.bj_entropy_decode.restype = ci
        L.bj_entropy_decode.argtypes = [vp, ci, ci, ci, u32, u32, u32, u32, ctypes.POINTER(EntropyBuffers), vp, ci, vp]
        if L.bj_sizeof_entropy(1) != SCAN_DTYPE.itemsize or L.bj_sizeof_entropy(2) != ctypes.sizeof(EntropyBuffers):
            raise NativeLibraryError("struct bj_scan / bj_entropy_buffers layout mismatch")
        _BOUND = True
    return L


@dataclass
class ScanGroup:
    first: int
    count: int
    mode: int
    max_sub: int
    max_streams: int
    max_blocks: int
    max_lut: int


class BatchPlan:
    """Everything the host must compute for one batch: geometry, scan descriptors grouped into waves,
    tile table, Huffman LUT blob, buffer sizes.  `offsets[i]` is where file i starts in the raw buffer."""

    def __init__(self, parsed: Sequence[ParsedJpeg], offsets: Sequence[int], raw_bytes: int, serial_scans: bool = False):
        self.parsed = list(parsed)
        self.geom = BatchGeometry(self.parsed)
        self.raw_bytes = raw_bytes
        n_scans = sum(len(p.scans) for p in self.parsed)
        self.scans = np.zeros(n_scans, dtype=SCAN_DTYPE)
        self.any_progressive = any(p.progressive for p in self.parsed)
        self.needs_zero = self.any_progressive or any(not covers_all_components(p) for p in self.parsed)
        lut_parts: List[np.ndarray] = []
        lut_cache: Dict[tuple, Tuple[int, int, list, list]] = {}
        lut_size = 0
        # order: wave by wave (scans of equal dependency level, plan.scan_levels), inside a wave grouped by mode
        order4 = sorted((lv, MODES[p.scans[k].kind], i, k) for i, p in enumerate(self.parsed)
                        for k, lv in enumerate(scan_levels(p, serial_scans)))
        order = [(lv, m, i, k) for (lv, m, i, k) in order4]
        self.groups: List[ScanGroup] = []
        stream0 = 0
        sub0 = 0
        tile0 = 0
        tile_counts = []
        cur_key = None
        for k, (w, mode, i, sidx) in enumerate(order):
            p = self.parsed[i]
            sc: Scan = p.scans[sidx]
            rec = self.scans[k]
            raw_off = offsets[i] + sc.data_start
            raw_len = sc.data_end - sc.data_start
            if raw_len < 0 or raw_off < 0 or raw_off + raw_len > raw_bytes:
                raise CorruptedJpeg(f"File {i}: entropy-coded segment lies outside the file.")
            n_mcu = sc.mcus_x * sc.mcus_y
            ri = sc.ri if sc.ri > 0 else n_mcu
            n_streams = -(-n_mcu // ri)
            interleaved = len(sc.comps) > 1 or p.ncomp == 1
            key = (sc.dc_specs, sc.ac_specs)
            if key not in lut_cache:
                blob, dc_off, ac_off = build_scan_blob(sc.dc_specs, sc.ac_specs)
                lut_cache[key] = (lut_size, len(blob), dc_off, ac_off)
                lut_parts.append(blob)
                lut_size += len(blob)
            lut_off, lut_len, dc_off, ac_off = lut_cache[key]
            s0 = slot0_of(p)
            slot = 0
            if sum((p.components[ci].h * p.components[ci].v if len(sc.comps) > 1 else 1) for ci in sc.comps) > MAX_SLOTS:
                raise CorruptedJpeg("More than 10 blocks per MCU.")
            for kk, ci in enumerate(sc.comps):
                c = p.components[ci]
                nb = c.h * c.v if len(sc.comps) > 1 else 1
                for r in range(nb):
                    rec["slot_frame"][slot] = s0[ci] + r
                    rec["slot_comp"][slot] = kk
                    rec["slot_dc"][slot] = dc_off[kk]
                    rec["slot_ac"][slot] = ac_off[kk]
                    slot += 1
            if slot > MAX_SLOTS:
                raise CorruptedJpeg("More than 10 blocks per MCU.")
            c0 = p.components[sc.comps[0]]
            n_sub_max = -(-raw_len * 8 // SUBSEQ_BITS) + n_streams
            lead = raw_off & 15
            n_tiles = max(1, -(-(lead + raw_len) // UNSTUFF_TILE))
            rec["raw_off"], rec["raw_len"] = raw_off, raw_len
            rec["coef_block0"] = self.geom.block_offsets[i]
            rec["image"] = i
            rec["stream0"], rec["n_streams"], rec["ri"], rec["n_mcu"], rec["mcus_x"] = stream0, n_streams, ri, n_mcu, sc.mcus_x
            rec["sub0"], rec["n_sub_max"] = sub0, n_sub_max
            rec["lut_off"], rec["lut_len"] = lut_off, lut_len
            rec["tile0"] = tile0
            rec["frame_mcus_x"], rec["frame_bpm"] = p.mcus_x, p.blocks_per_mcu
            rec["nslots"], rec["mode"] = slot, mode
            rec["ss"], rec["se"], rec["ah"], rec["al"] = sc.ss, sc.se, sc.ah, sc.al
            rec["interleaved"] = 1 if interleaved else 0
            rec["comp_h"], rec["comp_v"], rec["comp_slot0"] = c0.h, c0.v, s0[sc.comps[0]]
            rec["ncomp_scan"] = len(sc.comps)
            if (w, mode) != cur_key:
                self.groups.append(ScanGroup(first=k, count=0, mode=mode, max_sub=0, max_streams=0, max_blocks=0, max_lut=0))
                cur_key = (w, mode)
            g = self.groups[-1]
            g.count += 1
            g.max_sub = max(g.max_sub, n_sub_max)
            g.max_streams = max(g.max_streams, n_streams)
            g.max_blocks = max(g.max_blocks, n_mcu * slot)
            g.max_lut = max(g.max_lut, lut_len)
            stream0 += n_streams
            sub0 += n_sub_max
            tile0 += n_tiles
            tile_counts.append(n_tiles)
        self.n_streams = stream0
        self.n_sub = sub0
        self.n_tiles = tile0
        self.tile_scan = np.repeat(np.arange(n_scans, dtype=np.uint32), tile_counts)
        self.lut = np.concatenate(lut_parts).astype(np.uint32)
        self.max_chain = max((-(-g.max_sub // ENTROPY_THREADS)) * g.count for g in self.groups
                             if g.mode in (0, 1, 3)) if any(g.mode in (0, 1, 3) for g in self.groups) else 1


def host_threads() -> int:
    """Host threads of the C gather / marker-walk helpers: BJ_HOST_THREADS, else the cores of the box divided among
    the ranks of a one-process-per-GPU launch (LOCAL_WORLD_SIZE), at most 16."""
    env = os.environ.get("BJ_HOST_THREADS")
    if env:
        return max(1, int(env))
    ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1))
    return max(1, min(16, (os.cpu_count() or 1) // ranks))


def covers_all_components(p: ParsedJpeg) -> bool:
    """True if the scans of a baseline image write every coefficient block (the write kernel stores whole blocks,
    so the coefficient buffer then needs no memset).  A truncated non-interleaved file leaves components unscanned:
    the reference keeps their planes at zero (:627-632), so the buffer must be cleared."""
    seen = set()
    for sc in p.scans:
        seen.update(sc.comps)
    return len(seen) == p.ncomp


_PINNED_POOL: Dict[object, torch.Tensor] = {}     # keyed slots (one owner each, e.g. loader._Uploader)
_PINNED_FREE: List[torch.Tensor] = []             # checkout / release list shared by all threads
_PINNED_LOCK = threading.Lock()


_PINNED_LARGEST = 0


def _pinned_take(total: int) -> torch.Tensor:
    """A pinned buffer of at least `total` bytes from the free list, else a new one.  New buffers are never smaller
    than the largest one handed out so far: pinning costs ~0.7 ms per MB, and with sub-batches of several sizes a
    free list of mixed sizes would keep running out of buffers that fit the large ones."""
    global _PINNED_LARGEST
    with _PINNED_LOCK:
        best = None
        for i, t in enumerate(_PINNED_FREE):
            if t.numel() >= total and (best is None or t.numel() < _PINNED_FREE[best].numel()):
                best = i
        if best is not None:
            return _PINNED_FREE.pop(best)
        size = max(max(total, 1 << 20) * 5 // 4, _PINNED_LARGEST)
        _PINNED_LARGEST = size
    return torch.empty(size, dtype=torch.uint8, pin_memory=True)


def release_pinned(buf: torch.Tensor) -> None:
    """Give a buffer obtained with pack_files(reuse_slot="checkout") back (after the copy that reads it is done)."""
    pool = getattr(buf, "_bj_pool", None)
    if pool is None:
        return
    with _PINNED_LOCK:
        _PINNED_FREE.append(pool)
        if len(_PINNED_FREE) > 8:                  # keep the largest few
            _PINNED_FREE.sort(key=lambda t: t.numel())
            _PINNED_FREE.pop(0)


def read_files_packed(paths: Sequence, read_threads: Optional[int] = None, walk: bool = True) -> Tuple[torch.Tensor, List[int], List[int]]:
    """Read files STRAIGHT into one pinned host buffer (each file 16-byte aligned) with the C helper's host threads:
    the kernel's copy out of the page cache is the only host copy -- no intermediate bytes objects, no gather, no
    interpreter lock around 4096 open/read/close calls.  With walk=True every file is marker-walked and hashed right
    after it was read (buf._bj_walk, as pack_files(walk=True) does).  The buffer comes from the checkout pool (give it
    back with release_pinned()).  Returns (buffer, offsets, sizes); a missing / unreadable file raises OSError."""
    import errno as _errno
    L = _native.lib()
    if not getattr(L, "_read_bound", False):
        L.bj_host_stat_files.restype = None
        L.bj_host_stat_files.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        L.bj_host_read_files.restype = None
        L.bj_host_read_files.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_int]
        L._read_bound = True
    n = len(paths)
    threads = read_threads if read_threads else max(host_threads(), 1)
    cpaths = (ctypes.c_char_p * n)(*[os.fsencode(f) for f in paths])
    sizes64 = np.empty(n, dtype=np.int64)
    L.bj_host_stat_files(cpaths, n, sizes64.ctypes.data, threads)
    bad = np.nonzero(sizes64 < 0)[0]
    if len(bad):
        i = int(bad[0])
        e = int(-sizes64[i])
        raise OSError(e, os.strerror(e), str(paths[i]))
    sizes = sizes64.astype(np.uint64)
    padded = (sizes + np.uint64(15)) & ~np.uint64(15)
    offs = np.zeros(n, dtype=np.uint64)
    if n > 1:
        np.cumsum(padded[:-1], out=offs[1:])
    total = int(padded.sum()) + 64
    if torch.cuda.is_available():
        pool = _pinned_take(total)
        buf = pool[:total]
        buf._bj_pool = pool
    else:
        buf = torch.empty(total, dtype=torch.uint8)
    status = np.zeros(n, dtype=np.int32)
    if walk and n:
        from .fastplan import ENTRY_DTYPE, MAX_ENTRIES
        entries = np.empty((n, MAX_ENTRIES), dtype=ENTRY_DTYPE)
        counts = np.empty(n, dtype=np.int32)
        hashes = np.empty((n, 2), dtype=np.uint64)
        L.bj_host_read_files(cpaths, sizes.ctypes.data, offs.ctypes.data, n, buf.data_ptr(), status.ctypes.data,
                             entries.ctypes.data, MAX_ENTRIES, counts.ctypes.data, hashes.ctypes.data, threads)
        buf._bj_walk = (entries, counts, hashes)
    else:
        L.bj_host_read_files(cpaths, sizes.ctypes.data, offs.ctypes.data, n, buf.data_ptr(), status.ctypes.data,
                             None, 0, None, None, threads)
    bad = np.nonzero(status)[0]
    if len(bad):
        i = int(bad[0])
        release_pinned(buf)
        e = int(status[i])
        raise OSError(e, os.strerror(e) if e != _errno.EIO else "file changed while it was being read", str(paths[i]))
    return buf, [int(o) for o in offs], [int(x) for x in sizes]


def pack_files(datas: Sequence[bytes], pin: bool = True, reuse_slot=None, walk: bool = False) -> Tuple[torch.Tensor, List[int]]:
    """Concatenate file images into one (pinned) host buffer, each file 16-byte aligned.
    Returns (buffer, offsets); the sizes are len(datas[i]).  reuse_slot: pinning memory is slow, so allocations
    are kept.  "checkout": take a buffer from a shared free list and give it back with release_pinned() when the
    copy out of it has completed (thread safe); any other hashable value: a slot owned by the caller, overwritten
    by the next pack into the same slot."""
    offsets, total = [], 0
    for d in datas:
        offsets.append(total)
        total += (len(d) + 15) & ~15
    total += 64
    pinned = pin and torch.cuda.is_available()
    if reuse_slot == "checkout" and pinned:
        # a buffer from the shared free list (or a new one); the caller gives it back with release_pinned() once the
        # copy that reads it has completed -- safe with any number of threads / devices decoding at the same time
        pool = _pinned_take(total)
        buf = pool[:total]
        buf._bj_pool = pool
    elif reuse_slot is not None and pinned:
        pool = _PINNED_POOL.get(reuse_slot)
        if pool is None or pool.numel() < total:
            pool = torch.empty(max(total, 1 << 20) * 5 // 4, dtype=torch.uint8, pin_memory=True)
            _PINNED_POOL[reuse_slot] = pool
        buf = pool[:total]
    else:
        buf = torch.empty(total, dtype=torch.uint8, pin_memory=pinned)
    n = len(datas)
    if n >= 8 and all(type(d) is bytes for d in datas):
        # threaded gather in C (csrc/bj_host.cu): the pointers come straight from the bytes objects.  With
        # walk=True every file is also marker-walked and hashed right after it was copied (cache-hot); the result
        # rides along on the returned tensor (buf._bj_walk) and saves fastplan.plan_batch its own pass over the bytes.
        L = _native.lib()
        if not getattr(L, "_pack_bound", False):
            L.bj_host_pack.restype = None
            L.bj_host_pack.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
            L.bj_host_pack_walk_keys.restype = None
            L.bj_host_pack_walk_keys.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                                 ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
            L._pack_bound = True
        ptrs = (ctypes.c_char_p * n)(*datas)
        sizes = np.fromiter((len(d) for d in datas), dtype=np.uint64, count=n)
        offs = np.asarray(offsets, dtype=np.uint64)
        threads = host_threads()
        if walk:
            from .fastplan import ENTRY_DTYPE, MAX_ENTRIES
            entries = np.empty((n, MAX_ENTRIES), dtype=ENTRY_DTYPE)
            counts = np.empty(n, dtype=np.int32)
            hashes = np.empty((n, 2), dtype=np.uint64)
            L.bj_host_pack_walk_keys(ptrs, sizes.ctypes.data, offs.ctypes.data, n, buf.data_ptr(), entries.ctypes.data,
                                     MAX_ENTRIES, counts.ctypes.data, hashes.ctypes.data, threads)
            buf._bj_walk = (entries, counts, hashes)
        else:
            L.bj_host_pack(ptrs, sizes.ctypes.data, offs.ctypes.data, n, buf.data_ptr(), threads)
    else:
        view = buf.numpy()
        for d, off in zip(datas, offsets):
            view[off:off + len(d)] = np.frombuffer(d, dtype=np.uint8)
    return buf, offsets


_DESC_FIELDS = ("scans", "tile_scan", "lut", "images", "qtabs")


def descriptor_blob(plan) -> Tuple[np.ndarray, Dict[str, Tuple[int, int]]]:
    """All small per-batch arrays the kernels read (scan records, tile table, Huffman LUTs, image records, quantisation
    tables) as ONE byte blob with 256-byte aligned sections: one asynchronous copy from pinned memory instead of five
    blocking ones from pageable memory (each of which would wait for everything queued on the stream)."""
    parts = {"scans": plan.scans, "tile_scan": plan.tile_scan, "lut": plan.lut, "images": plan.geom.images,
             "qtabs": plan.geom.qtabs}
    layout: Dict[str, Tuple[int, int]] = {}
    total = 0
    for k in _DESC_FIELDS:
        a = np.ascontiguousarray(parts[k])
        total = (total + 255) & ~255
        layout[k] = (total, a.nbytes)
        total += a.nbytes
    blob = np.zeros(max(total, 16), dtype=np.uint8)
    for k in _DESC_FIELDS:
        a = np.ascontiguousarray(parts[k])
        o, n = layout[k]
        blob[o:o + n] = a.view(np.uint8).reshape(-1)
    return blob, layout


def upload_descriptors(plan, device, stream: torch.cuda.Stream, pinned: Optional[torch.Tensor] = None):
    """Copy descriptor_blob(plan) to the device on `stream` (non-blocking, from pinned memory).  Returns
    (device blob, layout, pinned staging buffer -- keep it alive until the copy has completed)."""
    blob, layout = descriptor_blob(plan)
    if pinned is None or pinned.numel() < blob.size:
        pinned = torch.empty(max(blob.size, 1 << 16) * 2, dtype=torch.uint8, pin_memory=True)
    pinned[:blob.size].numpy()[:] = blob
    with torch.cuda.device(device), torch.cuda.stream(stream):
        dev_blob = torch.empty(blob.size, dtype=torch.uint8, device=device)
        dev_blob.copy_(pinned[:blob.size], non_blocking=True)
    return dev_blob, layout, pinned


class _LazyViews:
    """Sequence of per-image (H, W, 3) / (H, W) views of the flat output buffer; a view is created when it is first
    asked for (a 4096-image batch would otherwise spend tens of milliseconds making views nobody may look at)."""

    def __init__(self, geom, out: torch.Tensor):
        """geom: anything with out_offsets / out_shapes (BatchGeometry, scaled.OutputLayout)."""
        self._g, self._out = geom, out
        self._cache: Dict[int, torch.Tensor] = {}

    def __len__(self) -> int:
        return len(self._g.out_offsets)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        v = self._cache.get(i)
        if v is None:
            off, shape = self._g.out_offsets[i], self._g.out_shapes[i]
            n = 1
            for d in shape:
                n *= int(d)
            v = self._out[off:off + n].view(*shape)
            self._cache[i] = v
        return v

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class DecodedBatch:
    """Result of decoding a batch on one device."""

    def __init__(self, plan: BatchPlan, out: torch.Tensor, coef: torch.Tensor, err: torch.Tensor, stats: dict,
                 layout=None):
        """layout: scaled.OutputLayout of `out` when the batch was decoded at reduced size or cropped (None: the
        planner's)."""
        self.plan = plan
        self.out = out
        self.coef = coef
        self.err = err
        self.stats = stats
        self._layout = layout
        self.images = _LazyViews(layout if layout is not None else plan.geom, out)    # (H, W, 3) / (H, W) uint8 device
                                                                                       # tensors, made on first use

    @property
    def layout(self):
        """scaled.OutputLayout: where each image's pixels lie in `out` (offset, pitch, size, channels)."""
        if self._layout is None:
            from .scaled import OutputLayout
            self._layout = OutputLayout.from_geometry(self.plan.geom)
        return self._layout

    def image_array(self, i: int) -> torch.Tensor:
        """The reference's layout: (W, H, 3) or (W, H) view (jpeg_decoder.py:626, :1373-1386)."""
        return self.images[i].transpose(0, 1)

    def start_host_copy(self, copy_stream: Optional[torch.cuda.Stream] = None, after: Optional[torch.cuda.Stream] = None) -> None:
        """Begin ONE device->host copy of all pixels of the batch into pinned memory (on `copy_stream`, after the work
        enqueued on `after` so far).  `host_image(i)` then hands out numpy views of that buffer: what the reference
        returns (`image_array`, host memory) at batch scale costs one large PCIe transfer instead of a pageable copy
        per image."""
        if getattr(self, "_host", None) is not None:
            return
        dev = self.out.device
        with torch.cuda.device(dev):
            cs = copy_stream if copy_stream is not None else torch.cuda.current_stream(dev)
            src = after if after is not None else torch.cuda.current_stream(dev)
            if cs is not src:
                ev = torch.cuda.Event()
                ev.record(src)
                cs.wait_event(ev)
            host = torch.empty(self.out.numel(), dtype=self.out.dtype, pin_memory=True)
            with torch.cuda.stream(cs):
                host.copy_(self.out, non_blocking=True)
                self.out.record_stream(cs)
                done = torch.cuda.Event()
                done.record(cs)
        self._host, self._host_done = host, done
        self._host_views = _LazyViews(self._layout if self._layout is not None else self.plan.geom, host)

    def host_image(self, i: int) -> Optional[np.ndarray]:
        """(H, W, 3) / (H, W) numpy view of image i in the pinned host copy (None if start_host_copy was not called)."""
        if getattr(self, "_host", None) is None:
            return None
        if self._host_done is not None:
            self._host_done.synchronize()
            self._host_done = None
        return self._host_views[i].numpy()

    def release_work_buffers(self, keep_coefficients: bool = False) -> None:
        """Drop everything but the pixels: the pipeline object with the un-stuffed bitstream, the decoder states and
        (unless asked to keep them) the coefficient planes -- as much memory again as the RGB output.  Safe right
        after the launches: the buffers were allocated on the stream the kernels run on, so the caching allocator
        hands them to later work of that stream only."""
        pipe = self.stats.pop("_pipe", None)
        if pipe is not None:
            coef = pipe.coef
            for name in ("raw", "words", "tile_sum", "stream_start", "stream_end", "stream_sub", "sub_entry", "sub_exit",
                         "sub_count", "sub_prefix", "chain", "coef", "blk_pos", "B"):
                setattr(pipe, name, None)
            if keep_coefficients:
                self.coef = coef
        if not keep_coefficients:
            self.coef = None

    def coefficient_grids(self, i: int) -> List[np.ndarray]:
        from .layout import device_to_grids, total_blocks
        if self.coef is None:
            raise RuntimeError("the coefficient planes of this sub-batch were released after decoding; "
                               "use decode_batch(..., keep_coefficients=True) or decode_stream(..., keep_coefficients=True)")
        p = self.plan.parsed[i]
        b0 = self.plan.geom.block_offsets[i]
        buf = self.coef[b0:b0 + total_blocks(p)].cpu().numpy()
        return device_to_grids(p, buf)


def error_for(word: int, i: int) -> Optional[Exception]:
    """The exception a device error word stands for (None if the image decoded): jpeg_decoder.py:1714-1725."""
    e = int(word)
    if e == 0:
        return None
    if e & _native.ERR_BAD_CODE:
        return CorruptedJpeg(f"Failed to decode image {i} (no Huffman code matches the data).")       # :718-719
    if e & (_native.ERR_OVERRUN | _native.ERR_RST_COUNT | _native.ERR_COEF_INDEX):
        return CorruptedJpeg(f"Failed to decode image {i} (entropy-coded data ended early or is inconsistent).")
    return NativeLibraryError(f"image {i}: device decode error {e:#x}")


def raise_for_errors(err_words: np.ndarray) -> None:
    """Map device error words to the reference's exception classes; raises for the first bad image."""
    bad = np.nonzero(err_words)[0]
    if len(bad):
        raise error_for(err_words[int(bad[0])], int(bad[0]))


class DevicePipeline:
    """Device buffers + launch sequence for one BatchPlan on one GPU.  Buffers are allocated once and
    can be reused for any number of batches with the same plan (bench.py does that); `upload` moves
    the file bytes, `launch` enqueues every kernel on the stream."""

    STAGES = ("unstuff", "plan", "spec", "fix", "write", "other_scans", "pixels")
    EXTRA_PHASE_FLAGS = 0                   # OR-ed into `phases` of bj_entropy_decode; tests set BJ_PHASE_NO_BITMAP (8)

    def __init__(self, plan: BatchPlan, device=None, stream: Optional[torch.cuda.Stream] = None,
                 raw: Optional[torch.Tensor] = None, desc: Optional[Tuple[torch.Tensor, Dict[str, Tuple[int, int]]]] = None):
        """raw: device copy of the packed file bytes, if the caller has already started it (see
        decode_batch_on_device: the H2D copy runs while the host is still planning).
        desc: (device blob, layout) from upload_descriptors(), if the caller uploaded the descriptors already."""
        self.plan = plan
        self.dev = require_cuda(device)
        self.L = _bind()
        self.extra_phase_flags = self.EXTRA_PHASE_FLAGS
        g = plan.geom
        dev = self.dev
        with torch.cuda.device(dev):
            self.stream = stream if stream is not None else torch.cuda.current_stream(dev)
            with torch.cuda.stream(self.stream):
                if desc is None:
                    desc_blob, layout, self._desc_pinned = upload_descriptors(plan, dev, self.stream)
                else:
                    desc_blob, layout = desc
                self._desc = desc_blob

                def sect(k):
                    o, n = layout[k]
                    return desc_blob[o:o + n]
                self.scans = sect("scans")
                self.tile_scan = sect("tile_scan")
                self.lut = sect("lut")
                self.dg = DeviceGeometry(g, dev, images=sect("images"), qtabs=sect("qtabs"))
                self.raw = raw if raw is not None else torch.empty(plan.raw_bytes, dtype=torch.uint8, device=dev)
                if self.raw.numel() != plan.raw_bytes or not self.raw.is_cuda:
                    raise ValueError("raw: wrong size or not a device tensor")
                self.words_len = plan.raw_bytes // 4 + 64
                self.words = torch.empty(self.words_len, dtype=torch.int32, device=dev)
                self.tile_sum = torch.empty(plan.n_tiles + 1, dtype=torch.int64, device=dev)
                self.stream_start = torch.empty(plan.n_streams, dtype=torch.int64, device=dev)
                self.stream_end = torch.empty(plan.n_streams, dtype=torch.int64, device=dev)
                self.stream_sub = torch.empty(plan.n_streams, dtype=torch.int32, device=dev)
                n_sub = max(plan.n_sub, 1)
                self.sub_entry = torch.empty(n_sub, dtype=torch.int64, device=dev)
                self.sub_exit = torch.empty(n_sub, dtype=torch.int64, device=dev)
                self.sub_count = torch.empty(n_sub * 4, dtype=torch.int32, device=dev)
                self.sub_prefix = torch.empty(n_sub * 4, dtype=torch.int32, device=dev)
                self.chain = torch.empty(plan.max_chain * 8, dtype=torch.int32, device=dev)
                self.coef = torch.empty((g.total_blocks, 64), dtype=torch.int16, device=dev)
                self.err = torch.zeros(len(plan.parsed), dtype=torch.int32, device=dev)
                self.sync_changes = torch.zeros(1, dtype=torch.int32, device=dev)
                # per-block start positions, only for batches with AC refinement scans
                self.blk_pos = (torch.empty(g.total_blocks, dtype=torch.int32, device=dev)
                                if any(grp.mode == 4 for grp in plan.groups) else None)
                self.out = None
                self.layout = None
        self.B = EntropyBuffers(self.words.data_ptr(), self.words_len, self.stream_start.data_ptr(),
                                self.stream_end.data_ptr(), self.stream_sub.data_ptr(), self.sub_entry.data_ptr(),
                                self.sub_exit.data_ptr(), self.sub_count.data_ptr(), self.sub_prefix.data_ptr(),
                                self.lut.data_ptr(), self.coef.data_ptr(), self.err.data_ptr(),
                                self.sync_changes.data_ptr(),
                                self.blk_pos.data_ptr() if self.blk_pos is not None else None)
        self.kernel_launches_per_step = 0

    def device_bytes(self) -> int:
        ts = [self.scans, self.tile_scan, self.lut, self.raw, self.words, self.tile_sum, self.stream_start,
              self.stream_end, self.stream_sub, self.sub_entry, self.sub_exit, self.sub_count, self.sub_prefix,
              self.chain, self.coef, self.err]
        return sum(t.numel() * t.element_size() for t in ts) + self.plan.geom.out_bytes

    def upload(self, raw_host: torch.Tensor) -> None:
        """H2D of the packed file bytes (async on the pipeline's stream when raw_host is pinned)."""
        with torch.cuda.device(self.dev), torch.cuda.stream(self.stream):
            self.raw.copy_(raw_host, non_blocking=True)

    def launch(self, out_kind: int = _native.OUT_RGB, upto_group: Optional[int] = None, events: Optional[dict] = None,
               scales=None, crops=None, compat: str = "reference"):
        """Enqueue un-stuffing, entropy decode and the pixel kernel.  With `events` (a dict), CUDA events
        are recorded around each stage: events[stage] = list of (start, end) pairs.
        scales: None (full size), or one scale / per-image scales in (1, 2, 4, 8) for RGB output at reduced size
        (scaled.launch); self.layout then describes the output.
        crops: None, or (n, 4) file boxes: only the pixels under each box are decoded, at the image's scale
        (crop.launch); self.layout then describes the output.
        compat: "reference", or "libjpeg-turbo": T.81 AC refinement and libjpeg-turbo's pixels (ijg.launch, full size
        only, with or without crops)."""
        L, plan, B = self.L, self.plan, self.B
        from .ijg import PHASE_T81_REFINE, check_compat
        ijg = check_compat(compat) == "libjpeg-turbo"
        if ijg:
            from .scaled import per_image
            if out_kind != _native.OUT_RGB:
                raise ValueError("a libjpeg-turbo decode gives RGB / grey output only")
            if scales is not None and (per_image(scales, len(plan.parsed)) != 1).any():
                check_compat(compat, scales)        # raises: full size only
        elif crops is not None:
            from . import crop
            if out_kind != _native.OUT_RGB:
                raise ValueError("a crop decode gives RGB / grey output only")
        elif scales is not None:
            from . import scaled
            if out_kind != _native.OUT_RGB:
                raise ValueError("a reduced-size decode gives RGB / grey output only")
            scales = scaled.per_image(scales, len(plan.parsed))
            if (scales == 1).all():
                scales = None
        s = self.stream
        cs = s.cuda_stream
        n_launch = 0

        def timed(name, fn):
            if events is None:
                fn()
                return
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            fn()
            b.record(s)
            events.setdefault(name, []).append((a, b))

        with torch.cuda.device(self.dev), torch.cuda.stream(s):
            if getattr(plan, "needs_zero", plan.any_progressive):
                self.coef.zero_()
            self.err.zero_()
            timed("unstuff", lambda: _native.check(L.bj_unstuff(
                self.raw.data_ptr(), self.scans.data_ptr(), len(plan.scans), self.tile_scan.data_ptr(), plan.n_tiles,
                self.tile_sum.data_ptr(), self.words.data_ptr(), self.stream_start.data_ptr(),
                self.stream_end.data_ptr(), plan.n_streams, cs), "bj_unstuff"))
            n_launch += 3
            timed("plan", lambda: _native.check(L.bj_entropy_plan(
                self.scans.data_ptr(), 0, len(plan.scans), self.tile_sum.data_ptr(), ctypes.byref(B), cs),
                "bj_entropy_plan"))
            n_launch += 1
            for gi, grp in enumerate(plan.groups):
                if upto_group is not None and gi >= upto_group:
                    break

                def call(phases, grp=grp):
                    phases |= self.extra_phase_flags
                    if ijg and grp.mode == 4:
                        phases |= PHASE_T81_REFINE
                    _native.check(L.bj_entropy_decode(
                        self.scans.data_ptr(), grp.first, grp.count, grp.mode, grp.max_sub, grp.max_streams,
                        grp.max_blocks, grp.max_lut, ctypes.byref(B), self.chain.data_ptr(), phases, cs),
                        "bj_entropy_decode")
                if grp.mode in (0, 1, 3):
                    if events is not None and grp.mode == 0:
                        timed("spec", lambda: call(1))
                        timed("fix", lambda: call(2))
                        timed("write", lambda: call(4))
                    else:
                        timed("other_scans" if grp.mode else "entropy", lambda: call(7))
                    n_launch += 4
                else:
                    timed("other_scans", lambda: call(7))
                    n_launch += 2 if grp.mode == 4 else 1
            if ijg:
                from . import ijg as ijg_mod
                holder = {}

                def pix_ijg():
                    holder["out"], holder["layout"] = ijg_mod.launch(self.dg, self.coef, crops, s)
                timed("pixels", pix_ijg)
                self.out, self.layout = holder["out"], holder["layout"]
                self._out_kind = None                   # the next reference launch allocates its own output
                n_launch += 2
            elif crops is not None:
                holder = {}

                def pix_crop():
                    holder["out"], holder["layout"] = crop.launch(self.dg, self.coef, 1 if scales is None else scales,
                                                                  crops, s)
                timed("pixels", pix_crop)
                self.out, self.layout = holder["out"], holder["layout"]
                self._out_kind = None                   # the next full-size launch allocates its own output
                n_launch += 1
            elif scales is not None:
                holder = {}

                def pix_scaled():
                    holder["out"], holder["layout"] = scaled.launch(self.dg, self.coef, scales, s)
                timed("pixels", pix_scaled)
                self.out, self.layout = holder["out"], holder["layout"]
                self._out_kind = None                   # the next full-size launch allocates its own output
                n_launch += int((scales > 1).any()) + int((scales == 1).any())
            else:
                if self.out is None or self._out_kind != out_kind:
                    self.out = None
                holder = {}

                def pix():
                    holder["out"] = run_pixels(self.dg, self.coef, _native.IN_COEF, out_kind, out=self.out, stream=s)
                timed("pixels", pix)
                self.out = holder["out"]
                self._out_kind = out_kind
                self.layout = None
                n_launch += 1
        self.kernel_launches_per_step = n_launch
        return self.out

    def result(self) -> "DecodedBatch":
        return DecodedBatch(self.plan, self.out, self.coef, self.err, {"sync_changes": self.sync_changes, "_pipe": self},
                            layout=self.layout)


def decode_batch_on_device(datas: Optional[Sequence[bytes]], device=None, parsed: Optional[Sequence[ParsedJpeg]] = None,
                           packed: Optional[Tuple[torch.Tensor, List[int]]] = None, check: bool = True,
                           stream: Optional[torch.cuda.Stream] = None, upto_wave: Optional[int] = None,
                           plan: Optional[BatchPlan] = None, out_kind: int = _native.OUT_RGB,
                           raw_dev: Optional[torch.Tensor] = None, raw_ready: Optional[torch.cuda.Event] = None,
                           desc=None, scales=None, crops=None, compat: str = "reference") -> DecodedBatch:
    """Decode a batch of JPEG file images on one GPU.  Returns device tensors; with check=True the
    per-image error words are read back (one synchronisation) and turned into exceptions.
    upto_wave=k stops the entropy stage after the first k scan groups (tests: per-scan parity).
    scales: None (full size), one scale or per-image scales in (1, 2, 4, 8), or a function of the planned batch's
    bj_image records that returns them (DevicePipeline.launch).
    crops: None, one file box, (n, 4) file boxes, or a function of the planned batch's bj_image records that returns
    them (crop.py); a box outside its image raises ValueError before anything is launched.
    compat: "reference" or "libjpeg-turbo" (ijg.py; full size only)."""
    require_cuda(device)
    if packed is None:
        packed = pack_files(datas, reuse_slot="checkout" if check else None,
                            walk=parsed is None and plan is None and len(datas) >= FAST_PLAN_MIN_FILES and upto_wave is None)
    raw_host, offsets = packed
    # start the host->device copy of the file bytes now: it overlaps the host-side planning below
    # (raw_dev / raw_ready: the caller already started it on another stream -- loader.py)
    dev = require_cuda(device)
    with torch.cuda.device(dev):
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        if raw_dev is None:
            with torch.cuda.stream(st):
                raw_dev = torch.empty(raw_host.numel(), dtype=torch.uint8, device=dev)
                raw_dev.copy_(raw_host, non_blocking=True)
        elif raw_ready is not None:
            st.wait_event(raw_ready)
    if plan is None:
        if parsed is None and datas is not None and len(datas) >= FAST_PLAN_MIN_FILES and upto_wave is None:
            from .fastplan import plan_batch
            plan = plan_batch(raw_host, offsets, [len(d) for d in datas], walked=getattr(raw_host, "_bj_walk", None))
        else:
            if parsed is None:
                parsed = [parse_jpeg(d) for d in datas]
            plan = BatchPlan(parsed, offsets, raw_host.numel(), serial_scans=upto_wave is not None)
    if crops is not None:
        from .crop import file_boxes
        crops = file_boxes(crops, plan.geom.images)
    pipe = DevicePipeline(plan, device, stream, raw=raw_dev, desc=desc)
    if callable(scales):
        scales = scales(plan.geom.images)
    pipe.launch(out_kind=out_kind, upto_group=upto_wave, scales=scales, crops=crops, compat=compat)
    res = pipe.result()
    if check:
        err = pipe.err.cpu().numpy()               # synchronises: the upload has long completed
        release_pinned(raw_host)
        raise_for_errors(err)
    return res
