"""CPU checks of the crop decode (pyjpegdecoder_b200/crop.py): argument errors (raised before any device work), the
box rule against a brute-force count of the scaled pixels and MCUs a box touches, the output layout, the bj_crop_job
mirror, and the crops decode_to_tensor(roi=) asks for."""
import numpy as np
import pytest

from pyjpegdecoder_b200 import crop

# (hmax, vmax) of the layouts: 4:4:4 / grey, 4:2:2, 4:4:0, 4:2:0
SAMPLING = [(1, 1), (2, 1), (1, 2), (2, 2)]


def _images(sizes, ncomp=3, hmax=1, vmax=1, strip=8):
    from pyjpegdecoder_b200._native import IMAGE_DTYPE
    rec = np.zeros(len(sizes), IMAGE_DTYPE)
    rec["width"] = [w for w, _ in sizes]
    rec["height"] = [h for _, h in sizes]
    rec["ncomp"] = ncomp
    rec["hmax"], rec["vmax"] = hmax, vmax
    rec["mcus_x"] = [-(-w // (8 * hmax)) for w, _ in sizes]
    rec["mcus_y"] = [-(-h // (8 * vmax)) for _, h in sizes]
    rec["blocks_per_mcu"] = hmax * vmax + (2 if ncomp == 3 else 0)
    rec["strip_mcus"] = strip
    return rec


@pytest.mark.parametrize("bad, msg", [
    ((0, 0, 10), "integer pixels"),
    ((0, 0, 10, 10.0), "integer pixels"),
    ((0, 0, True, 10), "integer pixels"),
    (("0", 0, 10, 10), "per-file crop boxes need a sized|boxes for"),
    ((-1, 0, 10, 10), "x0 >= 0"),
    ((0, -3, 10, 10), "x0 >= 0"),
    ((5, 0, 5, 10), "x1 > x0"),
    ((0, 7, 10, 2), "x1 > x0"),
    (np.array([0, 0, 4, 4], np.float64), "integer pixels"),
    (np.zeros((2, 3), np.int64), "shape"),
    (np.ones((2, 4), np.float32), "integer dtype"),
    ([(0, 0, 4, 4)] * 3, "3 boxes for 2 files"),
    ([(0, 0, 4, 4), (1, 1, 1, 2)], "x1 > x0"),
    (7, "one box"),
])
def test_argument_errors(bad, msg):
    with pytest.raises(ValueError, match=msg):
        crop.check_crop(bad, 2)


def test_one_box_and_per_file_boxes():
    one = crop.check_crop((1, 2, 30, 40), 3)
    assert not one.per_file and one([], [0, 1, 2]).tolist() == [[1, 2, 30, 40]] * 3
    arr = crop.check_crop(np.array([[0, 0, 4, 4], [1, 1, 5, 5]], np.int32), 2)
    assert arr.per_file and arr(None, [1]).tolist() == [[1, 1, 5, 5]]
    four = crop.check_crop([(0, 0, 1, 1), (0, 0, 2, 2), (0, 0, 3, 3), (0, 0, 4, 4)], 4)
    assert four.per_file and four.boxes[3].tolist() == [0, 0, 4, 4]
    assert crop.check_crop(np.array([3, 4, 5, 6], np.uint16), 9).boxes.tolist() == [3, 4, 5, 6]
    assert crop.check_crop(None, 2) is None
    with pytest.raises(ValueError, match="sized"):
        crop.check_crop([(0, 0, 1, 1)], None)


def test_outside_boxes():
    b = np.array([[10, 0, 20, 5], [0, 9, 3, 20], [9, 8, 100, 100]])
    assert crop.outside(b, [10, 10, 10], [9, 9, 9]).tolist() == [True, True, False]
    with pytest.raises(ValueError, match="outside the 10 x 9 image"):
        crop.scaled_boxes(b, [10] * 3, [9] * 3, [1] * 3)
    with pytest.raises(ValueError, match="outside"):
        crop.file_boxes(b[:1], _images([(10, 9)]))


@pytest.mark.parametrize("hmax, vmax", SAMPLING)
@pytest.mark.parametrize("s", [1, 2, 4, 8])
def test_box_rule_against_brute_force(hmax, vmax, s):
    """Scaled box = the scaled pixels whose full-size footprint [k s, (k+1) s) meets the clipped box; window = the
    MCUs holding those pixels."""
    mw, mh = 8 * hmax // s, 8 * vmax // s
    for W, H in [(1, 1), (5, 3), (17, 9), (33, 18)]:
        Ws, Hs = -(-W // s), -(-H // s)
        boxes = [(x0, y0, x1, y1) for x0 in range(W) for x1 in range(x0 + 1, W + 3)
                 for y0 in range(0, H, max(1, H // 3)) for y1 in (y0 + 1, H, H + 4) if y1 > y0]
        b = np.asarray(boxes, np.int64)
        n = len(b)
        sb = crop.scaled_boxes(b, [W] * n, [H] * n, [s] * n)
        win = crop.windows(sb, [hmax] * n, [vmax] * n, [s] * n)
        for (x0, y0, x1, y1), got, w in zip(boxes, sb, win):
            xs = [k for k in range(Ws) if k * s < min(x1, W) and (k + 1) * s > x0]
            ys = [k for k in range(Hs) if k * s < min(y1, H) and (k + 1) * s > y0]
            assert got.tolist() == [xs[0], ys[0], xs[-1] + 1, ys[-1] + 1], (W, H, s, (x0, y0, x1, y1))
            mx = sorted({k // mw for k in xs})
            my = sorted({k // mh for k in ys})
            assert w.tolist() == [mx[0], my[0], mx[-1] + 1, my[-1] + 1]
            assert mx == list(range(mx[0], mx[-1] + 1))


def test_layout_offsets_aligned_and_sizes():
    rec = _images([(1920, 1080), (61, 517), (333, 71), (7, 9)])
    rec["ncomp"][1] = 1
    boxes = np.array([[3, 5, 964, 546], [0, 0, 61, 517], [1, 1, 2, 2], [0, 0, 100, 100]])
    sb = crop.scaled_boxes(boxes, rec["width"], rec["height"], [1, 2, 4, 1])
    lay = crop.layout(rec, sb)
    assert lay.out_shapes == [(541, 961, 3), (259, 31), (1, 1, 3), (9, 7, 3)]
    assert (lay.offsets % 16 == 0).all()
    assert lay.pitches.tolist() == [961 * 3, 31, 3, 21]
    ends = lay.offsets + lay.heights * lay.pitches
    assert (ends[:-1] <= lay.offsets[1:]).all()
    assert lay.out_bytes == int(ends[-1])


def test_jobs_and_strips():
    rec = _images([(1920, 1080)] * 3, hmax=2, vmax=2, strip=32)
    rec["layout"] = 1
    rec["blocks_per_mcu"] = 6
    boxes = np.array([[0, 0, 1920, 1080], [480, 270, 1440, 810], [0, 0, 1920, 1080]])
    jobs, lay, max_strips, kinds = crop.jobs_for(rec, boxes, np.array([1, 1, 4]))
    assert kinds == (1 << 1) | crop.CROP_SCALED
    # full frame at s = 1: 68 MCU rows x ceil(120 / 32) strips; centre box: 35 rows x ceil(60 / 32)
    assert max_strips == 68 * 4
    assert jobs["log2_scale"].tolist() == [0, 0, 2]
    assert jobs[1][["x0", "y0", "x1", "y1"]].tolist() == (480, 270, 1440, 810)
    assert jobs[2][["x1", "y1"]].tolist() == (480, 270)
    assert jobs["out_offset"].tolist() == lay.offsets.tolist()


def test_crop_job_mirror_matches_the_library():
    L = crop._bind()
    assert L.bj_sizeof(3) == crop.CROP_JOB_DTYPE.itemsize == 40


@pytest.mark.parametrize("bad", [(0, 0, 1.5, 3), (0, 0, 0, 3), [(0, 0, 2, 2)] * 3])
def test_bad_crops_are_rejected_before_device_work(bad, monkeypatch):
    from pyjpegdecoder_b200 import decode_batch, decode_stream, loader, stages   # noqa: F401

    def no_device(*a, **k):
        raise AssertionError("device work started before the arguments were checked")
    monkeypatch.setattr(stages, "require_cuda", no_device)
    monkeypatch.setattr(loader, "require_cuda", no_device)
    with pytest.raises(ValueError):
        decode_batch([b"x", b"y"], crop=bad)
    with pytest.raises(ValueError):
        next(decode_stream([b"x", b"y"], crop=bad))
    with pytest.raises(ValueError, match="sized"):
        next(decode_stream(iter([b"x", b"y"]), crop=[(0, 0, 1, 1), (0, 0, 2, 2)]))


@pytest.mark.parametrize("seed", range(6))
def test_decode_to_tensor_requests_todays_box(seed):
    """The crop decode_to_tensor asks for, taken through the box rule at the file's scale, is exactly today's
    pixel_boxes box on the image decoded at that scale: each resize job keeps its box size and its source bytes."""
    from pyjpegdecoder_b200.tensor_out import _AutoScales, _check_roi, _RoiCrops, pixel_boxes
    rng = np.random.default_rng(seed)
    n = 64
    sizes = [(int(rng.integers(1, 3000)), int(rng.integers(1, 3000))) for _ in range(n)]
    rec = _images(sizes)
    size = (int(rng.integers(1, 400)), int(rng.integers(1, 400)))
    x0, y0 = rng.uniform(0, 0.9, n), rng.uniform(0, 0.9, n)
    per_file = np.stack([x0, y0, x0 + rng.uniform(1e-3, 1 - x0), y0 + rng.uniform(1e-3, 1 - y0)], 1)
    for roi in ("center", (0.1, 0.2, 0.7, 0.9), per_file.tolist()):
        roi = _check_roi(roi, n)
        for scale in (1, 2, 4, 8, "auto"):
            scales = _AutoScales(roi, size) if scale == "auto" else (None if scale == 1 else scale)
            idx = np.arange(n)
            got = _RoiCrops(roi, size, scales)(rec, idx)
            s = scales(rec, idx) if callable(scales) else np.full(n, scale)
            W, H = rec["width"].astype(np.int64), rec["height"].astype(np.int64)
            want = pixel_boxes(roi, -(-W // s), -(-H // s), size)
            assert not crop.outside(got, W, H).any()
            assert np.array_equal(crop.scaled_boxes(got, W, H, s), want)
