"""CPU checks of decode_to_tensor (pyjpegdecoder_b200/tensor_out.py): the filter weights of csrc/bj_resize_math.cuh
against torch's antialiased bilinear interpolate, the roi -> pixel-box rule, argument errors (raised before any device
work) and the bj_resize_job mirror."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from hostsim import build


@pytest.fixture(scope="module")
def hs():
    L = build("resize_hostsim")
    L.hs_resize_weights.restype = None
    L.hs_resize_weights.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return L


def _weights(hs, n, m):
    w = np.empty((m, n), np.float32)
    lo = np.empty(m, np.int32)
    hi = np.empty(m, np.int32)
    hs.hs_resize_weights(n, m, w.ctypes.data, lo.ctypes.data, hi.ctypes.data)
    return w, lo, hi


def _pairs():
    rng = np.random.default_rng(2024)
    fixed = [(1, 1), (1, 7), (9, 1), (1, 300), (3000, 1), (224, 224), (88, 224), (120, 224), (1080, 224), (1920, 224),
             (61, 40), (97, 300), (4000, 2), (3000, 2), (2500, 2), (5, 5), (2, 3), (3, 2), (1000, 1000), (7, 1000)]
    out = list(fixed)
    while len(out) < 220:
        kind = rng.integers(0, 4)
        if kind == 0:                        # downscale
            m = int(rng.integers(1, 300)); n = int(m * rng.uniform(1.0, 12.0)) + 1
        elif kind == 1:                      # upscale
            n = int(rng.integers(1, 200)); m = int(n * rng.uniform(1.0, 8.0)) + 1
        elif kind == 2:                      # identity
            n = m = int(rng.integers(1, 500))
        else:                                # extreme downscale (n / m > 1000)
            m = int(rng.integers(1, 4)); n = int(m * rng.uniform(1001, 1400))
        out.append((n, m))
    return out


PAIRS = _pairs()


def test_weight_pairs_cover_the_required_cases():
    assert len(PAIRS) >= 200
    assert any(n == 1 for n, _ in PAIRS) and any(m == 1 for _, m in PAIRS)
    assert any(n < m for n, m in PAIRS) and any(n == m for n, m in PAIRS) and any(n / m > 1000 for n, m in PAIRS)


def test_weights_sum_to_one_and_identity_is_exact(hs):
    for n, m in PAIRS:
        w, lo, hi = _weights(hs, n, m)
        assert np.all(lo >= 0) and np.all(hi <= n) and np.all(hi > lo), (n, m)
        assert np.all(np.diff(lo) >= 0) and np.all(np.diff(hi) >= 0), (n, m)     # the kernel's tile box relies on it
        s = w.astype(np.float64).sum(1)
        assert np.abs(s - 1).max() <= 1e-6, (n, m, np.abs(s - 1).max())
        if n == m:
            assert np.array_equal(w, np.eye(n, dtype=np.float32)), n


def test_weights_match_torch_antialiased_bilinear(hs):
    """Each pair resizes one axis of a random image (the other axis, 5 pixels, stays), alternately the height and the
    width; compared with F.interpolate on the CPU."""
    rng = np.random.default_rng(7)
    for k, (n, m) in enumerate(PAIRS):
        w, _, _ = _weights(hs, n, m)
        w = w.astype(np.float64)
        if k % 2 == 0:
            img = rng.integers(0, 256, (n, 5)).astype(np.float32)
            got, size = w @ img, (m, 5)
        else:
            img = rng.integers(0, 256, (5, n)).astype(np.float32)
            got, size = img @ w.T, (5, m)
        want = F.interpolate(torch.from_numpy(img)[None, None], size=size, mode="bilinear", antialias=True,
                             align_corners=False)[0, 0].numpy()
        assert np.abs(got - want).max() <= 0.01, (n, m, np.abs(got - want).max())


def test_pixel_boxes_rule():
    from pyjpegdecoder_b200.tensor_out import _check_roi, pixel_boxes
    W, H = np.array([1920, 88, 100, 7]), np.array([1080, 120, 100, 3])
    assert pixel_boxes(None, W, H, (224, 224)).tolist() == [[0, 0, 1920, 1080], [0, 0, 88, 120], [0, 0, 100, 100],
                                                           [0, 0, 7, 3]]
    box = _check_roi((0.1, 0.2, 0.6, 0.9), 4)
    got = pixel_boxes(box, W, H, (224, 224))
    for (x0, y0, x1, y1), w, h in zip(got, W, H):
        px0 = min(np.floor(0.1 * w + 0.5), w - 1)
        py0 = min(np.floor(0.2 * h + 0.5), h - 1)
        assert (x0, y0) == (px0, py0)
        assert x1 == max(px0 + 1, min(w, np.floor(0.6 * w + 0.5)))
        assert y1 == max(py0 + 1, min(h, np.floor(0.9 * h + 0.5)))
    # a box thinner than a pixel still covers one pixel; boxes ending at 1 end at the edge
    tiny = pixel_boxes(_check_roi((0.999, 0.0, 1.0, 1.0), 1), [7], [3], (2, 2))
    assert tiny.tolist() == [[6, 0, 7, 3]]
    per = _check_roi([(0, 0, 1, 1), (0.5, 0.5, 1, 1), (0, 0, 0.5, 0.5), (0.25, 0, 0.75, 1)], 4)
    assert pixel_boxes(per, W, H, (224, 224)).tolist() == [[0, 0, 1920, 1080], [44, 60, 88, 120], [0, 0, 50, 50],
                                                          [2, 0, 5, 3]]


def test_center_box_landscape_portrait_square():
    from pyjpegdecoder_b200.tensor_out import pixel_boxes
    # landscape into a square: full height, centred width
    assert pixel_boxes("center", [1920], [1080], (224, 224)).tolist() == [[420, 0, 1500, 1080]]
    # portrait into a square: full width, centred height
    assert pixel_boxes("center", [88], [120], (224, 224)).tolist() == [[0, 16, 88, 104]]
    # square into a square: the whole image
    assert pixel_boxes("center", [100], [100], (224, 224)).tolist() == [[0, 0, 100, 100]]
    # output wider than the image: full width; bw = W, bh = floor(W * h / w + 0.5)
    assert pixel_boxes("center", [100], [100], (37, 301)).tolist() == [[0, 44, 100, 56]]
    # never empty
    assert pixel_boxes("center", [3], [1000], (1, 1000)).tolist() == [[0, 499, 3, 500]]
    b = pixel_boxes("center", [1000], [3], (1000, 1))
    assert b[0, 2] - b[0, 0] >= 1 and b[0, 3] - b[0, 1] == 3


@pytest.mark.parametrize("kwargs, what", [
    (dict(size=(0, 224)), "size"),
    (dict(size=(224, -1)), "size"),
    (dict(size=(224,)), "size"),
    (dict(roi=(0.5, 0.0, 0.5, 1.0)), "x1 <= x0"),
    (dict(roi=(0.0, 0.0, 1.5, 1.0)), "outside [0, 1]"),
    (dict(roi=(-0.1, 0.0, 0.5, 1.0)), "outside [0, 1]"),
    (dict(roi=[(0, 0, 1, 1)] * 3), "roi length"),
    (dict(roi="middle"), "roi string"),
    (dict(mean=(0.5, 0.5, 0.5)), "mean without std"),
    (dict(std=(0.5, 0.5, 0.5)), "std without mean"),
    (dict(mean=(0.5, 0.5), std=(0.5, 0.5)), "wrong length"),
    (dict(mean=(0.5, 0.5, 0.5), std=(0.5, 0.0, 0.5)), "zero std"),
    (dict(dtype=torch.uint8, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)), "mean with uint8"),
    (dict(dtype=torch.int32), "dtype"),
    (dict(on_error="ignore"), "on_error"),
    (dict(chunk=0), "chunk"),
])
def test_argument_errors_are_raised_before_device_work(kwargs, what, monkeypatch):
    from pyjpegdecoder_b200 import decode_to_tensor, loader, stages   # noqa: F401 (modules that bind require_cuda
                                                                      # at import are imported before the patch)

    def no_device(*a, **k):
        raise AssertionError("device work started before the arguments were checked")
    monkeypatch.setattr(stages, "require_cuda", no_device)
    with pytest.raises(ValueError):
        decode_to_tensor([b"x", b"y"], **kwargs)


def test_resize_job_mirror_matches_the_library():
    from pyjpegdecoder_b200 import _native
    from pyjpegdecoder_b200.tensor_out import RESIZE_JOB_DTYPE, ResizeParams, _bind
    L = _bind()
    assert L.bj_sizeof(1) == RESIZE_JOB_DTYPE.itemsize == 40
    assert ctypes.sizeof(ResizeParams) == 40
    assert _native.lib().bj_sizeof(0) == 72


def test_decode_to_tensor_needs_a_gpu_and_never_falls_back():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from pyjpegdecoder_b200 import NativeLibraryError, decode_to_tensor
    with pytest.raises(NativeLibraryError):
        decode_to_tensor([b"\xff\xd8"], size=(8, 8))
