"""CPU checks of decode_to_tensor(resample="pil-bilinear" | "pil-bicubic", resize=): tests/pil_resample_ref.py equals
Pillow's Image.resize, which pins the definition to Pillow on any machine; csrc/bj_resize_pil_math.cuh (host build,
tests/hostsim/resize_pil_hostsim.cpp) equals the reference on the coefficient tables and on both passes, and stays
inside the int32 bound it derives; the resize= geometry equals torchvision's Resize + CenterCrop; argument errors;
the bj_resize_pil_job mirror."""
import ctypes

import numpy as np
import pytest
from PIL import Image

import pil_resample_ref as ref
from hostsim import build

FILTERS = {"bilinear": (0, Image.BILINEAR), "bicubic": (1, Image.BICUBIC)}


@pytest.fixture(scope="module")
def hs():
    L = build("resize_pil_hostsim")
    L.hs_pil_ksize.restype = ctypes.c_int
    L.hs_pil_ksize.argtypes = [ctypes.c_int] * 3
    L.hs_pil_coeffs.restype = None
    L.hs_pil_coeffs.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3
    L.hs_pil_resize.restype = None
    L.hs_pil_resize.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.c_void_p]
    L.hs_pil_partial_extremes.restype = None
    L.hs_pil_partial_extremes.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 2
    return L


def _cases():
    """(H, W, h, w): 1 x 1 up to several hundred, upscales, downscales up to 64x, one axis only."""
    rng = np.random.default_rng(5)
    out = [(1, 1, 1, 1), (1, 1, 7, 5), (5, 3, 1, 1), (2, 3, 3, 2), (17, 20, 17, 9), (17, 20, 40, 20), (9, 640, 9, 10),
           (640, 9, 10, 9), (448, 384, 7, 6), (384, 448, 6, 7), (300, 257, 300, 257), (31, 29, 311, 290),
           (120, 88, 224, 224), (341, 500, 256, 375)]
    for _ in range(24):
        H, W = (int(v) for v in rng.integers(1, 420, 2))
        h, w = (int(v) for v in rng.integers(1, 330, 2))
        out.append((H, W, h, w))
    return out


CASES = _cases()


def _img(H, W, channels, seed):
    rng = np.random.default_rng(seed)
    shape = (H, W) if channels == 1 else (H, W, channels)
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    # saturated patches: the clip8 ends of both passes
    img[: H // 3, : W // 3] = 255
    img[H // 2:, W // 2:][::2] = 0
    return img


@pytest.mark.parametrize("name", sorted(FILTERS))
@pytest.mark.parametrize("mode", ["RGB", "L"])
def test_reference_equals_pillow(name, mode):
    for k, (H, W, h, w) in enumerate(CASES):
        img = _img(H, W, 3 if mode == "RGB" else 1, k)
        want = np.asarray(Image.fromarray(img, mode).resize((w, h), FILTERS[name][1]))
        got = ref.resize(img, w, h, name)
        assert np.array_equal(got, want), (H, W, h, w, name, mode)


def _hs_coeffs(hs, n, m, f):
    ks = hs.hs_pil_ksize(n, m, f)
    xmin = np.empty(m, np.int32)
    cnt = np.empty(m, np.int32)
    k = np.empty((m, ks), np.int32)
    hs.hs_pil_coeffs(n, m, f, xmin.ctypes.data, cnt.ctypes.data, k.ctypes.data)
    return xmin, cnt, k


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_header_coefficients_equal_the_reference(hs, name):
    pairs = {(n, m) for H, W, h, w in CASES for n, m in ((H, h), (W, w))} | {(4160, 65), (2340, 7), (1, 300)}
    for n, m in sorted(pairs):
        xmin, cnt, k = _hs_coeffs(hs, n, m, FILTERS[name][0])
        rx, rn, rk = ref.coeffs(n, m, name)
        assert np.array_equal(xmin, rx) and np.array_equal(cnt, rn) and np.array_equal(k, rk), (n, m, name)


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_header_passes_equal_the_reference(hs, name):
    for k, (H, W, h, w) in enumerate(CASES[:20]):
        for C in (3, 1):
            img = np.ascontiguousarray(_img(H, W, C, 100 + k).reshape(H, W, C))
            out = np.empty((h, w, C), np.uint8)
            hs.hs_pil_resize(img.ctypes.data, W, H, C, w, h, FILTERS[name][0], out.ctypes.data)
            assert np.array_equal(out, ref.resize(img, w, h, name)), (H, W, h, w, C, name)


def test_partial_sums_reach_the_bound_and_stay_in_int32(hs):
    """The header's bound: every partial sum lies in [2^21 - 255 K-, 2^21 + 255 K+] and in
    (2^21 - 255 * 0.95 * 2^22, 2^21 + 255 * 1.95 * 2^22); the adversarial inputs reach the row bound exactly."""
    r = 1 << 21
    top, bottom = r + 255 * 1.95 * (1 << 22), r - 255 * 0.95 * (1 << 22)
    seen_hi = seen_lo = r
    ins = [1, 2, 3, 5, 7, 13, 100, 640, 1920, 4160]
    for name in sorted(FILTERS):
        f = FILTERS[name][0]
        for n in ins:
            # ratios around the cases of the derivation: upscales, 1 <= s < 2, 2 <= s < 3, s >= 3, s up to 64 and more
            for m in sorted({max(1, int(n / s)) for s in (0.3, 1.0, 1.1, 1.37, 1.5, 1.9, 2.0, 2.5, 2.9, 3.3, 8.6, 64.0,
                                                           n)} | {n * 3}):
                hi, lo = ctypes.c_int64(), ctypes.c_int64()
                hs.hs_pil_partial_extremes(n, m, f, ctypes.byref(hi), ctypes.byref(lo))
                _, cnt, k = ref.coeffs(n, m, name)
                kp = np.where(k > 0, k, 0).sum(1).max()
                kn = np.where(k < 0, -k, 0).sum(1).max()
                assert hi.value == r + 255 * kp and lo.value == r - 255 * kn, (n, m, name)
                assert bottom < lo.value <= hi.value < top < 2 ** 31, (n, m, name)
                seen_hi, seen_lo = max(seen_hi, hi.value), min(seen_lo, lo.value)
    assert seen_lo < r < seen_hi        # bicubic's negative lobes were exercised


@pytest.mark.parametrize("size", [(224, 224), (223, 225), (225, 223), (1, 1), (7, 300)])
@pytest.mark.parametrize("r", [300, 301, 511])
def test_resize_geometry_equals_torchvision(size, r):
    from torchvision import transforms as T
    from pyjpegdecoder_b200.tensor_out import resize_geometry
    h, w = size
    dims = [(301, 301), (333, 517), (517, 333), (640, 427), (427, 640), (301, 302), (303, 1001), (999, 401)]
    W = np.array([d[0] for d in dims])
    H = np.array([d[1] for d in dims])
    vw, vh, wx, wy = resize_geometry(W, H, r, size)
    tf = T.Compose([T.Resize(r, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(size)])
    for i, (Wi, Hi) in enumerate(dims):
        img = _img(Hi, Wi, 3, i)
        want = np.asarray(tf(Image.fromarray(img)))
        full = ref.resize(img, int(vw[i]), int(vh[i]), "bicubic") if (vw[i], vh[i]) != (Wi, Hi) else img
        got = full[wy[i]:wy[i] + h, wx[i]:wx[i] + w]
        assert np.array_equal(got, want), (Wi, Hi, r, size)


@pytest.mark.parametrize("kwargs", [
    dict(resample="pil-lanczos"),
    dict(resample="PIL-bilinear"),
    dict(resample=None),
    dict(resize=256),                                           # resample="torch"
    dict(resize=256, resample="pil-bilinear", roi="center"),
    dict(resize=256, resample="pil-bicubic", roi=(0.0, 0.0, 0.5, 0.5)),
    dict(resize=223, resample="pil-bilinear"),                  # below size
    dict(resize=256, resample="pil-bilinear", size=(224, 300)),  # a portrait image would be 256 wide
    dict(resize=0, resample="pil-bilinear", size=(1, 1)),
    dict(resize=256.0, resample="pil-bilinear"),
    dict(resize=True, resample="pil-bilinear", size=(1, 1)),
])
def test_argument_errors_are_raised_before_device_work(kwargs, monkeypatch):
    from pyjpegdecoder_b200 import decode_to_tensor, loader, stages   # noqa: F401 (modules that bind require_cuda
                                                                      # at import are imported before the patch)

    def no_device(*a, **k):
        raise AssertionError("device work started before the arguments were checked")
    monkeypatch.setattr(stages, "require_cuda", no_device)
    kwargs = dict(kwargs)
    size = kwargs.pop("size", (224, 224))
    with pytest.raises(ValueError):
        decode_to_tensor([b"x", b"y"], size=size, **kwargs)


def test_resize_pil_job_mirror_matches_the_library():
    from pyjpegdecoder_b200.tensor_out import RESIZE_PIL_JOB_DTYPE, _bind
    L = _bind()
    assert L.bj_sizeof(4) == RESIZE_PIL_JOB_DTYPE.itemsize == 56
