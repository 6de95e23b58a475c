"""GPU checks of decode_to_tensor(resample="pil-bilinear" | "pil-bicubic", resize=) (csrc/bj_resize_pil.cu): with
compat="libjpeg-turbo" the uint8 output is torch.equal to Pillow's Image.open -> convert("RGB") -> crop -> resize for
every roi kind, both filters, up- and downscales; resize= equals torchvision's Resize + CenterCrop; float dtypes are the
fold of the uint8 result; streamed, on_error="return", channels_last and greyscale paths give the same bytes;
compat="reference" and reduced scales equal the numpy reference on their decoded pixels."""
import io

import numpy as np
import pytest

import ijg_ref
import pil_resample_ref as ref
from conftest import GOLDEN
from test_ijg_cpu import WRAP
from test_tensor_out_gpu import MEAN, STD, _golden, _pil, _rois

pytestmark = pytest.mark.gpu

LJT = "libjpeg-turbo"
FILTERS = {"pil-bilinear": "bilinear", "pil-bicubic": "bicubic"}


def _pil_filter(resample):
    from PIL import Image
    return Image.BILINEAR if resample == "pil-bilinear" else Image.BICUBIC


@pytest.fixture(scope="module")
def files():
    return _golden() + [(GOLDEN / "base_image.jpg").read_bytes(), _pil(1920, 1080, 1), _pil(1920, 1080, 2),
                        _pil(1080, 1920, 3, progressive=True), _pil(61, 517, 4, mode="L"), _pil(333, 71, 5)]


def _opened(files):
    """Pillow's decode; for WRAP, whose dequantised products leave int16 where Pillow's SIMD IDCT and libjpeg-turbo's C
    arithmetic disagree, the C arithmetic (ijg_ref) that compat="libjpeg-turbo" reproduces."""
    from PIL import Image
    wrap = (GOLDEN / "cases" / f"{WRAP}.jpg").read_bytes()
    return [Image.fromarray(ijg_ref.decode(f)) if f == wrap else Image.open(io.BytesIO(f)).convert("RGB")
            for f in files]


def _want(imgs, roi, size, resample):
    import torch
    from pyjpegdecoder_b200.tensor_out import _check_roi, pixel_boxes
    boxes = pixel_boxes(_check_roi(roi, len(imgs)), [i.width for i in imgs], [i.height for i in imgs], size)
    out = [np.asarray(im.crop(tuple(int(v) for v in b)).resize((size[1], size[0]), _pil_filter(resample)))
           for im, b in zip(imgs, boxes)]
    return torch.from_numpy(np.stack(out)).permute(0, 3, 1, 2).contiguous()


@pytest.mark.parametrize("size", [(224, 224), (37, 301), (600, 1000), (37, 30)])   # (37, 30): chunked tap tables
@pytest.mark.parametrize("roi_name", ["none", "box", "per_image", "center"])
@pytest.mark.parametrize("resample", sorted(FILTERS))
def test_uint8_equals_pillow(files, size, roi_name, resample):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    roi = _rois(len(files))[roi_name]
    got = decode_to_tensor(files, size, roi=roi, dtype=torch.uint8, compat=LJT, resample=resample, device="cuda:0")
    want = _want(_opened(files), roi, size, resample)
    for i in range(len(files)):
        assert torch.equal(got[i].cpu(), want[i]), (i, size, roi_name, resample)


@pytest.mark.parametrize("resample", sorted(FILTERS))
def test_resize_center_crop_equals_torchvision(files, resample):
    import torch
    from torchvision import transforms as T
    from pyjpegdecoder_b200 import decode_to_tensor
    mode = T.InterpolationMode.BILINEAR if resample == "pil-bilinear" else T.InterpolationMode.BICUBIC
    tf = T.Compose([T.Resize(256, interpolation=mode), T.CenterCrop(224), T.PILToTensor()])
    want = torch.stack([tf(im) for im in _opened(files)])
    got = decode_to_tensor(files, (224, 224), dtype=torch.uint8, compat=LJT, resample=resample, resize=256,
                           device="cuda:0")
    assert torch.equal(got.cpu(), want)
    # the whole preprocessing of a timm / torchvision eval transform, in fp32
    tf32 = T.Compose([T.Resize(256, interpolation=mode), T.CenterCrop(224), T.ToTensor(), T.Normalize(MEAN, STD)])
    want32 = torch.stack([tf32(im) for im in _opened(files)])
    got32 = decode_to_tensor(files, (224, 224), dtype=torch.float32, mean=MEAN, std=STD, compat=LJT,
                             resample=resample, resize=256, device="cuda:0")
    assert (got32.cpu() - want32).abs().max().item() <= 1e-6


@pytest.mark.parametrize("resample", sorted(FILTERS))
def test_resize_of_extreme_aspects_equals_torchvision(resample):
    """Virtual sizes beyond 65535: a 20000 x 70 panorama at resize=256 is 73142 wide, an 8192 x 256 strip at
    resize=2048 is 65536 wide."""
    import torch
    from torchvision import transforms as T
    from pyjpegdecoder_b200 import decode_to_tensor
    mode = T.InterpolationMode.BILINEAR if resample == "pil-bilinear" else T.InterpolationMode.BICUBIC
    for (w, h), r in (((20000, 70), 256), ((8192, 256), 2048)):
        f = _pil(w, h, 9)
        tf = T.Compose([T.Resize(r, interpolation=mode), T.CenterCrop(224), T.PILToTensor()])
        want = tf(_opened([f])[0])
        got = decode_to_tensor([f], (224, 224), dtype=torch.uint8, compat=LJT, resample=resample, resize=r,
                               device="cuda:0")
        assert torch.equal(got[0].cpu(), want), (w, h, r)


def test_virtual_size_beyond_int32_raises():
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    f = _pil(65500, 1, 10)                                 # resize=40000 makes it 40000 * 65500 > 2^31 - 1 long
    with pytest.raises(ValueError, match="pixels long"):
        decode_to_tensor([f], (224, 224), dtype=torch.uint8, resample="pil-bilinear", resize=40000, device="cuda:0")


@pytest.mark.parametrize("dtype_name", ["float16", "bfloat16", "float32"])
def test_float_dtypes_are_the_fold_of_uint8(files, dtype_name):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    dtype = getattr(torch, dtype_name)
    kw = dict(roi="center", compat=LJT, resample="pil-bicubic", device="cuda:0")
    u8 = decode_to_tensor(files, (160, 200), dtype=torch.uint8, **kw)
    for mean, std in ((None, None), (MEAN, STD)):
        got = decode_to_tensor(files, (160, 200), dtype=dtype, mean=mean, std=std, **kw)
        m = torch.tensor(mean if mean else (0.0, 0.0, 0.0), dtype=torch.float64, device="cuda:0").view(1, 3, 1, 1)
        s = torch.tensor(std if std else (1.0, 1.0, 1.0), dtype=torch.float64, device="cuda:0").view(1, 3, 1, 1)
        a = (1.0 / (255.0 * s)).float().double()          # the fold's fp32 constants (tensor_out._fold_norm)
        b = (-m / s).float().double()
        # v * a + b is exact in fp64, so one rounding to fp32 is the kernel's fmaf
        want = (u8.double() * a + b).float().to(dtype)
        assert torch.equal(got, want), (dtype_name, mean)


def test_paths_agree(files):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    kw = dict(dtype=torch.uint8, compat=LJT, resample="pil-bilinear", device="cuda:0")
    base = decode_to_tensor(files, (96, 128), roi="center", **kw)
    streamed = decode_to_tensor(files, (96, 128), roi="center", chunk=max(2, len(files) // 3), **kw)
    assert len(files) > 1.5 * max(2, len(files) // 3)
    assert torch.equal(streamed, base)
    cl = decode_to_tensor(files, (96, 128), roi="center", channels_last=True, **kw)
    assert cl.is_contiguous(memory_format=torch.channels_last) and torch.equal(cl, base)
    bad = files[:3] + [b"\xff\xd8 not a jpeg"] + files[3:]
    t, errs = decode_to_tensor(bad, (96, 128), roi="center", on_error="return", **kw)
    assert errs[3] is not None and all(e is None for k, e in enumerate(errs) if k != 3)
    assert torch.equal(t[:3], base[:3]) and torch.equal(t[4:], base[3:]) and not t[3].any()
    for chunk in (None, 4):
        a = decode_to_tensor(files, (224, 224), resize=256, chunk=chunk, **kw)
        b, errs = decode_to_tensor(files, (224, 224), resize=256, chunk=chunk, on_error="return", **kw)
        assert torch.equal(a, b) and all(e is None for e in errs)


def test_greyscale_gives_three_equal_channels():
    import torch
    from PIL import Image
    from pyjpegdecoder_b200 import decode_to_tensor
    grey = [_pil(61, 517, 4, mode="L"), _pil(641, 479, 6, mode="L", progressive=True)]
    got = decode_to_tensor(grey, (100, 90), dtype=torch.uint8, compat=LJT, resample="pil-bicubic", device="cuda:0")
    for g, f in zip(got, grey):
        want = np.asarray(Image.open(io.BytesIO(f)).resize((90, 100), Image.BICUBIC))
        for c in range(3):
            assert torch.equal(g[c].cpu(), torch.from_numpy(want.copy()))


@pytest.mark.parametrize("resample", sorted(FILTERS))
def test_reference_compat_and_scales_equal_the_numpy_reference(resample):
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    from pyjpegdecoder_b200.scaled import auto_scales
    from pyjpegdecoder_b200.tensor_out import resize_geometry
    name = FILTERS[resample]
    files = [_pil(1920, 1080, 1), _pil(1080, 1920, 3, progressive=True), _pil(333, 71, 5), _pil(61, 517, 4, mode="L")]

    def decoded(scale):
        return [d.image_tensor.cpu().numpy() for d in decode_batch(files, device="cuda:0", scale=scale)]

    def rgb(a):
        return np.repeat(a[..., None], 3, -1) if a.ndim == 2 else a

    for scale in (1, 2, 8):
        got = decode_to_tensor(files, (120, 160), dtype=torch.uint8, resample=resample, scale=scale, device="cuda:0")
        for g, img in zip(got, decoded(scale)):
            assert np.array_equal(g.permute(1, 2, 0).cpu().numpy(), ref.resize(rgb(img), 160, 120, name)), scale
    got = decode_to_tensor(files, (96, 96), dtype=torch.uint8, resample=resample, resize=128, scale="auto",
                           device="cuda:0")
    W = np.array([1920, 1080, 333, 61])
    H = np.array([1080, 1920, 71, 517])
    scales = auto_scales(W, H, None, (128, 128))
    assert scales.tolist() == [8, 8, 1, 1]
    for i, s in enumerate(scales):
        img = rgb(decoded(int(s))[i])
        vw, vh, wx, wy = (int(v[0]) for v in resize_geometry([img.shape[1]], [img.shape[0]], 128, (96, 96)))
        want = ref.resize(img, vw, vh, name)[wy:wy + 96, wx:wx + 96]
        assert np.array_equal(got[i].permute(1, 2, 0).cpu().numpy(), want), i
