"""GPU checks of decode_to_tensor (csrc/bj_resize.cu through pyjpegdecoder_b200/tensor_out.py): identity resizes are
bit-exact with decode_batch, every dtype / roi / size agrees with torch's antialiased bilinear interpolate on the
decoded pixels, layouts and sub-batching do not change a value, memory stays flat, bad files behave like decode_batch."""
import io
from collections import defaultdict

import numpy as np
import pytest

from conftest import GOLDEN, golden_case_names

pytestmark = pytest.mark.gpu

MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)


def _golden():
    return [(GOLDEN / "cases" / f"{n}.jpg").read_bytes() for n in golden_case_names()]


def _pil(w, h, seed, mode="RGB", **kw):
    from PIL import Image
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.stack([128 + 100 * np.sin(x / 37 + y / 91), 128 + 100 * np.cos(x / 53 - y / 29),
                    128 + 100 * np.sin((x + y) / 71)], -1) + rng.normal(0, 12, (h, w, 3))
    img = np.clip(img, 0, 255).astype(np.uint8)
    b = io.BytesIO()
    Image.fromarray(img[..., 1] if mode == "L" else img).save(b, "JPEG", quality=85, **kw)
    return b.getvalue()


def _full(t):
    """(3, H, W) uint8 of a decoded (H, W, 3) / (H, W) image tensor (grey expanded like PIL's convert("RGB"))."""
    return t.permute(2, 0, 1) if t.dim() == 3 else t[None].expand(3, -1, -1)


def test_identity_is_bit_exact_per_size_group():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    files = _golden()
    decs = decode_batch(files, device="cuda:0")
    groups = defaultdict(list)
    for f, d in zip(files, decs):
        groups[tuple(d.image_tensor.shape[:2])].append((f, d))
    assert len(groups) >= 3
    for (H, W), items in groups.items():
        got = decode_to_tensor([f for f, _ in items], size=(H, W), dtype=torch.uint8, device="cuda:0")
        want = torch.stack([_full(d.image_tensor) for _, d in items])
        assert torch.equal(got, want), (H, W)


@pytest.fixture(scope="module")
def mixed():
    from pyjpegdecoder_b200 import decode_batch
    files = _golden() + [_pil(1920, 1080, 1), _pil(4000, 3000, 2), _pil(333, 71, 3), _pil(61, 517, 4, mode="L"),
                         _pil(1279, 719, 5, progressive=True), _pil(97, 131, 6, mode="L", progressive=True),
                         _pil(4000, 3000, 7, subsampling=0)]
    imgs = [_full(d.image_tensor).clone() for d in decode_batch(files, device="cuda:0")]
    return files, imgs


def _rois(n):
    rng = np.random.default_rng(11)
    per = []
    for _ in range(n):
        x0, y0 = rng.uniform(0, 0.7, 2)
        per.append((x0, y0, x0 + rng.uniform(0.05, 0.3), y0 + rng.uniform(0.05, 0.3)))
    return {"none": None, "box": (0.1, 0.05, 0.8, 0.9), "per_image": per, "center": "center"}


def _reference(imgs, roi, size):
    import torch
    import torch.nn.functional as F
    from pyjpegdecoder_b200.tensor_out import _check_roi, pixel_boxes
    H = [t.shape[1] for t in imgs]
    W = [t.shape[2] for t in imgs]
    boxes = pixel_boxes(_check_roi(roi, len(imgs)), W, H, size)
    out = []
    for t, (x0, y0, x1, y1) in zip(imgs, boxes):
        src = t[:, y0:y1, x0:x1].float()[None]
        try:
            out.append(F.interpolate(src, size, mode="bilinear", antialias=True, align_corners=False)[0])
        except RuntimeError:
            # torch's CUDA kernel keeps all taps of an output in shared memory and refuses very large ratios
            # (4000 x 3000 -> 1 x 1): the same separable filter as two one-axis passes on the CPU
            x = F.interpolate(src.cpu(), (src.shape[2], size[1]), mode="bilinear", antialias=True, align_corners=False)
            x = F.interpolate(x, size, mode="bilinear", antialias=True, align_corners=False)
            out.append(x[0].to(t.device))
    return torch.stack(out)


@pytest.mark.parametrize("size", [(224, 224), (37, 301), (1, 1)])
@pytest.mark.parametrize("roi_name", ["none", "box", "per_image", "center"])
def test_parity_with_torch_interpolate(mixed, size, roi_name):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    files, imgs = mixed
    roi = _rois(len(files))[roi_name]
    ref = _reference(imgs, roi, size)                                  # 0..255 scale, float32
    f32 = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, device="cuda:0")
    assert f32.shape == (len(files), 3) + size
    err = (f32 * 255 - ref).abs().max().item()
    assert err <= 0.02, err
    u8 = decode_to_tensor(files, size, roi=roi, dtype=torch.uint8, device="cuda:0")
    assert (u8.float() - torch.round(ref).clamp(0, 255)).abs().max().item() <= 1
    m = torch.tensor(MEAN, device="cuda:0").view(1, 3, 1, 1)
    s = torch.tensor(STD, device="cuda:0").view(1, 3, 1, 1)
    norm = (ref / 255 - m) / s
    f32n = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, mean=MEAN, std=STD, device="cuda:0")
    # where the kernel's fp32 value differs from torch's fp32 value (summation order, at most the 0.02 checked above),
    # the rounded values may differ by that difference on top of the ulp: carried through per element, not as a bound
    # (plus a few fp32 ulps of the offset -mean/std, lost where v * a + b cancels to near 0)
    carried = (f32 * 255 - ref).abs() / 255 / s + 4 * 2.0 ** -24 * (m / s).abs()
    for dt, mant, emin in ((torch.float16, 10, -14), (torch.bfloat16, 7, -126)):
        got = decode_to_tensor(files, size, roi=roi, dtype=dt, mean=MEAN, std=STD, device="cuda:0")
        assert torch.equal(got, f32n.to(dt)), dt                       # the fp32 value rounded to nearest even
        want = norm.to(dt).float()
        _, e = torch.frexp(want)
        ulp = torch.exp2((torch.clamp(e - 1, min=emin) - mant).float())  # spacing of dt at the rounded reference
        excess = (got.float() - want).abs() - ulp - carried
        assert excess.max().item() <= 0, (dt, excess.max().item())


def test_channels_last_has_the_same_values(mixed):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    files, _ = mixed
    for dt in (torch.uint8, torch.float16, torch.float32):
        a = decode_to_tensor(files, (37, 301), roi="center", dtype=dt, device="cuda:0")
        b = decode_to_tensor(files, (37, 301), roi="center", dtype=dt, channels_last=True, device="cuda:0")
        assert b.is_contiguous(memory_format=torch.channels_last) and a.is_contiguous()
        assert torch.equal(a, b), dt


def test_streaming_equals_one_batch():
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    distinct = [_pil(160 + 8 * (i % 5), 120 + 4 * (i % 7), 100 + i, mode="L" if i % 9 == 0 else "RGB")
                for i in range(40)]
    files = [distinct[i % len(distinct)] for i in range(1100)]
    sub = decode_to_tensor(files, (64, 96), dtype=torch.float16, mean=MEAN, std=STD, chunk=256, device="cuda:0")
    one = decode_to_tensor(files, (64, 96), dtype=torch.float16, mean=MEAN, std=STD, chunk=2048, device="cuda:0")
    assert torch.equal(sub, one)


def _peak(fn):
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    res = fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, res


def test_memory_stays_flat_with_the_number_of_files():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    distinct = [_pil(640, 480, 200 + i) for i in range(16)]

    def tensor_peak(n):
        files = [distinct[i % 16] for i in range(n)]
        peak, out = _peak(lambda: decode_to_tensor(files, (224, 224), dtype=torch.float16, chunk=128, device="cuda:0"))
        return peak - out.numel() * out.element_size()

    def batch_peak(n):
        files = [distinct[i % 16] for i in range(n)]
        peak, res = _peak(lambda: decode_batch(files, chunk=128, device="cuda:0"))
        del res
        return peak

    small, large = tensor_peak(512), tensor_peak(2048)
    assert large <= 1.25 * small, (small, large)
    b_small, b_large = batch_peak(512), batch_peak(2048)
    # decode_batch keeps every image: it grows with the files (beyond the sub-batches in flight both calls have)
    assert b_large - b_small >= 4 * max(large - small, 0) and b_large >= 2 * b_small, (b_small, b_large, small, large)


def test_bad_files_return_errors_or_raise():
    import torch
    from pyjpegdecoder_b200 import CorruptedJpeg, JpegError, NotJpeg, decode_batch, decode_to_tensor
    from pyjpegdecoder_b200.parser import parse_jpeg
    names = golden_case_names()[:8]
    good = [(GOLDEN / "cases" / f"{n}.jpg").read_bytes() for n in names]
    files = list(good)
    files.insert(1, b"not a jpeg at all")
    files.insert(4, good[0][: len(good[0]) // 2])                 # header intact, entropy data and EOI missing
    sc = parse_jpeg(good[2]).scans[0]
    broken = bytearray(good[2])
    mid = (sc.data_start + sc.data_end) // 2
    broken[mid:mid + 64] = b"\xff\x00" * 32                      # stuffed 0xFF bytes: 256 one-bits, no Huffman code
    files.append(bytes(broken))                                   # (the device reports BJ_ERR_BAD_CODE)
    bad = {1: NotJpeg, 4: CorruptedJpeg, len(files) - 1: CorruptedJpeg}
    out, errors = decode_to_tensor(files, (40, 56), dtype=torch.float32, mean=MEAN, std=STD, on_error="return",
                                   chunk=4, device="cuda:0")
    assert len(errors) == len(files)
    reported = decode_batch(files, device="cuda:0", on_error="return")
    for i, e in enumerate(errors):
        if i in bad:
            assert type(e) is bad[i] and type(reported[i]) is bad[i], (i, e, reported[i])
            assert not out[i].any(), i
        else:
            assert e is None, (i, e)
    ok = [i for i in range(len(files)) if i not in bad]
    alone = decode_to_tensor([files[i] for i in ok], (40, 56), dtype=torch.float32, mean=MEAN, std=STD, device="cuda:0")
    assert torch.equal(out[ok], alone)
    with pytest.raises(JpegError):
        decode_to_tensor(files, (40, 56), device="cuda:0")
