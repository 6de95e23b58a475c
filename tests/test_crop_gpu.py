"""GPU checks of the crop decode (bj_pixels_crop through decode_batch / decode_stream / JpegDecoder / decode_to_tensor):
at every scale a crop is torch.equal to the same-scale full decode sliced by the box rule, every public path gives the
same bytes, decode_to_tensor(roi=) gives exactly the values of today's decode-everything-then-resize, and a cropped
batch's output buffer holds only the crops."""
import numpy as np
import pytest

from conftest import GOLDEN, golden_case_names
from test_tensor_out_gpu import MEAN, STD, _pil, _rois

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)


@pytest.fixture(scope="module")
def files():
    golden = [(GOLDEN / "cases" / f"{n}.jpg").read_bytes() for n in golden_case_names()]
    return golden + [_pil(1920, 1080, 1), _pil(4000, 3000, 2, subsampling=0), _pil(1279, 719, 5, progressive=True),
                     _pil(61, 517, 4, mode="L"), _pil(333, 71, 3, subsampling=1)]


@pytest.fixture(scope="module")
def full(files):
    from pyjpegdecoder_b200 import decode_batch
    out = {}
    for s in SCALES:
        decs = decode_batch(files, device="cuda:0", scale=s)
        out[s] = [d.image_tensor.clone() for d in decs]
    rec = decs[0]._batch.plan.geom.images
    return out, rec["width"].astype(int), rec["height"].astype(int), rec["hmax"].astype(int), rec["vmax"].astype(int)


def _boxes(W, H, hm, vm):
    """name -> one box per file."""
    kinds = {}
    kinds["whole"] = [(0, 0, w, h) for w, h in zip(W, H)]
    kinds["top_left"] = [(0, 0, 1, 1) for _ in W]
    kinds["top_right"] = [(w - 1, 0, w, 1) for w in W]
    kinds["bottom_left"] = [(0, h - 1, 1, h) for h in H]
    kinds["bottom_right"] = [(w - 1, h - 1, w, h) for w, h in zip(W, H)]
    al = []
    for w, h, a, b in zip(W, H, hm, vm):
        mw, mh = 8 * a, 8 * b
        x0, y0 = mw * ((w // mw) // 2), mh * ((h // mh) // 2)
        al.append((x0, y0, min(w, x0 + 2 * mw), min(h, y0 + mh)) if x0 < w and y0 < h else (0, 0, mw, mh))
    kinds["mcu_aligned"] = al
    kinds["odd"] = [(w // 3, h // 5, max(w // 3 + 1, min(w, 2 * w // 3 + 5)), max(h // 5 + 1, min(h, 4 * h // 5 + 3)))
                    for w, h in zip(W, H)]
    kinds["row"] = [(0, h // 2, w, h // 2 + 1) for w, h in zip(W, H)]
    kinds["column"] = [(w // 2, 0, w // 2 + 1, h) for w, h in zip(W, H)]
    kinds["padded_edge"] = [(max(0, w - 13), max(0, h - 7), w, h) for w, h in zip(W, H)]
    kinds["past_image"] = [(w // 2, h // 3, w + 100, h + 50) for w, h in zip(W, H)]
    return kinds


def _rule(box, w, h, s):
    x0, y0, x1, y1 = box
    return x0 // s, y0 // s, -(-min(x1, w) // s), -(-min(y1, h) // s)


@pytest.mark.parametrize("s", SCALES)
def test_crop_equals_the_same_scale_decode_sliced(files, full, s, monkeypatch):
    import torch
    from pyjpegdecoder_b200 import crop, decode_batch
    imgs, W, H, hm, vm = full
    calls = []
    real = crop.launch
    monkeypatch.setattr(crop, "launch", lambda *a, **k: calls.append(1) or real(*a, **k))
    for name, boxes in _boxes(W, H, hm, vm).items():
        calls.clear()
        decs = decode_batch(files, device="cuda:0", scale=s, crop=boxes)
        assert len(calls) == 1                                  # one bj_pixels_crop call for the whole batch
        for i, d in enumerate(decs):
            rx0, ry0, rx1, ry1 = _rule(boxes[i], W[i], H[i], s)
            got = d.image_tensor
            assert got.is_contiguous() and torch.equal(got, imgs[s][i][ry0:ry1, rx0:rx1]), (name, i, boxes[i])
            assert (d.image_width, d.image_height) == (W[i], H[i])


def test_mixed_scales_in_one_call(files, full):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    imgs, W, H, hm, vm = full
    sc = np.asarray([SCALES[i % 4] for i in range(len(files))])
    boxes = _boxes(W, H, hm, vm)["odd"]
    decs = decode_batch(files, device="cuda:0", crop=boxes, _scales=sc)
    for i, d in enumerate(decs):
        rx0, ry0, rx1, ry1 = _rule(boxes[i], W[i], H[i], int(sc[i]))
        assert torch.equal(d.image_tensor, imgs[int(sc[i])][i][ry0:ry1, rx0:rx1]), i


def test_paths_agree(tmp_path):
    import torch
    from pyjpegdecoder_b200 import JpegDecoder, decode_batch, decode_stream
    distinct = [_pil(160 + 8 * (i % 5), 120 + 4 * (i % 7), 100 + i, mode="L" if i % 9 == 0 else "RGB",
                     subsampling=i % 3) for i in range(40)]
    files = [distinct[i % len(distinct)] for i in range(1100)]
    rng = np.random.default_rng(3)
    boxes = []
    for _ in files:
        x0, y0 = int(rng.integers(0, 150)), int(rng.integers(0, 110))
        boxes.append((x0, y0, x0 + int(rng.integers(1, 80)), y0 + int(rng.integers(1, 60))))
    for s in (1, 4):
        one = decode_batch(files, device="cuda:0", scale=s, crop=boxes, chunk=2048)
        sub = decode_batch(files, device="cuda:0", scale=s, crop=boxes, chunk=256, to_host=True)
        streamed = [d for part in decode_stream(files, chunk=300, device="cuda:0", scale=s, crop=boxes) for d in part]
        tolerant = decode_batch(files[:300], device="cuda:0", scale=s, crop=boxes[:300], on_error="return")
        for i, (a, b, c) in enumerate(zip(one, sub, streamed)):
            assert torch.equal(a.image_tensor, b.image_tensor) and torch.equal(a.image_tensor, c.image_tensor), (s, i)
            assert np.array_equal(b.image_array, a.image_tensor.cpu().numpy().swapaxes(0, 1))
            if i < 300:
                assert torch.equal(tolerant[i].image_tensor, a.image_tensor)
        p = tmp_path / "f.jpg"
        p.write_bytes(files[7])
        single = JpegDecoder(p, device="cuda:0", scale=s, crop=boxes[7])
        assert torch.equal(single.image_tensor, one[7].image_tensor)
        assert np.array_equal(single.image_array, one[7].image_tensor.cpu().numpy().swapaxes(0, 1))


def test_bad_files_and_outside_boxes(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.parser import parse_jpeg
    good = files[-5:]
    sc = parse_jpeg(good[2]).scans[0]
    broken = bytearray(good[2])
    mid = (sc.data_start + sc.data_end) // 2
    broken[mid:mid + 64] = b"\xff\x00" * 32
    bad = [good[0], b"not a jpeg", good[1], good[0][: len(good[0]) // 2], bytes(broken), good[3]]
    box = (5, 3, 40, 30)
    full = decode_batch(bad, device="cuda:0", on_error="return")
    for s in (1, 2):
        got = decode_batch(bad, device="cuda:0", on_error="return", scale=s, crop=box)
        for i in (1, 3, 4):
            assert isinstance(full[i], Exception) and type(got[i]) is type(full[i]), (s, i, got[i], full[i])
        ok = decode_batch([good[0], good[1], good[3]], device="cuda:0", scale=s, crop=box)
        for i, k in ((0, 0), (2, 1), (5, 2)):
            assert torch.equal(got[i].image_tensor, ok[k].image_tensor), i
    # the grey 61 x 517 file: a box right of x = 61 lies outside it only
    boxes = [(0, 0, 10, 10), (70, 0, 80, 10), (0, 0, 10, 10)]
    res = decode_batch([good[0], good[3], good[1]], device="cuda:0", crop=boxes, on_error="return")
    assert isinstance(res[1], ValueError) and "outside" in str(res[1])
    assert res[0].image_tensor.shape[:2] == (10, 10) and res[2].image_tensor.shape[:2] == (10, 10)
    with pytest.raises(ValueError, match="outside"):
        decode_batch([good[0], good[3]], device="cuda:0", crop=boxes[:2])


def _reference(files, roi, size, dtype, mean, std, channels_last, scale):
    """Today's decode_to_tensor: the whole files decoded (at the chosen scales), then resized by _Resizer with the
    pixel_boxes boxes."""
    import torch
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.tensor_out import _AutoScales, _check_roi, _fold_norm, _Resizer
    roi = _check_roi(roi, len(files))
    scales = _AutoScales(roi, size) if scale == "auto" else (None if scale == 1 else scale)
    a, b = _fold_norm(dtype, mean, std)
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    out = torch.empty((len(files), 3) + tuple(size), dtype=dtype, device="cuda:0", memory_format=fmt)
    rs = _Resizer(out, roi, size, dtype, a, b, channels_last)
    decs = decode_batch(files, device="cuda:0", _scales=scales)
    rs.resize(decs[0]._batch, [(i, i) for i in range(len(files))], torch.cuda.current_stream())
    rs.finish()
    return out


@pytest.mark.parametrize("roi_name", ["center", "box", "per_image"])
@pytest.mark.parametrize("scale", [1, 2, "auto"])
def test_decode_to_tensor_is_todays_output(files, roi_name, scale):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    roi = _rois(len(files))[roi_name]
    for dtype, mean, std, cl in ((torch.uint8, None, None, False), (torch.float32, MEAN, STD, True),
                                 (torch.float32, None, None, False)):
        for size in ((224, 224), (37, 301)):
            want = _reference(files, roi, size, dtype, mean, std, cl, scale)
            got = decode_to_tensor(files, size, roi=roi, dtype=dtype, mean=mean, std=std, channels_last=cl,
                                   device="cuda:0", scale=scale)
            assert torch.equal(got, want), (dtype, size, cl)
    streamed = decode_to_tensor(files, (64, 48), roi=roi, device="cuda:0", scale=scale, chunk=16)
    tolerant, errors = decode_to_tensor(files, (64, 48), roi=roi, device="cuda:0", scale=scale, chunk=16,
                                        on_error="return")
    want = _reference(files, roi, (64, 48), torch.float32, None, None, False, scale)
    assert torch.equal(streamed, want) and torch.equal(tolerant, want) and not any(errors)


def test_output_buffer_holds_exactly_the_crops():
    from pyjpegdecoder_b200 import decode_batch
    f = [_pil(1920, 1080, 1 + i) for i in range(8)]
    box = (480, 270, 1440, 810)
    decs = decode_batch(f, device="cuda:0", crop=box)
    per = 960 * 540 * 3                                        # a multiple of 16: no alignment gap between crops
    assert decs[0]._batch.out.numel() == 8 * per
    odd = decode_batch(f, device="cuda:0", crop=(1, 1, 8, 6))
    assert odd[0]._batch.out.numel() == 7 * ((7 * 5 * 3 + 15) & ~15) + 7 * 5 * 3
