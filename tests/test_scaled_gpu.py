"""GPU checks of the reduced-size decode (csrc/bj_pixels_scaled.cu through decode_batch / decode_stream /
decode_to_tensor(scale=)): the device pixels are bit-identical to the host model of the kernel on the same coefficient
buffer and close to the fp64 definition, scale 1 is today's decode, every public path gives the same bytes, and
decode_to_tensor at a scale equals torch's antialiased resize of the scaled decode."""
from collections import defaultdict

import numpy as np
import pytest

from conftest import GOLDEN, golden_case_names
from scaled_ref import image_f64, image_hostsim
from test_tensor_out_gpu import MEAN, STD, _full, _pil, _reference, _rois

pytestmark = pytest.mark.gpu

LOG2 = {2: 1, 4: 2, 8: 3}


@pytest.fixture(scope="module")
def files():
    golden = [(GOLDEN / "cases" / f"{n}.jpg").read_bytes() for n in golden_case_names()]
    return golden + [_pil(1920, 1080, 1), _pil(4000, 3000, 2, subsampling=0), _pil(1279, 719, 5, progressive=True),
                     _pil(61, 517, 4, mode="L"), _pil(333, 71, 3, subsampling=1)]


@pytest.mark.parametrize("s", [2, 4, 8])
def test_bit_identical_to_the_host_model_and_close_to_fp64(files, s):
    from pyjpegdecoder_b200 import decode_batch
    decs = decode_batch(files, device="cuda:0", scale=s, keep_coefficients=True)
    batch = decs[0]._batch
    assert all(d._batch is batch for d in decs)
    coef = batch.coef.cpu().numpy()
    rec, qt = batch.plan.geom.images, batch.plan.geom.qtabs
    n_diff = n_all = 0
    for i, d in enumerate(decs):
        got = d.image_tensor.cpu().numpy()
        assert (d.image_width, d.image_height) == (int(rec[i]["width"]), int(rec[i]["height"]))
        model = image_hostsim(rec[i], LOG2[s], coef, qt)
        assert got.shape == model.shape and np.array_equal(got, model), (i, s)
        diff = np.abs(got.astype(int) - image_f64(rec[i], LOG2[s], coef, qt))
        assert diff.max() <= 2, (i, s, diff.max())
        n_diff += int((diff > 0).sum())
        n_all += diff.size
    assert n_diff <= 0.001 * n_all, (s, n_diff, n_all)


def test_scale_one_is_todays_decode(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    a = decode_batch(files, device="cuda:0")
    b = decode_batch(files, device="cuda:0", scale=1)
    assert all(torch.equal(x.image_tensor, y.image_tensor) for x, y in zip(a, b))
    # the same layout; the up to 15 alignment bytes between images are not written by any kernel, so only the
    # images' own bytes are compared
    la, lb = a[0]._batch.layout, b[0]._batch.layout
    assert la.out_offsets == lb.out_offsets and la.out_shapes == lb.out_shapes and la.out_bytes == lb.out_bytes
    assert a[0]._batch.out.numel() == b[0]._batch.out.numel()


def test_streamed_equals_one_batch_and_host_copy_equals_device():
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_stream
    distinct = [_pil(160 + 8 * (i % 5), 120 + 4 * (i % 7), 100 + i, mode="L" if i % 9 == 0 else "RGB")
                for i in range(40)]
    files = [distinct[i % len(distinct)] for i in range(1100)]
    one = decode_batch(files, device="cuda:0", scale=4, chunk=2048)
    sub = decode_batch(files, device="cuda:0", scale=4, chunk=256, to_host=True)      # through decode_stream
    streamed = [d for part in decode_stream(files, chunk=300, device="cuda:0", scale=4) for d in part]
    for a, b, c in zip(one, sub, streamed):
        assert torch.equal(a.image_tensor, b.image_tensor) and torch.equal(a.image_tensor, c.image_tensor)
        assert np.array_equal(b.image_array, a.image_tensor.cpu().numpy().swapaxes(0, 1))
    small = decode_batch(files[:40], device="cuda:0", scale=8, to_host=True)
    for d in small:
        assert np.array_equal(d.image_array, d.image_tensor.cpu().numpy().swapaxes(0, 1))
        assert d.image_tensor.shape[:2] == (-(-d.image_height // 8), -(-d.image_width // 8))


def test_bad_files_give_the_same_errors_as_at_full_size(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.parser import parse_jpeg
    good = files[:6]
    sc = parse_jpeg(good[2]).scans[0]
    broken = bytearray(good[2])
    mid = (sc.data_start + sc.data_end) // 2
    broken[mid:mid + 64] = b"\xff\x00" * 32
    bad = [good[0], b"not a jpeg", good[1], good[0][: len(good[0]) // 2], bytes(broken), good[3]]
    full = decode_batch(bad, device="cuda:0", on_error="return")
    ok = decode_batch([good[0], good[1], good[3]], device="cuda:0", scale=4)
    for s in (2, 4):
        got = decode_batch(bad, device="cuda:0", on_error="return", scale=s)
        for i in (1, 3, 4):
            assert isinstance(full[i], Exception) and type(got[i]) is type(full[i]), (s, i, got[i], full[i])
        if s == 4:
            for i, k in ((0, 0), (2, 1), (5, 2)):
                assert torch.equal(got[i].image_tensor, ok[k].image_tensor), i


@pytest.fixture(scope="module")
def scaled_imgs(files):
    from pyjpegdecoder_b200 import decode_batch
    return {s: [_full(d.image_tensor).clone() for d in decode_batch(files, device="cuda:0", scale=s)] for s in (2, 4)}


@pytest.mark.parametrize("s", [2, 4])
@pytest.mark.parametrize("size", [(224, 224), (37, 301)])
@pytest.mark.parametrize("roi_name", ["none", "box", "per_image", "center"])
def test_decode_to_tensor_at_a_scale_matches_torch_on_the_scaled_decode(files, scaled_imgs, s, size, roi_name):
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    roi = _rois(len(files))[roi_name]
    ref = _reference(scaled_imgs[s], roi, size)
    f32 = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, device="cuda:0", scale=s)
    assert (f32 * 255 - ref).abs().max().item() <= 0.02
    u8 = decode_to_tensor(files, size, roi=roi, dtype=torch.uint8, device="cuda:0", scale=s)
    assert (u8.float() - torch.round(ref).clamp(0, 255)).abs().max().item() <= 1
    f32n = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, mean=MEAN, std=STD, device="cuda:0", scale=s)
    for dt in (torch.float16, torch.bfloat16):
        got = decode_to_tensor(files, size, roi=roi, dtype=dt, mean=MEAN, std=STD, device="cuda:0", scale=s)
        assert torch.equal(got, f32n.to(dt)), dt


def test_auto_equals_the_per_scale_calls_grouped_by_the_rule(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    from pyjpegdecoder_b200.scaled import auto_scales
    size = (32, 32)
    heads = decode_batch(files, device="cuda:0")
    W = [d.image_width for d in heads]
    H = [d.image_height for d in heads]
    for roi in (None, "center"):
        rule = auto_scales(W, H, roi, size)
        assert len(set(rule.tolist())) >= 3                         # a mix: the s = 1 images go through bj_pixels
        got = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, device="cuda:0", scale="auto")
        groups = defaultdict(list)
        for i, s in enumerate(rule.tolist()):
            groups[s].append(i)
        for s, idx in groups.items():
            want = decode_to_tensor([files[i] for i in idx], size, roi=roi, dtype=torch.float32, device="cuda:0", scale=s)
            assert torch.equal(got[idx], want), (roi, s)
        # streamed (chunk of 8: more than 1.5 chunks of files) and on_error="return" give the same values
        streamed = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, device="cuda:0", scale="auto", chunk=8)
        tolerant, errors = decode_to_tensor(files, size, roi=roi, dtype=torch.float32, device="cuda:0", scale="auto",
                                            chunk=8, on_error="return")
        assert torch.equal(streamed, got) and torch.equal(tolerant, got) and not any(errors)
    per = _rois(len(files))["per_image"]
    got = decode_to_tensor(files, size, roi=per, dtype=torch.float32, device="cuda:0", scale="auto", chunk=8)
    rule = auto_scales(W, H, np.asarray(per), size)
    for s in set(rule.tolist()):
        idx = [i for i in range(len(files)) if rule[i] == s]
        want = decode_to_tensor([files[i] for i in idx], size, roi=[per[i] for i in idx], dtype=torch.float32,
                                device="cuda:0", scale=s)
        assert torch.equal(got[idx], want), s


def test_auto_against_full_size_on_1080p():
    import torch
    from pyjpegdecoder_b200 import decode_to_tensor
    f = [_pil(1920, 1080, 1)]
    full = decode_to_tensor(f, (224, 224), dtype=torch.float32, device="cuda:0") * 255
    auto = decode_to_tensor(f, (224, 224), dtype=torch.float32, device="cuda:0", scale="auto") * 255
    d = (auto - full).abs()
    assert d.mean().item() <= 1.0 and d.max().item() <= 6, (d.mean().item(), d.max().item())


def test_scaled_output_is_a_sixteenth_at_quarter_scale():
    from pyjpegdecoder_b200 import decode_batch
    f = [_pil(1920, 1080, 1 + i) for i in range(8)]
    full = decode_batch(f, device="cuda:0")[0]._batch.out.numel()
    quarter = decode_batch(f, device="cuda:0", scale=4)[0]._batch.out.numel()
    assert quarter <= full / 16 + 16 * len(f), (quarter, full)
