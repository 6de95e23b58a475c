"""GPU checks of compat="libjpeg-turbo" (bj_pixels_ijg and the T.81 AC refinement): device pixels are torch.equal to
Pillow's decode (libjpeg-turbo) on every golden fixture, the reference's 4160 x 2340 example, synthetic files and a
mixed batch of random encodings; device coefficients equal the conformant oracle; crops equal the full decode sliced;
every public path gives the same bytes; decode_to_tensor resizes those pixels."""
import io

import numpy as np
import pytest

import ijg_ref
import oracle
from conftest import GOLDEN, golden_case_names
from test_crop_gpu import _boxes
from test_ijg_cpu import WRAP, _pillow, _random_files, _writer_files
from test_tensor_out_gpu import _full, _pil, _reference

pytestmark = pytest.mark.gpu

LJT = "libjpeg-turbo"


@pytest.fixture(scope="module")
def files():
    names = golden_case_names()
    golden = [(GOLDEN / "cases" / f"{n}.jpg").read_bytes() for n in names]
    extra = [(GOLDEN / "base_image.jpg").read_bytes(), _pil(1920, 1080, 1), _pil(4000, 3000, 2, subsampling=0),
             _pil(1279, 719, 5, progressive=True), _pil(61, 517, 4, mode="L"), _pil(333, 71, 3, subsampling=1),
             _pil(641, 479, 6, progressive=True, mode="L")]
    return names + [f"extra{i}" for i in range(len(extra))], golden + extra


def _want(name, data):
    return ijg_ref.decode(data) if name == WRAP else _pillow(data)


def test_pixels_equal_pillow(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    names, datas = files
    decs = decode_batch(datas, device="cuda:0", compat=LJT)
    for n, d, dec in zip(names, datas, decs):
        assert torch.equal(dec.image_tensor.cpu(), torch.from_numpy(_want(n, d).copy())), n


def test_mixed_batch_of_random_encodings():
    import torch
    from pyjpegdecoder_b200 import decode_batch
    from PIL import Image
    rng = np.random.default_rng(4)
    items = _random_files() + _writer_files()
    while len(items) < 300:
        w, h = int(rng.integers(1, 400)), int(rng.integers(1, 300))
        mode = ["L", 0, 1, 2][len(items) % 4]
        img = np.clip(rng.normal(128, 20, (h, w, 3)) + np.linspace(0, 80, w)[None, :, None], 0, 255).astype(np.uint8)
        kw = dict(quality=int(rng.integers(20, 101)), progressive=bool(len(items) % 3 == 0))
        if mode != "L":
            kw["subsampling"] = mode
        if len(items) % 5 == 0 and not kw["progressive"]:   # Pillow cannot write larger progressive files with DRI
            kw["restart_marker_blocks"] = 2
        b = io.BytesIO()
        Image.fromarray(img[..., 0] if mode == "L" else img).save(b, "JPEG", **kw)
        items.append((f"rand{len(items)}", b.getvalue()))
    decs = decode_batch([d for _, d in items], device="cuda:0", compat=LJT)
    for (n, d), dec in zip(items, decs):
        assert torch.equal(dec.image_tensor.cpu(), torch.from_numpy(_pillow(d))), n


def test_coefficients_equal_the_conformant_oracle(files):
    from pyjpegdecoder_b200 import decode_batch
    names, datas = files
    prog = [(n, d) for n, d in zip(names, datas) if n.startswith("prog")]
    decs = decode_batch([d for _, d in prog], device="cuda:0", compat=LJT)
    for (n, d), dec in zip(prog, decs):
        want = oracle.decode(d, flags=oracle.FLAG_CONFORMANT_REFINE, want=("coef",)).coef
        for got, w in zip(dec.coefficient_planes(), want):
            assert np.array_equal(got, w), n


def test_crops_equal_the_full_decode_sliced(files, monkeypatch):
    import torch
    from pyjpegdecoder_b200 import decode_batch, ijg
    _, datas = files
    full = decode_batch(datas, device="cuda:0", compat=LJT)
    rec = full[0]._batch.plan.geom.images
    W, H = rec["width"].astype(int), rec["height"].astype(int)
    calls = []
    real = ijg.launch
    monkeypatch.setattr(ijg, "launch", lambda *a, **k: calls.append(1) or real(*a, **k))
    for name, boxes in _boxes(W, H, rec["hmax"].astype(int), rec["vmax"].astype(int)).items():
        calls.clear()
        decs = decode_batch(datas, device="cuda:0", crop=boxes, compat=LJT)
        assert len(calls) == 1
        for i, d in enumerate(decs):
            x0, y0, x1, y1 = boxes[i]
            want = full[i].image_tensor[y0:min(y1, H[i]), x0:min(x1, W[i])]
            assert d.image_tensor.is_contiguous() and torch.equal(d.image_tensor, want), (name, i, boxes[i])


def test_paths_agree(tmp_path):
    import torch
    from pyjpegdecoder_b200 import JpegDecoder, decode_batch, decode_stream
    distinct = [_pil(160 + 8 * (i % 5), 120 + 4 * (i % 7), 100 + i, mode="L" if i % 9 == 0 else "RGB",
                     subsampling=i % 3, progressive=i % 4 == 1) for i in range(40)]
    files = [distinct[i % len(distinct)] for i in range(800)]
    want = [torch.from_numpy(_pillow(d)) for d in distinct]
    one = decode_batch(files, device="cuda:0", compat=LJT, chunk=2048)
    sub = decode_batch(files, device="cuda:0", compat=LJT, chunk=256, to_host=True)
    streamed = [d for part in decode_stream(files, chunk=300, device="cuda:0", compat=LJT) for d in part]
    for i, (a, b, c) in enumerate(zip(one, sub, streamed)):
        w = want[i % len(distinct)]
        assert torch.equal(a.image_tensor.cpu(), w) and torch.equal(b.image_tensor.cpu(), w), i
        assert torch.equal(c.image_tensor.cpu(), w), i
        assert np.array_equal(b.image_array, w.numpy().swapaxes(0, 1)), i
    p = tmp_path / "f.jpg"
    p.write_bytes(distinct[5])
    single = JpegDecoder(p, device="cuda:0", compat=LJT)
    assert torch.equal(single.image_tensor.cpu(), want[5])
    assert np.array_equal(single.image_array, want[5].numpy().swapaxes(0, 1))
    kept = decode_batch(files[:40], device="cuda:0", compat=LJT, chunk=16, keep_coefficients=True)
    ref = decode_batch(files[:40], device="cuda:0", compat=LJT)
    for a, b in zip(kept, ref):
        for x, y in zip(a.coefficient_planes(), b.coefficient_planes()):
            assert np.array_equal(x, y)


def test_bad_file_among_good_ones(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch
    from pyjpegdecoder_b200.parser import parse_jpeg
    good = files[1][-5:]
    sc = parse_jpeg(good[2]).scans[0]
    broken = bytearray(good[2])
    mid = (sc.data_start + sc.data_end) // 2
    broken[mid:mid + 64] = b"\xff\x00" * 32
    bad = [good[0], b"not a jpeg", good[1], good[0][: len(good[0]) // 2], bytes(broken), good[3]]
    ref = decode_batch(bad, device="cuda:0", on_error="return")
    got = decode_batch(bad, device="cuda:0", on_error="return", compat=LJT)
    for i in (1, 3, 4):
        assert isinstance(ref[i], Exception) and type(got[i]) is type(ref[i]), (i, got[i], ref[i])
    for i, k in ((0, 0), (2, 1), (5, 3)):
        assert torch.equal(got[i].image_tensor.cpu(), torch.from_numpy(_pillow(good[k]))), i


def test_decode_to_tensor(files):
    import torch
    from pyjpegdecoder_b200 import decode_batch, decode_to_tensor
    from pyjpegdecoder_b200.tensor_out import _check_roi, _fold_norm, _Resizer
    _, datas = files
    datas = datas[-7:]
    size = (96, 128)
    for roi in (None, "center", (0.1, 0.2, 0.7, 0.9)):
        got = decode_to_tensor(datas, size, roi=roi, compat=LJT, dtype=torch.float32)
        decs = decode_batch(datas, device="cuda:0", compat=LJT)
        want = torch.empty_like(got)
        a, b = _fold_norm(torch.float32, None, None)
        rs = _Resizer(want, _check_roi(roi, len(datas)), size, torch.float32, a, b, False)
        rs.resize(decs[0]._batch, [(i, i) for i in range(len(datas))], torch.cuda.current_stream())
        rs.finish()
        assert torch.equal(got, want), roi
        pil = [_full(torch.from_numpy(_pillow(d)).cuda()) for d in datas]
        ref = _reference(pil, roi, size)
        err = (got * 255 - ref).abs().max().item()
        assert err <= 0.02, (roi, err)
