"""CPU checks of the reduced-size decode (csrc/bj_scaled_math.cuh through tests/hostsim/scaled_hostsim.cpp, and
pyjpegdecoder_b200/scaled.py): the fp32 samples against an fp64 evaluation of the definition with the header's error
bound, the host model of the kernel on whole images, the output layout and the "auto" rule, argument errors (raised
before any device work) and the bj_scaled_job mirror."""
import numpy as np
import pytest
import torch

from scaled_ref import ZZ_NATURAL, bound, hostsim, image_f64, image_hostsim, tile_f64

SIDES = [(nx, ny) for nx in (1, 2, 4, 8) for ny in (1, 2, 4, 8)]


def _blocks(rng):
    """(kind, coef zig-zag, q zig-zag) test blocks."""
    out = []
    for _ in range(40):                                              # dense, typical magnitudes
        out.append(("dense", rng.integers(-60, 61, 64), rng.integers(1, 40, 64)))
    for _ in range(40):                                              # sparse: a few non-zero coefficients
        c = np.zeros(64, np.int64)
        k = rng.choice(64, int(rng.integers(1, 6)), replace=False)
        c[k] = rng.integers(-200, 201, len(k))
        out.append(("sparse", c, rng.integers(1, 100, 64)))
    for dc in range(-1024, 1024, 53):                                # DC only
        c = np.zeros(64, np.int64)
        c[0] = dc
        out.append(("dc", c, np.full(64, int(rng.integers(1, 9)))))
    for _ in range(20):                                              # saturated: products at the int16 limits
        c = rng.choice([-1, 1], 64) * 2047
        out.append(("saturated", c, np.full(64, 16)))                # +-32752
    for _ in range(20):                                              # the int16 product wraps
        out.append(("wrap", rng.integers(-2047, 2048, 64), rng.integers(100, 256, 64)))
    return out


def _hs_block(nx, ny, coef, q):
    lnx, lny = nx.bit_length() - 1, ny.bit_length() - 1
    c = np.ascontiguousarray(coef, np.int16)
    qq = np.ascontiguousarray(q, np.int16)
    f = np.empty(ny * nx, np.float32)
    s = np.empty(ny * nx, np.float32)
    hostsim().hs_scaled_block(lnx, lny, c.ctypes.data, qq.ctypes.data, f.ctypes.data, s.ctypes.data)
    return f.reshape(ny, nx), s.reshape(ny, nx)


def test_prefix_lengths():
    nat = ZZ_NATURAL
    for nx, ny in SIDES:
        want = 1 + max(k for k in range(64) if nat[k] % 8 < nx and nat[k] // 8 < ny)
        assert hostsim().hs_scaled_prefix(nx, ny) == want, (nx, ny)
    assert [hostsim().hs_scaled_prefix(n, n) for n in (1, 2, 4, 8)] == [1, 5, 25, 64]


@pytest.mark.parametrize("nx, ny", SIDES)
def test_samples_match_fp64_definition_within_the_stated_bound(nx, ny):
    rng = np.random.default_rng(100 + 8 * nx + ny)
    kinds = set()
    for kind, coef, q in _blocks(rng):
        f32, s32 = _hs_block(nx, ny, coef, q)
        f64, sum_abs = tile_f64(coef, q, nx, ny)
        b = bound(sum_abs)
        err = np.abs(f32.astype(np.float64) - f64)
        assert err.max() <= b, (kind, nx, ny, err.max(), b)
        want = np.round(f64) + 128
        near_tie = np.abs(np.abs(f64 - np.floor(f64)) - 0.5) <= b
        assert np.all((s32 == want) | near_tie), (kind, nx, ny)
        kinds.add(kind)
        if kind == "wrap":
            prod = coef.astype(np.int64) * q
            assert (np.abs(prod) > 32767).any()
    assert kinds == {"dense", "sparse", "dc", "saturated", "wrap"}


def test_block_mean_is_kept():
    """DC only: every sample of every tile size is DC * q / 8 (rounded) + 128, like the 8 x 8 IDCT's."""
    for nx, ny in SIDES:
        for dc in (-1000, -37, 0, 5, 12, 999):
            c = np.zeros(64, np.int64)
            c[0] = dc
            _, s = _hs_block(nx, ny, c, np.full(64, 2))
            assert np.all(s == np.round(dc * 2 / 8) + 128), (nx, ny, dc)


def _record(w, h, hs, vs, rng):
    """A bj_image record (and coefficient buffer, table) for a w x h image with per-component sampling hs / vs."""
    from pyjpegdecoder_b200._native import IMAGE_DTYPE
    nc = len(hs)
    hmax, vmax = max(hs), max(vs)
    rec = np.zeros(1, IMAGE_DTYPE)[0]
    mx, my = -(-w // (8 * hmax)), -(-h // (8 * vmax))
    bpm = sum(a * b for a, b in zip(hs, vs))
    rec["width"], rec["height"], rec["mcus_x"], rec["mcus_y"] = w, h, mx, my
    rec["ncomp"], rec["hmax"], rec["vmax"], rec["blocks_per_mcu"] = nc, hmax, vmax, bpm
    s0 = 0
    for c in range(nc):
        rec["hs"][c], rec["vs"][c], rec["slot0"][c], rec["qtab"][c] = hs[c], vs[c], s0, min(c, 1)
        s0 += hs[c] * vs[c]
    rec["coef_block0"] = 3                                      # the model must honour the image's first block
    coef = rng.integers(-30, 31, (3 + mx * my * bpm, 64)).astype(np.int16)
    coef[:, 0] = rng.integers(-60, 61, len(coef))
    qt = rng.integers(1, 12, (2, 64)).astype(np.int16)
    return rec, coef, qt


@pytest.mark.parametrize("hs, vs", [((1,), (1,)), ((1, 1, 1), (1, 1, 1)), ((2, 1, 1), (1, 1, 1)),
                                    ((1, 1, 1), (2, 1, 1)), ((2, 1, 1), (2, 1, 1)), ((2, 2, 1), (2, 1, 1))])
def test_host_model_of_whole_images_matches_fp64(hs, vs):
    """The host model places every tile and converts colour as the definition says: equal to the fp64 evaluation
    except for a few values next to a rounding tie (fp32 colour), and never by more than one level."""
    rng = np.random.default_rng(sum(hs) * 10 + sum(vs))
    for w, h in ((61, 45), (33, 17), (8, 8)):
        rec, coef, qt = _record(w, h, hs, vs, rng)
        for l in (1, 2, 3):
            got = image_hostsim(rec, l, coef, qt)
            want = image_f64(rec, l, coef, qt)
            s = 1 << l
            assert got.shape == want.shape == ((-(-h // s), -(-w // s), 3) if len(hs) == 3 else (-(-h // s), -(-w // s)))
            d = np.abs(got.astype(int) - want)
            assert d.max() <= 1 and (d > 0).mean() <= 0.01, (hs, vs, w, h, l, d.max(), (d > 0).mean())


def _images(sizes, ncomp=3):
    from pyjpegdecoder_b200._native import IMAGE_DTYPE
    rec = np.zeros(len(sizes), IMAGE_DTYPE)
    rec["width"] = [w for w, _ in sizes]
    rec["height"] = [h for _, h in sizes]
    rec["ncomp"] = ncomp
    return rec


def test_output_layout_shapes_and_alignment():
    from pyjpegdecoder_b200.scaled import OutputLayout
    sizes = [(1920, 1080), (61, 517), (333, 71), (1, 1), (7, 9), (4000, 3000)]
    rec = _images(sizes)
    rec["ncomp"][1] = 1
    for scales in ([2] * 6, [4] * 6, [8] * 6, [1, 2, 4, 8, 2, 1]):
        lay = OutputLayout.scaled(rec, np.asarray(scales))
        for i, ((w, h), s) in enumerate(zip(sizes, scales)):
            ch = 1 if i == 1 else 3
            W, H = -(-w // s), -(-h // s)
            assert lay.out_shapes[i] == ((H, W) if ch == 1 else (H, W, 3))
            assert lay.pitches[i] == W * ch and lay.offsets[i] % 16 == 0
            if i:
                prev = lay.offsets[i - 1] + lay.heights[i - 1] * lay.pitches[i - 1]
                assert prev <= lay.offsets[i] < prev + 16
        assert lay.out_bytes == lay.offsets[-1] + lay.heights[-1] * lay.pitches[-1]
    full = OutputLayout.scaled(_images([(1920, 1080)] * 4), np.full(4, 1))
    quarter = OutputLayout.scaled(_images([(1920, 1080)] * 4), np.full(4, 4))
    assert quarter.out_bytes <= full.out_bytes / 16 + 16 * 4


def test_full_layout_equals_the_planners_records():
    from pyjpegdecoder_b200.parser import parse_jpeg
    from pyjpegdecoder_b200.plan import BatchGeometry
    from pyjpegdecoder_b200.scaled import OutputLayout
    from conftest import GOLDEN, golden_case_names
    parsed = [parse_jpeg((GOLDEN / "cases" / f"{n}.jpg").read_bytes()) for n in golden_case_names()[:12]]
    g = BatchGeometry(parsed)
    a, b = OutputLayout.from_geometry(g), OutputLayout.scaled(g.images, np.ones(len(parsed), np.int64))
    assert a.out_offsets == b.out_offsets == g.out_offsets and a.out_shapes == b.out_shapes == g.out_shapes
    assert a.out_bytes == b.out_bytes == g.out_bytes and np.array_equal(a.pitches, g.images["out_pitch"])


ROIS = {"none": None, "box": np.array([0.1, 0.05, 0.8, 0.9]), "center": "center"}


@pytest.mark.parametrize("roi_name", ["none", "box", "center", "per_image"])
def test_auto_rule_landscape_portrait_square(roi_name):
    from pyjpegdecoder_b200.scaled import auto_scales
    from pyjpegdecoder_b200.tensor_out import _check_roi, pixel_boxes
    W, H = np.array([1920, 1080, 1000]), np.array([1080, 1920, 1000])
    roi = ROIS.get(roi_name)
    if roi_name == "per_image":
        roi = _check_roi([(0, 0, 1, 1), (0.5, 0.5, 1, 1), (0.2, 0.1, 0.7, 0.35)], 3)
    size = (224, 224)
    got = auto_scales(W, H, roi, size)
    for i in range(3):
        ok = [s for s in (1, 2, 4, 8)
              if (lambda b: b[2] - b[0] >= 224 and b[3] - b[1] >= 224)(
                  pixel_boxes(roi if not (isinstance(roi, np.ndarray) and roi.ndim == 2) else roi[i:i + 1],
                              [-(-W[i] // s)], [-(-H[i] // s)], size)[0])]
        assert got[i] == max(ok + [1]), (roi_name, i, got[i], ok)
    if roi_name == "none":
        assert got.tolist() == [4, 4, 4]                       # 480 x 270 is still >= 224 x 224, 240 x 135 is not
    if roi_name == "center":
        assert got.tolist() == [4, 4, 4]


def test_auto_returns_one_when_any_reduction_would_upscale():
    from pyjpegdecoder_b200.scaled import auto_scales
    assert auto_scales([300, 448, 447, 446], [300, 448, 447, 446], None, (224, 224)).tolist() == [1, 2, 2, 1]
    assert auto_scales([1920], [1080], None, (1080, 1920)).tolist() == [1]
    assert auto_scales([1920], [1080], None, (135, 240)).tolist() == [8]


def test_scaled_job_mirror_matches_the_library():
    from pyjpegdecoder_b200.scaled import SCALED_JOB_DTYPE, _bind
    L = _bind()
    assert L.bj_sizeof(2) == SCALED_JOB_DTYPE.itemsize == 24
    assert L.bj_sizeof(0) == 72 and L.bj_sizeof(1) == 40


@pytest.mark.parametrize("scale", [0, 3, 16, -2, 2.0, "2", "auto", None, True])
def test_bad_scales_are_rejected_before_device_work(scale, monkeypatch):
    from pyjpegdecoder_b200 import decode_batch, decode_stream, decode_to_tensor, loader, stages   # noqa: F401

    def no_device(*a, **k):
        raise AssertionError("device work started before the arguments were checked")
    monkeypatch.setattr(stages, "require_cuda", no_device)
    monkeypatch.setattr(loader, "require_cuda", no_device)
    with pytest.raises(ValueError):
        decode_batch([b"x", b"y"], scale=scale)
    with pytest.raises(ValueError):
        next(iter(decode_stream([b"x", b"y"], scale=scale)))
    if scale != "auto":
        with pytest.raises(ValueError):
            decode_to_tensor([b"x", b"y"], size=(8, 8), scale=scale)
    with pytest.raises(ValueError):
        decode_to_tensor([b"x", b"y"], size=(8, 8), scale="Auto")


def test_scaled_decode_needs_a_gpu_and_never_falls_back():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from pyjpegdecoder_b200 import NativeLibraryError, decode_batch, decode_to_tensor
    with pytest.raises(NativeLibraryError):
        decode_batch([b"\xff\xd8"], scale=4)
    with pytest.raises(NativeLibraryError):
        decode_to_tensor([b"\xff\xd8"], size=(8, 8), scale="auto")
