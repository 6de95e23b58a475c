"""CPU checks of compat="libjpeg-turbo": tests/ijg_ref.py (a numpy statement of libjpeg-turbo's default decompression)
equals Pillow's decode, which pins the definition to libjpeg-turbo on any machine; csrc/bj_ijg_math.cuh (host build,
tests/hostsim/ijg_hostsim.cpp) equals ijg_ref rule by rule; the entropy header's T.81 refinement gives the conformant
oracle's coefficients; the halo window rule equals a brute-force dependency count; argument errors."""
import ctypes
import io

import numpy as np
import pytest

import ijg_ref
import oracle
from conftest import GOLDEN, golden_case_names
from hostsim import build
from jpeg_writer import image_to_components, std_qtables, write_baseline

WRAP = "wwrap_16x16_ss0"   # dequantised products beyond int16: libjpeg-turbo's SIMD and C paths disagree there


def _pillow(data):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(data)))


def _img(w, h, seed):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    img = np.stack([127 + 90 * np.sin(x / (5 + 20 * rng.random()) + y / (7 + 20 * rng.random())) for _ in range(3)], -1)
    return np.clip(img + rng.normal(0, 25, (h, w, 3)), 0, 255).astype(np.uint8)


def _random_files():
    from PIL import Image
    rng = np.random.default_rng(11)
    sizes = [(1, 1), (2, 1), (2, 5), (3, 3), (4, 9), (3, 17), (17, 2), (33, 31), (97, 61), (250, 7), (129, 130)]
    out = []
    for k, (w, h) in enumerate(sizes):
        for prog in (False, True):
            for mode in ("L", 0, 1, 2):
                kw = dict(quality=int(rng.integers(30, 101)), progressive=prog)
                if mode != "L":
                    kw["subsampling"] = mode
                if k % 3 == 1:
                    kw["restart_marker_blocks"] = int(rng.integers(1, 4))
                img = _img(w, h, 100 * k + (0 if mode == "L" else mode + 1))
                b = io.BytesIO()
                Image.fromarray(img[..., 0] if mode == "L" else img).save(b, "JPEG", **kw)
                out.append((f"{w}x{h}_{'p' if prog else 'b'}_{mode}", b.getvalue()))
    return out


def _writer_files():
    q = std_qtables(80)
    out = []
    for k, samp in enumerate([[(1, 2), (1, 1), (1, 1)], [(2, 2), (1, 2), (2, 1)], [(1, 1), (2, 2), (1, 1)],
                              [(2, 1), (1, 1), (2, 1)], [(1, 2), (1, 2), (1, 1)]]):
        for w, h in ((37, 29), (3, 11), (64, 48)):
            img = _img(w, h, 7 + k)
            out.append((f"writer_{k}_{w}x{h}", write_baseline(w, h, image_to_components(img, samp, q), q,
                                                                 restart_interval=2 if k % 2 else 0)))
    return out


@pytest.mark.parametrize("name", [n for n in golden_case_names() if n != WRAP])
def test_ref_equals_pillow_on_golden_fixtures(name):
    data = (GOLDEN / "cases" / f"{name}.jpg").read_bytes()
    assert np.array_equal(ijg_ref.decode(data), _pillow(data))


def test_ref_equals_pillow_on_base_image():
    data = (GOLDEN / "base_image.jpg").read_bytes()
    assert np.array_equal(ijg_ref.decode(data), _pillow(data))


def test_ref_equals_pillow_on_random_encodings():
    for name, data in _random_files():
        got, want = ijg_ref.decode(data), _pillow(data)
        assert got.shape == want.shape and np.array_equal(got, want), name


def test_ref_equals_pillow_on_unusual_sampling():
    for name, data in _writer_files():
        got, want = ijg_ref.decode(data), _pillow(data)
        assert got.shape == want.shape and np.array_equal(got, want), name


_HS = None


def hostsim():
    global _HS
    if _HS is None:
        _HS = build("ijg_hostsim")
        vp, ci = ctypes.c_void_p, ctypes.c_int
        _HS.hs_ijg_idct.argtypes = [ci, vp, vp]
        _HS.hs_ijg_upsample.argtypes = [vp, ci, ci, ci, ci, ci, ci, vp]
        _HS.hs_ijg_rgb.argtypes = [ci, vp, vp]
        _HS.hs_ijg_window.argtypes = [vp, vp, vp]
    return _HS


def _idct_blocks(rng):
    out = [rng.integers(-600, 601, (200, 8, 8)) * rng.integers(1, 30, (200, 1, 1))]                   # dense
    sp = np.zeros((200, 64), np.int64)
    for b in sp:
        k = rng.choice(64, int(rng.integers(1, 6)), replace=False)
        b[k] = rng.integers(-3000, 3001, len(k))
    out.append(sp.reshape(-1, 8, 8))                                                                    # sparse
    dc = np.zeros((400, 8, 8), np.int64)
    dc[:, 0, 0] = np.arange(-2000, 2000, 10) * 8                                                        # DC only
    out.append(dc)
    out.append(rng.choice([-1, 1], (100, 8, 8)) * 2047 * 16)                                            # saturated
    edge = rng.choice([-32768, -32767, 32767, 32768], (100, 8, 8))                                      # 32-bit edge
    out.append(edge)
    big = rng.integers(-2047, 2048, (100, 8, 8)) * rng.integers(1, 32768, (100, 8, 8))                  # int16 products
    out.append(big)                                                                                     # overflow: 64-bit
    out.append(rng.integers(-(2 ** 30), 2 ** 30, (100, 8, 8)))
    return np.concatenate(out)


def test_idct_equals_ref_including_range_limit_wrap():
    d = _idct_blocks(np.random.default_rng(5))
    want = ijg_ref.islow(d)
    dd = np.ascontiguousarray(d.astype(np.int32))
    got = np.empty((len(d), 8, 8), np.uint8)
    hostsim().hs_ijg_idct(len(d), dd.ctypes.data, got.ctypes.data)
    assert np.array_equal(got, want)
    # the wrap of range_limit is exercised: samples from results far outside [-128, 127]
    assert (want == 0).any() and (want == 255).any()


@pytest.mark.parametrize("rh,rv", [(1, 1), (2, 1), (1, 2), (2, 2)])
def test_upsampling_equals_ref_at_both_edges(rh, rv):
    rng = np.random.default_rng(rh * 10 + rv)
    for dw in (1, 2, 3, 4, 5, 9, 16):
        for dh in (1, 2, 3, 7):
            pl = np.ascontiguousarray(rng.integers(0, 256, (dh, dw)).astype(np.uint8))
            want = ijg_ref.upsample(pl, rh, rv)
            for w_out in {rh * dw, rh * dw - (rh - 1)}:          # an even and an odd output width
                for h_out in {rv * dh, rv * dh - (rv - 1)}:
                    got = np.empty((h_out, w_out), np.int32)
                    hostsim().hs_ijg_upsample(pl.ctypes.data, dw, dh, rh, rv, w_out, h_out, got.ctypes.data)
                    assert np.array_equal(got, want[:h_out, :w_out]), (dw, dh, w_out, h_out)


def test_colour_equals_ref_over_all_inputs():
    cb, cr = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    for y in range(256):
        ycc = np.ascontiguousarray(np.stack([np.full_like(cb, y), cb, cr], -1).astype(np.uint8).reshape(-1, 3))
        got = np.empty_like(ycc)
        hostsim().hs_ijg_rgb(len(ycc), ycc.ctypes.data, got.ctypes.data)
        want = ijg_ref.ycc(np.int64(y), cb.reshape(-1).astype(np.int64), cr.reshape(-1).astype(np.int64))
        assert np.array_equal(got, want), y


def test_t81_refinement_in_the_entropy_header_equals_the_conformant_oracle(monkeypatch):
    import entropy_sim
    # entropy_sim drives the library it builds; build the T.81 variant instead and route its AC-refinement streams
    # through hs_acrefine_stream_t81 (same arguments)
    monkeypatch.setattr(entropy_sim, "_L", None)
    monkeypatch.setattr(entropy_sim, "build", lambda name: build("entropy_t81_hostsim"))
    lib = entropy_sim.lib()
    lib.hs_acrefine_stream_t81.restype = ctypes.c_uint32
    lib.hs_acrefine_stream_t81.argtypes = lib.hs_acrefine_stream.argtypes
    monkeypatch.setattr(lib, "hs_acrefine_stream", lib.hs_acrefine_stream_t81)
    names = [n for n in golden_case_names() if n.startswith("prog")]
    assert names
    differs = 0
    for n in names:
        data = (GOLDEN / "cases" / f"{n}.jpg").read_bytes()
        p, per_scan, _ = entropy_sim.decode_file(data)
        want = oracle.decode(data, flags=oracle.FLAG_CONFORMANT_REFINE, want=("coef",)).coef
        ref = oracle.decode(data, want=("coef",)).coef
        for g, w, r in zip(per_scan[-1], want, ref):
            assert np.array_equal(g, w), n
            differs += not np.array_equal(w, r)
    assert differs                                      # the two rules do differ on these files


def _brute_window(rec, box):
    """MCU window from the samples ijg_sample reads for every pixel of the box (bounding rectangle, box MCUs included)."""
    W, H, hm, vm = int(rec["width"]), int(rec["height"]), int(rec["hmax"]), int(rec["vmax"])
    x0, y0, x1, y1 = box
    mx = {x0 // (8 * hm), (x1 - 1) // (8 * hm)}
    my = {y0 // (8 * vm), (y1 - 1) // (8 * vm)}
    for c in range(int(rec["ncomp"])):
        h, v = int(rec["hs"][c]), int(rec["vs"][c])
        rh, rv = hm // h, vm // v
        dw, dh = -(-W * h // hm), -(-H * v // vm)
        cols, rows = set(), set()

        def at(sx, sy):
            cols.add(sx // (8 * h))
            rows.add(sy // (8 * v))
            return 0
        xs = sorted({x0, x0 + 1, x1 - 2, x1 - 1} & set(range(x0, x1)))
        ys = sorted({y0, y0 + 1, y1 - 2, y1 - 1} & set(range(y0, y1)))
        for y in ys:
            for x in xs:
                _sample(at, x, y, rh, rv, dw, dh)
        mx |= cols
        my |= rows
    return min(mx), min(my), max(mx) + 1, max(my) + 1


def _sample(at, x, y, rh, rv, dw, dh):
    """The reads of bj::ijg_sample (the values do not matter here)."""
    if rh == 1 and rv == 1:
        return at(x, y)
    if rh == 2 and dw <= 2:
        return at(x >> 1, y >> 1 if rv == 2 else y)
    if rh == 1:
        i = y >> 1
        return at(x, i) + at(x, min(i + 1, dh - 1) if y & 1 else max(i - 1, 0))
    j = x >> 1
    if rv == 1:
        if (x & 1 and j == dw - 1) or (not x & 1 and j == 0):
            return at(j, y)
        return at(j, y) + at(j + 1 if x & 1 else j - 1, y)
    i = y >> 1
    n = min(i + 1, dh - 1) if y & 1 else max(i - 1, 0)
    s = at(j, i) + at(j, n)
    if (x & 1 and j == dw - 1) or (not x & 1 and j == 0):
        return s
    jj = j + 1 if x & 1 else j - 1
    return s + at(jj, i) + at(jj, n)


LAYOUTS = {"420": [(2, 2), (1, 1), (1, 1)], "422": [(2, 1), (1, 1), (1, 1)], "440": [(1, 2), (1, 1), (1, 1)],
           "444": [(1, 1)] * 3, "grey": [(1, 1)], "gen_a": [(2, 2), (1, 2), (2, 1)], "gen_b": [(1, 1), (2, 2), (1, 1)],
           "gen_c": [(2, 1), (1, 1), (2, 1)], "gen_d": [(1, 2), (1, 2), (1, 1)]}


def _rec(w, h, samp):
    from pyjpegdecoder_b200 import _native
    r = np.zeros(1, dtype=_native.IMAGE_DTYPE)[0]
    r["width"], r["height"], r["ncomp"] = w, h, len(samp)
    r["hmax"], r["vmax"] = max(s[0] for s in samp), max(s[1] for s in samp)
    for c, (a, b) in enumerate(samp):
        r["hs"][c], r["vs"][c] = a, b
    r["mcus_x"], r["mcus_y"] = -(-w // (8 * int(r["hmax"]))), -(-h // (8 * int(r["vmax"])))
    return r


def test_window_rule_equals_brute_force_dependencies():
    from pyjpegdecoder_b200 import ijg
    from pyjpegdecoder_b200.crop import CROP_JOB_DTYPE
    rng = np.random.default_rng(2)
    L = hostsim()
    for name, samp in LAYOUTS.items():
        for w, h in ((1, 1), (3, 2), (4, 5), (5, 3), (40, 37), (77, 50)):
            rec = _rec(w, h, samp)
            boxes = [(0, 0, w, h), (0, 0, 1, 1), (w - 1, h - 1, w, h)]
            for _ in range(30):
                x0, y0 = int(rng.integers(0, w)), int(rng.integers(0, h))
                boxes.append((x0, y0, int(rng.integers(x0 + 1, w + 1)), int(rng.integers(y0 + 1, h + 1))))
            recs = np.stack([rec] * len(boxes))
            py = ijg.windows(recs, np.asarray(boxes))
            for b, pw in zip(boxes, py):
                want = _brute_window(rec, b)
                assert tuple(int(v) for v in pw[[0, 1, 2, 3]]) == (want[0], want[1], want[2], want[3]), (name, w, h, b)
                job = np.zeros(1, CROP_JOB_DTYPE)
                job["x0"], job["y0"], job["x1"], job["y1"] = b
                r1 = np.ascontiguousarray(np.asarray([rec]))
                got = np.zeros(4, np.int32)
                L.hs_ijg_window(r1.ctypes.data, job.ctypes.data, got.ctypes.data)
                assert tuple(got) == tuple(int(v) for v in pw), (name, w, h, b)


def test_argument_errors():
    from pyjpegdecoder_b200 import JpegDecoder, decode_batch, decode_stream, decode_to_tensor
    data = (GOLDEN / "cases" / f"{golden_case_names()[0]}.jpg").read_bytes()
    with pytest.raises(ValueError, match="compat"):
        decode_batch([data], compat="pillow")
    with pytest.raises(ValueError, match="compat"):
        decode_batch([data], compat=None)
    with pytest.raises(ValueError, match="full size"):
        decode_batch([data], compat="libjpeg-turbo", scale=2)
    with pytest.raises(ValueError, match="full size"):
        next(iter(decode_stream([data], compat="libjpeg-turbo", scale=4)))
    with pytest.raises(ValueError, match="full size"):
        JpegDecoder(data, compat="libjpeg-turbo", scale=8)
    with pytest.raises(ValueError, match="compat"):
        JpegDecoder(data, compat="LIBJPEG")
    for scale in (2, "auto"):
        with pytest.raises(ValueError, match="full size"):
            decode_to_tensor([data], (8, 8), compat="libjpeg-turbo", scale=scale)
    with pytest.raises(ValueError, match="compat"):
        decode_to_tensor([data], (8, 8), compat="opencv")


def test_workspace_layout_and_jobs():
    from pyjpegdecoder_b200 import ijg
    recs = np.stack([_rec(1920, 1080, LAYOUTS["420"]), _rec(61, 17, LAYOUTS["grey"]), _rec(37, 29, LAYOUTS["gen_a"])])
    jobs, lay, strips, ws = ijg.jobs_for(recs)
    assert lay is None and strips == 68
    offs = jobs["reserved"].astype(np.int64) * 256
    assert offs[0] == 0 and offs[1] == -(-(1920 * 1088 + 2 * 960 * 544) // 256) * 256
    assert offs[2] - offs[1] == 64 * 24                       # grey 61 x 17: 8 x 3 blocks
    assert ws == offs[2] + 48 * 32 + 24 * 32 + 48 * 16        # 37 x 29 in 3 x 2 MCUs of 16 x 16: Y 2x2, Cb 1x2, Cr 2x1
    assert list(jobs["x1"]) == [1920, 61, 37] and list(jobs["y1"]) == [1080, 17, 29]
