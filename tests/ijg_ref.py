"""numpy statement of libjpeg-turbo's default decompression (csrc/bj_ijg_math.cuh): ISLOW IDCT with range_limit,
jdsample.c fancy upsampling at each component's real size, jdcolor.c's YCbCr -> RGB.  TEST-ONLY reference: applied
to T.81 coefficients (oracle.decode(flags=FLAG_CONFORMANT_REFINE)) it pins the definition to Pillow's decode."""
import numpy as np

import oracle
from pyjpegdecoder_b200.layout import ZIGZAG_UV
from pyjpegdecoder_b200.parser import parse_jpeg

FIX = dict(a=2446, b=3196, c=4433, d=6270, e=7373, f=9633, g=12299, h=15137, i=16069, j=16819, k=20995, l=25172)


def idct_1d(x, shift):
    """One jpeg_idct_islow pass over the last axis (int64, as JLONG), descaled with round half up, then (int)."""
    z2, z3 = x[..., 2], x[..., 6]
    z1 = (z2 + z3) * FIX['c']
    tmp2 = z1 - z3 * FIX['h']
    tmp3 = z1 + z2 * FIX['d']
    tmp0 = (x[..., 0] + x[..., 4]) << 13
    tmp1 = (x[..., 0] - x[..., 4]) << 13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    o0, o1, o2, o3 = x[..., 7], x[..., 5], x[..., 3], x[..., 1]
    z1, z2, z3, z4 = o0 + o3, o1 + o2, o0 + o2, o1 + o3
    z5 = (z3 + z4) * FIX['f']
    o0, o1, o2, o3 = o0 * FIX['a'], o1 * FIX['j'], o2 * FIX['l'], o3 * FIX['g']
    z1, z2, z3, z4 = -z1 * FIX['e'], -z2 * FIX['k'], -z3 * FIX['i'], -z4 * FIX['b']
    z3 = z3 + z5
    z4 = z4 + z5
    o0, o1, o2, o3 = o0 + z1 + z3, o1 + z2 + z4, o2 + z2 + z3, o3 + z1 + z4
    r = lambda v: ((v + (1 << (shift - 1))) >> shift).astype(np.int32).astype(np.int64)
    return np.stack([r(t10 + o3), r(t11 + o2), r(t12 + o1), r(t13 + o0),
                     r(t13 - o0), r(t12 - o1), r(t11 - o2), r(t10 - o3)], -1)


def range_limit(x):
    i = x & 1023
    return np.where(i < 128, i + 128, np.where(i < 512, 255, np.where(i < 896, 0, i - 896))).astype(np.uint8)


def islow(d):
    """(..., 8, 8) dequantised coefficients [row][column] (int64) -> (..., 8, 8) uint8 samples."""
    ws = np.swapaxes(idct_1d(np.swapaxes(d, -1, -2), 11), -1, -2)
    return range_limit(idct_1d(ws, 18))


def dequantise(coef_zz, q_zz):
    """(..., 64) zig-zag coefficients times the table, as int (no int16 wrap) -> (..., 8, 8) natural order."""
    d = np.zeros(coef_zz.shape[:-1] + (8, 8), np.int64)
    for i, (u, v) in enumerate(ZIGZAG_UV):
        d[..., v, u] = coef_zz[..., i].astype(np.int64) * int(np.int16(q_zz[i]))
    return d


def _pad(p, axis, before, after):
    n = p.shape[axis]
    idx = np.concatenate([[0] if before else [], np.arange(n), [n - 1] if after else []]).astype(np.int64)
    return np.take(p, idx, axis=axis)


def h2v1(p):
    p = p.astype(np.int64)
    l, r = _pad(p, 1, True, False)[:, :-1], _pad(p, 1, False, True)[:, 1:]
    out = np.empty((p.shape[0], 2 * p.shape[1]), np.int64)
    out[:, 0::2] = (3 * p + l + 1) >> 2
    out[:, 1::2] = (3 * p + r + 2) >> 2
    out[:, 0], out[:, -1] = p[:, 0], p[:, -1]
    return out


def h1v2(p):
    p = p.astype(np.int64)
    up, dn = _pad(p, 0, True, False)[:-1], _pad(p, 0, False, True)[1:]
    out = np.empty((2 * p.shape[0], p.shape[1]), np.int64)
    out[0::2] = (3 * p + up + 1) >> 2
    out[1::2] = (3 * p + dn + 2) >> 2
    return out


def h2v2(p):
    p = p.astype(np.int64)
    up, dn = _pad(p, 0, True, False)[:-1], _pad(p, 0, False, True)[1:]
    out = np.empty((2 * p.shape[0], 2 * p.shape[1]), np.int64)
    for k, nb in ((0, up), (1, dn)):
        cs = 3 * p + nb
        l, r = _pad(cs, 1, True, False)[:, :-1], _pad(cs, 1, False, True)[:, 1:]
        o = np.empty((cs.shape[0], 2 * cs.shape[1]), np.int64)
        o[:, 0::2] = (3 * cs + l + 8) >> 4
        o[:, 1::2] = (3 * cs + r + 7) >> 4
        o[:, 0], o[:, -1] = (4 * cs[:, 0] + 8) >> 4, (4 * cs[:, -1] + 7) >> 4
        out[k::2] = o
    return out


def upsample(pl, rh, rv):
    """A component's real-size plane (dh, dw) upsampled by jinit_upsampler's choice for ratio (rh, rv)."""
    dw = pl.shape[1]
    if (rh, rv) == (1, 1):
        return pl.astype(np.int64)
    if (rh, rv) == (2, 1) and dw > 2:
        return h2v1(pl)
    if (rh, rv) == (1, 2):
        return h1v2(pl)
    if (rh, rv) == (2, 2) and dw > 2:
        return h2v2(pl)
    return np.repeat(np.repeat(pl.astype(np.int64), rv, 0), rh, 1)


def ycc(y, cb, cr):
    cb, cr = cb - 128, cr - 128
    R = y + ((91881 * cr + 32768) >> 16)
    G = y + ((-22554 * cb + 32768 - 46802 * cr) >> 16)
    B = y + ((116130 * cb + 32768) >> 16)
    return np.clip(np.stack([R, G, B], -1), 0, 255).astype(np.uint8)


def decode_coef(p, coef, qtables):
    """Pixels from a parsed file's per-component coefficient grids (blocks_v, blocks_h, 64)."""
    W, H, hm, vm = p.width, p.height, p.hmax, p.vmax
    planes = []
    for c, comp in enumerate(p.components):
        dw, dh = -(-W * comp.h // hm), -(-H * comp.v // vm)
        g = coef[c]
        s = islow(dequantise(g, np.asarray(qtables[comp.tq])))
        pl = s.transpose(0, 2, 1, 3).reshape(g.shape[0] * 8, g.shape[1] * 8)[:dh, :dw]
        planes.append(upsample(pl, hm // comp.h, vm // comp.v)[:H, :W])
    if len(planes) == 1:
        return planes[0].astype(np.uint8)
    return ycc(*planes)


def decode(data: bytes):
    """libjpeg-turbo's pixels of a file from the oracle's T.81 coefficients."""
    p = parse_jpeg(data)
    d = oracle.decode(data, flags=oracle.FLAG_CONFORMANT_REFINE, want=("coef",))
    return decode_coef(p, d.coef, p.qtables)
