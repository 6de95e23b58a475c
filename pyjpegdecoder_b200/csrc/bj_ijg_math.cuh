// bj_ijg_math.cuh -- the integer arithmetic of libjpeg-turbo's default decompressor, host and device
// (bj_pixels_ijg.cu, compat="libjpeg-turbo").
//
// jpeg_read_scanlines with JDCT_ISLOW, do_fancy_upsampling = TRUE and no merged upsampling -- what Pillow's
// Image.open(f), torchvision's CPU decode and OpenCV give -- is pure integer arithmetic, so it is restated here rule by
// rule, each citing the libjpeg-turbo function it restates:
//   dequantise   coef * q as int (jidctint.c DEQUANTIZE: JCOEF times ISLOW_MULT_TYPE, both 16-bit; no int16 wrap)
//   IDCT         jpeg_idct_islow (jidctint.c), output through range_limit (prepare_range_limit_table, jdmaster.c)
//   upsampling   jinit_upsampler's choice per component and h2v1_fancy_upsample / h1v2_fancy_upsample /
//                h2v2_fancy_upsample / h2v1_upsample / h2v2_upsample (jdsample.c), edges replicated at the
//                component's real size (jdmainct.c context rows)
//   colour       build_ycc_rgb_table / ycc_rgb_convert (jdcolor.c), SCALEBITS 16
// Everything is __host__ __device__ and integer only, so tests/hostsim/ijg_hostsim.cpp (g++) computes the same bytes.
#pragma once
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_pixel_math.cuh"

namespace bj {

// ---- jpeg_idct_islow ------------------------------------------------------------------------------------------------
// CONST_BITS 13, PASS1_BITS 2.  JLONG intermediates are 64-bit in libjpeg-turbo; a 1-D pass may use 32-bit ones when
// its 8 inputs satisfy |x| <= BJ_IJG_INT32_MAX_IN.  Bound: every intermediate of one pass (even and odd part, the
// partial sums, the final tmp1x +- tmp_y) is a linear form in the inputs whose absolute weights sum to at most 61214
// (z2 + z3 of the odd part of output 2 / 5 and tmp11 + tmp2 come closest), so |intermediate| <= 61214 * 32767 + 2^17
// (the descale rounding term) = 2005919666 < 2^31 - 1.  Larger inputs (dequantised products of coefficients and
// tables that a conforming 8-bit encoder does not write) take the 64-bit pass.
#define BJ_IJG_INT32_MAX_IN 32767

constexpr int kIjgFix0298631336 = 2446, kIjgFix0390180644 = 3196, kIjgFix0541196100 = 4433,
              kIjgFix0765366865 = 6270, kIjgFix0899976223 = 7373, kIjgFix1175875602 = 9633,
              kIjgFix1501321110 = 12299, kIjgFix1847759065 = 15137, kIjgFix1961570560 = 16069,
              kIjgFix2053119869 = 16819, kIjgFix2562915447 = 20995, kIjgFix3072711026 = 25172;

// One 1-D pass of jpeg_idct_islow on x[0..7] (stride `st`), descaled by `shift` with round half up (DESCALE), each
// result truncated to int as libjpeg-turbo's (int) casts do.
template <class T>
BJ_HD void ijg_idct_pass(const int* x, int st, int shift, int* out, int ost) {
    T z2 = (T)x[2 * st], z3 = (T)x[6 * st];
    T z1 = (z2 + z3) * kIjgFix0541196100;
    T tmp2 = z1 + z3 * -kIjgFix1847759065;
    T tmp3 = z1 + z2 * kIjgFix0765366865;
    z2 = (T)x[0];
    z3 = (T)x[4 * st];
    T tmp0 = (z2 + z3) * 8192;                       // LEFT_SHIFT(z2 + z3, CONST_BITS)
    T tmp1 = (z2 - z3) * 8192;
    const T tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = (T)x[7 * st];
    tmp1 = (T)x[5 * st];
    tmp2 = (T)x[3 * st];
    tmp3 = (T)x[1 * st];
    z1 = tmp0 + tmp3;
    z2 = tmp1 + tmp2;
    z3 = tmp0 + tmp2;
    T z4 = tmp1 + tmp3;
    const T z5 = (z3 + z4) * kIjgFix1175875602;
    tmp0 = tmp0 * kIjgFix0298631336;
    tmp1 = tmp1 * kIjgFix2053119869;
    tmp2 = tmp2 * kIjgFix3072711026;
    tmp3 = tmp3 * kIjgFix1501321110;
    z1 = z1 * -kIjgFix0899976223;
    z2 = z2 * -kIjgFix2562915447;
    z3 = z3 * -kIjgFix1961570560;
    z4 = z4 * -kIjgFix0390180644;
    z3 += z5;
    z4 += z5;
    tmp0 += z1 + z3;
    tmp1 += z2 + z4;
    tmp2 += z2 + z3;
    tmp3 += z1 + z4;
    const T half = (T)1 << (shift - 1);
    out[0] = (int)((tmp10 + tmp3 + half) >> shift);
    out[7 * ost] = (int)((tmp10 - tmp3 + half) >> shift);
    out[1 * ost] = (int)((tmp11 + tmp2 + half) >> shift);
    out[6 * ost] = (int)((tmp11 - tmp2 + half) >> shift);
    out[2 * ost] = (int)((tmp12 + tmp1 + half) >> shift);
    out[5 * ost] = (int)((tmp12 - tmp1 + half) >> shift);
    out[3 * ost] = (int)((tmp13 + tmp0 + half) >> shift);
    out[4 * ost] = (int)((tmp13 - tmp0 + half) >> shift);
}

BJ_HD bool ijg_small(const int* x, int st) {
    bool ok = true;
    for (int i = 0; i < 8; i++) ok &= x[i * st] >= -BJ_IJG_INT32_MAX_IN && x[i * st] <= BJ_IJG_INT32_MAX_IN;
    return ok;
}

// range_limit[x & 1023] of jpeg_idct_islow, x the row-pass result before +128 (prepare_range_limit_table, jdmaster.c):
// [0, 127] -> x + 128, [128, 511] -> 255, [512, 895] -> 0, [896, 1023] -> x - 896 (the negative x in [-128, -1]).
BJ_HD uint32_t ijg_range_limit(int x) {
    const int i = x & 1023;
    return i < 128 ? (uint32_t)(i + 128) : i < 512 ? 255u : i < 896 ? 0u : (uint32_t)(i - 896);
}

// d: the 64 dequantised coefficients in natural order [row][column]; ws: 64 ints of scratch.  s: the 64 samples,
// row-major.  Columns first (descale by CONST_BITS - PASS1_BITS = 11), then rows (CONST_BITS + PASS1_BITS + 3 = 18).
BJ_HD void ijg_idct_block(const int* d, int* ws, uint8_t* s) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 8; c++) {
        if (ijg_small(d + c, 8)) ijg_idct_pass<int>(d + c, 8, 11, ws + c, 8);
        else ijg_idct_pass<long long>(d + c, 8, 11, ws + c, 8);
    }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 8; r++) {
        int o[8];
        if (ijg_small(ws + 8 * r, 1)) ijg_idct_pass<int>(ws + 8 * r, 1, 18, o, 1);
        else ijg_idct_pass<long long>(ws + 8 * r, 1, 18, o, 1);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = 0; k < 8; k++) s[8 * r + k] = (uint8_t)ijg_range_limit(o[k]);
    }
}

// ---- upsampling (jdsample.c) -----------------------------------------------------------------------------------------
// Sample of one component at output pixel (x, y), for the component's ratio (rh, rv) = (hmax / h, vmax / v) in {1, 2}
// and real downsampled size dw = ceil(W h / hmax), dh = ceil(H v / vmax).  at(sx, sy) reads the component's samples;
// it is only called with 0 <= sx < dw, 0 <= sy < dh.  jinit_upsampler's choice:
//   (1, 1)                      the sample itself
//   (2, 1), dw > 2              h2v1_fancy_upsample: (3a + left + 1) >> 2, (3a + right + 2) >> 2, edge columns copied
//   (1, 2)                      h1v2_fancy_upsample: (3a + above + 1) >> 2, (3a + below + 2) >> 2
//   (2, 2), dw > 2              h2v2_fancy_upsample: column sums s = 3 cur + nearer row, then (3s + sl + 8) >> 4,
//                               (3s + sr + 7) >> 4, edge columns (4s + 8) >> 4, (4s + 7) >> 4
//   (2, 1) / (2, 2), dw <= 2    h2v1_upsample / h2v2_upsample: replication
// The rows above the first and below the last real row are those rows themselves (jdmainct.c's context pointers).
template <class At>
BJ_HD int ijg_sample(const At& at, int x, int y, int rh, int rv, int dw, int dh) {
    if (rh == 1 && rv == 1) return at(x, y);
    if (rh == 2 && dw <= 2) return at(x >> 1, rv == 2 ? y >> 1 : y);
    if (rh == 1) {
        const int i = y >> 1, a = at(x, i);
        if (y & 1) return (3 * a + at(x, i + 1 < dh ? i + 1 : dh - 1) + 2) >> 2;
        return (3 * a + at(x, i > 0 ? i - 1 : 0) + 1) >> 2;
    }
    const int j = x >> 1;
    if (rv == 1) {
        const int a = at(j, y);
        if (x & 1) return j == dw - 1 ? a : (3 * a + at(j + 1, y) + 2) >> 2;
        return j == 0 ? a : (3 * a + at(j - 1, y) + 1) >> 2;
    }
    const int i = y >> 1, n = (y & 1) ? (i + 1 < dh ? i + 1 : dh - 1) : (i > 0 ? i - 1 : 0);
    const int s = 3 * at(j, i) + at(j, n);
    if (x & 1) return j == dw - 1 ? (4 * s + 7) >> 4 : (3 * s + 3 * at(j + 1, i) + at(j + 1, n) + 7) >> 4;
    return j == 0 ? (4 * s + 8) >> 4 : (3 * s + 3 * at(j - 1, i) + at(j - 1, n) + 8) >> 4;
}

// ---- colour (jdcolor.c) ---------------------------------------------------------------------------------------------
// R = y + Cr_r_tab[cr], G = y + ((Cb_g_tab[cb] + Cr_g_tab[cr]) >> 16), B = y + Cb_b_tab[cb], then range_limit (a clamp
// to [0, 255] for these sums).  FIX(v) = (int)(v * 65536 + 0.5).
BJ_HD uint32_t ijg_clamp(int v) { return v < 0 ? 0u : v > 255 ? 255u : (uint32_t)v; }

BJ_HD void ijg_ycc_rgb(int y, int cb, int cr, uint32_t& R, uint32_t& G, uint32_t& B) {
    cb -= 128;
    cr -= 128;
    R = ijg_clamp(y + ((91881 * cr + 32768) >> 16));                 // FIX(1.40200)
    G = ijg_clamp(y + ((-22554 * cb + 32768 - 46802 * cr) >> 16));   // FIX(0.34414), FIX(0.71414)
    B = ijg_clamp(y + ((116130 * cb + 32768) >> 16));                // FIX(1.77200)
}

// ---- the MCU window of a job (include/b200jpeg.h, bj_pixels_ijg) -------------------------------------------------------
// The box's own MCUs, grown to every MCU holding a sample that ijg_sample reads for a pixel of the box.  Only fancy
// upsampling reads neighbours, and only one sample beyond the pixel's own, so the growth is at most one MCU per side and
// happens only where the box edge meets a sample whose neighbour lies in the next MCU.
BJ_HD void ijg_need(int p0, int p1, int n, int& lo, int& hi) {   // samples read for pixels [p0, p1) at ratio 2
    const int j0 = p0 >> 1, j1 = (p1 - 1) >> 1;
    lo = (!(p0 & 1) && j0 > 0) ? j0 - 1 : j0;
    hi = (((p1 - 1) & 1) && j1 < n - 1) ? j1 + 1 : j1;
}

BJ_HD void ijg_window(const bj_image& im, const bj_crop_job& jb, int& mx0, int& my0, int& mx1, int& my1) {
    const int mw = 8 * im.hmax, mh = 8 * im.vmax;
    mx0 = (int)jb.x0 / mw;
    my0 = (int)jb.y0 / mh;
    mx1 = ((int)jb.x1 + mw - 1) / mw;
    my1 = ((int)jb.y1 + mh - 1) / mh;
    for (int c = 0; c < im.ncomp; c++) {
        const int rh = im.hmax / im.hs[c], rv = im.vmax / im.vs[c];
        const int dw = (int)((im.width * (uint32_t)im.hs[c] + im.hmax - 1) / im.hmax);
        const int dh = (int)((im.height * (uint32_t)im.vs[c] + im.vmax - 1) / im.vmax);
        const bool fancy_h = rh == 2 && dw > 2;
        const bool fancy_v = rv == 2 && (rh == 1 || dw > 2);
        int lo, hi;
        if (fancy_h) {
            ijg_need((int)jb.x0, (int)jb.x1, dw, lo, hi);
            const int a = lo / (8 * im.hs[c]), b = hi / (8 * im.hs[c]) + 1;
            mx0 = a < mx0 ? a : mx0;
            mx1 = b > mx1 ? b : mx1;
        }
        if (fancy_v) {
            ijg_need((int)jb.y0, (int)jb.y1, dh, lo, hi);
            const int a = lo / (8 * im.vs[c]), b = hi / (8 * im.vs[c]) + 1;
            my0 = a < my0 ? a : my0;
            my1 = b > my1 ? b : my1;
        }
    }
}

}  // namespace bj
