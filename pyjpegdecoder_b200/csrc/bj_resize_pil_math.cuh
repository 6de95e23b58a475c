// bj_resize_pil_math.cuh -- Pillow's 8-bit BILINEAR / BICUBIC resample (libImaging/Resample.c), host and device.
//
// Each function restates one rule of Resample.c and names it.  The coefficients are plain IEEE double arithmetic in
// Pillow's operation order; everything after them is integer.  Two conditions make the result Pillow's, bit for bit:
//   - no FMA contraction and no fast-math: the library builds with nvcc -fmad=false, the host tests with
//     g++ -ffp-contract=off (Pillow's x86-64 build uses SSE2 doubles, which never fuse);
//   - division by the weight sum is a real IEEE division (not a multiply by the reciprocal).
//
// Skipped passes.  ImagingResample skips the horizontal (vertical) pass when the output width (height) equals the
// input's.  The pass it skips would be the identity, so the kernel runs every pass: with out == in, scale = 1,
// filterscale = 1, center = xx + 0.5, and the taps' filter arguments are the integers j - xx.  Bilinear is 1 at 0 and
// 0 at +-1; bicubic (a = -0.5) is 1 at 0, and 0 at +-1 and +-2 (((1 - 5) + 8) - 4 = 0, 2 is outside |x| < 2).  The window
// always holds tap xx (0 <= xx < in), so the weights are exactly 1 there and 0 elsewhere, the sum is 1.0, the coefficient
// is 2^22, and clip8(2^21 + v 2^22) = v for 0 <= v <= 255.
//
// int32 bound (any summation order).  A pass computes S = 2^21 + sum_j src_j k_j, 0 <= src_j <= 255.  Every partial
// sum over any subset of the taps lies in [2^21 - 255 K-, 2^21 + 255 K+], K+ (K-) the sum of the positive (|negative|)
// coefficients of the row; src = 255 exactly where k > 0 (k < 0) reaches the bound (tests/test_resize_pil_cpu.py).
// With normalised weights w_j = f_j / W, W = P - N the weight sum, P (N) the sum of the positive (|negative|) filter
// values, and k = (int)(w 2^22 +- 0.5): K+ <= 2^22 P / W + n / 2 and K- <= 2^22 N / W + n / 2, n <= ksize taps.
// Let s = filterscale >= 1 (taps at filter-argument spacing 1 / s) and r = N / P, so P / W = 1 / (1 - r).
//   Bilinear: N = 0, K+ <= 2^22 + n / 2 with n <= 2 ceil(s) + 1 <= 131071 (in <= 65535): S < 2^21 + 255 1.02 2^22.
//   Bicubic: |f| <= 2/27 on the lobes 1 < |x| < 2 (maximum at 4/3), f decreases from 1 to 0 on [0, 1].  The centre
//   c = (xx + 0.5) in / out lies at least s / 2 pixels inside both edges when downscaling, so the m = floor(s) pixel
//   centres nearest c are all in the window and the i-th of them has |x| <= i / (2 s).
//     upscale (s = 1, at most one lobe tap per side; the pixel holding c gives f(1/2) = 9/16):
//         r <= (4/27) / (9/16) < 0.27;
//     1 <= s < 2 (at most two lobe taps per side, 1/2 apart or more, the second at |x| >= 3/2 where |f| <= 1/16):
//         r <= 2 (2/27 + 1/16) / (9/16) < 0.486;
//     2 <= s < 3: P >= f(1/4) + f(1/2) = 1.4297, N <= 6 (2/27): r < 0.32;
//     s >= 3: P >= 2 m int_0^{1/2} f - f(0) = 0.8385 m - 1 (Riemann sum of a decreasing f), N <= 2 (m + 1)(2/27):
//         r <= 0.1482 (m + 1) / (0.8385 m - 1) < 0.40.
//   For s < 3, n <= 15 and P / W < 1 / (1 - 0.486) < 1.946, so K+ < 1.946 2^22 + 8; for s >= 3, P / W < 1.67 and
//   n / 2 <= (4 s + 3) / 2 < 131073 < 0.032 2^22.  Either way K+ < 1.95 2^22 and K- < 0.95 2^22, so every partial sum
//   lies in (2^21 - 255 0.95 2^22, 2^21 + 255 1.95 2^22) = (-1.01e9, 2.088e9), inside int32.  W is a double sum of at
//   most ksize terms, so its rounding changes these ratios by less than 1e-10.
// Integer sums are therefore exact and order-independent: tiles and chunks may split the taps freely.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define BJ_PIL_HD __host__ __device__ __forceinline__
#else
#define BJ_PIL_HD inline
#endif

namespace bj {

constexpr int kPilPrecisionBits = 32 - 8 - 2;   // Resample.c: PRECISION_BITS

// the filter argument (bj_resize_pil's BJ_PIL_BILINEAR / BJ_PIL_BICUBIC)
constexpr int kPilBilinear = 0;
constexpr int kPilBicubic = 1;

// Resample.c: bilinear_filter
BJ_PIL_HD double pil_bilinear(double x) {
    if (x < 0.0) x = -x;
    if (x < 1.0) return 1.0 - x;
    return 0.0;
}

// Resample.c: bicubic_filter, a = -0.5, Pillow's operation order ((a + 2.0) and (a + 3.0) are the exact constants
// 1.5 and 2.5 in both builds)
BJ_PIL_HD double pil_bicubic(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

BJ_PIL_HD double pil_filter(int filter, double x) { return filter == kPilBicubic ? pil_bicubic(x) : pil_bilinear(x); }

// Resample.c: struct filter .support
BJ_PIL_HD double pil_support(int filter) { return filter == kPilBicubic ? 2.0 : 1.0; }

// One axis of precompute_coeffs for inSize = in, box [0, in), outSize = out.
struct PilAxis {
    double scale, filterscale, support, ss;
    int in, ksize;
};

// precompute_coeffs: scale = (in1 - in0) / outSize, filterscale = max(scale, 1), support = filter support *
// filterscale, ksize = (int)ceil(support) * 2 + 1, ss = 1.0 / filterscale
BJ_PIL_HD PilAxis pil_axis(int in, int out, int filter) {
    PilAxis a;
    a.in = in;
    a.scale = (double)(float)((float)in - 0.0f) / out;   // in0 / in1 are floats in Pillow: exact for in < 2^24
    a.filterscale = a.scale < 1.0 ? 1.0 : a.scale;
    a.support = pil_support(filter) * a.filterscale;
    a.ksize = (int)ceil(a.support) * 2 + 1;
    a.ss = 1.0 / a.filterscale;
    return a;
}

// The window of output xx: taps [xmin, xmin + n), the centre and the sum of the unnormalised weights.
struct PilWindow {
    int xmin, n;
    double center, ww;
};

// precompute_coeffs, per output: center = in0 + (xx + 0.5) * scale, xmin = max((int)(center - support + 0.5), 0),
// xmax = min((int)(center + support + 0.5), inSize) - xmin
BJ_PIL_HD PilWindow pil_window(const PilAxis& a, int xx) {
    PilWindow w;
    w.center = 0.0 + (xx + 0.5) * a.scale;
    int xmin = (int)(w.center - a.support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(w.center + a.support + 0.5);
    if (xmax > a.in) xmax = a.in;
    w.xmin = xmin;
    w.n = xmax - xmin;
    w.ww = 0.0;
    return w;
}

// precompute_coeffs: w = filter((x + xmin - center + 0.5) * ss), tap x = 0 .. n - 1 of the window
BJ_PIL_HD double pil_weight(const PilAxis& a, const PilWindow& w, int filter, int x) {
    return pil_filter(filter, (x + w.xmin - w.center + 0.5) * a.ss);
}

// precompute_coeffs: ww += w over the taps, in order
BJ_PIL_HD void pil_window_sum(const PilAxis& a, PilWindow& w, int filter) {
    double ww = 0.0;
    for (int x = 0; x < w.n; x++) ww += pil_weight(a, w, filter, x);
    w.ww = ww;
}

// normalize_coeffs_8bpc: (int)(+-0.5 + k * (1 << PRECISION_BITS)), the sign of k
BJ_PIL_HD int32_t pil_fixed(double k) {
    return k < 0 ? (int32_t)(-0.5 + k * (1 << kPilPrecisionBits)) : (int32_t)(0.5 + k * (1 << kPilPrecisionBits));
}

// The int32 coefficient of tap x of the window: precompute_coeffs' k[x] /= ww (when ww != 0), then
// normalize_coeffs_8bpc
BJ_PIL_HD int32_t pil_coeff(const PilAxis& a, const PilWindow& w, int filter, int x) {
    double k = pil_weight(a, w, filter, x);
    if (w.ww != 0.0) k /= w.ww;
    return pil_fixed(k);
}

// ImagingResampleHorizontal_8bpc / ImagingResampleVertical_8bpc: ss0 = 1 << (PRECISION_BITS - 1) is the rounding
// term every pass starts from
constexpr int32_t kPilRound = 1 << (kPilPrecisionBits - 1);

// Resample.c: clip8 -- 255 when the sum >= 1 << (PRECISION_BITS + 8), 0 when it is <= 0, else the sum >> PRECISION_BITS
BJ_PIL_HD uint8_t pil_clip8(int32_t in) {
    if (in >= (1 << kPilPrecisionBits << 8)) return 255;
    if (in <= 0) return 0;
    return (uint8_t)(in >> kPilPrecisionBits);
}

}  // namespace bj
