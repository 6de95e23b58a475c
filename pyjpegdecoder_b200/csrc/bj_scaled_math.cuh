// bj_scaled_math.cuh -- per-block arithmetic of the reduced-size decode (bj_pixels_scaled.cu), host and device.
//
// Decoding at scale 1/s (s = 2, 4, 8) in the DCT domain.  Component c of an image with maximum sampling factors
// (hmax, vmax) gives, from each of its blocks, an NY x NX tile with NX = 8 * (hmax / h_c) / s and
// NY = 8 * (vmax / v_c) / s, both in {1, 2, 4, 8}: every component then comes out at the scaled image's own
// resolution and no chroma upsampling is needed.  The sample at (x, y) of a tile is
//     f(x, y) = 1/4 * sum_{u < NX, v < NY} C(u) C(v) F(u, v) cos((2x+1) u pi / 2NX) cos((2y+1) v pi / 2NY),
//     C(0) = 1/sqrt 2, C(k > 0) = 1,       sample = round_half_even(f) + 128 (no clamp),
// with F the dequantised coefficients (int16 product, wrapping like bj_pixels and jpeg_decoder.py:869): the JPEG
// IDCT restricted to the low-frequency NX x NY corner, with the cosine argument of an N-point transform.  It keeps
// the block mean; for N = 8 it is the ordinary IDCT.  Colour is the full path's fp32 rule: ycc_to_rgb_fast, clip to
// [0, 255], round half to even; greyscale samples are clamped to [0, 255].
//
// Every function is __host__ __device__ and uses explicit fmaf only (the library builds with -fmad=false), so
// tests/hostsim/scaled_hostsim.cpp, built with g++ -ffp-contract=off, computes bit-identical samples.
#pragma once
#include <stdint.h>

#include "bj_pixel_math.cuh"

namespace bj {

// ---- how f is computed ------------------------------------------------------------------------------------------
// Each 1-D pass runs on basis values scaled by 2 sqrt 2: k_0 = 1 and k_u = sqrt 2 cos(u pi / 16) (so the pi/4 terms are
// +-1 as well), and f is the two-pass result times 1/8, which is exact.  Blocks whose non-zero corner coefficients all
// sit at frequencies 0 or pi/4 of each axis (DC-only blocks above all) therefore give f = (integer sum) / 8 exactly:
// the exact rounding ties of such blocks (DC = 4 mod 8) are rounded half to even as the definition says, where the
// unscaled constants (C4 = 1/(2 sqrt 2) in fp32) would push every one of them the same way.
//
// ---- fp32 error bound of f (before rounding) -------------------------------------------------------------------
//     |f_fp32 - f_exact| <= BJ_SCALED_ERR_C * 2^-24 * (sum_{u<NX, v<NY} |F(u, v)| + BJ_SCALED_ERR_K)
// First-order rounding analysis, u = 2^-24, the way bj_pixel_math.cuh bounds idct8x8_packed.  One 1-D pass computes
// out_n = sum_k c_nk X_k with |c_nk| <= cmax = sqrt 2 cos(pi/16) = 1.387.  Along the path from input k to an output,
// every operation rounds once (at most u times a magnitude <= sum_k |c_nk X_k|) and every fp32 constant other than 1
// carries a relative error <= u; the largest number R of such events on any path is
//     N = 1: none                                                                R = 0
//     N = 2: final add                                                           R = 1
//     N = 4: x1: constant, product, fma, final add                              R = 4
//     N = 8: x1: constant, product, 3 fmas, final add                           R = 6
// so one pass adds at most u R cmax sum |X| and passes on incoming errors with gain <= cmax per input.  Two passes
// (columns, then rows): the first gives |g_v| <= cmax sum_u |F(u, v)| with error <= u R1 cmax sum_u |F(u, v)|; the
// second adds u R2 cmax sum_v |g_v| and carries cmax sum_v err(g_v), in all u (R1 + R2) cmax^2 sum |F|, and the exact
// factor 1/8 gives  |err f| <= u * 12 * 1.924 / 8 * sum |F| = 2.89 u sum |F|.
// C = 3.25 leaves room for the second-order terms (R^2 u^2, below 1e-12 relative); K = 1 covers an all-zero corner.
// tests/test_scaled_cpu.py checks the bound against an fp64 evaluation of the definition.
#define BJ_SCALED_ERR_C 3.25f
#define BJ_SCALED_ERR_K 1.0f

// sqrt 2 cos(k pi / 16)
#define BJ_K1 1.3870398453221475f
#define BJ_K2 1.3065629648763766f
#define BJ_K3 1.1758756024193588f
#define BJ_K5 0.7856949583871023f
#define BJ_K6 0.5411961001461971f
#define BJ_K7 0.2758993792829431f

// Zig-zag prefix a block needs for its NX x NY corner: 1 + the largest zig-zag index of a natural position
// (u < NX, v < NY).  (1, 1) -> 1, (2, 2) -> 5, (4, 4) -> 25, (8, 8) -> 64.
constexpr BJ_HD int scaled_prefix(int nx, int ny) {
    constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
    int p = 0;
    for (int k = 0; k < 64; k++)
        if ((zz[k] & 7) < nx && (zz[k] >> 3) < ny) p = k + 1;
    return p;
}

// Dequantisation, as bj_pixels: int16 * int16 -> int16 wraps.
BJ_HD float scaled_dequant(int coef, int q) { return (float)(int16_t)(coef * q); }

// N-point inverse DCT scaled by 2 sqrt 2, in place over x[0], x[S], ..., x[(N-1) S]:
// out[n] = X[0] + sum_{k>0} sqrt 2 cos((2n+1) k pi / 2N) X[k].  The 8-point form is idct8's butterfly with these
// constants.
template <int N, int S>
BJ_HD void idct_n(float* x) {
    if constexpr (N == 1) {
        (void)x;
    } else if constexpr (N == 2) {
        const float a = x[0] + x[S], b = x[0] - x[S];
        x[0] = a; x[S] = b;
    } else if constexpr (N == 4) {
        const float e0 = x[0] + x[2 * S], e1 = x[0] - x[2 * S];
        const float o0 = fmaf(BJ_K6, x[3 * S], BJ_K2 * x[S]);
        const float o1 = fmaf(-BJ_K2, x[3 * S], BJ_K6 * x[S]);
        x[0] = e0 + o0; x[3 * S] = e0 - o0;
        x[S] = e1 + o1; x[2 * S] = e1 - o1;
    } else {
        const float s04 = x[0] + x[4 * S], d04 = x[0] - x[4 * S];
        const float f0 = fmaf(BJ_K6, x[6 * S], BJ_K2 * x[2 * S]);
        const float f1 = fmaf(-BJ_K2, x[6 * S], BJ_K6 * x[2 * S]);
        const float a0 = s04 + f0, a3 = s04 - f0, a1 = d04 + f1, a2 = d04 - f1;
        const float x1 = x[S], x3 = x[3 * S], x5 = x[5 * S], x7 = x[7 * S];
        const float o0 = fmaf(BJ_K7, x7, fmaf(BJ_K5, x5, fmaf(BJ_K3, x3, BJ_K1 * x1)));
        const float o1 = fmaf(-BJ_K5, x7, fmaf(-BJ_K1, x5, fmaf(-BJ_K7, x3, BJ_K3 * x1)));
        const float o2 = fmaf(BJ_K3, x7, fmaf(BJ_K7, x5, fmaf(-BJ_K1, x3, BJ_K5 * x1)));
        const float o3 = fmaf(-BJ_K1, x7, fmaf(BJ_K3, x5, fmaf(-BJ_K5, x3, BJ_K7 * x1)));
        x[0] = a0 + o0; x[7 * S] = a0 - o0;
        x[S] = a1 + o1; x[6 * S] = a1 - o1;
        x[2 * S] = a2 + o2; x[5 * S] = a2 - o2;
        x[3 * S] = a3 + o3; x[4 * S] = a3 - o3;
    }
}

// Sample from f: round half to even (|f| < 2^22, which holds for any int16 coefficients) + 128, exact in fp32.
BJ_HD float scaled_sample(float f) { return ((f + BJ_MAGIC) - BJ_MAGIC) + 128.0f; }

// One block's NY x NX tile.  coef(k): quantised coefficient at zig-zag index k (only k < scaled_prefix(NX, NY) are
// read); q: the component's table in zig-zag order.  out[y * stride + x] = sample, or f itself with raw = true.
template <int NX, int NY, class Coef>
BJ_HD void scaled_tile_t(const Coef& coef, const int16_t* q, float* out, int stride, bool raw) {
    constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
    constexpr int P = scaled_prefix(NX, NY);
    float X[NY * NX];
#pragma unroll
    for (int k = 0; k < P; k++) {
        const int u = zz[k] & 7, v = zz[k] >> 3;
        if (u < NX && v < NY) X[v * NX + u] = scaled_dequant(coef(k), q[k]);
    }
#pragma unroll
    for (int u = 0; u < NX; u++) idct_n<NY, NX>(&X[u]);       // columns (vertical frequency v)
#pragma unroll
    for (int y = 0; y < NY; y++) idct_n<NX, 1>(&X[y * NX]);   // rows
#pragma unroll
    for (int y = 0; y < NY; y++)
#pragma unroll
        for (int x = 0; x < NX; x++) {
            const float f = X[y * NX + x] * 0.125f;
            out[y * stride + x] = raw ? f : scaled_sample(f);
        }
}

// scaled_tile_t for run-time log2 NX, log2 NY in [0, 3].
template <class Coef>
BJ_HD void scaled_tile(int lnx, int lny, const Coef& coef, const int16_t* q, float* out, int stride, bool raw = false) {
#define BJ_ST(A, B) case A * 4 + B: scaled_tile_t<1 << A, 1 << B>(coef, q, out, stride, raw); break;
    switch (lnx * 4 + lny) {
        BJ_ST(0, 0) BJ_ST(0, 1) BJ_ST(0, 2) BJ_ST(0, 3)
        BJ_ST(1, 0) BJ_ST(1, 1) BJ_ST(1, 2) BJ_ST(1, 3)
        BJ_ST(2, 0) BJ_ST(2, 1) BJ_ST(2, 2) BJ_ST(2, 3)
        BJ_ST(3, 0) BJ_ST(3, 1) BJ_ST(3, 2) BJ_ST(3, 3)
        default: break;
    }
#undef BJ_ST
}

// log2 of a component's tile side: 3 + log2(max / sampling) - log2 s (the ratio is 1 or 2).
BJ_HD int scaled_log2_side(int max_sampling, int sampling, int log2_scale) {
    return 3 + (max_sampling > sampling ? 1 : 0) - log2_scale;
}

// Clip to [0, 255], then round half to even (jpeg_decoder.py:1698-1700).
BJ_HD uint32_t scaled_u8(float v) { return (uint32_t)((fminf(fmaxf(v, 0.0f), 255.0f) + BJ_MAGIC) - BJ_MAGIC); }

// RGB bytes of one pixel from its Y, Cb, Cr samples.
BJ_HD void scaled_rgb(float Y, float Cb, float Cr, uint32_t& R, uint32_t& G, uint32_t& B) {
    float r, g, b, err;
    ycc_to_rgb_fast(Y, Cb, Cr, r, g, b, err);
    R = scaled_u8(r); G = scaled_u8(g); B = scaled_u8(b);
}

}  // namespace bj
