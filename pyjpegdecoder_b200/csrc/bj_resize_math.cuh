// bj_resize_math.cuh -- filter weights of the antialiased bilinear resize (bj_resize.cu), host and device.
//
// The same arithmetic as torch.nn.functional.interpolate(mode="bilinear", align_corners=False, antialias=True)
// (upsample_antialias::_compute_weights_span / _compute_weights), per axis, in fp32:
//   scale = n / m, support = max(scale, 1), inv = 1 / scale if scale >= 1 else 1
//   output i: c = scale * (i + 0.5), lo = max(int(c - support + 0.5), 0), hi = min(int(c + support + 0.5), n)
//   tap j in [lo, hi): w = max(0, 1 - |(j - c + 0.5) * inv|), normalised to sum 1.
// The kernel computes the weights while it accumulates (no per-image weight tables): tap k = j - lo of an
// output weighs bj_rs_weight(win.base + k * inv); the normalisation 1 / sum(w) is applied once to the result.
// tests/hostsim/resize_hostsim.cpp builds this header with g++ and checks it against torch on the CPU.
#pragma once

#include <math.h>

#if defined(__CUDACC__)
#define BJ_RS_HD __host__ __device__ __forceinline__
#else
#define BJ_RS_HD inline
#endif

namespace bj {

struct RsAxis {
    float scale, support, inv;
    int n, m;
};

struct RsWindow {
    int lo, hi;   // taps [lo, hi) of the source axis
    float base;   // (lo - c + 0.5) * inv: filter argument of tap lo
};

BJ_RS_HD RsAxis rs_axis(int n, int m) {
    RsAxis a;
    a.n = n;
    a.m = m;
    a.scale = (float)n / (float)m;
    a.support = a.scale >= 1.0f ? a.scale : 1.0f;
    a.inv = a.scale >= 1.0f ? 1.0f / a.scale : 1.0f;
    return a;
}

BJ_RS_HD RsWindow rs_window(const RsAxis& a, int i) {
    RsWindow w;
    const float c = a.scale * ((float)i + 0.5f);
    int lo = (int)(c - a.support + 0.5f);
    int hi = (int)(c + a.support + 0.5f);
    w.lo = lo > 0 ? lo : 0;
    w.hi = hi < a.n ? hi : a.n;
    w.base = ((float)w.lo - c + 0.5f) * a.inv;
    return w;
}

// unnormalised weight of the tap whose filter argument is t
BJ_RS_HD float rs_weight(float t) { return fmaxf(1.0f - fabsf(t), 0.0f); }

// filter argument of tap k (= j - lo) of window w
BJ_RS_HD float rs_arg(const RsAxis& a, const RsWindow& w, float k) { return fmaf(k, a.inv, w.base); }

// 1 / sum of the window's weights (the sum is > 0 for every window rs_window returns).  Compensated summation: a
// plain fp32 sum over the thousands of taps of a large downscale drifts by ~1e-6.
BJ_RS_HD float rs_norm(const RsAxis& a, const RsWindow& w) {
    float s = 0.0f, comp = 0.0f;
    float k = 0.0f;
    for (int j = w.lo; j < w.hi; j++, k += 1.0f) {
        const float y = rs_weight(rs_arg(a, w, k)) - comp;
        const float t = s + y;
        comp = (t - s) - y;
        s = t;
    }
    return 1.0f / s;
}

}  // namespace bj
