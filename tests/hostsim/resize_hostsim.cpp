// Host build of the resize filter weights in pyjpegdecoder_b200/csrc/bj_resize_math.cuh.
// TEST-ONLY: the CPU test-suite checks the exact fp32 weights the CUDA kernel uses (the header is __host__ __device__
// and uses explicit fmaf only).  Never used by the product.
#include <cstdint>
#include <cmath>
#include "../../pyjpegdecoder_b200/csrc/bj_resize_math.cuh"

extern "C" {

// Dense (m, n) matrix of the normalised weights of an n -> m resize, as the kernel applies them:
// w(i, j) = rs_weight(rs_arg(k = j - lo)) * rs_norm.  lo / hi: the window of each output.
void hs_resize_weights(int n, int m, float* w, int32_t* lo, int32_t* hi) {
    const bj::RsAxis a = bj::rs_axis(n, m);
    for (int i = 0; i < m; i++) {
        const bj::RsWindow win = bj::rs_window(a, i);
        const float norm = bj::rs_norm(a, win);
        lo[i] = win.lo;
        hi[i] = win.hi;
        for (int j = 0; j < n; j++) w[(int64_t)i * n + j] = 0.0f;
        float k = 0.0f;
        for (int j = win.lo; j < win.hi; j++, k += 1.0f) w[(int64_t)i * n + j] = bj::rs_weight(bj::rs_arg(a, win, k)) * norm;
    }
}

}  // extern "C"
