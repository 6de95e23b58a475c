// Host build of the libjpeg-turbo arithmetic in pyjpegdecoder_b200/csrc/bj_ijg_math.cuh.
// TEST-ONLY: exposes the header's IDCT, upsampling, colour and window rules to the CPU suite, which compares them with
// tests/ijg_ref.py.  Never used by the product.
#include <cstdint>
#include "../../include/b200jpeg.h"
#include "../../pyjpegdecoder_b200/csrc/bj_ijg_math.cuh"

extern "C" {

// n blocks: d = 64 dequantised coefficients each, natural order; s = 64 samples each.
void hs_ijg_idct(int n, const int* d, uint8_t* s) {
    int ws[64];
    for (int i = 0; i < n; i++) bj::ijg_idct_block(d + 64 * i, ws, s + 64 * i);
}

// The upsampled (H_out, W_out) plane of one component from its real-size samples (dh, dw), row-major.
void hs_ijg_upsample(const uint8_t* plane, int dw, int dh, int rh, int rv, int w_out, int h_out, int* out) {
    auto at = [plane, dw](int x, int y) { return (int)plane[y * dw + x]; };
    for (int y = 0; y < h_out; y++)
        for (int x = 0; x < w_out; x++) out[y * w_out + x] = bj::ijg_sample(at, x, y, rh, rv, dw, dh);
}

// n pixels: ycc[3 i..3 i + 2] -> rgb[3 i..3 i + 2]
void hs_ijg_rgb(int n, const uint8_t* ycc, uint8_t* rgb) {
    for (int i = 0; i < n; i++) {
        uint32_t R, G, B;
        bj::ijg_ycc_rgb(ycc[3 * i], ycc[3 * i + 1], ycc[3 * i + 2], R, G, B);
        rgb[3 * i] = (uint8_t)R; rgb[3 * i + 1] = (uint8_t)G; rgb[3 * i + 2] = (uint8_t)B;
    }
}

void hs_ijg_window(const bj_image* im, const bj_crop_job* jb, int* w) { bj::ijg_window(*im, *jb, w[0], w[1], w[2], w[3]); }

}  // extern "C"
