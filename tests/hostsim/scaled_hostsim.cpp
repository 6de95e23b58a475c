// Host build of the reduced-size decode arithmetic in pyjpegdecoder_b200/csrc/bj_scaled_math.cuh.
// TEST-ONLY: a sequential host model of bj_pixels_scaled that calls the header's functions (the header is
// __host__ __device__ and uses explicit fmaf only), so the CPU suite checks the exact fp32 arithmetic of the kernel and
// the GPU suite compares the kernel's bytes with this model.  Never used by the product.
#include <cstdint>
#include <cmath>
#include <vector>
#include "../../include/b200jpeg.h"
#include "../../pyjpegdecoder_b200/csrc/bj_scaled_math.cuh"

extern "C" {

int hs_scaled_prefix(int nx, int ny) { return bj::scaled_prefix(nx, ny); }

// One block: coef / q are 64 entries in zig-zag order.  f: the NY x NX values before rounding; samples: after.
void hs_scaled_block(int lnx, int lny, const int16_t* coef, const int16_t* q, float* f, float* samples) {
    auto cf = [coef](int k) { return (int)coef[k]; };
    bj::scaled_tile(lnx, lny, cf, q, f, 1 << lnx, true);
    bj::scaled_tile(lnx, lny, cf, q, samples, 1 << lnx, false);
}

// One job of bj_pixels_scaled over an MCU-major coefficient buffer (blocks of 64 int16, zig-zag order).
void hs_scaled_image(const bj_image* im, const bj_scaled_job* job, const int16_t* coef, const int16_t* qtabs,
                     uint8_t* out) {
    const int l = (int)job->log2_scale;
    const int mcu_w = (8 * im->hmax) >> l, mcu_h = (8 * im->vmax) >> l;
    const int PW = (int)im->mcus_x * mcu_w, PH = (int)im->mcus_y * mcu_h;
    std::vector<float> planes((size_t)im->ncomp * PW * PH);
    for (int my = 0; my < (int)im->mcus_y; my++)
        for (int mx = 0; mx < (int)im->mcus_x; mx++)
            for (int c = 0; c < im->ncomp; c++) {
                const int lx = bj::scaled_log2_side(im->hmax, im->hs[c], l);
                const int ly = bj::scaled_log2_side(im->vmax, im->vs[c], l);
                for (int r = 0; r < im->hs[c] * im->vs[c]; r++) {
                    const int bx = r % im->hs[c], by = r / im->hs[c];
                    const int64_t blk = (int64_t)im->coef_block0 + ((int64_t)my * im->mcus_x + mx) * im->blocks_per_mcu +
                                        im->slot0[c] + r;
                    const int16_t* b = coef + blk * 64;
                    auto cf = [b](int k) { return (int)b[k]; };
                    const int x = mx * mcu_w + (bx << lx), y = my * mcu_h + (by << ly);
                    bj::scaled_tile(lx, ly, cf, qtabs + (size_t)im->qtab[c] * 64,
                                    &planes[((size_t)c * PH + y) * PW + x], PW);
                }
            }
    const int out_w = ((int)im->width + (1 << l) - 1) >> l, out_h = ((int)im->height + (1 << l) - 1) >> l;
    const size_t plane = (size_t)PW * PH;
    for (int y = 0; y < out_h; y++)
        for (int x = 0; x < out_w; x++) {
            const float* P = &planes[(size_t)y * PW + x];
            uint8_t* d = out + job->out_offset + (size_t)y * job->out_pitch;
            if (im->ncomp == 3) {
                uint32_t R, G, B;
                bj::scaled_rgb(P[0], P[plane], P[2 * plane], R, G, B);
                d[3 * x] = (uint8_t)R; d[3 * x + 1] = (uint8_t)G; d[3 * x + 2] = (uint8_t)B;
            } else {
                d[x] = (uint8_t)bj::scaled_u8(P[0]);
            }
        }
}

}  // extern "C"
