// Host build of Pillow's resample arithmetic in pyjpegdecoder_b200/csrc/bj_resize_pil_math.cuh.
// TEST-ONLY: the CPU suite compares the header's coefficient tables and passes with tests/pil_resample_ref.py, and
// checks the int32 partial-sum bound the header derives.  Never used by the product.
#include <cstdint>
#include <vector>
#include "../../pyjpegdecoder_b200/csrc/bj_resize_pil_math.cuh"

extern "C" {

int hs_pil_ksize(int in, int out, int filter) { return bj::pil_axis(in, out, filter).ksize; }

// The (out, ksize) int32 coefficient table of an in -> out axis and each output's window [xmin, xmin + n).
void hs_pil_coeffs(int in, int out, int filter, int32_t* xmin, int32_t* n, int32_t* k) {
    const bj::PilAxis a = bj::pil_axis(in, out, filter);
    for (int xx = 0; xx < out; xx++) {
        bj::PilWindow w = bj::pil_window(a, xx);
        bj::pil_window_sum(a, w, filter);
        xmin[xx] = w.xmin;
        n[xx] = w.n;
        for (int x = 0; x < a.ksize; x++) k[(int64_t)xx * a.ksize + x] = x < w.n ? bj::pil_coeff(a, w, filter, x) : 0;
    }
}

// Image.resize((w, h)) of a uint8 (H, W, C) image the way the kernel computes it: horizontal pass (int32, clip8 to
// uint8), then vertical pass, every pass run (also when a size is unchanged).
void hs_pil_resize(const uint8_t* img, int W, int H, int C, int w, int h, int filter, uint8_t* out) {
    const bj::PilAxis ax = bj::pil_axis(W, w, filter), ay = bj::pil_axis(H, h, filter);
    std::vector<uint8_t> t((size_t)H * w * C);
    for (int ox = 0; ox < w; ox++) {
        bj::PilWindow win = bj::pil_window(ax, ox);
        bj::pil_window_sum(ax, win, filter);
        std::vector<int32_t> k(win.n);
        for (int x = 0; x < win.n; x++) k[x] = bj::pil_coeff(ax, win, filter, x);
        for (int y = 0; y < H; y++)
            for (int c = 0; c < C; c++) {
                int32_t s = bj::kPilRound;
                for (int x = 0; x < win.n; x++) s += k[x] * (int32_t)img[((size_t)y * W + win.xmin + x) * C + c];
                t[((size_t)y * w + ox) * C + c] = bj::pil_clip8(s);
            }
    }
    for (int oy = 0; oy < h; oy++) {
        bj::PilWindow win = bj::pil_window(ay, oy);
        bj::pil_window_sum(ay, win, filter);
        std::vector<int32_t> k(win.n);
        for (int y = 0; y < win.n; y++) k[y] = bj::pil_coeff(ay, win, filter, y);
        for (int ox = 0; ox < w; ox++)
            for (int c = 0; c < C; c++) {
                int32_t s = bj::kPilRound;
                for (int y = 0; y < win.n; y++) s += k[y] * (int32_t)t[((size_t)(win.xmin + y) * w + ox) * C + c];
                out[((size_t)oy * w + ox) * C + c] = bj::pil_clip8(s);
            }
    }
}

// The adversarial inputs of the header's bound, per output of an in -> out axis: src = 255 where k > 0 (k < 0) and 0
// elsewhere, summed from 2^21 in tap order in int64.  hi / lo: the largest / smallest partial sum over all outputs.
void hs_pil_partial_extremes(int in, int out, int filter, int64_t* hi, int64_t* lo) {
    const bj::PilAxis a = bj::pil_axis(in, out, filter);
    int64_t mx = bj::kPilRound, mn = bj::kPilRound;
    for (int xx = 0; xx < out; xx++) {
        bj::PilWindow w = bj::pil_window(a, xx);
        bj::pil_window_sum(a, w, filter);
        int64_t sp = bj::kPilRound, sn = bj::kPilRound;
        for (int x = 0; x < w.n; x++) {
            const int32_t k = bj::pil_coeff(a, w, filter, x);
            if (k > 0) sp += 255 * (int64_t)k;
            if (k < 0) sn += 255 * (int64_t)k;
            mx = sp > mx ? sp : mx;
            mn = sn < mn ? sn : mn;
        }
    }
    *hi = mx;
    *lo = mn;
}

}  // extern "C"
