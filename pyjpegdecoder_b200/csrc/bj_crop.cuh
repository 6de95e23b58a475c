// bj_crop.cuh -- what the crop variants of the pixel kernels share (include/b200jpeg.h, bj_pixels_crop): the strip of
// a job's MCU window a CTA decodes, and the store of a staged strip's part of the box to rows of any alignment.
#pragma once
#include <stdint.h>

#include "../../include/b200jpeg.h"

namespace bj {

// The strip of MCUs [m0, m0 + M) of MCU row my that CTA `bx` decodes: strips of up to `strip` MCUs walk the job's MCU
// window [mx0, mx1) x [my0, my1) (the window rule of include/b200jpeg.h; mw x mh: MCU size at the job's scale).
// Returns false if the CTA has no strip.
__device__ __forceinline__ bool crop_strip(const bj_crop_job& jb, int mw, int mh, int strip, int bx, int& my, int& m0,
                                           int& M) {
    const int mx0 = (int)jb.x0 / mw, mx1 = ((int)jb.x1 + mw - 1) / mw;
    const int my0 = (int)jb.y0 / mh, my1 = ((int)jb.y1 + mh - 1) / mh;
    const int spr = (mx1 - mx0 + strip - 1) / strip;
    if (bx >= (my1 - my0) * spr) return false;
    my = my0 + bx / spr;
    m0 = mx0 + (bx % spr) * strip;
    M = min(strip, mx1 - m0);
    return true;
}

// The part of the box a strip covers: strip pixels [x0, x0 + cols) x [y0, y0 + rows) clipped to the box.  Writes the
// staging offsets (sx: first column, sy: first row, both strip-relative), the size, and the destination of the
// first byte.  Returns false if the strip and the box do not meet.
__device__ __forceinline__ bool crop_part(const bj_crop_job& jb, int x0, int y0, int cols, int rows, int ch, uint8_t* out,
                                          int& sx, int& sy, int& w, int& h, uint8_t*& gout) {
    const int cx0 = max(x0, (int)jb.x0), cx1 = min(x0 + cols, (int)jb.x1);
    const int cy0 = max(y0, (int)jb.y0), cy1 = min(y0 + rows, (int)jb.y1);
    sx = cx0 - x0;
    sy = cy0 - y0;
    w = cx1 - cx0;
    h = cy1 - cy0;
    gout = out + jb.out_offset + (int64_t)(cy0 - (int)jb.y0) * jb.out_pitch + (int64_t)(cx0 - (int)jb.x0) * ch;
    return w > 0 && h > 0;
}

// rows x nbytes bytes from the staged rows (row r at stage + r * sstride + soff; sstride a multiple of 4) to
// gout + r * pitch, for any alignment of either side.  Threads t = 0..nt-1 walk the 16-byte chunks of the destination
// rows: a chunk inside the row is put together from five aligned 4-byte shared loads by funnel shifts and leaves as
// one 16-byte store; the partial chunks at both ends of a row go byte by byte.
__device__ __forceinline__ void crop_store(uint8_t* gout, uint32_t pitch, const unsigned char* stage, int sstride,
                                           int soff, int nbytes, int rows, int t, int nt) {
    if (nbytes <= 0) return;
    for (int i = t; i < rows * ((nbytes + 15) / 16 + 1); i += nt) {
        const int nv = (nbytes + 15) / 16 + 1;
        const int r = i / nv, v = i - r * nv;
        unsigned char* g = gout + (int64_t)r * pitch;
        const int lead = (int)(reinterpret_cast<uintptr_t>(g) & 15);
        const int lo = 16 * v - lead, hi = lo + 16;                   // chunk v in row bytes: [lo, hi)
        const unsigned char* s = stage + r * sstride + soff;
        if (lo >= 0 && hi <= nbytes) {
            const int a = soff + lo, sh = 8 * (a & 3);
            const uint32_t* w = reinterpret_cast<const uint32_t*>(stage + r * sstride + (a & ~3));
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = sh ? w[4] : 0u;
            *reinterpret_cast<uint4*>(g + lo) = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh),
                                                           __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
        } else {
            for (int b = max(lo, 0); b < min(hi, nbytes); b++) g[b] = s[b];
        }
    }
}

}  // namespace bj
