// bj_resize.cu -- antialiased bilinear resize + per-channel normalise of a whole batch of decoded images into one
// (N, 3, h, w) tensor, NCHW or NHWC, uint8 / fp16 / bf16 / fp32, in one launch (sm_100a).
//
// The filter is torch.nn.functional.interpolate(mode="bilinear", align_corners=False, antialias=True); its weights
// come from bj_resize_math.cuh, computed while accumulating (fp32).  See include/b200jpeg.h for the ABI.
//
// One CTA = one 32 x 32 output tile of one image (grid: tiles x images).  The tile's source box is walked in chunks
// of 16 source rows x up to 320 (RGB) / 960 (grey) source pixels, so any ratio works, from 2-tap upscales to
// thousands of taps per output:
//   stage       one warp per row: the chunk's rows leave global memory as coalesced aligned 4-byte loads (rows are
//               not aligned: the partial words at both ends are read byte by byte), become fp32 and go to shared
//               memory
//   horizontal  one thread per (source row, output column), all channels: partial sums over the chunk's taps are
//               kept in registers across column chunks, then written to shared memory
//   vertical    one thread per (output row, output column), all channels, accumulates the chunk's rows
// Neighbouring tiles share the source rows / columns under the overlap of their filter windows: a downscaling tile
// of 32 outputs reads the source of about 33 outputs per axis, 1.056 times the source box in all for
// 1080p -> 224 x 224 (tools/tensor_bench.py reports the factor).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_resize_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

constexpr int kThreads = 256;
constexpr int kTile = 32;      // output rows and columns per CTA
constexpr int kRows = 16;      // source rows per chunk
constexpr int kRowW = 978;     // floats per staged row (row stride = 18 mod 32 banks: the 16 rows a half-warp reads
                               // in the horizontal pass fall into distinct banks)
constexpr int kRowBytes = 961; // source bytes of a chunk row: + up to 3 bytes of alignment lead, in words, <= 978
constexpr int kWordsPerLane = 8; // (961 + 6) / 4 = 241 words of a staged row <= 8 x 32 lanes

struct Smem {
    alignas(16) float s[kRows * kRowW];   // staged source chunk, fp32, row rr starts at s[rr * kRowW + shift[rr]]
    float h[kRows * 3 * kTile];           // horizontal results [row][channel][output column]
    int lox[kTile], hix[kTile], loy[kTile], hiy[kTile];
    float basex[kTile], normx[kTile], basey[kTile], normy[kTile];
    int shift[kRows];
};

__device__ __forceinline__ float u8f(uint32_t w, int k) {
    // byte k of w as an exact fp32 value: 2^23 + b has b in its low mantissa bits
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7440u | (unsigned)k)) - 8388608.0f;
}

__device__ __forceinline__ void store_out(void* dst, uint32_t dtype, size_t idx, float v) {
    switch (dtype) {
    case BJ_DTYPE_U8: {
        const float r = fminf(fmaxf(rintf(v), 0.0f), 255.0f);
        static_cast<uint8_t*>(dst)[idx] = (uint8_t)r;
        break;
    }
    case BJ_DTYPE_F16: static_cast<__half*>(dst)[idx] = __float2half_rn(v); break;
    case BJ_DTYPE_BF16: static_cast<__nv_bfloat16*>(dst)[idx] = __float2bfloat16_rn(v); break;
    default: static_cast<float*>(dst)[idx] = v; break;
    }
}

template <int C>
__device__ __forceinline__ void resize_tile(const bj_resize_job& jb, const uint8_t* __restrict__ src, void* dst,
                                            const bj_resize_params& p, int ty, int tx, Smem& sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int out_h = (int)p.out_h, out_w = (int)p.out_w;
    const bj::RsAxis ax = bj::rs_axis((int)(jb.x1 - jb.x0), out_w);
    const bj::RsAxis ay = bj::rs_axis((int)(jb.y1 - jb.y0), out_h);
    const int ox0 = tx * kTile, oy0 = ty * kTile;
    const int nox = min(kTile, out_w - ox0), noy = min(kTile, out_h - oy0);
    if (tid < 2 * kTile) {
        const bool is_x = tid < kTile;
        const int i = tid & (kTile - 1);
        const bool valid = i < (is_x ? nox : noy);
        bj::RsWindow w{0, 0, 0.0f};
        float norm = 0.0f;
        if (valid) {
            w = bj::rs_window(is_x ? ax : ay, (is_x ? ox0 : oy0) + i);
            norm = bj::rs_norm(is_x ? ax : ay, w);
        }
        (is_x ? sm.lox : sm.loy)[i] = w.lo;
        (is_x ? sm.hix : sm.hiy)[i] = w.hi;
        (is_x ? sm.basex : sm.basey)[i] = w.base;
        (is_x ? sm.normx : sm.normy)[i] = norm;
    }
    __syncthreads();
    // window bounds grow with the output index: the tile's source box is [cx0, cx1) x [ry0, ry1)
    const int cx0 = sm.lox[0], cx1 = sm.hix[nox - 1];
    const int ry0 = sm.loy[0], ry1 = sm.hiy[noy - 1];
    constexpr int kChunkPx = (kRowBytes / C) < 960 ? (kRowBytes / C) : 960;
    const uint8_t* img = src + jb.src_offset + (size_t)jb.x0 * C;

    float acc[4][C];
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
        for (int c = 0; c < C; c++) acc[k][c] = 0.0f;

    for (int r0 = ry0; r0 < ry1; r0 += kRows) {
        const int nr = min(kRows, ry1 - r0);
        float hacc[2][C];
#pragma unroll
        for (int k = 0; k < 2; k++)
#pragma unroll
            for (int c = 0; c < C; c++) hacc[k][c] = 0.0f;

        for (int xc = cx0; xc < cx1; xc += kChunkPx) {
            const int ccw = min(kChunkPx, cx1 - xc);
            const int nbytes = ccw * C;
            const int nw = (nbytes + 6) >> 2;             // 4-byte words a row can touch (alignment lead <= 3)
            // one warp per row, lanes on consecutive words (coalesced 4-byte loads); a warp's two rows (16 rows, 8
            // warps) and all words of a row (<= 241 = 8 per lane) are loaded before the first one is used, so the
            // loads of a chunk wait for memory once instead of once per word
            uint32_t wv[2][kWordsPerLane];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int rr = warp + h * (kThreads / 32);
                const uint8_t* row = img + (size_t)(jb.y0 + r0 + min(rr, nr - 1)) * jb.src_pitch + (size_t)xc * C;
                const uintptr_t g = (uintptr_t)row, a0 = g & ~(uintptr_t)3;
                if (lane == 0 && rr < nr) sm.shift[rr] = (int)(g - a0);
#pragma unroll
                for (int u = 0; u < kWordsPerLane; u++) {
                    const int q = lane + 32 * u;
                    const uintptr_t a = a0 + 4 * (uintptr_t)q;
                    uint32_t w = 0;
                    if (rr < nr && q < nw) {
                        if (a >= g && a + 4 <= g + nbytes) {
                            w = __ldg(reinterpret_cast<const uint32_t*>(a));
                        } else {                           // the partial words at both ends: only the row's bytes
#pragma unroll
                            for (int b = 0; b < 4; b++)
                                if (a + b >= g && a + b < g + nbytes)
                                    w |= (uint32_t)*reinterpret_cast<const uint8_t*>(a + b) << (8 * b);
                        }
                    }
                    wv[h][u] = w;
                }
            }
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int rr = warp + h * (kThreads / 32);
                float2* d = reinterpret_cast<float2*>(&sm.s[rr * kRowW]);
#pragma unroll
                for (int u = 0; u < kWordsPerLane; u++) {
                    const int q = lane + 32 * u;
                    if (rr < nr && q < nw) {
                        d[2 * q] = make_float2(u8f(wv[h][u], 0), u8f(wv[h][u], 1));
                        d[2 * q + 1] = make_float2(u8f(wv[h][u], 2), u8f(wv[h][u], 3));
                    }
                }
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const int i = tid + k * kThreads;
                const int rr = i & (kRows - 1), oxl = i >> 4;
                if (rr < nr && oxl < nox) {
                    const int wlo = sm.lox[oxl];
                    const int lo = max(wlo, xc), hi = min(sm.hix[oxl], xc + ccw);
                    const float base = sm.basex[oxl];
                    const float* s = &sm.s[rr * kRowW + sm.shift[rr] + (lo - xc) * C];
                    float kk = (float)(lo - wlo);
                    for (int j = lo; j < hi; j++, kk += 1.0f, s += C) {
                        const float w = bj::rs_weight(fmaf(kk, ax.inv, base));
#pragma unroll
                        for (int c = 0; c < C; c++) hacc[k][c] = fmaf(w, s[c], hacc[k][c]);
                    }
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int i = tid + k * kThreads;
            const int rr = i & (kRows - 1), oxl = i >> 4;
            if (rr < nr && oxl < nox) {
#pragma unroll
                for (int c = 0; c < C; c++) sm.h[(rr * C + c) * kTile + oxl] = hacc[k][c];
            }
        }
        __syncthreads();
        // (the next chunk writes h only after the __syncthreads behind its staging: no barrier needed here)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int oyl = warp + 8 * k;
            if (oyl < noy && lane < nox) {
                const int wlo = sm.loy[oyl];
                const int lo = max(wlo, r0), hi = min(sm.hiy[oyl], r0 + nr);
                const float base = sm.basey[oyl];
                float kk = (float)(lo - wlo);
                for (int r = lo; r < hi; r++, kk += 1.0f) {
                    const float w = bj::rs_weight(fmaf(kk, ay.inv, base));
                    const float* hrow = &sm.h[(r - r0) * C * kTile + lane];
#pragma unroll
                    for (int c = 0; c < C; c++) acc[k][c] = fmaf(w, hrow[c * kTile], acc[k][c]);
                }
            }
        }
    }

#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int oyl = warp + 8 * k;
        if (oyl < noy && lane < nox) {
            const float norm = sm.normx[lane] * sm.normy[oyl];
            const int oy = oy0 + oyl, ox = ox0 + lane;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const float v = fmaf(acc[k][C == 3 ? c : 0] * norm, p.a[c], p.b[c]);
                const size_t idx = p.channels_last
                    ? (((size_t)jb.dst_index * out_h + oy) * out_w + ox) * 3 + c
                    : (((size_t)jb.dst_index * 3 + c) * out_h + oy) * out_w + ox;
                store_out(dst, p.dtype, idx, v);
            }
        }
    }
}

__global__ void __launch_bounds__(kThreads, 3)
bj_resize_kernel(const bj_resize_job* __restrict__ jobs, const uint8_t* __restrict__ src, void* dst,
                 const bj_resize_params p, int tiles_x) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const bj_resize_job jb = jobs[blockIdx.y];
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    if (jb.x1 <= jb.x0 || jb.y1 <= jb.y0) return;
    if (jb.channels == 3)
        resize_tile<3>(jb, src, dst, p, ty, tx, sm);
    else if (jb.channels == 1)
        resize_tile<1>(jb, src, dst, p, ty, tx, sm);
}

}  // namespace

extern "C" bj_status bj_resize(const bj_resize_job* jobs, int n_jobs, const uint8_t* src, void* dst,
                               const bj_resize_params* p, void* stream) {
    static_assert(sizeof(bj_resize_job) == 40, "bj_resize_job layout");
    if (!jobs || n_jobs <= 0 || !src || !dst || !p) return BJ_E_ARG;
    if (p->out_h < 1 || p->out_w < 1 || p->out_h > 65535 || p->out_w > 65535 || p->dtype > BJ_DTYPE_F32 ||
        p->channels_last > 1)
        return BJ_E_ARG;
    cudaError_t e = cudaFuncSetAttribute(bj_resize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_resize/attr");
    const int tiles_x = (int)((p->out_w + kTile - 1) / kTile), tiles_y = (int)((p->out_h + kTile - 1) / kTile);
    // the job index rides on grid.y (at most 65535): larger batches run as slices (jobs hold absolute offsets)
    for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
        const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
        bj_resize_kernel<<<dim3((unsigned)(tiles_x * tiles_y), (unsigned)n), kThreads, sizeof(Smem),
                           (cudaStream_t)stream>>>(jobs + j0, src, dst, *p, tiles_x);
        e = cudaGetLastError();
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_resize/launch");
    }
    return BJ_OK;
}
