// bj_resize_pil.cu -- Pillow's BILINEAR / BICUBIC resize (Image.resize), bit for bit, + per-channel normalise of a
// whole batch of decoded images into one (N, 3, h, w) tensor, NCHW or NHWC, uint8 / fp16 / bf16 / fp32, in one launch
// (sm_100a).  The arithmetic is bj_resize_pil_math.cuh; see include/b200jpeg.h for the ABI.
//
// One CTA = one 32 x 32 output tile of one job (grid: tiles x jobs).  Each job resizes its box to a virtual
// (virt_h, virt_w) image of which only the out_h x out_w window at (win_x, win_y) exists, so a tile's outputs are
// virtual outputs win + tile offset + i and use the full resize's coefficients.
//   setup       one thread per tile column / row: Pillow's window and double weight sum of that output
//   tables      the tile's int32 coefficients, in shared memory: the whole window of every output when ksize fits
//               the table (kCapX horizontal taps, kCapY vertical ones), else only the taps of the chunk being
//               processed, recomputed per chunk (extreme downscales)
//   row chunks  the source rows the tile's vertical taps reach, kRows at a time:
//     stage       one warp per row: coalesced aligned 4-byte loads of up to kCapX source pixels (the partial words at
//                 both ends are read byte by byte), into shared memory as bytes
//     horizontal  one thread per (source row, output column): int32 partial sums across column chunks, then
//                 clip8 -> the uint8 intermediate in shared memory (Pillow's imTemp rows of this tile)
//     vertical    one thread per (output row, output column) accumulates the chunk's rows in int32
//   store       clip8, then v * a[c] + b[c] in the requested dtype
// All sums are exact int32 (the header bounds every partial sum), so splitting the taps into chunks changes nothing.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_resize_pil_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

constexpr int kThreads = 256;
constexpr int kTile = 32;        // output rows and columns per CTA
constexpr int kRows = 32;        // source rows per chunk
constexpr int kCapX = 128;       // horizontal taps per output column in the table; source columns per staged chunk
constexpr int kCapY = 64;        // vertical taps per output row in the table (>= kRows)
constexpr int kRowBytes = 388;   // staged row: 128 RGB pixels + up to 3 bytes of alignment lead = 97 words; an odd
                                 // word stride puts the 32 rows a warp reads in the horizontal pass in distinct banks
constexpr int kWordsPerLane = 4; // 97 words of a staged row <= 4 x 32 lanes
static_assert(BJ_PIL_BILINEAR == bj::kPilBilinear && BJ_PIL_BICUBIC == bj::kPilBicubic, "filter numbering");
static_assert(kRows <= kCapY, "a vertical chunk's taps fit the table");
static_assert(3 * kCapX + 3 <= kRowBytes, "a staged chunk fits its row");

struct Smem {
    int32_t kx[kTile * kCapX];
    int32_t ky[kTile * kCapY];
    alignas(16) uint8_t stage[kRows * kRowBytes];
    uint8_t t[kRows * 3 * kTile];    // horizontal results [row][channel][output column]
    double cx[kTile], wwx[kTile], cy[kTile], wwy[kTile];
    int xmin[kTile], xn[kTile], ymin[kTile], yn[kTile];
    int shift[kRows];
};

// The coefficients of the tile's nout outputs for the source taps in [a, b): tap j of output i at
// tab[i * cap + j - max(lo[i], a)].  With a = 0 and b = the axis length this is every output's whole window.
__device__ __forceinline__ void fill_table(int32_t* tab, int cap, const bj::PilAxis& ax, int filter, const int* lo,
                                           const int* n, const double* c, const double* ww, int nout, int a, int b) {
    for (int e = threadIdx.x; e < nout * cap; e += kThreads) {
        const int i = e / cap, t = e - i * cap;
        const int base = max(lo[i], a), j = base + t;
        if (j < min(lo[i] + n[i], b)) {
            const bj::PilWindow w{lo[i], n[i], c[i], ww[i]};
            tab[e] = bj::pil_coeff(ax, w, filter, j - lo[i]);
        }
    }
}

__device__ __forceinline__ void store_out(void* dst, uint32_t dtype, size_t idx, int v, float a, float b) {
    switch (dtype) {
    case BJ_DTYPE_U8: static_cast<uint8_t*>(dst)[idx] = (uint8_t)v; break;
    case BJ_DTYPE_F16: static_cast<__half*>(dst)[idx] = __float2half_rn(fmaf((float)v, a, b)); break;
    case BJ_DTYPE_BF16: static_cast<__nv_bfloat16*>(dst)[idx] = __float2bfloat16_rn(fmaf((float)v, a, b)); break;
    default: static_cast<float*>(dst)[idx] = fmaf((float)v, a, b); break;
    }
}

template <int C>
__device__ __forceinline__ void resize_tile(const bj_resize_pil_job& jb, const uint8_t* __restrict__ src, void* dst,
                                            const bj_resize_params& p, int filter, int ty, int tx, Smem& sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int out_h = (int)p.out_h, out_w = (int)p.out_w;
    const bj::PilAxis ax = bj::pil_axis((int)(jb.x1 - jb.x0), (int)jb.virt_w, filter);
    const bj::PilAxis ay = bj::pil_axis((int)(jb.y1 - jb.y0), (int)jb.virt_h, filter);
    const int ox0 = tx * kTile, oy0 = ty * kTile;
    const int nox = min(kTile, out_w - ox0), noy = min(kTile, out_h - oy0);
    if (tid < 2 * kTile) {
        const bool is_x = tid < kTile;
        const int i = tid & (kTile - 1);
        if (i < (is_x ? nox : noy)) {
            bj::PilWindow w = bj::pil_window(is_x ? ax : ay, is_x ? (int)jb.win_x + ox0 + i : (int)jb.win_y + oy0 + i);
            bj::pil_window_sum(is_x ? ax : ay, w, filter);
            (is_x ? sm.xmin : sm.ymin)[i] = w.xmin;
            (is_x ? sm.xn : sm.yn)[i] = w.n;
            (is_x ? sm.cx : sm.cy)[i] = w.center;
            (is_x ? sm.wwx : sm.wwy)[i] = w.ww;
        }
    }
    __syncthreads();
    // windows grow with the output index: the tile's source box is [cx0, cx1) x [ry0, ry1)
    const int cx0 = sm.xmin[0], cx1 = sm.xmin[nox - 1] + sm.xn[nox - 1];
    const int ry0 = sm.ymin[0], ry1 = sm.ymin[noy - 1] + sm.yn[noy - 1];
    const bool whole_x = ax.ksize <= kCapX, whole_y = ay.ksize <= kCapY;
    if (whole_x) fill_table(sm.kx, kCapX, ax, filter, sm.xmin, sm.xn, sm.cx, sm.wwx, nox, 0, ax.in);
    if (whole_y) fill_table(sm.ky, kCapY, ay, filter, sm.ymin, sm.yn, sm.cy, sm.wwy, noy, 0, ay.in);
    const uint8_t* img = src + jb.src_offset + (size_t)jb.x0 * C;

    int32_t acc[4][C];
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
        for (int c = 0; c < C; c++) acc[k][c] = 0;

    for (int r0 = ry0; r0 < ry1; r0 += kRows) {
        const int nr = min(kRows, ry1 - r0);
        if (!whole_y) fill_table(sm.ky, kCapY, ay, filter, sm.ymin, sm.yn, sm.cy, sm.wwy, noy, r0, r0 + nr);
        int32_t hacc[4][C];
#pragma unroll
        for (int k = 0; k < 4; k++)
#pragma unroll
            for (int c = 0; c < C; c++) hacc[k][c] = 0;

        for (int xc = cx0; xc < cx1; xc += kCapX) {
            const int ncw = min(kCapX, cx1 - xc);
            if (!whole_x) fill_table(sm.kx, kCapX, ax, filter, sm.xmin, sm.xn, sm.cx, sm.wwx, nox, xc, xc + ncw);
            const int nbytes = ncw * C;
#pragma unroll
            for (int h = 0; h < kRows / 8; h++) {
                const int rr = warp + 8 * h;
                if (rr >= nr) continue;
                const uint8_t* row = img + (size_t)(jb.y0 + r0 + rr) * jb.src_pitch + (size_t)xc * C;
                const uintptr_t g = (uintptr_t)row, a0 = g & ~(uintptr_t)3;
                const int nw = (int)((g - a0 + nbytes + 3) >> 2);
                if (lane == 0) sm.shift[rr] = (int)(g - a0);
                uint32_t* d = reinterpret_cast<uint32_t*>(&sm.stage[rr * kRowBytes]);
#pragma unroll
                for (int u = 0; u < kWordsPerLane; u++) {
                    const int q = lane + 32 * u;
                    if (q < nw) {
                        const uintptr_t a = a0 + 4 * (uintptr_t)q;
                        uint32_t w = 0;
                        if (a >= g && a + 4 <= g + nbytes) {
                            w = __ldg(reinterpret_cast<const uint32_t*>(a));
                        } else {                           // the partial words at both ends: only the row's bytes
#pragma unroll
                            for (int b = 0; b < 4; b++)
                                if (a + b >= g && a + b < g + nbytes)
                                    w |= (uint32_t)*reinterpret_cast<const uint8_t*>(a + b) << (8 * b);
                        }
                        d[q] = w;
                    }
                }
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int i = tid + k * kThreads;
                const int rr = i & (kRows - 1), oxl = i >> 5;
                if (rr < nr && oxl < nox) {
                    const int wlo = sm.xmin[oxl];
                    const int lo = max(wlo, xc), hi = min(wlo + sm.xn[oxl], xc + ncw);
                    const int32_t* kk = &sm.kx[oxl * kCapX + lo - (whole_x ? wlo : lo)];
                    const uint8_t* s = &sm.stage[rr * kRowBytes + sm.shift[rr] + (lo - xc) * C];
                    for (int j = 0; j < hi - lo; j++, s += C) {
                        const int32_t kv = kk[j];
#pragma unroll
                        for (int c = 0; c < C; c++) hacc[k][c] += kv * (int32_t)s[c];
                    }
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = tid + k * kThreads;
            const int rr = i & (kRows - 1), oxl = i >> 5;
            if (rr < nr && oxl < nox) {
#pragma unroll
                for (int c = 0; c < C; c++) sm.t[(rr * C + c) * kTile + oxl] = bj::pil_clip8(bj::kPilRound + hacc[k][c]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int oyl = warp + 8 * k;
            if (oyl < noy && lane < nox) {
                const int wlo = sm.ymin[oyl];
                const int lo = max(wlo, r0), hi = min(wlo + sm.yn[oyl], r0 + nr);
                const int32_t* kk = &sm.ky[oyl * kCapY + lo - (whole_y ? wlo : lo)];
                for (int r = lo; r < hi; r++) {
                    const int32_t kv = kk[r - lo];
                    const uint8_t* trow = &sm.t[(r - r0) * C * kTile + lane];
#pragma unroll
                    for (int c = 0; c < C; c++) acc[k][c] += kv * (int32_t)trow[c * kTile];
                }
            }
        }
        __syncthreads();   // the next chunk refills ky (chunked tables) and rewrites t
    }

#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int oyl = warp + 8 * k;
        if (oyl < noy && lane < nox) {
            const int oy = oy0 + oyl, ox = ox0 + lane;
            int v[C];
#pragma unroll
            for (int c = 0; c < C; c++) v[c] = bj::pil_clip8(bj::kPilRound + acc[k][c]);
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const size_t idx = p.channels_last
                    ? (((size_t)jb.dst_index * out_h + oy) * out_w + ox) * 3 + c
                    : (((size_t)jb.dst_index * 3 + c) * out_h + oy) * out_w + ox;
                store_out(dst, p.dtype, idx, v[C == 3 ? c : 0], p.a[c], p.b[c]);
            }
        }
    }
}

__global__ void __launch_bounds__(kThreads, 4)   // 64 registers (4 bytes spilled): 4 CTAs per SM, 1.06x faster than 3
bj_resize_pil_kernel(const bj_resize_pil_job* __restrict__ jobs, const uint8_t* __restrict__ src, void* dst,
                     const bj_resize_params p, int filter, int tiles_x) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const bj_resize_pil_job jb = jobs[blockIdx.y];
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    // virtual sizes up to INT32_MAX: they enter only the double coefficient arithmetic and the int output index
    if (jb.x1 <= jb.x0 || jb.y1 <= jb.y0 || jb.virt_w < 1 || jb.virt_h < 1 || jb.virt_w > 0x7fffffffu ||
        jb.virt_h > 0x7fffffffu || jb.win_x + p.out_w > jb.virt_w || jb.win_y + p.out_h > jb.virt_h)
        return;
    if (jb.channels == 3)
        resize_tile<3>(jb, src, dst, p, filter, ty, tx, sm);
    else if (jb.channels == 1)
        resize_tile<1>(jb, src, dst, p, filter, ty, tx, sm);
}

}  // namespace

extern "C" bj_status bj_resize_pil(const bj_resize_pil_job* jobs, int n_jobs, const uint8_t* src, void* dst,
                                   const bj_resize_params* p, int filter, void* stream) {
    static_assert(sizeof(bj_resize_pil_job) == 56, "bj_resize_pil_job layout");
    if (!jobs || n_jobs <= 0 || !src || !dst || !p) return BJ_E_ARG;
    if (p->out_h < 1 || p->out_w < 1 || p->out_h > 65535 || p->out_w > 65535 || p->dtype > BJ_DTYPE_F32 ||
        p->channels_last > 1 || (filter != BJ_PIL_BILINEAR && filter != BJ_PIL_BICUBIC))
        return BJ_E_ARG;
    cudaError_t e = cudaFuncSetAttribute(bj_resize_pil_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)sizeof(Smem));
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_resize_pil/attr");
    const int tiles_x = (int)((p->out_w + kTile - 1) / kTile), tiles_y = (int)((p->out_h + kTile - 1) / kTile);
    // the job index rides on grid.y (at most 65535): larger batches run as slices (jobs hold absolute offsets)
    for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
        const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
        bj_resize_pil_kernel<<<dim3((unsigned)(tiles_x * tiles_y), (unsigned)n), kThreads, sizeof(Smem),
                               (cudaStream_t)stream>>>(jobs + j0, src, dst, *p, filter, tiles_x);
        e = cudaGetLastError();
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_resize_pil/launch");
    }
    return BJ_OK;
}
