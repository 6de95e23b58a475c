// bj_pixels.cu -- fused de-zigzag + dequantise + 8x8 IDCT + level shift, chroma upsampling and
// YCbCr->RGB for a whole batch of images in one launch (sm_100a).
//
// Replaces jpeg_decoder.py:868-891 (baseline per-block pixel work), :1306-1366 (progressive final
// stage) and :1368-1386 + :1683-1700 (crop, colour, clip).  See include/b200jpeg.h for the data
// layout and DESIGN.md for the roofline accounting (128 B of coefficients in, W*H*3 bytes out).
//
// One CTA = one strip of up to 192/blocks_per_mcu MCUs of one MCU row of one image:
//   load    the strip's coefficients are one contiguous run of 128-byte blocks (MCU-major layout):
//           coalesced 16-byte loads into shared memory, 16-byte chunks XOR-swizzled by block index.
//   phase A one thread per 8x8 block: de-zigzag + int16 dequantise + separable fp32 IDCT entirely in
//           registers (34 flops per 8-point pass).  The reference rounds an fp64 sum; a sample is
//           accepted from fp32 only if it is farther from a rounding tie than the fp32 error bound,
//           otherwise the whole block is recomputed warp-cooperatively in fp64 in numpy's pairwise
//           summation order (bit-exact with jpeg_decoder.py:1570).
//   phase B warps walk (pixel row, 8-pixel run) pairs, lanes walk MCUs: chroma is interpolated
//           with the reference's 3-tap Delaunay weights (integers /15, exact), colour conversion runs
//           in fp32 with the same near-tie test and an fp64 per-pixel fallback; RGB bytes are staged
//           in shared memory and leave with 128-bit coalesced stores.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200jpeg.h"
#include "bj_crop.cuh"
#include "bj_pixel_math.cuh"

namespace {

constexpr int kThreads = 192;
constexpr int kMaxBlocks = 192;  // blocks per strip
constexpr int kWarps = kThreads / 32;

__constant__ uint8_t c_zz_nat[64] = {BJ_ZZ_NATURAL};

struct Smem {
    // tile A: coefficients (int16, 128 B per block, swizzled); reused as the RGB staging buffer
    alignas(16) unsigned char a[kMaxBlocks * 128 + 512];
    // tile B: samples as fp32 (256 B per block, swizzled)
    alignas(16) float b[kMaxBlocks * 64];
    // 4-corner interpolation weights per upsampling kind and MCU pixel (b*16+a)
    alignas(16) float4 w[2][256];
    uint8_t wsel[4];  // component -> weight table
    alignas(16) int16_t qt[BJ_MAX_COMP][64];
    uint8_t slot_comp[16];
    uint8_t nat_zz[64];  // reference flat index u*8+v -> zig-zag index
};

__device__ __forceinline__ int swzA(int blk, int chunk) { return blk * 128 + ((chunk ^ (blk & 7)) << 4); }          // bytes
__device__ __forceinline__ int swzB(int blk, int chunk) { return blk * 64 + (((chunk ^ (blk & 15)) & 15) << 2); }   // floats

__device__ __forceinline__ float int_to_float_magic(int v) { return __int_as_float(v + BJ_MAGIC_BITS) - BJ_MAGIC; }

// ---- phase A: exact recompute of one block by a whole warp ------------------------------------
// Follows InverseDCT.__call__ (:1561-1573): for every output sample the 64 products
// block[u,v] * table[x,y,u,v] are summed by numpy's pairwise routine: accumulator j = v collects
// u = 0..7 in order, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)).  Zero coefficients contribute +-0.0
// and are skipped (r + 0.0 == r).  tabT is the table transposed to [u*8+v][x*8+y].
__device__ void recompute_block_exact(Smem& sm, int blk, const int16_t* qt, const double* __restrict__ tabT, int lane) {
    double r0[8], r1[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r0[j] = r1[j] = 0.0;
    const unsigned char* A = sm.a;
#pragma unroll
    for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int v = 0; v < 8; v++) {
            int n = u * 8 + v;
            int k = sm.nat_zz[n];
            int c = *reinterpret_cast<const int16_t*>(A + swzA(blk, k >> 3) + ((k & 7) << 1));
            if (c != 0) {  // warp-uniform
                int prod = (int16_t)(c * (int)qt[k]);
                double p = (double)prod;
                const double* t = tabT + n * 64;
                r0[v] = __dadd_rn(r0[v], __dmul_rn(p, t[lane]));
                r1[v] = __dadd_rn(r1[v], __dmul_rn(p, t[lane + 32]));
            }
        }
    }
    double s0 = __dadd_rn(__dadd_rn(__dadd_rn(r0[0], r0[1]), __dadd_rn(r0[2], r0[3])),
                          __dadd_rn(__dadd_rn(r0[4], r0[5]), __dadd_rn(r0[6], r0[7])));
    double s1 = __dadd_rn(__dadd_rn(__dadd_rn(r1[0], r1[1]), __dadd_rn(r1[2], r1[3])),
                          __dadd_rn(__dadd_rn(r1[4], r1[5]), __dadd_rn(r1[6], r1[7])));
    // sample index s = x*8+y (reference order); tile B is [y][x]
    int x0 = lane >> 3, y0 = lane & 7;
    float v0 = (float)((int16_t)(__double2int_rn(s0)) + 128);
    float v1 = (float)((int16_t)(__double2int_rn(s1)) + 128);
    sm.b[swzB(blk, 2 * y0 + (x0 >> 2)) + (x0 & 3)] = v0;
    int x1 = x0 + 4;
    sm.b[swzB(blk, 2 * y0 + (x1 >> 2)) + (x1 & 3)] = v1;
}

// ---- phase B helpers ---------------------------------------------------------------------------
__device__ __forceinline__ void load_row8(const Smem& sm, int blk, int row, float* o) {
    float4 lo = *reinterpret_cast<const float4*>(&sm.b[swzB(blk, 2 * row)]);
    float4 hi = *reinterpret_cast<const float4*>(&sm.b[swzB(blk, 2 * row + 1)]);
    o[0] = lo.x; o[1] = lo.y; o[2] = lo.z; o[3] = lo.w;
    o[4] = hi.x; o[5] = hi.y; o[6] = hi.z; o[7] = hi.w;
}

// cell index of output column a = 8*HX + p when the component is upsampled horizontally
template <int A> struct Cell { static constexpr int i = (A == 15) ? 6 : (7 * A) / 15; };

// 8 samples of component c for pixel row r, run HX of MCU m.  RH: horizontal ratio (1 or 2).
template <int RH, int HX>
__device__ __forceinline__ void comp_run(const Smem& sm, const bj_image& im, int c, int mblk0, int r, float* o) {
    const int hs = im.hs[c], vs = im.vs[c];
    const int rv = im.vmax / vs;
    if (RH == 1 && rv == 1) {
        int blk = mblk0 + im.slot0[c] + (r >> 3) * hs + (hs > 1 ? HX : 0);
        load_row8(sm, blk, r & 7, o);
        return;
    }
    int brow, j;
    if (rv == 2) { brow = 0; j = (r == 15) ? 6 : (7 * r) / 15; }
    else { brow = r >> 3; j = r & 7; }
    int j2 = j < 7 ? j + 1 : 7;
    int bcol = (RH == 2) ? 0 : (hs > 1 ? HX : 0);
    int blk = mblk0 + im.slot0[c] + brow * hs + bcol;
    float p0[8], p1[8];
    load_row8(sm, blk, j, p0);
    load_row8(sm, blk, j2, p1);
    const float4* w = &sm.w[sm.wsel[c]][(r & (8 * im.vmax - 1)) * 16 + 8 * HX];
#define BJ_PIX(P)                                                                              \
    {                                                                                          \
        constexpr int i = (RH == 2) ? Cell<8 * HX + P>::i : P;                                 \
        constexpr int i2 = i < 7 ? i + 1 : 7;                                                  \
        float4 ww = w[P];                                                                      \
        float n = fmaf(ww.w, p1[i2], fmaf(ww.z, p1[i], fmaf(ww.y, p0[i2], ww.x * p0[i])));     \
        o[P] = bj::div15_round(n);                                                             \
    }
    BJ_PIX(0) BJ_PIX(1) BJ_PIX(2) BJ_PIX(3) BJ_PIX(4) BJ_PIX(5) BJ_PIX(6) BJ_PIX(7)
#undef BJ_PIX
}

template <int HX>
__device__ __forceinline__ void comp_run_any(const Smem& sm, const bj_image& im, int c, int mblk0, int r, float* o) {
    if (im.hmax / im.hs[c] == 2) comp_run<2, HX>(sm, im, c, mblk0, r, o);
    else comp_run<1, HX>(sm, im, c, mblk0, r, o);
}

// exact colour conversion of one pixel, fp64, evaluation order of :1693-1695
__device__ __noinline__ void ycc_to_rgb_exact(float Yf, float Cbf, float Crf, int& R, int& G, int& B) {
    double Y = Yf, cb = __dsub_rn((double)Cbf, 128.0), cr = __dsub_rn((double)Crf, 128.0);
    double r = __dadd_rn(Y, __dmul_rn(1.402, cr));
    double g = __dsub_rn(__dsub_rn(Y, __dmul_rn(0.34414, cb)), __dmul_rn(0.71414, cr));
    double b = __dadd_rn(Y, __dmul_rn(1.772, cb));
    r = fmin(fmax(r, 0.0), 255.0);
    g = fmin(fmax(g, 0.0), 255.0);
    b = fmin(fmax(b, 0.0), 255.0);
    R = __double2int_rn(r);
    G = __double2int_rn(g);
    B = __double2int_rn(b);
}

__device__ __forceinline__ int clamp_round_u8(float v, float err, bool& tie) {
    float w = v + BJ_MAGIC;
    float r = w - BJ_MAGIC;
    // a tie matters only inside the clip range (:1698 clips before rounding)
    tie = tie || ((0.5f - fabsf(v - r)) < err && v > -1.0f && v < 256.0f);
    int iv = __float_as_int(w) - BJ_MAGIC_BITS;
    return min(max(iv, 0), 255);
}

template <int HX>
__device__ __forceinline__ void pixel_run(Smem& sm, const bj_image& im, int out_kind, int m, int mblk0, int r,
                                          int row_stride_s, int cols, void* out, int64_t gbase, uint32_t* stats) {
    float y[8];
    comp_run_any<HX>(sm, im, 0, mblk0, r, y);
    const int px0 = m * 8 * im.hmax + 8 * HX;  // pixel x inside the strip
    if (im.ncomp == 1) {
        if (out_kind == BJ_OUT_RGB) {
            unsigned char* s = sm.a + r * row_stride_s + px0;
            uint32_t lo = 0, hi = 0;
#pragma unroll
            for (int p = 0; p < 4; p++) {
                int a = min(max((int)y[p], 0), 255), b = min(max((int)y[p + 4], 0), 255);  // (:1385-1386)
                lo |= (uint32_t)a << (8 * p);
                hi |= (uint32_t)b << (8 * p);
            }
            *reinterpret_cast<uint2*>(s) = make_uint2(lo, hi);
        } else {
            int16_t* o = reinterpret_cast<int16_t*>(out) + gbase + (int64_t)r * im.out_pitch + px0;
#pragma unroll
            for (int p = 0; p < 8; p++)
                if (px0 + p < cols) o[p] = (int16_t)y[p];
        }
        return;
    }
    float cb[8], cr[8];
    comp_run_any<HX>(sm, im, 1, mblk0, r, cb);
    comp_run_any<HX>(sm, im, 2, mblk0, r, cr);
    if (out_kind == BJ_OUT_CANVAS) {
        int16_t* o = reinterpret_cast<int16_t*>(out) + gbase + (int64_t)r * im.out_pitch + (int64_t)px0 * 3;
#pragma unroll
        for (int p = 0; p < 8; p++) {
            if (px0 + p >= cols) break;
            o[3 * p] = (int16_t)y[p];
            o[3 * p + 1] = (int16_t)cb[p];
            o[3 * p + 2] = (int16_t)cr[p];
        }
        return;
    }
    uint32_t bytes[6] = {0, 0, 0, 0, 0, 0};
    int nslow = 0;
#pragma unroll
    for (int p = 0; p < 8; p++) {
        float R, G, B, err;
        bj::ycc_to_rgb_fast(y[p], cb[p], cr[p], R, G, B, err);
        bool tie = false;
        int ri = clamp_round_u8(R, err, tie);
        int gi = clamp_round_u8(G, err, tie);
        int bi = clamp_round_u8(B, err, tie);
        if (tie) {
            ycc_to_rgb_exact(y[p], cb[p], cr[p], ri, gi, bi);
            nslow++;
        }
        bytes[(3 * p) >> 2] |= (uint32_t)ri << (8 * ((3 * p) & 3));
        bytes[(3 * p + 1) >> 2] |= (uint32_t)gi << (8 * ((3 * p + 1) & 3));
        bytes[(3 * p + 2) >> 2] |= (uint32_t)bi << (8 * ((3 * p + 2) & 3));
    }
    if (stats && nslow) atomicAdd(&stats[1], (uint32_t)nslow);
    unsigned char* s = sm.a + r * row_stride_s + px0 * 3;  // 24-byte aligned -> 8-byte stores
    uint2* s2 = reinterpret_cast<uint2*>(s);
    s2[0] = make_uint2(bytes[0], bytes[1]);
    s2[1] = make_uint2(bytes[2], bytes[3]);
    s2[2] = make_uint2(bytes[4], bytes[5]);
}

// CROP: one CTA per strip of a bj_crop_job's MCU window (generic layout, scale 1, coefficients in, RGB out), storing
// only the box; in_kind, out_kind and only_generic_layout are then ignored.
template <bool CROP>
__global__ void __launch_bounds__(kThreads, 3)
bj_pixels_kernel(const bj_image* __restrict__ images, const void* __restrict__ in, int in_kind_arg,
                 const int16_t* __restrict__ qtabs, const double* __restrict__ tabT, void* __restrict__ out,
                 int out_kind_arg, int only_generic_layout, uint32_t* __restrict__ stats,
                 const bj_crop_job* __restrict__ jobs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    __shared__ bj_image im;
    const int in_kind = CROP ? BJ_IN_COEF : in_kind_arg;
    const int out_kind = CROP ? BJ_OUT_RGB : out_kind_arg;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    bj_crop_job jb{};
    if constexpr (CROP) jb = jobs[blockIdx.y];
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&images[CROP ? jb.image : blockIdx.y]);
        if (tid < (int)(sizeof(bj_image) / 4)) reinterpret_cast<uint32_t*>(&im)[tid] = src[tid];
    }
    __syncthreads();
    int my, m0, M;
    if constexpr (CROP) {
        if (im.layout != BJ_LAYOUT_GENERIC || jb.log2_scale != 0) return;  // other kernels' jobs
        if (!bj::crop_strip(jb, 8 * im.hmax, 8 * im.vmax, im.strip_mcus, blockIdx.x, my, m0, M)) return;
    } else {
        if (only_generic_layout && im.layout != BJ_LAYOUT_GENERIC) return;  // handled by bj_pixels_fast.cu
        const int strips_total = im.mcus_y * im.strips_per_row;
        if ((int)blockIdx.x >= strips_total) return;
        my = blockIdx.x / im.strips_per_row;
        m0 = (blockIdx.x % im.strips_per_row) * im.strip_mcus;
        M = min((int)im.strip_mcus, (int)im.mcus_x - m0);
    }
    const int bpm = im.blocks_per_mcu;
    const int nblk = M * bpm;
    const int64_t gblk0 = (int64_t)im.coef_block0 + ((int64_t)my * im.mcus_x + m0) * bpm;

    // ---- set-up tables -------------------------------------------------------------------------
    if (tid < 64) {
        int k = tid, nat = c_zz_nat[k];  // nat = v*8+u
        sm.nat_zz[(nat & 7) * 8 + (nat >> 3)] = (uint8_t)k;
    }
    for (int i = tid; i < im.ncomp * 64; i += kThreads) {
        int c = i >> 6;
        sm.qt[c][i & 63] = qtabs[(size_t)im.qtab[c] * 64 + (i & 63)];
    }
    if (tid < 16) {
        int s = tid, c = 0;
        for (int k = 0; k < im.ncomp; k++)
            if (s >= im.slot0[k]) c = k;
        sm.slot_comp[s] = (uint8_t)c;
    }
    // weight tables: one per distinct upsampling kind (rh, rv) != (1,1); at most two per image
    int kind0 = 0, kind1 = 0;
    for (int c = 0; c < im.ncomp; c++) {
        int kind = (im.hmax / im.hs[c]) * 4 + (im.vmax / im.vs[c]);
        int sel = 0;
        if (kind != 5) {
            if (kind0 == 0 || kind0 == kind) { kind0 = kind; sel = 0; }
            else { kind1 = kind; sel = 1; }
        }
        if (tid == 0) sm.wsel[c] = (uint8_t)sel;
    }
    for (int i = tid; i < 512; i += kThreads) {
        int kind = (i >> 8) ? kind1 : kind0;
        if (kind == 0) continue;
        int b = (i >> 4) & 15, a = i & 15;
        int rh = kind >> 2, rv = kind & 3;
        int ii = a & 7, s = 0, jj = b & 7, t = 0;
        if (rh == 2) bj::up_cell(a, ii, s);
        if (rv == 2) bj::up_cell(b, jj, t);
        int w00, w10, w01, w11;
        bj::up_weights_2d(ii, jj, s, t, w00, w10, w01, w11);
        sm.w[i >> 8][i & 255] = make_float4((float)w00, (float)w10, (float)w01, (float)w11);
    }

    // ---- load ----------------------------------------------------------------------------------
    if (in_kind == BJ_IN_COEF) {
        const uint4* g = reinterpret_cast<const uint4*>(reinterpret_cast<const int16_t*>(in) + gblk0 * 64);
        for (int i = tid; i < nblk * 8; i += kThreads) {
            uint4 v = __ldg(g + i);
            *reinterpret_cast<uint4*>(sm.a + swzA(i >> 3, i & 7)) = v;
        }
    } else {
        const uint4* g = reinterpret_cast<const uint4*>(reinterpret_cast<const int16_t*>(in) + gblk0 * 64);
        for (int i = tid; i < nblk * 8; i += kThreads) {  // 8 int16 = one row of a block
            uint4 v = __ldg(g + i);
            int blk = i >> 3, row = i & 7;
            const int16_t* h = reinterpret_cast<const int16_t*>(&v);
            float4 lo = make_float4(h[0], h[1], h[2], h[3]), hi = make_float4(h[4], h[5], h[6], h[7]);
            *reinterpret_cast<float4*>(&sm.b[swzB(blk, 2 * row)]) = lo;
            *reinterpret_cast<float4*>(&sm.b[swzB(blk, 2 * row + 1)]) = hi;
        }
    }
    __syncthreads();

    // ---- phase A: IDCT -------------------------------------------------------------------------
    if (in_kind == BJ_IN_COEF) {
        const int blk = tid;
        bool flagged = false;
        int comp = 0;
        if (blk < nblk) {
            comp = sm.slot_comp[blk % bpm];
            float f[64];
            float S = 0.f;
#pragma unroll
            for (int c = 0; c < 8; c++) {
                uint4 v = *reinterpret_cast<const uint4*>(sm.a + swzA(blk, c));
                uint4 q = *reinterpret_cast<const uint4*>(&sm.qt[comp][c * 8]);
                const uint32_t vw[4] = {v.x, v.y, v.z, v.w}, qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    int coef = (int16_t)(vw[e >> 1] >> (16 * (e & 1)));
                    int qq = (int16_t)(qw[e >> 1] >> (16 * (e & 1)));
                    int prod = (int16_t)(coef * qq);  // int16 * int16 -> int16 wraps (:869, :1348)
                    float x = int_to_float_magic(prod);
                    constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
                    f[zz[c * 8 + e]] = x;
                    S += fabsf(x);
                }
            }
            bj::idct8x8_fast(f);
            const float T = fmaf(S, BJ_IDCT_ERR_REL, BJ_IDCT_ERR_ABS);
            float mind = 1.0f;
#pragma unroll
            for (int y = 0; y < 8; y++) {
                float o[8];
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    float td;
                    float r = bj::round_tie(f[y * 8 + x], td);
                    mind = fminf(mind, td);
                    o[x] = r + 128.0f;
                }
                *reinterpret_cast<float4*>(&sm.b[swzB(blk, 2 * y)]) = make_float4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<float4*>(&sm.b[swzB(blk, 2 * y + 1)]) = make_float4(o[4], o[5], o[6], o[7]);
            }
            flagged = mind < T;
        }
        // warp-cooperative exact recompute of flagged blocks
        unsigned mask = __ballot_sync(0xffffffffu, flagged);
        if (mask) {
            __syncwarp();
            if (stats && lane == 0) atomicAdd(&stats[0], (uint32_t)__popc(mask));
            while (mask) {
                int src = __ffs(mask) - 1;
                mask &= mask - 1;
                int b2 = (warp << 5) + src;
                int c2 = __shfl_sync(0xffffffffu, comp, src);
                recompute_block_exact(sm, b2, sm.qt[c2], tabT, lane);
            }
        }
    }
    __syncthreads();

    // ---- samples out ---------------------------------------------------------------------------
    if (out_kind == BJ_OUT_SAMPLES) {
        uint4* g = reinterpret_cast<uint4*>(reinterpret_cast<int16_t*>(out) + gblk0 * 64);
        for (int i = tid; i < nblk * 8; i += kThreads) {
            int blk = i >> 3, row = i & 7;
            float4 lo = *reinterpret_cast<const float4*>(&sm.b[swzB(blk, 2 * row)]);
            float4 hi = *reinterpret_cast<const float4*>(&sm.b[swzB(blk, 2 * row + 1)]);
            int16_t h[8] = {(int16_t)lo.x, (int16_t)lo.y, (int16_t)lo.z, (int16_t)lo.w,
                            (int16_t)hi.x, (int16_t)hi.y, (int16_t)hi.z, (int16_t)hi.w};
            g[i] = *reinterpret_cast<const uint4*>(h);
        }
        return;
    }

    // ---- phase B: upsample + colour ------------------------------------------------------------
    const int mcu_w = 8 * im.hmax, mcu_h = 8 * im.vmax;
    const int ch = (im.ncomp == 3) ? 3 : 1;
    const int x0 = m0 * mcu_w, y0 = my * mcu_h;
    const int cols = min(M * mcu_w, (int)im.width - x0);   // visible pixel columns of the strip
    const int rows = min(mcu_h, (int)im.height - y0);      // visible rows
    const int row_stride_s = ((M * mcu_w * ch) + 15) & ~15;
    const int64_t gbase = (int64_t)im.out_offset + (int64_t)y0 * im.out_pitch + (int64_t)x0 * ch;
    const int pairs = mcu_h * im.hmax;
    const int chunks = (M + 31) >> 5;
    for (int it = warp; it < pairs * chunks; it += kWarps) {
        int pair = it % pairs, chunk = it / pairs;
        int r = pair / im.hmax, hx = pair % im.hmax;
        int m = (chunk << 5) + lane;
        if (r >= rows || m >= M) continue;
        if constexpr (CROP) {
            if (y0 + r < (int)jb.y0 || y0 + r >= (int)jb.y1) continue;   // rows outside the box are not stored
        }
        if (hx) pixel_run<1>(sm, im, out_kind, m, m * bpm, r, row_stride_s, cols, out, gbase, stats);
        else pixel_run<0>(sm, im, out_kind, m, m * bpm, r, row_stride_s, cols, out, gbase, stats);
    }
    if (out_kind != BJ_OUT_RGB) return;
    __syncthreads();

    if constexpr (CROP) {
        int sx, sy, w, h;
        uint8_t* g;
        if (bj::crop_part(jb, x0, y0, cols, rows, ch, reinterpret_cast<uint8_t*>(out), sx, sy, w, h, g))
            bj::crop_store(g, jb.out_pitch, sm.a + sy * row_stride_s, row_stride_s, sx * ch, w * ch, h, tid, kThreads);
        return;
    }
    // ---- coalesced copy-out of the staged rows -------------------------------------------------
    unsigned char* gout = reinterpret_cast<unsigned char*>(out) + gbase;
    const int nbytes = cols * ch;
    const bool aligned = ((reinterpret_cast<uintptr_t>(gout) & 15) == 0) && ((im.out_pitch & 15) == 0);
    if (aligned) {
        const int nvec = nbytes >> 4;
        for (int i = tid; i < rows * nvec; i += kThreads) {
            int r = i / nvec, v = i - r * nvec;
            uint4 val = *reinterpret_cast<const uint4*>(sm.a + r * row_stride_s + (v << 4));
            *reinterpret_cast<uint4*>(gout + (int64_t)r * im.out_pitch + (v << 4)) = val;
        }
        const int tail = nbytes & 15;
        if (tail) {
            for (int i = tid; i < rows * tail; i += kThreads) {
                int r = i / tail, b = (nvec << 4) + (i - r * tail);
                gout[(int64_t)r * im.out_pitch + b] = sm.a[r * row_stride_s + b];
            }
        }
    } else {
        for (int i = tid; i < rows * nbytes; i += kThreads) {
            int r = i / nbytes, b = i - r * nbytes;
            gout[(int64_t)r * im.out_pitch + b] = sm.a[r * row_stride_s + b];
        }
    }
}

thread_local char g_err[256] = "";

}  // namespace

extern "C" {

int bj_version(void) { return BJ_VERSION; }
int bj_sizeof(int what) {
    return what == 0 ? (int)sizeof(bj_image) : what == 1 ? (int)sizeof(bj_resize_job)
         : what == 2 ? (int)sizeof(bj_scaled_job) : what == 3 ? (int)sizeof(bj_crop_job)
         : what == 4 ? (int)sizeof(bj_resize_pil_job) : -1;
}
const char* bj_last_cuda_error(void) { return g_err; }

bj_status bj_set_cuda_error(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof g_err, "%s: %s", where, cudaGetErrorString(e));
    return BJ_E_CUDA;
}

bj_status bj_pixels_fast_launch(const bj_image* images, int n_images, int max_strips, const int16_t* coef,
                                const int16_t* qtabs, const double* tabT, uint8_t* out, uint32_t layout_mask,
                                uint32_t* stats, void* stream);
bj_status bj_pixels_420_launch(const bj_image* images, int n_images, int max_strips, const int16_t* coef,
                               uint64_t total_blocks, const int16_t* qtabs, const double* tabT, uint8_t* out,
                               uint32_t* stats, void* stream);

bj_status bj_pixels_fast_crop_launch(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                                     const int16_t* coef, const int16_t* qtabs, const double* tabT, uint8_t* out,
                                     uint32_t layout_mask, uint32_t* stats, void* stream);
bj_status bj_pixels_420_crop_launch(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                                    const int16_t* coef, uint64_t total_blocks, const int16_t* qtabs, const double* tabT,
                                    uint8_t* out, uint32_t* stats, void* stream);
bj_status bj_pixels_scaled_crop_launch(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                                       const int16_t* coef, const int16_t* qtabs, uint8_t* out, void* stream);

bj_status bj_pixels(const bj_image* images, int n_images, int max_strips, const void* in, int in_kind,
                    uint64_t total_blocks, const int16_t* qtabs, const double* idct_table_t, void* out, int out_kind,
                    uint32_t layout_mask, uint32_t* stats, void* stream) {
    if (!images || n_images <= 0 || max_strips <= 0 || !in || !qtabs || !idct_table_t || !out) return BJ_E_ARG;
    if (n_images > 65535) {
        // the image index rides on grid.y: larger batches run as slices (image records hold absolute buffer offsets)
        for (int i0 = 0; i0 < n_images; i0 += 65535) {
            const int n = n_images - i0 < 65535 ? n_images - i0 : 65535;
            bj_status st = bj_pixels(images + i0, n, max_strips, in, in_kind, total_blocks, qtabs, idct_table_t, out, out_kind,
                                     layout_mask, stats, stream);
            if (st != BJ_OK) return st;
        }
        return BJ_OK;
    }
    if (in_kind != BJ_IN_COEF && in_kind != BJ_IN_SAMPLES) return BJ_E_ARG;
    if (out_kind < BJ_OUT_RGB || out_kind > BJ_OUT_CANVAS) return BJ_E_ARG;
    static_assert(sizeof(bj_image) == 72, "bj_image layout");
    int only_generic = 0;
    if (in_kind == BJ_IN_COEF && out_kind == BJ_OUT_RGB && layout_mask != 0) {
        if (layout_mask & (1u << BJ_LAYOUT_420)) {
            bj_status st = bj_pixels_420_launch(images, n_images, max_strips, (const int16_t*)in, total_blocks, qtabs,
                                                idct_table_t, (uint8_t*)out, stats, stream);
            if (st != BJ_OK) return st;
        }
        if (layout_mask & ~(1u | (1u << BJ_LAYOUT_420))) {
            bj_status st = bj_pixels_fast_launch(images, n_images, max_strips, (const int16_t*)in, qtabs, idct_table_t,
                                                 (uint8_t*)out, layout_mask & ~(1u << BJ_LAYOUT_420), stats, stream);
            if (st != BJ_OK) return st;
        }
        if (!(layout_mask & 1u)) return BJ_OK;
        only_generic = 1;
    }
    cudaError_t e = cudaFuncSetAttribute(bj_pixels_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels/attr");
    dim3 grid((unsigned)max_strips, (unsigned)n_images);
    bj_pixels_kernel<false><<<grid, kThreads, sizeof(Smem), (cudaStream_t)stream>>>(images, in, in_kind, qtabs, idct_table_t, out,
                                                                                  out_kind, only_generic, stats, nullptr);
    e = cudaGetLastError();
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels/launch");
    return BJ_OK;
}

bj_status bj_pixels_crop(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips, const int16_t* coef,
                         uint64_t total_blocks, const int16_t* qtabs, const double* idct_table_t, uint8_t* out,
                         uint32_t kinds, uint32_t* stats, void* stream) {
    static_assert(sizeof(bj_crop_job) == 40, "bj_crop_job layout");
    if (!images || !jobs || n_jobs <= 0 || max_strips <= 0 || !coef || !qtabs || !idct_table_t || !out) return BJ_E_ARG;
    if (n_jobs > 65535) {
        // the job index rides on grid.y: larger batches run as slices (jobs hold absolute offsets)
        for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
            const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
            bj_status st = bj_pixels_crop(images, jobs + j0, n, max_strips, coef, total_blocks, qtabs, idct_table_t, out,
                                          kinds, stats, stream);
            if (st != BJ_OK) return st;
        }
        return BJ_OK;
    }
    bj_status st = BJ_OK;
    if (kinds & (1u << BJ_LAYOUT_420))
        st = bj_pixels_420_crop_launch(images, jobs, n_jobs, max_strips, coef, total_blocks, qtabs, idct_table_t, out,
                                       stats, stream);
    const uint32_t fast = kinds & ((1u << BJ_LAYOUT_422) | (1u << BJ_LAYOUT_440) | (1u << BJ_LAYOUT_444) | (1u << BJ_LAYOUT_GRAY));
    if (st == BJ_OK && fast)
        st = bj_pixels_fast_crop_launch(images, jobs, n_jobs, max_strips, coef, qtabs, idct_table_t, out, fast, stats,
                                        stream);
    if (st == BJ_OK && (kinds & BJ_CROP_SCALED))
        st = bj_pixels_scaled_crop_launch(images, jobs, n_jobs, max_strips, coef, qtabs, out, stream);
    if (st != BJ_OK || !(kinds & (1u << BJ_LAYOUT_GENERIC))) return st;
    cudaError_t e = cudaFuncSetAttribute(bj_pixels_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_crop/attr");
    bj_pixels_kernel<true><<<dim3((unsigned)max_strips, (unsigned)n_jobs), kThreads, sizeof(Smem), (cudaStream_t)stream>>>(
        images, coef, BJ_IN_COEF, qtabs, idct_table_t, out, BJ_OUT_RGB, 1, stats, jobs);
    e = cudaGetLastError();
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_crop/launch");
    return BJ_OK;
}

}  // extern "C"
