// bj_pixels_fast.cu -- layout-specialised fused pixel kernel (sm_100a): de-zigzag + dequantise +
// 8x8 IDCT + level shift + chroma upsampling + YCbCr->RGB + clamp, coefficients in, RGB bytes out.
//
// Same arithmetic contract as the generic kernel in bj_pixels.cu (bit-exact with the reference's
// fp64 path, jpeg_decoder.py:869-891, :1306-1366, :1368-1386, :1683-1700) but the sampling layout is
// a template parameter (4:2:0, 4:2:2, 4:4:0, 4:4:4, greyscale), so every index computation, division
// and branch on the geometry folds at compile time.
//
// WARP-AUTONOMOUS design: a warp owns 32/blocks_per_mcu whole MCUs (4:2:0: 5 MCUs = 30 blocks) and
// does everything for them -- cp.async load of its contiguous 128-byte coefficient blocks into its
// private, bank-swizzled shared-memory tile, one lane per block for the register IDCT, the exact
// recompute of flagged blocks, the per-pixel colour stage and the stores of its 16-row output
// segment -- with __syncwarp() only.  After the one-time table set-up there is no CTA barrier, so the
// 18 warps of an SM run at independent phases and hide each other's load/store latency.
//   * luma samples stay int16 in shared memory (128 B per block); only chroma is kept as fp32
//     because it is interpolated.  R/G/B = clamp(Y + round(offset(Cb,Cr))): the rounding tie test
//     only involves the chroma offsets (Y is an integer), see bj_pixel_math.cuh;
//   * add + clamp is one VIADDMNMX (__viaddmin_s32_relu);
//   * the exact fp64 recompute of a flagged block iterates over its non-zero coefficients only
//     (ballot masks), in numpy's pairwise order.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_crop.cuh"
#include "bj_pixel_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

constexpr int kWarps = 6;
constexpr int kThreads = kWarps * 32;
constexpr int kWStride = 17;  // float4 entries per weight-table row (16 + 1 pad: lanes read different rows)

template <int HMAX_, int VMAX_, int NCOMP_>
struct Lay {
    static constexpr int HMAX = HMAX_, VMAX = VMAX_, NCOMP = NCOMP_;
    static constexpr int NY = HMAX * VMAX;
    static constexpr int BPM = NY + (NCOMP == 3 ? 2 : 0);
    static constexpr int MCU_W = 8 * HMAX, MCU_H = 8 * VMAX;
    static constexpr bool UPS = (NCOMP == 3) && (NY > 1);
    static constexpr int CH = NCOMP == 3 ? 3 : 1;
    static constexpr int MPW = 32 / BPM;          // MCUs per warp
    static constexpr int STRIP = kWarps * MPW;    // MCUs per CTA (must match plan.py: choose_strip)
    static constexpr int MCU_B = NY * 128 + (NCOMP == 3 ? 512 : 0);  // sample-tile bytes per MCU
    static constexpr int A_BYTES = 32 * 128;      // coefficient tile of a warp, reused as RGB staging
    static constexpr int B_BYTES = MPW * MCU_B;
    static constexpr int WARP_BYTES = A_BYTES + B_BYTES;
    static constexpr int ROW_BYTES = MPW * MCU_W * CH;  // one staged output row of a warp
    static constexpr int W_BYTES = UPS ? 16 * kWStride * 16 : 0;
    static constexpr int SMEM = kWarps * WARP_BYTES + W_BYTES + 3 * 128;
    static_assert(ROW_BYTES % 16 == 0 && ROW_BYTES * MCU_H <= A_BYTES, "staging must fit the coefficient tile");
};

// reference flat index u*8+v -> zig-zag index (zagzig, jpeg_decoder.py:1672-1681, inverted)
__constant__ uint8_t c_nat_zz[64] = {0, 2, 3, 9, 10, 20, 21, 35, 1, 4, 8, 11, 19, 22, 34, 36, 5, 7, 12, 18, 23, 33,
                                     37, 48, 6, 13, 17, 24, 32, 38, 47, 49, 14, 16, 25, 31, 39, 46, 50, 57, 15, 26,
                                     30, 40, 45, 51, 56, 58, 27, 29, 41, 44, 52, 55, 59, 62, 28, 42, 43, 53, 54, 60,
                                     61, 63};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

template <class L>
struct Tiles {
    unsigned char* a;   // this warp's coefficients (32 x 128 B, swizzled) / RGB staging
    unsigned char* b;   // this warp's samples
    const float4* w;    // interpolation weights [b * kWStride + a]
    const int16_t* qt;  // [3][64]
    __device__ __forceinline__ unsigned char* coef_chunk(int blk, int c) const { return a + blk * 128 + ((c ^ (blk & 7)) << 4); }
    // luma block ys of MCU m, row y: 8 int16
    __device__ __forceinline__ unsigned char* yrow(int m, int ys, int y) const {
        return b + m * L::MCU_B + ys * 128 + ((y ^ ((m + ys) & 7)) << 4);
    }
    // chroma block k (0 = Cb, 1 = Cr) of MCU m, row y: 8 floats, contiguous; rows are XOR-swizzled in steps of 32
    // bytes so that the lanes of phase A (one block each, same row at the same time) spread over the banks
    __device__ __forceinline__ float* crow(int m, int k, int y) const {
        return reinterpret_cast<float*>(b + m * L::MCU_B + L::NY * 128 + k * 256 + ((y * 32) ^ (((m + k) & 7) * 32)));
    }
    // 16-byte chunk c of that block (row y = chunks 2y, 2y+1): 4 floats
    __device__ __forceinline__ float* cchunk(int m, int k, int c) const { return crow(m, k, c >> 1) + (c & 1) * 4; }
};

// ---- exact recompute of one block by a whole warp (InverseDCT.__call__, :1561-1573) ---------------
// Lane l owns output samples s = l and l + 32 (s = x*8 + y).  Accumulator j = v collects the products
// of u = 0..7 in order, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)): numpy's pairwise sum of the 64
// products in C order [u][v]; zero coefficients only add +-0.0 and are skipped.
template <class L>
__device__ __noinline__ void recompute_block_exact(const Tiles<L>& t, int blk, const double* __restrict__ tabT, int lane) {
    const int m = blk / L::BPM, slot = blk - m * L::BPM;
    const int comp = slot < L::NY ? 0 : slot - L::NY + 1;
    const int16_t* qt = t.qt + comp * 64;
    // natural-order non-zero masks: lane l looks at n = l and n = l + 32
    int k0 = c_nat_zz[lane], k1 = c_nat_zz[lane + 32];
    int c0 = *reinterpret_cast<const int16_t*>(t.coef_chunk(blk, k0 >> 3) + ((k0 & 7) << 1));
    int c1 = *reinterpret_cast<const int16_t*>(t.coef_chunk(blk, k1 >> 3) + ((k1 & 7) << 1));
    int p0 = (int16_t)(c0 * (int)qt[k0]), p1 = (int16_t)(c1 * (int)qt[k1]);  // int16 product wraps (:869)
    const unsigned nz_lo = __ballot_sync(0xffffffffu, p0 != 0), nz_hi = __ballot_sync(0xffffffffu, p1 != 0);
    double r0[8], r1[8];
#pragma unroll
    for (int v = 0; v < 8; v++) r0[v] = r1[v] = 0.0;
    // rolled over u (this path runs for about one block in a hundred: compact code matters more than its speed,
    // the kernel's hot code has to stay inside the instruction cache)
#pragma unroll 1
    for (int u = 0; u < 8; u++) {
        const unsigned bits = (((u < 4) ? nz_lo : nz_hi) >> ((u & 3) * 8)) & 0xFFu;  // warp-uniform
        if (!bits) continue;
        const int psel = (u < 4) ? p0 : p1;
        const double* tu = tabT + u * 8 * 64;
#pragma unroll
        for (int v = 0; v < 8; v++) {
            if (bits & (1u << v)) {
                const int prod = __shfl_sync(0xffffffffu, psel, ((u & 3) << 3) + v);
                const double p = (double)prod;
                const double* tt = tu + v * 64;
                r0[v] = __dadd_rn(r0[v], __dmul_rn(p, tt[lane]));
                r1[v] = __dadd_rn(r1[v], __dmul_rn(p, tt[lane + 32]));
            }
        }
    }
    double s0 = __dadd_rn(__dadd_rn(__dadd_rn(r0[0], r0[1]), __dadd_rn(r0[2], r0[3])),
                          __dadd_rn(__dadd_rn(r0[4], r0[5]), __dadd_rn(r0[6], r0[7])));
    double s1 = __dadd_rn(__dadd_rn(__dadd_rn(r1[0], r1[1]), __dadd_rn(r1[2], r1[3])),
                          __dadd_rn(__dadd_rn(r1[4], r1[5]), __dadd_rn(r1[6], r1[7])));
    const int x0 = lane >> 3, y0 = lane & 7, x1 = x0 + 4;
    const int v0 = (int16_t)(__double2int_rn(s0)) + 128, v1 = (int16_t)(__double2int_rn(s1)) + 128;
    if (comp == 0) {
        int16_t* row = reinterpret_cast<int16_t*>(t.yrow(m, slot, y0));
        row[x0] = (int16_t)v0;
        row[x1] = (int16_t)v1;
    } else {
        t.cchunk(m, comp - 1, 2 * y0 + (x0 >> 2))[x0 & 3] = (float)v0;
        t.cchunk(m, comp - 1, 2 * y0 + (x1 >> 2))[x1 & 3] = (float)v1;
    }
}

// exact colour conversion of one pixel, fp64, evaluation order of :1693-1695, clip (:1698), round (:1700)
__device__ __noinline__ uint32_t ycc_to_rgb_exact_packed(int Yi, float Cbf, float Crf) {
    double Y = (double)Yi, cb = __dsub_rn((double)Cbf, 128.0), cr = __dsub_rn((double)Crf, 128.0);
    double r = __dadd_rn(Y, __dmul_rn(1.402, cr));
    double g = __dsub_rn(__dsub_rn(Y, __dmul_rn(0.34414, cb)), __dmul_rn(0.71414, cr));
    double b = __dadd_rn(Y, __dmul_rn(1.772, cb));
    r = fmin(fmax(r, 0.0), 255.0);
    g = fmin(fmax(g, 0.0), 255.0);
    b = fmin(fmax(b, 0.0), 255.0);
    return (uint32_t)__double2int_rn(r) | ((uint32_t)__double2int_rn(g) << 8) | ((uint32_t)__double2int_rn(b) << 16);
}

// Interpolation weight table of a layout, built at COMPILE time (it only depends on the sampling factors) and
// placed in global memory: the kernel prologue copies 4 KB instead of recomputing 256 entries per CTA.
// Entry a' of row b: a' < 8 -> output column a'; a' >= 8 (right half, HMAX == 2) -> column 23 - a', i.e. the right
// half stored right-to-left with the left/right taps swapped (see pixel_run).
template <int HMAX, int VMAX>
struct WeightTable {
    float4 v[256];
    constexpr WeightTable() : v{} {
        for (int i = 0; i < 256; i++) {
            const int b = i >> 4, ap = i & 15;
            const bool mirror = (HMAX == 2) && ap >= 8;
            const int a = mirror ? 23 - ap : ap;
            int ii = a & 7, s = 0, jj = b & 7, tt = 0;
            if (HMAX == 2) bj::up_cell(a, ii, s);
            if (VMAX == 2) bj::up_cell(b, jj, tt);
            int w00 = 0, w10 = 0, w01 = 0, w11 = 0;
            bj::up_weights_2d(ii, jj, s, tt, w00, w10, w01, w11);
            v[i].x = (float)(mirror ? w10 : w00);
            v[i].y = (float)(mirror ? w00 : w10);
            v[i].z = (float)(mirror ? w11 : w01);
            v[i].w = (float)(mirror ? w01 : w11);
        }
    }
};
template <int HMAX, int VMAX>
__device__ const WeightTable<HMAX, VMAX> g_weight_table{};

template <int A> struct Cell { static constexpr int i = (A == 15) ? 6 : (7 * A) / 15; };

// Exact colour conversion of a whole 8-pixel run, straight from the sample tile: the out-of-line, compact
// (rolled) path behind pixel_run's tie / range guards.  Runs for a tiny fraction of the runs; what matters is
// that it adds little code next to the hot path.
template <class L>
__device__ __noinline__ void pixel_run_exact(const Tiles<L>& t, int m, int r, int hx) {
    const int ys = (r >> 3) * L::HMAX + hx, yy = r & 7;
    const int16_t* yrow = reinterpret_cast<const int16_t*>(t.yrow(m, ys, yy));
    unsigned char* stage = t.a + r * L::ROW_BYTES + (m * L::MCU_W + 8 * hx) * L::CH;
    const int j = (L::VMAX == 2) ? ((r == 15) ? 6 : (7 * r) / 15) : yy;
    const int j2 = j < 7 ? j + 1 : 7;
#pragma unroll 1
    for (int p = 0; p < 8; p++) {
        float c[2];
        if (!L::UPS) {
            c[0] = t.cchunk(m, 0, 2 * yy + (p >> 2))[p & 3];
            c[1] = t.cchunk(m, 1, 2 * yy + (p >> 2))[p & 3];
        } else {
            const int a = 8 * hx + p;
            const int i = (L::HMAX == 2) ? ((a == 15) ? 6 : (7 * a) / 15) : p;
            const int i2 = i < 7 ? i + 1 : 7;
            float4 w = t.w[r * kWStride + a];
            if (L::HMAX == 2 && hx) {  // right half: stored right-to-left with the taps swapped (see pixel_run)
                const float4 e = t.w[r * kWStride + 23 - a];
                w = make_float4(e.y, e.x, e.w, e.z);
            }
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const float p00 = t.cchunk(m, k, 2 * j + (i >> 2))[i & 3], p10 = t.cchunk(m, k, 2 * j + (i2 >> 2))[i2 & 3];
                const float p01 = t.cchunk(m, k, 2 * j2 + (i >> 2))[i & 3], p11 = t.cchunk(m, k, 2 * j2 + (i2 >> 2))[i2 & 3];
                const float n = fmaf(w.w, p11, fmaf(w.z, p01, fmaf(w.y, p10, w.x * p00)));  // integers: exact in any order
                c[k] = fmaf(n, 1.0f / 15.0f, BJ_MAGIC) - BJ_MAGIC;
            }
        }
        const uint32_t rgb = ycc_to_rgb_exact_packed((int)yrow[p], c[0], c[1]);
        stage[3 * p] = (unsigned char)rgb;
        stage[3 * p + 1] = (unsigned char)(rgb >> 8);
        stage[3 * p + 2] = (unsigned char)(rgb >> 16);
    }
}

// One 8-pixel run: pixel row r (0..MCU_H-1) of MCU m (warp-local), horizontal half hx.
// `wide` (warp-level knowledge from phase A): some sample of this MCU may lie outside the range in which the
// fp32 colour offsets are proven exact (|Cb-128| >= 125: B can tie; |Cr-128| >= 250; |Y| huge) -> exact path.
// For layouts with two luma blocks per MCU row (HMAX == 2) the half `hx` is a RUN-TIME value, so that one lane
// can take one run and the (MCU, row, half) triples fill the warp exactly (4:2:0: 160 runs = 5 x 32 lanes; with a
// lane per (MCU, row) doing both halves in turn it was 80 pairs on 96 lane slots).  One code body serves both
// halves because the right half is the mirror image of the left one: output column a = 15 - a' reads source
// cells 6 - i(a'), so the right half walks its pixels right-to-left over the mirrored chroma columns with the
// left half's compile-time tap indices; the weight table holds the right half's entries mirrored and with the
// left/right taps swapped, and luma pairs / RGB pairs are flipped with one byte-permute each.
// ww: the lane's eight interpolation weight vectors (row r, half hx); loaded once per tile by the caller -- a
// lane always works on the same (row, half), only the MCU changes from run to run.
template <class L>
__device__ __forceinline__ void pixel_run(const Tiles<L>& t, int m, int r, int hx, const float4 (&ww)[8], bool wide,
                                          uint32_t* stats) {
    const int ys = (r >> 3) * L::HMAX + hx, yy = r & 7;
    const uint4 yv = *reinterpret_cast<const uint4*>(t.yrow(m, ys, yy));
    const uint32_t flip = (L::HMAX == 2 && hx) ? 0x5476u : 0x3210u;  // byte-permute selector: second operand, halves swapped
    uint32_t yw[4] = {yv.x, yv.y, yv.z, yv.w};
    if (L::HMAX == 2) {
        const uint32_t y0 = __byte_perm(yv.x, yv.w, flip), y1 = __byte_perm(yv.y, yv.z, flip);
        const uint32_t y2 = __byte_perm(yv.z, yv.y, flip), y3 = __byte_perm(yv.w, yv.x, flip);
        yw[0] = y0; yw[1] = y1; yw[2] = y2; yw[3] = y3;
    }
    unsigned char* stage = t.a + r * L::ROW_BYTES + (m * L::MCU_W + 8 * hx) * L::CH;
    if (L::NCOMP == 1) {
        int Y[8];
#pragma unroll
        for (int p = 0; p < 8; p++) Y[p] = (int)(int16_t)(yw[p >> 1] >> (16 * (p & 1)));
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int p = 0; p < 4; p++) {
            lo |= (uint32_t)min(max(Y[p], 0), 255) << (8 * p);  // (:1385-1386)
            hi |= (uint32_t)min(max(Y[p + 4], 0), 255) << (8 * p);
        }
        *reinterpret_cast<uint2*>(stage) = make_uint2(lo, hi);
        return;
    }
    // chroma minus 128 for the 8 pixels
    float cbm[8], crm[8];
    if (!L::UPS) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
            float4 lo = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * yy));
            float4 hi = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * yy + 1));
            float* o = k ? crm : cbm;
            o[0] = lo.x - 128.f; o[1] = lo.y - 128.f; o[2] = lo.z - 128.f; o[3] = lo.w - 128.f;
            o[4] = hi.x - 128.f; o[5] = hi.y - 128.f; o[6] = hi.z - 128.f; o[7] = hi.w - 128.f;
        }
    } else {
        int j = (L::VMAX == 2) ? ((r == 15) ? 6 : (7 * r) / 15) : r;
        int j2 = j < 7 ? j + 1 : 7;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            float* o = k ? crm : cbm;
            if (L::HMAX == 2) {
                // window of five source columns: 0..4 for the left half, 7..3 (mirrored) for the right half
                float p0[5], p1[5];
                {
                    const float* r0 = t.crow(m, k, j);
                    const float* r1 = t.crow(m, k, j2);
                    const float4 a = *reinterpret_cast<const float4*>(r0 + 4 * hx);
                    const float4 b = *reinterpret_cast<const float4*>(r1 + 4 * hx);
                    p0[4] = r0[hx ? 3 : 4];   // the fifth column of the window: 4 (left half) or 3 (mirrored right half)
                    p1[4] = r1[hx ? 3 : 4];
                    p0[0] = hx ? a.w : a.x; p0[1] = hx ? a.z : a.y; p0[2] = hx ? a.y : a.z; p0[3] = hx ? a.x : a.w;
                    p1[0] = hx ? b.w : b.x; p1[1] = hx ? b.z : b.y; p1[2] = hx ? b.y : b.z; p1[3] = hx ? b.x : b.w;
                }
#define BJ_PIX(P)                                                                                          \
    {                                                                                                      \
        constexpr int i = Cell<P>::i;                                                                      \
        float n = fmaf(ww[P].w, p1[i + 1], fmaf(ww[P].z, p1[i], fmaf(ww[P].y, p0[i + 1], ww[P].x * p0[i]))); \
        /* N/15 rounded (never a tie), minus 128: both subtractions folded into one exact fp32 add */      \
        o[P] = fmaf(n, 1.0f / 15.0f, BJ_MAGIC) - (BJ_MAGIC + 128.0f);                                      \
    }
                BJ_PIX(0) BJ_PIX(1) BJ_PIX(2) BJ_PIX(3) BJ_PIX(4) BJ_PIX(5) BJ_PIX(6) BJ_PIX(7)
#undef BJ_PIX
            } else {
                float p0[8], p1[8];
                {
                    float4 a0 = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * j));
                    float4 a1 = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * j + 1));
                    float4 b0 = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * j2));
                    float4 b1 = *reinterpret_cast<const float4*>(t.cchunk(m, k, 2 * j2 + 1));
                    p0[0] = a0.x; p0[1] = a0.y; p0[2] = a0.z; p0[3] = a0.w; p0[4] = a1.x; p0[5] = a1.y; p0[6] = a1.z; p0[7] = a1.w;
                    p1[0] = b0.x; p1[1] = b0.y; p1[2] = b0.z; p1[3] = b0.w; p1[4] = b1.x; p1[5] = b1.y; p1[6] = b1.z; p1[7] = b1.w;
                }
#define BJ_PIX(P)                                                                                          \
    {                                                                                                      \
        constexpr int i = P;                                                                               \
        constexpr int i2 = i < 7 ? i + 1 : 7;                                                              \
        float n = fmaf(ww[P].w, p1[i2], fmaf(ww[P].z, p1[i], fmaf(ww[P].y, p0[i2], ww[P].x * p0[i])));     \
        o[P] = fmaf(n, 1.0f / 15.0f, BJ_MAGIC) - (BJ_MAGIC + 128.0f);                                      \
    }
                BJ_PIX(0) BJ_PIX(1) BJ_PIX(2) BJ_PIX(3) BJ_PIX(4) BJ_PIX(5) BJ_PIX(6) BJ_PIX(7)
#undef BJ_PIX
            }
        }
    }
    // colour: offsets from chroma in fp32, integer add + clamp; see bj_pixel_math.cuh for the tie rules
    // Two pixels per instruction: the low halves of the magic-biased offsets are round(offset) as int16 (the
    // bias 0x4B400000 has a zero low half), luma is already a packed int16 pair, and one DPX
    // add-min-relu (VIADDMNMX.S16x2) gives clamp(Y + round(offset), 0, 255) for both.  |Y + offset| stays far
    // below 2^15 because `wide` MCUs (huge samples) never get here.
    uint32_t rg[4], bb[4];  // per pixel pair: bytes (R0, G0, R1, G1) and halves (B0, B1)
    float dgmax = 0.f;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        float wr[2], wg[2], wb[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const float cb = cbm[2 * k + h], cr = crm[2 * k + h];
            // offset + 1.5 * 2^23 in one rounding: the low mantissa bits are round-to-nearest(offset)
            wr[h] = fmaf(1.402f, cr, BJ_MAGIC);
            wb[h] = fmaf(1.772f, cb, BJ_MAGIC);
            const float gC = fmaf(-0.71414f, cr, -0.34414f * cb);
            wg[h] = gC + BJ_MAGIC;
            dgmax = fmaxf(dgmax, fabsf(gC - (wg[h] - BJ_MAGIC)));
        }
        const uint32_t RR = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wr[0]), __float_as_uint(wr[1]), 0x5410), yw[k], 0x00FF00FFu);
        const uint32_t GG = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wg[0]), __float_as_uint(wg[1]), 0x5410), yw[k], 0x00FF00FFu);
        bb[k] = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wb[0]), __float_as_uint(wb[1]), 0x5410), yw[k], 0x00FF00FFu);
        rg[k] = __byte_perm(RR, GG, 0x6240);
    }
    if (wide || dgmax > 0.5f - BJ_G_ERR) {
        pixel_run_exact<L>(t, m, r, hx);
        if (stats) atomicAdd(&stats[1], 8u);
        return;
    }
    if (L::HMAX == 2) {  // back to left-to-right order
        const uint32_t r0 = __byte_perm(rg[0], rg[3], flip), r1 = __byte_perm(rg[1], rg[2], flip);
        const uint32_t r2 = __byte_perm(rg[2], rg[1], flip), r3 = __byte_perm(rg[3], rg[0], flip);
        const uint32_t b0 = __byte_perm(bb[0], bb[3], flip), b1 = __byte_perm(bb[1], bb[2], flip);
        const uint32_t b2 = __byte_perm(bb[2], bb[1], flip), b3 = __byte_perm(bb[3], bb[0], flip);
        rg[0] = r0; rg[1] = r1; rg[2] = r2; rg[3] = r3;
        bb[0] = b0; bb[1] = b1; bb[2] = b2; bb[3] = b3;
    }
    // 8 pixels x 3 bytes = 6 words: R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3 | ...
    uint32_t o[6];
#pragma unroll
    for (int q = 0; q < 2; q++) {
        const uint32_t t0 = rg[2 * q], t1 = rg[2 * q + 1], b0 = bb[2 * q], b1 = bb[2 * q + 1];
        o[3 * q] = __byte_perm(t0, b0, 0x2410);                             // R0 G0 B0 R1
        o[3 * q + 1] = __byte_perm(__byte_perm(t0, b0, 0x0063), t1, 0x5410);  // G1 B1 | R2 G2
        o[3 * q + 2] = __byte_perm(t1, b1, 0x6324);                         // B2 R3 G3 B3
    }
    uint2* s2 = reinterpret_cast<uint2*>(stage);
    s2[0] = make_uint2(o[0], o[1]);
    s2[1] = make_uint2(o[2], o[3]);
    s2[2] = make_uint2(o[4], o[5]);
}

// CROP: one CTA per strip of a bj_crop_job's MCU window (jobs of this layout at scale 1), storing only the box.
template <int HMAX, int VMAX, int NCOMP, int LAYOUT, bool CROP>
__global__ void __launch_bounds__(kThreads, 3)
bj_pixels_fast_kernel(const bj_image* __restrict__ images, const int16_t* __restrict__ coef,
                      const int16_t* __restrict__ qtabs, const double* __restrict__ tabT,
                      uint8_t* __restrict__ out, uint32_t* __restrict__ stats, const bj_crop_job* __restrict__ jobs) {
    using L = Lay<HMAX, VMAX, NCOMP>;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ bj_image im;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // The descriptor goes to shared memory for later use (visible after the barrier below); what the prologue needs
    // is read straight from global memory by every thread (one broadcast transaction each), which saves a barrier
    // and a shared-memory round trip in front of the tile request.
    bj_crop_job jb{};
    if constexpr (CROP) jb = jobs[blockIdx.y];
    const bj_image* const gi = &images[CROP ? jb.image : blockIdx.y];
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(gi);
        if (tid < (int)(sizeof(bj_image) / 4)) reinterpret_cast<uint32_t*>(&im)[tid] = src[tid];
    }
    if ((int)__ldg(&gi->layout) != LAYOUT) return;
    const int g_mcus_x = (int)__ldg(&gi->mcus_x);
    int my, m0, M;
    if constexpr (CROP) {
        if (jb.log2_scale != 0) return;
        int sm0, sM;
        if (!bj::crop_strip(jb, L::MCU_W, L::MCU_H, L::STRIP, blockIdx.x, my, sm0, sM)) return;
        m0 = sm0 + warp * L::MPW;
        M = min(L::MPW, sm0 + sM - m0);
    } else {
        const int g_mcus_y = (int)__ldg(&gi->mcus_y);
        const int strips_per_row = (g_mcus_x + L::STRIP - 1) / L::STRIP;
        if ((int)blockIdx.x >= g_mcus_y * strips_per_row) return;
        my = blockIdx.x / strips_per_row;
        m0 = (blockIdx.x - my * strips_per_row) * L::STRIP + warp * L::MPW;
        M = min(L::MPW, g_mcus_x - m0);
    }

    // ---- this warp's tile: requested first, so that the table set-up below runs while it is in flight -------
    float4* wtab = reinterpret_cast<float4*>(smem + kWarps * L::WARP_BYTES);
    int16_t* qt = reinterpret_cast<int16_t*>(smem + kWarps * L::WARP_BYTES + L::W_BYTES);
    Tiles<L> t;
    t.a = smem + warp * L::WARP_BYTES;
    t.b = t.a + L::A_BYTES;
    t.w = wtab;
    t.qt = qt;
    const int nblk = M > 0 ? M * L::BPM : 0;
    if (M > 0) {
        const uint4* g = reinterpret_cast<const uint4*>(coef + ((int64_t)__ldg(&gi->coef_block0) + ((int64_t)my * g_mcus_x + m0) * L::BPM) * 64);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            int i = lane + 32 * k;  // 16-byte chunk index inside the warp's tile
            if (i < nblk * 8) cp_async16(t.coef_chunk(i >> 3, i & 7), g + i);
        }
    }
    // ---- CTA-wide tables (the only CTA barrier of the kernel) ---------------------------------------
    for (int i = tid; i < NCOMP * 64; i += kThreads) qt[i] = qtabs[(size_t)__ldg(&gi->qtab[i >> 6]) * 64 + (i & 63)];
    if (L::UPS) {
        for (int i = tid; i < 256; i += kThreads) wtab[(i >> 4) * kWStride + (i & 15)] = g_weight_table<HMAX, VMAX>.v[i];
    }
    cp_async_wait_all();
    __syncthreads();
    if (M <= 0) return;

    // ---- phase A: one lane per block ---------------------------------------------------------------
    unsigned wide_mask;  // blocks whose samples may leave the range the fast colour path is proven for
    {
        const int blk = lane;
        const int m = blk / L::BPM, slot = blk - m * L::BPM;
        bool flagged = false, wide_blk = false;
        if (blk < nblk) {
            const int comp = slot < L::NY ? 0 : slot - L::NY + 1;
            float f[64];
            float S = 0.f;
#pragma unroll
            for (int c = 0; c < 8; c++) {
                uint4 v = *reinterpret_cast<const uint4*>(t.coef_chunk(blk, c));
                uint4 q = *reinterpret_cast<const uint4*>(t.qt + comp * 64 + c * 8);
                const uint32_t vw[4] = {v.x, v.y, v.z, v.w}, qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    int cf = (int16_t)(vw[e >> 1] >> (16 * (e & 1)));
                    int qq = (int16_t)(qw[e >> 1] >> (16 * (e & 1)));
                    float x = (float)(int16_t)(cf * qq);  // int16 * int16 -> int16 wraps (:869, :1348)
                    constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
                    f[zz[c * 8 + e]] = x;
                    if (c * 8 + e) S += fabsf(x);
                }
            }
            const float dc_abs = fabsf(f[0]);
            const float T = fmaf(S, BJ_IDCT_ERR_REL, fmaf(dc_abs, BJ_IDCT_ERR_DC, BJ_IDCT_ERR_ABS));
            bj::idct8x8_fast(f);
            // round + level shift in one add: the low mantissa bits of v + (1.5 * 2^23 + 128) are rint(v) + 128
            constexpr float kMagicShift = BJ_MAGIC + 128.0f;
            float maxd = 0.f;
#pragma unroll
            for (int y = 0; y < 8; y++) {
                float w[8];
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    float v = f[y * 8 + x];
                    w[x] = v + kMagicShift;
                    maxd = fmaxf(maxd, fabsf(v - (w[x] - kMagicShift)));
                }
                if (comp == 0) {
                    // int16 pairs = the low halves of the biased floats (the bias has a zero low half)
                    *reinterpret_cast<uint4*>(t.yrow(m, slot, y)) =
                        make_uint4(__byte_perm(__float_as_uint(w[0]), __float_as_uint(w[1]), 0x5410),
                                   __byte_perm(__float_as_uint(w[2]), __float_as_uint(w[3]), 0x5410),
                                   __byte_perm(__float_as_uint(w[4]), __float_as_uint(w[5]), 0x5410),
                                   __byte_perm(__float_as_uint(w[6]), __float_as_uint(w[7]), 0x5410));
                } else {
                    // rint(v) + 128 = w - MAGIC, exact
                    float4* row = reinterpret_cast<float4*>(t.crow(m, comp - 1, y));
                    row[0] = make_float4(w[0] - BJ_MAGIC, w[1] - BJ_MAGIC, w[2] - BJ_MAGIC, w[3] - BJ_MAGIC);
                    row[1] = make_float4(w[4] - BJ_MAGIC, w[5] - BJ_MAGIC, w[6] - BJ_MAGIC, w[7] - BJ_MAGIC);
                }
            }
            flagged = maxd > 0.5f - T;
            // |sample - 128| <= |DC| / 8 + sum|AC| / 4 + 1/2 (every basis value is at most 1/8 resp. 1/4)
            const float bound = fmaf(0.25f, S, fmaf(0.125f, dc_abs, 0.5f));
            wide_blk = bound >= (comp == 0 ? 30000.0f : comp == 1 ? 125.0f : BJ_CHROMA_GUARD);
        }
        wide_mask = __ballot_sync(0xffffffffu, wide_blk);
        unsigned mask = __ballot_sync(0xffffffffu, flagged);
        __syncwarp();
        if (mask) {
            if (stats && lane == 0) atomicAdd(&stats[0], (uint32_t)__popc(mask));
            while (mask) {
                int src = __ffs(mask) - 1;
                mask &= mask - 1;
                recompute_block_exact<L>(t, src, tabT, lane);
            }
            __syncwarp();
        }
    }

    // ---- phase B: lanes = (MCU, pixel row) pairs of this warp -----------------------------------------
    const int x0 = m0 * L::MCU_W, y0 = my * L::MCU_H;
    const int cols = min(M * L::MCU_W, (int)im.width - x0);
    const int rows = min(L::MCU_H, (int)im.height - y0);
    const int nunits = M * L::MCU_H * L::HMAX;  // 8-pixel runs: (MCU, half, row)
    {
        // 32 is a multiple of MCU_H * HMAX: lane -> (row, half) is the same in every pass, only the MCU advances
        static_assert(32 % (L::MCU_H * L::HMAX) == 0, "lane -> (row, half) must not depend on the pass");
        const int r = lane % L::MCU_H, hx = (lane / L::MCU_H) % L::HMAX;
        float4 ww[8];
#pragma unroll
        for (int p = 0; p < 8; p++) ww[p] = L::UPS ? t.w[r * kWStride + 8 * hx + p] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
        for (int u0 = 0; u0 < nunits; u0 += 32) {
            const int u = u0 + lane;
            const int m = u / (L::MCU_H * L::HMAX);
            bool row_ok = r < rows;
            if constexpr (CROP) row_ok = row_ok && y0 + r >= (int)jb.y0 && y0 + r < (int)jb.y1;   // rows outside the box are not stored
            if (u < nunits && row_ok) {
                const bool wide = ((wide_mask >> (m * L::BPM)) & ((1u << L::BPM) - 1u)) != 0u;
                pixel_run<L>(t, m, r, hx, ww, wide, stats);
            }
        }
    }
    __syncwarp();

    // ---- store this warp's rows -------------------------------------------------------------------------
    if constexpr (CROP) {
        int sx, sy, w, h;
        uint8_t* g;
        if (bj::crop_part(jb, x0, y0, cols, rows, L::CH, out, sx, sy, w, h, g))
            bj::crop_store(g, jb.out_pitch, t.a + sy * L::ROW_BYTES, L::ROW_BYTES, sx * L::CH, w * L::CH, h, lane, 32);
        return;
    }
    uint8_t* gout = out + (int64_t)im.out_offset + (int64_t)y0 * im.out_pitch + (int64_t)x0 * L::CH;
    const int nbytes = cols * L::CH;
    const bool aligned = ((reinterpret_cast<uintptr_t>(gout) & 15) == 0) && ((im.out_pitch & 15) == 0);
    if (aligned && nbytes == L::ROW_BYTES) {
        constexpr int NVEC = L::ROW_BYTES / 16;
        for (int i = lane; i < rows * NVEC; i += 32) {
            const int r = i / NVEC, v = i - r * NVEC;
            uint4 val = *reinterpret_cast<const uint4*>(t.a + r * L::ROW_BYTES + (v << 4));
            __stcs(reinterpret_cast<uint4*>(gout + (int64_t)r * im.out_pitch + (v << 4)), val);
        }
    } else if (aligned) {
        const int nvec = nbytes >> 4, tail = nbytes & 15;
#pragma unroll 1
        for (int r = 0; r < rows; r++) {
#pragma unroll 1
            for (int v = lane; v < nvec; v += 32)
                __stcs(reinterpret_cast<uint4*>(gout + (int64_t)r * im.out_pitch + (v << 4)),
                       *reinterpret_cast<const uint4*>(t.a + r * L::ROW_BYTES + (v << 4)));
            if (lane < tail) gout[(int64_t)r * im.out_pitch + (nvec << 4) + lane] = t.a[r * L::ROW_BYTES + (nvec << 4) + lane];
        }
    } else {
#pragma unroll 1
        for (int r = 0; r < rows; r++)
#pragma unroll 1
            for (int b = lane; b < nbytes; b += 32) gout[(int64_t)r * im.out_pitch + b] = t.a[r * L::ROW_BYTES + b];
    }
}

// n_images: grid.y, the images (jobs == nullptr) or the crop jobs
template <int HMAX, int VMAX, int NCOMP, int LAYOUT, bool CROP = false>
cudaError_t launch(const bj_image* images, int n_images, int max_strips, const int16_t* coef, const int16_t* qtabs,
                   const double* tabT, uint8_t* out, uint32_t* stats, cudaStream_t st, const bj_crop_job* jobs = nullptr) {
    using L = Lay<HMAX, VMAX, NCOMP>;
    auto k = bj_pixels_fast_kernel<HMAX, VMAX, NCOMP, LAYOUT, CROP>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, L::SMEM);
    if (e != cudaSuccess) return e;
    k<<<dim3((unsigned)max_strips, (unsigned)n_images), kThreads, L::SMEM, st>>>(images, coef, qtabs, tabT, out, stats, jobs);
    return cudaGetLastError();
}

}  // namespace

// MCUs per CTA of the specialised kernel for a layout (0 for the generic layout); the host sizes the
// grid with it (strips_per_row = ceil(mcus_x / strip)).
extern "C" int bj_pixels_420_strip(void);
extern "C" int bj_pixels_fast_strip(int layout) {
    switch (layout) {
        case BJ_LAYOUT_420: return bj_pixels_420_strip();  // bj_pixels_mma.cu
        case BJ_LAYOUT_422: return Lay<2, 1, 3>::STRIP;
        case BJ_LAYOUT_440: return Lay<1, 2, 3>::STRIP;
        case BJ_LAYOUT_444: return Lay<1, 1, 3>::STRIP;
        case BJ_LAYOUT_GRAY: return Lay<1, 1, 1>::STRIP;
        default: return 0;
    }
}

// Launch the specialised kernels for every layout present in layout_mask (bits BJ_LAYOUT_420..GRAY).
extern "C" bj_status bj_pixels_fast_launch(const bj_image* images, int n_images, int max_strips, const int16_t* coef,
                                           const int16_t* qtabs, const double* tabT, uint8_t* out, uint32_t layout_mask,
                                           uint32_t* stats, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_420)))
        e = launch<2, 2, 3, BJ_LAYOUT_420>(images, n_images, max_strips, coef, qtabs, tabT, out, stats, st);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_422)))
        e = launch<2, 1, 3, BJ_LAYOUT_422>(images, n_images, max_strips, coef, qtabs, tabT, out, stats, st);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_440)))
        e = launch<1, 2, 3, BJ_LAYOUT_440>(images, n_images, max_strips, coef, qtabs, tabT, out, stats, st);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_444)))
        e = launch<1, 1, 3, BJ_LAYOUT_444>(images, n_images, max_strips, coef, qtabs, tabT, out, stats, st);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_GRAY)))
        e = launch<1, 1, 1, BJ_LAYOUT_GRAY>(images, n_images, max_strips, coef, qtabs, tabT, out, stats, st);
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels/fast");
    return BJ_OK;
}

// Crop jobs (bj_pixels_crop) of the specialised layouts in layout_mask other than 4:2:0 (bj_pixels_mma.cu).
extern "C" bj_status bj_pixels_fast_crop_launch(const bj_image* images, const bj_crop_job* jobs, int n_jobs,
                                                int max_strips, const int16_t* coef, const int16_t* qtabs,
                                                const double* tabT, uint8_t* out, uint32_t layout_mask,
                                                uint32_t* stats, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_422)))
        e = launch<2, 1, 3, BJ_LAYOUT_422, true>(images, n_jobs, max_strips, coef, qtabs, tabT, out, stats, st, jobs);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_440)))
        e = launch<1, 2, 3, BJ_LAYOUT_440, true>(images, n_jobs, max_strips, coef, qtabs, tabT, out, stats, st, jobs);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_444)))
        e = launch<1, 1, 3, BJ_LAYOUT_444, true>(images, n_jobs, max_strips, coef, qtabs, tabT, out, stats, st, jobs);
    if (e == cudaSuccess && (layout_mask & (1u << BJ_LAYOUT_GRAY)))
        e = launch<1, 1, 1, BJ_LAYOUT_GRAY, true>(images, n_jobs, max_strips, coef, qtabs, tabT, out, stats, st, jobs);
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_crop/fast");
    return BJ_OK;
}
