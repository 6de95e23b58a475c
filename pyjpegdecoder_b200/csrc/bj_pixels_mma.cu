// bj_pixels_mma.cu -- fused pixel kernel for 4:2:0 images (sm_100a): de-zigzag + dequantise + 8x8 IDCT +
// level shift + chroma upsampling + YCbCr->RGB + clamp + crop, coefficients in, RGB bytes out.
//
// Same arithmetic contract as the other pixel kernels (bit-exact with the reference's fp64 path,
// jpeg_decoder.py:869-891, :1306-1366, :1368-1386, :1561-1573, :1588-1626, :1683-1700); what is new is how the
// work is mapped onto Blackwell:
//   * one CTA = 32 MCUs (192 blocks = 24 KB of coefficients, 16 x 1536 B of RGB).  The coefficient tile arrives
//     with ONE 2-D TMA load (cp.async.bulk.tensor, SWIZZLE_128B: the hardware applies the 16-byte-chunk XOR
//     swizzle that makes the one-lane-per-block reads conflict-free) on an mbarrier; the RGB rows leave with
//     cp.async.bulk shared->global.  No per-thread address arithmetic for the bulk data.
//   * phase A, one lane per block: warps 0-3 take the 128 luma blocks, warps 4-5 the 64 chroma blocks, so each
//     warp runs ONE code path: luma dense, chroma the 4x4 low-frequency variant when (as nearly always) every
//     chroma block of the warp is confined to that corner.  The separable IDCT is written for the packed-fp32
//     pipe (FFMA2 / FADD2 / FMUL2: two columns, then two rows, per instruction); rounding + level shift is one
//     packed add of 1.5*2^23 + 128, the tie test two more packed ops and one 3-input FMNMX3.  Samples within the
//     fp32 error bound of a rounding tie are recomputed exactly (fp64, numpy's pairwise order), as before.
//   * phase B: the reference's 3-tap Delaunay interpolation of an 8x8 chroma block to 16x16 is a linear map with
//     small integer weights -> it runs on the tensor cores (mma.sync m16n8k16, f16 x f16 -> f32: weights 0..15 and
//     samples are exact in f16, the sums stay below 2^17: exact in any accumulation order).  One MMA pair
//     gives every lane the numerators of (Cb, Cr) for 4 adjacent pixels of one MCU row; /15 rounding, colour
//     offsets and the G tie test are packed fp32 ops, add+clamp two pixels per DPX VIADDMNMX.S16x2.
//   * anything outside the range the fast arithmetic is proven for (huge samples, |Cb-128| >= 125, G within
//     BJ_G_ERR of a tie) takes an out-of-line exact path per 4-pixel run (pixel_quad_exact).
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_crop.cuh"
#include "bj_pixel_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

using bj::F2;
using bj::f2;
using bj::f2add;
using bj::f2fma;
using bj::f2mul;
using bj::f2s;

constexpr int kWarps = 5;               // 4 luma warps + 1 chroma warp (two rounds of 32 blocks)
constexpr int kThreads = kWarps * 32;
constexpr int kMcus = 32;              // MCUs per CTA (must match plan.py FAST_STRIP[LAYOUT_420])
constexpr int kTileBlocks = kMcus * 6; // 192 coefficient blocks
constexpr int kRowBytes = kMcus * 48;  // one staged RGB row of the strip

// shared memory map (offsets from a 1024-byte aligned base)
constexpr int OFF_COEF = 0;                    // 24576: TMA tile [192][128 B], later RGB staging [16][1536]
constexpr int OFF_Y = OFF_COEF + 24576;        // 16384: luma samples int16 [32 MCUs][4][8][8]
constexpr int OFF_C = OFF_Y + 16384;           //  8192: chroma samples f16 (int16 for wide blocks) [32 MCUs][8 rows][4 column pairs][Cb, Cr]
constexpr int OFF_Q = OFF_C + 8192;            //   768: quantisation tables as float [3][64]
constexpr int OFF_BASIS = OFF_Q + 768;         //   512: 1-D IDCT basis in double precision (exact recompute)
constexpr int OFF_NATZZ = OFF_BASIS + 512;     //    64: reference flat index u*8+v -> zig-zag index (exact recompute)
constexpr int OFF_MISC = OFF_NATZZ + 64;       //    32: mbarrier, wide masks
constexpr int SMEM_USED = OFF_MISC + 32;
constexpr int SMEM_BYTES = SMEM_USED;

struct Misc {
    unsigned long long mbar;
    uint32_t wide_mcu;     // bit m: MCU m has a block outside the fast colour path's range
    uint32_t wide_c[2];    // bit 2m+comp: that chroma block is stored as int16, not f16
};

// ---- PTX wrappers -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* mbar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* mbar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(mbar)), "r"(parity) : "memory");
}
// 2-D tiled TMA load: box (64 int16, 192 rows) at row `row` of the coefficient buffer
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, void* mbar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(mbar))
        : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read() {
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

__device__ __forceinline__ void mma_f16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};\n"
                 : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.0f));
}

// ---- tile addressing ------------------------------------------------------------------------------------------
struct Tiles {
    unsigned char* base;
    // 16-byte chunk c of tile row R of the coefficient tile (SWIZZLE_128B: chunk ^= row & 7)
    __device__ __forceinline__ const unsigned char* coef_chunk(int R, int c) const { return base + OFF_COEF + R * 128 + ((c ^ (R & 7)) << 4); }
    // luma block s of MCU m, row y (8 int16).  key: distinct for the 8 lanes of a store phase in phase A AND for
    // the (4 MCUs) x (2 blocks of a row) a half-warp reads at once in phase B
    __device__ __forceinline__ unsigned char* yrow(int m, int s, int y) const {
        const int key = (s & 1) | (((m + (s >> 1)) & 3) << 1);
        return base + OFF_Y + (m * 4 + s) * 128 + ((y ^ key) << 4);
    }
    // chroma samples (f16, or int16 for wide blocks) of MCU m, row y: 32 bytes, Cb and Cr interleaved in column
    // pairs [Cb01 Cr01 Cb23 Cr23 | Cb45 Cr45 Cb67 Cr67], so that one 16-byte load is a whole A fragment of the
    // interpolation MMA.  The row index is XOR-swizzled with a bit permutation of m: conflict-free 16-byte loads in
    // phase B (two MCUs x two rows per quarter-warp), 2-way on the 4-byte stores of phase A.
    __device__ __forceinline__ unsigned char* crow32(int m, int y) const {
        const int swz = ((m & 1) << 1) | ((m >> 1) & 1) | (m & 4);
        return base + OFF_C + m * 256 + ((y ^ swz) << 5);
    }
    // column pair cp (columns 2cp, 2cp+1) of component comp in that row: 4 bytes
    __device__ __forceinline__ unsigned char* cpair(int m, int comp, int y, int cp) const { return crow32(m, y) + cp * 8 + comp * 4; }
    __device__ __forceinline__ unsigned char* stage(int row) const { return base + OFF_COEF + row * kRowBytes; }
    __device__ __forceinline__ const float* qf() const { return reinterpret_cast<const float*>(base + OFF_Q); }
    __device__ __forceinline__ Misc* misc() const { return reinterpret_cast<Misc*>(base + OFF_MISC); }
    __device__ __forceinline__ const double* basis() const { return reinterpret_cast<const double*>(base + OFF_BASIS); }
    __device__ __forceinline__ const uint8_t* nat_zz() const { return base + OFF_NATZZ; }
};

// Store two exactly recomputed samples (x0, y) and (x1, y) of a block: luma int16, chroma f16 (int16 when wide).
// Out of line and shared by both exact routines: cold code, kept small.
__device__ __noinline__ void store_exact_pair(const Tiles t, int m, int s, int comp, bool as_int16, int y, int x0, int v0, int x1, int v1) {
    unsigned char* p0 = comp == 0 ? t.yrow(m, s, y) + 2 * x0 : t.cpair(m, comp - 1, y, x0 >> 1) + 2 * (x0 & 1);
    unsigned char* p1 = comp == 0 ? t.yrow(m, s, y) + 2 * x1 : t.cpair(m, comp - 1, y, x1 >> 1) + 2 * (x1 & 1);
    const bool i16 = comp == 0 || as_int16;
    // |v| <= 2048 in a chroma block that is not wide: exact in f16
    *reinterpret_cast<uint16_t*>(p0) = i16 ? (uint16_t)v0 : __half_as_ushort(__int2half_rn(v0));
    *reinterpret_cast<uint16_t*>(p1) = i16 ? (uint16_t)v1 : __half_as_ushort(__int2half_rn(v1));
}

// reference flat index u*8+v -> zig-zag index (zagzig, jpeg_decoder.py:1672-1681, inverted)
__constant__ uint8_t c_nat_zz[64] = {0, 2, 3, 9, 10, 20, 21, 35, 1, 4, 8, 11, 19, 22, 34, 36, 5, 7, 12, 18, 23, 33,
                                     37, 48, 6, 13, 17, 24, 32, 38, 47, 49, 14, 16, 25, 31, 39, 46, 50, 57, 15, 26,
                                     30, 40, 45, 51, 56, 58, 27, 29, 41, 44, 52, 55, 59, 62, 28, 42, 43, 53, 54, 60,
                                     61, 63};

// ---- exact recompute of one block by a whole warp (InverseDCT.__call__, :1561-1573) ---------------
// Lane l owns output samples s = l and l + 32 (s = x*8 + y).  Accumulator j = v collects the products
// of u = 0..7 in order, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)): numpy's pairwise sum of the 64
// products in C order [u][v]; zero coefficients only add +-0.0 and are skipped.
// R: tile row of the block; comp 0 = luma (block s of MCU m), 1/2 = Cb/Cr; as_int16: chroma block is `wide`.
__device__ __noinline__ void recompute_block_exact(const Tiles t, int R, int m, int s, int comp, bool as_int16,
                                                   const double* __restrict__ tabT, int lane) {
    const float* qf = t.qf() + comp * 64;
    int k0 = c_nat_zz[lane], k1 = c_nat_zz[lane + 32];
    int c0 = *reinterpret_cast<const int16_t*>(t.coef_chunk(R, k0 >> 3) + ((k0 & 7) << 1));
    int c1 = *reinterpret_cast<const int16_t*>(t.coef_chunk(R, k1 >> 3) + ((k1 & 7) << 1));
    int p0 = (int16_t)(c0 * (int)qf[k0]), p1 = (int16_t)(c1 * (int)qf[k1]);  // int16 product wraps (:869)
    const unsigned nz_lo = __ballot_sync(0xffffffffu, p0 != 0), nz_hi = __ballot_sync(0xffffffffu, p1 != 0);
    double r0[8], r1[8];
#pragma unroll
    for (int v = 0; v < 8; v++) r0[v] = r1[v] = 0.0;
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
    store_exact_pair(t, m, s, comp, as_int16, y0, x0, v0, x1, v1);
}

// c(n, k) = a_k cos((2n + 1) k pi / 16), a_0 = 1 / (2 sqrt 2), a_k = 1/2: the 1-D inverse DCT basis in double precision
__device__ const double g_idct_basis[64] = {
    0.35355339059327373, 0.4903926402016152, 0.46193976625564337, 0.4157348061512726, 0.3535533905932738, 0.27778511650980114, 0.19134171618254492, 0.09754516100806417,
    0.35355339059327373, 0.4157348061512726, 0.19134171618254492, -0.0975451610080641, -0.35355339059327373, -0.4903926402016152, -0.4619397662556434, -0.2777851165098011,
    0.35355339059327373, 0.27778511650980114, -0.19134171618254486, -0.4903926402016152, -0.35355339059327384, 0.09754516100806415, 0.46193976625564326, 0.41573480615127273,
    0.35355339059327373, 0.09754516100806417, -0.46193976625564337, -0.2777851165098011, 0.3535533905932737, 0.41573480615127273, -0.19134171618254495, -0.4903926402016153,
    0.35355339059327373, -0.0975451610080641, -0.4619397662556434, 0.2777851165098009, 0.35355339059327384, -0.41573480615127256, -0.19134171618254528, 0.4903926402016152,
    0.35355339059327373, -0.277785116509801, -0.19134171618254517, 0.4903926402016152, -0.35355339059327334, -0.09754516100806401, 0.46193976625564337, -0.4157348061512725,
    0.35355339059327373, -0.4157348061512727, 0.191341716182545, 0.09754516100806439, -0.35355339059327356, 0.4903926402016153, -0.4619397662556432, 0.27778511650980076,
    0.35355339059327373, -0.4903926402016152, 0.46193976625564326, -0.41573480615127256, 0.3535533905932733, -0.27778511650980076, 0.19134171618254478, -0.09754516100806429};

// ---- exact recompute, fast form: separable fp64 IDCT of one block by a whole warp -----------------------------
// The reference rounds the fp64 sum of 64 products taken in numpy's pairwise order (:1561-1573).  Any other fp64
// evaluation of the same sum differs from it by a few 1e-16 * sum|coef| (bound: 3e-15 * sum|coef|, see DESIGN.md), so
// unless a sample lies within 1e-13 * (sum|coef| + 8) of a rounding tie the two round to the same integer.  This
// routine evaluates the block separably (2 x 16 DFMA per lane instead of up to 128 DMUL + DADD), and reports back
// when some sample is inside that guard band (exact ties: DC-only blocks with DC = 4 mod 8, ...): the caller then
// runs recompute_block_exact, which follows numpy's order to the letter.
// Lane l = (a = l >> 3, b = l & 7) holds the products P[u][v] for (u, v) = (a, b) and (a + 4, b), and ends up with
// the samples (x, y) = (a, b) and (a + 4, b).  Returns true (warp-uniform) if the block is done.
__device__ __noinline__ bool recompute_block_sep(const Tiles t, int R, int m, int s, int comp, bool as_int16, float sum_abs, int lane) {
    const float* qf = t.qf() + comp * 64;
    const int a = lane >> 3, b = lane & 7;
    const int k0 = t.nat_zz()[lane], k1 = t.nat_zz()[lane + 32];
    const double* basis = t.basis();
    const int c0 = *reinterpret_cast<const int16_t*>(t.coef_chunk(R, k0 >> 3) + ((k0 & 7) << 1));
    const int c1 = *reinterpret_cast<const int16_t*>(t.coef_chunk(R, k1 >> 3) + ((k1 & 7) << 1));
    const int p0 = (int16_t)(c0 * (int)qf[k0]), p1 = (int16_t)(c1 * (int)qf[k1]);  // int16 product wraps (:869)
    // (rolled loops: this code runs for one block in ~270 and is fetched cold every time -- its instruction
    // footprint, not its instruction count, is what the rest of the CTA waits for)
    // pass 1: contract over v (vertical frequency) for y = b
    double h0 = 0.0, h1 = 0.0;
#pragma unroll 1
    for (int v = 0; v < 8; v++) {
        const double cv = basis[b * 8 + v];
        h0 = fma((double)__shfl_sync(0xffffffffu, p0, a * 8 + v), cv, h0);
        h1 = fma((double)__shfl_sync(0xffffffffu, p1, a * 8 + v), cv, h1);
    }
    // pass 2: contract over u (horizontal frequency) for x = a and a + 4
    double s0 = 0.0, s1 = 0.0;
#pragma unroll 1
    for (int ap = 0; ap < 4; ap++) {
        const double lo = __shfl_sync(0xffffffffu, h0, ap * 8 + b), hi = __shfl_sync(0xffffffffu, h1, ap * 8 + b);  // u = ap, ap + 4
        s0 = fma(lo, basis[a * 8 + ap], s0);
        s0 = fma(hi, basis[a * 8 + ap + 4], s0);
        s1 = fma(lo, basis[(a + 4) * 8 + ap], s1);
        s1 = fma(hi, basis[(a + 4) * 8 + ap + 4], s1);
    }
    const double r0 = rint(s0), r1 = rint(s1);
    const double guard = 1e-13 * ((double)sum_abs + 8.0);
    const bool unsure = (0.5 - fabs(s0 - r0) < guard) || (0.5 - fabs(s1 - r1) < guard);
    if (__any_sync(0xffffffffu, unsure)) return false;
    const int x0 = a, y0 = b, x1 = a + 4;
    const int v0 = (int16_t)(__double2int_rn(s0)) + 128, v1 = (int16_t)(__double2int_rn(s1)) + 128;
    store_exact_pair(t, m, s, comp, as_int16, y0, x0, v0, x1, v1);
    return true;
}

// exact colour conversion of one pixel, fp64, evaluation order of :1693-1695, clip (:1698), round (:1700)
__device__ __forceinline__ uint32_t ycc_to_rgb_exact_packed(int Yi, int Cbi, int Cri) {
    double Y = (double)Yi, cb = __dsub_rn((double)Cbi, 128.0), cr = __dsub_rn((double)Cri, 128.0);
    double r = __dadd_rn(Y, __dmul_rn(1.402, cr));
    double g = __dsub_rn(__dsub_rn(Y, __dmul_rn(0.34414, cb)), __dmul_rn(0.71414, cr));
    double b = __dadd_rn(Y, __dmul_rn(1.772, cb));
    r = fmin(fmax(r, 0.0), 255.0);
    g = fmin(fmax(g, 0.0), 255.0);
    b = fmin(fmax(b, 0.0), 255.0);
    return (uint32_t)__double2int_rn(r) | ((uint32_t)__double2int_rn(g) << 8) | ((uint32_t)__double2int_rn(b) << 16);
}

// Exact path of phase B for the 4 pixels a = 4q..4q+3 of row b of MCU m: integer interpolation
// floor((2N + 15) / 30) (ResizeGrid, :1588-1626) and fp64 colour, straight from the sample tiles.  Rare; compact.
__device__ __noinline__ void pixel_quad_exact(const Tiles t, int m, int b, int q) {
    const Misc* mi = t.misc();
    int jj, tt;
    bj::up_cell(b, jj, tt);
    unsigned char* st = t.stage(b) + m * 48 + q * 12;
#pragma unroll 1
    for (int p = 0; p < 4; p++) {
        const int a = 4 * q + p;
        int ii, ss;
        bj::up_cell(a, ii, ss);
        int w00, w10, w01, w11;
        bj::up_weights_2d(ii, jj, ss, tt, w00, w10, w01, w11);
        const int Y = reinterpret_cast<const int16_t*>(t.yrow(m, 2 * (b >> 3) + (a >> 3), b & 7))[a & 7];
        int c[2];
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const bool i16 = (mi->wide_c[(2 * m + k) >> 5] >> ((2 * m + k) & 31)) & 1u;
            int P[2][2];
#pragma unroll
            for (int dj = 0; dj < 2; dj++)
#pragma unroll
                for (int di = 0; di < 2; di++) {
                    const unsigned char* pr = t.cpair(m, k, jj + dj, (ii + di) >> 1);
                    P[dj][di] = i16 ? (int)reinterpret_cast<const int16_t*>(pr)[(ii + di) & 1]
                                    : __half2int_rn(reinterpret_cast<const __half*>(pr)[(ii + di) & 1]);
                }
            const int N = w00 * P[0][0] + w10 * P[0][1] + w01 * P[1][0] + w11 * P[1][1];
            const int n2 = 2 * N + 15;
            c[k] = n2 >= 0 ? n2 / 30 : -((-n2 + 29) / 30);
        }
        const uint32_t rgb = ycc_to_rgb_exact_packed(Y, c[0], c[1]);
        st[3 * p] = (unsigned char)rgb;
        st[3 * p + 1] = (unsigned char)(rgb >> 8);
        st[3 * p + 2] = (unsigned char)(rgb >> 16);
    }
}

// Interpolation weights as B fragments of mma.m16n8k16 (f16), built at compile time.
// Output row b, lane (g = lane >> 2 -> column n = g, q = lane & 3), two MMAs e = 0, 1:
//   column n of MMA e  <->  pixel a = 4 (n >> 1) + 2 e + (n & 1)      (so lane q of the D fragment owns pixels 4q..4q+3)
//   k = 2 q + e' (+8)  <->  source sample (row j(b) + (q >> 1), column 4 (q & 1) + e' (+2))   (see the A loads)
// entry [b][lane] = {b0, b1 of MMA 0, b0, b1 of MMA 1}, each two f16 (low half = even k).
struct WeightFrags {
    uint32_t v[16 * 32 * 4];
    static constexpr uint32_t h16(int n) {  // f16 bit pattern of the integer 0 <= n <= 15
        constexpr uint16_t tab[16] = {0x0000, 0x3C00, 0x4000, 0x4200, 0x4400, 0x4500, 0x4600, 0x4700,
                                      0x4800, 0x4880, 0x4900, 0x4980, 0x4A00, 0x4A80, 0x4B00, 0x4B80};
        return tab[n];
    }
    static constexpr int weight(int b, int a, int rsel, int col) {
        int ii = 0, ss = 0, jj = 0, tt = 0;
        bj::up_cell(a, ii, ss);
        bj::up_cell(b, jj, tt);
        int w00 = 0, w10 = 0, w01 = 0, w11 = 0;
        bj::up_weights_2d(ii, jj, ss, tt, w00, w10, w01, w11);
        if (rsel == 0) return col == ii ? w00 : (col == ii + 1 ? w10 : 0);
        return col == ii ? w01 : (col == ii + 1 ? w11 : 0);
    }
    constexpr WeightFrags() : v{} {
        for (int b = 0; b < 16; b++)
            for (int lane = 0; lane < 32; lane++) {
                const int n = lane >> 2, q = lane & 3;
                for (int e = 0; e < 2; e++) {
                    const int a = 4 * (n >> 1) + 2 * e + (n & 1);
                    for (int hi = 0; hi < 2; hi++) {
                        uint32_t w = 0;
                        for (int ep = 0; ep < 2; ep++) {
                            const int rsel = q >> 1, col = 4 * (q & 1) + 2 * hi + ep;
                            w |= h16(weight(b, a, rsel, col)) << (16 * ep);
                        }
                        v[(b * 32 + lane) * 4 + e * 2 + hi] = w;
                    }
                }
            }
    }
};
__device__ const WeightFrags g_weight_frags{};

// ---- phase A ---------------------------------------------------------------------------------------------------
// 1 if zig-zag index k lies in the 4x4 low-frequency corner (u, v <= 3)
__host__ __device__ constexpr bool in_lo4(int k) {
    constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
    return (zz[k] & 7) < 4 && (zz[k] >> 3) < 4;
}

struct BlockResult {
    bool flagged, wide;
    float sum_abs;   // >= sum of |dequantised coefficient| (guard band of the separable recompute)
};

// One block per lane: dequantise, IDCT, round, tie test, store samples.  LO4: only the 4x4 corner is non-zero.
// LUMA: store int16 rows into the luma tile, else f16 (int16 when wide) into the chroma tile.
template <bool LUMA, bool LO4>
__device__ __forceinline__ BlockResult block_idct(const Tiles t, const uint4 (&cv)[8], int m, int s, int comp) {
    const float* qf = t.qf() + comp * 64;
    F2 P[8][4];
    if (LO4) {
#pragma unroll
        for (int v = 0; v < 4; v++)
#pragma unroll
            for (int h = 0; h < 2; h++) P[v][h] = f2(0.f, 0.f);
    }
    float Sw = 0.f;
    const float4* q4 = reinterpret_cast<const float4*>(qf);
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if (LO4 && c > 3) continue;   // zig-zag 32..63 lie outside the corner
        const float4 qa = q4[2 * c], qb = q4[2 * c + 1];
        const float qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
        const uint32_t vw[4] = {cv[c].x, cv[c].y, cv[c].z, cv[c].w};
#pragma unroll
        for (int e = 0; e < 8; e++) {
            constexpr uint8_t zz[64] = {BJ_ZZ_NATURAL};
            const int K = c * 8 + e;
            if (LO4 && !in_lo4(K)) continue;
            const uint32_t w = vw[e >> 1];
            const int16_t ci = (e & 1) ? (int16_t)(w >> 16) : (int16_t)(w & 0xffffu);
            const float x = (float)ci * qv[e];  // exact; the int16 wrap of :869 is caught by the S bound below
            const int n = zz[K], v = n >> 3, u = n & 7;
            if (u & 1) P[v][u >> 1].y = x;
            else P[v][u >> 1].x = x;
            // error-weighted sum of the AC magnitudes (one FFMA, the weight is an immediate), see bj_pixel_math.cuh
            if (K) Sw = fmaf(fabsf(x), bj::idct_err_weight(v, u), Sw);
        }
    }
    const float dc_abs = fabsf(P[0][0].x);
    const float S = Sw * (1.0f / BJ_IDCT_W_MIN);   // >= sum |AC|
    // |sample - 128| <= |DC| / 8 + sum|AC| / 4 + 1/2 (every basis value is at most 1/8 resp. 1/4)
    const float bound = fmaf(0.25f, S, fmaf(0.125f, dc_abs, 0.5f));
    BlockResult res;
    res.wide = bound >= (comp == 0 ? 30000.0f : comp == 1 ? 125.0f : BJ_CHROMA_GUARD);
    const float dc_int = bj::dc_peel(P[0][0].x);   // DC/8 = dc_int + (what is left in P[0][0].x) / 8
    const float T = fmaf(fmaf(P[0][0].x, bj::idct_err_weight(0, 0), Sw), BJ_IDCT_ERR_U, BJ_IDCT_ERR_ABS);
    // round + level shift (+ the peeled DC) in one add: the low mantissa bits of v + (1.5 * 2^23 + 128 + I) are
    // rint(v) + 128 + I
    const float shift = (BJ_MAGIC + 128.0f) + dc_int;
    F2 Wa[4][8];
    float maxd;
    bj::idct8x8_round_packed<LO4>(P, shift, Wa, maxd);
#pragma unroll
    for (int yp = 0; yp < 4; yp++) {
        const F2 (&W)[8] = Wa[yp];
        if (LUMA) {
            // int16 pairs = the low halves of the biased floats (the bias has a zero low half)
            *reinterpret_cast<uint4*>(t.yrow(m, s, 2 * yp)) = make_uint4(__byte_perm(__float_as_uint(W[0].x), __float_as_uint(W[1].x), 0x5410),
                                                                          __byte_perm(__float_as_uint(W[2].x), __float_as_uint(W[3].x), 0x5410),
                                                                          __byte_perm(__float_as_uint(W[4].x), __float_as_uint(W[5].x), 0x5410),
                                                                          __byte_perm(__float_as_uint(W[6].x), __float_as_uint(W[7].x), 0x5410));
            *reinterpret_cast<uint4*>(t.yrow(m, s, 2 * yp + 1)) = make_uint4(__byte_perm(__float_as_uint(W[0].y), __float_as_uint(W[1].y), 0x5410),
                                                                              __byte_perm(__float_as_uint(W[2].y), __float_as_uint(W[3].y), 0x5410),
                                                                              __byte_perm(__float_as_uint(W[4].y), __float_as_uint(W[5].y), 0x5410),
                                                                              __byte_perm(__float_as_uint(W[6].y), __float_as_uint(W[7].y), 0x5410));
        } else {
            uint32_t h0[4], h1[4];
            if (res.wide) {
#pragma unroll
                for (int x = 0; x < 4; x++) {
                    h0[x] = __byte_perm(__float_as_uint(W[2 * x].x), __float_as_uint(W[2 * x + 1].x), 0x5410);
                    h1[x] = __byte_perm(__float_as_uint(W[2 * x].y), __float_as_uint(W[2 * x + 1].y), 0x5410);
                }
            } else {
                // rint(v) + 128 = W - MAGIC (exact), as f16 (|.| <= 2048 in a block that is not wide: exact)
#pragma unroll
                for (int x = 0; x < 4; x++) {
                    const F2 va = f2add(W[2 * x], f2s(-BJ_MAGIC)), vb = f2add(W[2 * x + 1], f2s(-BJ_MAGIC));   // exact
                    __half2 a = __floats2half2_rn(va.x, vb.x), b = __floats2half2_rn(va.y, vb.y);
                    h0[x] = *reinterpret_cast<uint32_t*>(&a);
                    h1[x] = *reinterpret_cast<uint32_t*>(&b);
                }
            }
            unsigned char* r0 = t.crow32(m, 2 * yp) + (comp - 1) * 4;
            unsigned char* r1 = t.crow32(m, 2 * yp + 1) + (comp - 1) * 4;
#pragma unroll
            for (int x = 0; x < 4; x++) {
                *reinterpret_cast<uint32_t*>(r0 + 8 * x) = h0[x];
                *reinterpret_cast<uint32_t*>(r1 + 8 * x) = h1[x];
            }
        }
    }
    // the fp32 products are only the reference's int16 products (:869) while nothing wraps
    res.sum_abs = S + dc_abs;
    res.flagged = (maxd > 0.5f - T) || (S + dc_abs > 32767.0f);
#ifdef BJ_EXP_NO_RECOMPUTE
    res.flagged = false;   // timing experiment only: results are wrong near ties
#endif
    return res;
}

template <bool LUMA>
__device__ __forceinline__ BlockResult block_dense_inl(const Tiles t, int R, int m, int s, int comp) {
    uint4 cv[8];
#pragma unroll
    for (int c = 0; c < 8; c++) cv[c] = *reinterpret_cast<const uint4*>(t.coef_chunk(R, c));
    return block_idct<LUMA, false>(t, cv, m, s, comp);
}
template <bool LUMA>
__device__ __noinline__ BlockResult block_dense(const Tiles t, int R, int m, int s, int comp) {
    uint4 cv[8];
#pragma unroll
    for (int c = 0; c < 8; c++) cv[c] = *reinterpret_cast<const uint4*>(t.coef_chunk(R, c));
    return block_idct<LUMA, false>(t, cv, m, s, comp);
}

// 96 registers x 160 threads x 4 CTAs = 61440 of the SM's 65536 registers; 50 KB of shared memory per CTA
// CROP: one CTA per strip of a bj_crop_job's MCU window (4:2:0 jobs at scale 1), storing only the box.
template <bool CROP>
__global__ void __maxnreg__(96)
bj_pixels_420_kernel(const __grid_constant__ CUtensorMap tmap, const bj_image* __restrict__ images,
                     const int16_t* __restrict__ qtabs, const double* __restrict__ tabT, uint8_t* __restrict__ out,
                     uint32_t* __restrict__ stats, const bj_crop_job* __restrict__ jobs) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];   // SWIZZLE_128B wants a 1024-byte aligned tile
    Tiles t;
    t.base = smem_raw;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // (the job is read again for the store rather than kept in registers through phase A and B; phase B computes
    // every row of the strip, not only the box's: a row filter there costs registers the kernel does not have)
    const bj_image* const gi = &images[CROP ? __ldg(&jobs[blockIdx.y].image) : blockIdx.y];
    if ((int)__ldg(&gi->layout) != BJ_LAYOUT_420) return;
    const int mcus_x = (int)__ldg(&gi->mcus_x);
    int my, m0, M;
    if constexpr (CROP) {
        const bj_crop_job jb = jobs[blockIdx.y];
        if (jb.log2_scale != 0) return;
        if (!bj::crop_strip(jb, 16, 16, kMcus, blockIdx.x, my, m0, M)) return;
    } else {
        const int mcus_y = (int)__ldg(&gi->mcus_y);
        const int strips_per_row = (mcus_x + kMcus - 1) / kMcus;
        if ((int)blockIdx.x >= mcus_y * strips_per_row) return;
        my = blockIdx.x / strips_per_row;
        m0 = (blockIdx.x - my * strips_per_row) * kMcus;
        M = min(kMcus, mcus_x - m0);
    }
    Misc* misc = t.misc();

    // ---- prologue: one thread requests the coefficient tile and the weight fragments ------------------------------
    if (tid == 0) {
        mbar_init(&misc->mbar, 1);
        mbar_expect_tx(&misc->mbar, kTileBlocks * 128);
        const long long row0 = (long long)__ldg(&gi->coef_block0) + ((long long)my * mcus_x + m0) * 6;
        tma_load_2d(t.base + OFF_COEF, &tmap, 0, (int)row0, &misc->mbar);
        misc->wide_mcu = 0;
        misc->wide_c[0] = misc->wide_c[1] = 0;
    }
    for (int i = tid; i < 192; i += kThreads) {
        float* qf = reinterpret_cast<float*>(t.base + OFF_Q);
        qf[i] = (float)qtabs[(size_t)__ldg(&gi->qtab[i >> 6]) * 64 + (i & 63)];
    }
    if (tid < 64) {   // tables of the exact recompute: shared-memory copies keep its (serial) latency short
        reinterpret_cast<double*>(t.base + OFF_BASIS)[tid] = g_idct_basis[tid];
        t.base[OFF_NATZZ + tid] = c_nat_zz[tid];
    }
    __syncthreads();
    mbar_wait(&misc->mbar, 0);

    // ---- phase A: one lane per block -------------------------------------------------------------------------
    if (warp < 4) {
        // luma: 16-lane groups = 4 MCUs ordered (0, 2, 1, 3) so that the 8 tile rows read by an 8-lane phase are
        // distinct modulo 8 (rows 6m + s)
        const int l4 = (lane >> 2) & 3;
        const int m = 8 * warp + 4 * (lane >> 4) + (((l4 & 1) << 1) | (l4 >> 1));
        const int s = lane & 3;
        const int R = 6 * m + s;
        BlockResult r{false, false, 0.f};
        if (m < M) r = block_dense_inl<true>(t, R, m, s, 0);
        unsigned mask = __ballot_sync(0xffffffffu, r.flagged);
        const unsigned wide = __ballot_sync(0xffffffffu, r.wide);
        if (wide && lane == 0) {
            unsigned mm = 0;
            for (unsigned w = wide; w; w &= w - 1) {
                const int l = __ffs(w) - 1, q4 = (l >> 2) & 3;
                mm |= 1u << (8 * warp + 4 * (l >> 4) + (((q4 & 1) << 1) | (q4 >> 1)));
            }
            atomicOr(&misc->wide_mcu, mm);
        }
        if (mask) {
            __syncwarp();
            if (stats && lane == 0) atomicAdd(&stats[0], (uint32_t)__popc(mask));
            while (mask) {
                const int l = __ffs(mask) - 1, q4 = (l >> 2) & 3;
                mask &= mask - 1;
                const int mm = 8 * warp + 4 * (l >> 4) + (((q4 & 1) << 1) | (q4 >> 1));
                const float sa = __shfl_sync(0xffffffffu, r.sum_abs, l);
                if (!recompute_block_sep(t, 6 * mm + (l & 3), mm, l & 3, 0, false, sa, lane))
                    recompute_block_exact(t, 6 * mm + (l & 3), mm, l & 3, 0, false, tabT, lane);
            }
        }
    } else {
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
            const int C = half * 32 + lane;
            const int m = C >> 1, comp = C & 1;
            const int R = 6 * m + 4 + comp;
            const bool active = m < M;
            if (__all_sync(0xffffffffu, !active)) break;
            uint4 cv[8];
            uint32_t other = 0;
            if (active) {
#pragma unroll
                for (int c = 0; c < 8; c++) cv[c] = *reinterpret_cast<const uint4*>(t.coef_chunk(R, c));
#pragma unroll
                for (int w = 0; w < 32; w++) {
                    const uint32_t msk = (in_lo4(2 * w) ? 0u : 0xffffu) | (in_lo4(2 * w + 1) ? 0u : 0xffff0000u);
                    const uint32_t word = (w & 3) == 0 ? cv[w >> 2].x : (w & 3) == 1 ? cv[w >> 2].y : (w & 3) == 2 ? cv[w >> 2].z : cv[w >> 2].w;
                    if (msk) other |= word & msk;
                }
            }
            BlockResult r{false, false, 0.f};
            if (__all_sync(0xffffffffu, other == 0)) {
                if (active) r = block_idct<false, true>(t, cv, m, 0, comp + 1);
            } else {
                if (active) r = block_dense<false>(t, R, m, 0, comp + 1);
            }
            unsigned mask = __ballot_sync(0xffffffffu, r.flagged);
            const unsigned wide = __ballot_sync(0xffffffffu, r.wide);
            if (wide && lane == 0) {
                unsigned mm = 0;
                for (unsigned w = wide; w; w &= w - 1) mm |= 1u << ((half * 32 + __ffs(w) - 1) >> 1);
                atomicOr(&misc->wide_mcu, mm);
                misc->wide_c[half] = wide;  // bit 2m+comp of the CTA-wide mask = bit `lane` of this round's word
            }
            if (mask) {
                __syncwarp();
                if (stats && lane == 0) atomicAdd(&stats[0], (uint32_t)__popc(mask));
                while (mask) {
                    const int l = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const int CC = half * 32 + l;
                    const float sa = __shfl_sync(0xffffffffu, r.sum_abs, l);
                    if (!recompute_block_sep(t, 6 * (CC >> 1) + 4 + (CC & 1), CC >> 1, 0, (CC & 1) + 1, (wide >> l) & 1u, sa, lane))
                        recompute_block_exact(t, 6 * (CC >> 1) + 4 + (CC & 1), CC >> 1, 0, (CC & 1) + 1, (wide >> l) & 1u, tabT, lane);
                }
            }
        }
    }
    __syncthreads();   // samples complete; the coefficient tile is dead from here on (it becomes the RGB staging)

    // ---- phase B: (group of 8 MCUs, pixel row) per warp iteration; lane (g, q) = MCU g of the group, pixels 4q..4q+3 ----
    const int x0 = m0 * 16, y0 = my * 16;
    const int cols = min(M * 16, (int)__ldg(&gi->width) - x0);
    const int rows = min(16, (int)__ldg(&gi->height) - y0);
    {
        const int g = lane >> 2, q = lane & 3;
        const uint32_t wide_mcu = misc->wide_mcu;
        const uint4* wfr = reinterpret_cast<const uint4*>(g_weight_frags.v) + lane;   // 8 KB, L1-resident
        const int n_it = ((M + 7) >> 3) * 16;
        // lane-invariant parts of the tile addresses (MCU g of group 0)
        const int cswz = ((g & 1) << 1) | ((g >> 1) & 1) | (g & 4);
        const unsigned char* cbase = t.base + OFF_C + g * 256 + (q & 1) * 16;
        const unsigned char* ybase = t.base + OFF_Y + g * 512 + (q >> 1) * 128 + (q & 1) * 8;
        unsigned char* sbase = t.base + OFF_COEF + g * 48 + q * 12;
#pragma unroll 1
        for (int it = warp; it < n_it; it += kWarps) {
            const int G = it >> 4, b = it & 15;
            if (b >= rows) continue;
            const int m = 8 * G + g;
            const int j = (int)((0x6665544332211000ull >> (4 * b)) & 7);   // source row of output row b: floor(7b/15), 6 for b = 15
            const uint4 wf = __ldg(wfr + b * 32);
            // A fragment: (Cb lo, Cr lo, Cb hi, Cr hi) column pairs of source row j + (q >> 1)
            const uint4 av = *reinterpret_cast<const uint4*>(cbase + G * 2048 + (((j + (q >> 1)) ^ cswz) << 5));
            // luma: pixels 4q..4q+3 of row b = block 2 (b >> 3) + (q >> 1), row b & 7, columns 4 (q & 1)..
            const int ykey = (q >> 1) | (((g + (b >> 3)) & 3) << 1);
            const uint2 yv = *reinterpret_cast<const uint2*>(ybase + G * 4096 + (b >> 3) * 256 + (((b & 7) ^ ykey) << 4));
            float d[4], e[4];
            mma_f16(d, av.x, av.y, av.z, av.w, wf.x, wf.y);  // (Cb p0, Cb p1, Cr p0, Cr p1) numerators
            mma_f16(e, av.x, av.y, av.z, av.w, wf.z, wf.w);  // (Cb p2, Cb p3, Cr p2, Cr p3)
            // N / 15 rounded (never a tie), minus 128: both subtractions folded into one exact fp32 add
            const F2 k15 = f2s(1.0f / 15.0f), kmg = f2s(BJ_MAGIC), kun = f2s(-(BJ_MAGIC + 128.0f));
            const F2 cb01 = f2add(f2fma(f2(d[0], d[1]), k15, kmg), kun), cr01 = f2add(f2fma(f2(d[2], d[3]), k15, kmg), kun);
            const F2 cb23 = f2add(f2fma(f2(e[0], e[1]), k15, kmg), kun), cr23 = f2add(f2fma(f2(e[2], e[3]), k15, kmg), kun);
            // colour offsets + 1.5 * 2^23 in one rounding: the low mantissa bits are round-to-nearest(offset)
            const F2 wr01 = f2fma(f2s(1.402f), cr01, kmg), wr23 = f2fma(f2s(1.402f), cr23, kmg);
            const F2 wb01 = f2fma(f2s(1.772f), cb01, kmg), wb23 = f2fma(f2s(1.772f), cb23, kmg);
            const F2 gc01 = f2fma(f2s(-0.71414f), cr01, f2mul(f2s(-0.34414f), cb01));
            const F2 gc23 = f2fma(f2s(-0.71414f), cr23, f2mul(f2s(-0.34414f), cb23));
            const F2 wg01 = f2add(gc01, kmg), wg23 = f2add(gc23, kmg);
            const F2 dg01 = f2add(gc01, f2fma(wg01, f2s(-1.0f), kmg)), dg23 = f2add(gc23, f2fma(wg23, f2s(-1.0f), kmg));
            const float dgmax = fmaxf(fmaxf(fmaxf(fabsf(dg01.x), fabsf(dg01.y)), fabsf(dg23.x)), fabsf(dg23.y));
            if (((wide_mcu >> m) & 1u) || dgmax > 0.5f - BJ_G_ERR) {
                if (m < M) {
                    pixel_quad_exact(t, m, b, q);
                    if (stats) atomicAdd(&stats[1], 4u);
                }
                continue;
            }
            // two pixels per DPX add-min-relu (VIADDMNMX.S16x2): clamp(Y + round(offset), 0, 255)
            const uint32_t R01 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wr01.x), __float_as_uint(wr01.y), 0x5410), yv.x, 0x00FF00FFu);
            const uint32_t G01 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wg01.x), __float_as_uint(wg01.y), 0x5410), yv.x, 0x00FF00FFu);
            const uint32_t B01 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wb01.x), __float_as_uint(wb01.y), 0x5410), yv.x, 0x00FF00FFu);
            const uint32_t R23 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wr23.x), __float_as_uint(wr23.y), 0x5410), yv.y, 0x00FF00FFu);
            const uint32_t G23 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wg23.x), __float_as_uint(wg23.y), 0x5410), yv.y, 0x00FF00FFu);
            const uint32_t B23 = __viaddmin_s16x2_relu(__byte_perm(__float_as_uint(wb23.x), __float_as_uint(wb23.y), 0x5410), yv.y, 0x00FF00FFu);
            // 4 pixels x 3 bytes: R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3
            const uint32_t t0 = __byte_perm(R01, G01, 0x6240);   // R0 G0 R1 G1
            const uint32_t t1 = __byte_perm(R23, G23, 0x6240);   // R2 G2 R3 G3
            const uint32_t o0 = __byte_perm(t0, B01, 0x2410);                              // R0 G0 B0 R1
            const uint32_t o1 = __byte_perm(__byte_perm(t0, B01, 0x0063), t1, 0x5410);     // G1 B1 | R2 G2
            const uint32_t o2 = __byte_perm(t1, B23, 0x6324);                              // B2 R3 G3 B3
            uint32_t* st = reinterpret_cast<uint32_t*>(sbase + b * kRowBytes + G * 384);
            st[0] = o0;
            st[1] = o1;
            st[2] = o2;
        }
    }
    fence_proxy_async();
    __syncthreads();

    // ---- store the strip's rows ---------------------------------------------------------------------------------
    if constexpr (CROP) {
        const bj_crop_job jb = jobs[blockIdx.y];
        int sx, sy, w, h;
        uint8_t* g;
        if (bj::crop_part(jb, x0, y0, cols, rows, 3, out, sx, sy, w, h, g))
            bj::crop_store(g, jb.out_pitch, t.stage(sy), kRowBytes, sx * 3, w * 3, h, tid, kThreads);
        return;
    }
    const uint32_t pitch = __ldg(&gi->out_pitch);
    uint8_t* gout = out + (int64_t)__ldg(&gi->out_offset) + (int64_t)y0 * pitch + (int64_t)x0 * 3;
    const int nbytes = cols * 3;
    const bool aligned = ((reinterpret_cast<uintptr_t>(gout) & 15) == 0) && ((pitch & 15) == 0);
    if (aligned && (nbytes & 15) == 0) {
        if (tid < rows) {
            bulk_store(gout + (int64_t)tid * pitch, t.stage(tid), (uint32_t)nbytes);
            bulk_commit_wait_read();
        }
    } else if (aligned) {
        const int nvec = nbytes >> 4, tail = nbytes & 15;
#pragma unroll 1
        for (int r = warp; r < rows; r += kWarps) {
#pragma unroll 1
            for (int v = lane; v < nvec; v += 32)
                __stcs(reinterpret_cast<uint4*>(gout + (int64_t)r * pitch + (v << 4)), *reinterpret_cast<const uint4*>(t.stage(r) + (v << 4)));
            if (lane < tail) gout[(int64_t)r * pitch + (nvec << 4) + lane] = t.stage(r)[(nvec << 4) + lane];
        }
    } else {
#pragma unroll 1
        for (int r = warp; r < rows; r += kWarps)
#pragma unroll 1
            for (int b = lane; b < nbytes; b += 32) gout[(int64_t)r * pitch + b] = t.stage(r)[b];
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

}  // namespace

extern "C" int bj_pixels_420_strip(void) { return kMcus; }

namespace {

// grid.y = n_images (jobs == nullptr) or the crop jobs
template <bool CROP>
bj_status launch_420(const bj_image* images, const bj_crop_job* jobs, int n_images, int max_strips, const int16_t* coef,
                     uint64_t total_blocks, const int16_t* qtabs, const double* tabT, uint8_t* out, uint32_t* stats,
                     void* stream) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return bj_set_cuda_error(cudaErrorNotSupported, "bj_pixels/420: cuTensorMapEncodeTiled unavailable");
    if (total_blocks == 0 || total_blocks > 0x7fffffffull) return BJ_E_ARG;
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {64, (cuuint64_t)total_blocks};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {64, (cuuint32_t)kTileBlocks};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<int16_t*>(coef), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return bj_set_cuda_error(cudaErrorInvalidValue, "bj_pixels/420: cuTensorMapEncodeTiled");
    cudaError_t e = cudaFuncSetAttribute(bj_pixels_420_kernel<CROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(bj_pixels_420_kernel<CROP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels/420");
    bj_pixels_420_kernel<CROP><<<dim3((unsigned)max_strips, (unsigned)n_images), kThreads, SMEM_BYTES, (cudaStream_t)stream>>>(
        tmap, images, qtabs, tabT, out, stats, jobs);
    e = cudaGetLastError();
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels/420");
    return BJ_OK;
}

}  // namespace

// 4:2:0 images of the batch: coefficient buffer (total_blocks x 64 int16) -> RGB.
extern "C" bj_status bj_pixels_420_launch(const bj_image* images, int n_images, int max_strips, const int16_t* coef,
                                          uint64_t total_blocks, const int16_t* qtabs, const double* tabT, uint8_t* out,
                                          uint32_t* stats, void* stream) {
    return launch_420<false>(images, nullptr, n_images, max_strips, coef, total_blocks, qtabs, tabT, out, stats, stream);
}

// 4:2:0 crop jobs at scale 1 (bj_pixels_crop).
extern "C" bj_status bj_pixels_420_crop_launch(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                                               const int16_t* coef, uint64_t total_blocks, const int16_t* qtabs,
                                               const double* tabT, uint8_t* out, uint32_t* stats, void* stream) {
    return launch_420<true>(images, jobs, n_jobs, max_strips, coef, total_blocks, qtabs, tabT, out, stats, stream);
}
