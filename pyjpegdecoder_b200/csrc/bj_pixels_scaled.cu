// bj_pixels_scaled.cu -- reduced-size decode (scale 1/2, 1/4, 1/8 in the DCT domain) of a whole batch of images in
// one launch (sm_100a): dequantise + N-point IDCT of each block's low-frequency corner + colour, straight from the
// coefficient buffer to RGB / grey at ceil(H/s) x ceil(W/s).  The arithmetic is bj_scaled_math.cuh; see
// include/b200jpeg.h for the ABI.
//
// One CTA = one strip of up to scaled_strip_mcus() MCUs of one MCU row of one job (grid: strips x jobs):
//   load    only the zig-zag prefix each block's corner needs, as coalesced 16-byte loads (consecutive threads walk
//           the (block, 16-byte chunk) pairs of the strip) into shared memory, chunks XOR-swizzled by block
//   tile    one thread per block: dequantise, separable N-point IDCT, round; the NY x NX tile goes into its
//           component's sample plane, which has the scaled strip's own resolution (no upsampling at any layout)
//   colour  one thread per output pixel: YCbCr -> RGB, the bytes are staged row by row in shared memory, each row at
//           the alignment (mod 16) of its destination
//   store   16-byte stores for the aligned middle of each row, byte stores at both ends
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_scaled_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

constexpr int kThreads = 192;
constexpr int kMaxBlocks = 192;    // blocks per strip (one per thread in the tile phase)
constexpr int kPlane = 6144;       // sample-plane floats per CTA: ncomp x 16 hmax vmax x strip MCUs at s = 2

struct Smem {
    alignas(16) unsigned char a[kMaxBlocks * 128];  // coefficient prefixes (swizzled); then the staged output rows
    alignas(16) float p[kPlane];                    // sample planes [comp][row][column]
    alignas(16) int16_t qt[BJ_MAX_COMP][64];
    uint8_t load_slot[BJ_MAX_SLOTS * 8], load_chunk[BJ_MAX_SLOTS * 8];  // the (slot, chunk) pairs of one MCU
    uint8_t slot_comp[BJ_MAX_SLOTS], slot_bx[BJ_MAX_SLOTS], slot_by[BJ_MAX_SLOTS];
    int lnx[BJ_MAX_COMP], lny[BJ_MAX_COMP];
    int n_load;
    int lead[8];                                    // destination address mod 16 of each output row
};

__device__ __forceinline__ int swzA(int blk, int chunk) { return blk * 128 + ((chunk ^ (blk & 7)) << 4); }

// MCUs per strip; the host computes max_strips with the same rule (pyjpegdecoder_b200/scaled.py)
__device__ __forceinline__ int scaled_strip_mcus(const bj_image& im) {
    const int by_blocks = kMaxBlocks / im.blocks_per_mcu;
    const int by_plane = kPlane / (im.ncomp * 16 * im.hmax * im.vmax);
    return by_blocks < by_plane ? by_blocks : by_plane;
}

__global__ void __launch_bounds__(kThreads, 3)
bj_pixels_scaled_kernel(const bj_image* __restrict__ images, const bj_scaled_job* __restrict__ jobs,
                        const int16_t* __restrict__ coef, const int16_t* __restrict__ qtabs, uint8_t* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    __shared__ bj_image im;
    const int tid = threadIdx.x;
    const bj_scaled_job jb = jobs[blockIdx.y];
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&images[jb.image]);
        if (tid < (int)(sizeof(bj_image) / 4)) reinterpret_cast<uint32_t*>(&im)[tid] = src[tid];
    }
    __syncthreads();
    const int l = (int)jb.log2_scale;
    if (l < 1 || l > 3) return;
    const int M_max = scaled_strip_mcus(im);
    const int strips_per_row = ((int)im.mcus_x + M_max - 1) / M_max;
    if ((int)blockIdx.x >= (int)im.mcus_y * strips_per_row) return;
    const int my = blockIdx.x / strips_per_row;
    const int m0 = (blockIdx.x - my * strips_per_row) * M_max;
    const int M = min(M_max, (int)im.mcus_x - m0);
    const int bpm = im.blocks_per_mcu;
    const int nblk = M * bpm;
    const int ch = im.ncomp == 3 ? 3 : 1;
    const int64_t gblk0 = (int64_t)im.coef_block0 + ((int64_t)my * im.mcus_x + m0) * bpm;

    // ---- set-up tables -------------------------------------------------------------------------------------------
    for (int i = tid; i < im.ncomp * 64; i += kThreads) {
        const int c = i >> 6;
        sm.qt[c][i & 63] = qtabs[(size_t)im.qtab[c] * 64 + (i & 63)];
    }
    if (tid < im.ncomp) {
        sm.lnx[tid] = bj::scaled_log2_side(im.hmax, im.hs[tid], l);
        sm.lny[tid] = bj::scaled_log2_side(im.vmax, im.vs[tid], l);
    }
    if (tid == 0) {
        int n = 0;
        for (int s = 0; s < bpm; s++) {
            int c = 0;
            for (int k = 0; k < im.ncomp; k++)
                if (s >= im.slot0[k]) c = k;
            const int r = s - im.slot0[c];
            sm.slot_comp[s] = (uint8_t)c;
            sm.slot_bx[s] = (uint8_t)(r % im.hs[c]);
            sm.slot_by[s] = (uint8_t)(r / im.hs[c]);
            const int lx = bj::scaled_log2_side(im.hmax, im.hs[c], l), ly = bj::scaled_log2_side(im.vmax, im.vs[c], l);
            const int chunks = (bj::scaled_prefix(1 << lx, 1 << ly) + 7) >> 3;
            for (int k = 0; k < chunks; k++, n++) {
                sm.load_slot[n] = (uint8_t)s;
                sm.load_chunk[n] = (uint8_t)k;
            }
        }
        sm.n_load = n;
    }
    __syncthreads();

    // ---- load: the needed 16-byte chunks of every block of the strip ------------------------------------------------
    {
        const int Q = sm.n_load;
        const uint4* g = reinterpret_cast<const uint4*>(coef + gblk0 * 64);
        for (int i = tid; i < M * Q; i += kThreads) {
            const int m = i / Q, j = i - m * Q;
            const int b = m * bpm + sm.load_slot[j], c = sm.load_chunk[j];
            *reinterpret_cast<uint4*>(sm.a + swzA(b, c)) = __ldg(g + b * 8 + c);
        }
    }
    __syncthreads();

    // ---- tile: one thread per block ----------------------------------------------------------------------------------
    const int mcu_w = (8 * im.hmax) >> l, mcu_h = (8 * im.vmax) >> l;   // scaled pixels per MCU
    const int PC = M * mcu_w;                                           // plane columns; plane rows = mcu_h
    if (tid < nblk) {
        const int m = tid / bpm, s = tid - m * bpm;
        const int c = sm.slot_comp[s];
        const int lx = sm.lnx[c], ly = sm.lny[c];
        const int col = ((m * im.hs[c] + sm.slot_bx[s]) << lx), row = sm.slot_by[s] << ly;
        const unsigned char* A = sm.a;
        const int blk = tid;
        auto cf = [A, blk](int k) { return (int)*reinterpret_cast<const int16_t*>(A + swzA(blk, k >> 3) + ((k & 7) << 1)); };
        bj::scaled_tile(lx, ly, cf, sm.qt[c], &sm.p[(c * mcu_h + row) * PC + col], PC);
    }
    __syncthreads();

    // ---- colour into the staged rows ---------------------------------------------------------------------------------
    const int out_w = ((int)im.width + (1 << l) - 1) >> l, out_h = ((int)im.height + (1 << l) - 1) >> l;
    const int x0 = m0 * mcu_w, y0 = my * mcu_h;
    const int cols = min(PC, out_w - x0), rows = min(mcu_h, out_h - y0);
    if (cols <= 0 || rows <= 0) return;
    uint8_t* gout = out + jb.out_offset + (int64_t)y0 * jb.out_pitch + (int64_t)x0 * ch;
    const int nbytes = cols * ch;
    const int rs = ((nbytes + 15) & ~15) + 16;                          // staged row stride
    if (tid < rows) sm.lead[tid] = (int)(reinterpret_cast<uintptr_t>(gout + (int64_t)tid * jb.out_pitch) & 15);
    __syncthreads();
    const int plane = mcu_h * PC;
    for (int i = tid; i < rows * cols; i += kThreads) {
        const int r = i / cols, x = i - r * cols;
        const float* P = &sm.p[r * PC + x];
        unsigned char* d = sm.a + r * rs + sm.lead[r] + x * ch;
        if (ch == 3) {
            uint32_t R, G, B;
            bj::scaled_rgb(P[0], P[plane], P[2 * plane], R, G, B);
            d[0] = (unsigned char)R; d[1] = (unsigned char)G; d[2] = (unsigned char)B;
        } else {
            d[0] = (unsigned char)bj::scaled_u8(P[0]);
        }
    }
    __syncthreads();

    // ---- store: 16-byte chunks of each destination row, partial chunks byte by byte ----------------------------------
    const int nv = (nbytes + 15) / 16 + 1;                               // chunks a row can touch
    for (int i = tid; i < rows * nv; i += kThreads) {
        const int r = i / nv, v = i - r * nv;
        const int lead = sm.lead[r];
        unsigned char* g = gout + (int64_t)r * jb.out_pitch;           // g = 16-byte boundary + lead
        const int lo = 16 * v - lead, hi = lo + 16;                     // chunk v in row bytes: [lo, hi)
        const unsigned char* s = sm.a + r * rs + lead;
        if (lo >= 0 && hi <= nbytes) {
            *reinterpret_cast<uint4*>(g + lo) = *reinterpret_cast<const uint4*>(s + lo);
        } else {
            for (int b = max(lo, 0); b < min(hi, nbytes); b++) g[b] = s[b];
        }
    }
}

}  // namespace

extern "C" bj_status bj_pixels_scaled(const bj_image* images, const bj_scaled_job* jobs, int n_jobs, int max_strips,
                                      const int16_t* coef, const int16_t* qtabs, uint8_t* out, void* stream) {
    static_assert(sizeof(bj_scaled_job) == 24, "bj_scaled_job layout");
    if (!images || !jobs || n_jobs <= 0 || max_strips <= 0 || !coef || !qtabs || !out) return BJ_E_ARG;
    cudaError_t e = cudaFuncSetAttribute(bj_pixels_scaled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)sizeof(Smem));
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_scaled/attr");
    // the job index rides on grid.y (at most 65535): larger batches run as slices (jobs hold absolute offsets)
    for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
        const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
        bj_pixels_scaled_kernel<<<dim3((unsigned)max_strips, (unsigned)n), kThreads, sizeof(Smem), (cudaStream_t)stream>>>(
            images, jobs + j0, coef, qtabs, out);
        e = cudaGetLastError();
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_scaled/launch");
    }
    return BJ_OK;
}
