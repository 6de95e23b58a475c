// bj_pixels_ijg.cu -- libjpeg-turbo-exact pixels (compat="libjpeg-turbo") for a batch of jobs (sm_100a): ISLOW IDCT,
// fancy upsampling across MCU boundaries and table-exact YCbCr -> RGB, bit for bit what libjpeg-turbo's default
// jpeg_read_scanlines writes.  The arithmetic is bj_ijg_math.cuh; see include/b200jpeg.h for the ABI.
//
// Fancy upsampling reads one chroma sample beyond each MCU edge, so the pixels of an MCU depend on its neighbours'
// blocks and the work runs as two launches through a workspace of uint8 sample planes:
//   bj_ijg_idct_kernel    one CTA per MCU row of the job's window (the box's MCUs plus the halo bj::ijg_window adds):
//                         coalesced 16-byte coefficient loads into shared memory, then one thread per block
//                         dequantises, runs ISLOW and writes its 8 x 8 samples into its component's plane
//   bj_ijg_colour_kernel  one CTA per MCU row of the box: one thread per output pixel upsamples every component from
//                         the planes and converts the colour; rows are staged in shared memory and leave through the
//                         funnel-shift store of bj_crop.cuh, so any row alignment works
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_crop.cuh"
#include "bj_ijg_math.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

constexpr int kIdctThreads = 128;      // blocks per load round of bj_ijg_idct_kernel
constexpr int kColThreads = 256;
constexpr int kColChunk = kColThreads; // output pixels per staged row segment of bj_ijg_colour_kernel
constexpr int kStageStride = kColChunk * 3 + 16;

__device__ __constant__ uint8_t c_zigzag_of[64] = {   // natural index (row * 8 + column) -> zig-zag index
    0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30, 41, 43, 9,  11, 18, 24, 31, 40, 44, 53,
    10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

__device__ __forceinline__ int swz(int blk, int chunk) { return blk * 128 + ((chunk ^ (blk & 7)) << 4); }

// Where component c's plane of a job starts in the workspace and how wide it is (include/b200jpeg.h, workspace rule).
struct Planes {
    int mx0, my0, mx1, my1;
    uint64_t off[BJ_MAX_COMP];
    int pw[BJ_MAX_COMP];
};

__device__ __forceinline__ void job_planes(const bj_image& im, const bj_crop_job& jb, Planes& p) {
    bj::ijg_window(im, jb, p.mx0, p.my0, p.mx1, p.my1);
    uint64_t o = (uint64_t)jb.reserved * 256;
    for (int c = 0; c < BJ_MAX_COMP; c++) {
        p.off[c] = o;
        p.pw[c] = (p.mx1 - p.mx0) * 8 * (c < im.ncomp ? im.hs[c] : 0);
        if (c < im.ncomp) o += (uint64_t)p.pw[c] * ((p.my1 - p.my0) * 8 * im.vs[c]);
    }
}

__device__ __forceinline__ void load_image(const bj_image* images, uint32_t i, bj_image& im) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&images[i]);
    if (threadIdx.x < sizeof(bj_image) / 4) reinterpret_cast<uint32_t*>(&im)[threadIdx.x] = src[threadIdx.x];
}

__global__ void __launch_bounds__(kIdctThreads)
bj_ijg_idct_kernel(const bj_image* __restrict__ images, const bj_crop_job* __restrict__ jobs,
                   const int16_t* __restrict__ coef, const int16_t* __restrict__ qtabs, uint8_t* __restrict__ ws) {
    __shared__ __align__(16) unsigned char a[kIdctThreads * 128];
    __shared__ int16_t qt[BJ_MAX_COMP][64];
    __shared__ uint8_t slot_comp[BJ_MAX_SLOTS], slot_bx[BJ_MAX_SLOTS], slot_by[BJ_MAX_SLOTS];
    __shared__ bj_image im;
    const int tid = threadIdx.x;
    const bj_crop_job jb = jobs[blockIdx.y];
    if (jb.log2_scale != 0) return;                       // full-size pixels only (include/b200jpeg.h)
    load_image(images, jb.image, im);
    __syncthreads();
    Planes P;
    job_planes(im, jb, P);
    const int my = P.my0 + (int)blockIdx.x;
    if (my >= P.my1) return;
    for (int i = tid; i < im.ncomp * 64; i += kIdctThreads) qt[i >> 6][i & 63] = qtabs[(size_t)im.qtab[i >> 6] * 64 + (i & 63)];
    if (tid < im.blocks_per_mcu) {
        int c = 0;
        for (int k = 0; k < im.ncomp; k++)
            if (tid >= im.slot0[k]) c = k;
        const int r = tid - im.slot0[c];
        slot_comp[tid] = (uint8_t)c;
        slot_bx[tid] = (uint8_t)(r % im.hs[c]);
        slot_by[tid] = (uint8_t)(r / im.hs[c]);
    }
    const int bpm = im.blocks_per_mcu;
    const int nblk = (P.mx1 - P.mx0) * bpm;
    // the window's blocks of this MCU row are contiguous in the coefficient buffer
    const uint4* g = reinterpret_cast<const uint4*>(coef + ((int64_t)im.coef_block0 + ((int64_t)my * im.mcus_x + P.mx0) * bpm) * 64);
    for (int base = 0; base < nblk; base += kIdctThreads) {
        const int n = min(kIdctThreads, nblk - base);
        __syncthreads();                                 // the previous round's reads of `a` are done
        for (int i = tid; i < n * 8; i += kIdctThreads) *reinterpret_cast<uint4*>(a + swz(i >> 3, i & 7)) = __ldg(g + base * 8 + i);
        __syncthreads();
        if (tid < n) {
            const int b = base + tid, m = b / bpm, s = b - m * bpm;
            const int c = slot_comp[s];
            int d[64], w[64];
            uint8_t smp[64];
#pragma unroll
            for (int k = 0; k < 64; k++) {
                const int z = c_zigzag_of[k];
                d[k] = (int)*reinterpret_cast<const int16_t*>(a + swz(tid, z >> 3) + ((z & 7) << 1)) * (int)qt[c][z];
            }
            bj::ijg_idct_block(d, w, smp);
            const int pw = P.pw[c];
            uint8_t* dst = ws + P.off[c] + (int64_t)((my - P.my0) * 8 * im.vs[c] + slot_by[s] * 8) * pw +
                           (m * im.hs[c] + slot_bx[s]) * 8;
#pragma unroll
            for (int r = 0; r < 8; r++) {
                uint2 v;
                v.x = smp[8 * r] | (smp[8 * r + 1] << 8) | (smp[8 * r + 2] << 16) | ((uint32_t)smp[8 * r + 3] << 24);
                v.y = smp[8 * r + 4] | (smp[8 * r + 5] << 8) | (smp[8 * r + 6] << 16) | ((uint32_t)smp[8 * r + 7] << 24);
                *reinterpret_cast<uint2*>(dst + (int64_t)r * pw) = v;
            }
        }
    }
}

__global__ void __launch_bounds__(kColThreads)
bj_ijg_colour_kernel(const bj_image* __restrict__ images, const bj_crop_job* __restrict__ jobs,
                     const uint8_t* __restrict__ ws, uint8_t* __restrict__ out) {
    __shared__ __align__(16) unsigned char stage[16 * kStageStride];
    __shared__ bj_image im;
    const int tid = threadIdx.x;
    const bj_crop_job jb = jobs[blockIdx.y];
    if (jb.log2_scale != 0) return;                       // full-size pixels only (include/b200jpeg.h)
    load_image(images, jb.image, im);
    __syncthreads();
    Planes P;
    job_planes(im, jb, P);
    const int mh = 8 * im.vmax;
    const int my = (int)jb.y0 / mh + (int)blockIdx.x;
    const int y0 = max(my * mh, (int)jb.y0), y1 = min((my + 1) * mh, (int)jb.y1);
    if (y0 >= y1) return;
    const int rows = y1 - y0;
    const int ch = im.ncomp == 3 ? 3 : 1;
    int rh[BJ_MAX_COMP], rv[BJ_MAX_COMP], dw[BJ_MAX_COMP], dh[BJ_MAX_COMP], ox[BJ_MAX_COMP], oy[BJ_MAX_COMP];
    for (int c = 0; c < BJ_MAX_COMP; c++) {
        const int k = c < im.ncomp ? c : 0;
        rh[c] = im.hmax / im.hs[k];
        rv[c] = im.vmax / im.vs[k];
        dw[c] = (int)((im.width * (uint32_t)im.hs[k] + im.hmax - 1) / im.hmax);
        dh[c] = (int)((im.height * (uint32_t)im.vs[k] + im.vmax - 1) / im.vmax);
        ox[c] = P.mx0 * 8 * im.hs[k];
        oy[c] = P.my0 * 8 * im.vs[k];
    }
    uint8_t* gout0 = out + jb.out_offset + (int64_t)(y0 - (int)jb.y0) * jb.out_pitch;
    // thread t owns column t of each chunk and walks its rows: the column's neighbour decisions are made once
    for (int x0 = (int)jb.x0; x0 < (int)jb.x1; x0 += kColChunk) {
        const int cols = min(kColChunk, (int)jb.x1 - x0);
        if (tid < cols) {
            const int X = x0 + tid;
            for (int r = 0; r < rows; r++) {
                const int Y = y0 + r;
                int v[BJ_MAX_COMP];
#pragma unroll
                for (int c = 0; c < BJ_MAX_COMP; c++) {
                    if (c >= ch) break;
                    const uint8_t* pl = ws + P.off[c];
                    const int pw = P.pw[c], oxc = ox[c], oyc = oy[c];
                    auto at = [pl, pw, oxc, oyc](int sx, int sy) { return (int)__ldg(pl + (uint32_t)((sy - oyc) * pw + (sx - oxc))); };
                    v[c] = bj::ijg_sample(at, X, Y, rh[c], rv[c], dw[c], dh[c]);
                }
                unsigned char* d = stage + r * kStageStride + tid * ch;
                if (ch == 3) {
                    uint32_t R, G, B;
                    bj::ijg_ycc_rgb(v[0], v[1], v[2], R, G, B);
                    d[0] = (unsigned char)R; d[1] = (unsigned char)G; d[2] = (unsigned char)B;
                } else {
                    d[0] = (unsigned char)v[0];
                }
            }
        }
        __syncthreads();
        bj::crop_store(gout0 + (int64_t)(x0 - (int)jb.x0) * ch, jb.out_pitch, stage, kStageStride, 0, cols * ch, rows, tid,
                       kColThreads);
        __syncthreads();
    }
}

}  // namespace

extern "C" bj_status bj_pixels_ijg(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                                   const int16_t* coef, const int16_t* qtabs, uint8_t* workspace, uint8_t* out,
                                   uint32_t kinds, void* stream) {
    if (!images || !jobs || n_jobs <= 0 || max_strips <= 0 || !coef || !qtabs || !workspace || !out) return BJ_E_ARG;
    if (!(kinds & BJ_IJG_ALL) || (kinds & ~(uint32_t)BJ_IJG_ALL)) return BJ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // the job index rides on grid.y (at most 65535): larger batches run as slices (jobs hold absolute offsets)
    for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
        const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
        if (kinds & BJ_IJG_IDCT)
            bj_ijg_idct_kernel<<<dim3((unsigned)max_strips, (unsigned)n), kIdctThreads, 0, st>>>(images, jobs + j0, coef,
                                                                                                  qtabs, workspace);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_ijg/idct");
    }
    for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
        const int n = n_jobs - j0 < 65535 ? n_jobs - j0 : 65535;
        if (kinds & BJ_IJG_COLOUR)
            bj_ijg_colour_kernel<<<dim3((unsigned)max_strips, (unsigned)n), kColThreads, 0, st>>>(images, jobs + j0,
                                                                                                   workspace, out);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_pixels_ijg/colour");
    }
    return BJ_OK;
}
