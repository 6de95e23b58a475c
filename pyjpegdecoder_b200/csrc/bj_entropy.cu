// bj_entropy.cu -- entropy decoding kernels (sm_100a): stream planning, speculative decode,
// chained fix-up + prefix sums, and the writing passes for baseline and progressive scans.
//
// Replaces the entropy half of baseline_dct_scan (jpeg_decoder.py:709-722, :805-866, :898-900) and
// progressive_dct_scan (:908-1304).  The per-thread decode logic lives in bj_entropy.cuh (shared with
// the CPU test-suite); this file is the orchestration:
//
//   plan     one CTA per scan: stream lengths -> subsequences per stream -> first subsequence of
//            every stream (exclusive scan), restart-marker count check.
//   spec     one thread per subsequence: decode from one subsequence early (assumed block start) to
//            obtain a speculative entry state, then the own subsequence: exit state, blocks started,
//            DC difference sums.  The scan's Huffman LUTs are staged in shared memory; the bitstream is
//            read through L1 (every lane walks its own 512-byte region).
//   fix      two launches.  fix_local: each CTA iterates in shared memory until every subsequence's entry
//            equals its predecessor's exit (re-decodes compacted into a dense list per round).  chain: one
//            CTA per scan repairs the CTA boundaries of fix_local in parallel, then computes the segmented
//            exclusive prefix sums (block index and DC predictors per subsequence).  Nothing waits on
//            another CTA.
//   write    baseline: each thread owns the blocks that START in its subsequence, assembles each in a
//            private shared-memory slot and stores it as one 128-byte line -- every block is written
//            exactly once, no memset, no atomics.  Progressive first scans store single coefficients.
//   dc refine / ac refine: see the kernels below.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_entropy.cuh"

extern "C" bj_status bj_set_cuda_error(cudaError_t e, const char* where);

namespace {

using namespace bj;

constexpr int T = BJ_ENTROPY_THREADS;
#ifndef BJ_WRITE_THREADS
#define BJ_WRITE_THREADS 128
#endif
constexpr int TW = BJ_WRITE_THREADS;  // subsequences per CTA of write_kernel (its LUT copy is amortised over more threads)
constexpr int S = BJ_SUBSEQ_BITS;
// Warm-up: 4096 bits synchronise 99.3 % of the entries (the synchronisation distance of the 4:2:0 state averages 823
// bits); with 8192-bit subsequences the speculative pass then decodes every bit 1.5 instead of 2 times.  Measured on the
// full bench (4096 images, 8 streams): S/warm 4096/4096 52.5 ms, 8192/4096 50.1, 8192/3072 50.9, 16384/4096 51.5.
#ifndef BJ_WARM_BITS
#define BJ_WARM_BITS (BJ_SUBSEQ_BITS < 4096 ? BJ_SUBSEQ_BITS : 4096)
#endif
constexpr int kWarm = BJ_WARM_BITS;  // bits decoded ahead of a subsequence to obtain its speculative entry state (<= S)
static_assert(kWarm > 0 && kWarm <= S, "warm-up must not reach further back than one subsequence");
constexpr int kMaxLutSmem = 12288;                  // most LUT entries ever staged in shared memory (48 KB)


struct GlobalSrc {
    const uint32_t* gw;
    uint32_t gn;
    // clamped, not branched: the buffer ends with 64 words of slack, a valid stream never reads past them, and what a
    // corrupt one reads there does not matter as long as it is deterministic
    __device__ __forceinline__ uint32_t word(uint32_t i) const { return __ldg(gw + min(i, gn - 1u)); }
    __device__ __forceinline__ void start(uint32_t) const {}
};

// ---- bitstream staging by a producer warp (write_kernel) ------------------------------------------------
// Every lane of a decoding warp walks its own subsequence, so with 32 lanes refilling their bit windows at different
// symbols some lane misses in (the small) L1 in practically every iteration of the symbol loop and the whole warp
// waits an L2 round trip for it: 42 % of write_kernel's stall samples sat on the first use of the refilled word
// (profiles/r2_full_summary.csv).  A register prefetch cannot hide that (ptxas copies the loop-carried window words at
// the loop head, which reads the load's destination in the same iteration), and per-lane cp.async completion does not
// exist in hardware: wait_group counts per WARP and the mbarrier form of the arrival wants a uniform address.  So one
// extra warp per CTA -- always converged -- copies the bitstream for the decoding threads: 16-byte groups with
// cp.async into a ring of kRing groups per decoding thread, driven by two words of shared memory per thread
// (cons: the group the thread is reading; fill: every group below it has landed).  The decoding threads only ever
// issue LDS.
#ifndef BJ_RING
#define BJ_RING 2
#endif
#ifndef BJ_PRODUCER_SLEEP
#define BJ_PRODUCER_SLEEP 6000
#endif
constexpr int kRing = BJ_RING;  // groups per decoding thread (a power of two)
constexpr uint32_t kConsIdle = 0xFFFFFFFEu, kConsDone = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t lds_volatile(uint32_t a) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_volatile(uint32_t a, uint32_t v) { asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v)); }
// The decoding threads use the weak forms inside `asm volatile` (one access per call, in program order, but no
// .volatile in the PTX): ptxas gives up the reconvergence points of a loop that contains a volatile access -- it
// could be one half of an inter-thread hand-shake -- and the lanes of write_kernel then run their symbol loops and
// block flushes one or two at a time (measured: 2.9x the executed warp instructions).
__device__ __forceinline__ uint32_t lds_weak(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_weak(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v)); }

template <int NT>
struct StagedSrc {
    uint32_t ring;   // shared-space address of this thread's ring: kRing groups of 16 bytes, contiguous
    uint32_t flags;  // shared-space address of cons[t]; fill[t] at flags + NT * 4
    const uint32_t* gw;
    uint32_t gn;
    mutable uint32_t ready;  // the group being read has landed in the ring (a full register: a bool gets packed)
    // No waiting anywhere: a group that has not landed yet (the first one or two of a thread, before the producer has
    // seen it) is read from global memory instead.
    // ONE seek per thread: the reader's look-ahead (BitReader::w2) may already have entered the next group, so a second
    // seek at the reader's own position can land one group back, in a slot the producer has reused by then.
    // write_kernel seeks once; a kernel that seeks twice (spec_kernel) would have to refuse groups below the highest
    // one entered -- measured there, and slower than plain loads anyway (profiles/README.md).
    __device__ __forceinline__ void enter(uint32_t i) const {  // i = first word of the group
        sts_weak(flags, i);
        ready = lds_weak(flags + NT * 4) > i ? 1u : 0u;
    }
    __device__ __forceinline__ void start(uint32_t w) const { enter(w & ~3u); }
    __device__ __forceinline__ uint32_t word(uint32_t i) const {
        if ((i & 3u) == 0u) enter(i);
        if (BJ_UNLIKELY(!ready)) return __ldg(gw + min(i, gn - 1u));
        return lds_weak(ring + ((i & (4u * kRing - 1u)) << 2));
    }
    __device__ __forceinline__ void done() const { sts_weak(flags, kConsDone); }
};

// shared memory of the staging: NT * (kRing * 4 + 2) words, 16-byte aligned
template <int NT>
__device__ __forceinline__ StagedSrc<NT> staged_src(uint32_t* stage, int t, const uint32_t* gw, uint32_t gn) {
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(stage);
    return StagedSrc<NT>{base + 16u * kRing * t, base + NT * kRing * 16 + 4u * t, gw, gn, 0u};
}
template <int NT>
__device__ __forceinline__ void staged_init(uint32_t* stage, int tid, int nthreads) {
    for (int i = tid; i < NT; i += nthreads) {
        stage[NT * kRing * 4 + i] = kConsIdle;
        stage[NT * kRing * 4 + NT + i] = 0u;
    }
}

// The producer warp: lane l serves the decoding threads l, l + 32, ...  Runs until all of them are done.
// cons[t] = first word of the group thread t is reading; fill[t] = every word below it has landed.
template <int NT>
__device__ __forceinline__ void staged_producer(uint32_t* stage, const uint32_t* __restrict__ gw, uint32_t gmax, int lane) {
    constexpr int PER = NT / 32;
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(stage);
    const uint32_t cons0 = base + NT * kRing * 16, fill0 = cons0 + NT * 4;
    uint32_t req[PER];  // next group to request for each of my threads (valid once the thread has started)
    bool live[PER];
#pragma unroll
    for (int k = 0; k < PER; k++) {
        req[k] = 0;
        live[k] = false;
    }
    for (;;) {
        bool all_done = true, issued = false;
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const int t = lane + 32 * k;
            const uint32_t cw = lds_volatile(cons0 + 4u * t);
            if (cw == kConsDone) continue;
            all_done = false;
            if (cw == kConsIdle) continue;
            const uint32_t c = cw >> 2;
            if (!live[k]) {
                live[k] = true;
                req[k] = c;
            }
#pragma unroll
            for (int j = 0; j < 2; j++) {  // at most two groups per thread and round
                if (req[k] < c + kRing) {
                    const uint32_t* p = gw + 4 * (size_t)min(req[k], gmax);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(base + (t * kRing + (req[k] & (kRing - 1))) * 16u), "l"(p) : "memory");
                    req[k]++;
                    issued = true;
                }
            }
        }
        if (__all_sync(0xFFFFFFFFu, all_done)) break;
        if (__any_sync(0xFFFFFFFFu, issued)) {
            asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;\n\tfence.acq_rel.cta;" ::: "memory");
#pragma unroll
            for (int k = 0; k < PER; k++)
                if (live[k]) sts_volatile(fill0 + 4u * (lane + 32 * k), req[k] << 2);
        }
        // One round every few microseconds is plenty (a decoding thread takes ~20 us per group; one that is faster
        // than the producer reads that group from global memory) and keeps the producer's polling out of the issue
        // slots of the decoding warps: 2 us -> 2.04 ms, 4 us -> 1.97, 8 us -> 1.96, 16 us -> 2.11 per 512 images.
        __nanosleep(BJ_PRODUCER_SLEEP);
    }
}

// Per-CTA scan context + the scan's Huffman LUTs (the bitstream itself is read through L1)
struct CtaShared {
    bj_scan sc;
    ScanCtx ctx;
    uint32_t scan_nsub;
    uint32_t lut_cap;
    uint32_t lut_in_smem;
    uint32_t lut[1];  // lut_cap entries follow
};

// The fix-up kernel is latency bound (a few subsequences are re-decoded per round), so it trades the
// shared-memory copies of the bit window and the LUTs for occupancy: it reads both through L1.
struct CtaSharedLite {
    bj_scan sc;
    ScanCtx ctx;
    uint32_t scan_nsub;
};

// ---- helpers -------------------------------------------------------------------------------------
template <class SH>
__device__ __forceinline__ void load_scan_header(SH& sh, const bj_scan* scans, int idx, const bj_entropy_buffers& B) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&scans[idx]);
    for (int i = threadIdx.x; i < (int)(sizeof(bj_scan) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(&sh.sc)[i] = src[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        const bj_scan& sc = sh.sc;
        for (int i = 0; i < BJ_MAX_SLOTS; i++) {
            sh.ctx.dc_tab[i] = sc.slot_dc[i];
            sh.ctx.ac_tab[i] = sc.slot_ac[i];
            sh.ctx.slot_comp[i] = sc.slot_comp[i];
        }
        ctx_finish(sh.ctx);
        sh.ctx.nslots = sc.nslots;
        sh.ctx.ss = sc.ss;
        sh.ctx.se = sc.se;
        sh.ctx.al = sc.al;
        // total subsequences of the scan = first subsequence of the last stream + its own count
        uint32_t last = sc.stream0 + sc.n_streams - 1;
        uint64_t bits = (B.stream_end[last] - B.stream_start[last]) * 8;
        sh.scan_nsub = B.stream_sub[last] + (uint32_t)((bits + S - 1) / S);
    }
    __syncthreads();
}

template <class SH>
__device__ __forceinline__ void load_scan(SH& sh, const bj_scan* scans, int idx, const bj_entropy_buffers& B,
                                          uint32_t lut_cap) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&scans[idx]);
    for (int i = threadIdx.x; i < (int)(sizeof(bj_scan) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(&sh.sc)[i] = src[i];
    __syncthreads();
    const bj_scan& sc = sh.sc;
    const bool in_smem = sc.lut_len <= lut_cap;
    if (in_smem)
        for (uint32_t i = threadIdx.x; i < sc.lut_len; i += blockDim.x) sh.lut[i] = __ldg(B.lut + sc.lut_off + i);
    if (threadIdx.x == 0) {
        sh.lut_in_smem = in_smem ? 1u : 0u;
        for (int i = 0; i < BJ_MAX_SLOTS; i++) {
            sh.ctx.dc_tab[i] = sc.slot_dc[i];
            sh.ctx.ac_tab[i] = sc.slot_ac[i];
            sh.ctx.slot_comp[i] = sc.slot_comp[i];
        }
        ctx_finish(sh.ctx);
        sh.ctx.nslots = sc.nslots;
        sh.ctx.ss = sc.ss;
        sh.ctx.se = sc.se;
        sh.ctx.al = sc.al;
        // total subsequences of the scan = first subsequence of the last stream + its own count
        uint32_t last = sc.stream0 + sc.n_streams - 1;
        uint64_t bits = (B.stream_end[last] - B.stream_start[last]) * 8;
        sh.scan_nsub = B.stream_sub[last] + (uint32_t)((bits + S - 1) / S);
    }
    __syncthreads();
}

struct SubInfo {
    bool valid;
    uint32_t stream;     // absolute stream index
    uint32_t l;          // subsequence index inside the stream
    uint64_t b0, b1;     // stream bit range
    uint64_t own, stop;  // own bit range (absolute)
    uint32_t own_rel, stop_rel, end_rel;  // the same relative to b0
    uint32_t nblk_stream;
    uint32_t mcu0;       // first MCU of the stream
};

template <class SH>
__device__ __forceinline__ SubInfo locate(const SH& sh, const bj_entropy_buffers& B, uint32_t lscan) {
    SubInfo s;
    const bj_scan& sc = sh.sc;
    s.valid = lscan < sh.scan_nsub;
    if (!s.valid) return s;
    // last stream m with stream_sub[m] <= lscan
    uint32_t lo = 0, hi = sc.n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (B.stream_sub[sc.stream0 + mid] <= lscan) lo = mid;
        else hi = mid - 1;
    }
    s.stream = sc.stream0 + lo;
    s.l = lscan - B.stream_sub[s.stream];
    s.b0 = B.stream_start[s.stream] * 8;
    s.b1 = B.stream_end[s.stream] * 8;
    s.own = s.b0 + (uint64_t)s.l * S;
    s.stop = min(s.own + (uint64_t)S, s.b1);
    s.own_rel = s.l * S;
    s.end_rel = (uint32_t)(s.b1 - s.b0);
    s.stop_rel = min(s.own_rel + (uint32_t)S, s.end_rel);
    s.mcu0 = lo * sc.ri;
    uint32_t mcus = min(sc.ri, sc.n_mcu - s.mcu0);
    s.nblk_stream = mcus * sc.nslots;
    if (s.own >= s.b1) s.valid = false;  // (cannot happen: nsub = ceil(bits / S))
    return s;
}

// Decode one subsequence from entry state st: exit state + counts.  `lut` must be passed with visible
// provenance (sh.lut -> LDS, or a global pointer).
template <class Src>
__device__ __forceinline__ void run_sub_core(int mode, const ScanCtx& ctx, const uint32_t* lut, const Src& src, uint64_t b0,
                                             uint32_t own_rel, uint32_t stop_rel, uint32_t end_rel, uint64_t st, uint64_t& ex,
                                             SubCount& k) {
    BitReader<Src> rd;
    rd.seek(&src, b0, (uint32_t)(state_pos(st) - b0));
    int z = state_z(st), slot = state_slot(st);
    k.blocks = 0;
    k.dc[0] = k.dc[1] = k.dc[2] = 0;
    if (mode == BJ_MODE_BASELINE) sync_run<BJ_M_BASE>(rd, z, slot, ctx, lut, own_rel, stop_rel, end_rel, k);
    else if (mode == BJ_MODE_DC_FIRST) sync_run<BJ_M_DCFIRST>(rd, z, slot, ctx, lut, own_rel, stop_rel, end_rel, k);
    else {
        struct NoSink { __device__ void store(uint32_t, int, int16_t) {} } ns;
        uint32_t blk = 0, adv = 0;
        acfirst_run<false>(rd, z, ctx, lut, own_rel, stop_rel, end_rel, blk, 0xFFFFFFFFu, adv, ns);
        k.blocks = adv;
    }
    ex = pack_state(rd.abs_pos(), z, slot);
}

template <class SH, class Src>
__device__ __forceinline__ void run_sub(const SH& sh, const bj_entropy_buffers& B, const Src& src, uint64_t b0,
                                        uint32_t own_rel, uint32_t stop_rel, uint32_t end_rel, uint64_t st, uint64_t& ex,
                                        SubCount& k) {
    if (sh.lut_in_smem) run_sub_core(sh.sc.mode, sh.ctx, sh.lut, src, b0, own_rel, stop_rel, end_rel, st, ex, k);
    else run_sub_core(sh.sc.mode, sh.ctx, B.lut + sh.sc.lut_off, src, b0, own_rel, stop_rel, end_rel, st, ex, k);
}

// ---- plan ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) plan_kernel(const bj_scan* __restrict__ scans, int scan_first,
                                                   const uint64_t* __restrict__ tile_sum, bj_entropy_buffers B) {
    const bj_scan& sc = scans[scan_first + blockIdx.x];
    __shared__ uint32_t part[256];
    __shared__ uint32_t carry;
    __shared__ int bad;
    if (threadIdx.x == 0) { carry = 0; bad = 0; }
    __syncthreads();
    const uint32_t n_tiles = ((uint32_t)(sc.raw_off & 15) + sc.raw_len + BJ_UNSTUFF_TILE - 1) / BJ_UNSTUFF_TILE;
    const uint64_t scan_end = tile_sum[sc.tile0 + (n_tiles ? n_tiles : 1)] & ((1ull << 40) - 1);
    for (uint32_t base = 0; base < sc.n_streams; base += 256) {
        uint32_t m = base + threadIdx.x;
        uint32_t nsub = 0;
        uint64_t st = 0, en = 0;
        if (m < sc.n_streams) {
            st = B.stream_start[sc.stream0 + m];
            en = (m + 1 < sc.n_streams) ? B.stream_start[sc.stream0 + m + 1] : scan_end;
            if (st == ~0ull || en == ~0ull || en < st) {  // restart marker missing
                bad = 1;
                st = en = scan_end;
            }
            nsub = (uint32_t)(((en - st) * 8 + S - 1) / S);
        }
        part[threadIdx.x] = nsub;
        __syncthreads();
        for (int o = 1; o < 256; o <<= 1) {
            uint32_t a = (threadIdx.x >= (unsigned)o) ? part[threadIdx.x - o] : 0;
            __syncthreads();
            part[threadIdx.x] += a;
            __syncthreads();
        }
        if (m < sc.n_streams) {
            B.stream_start[sc.stream0 + m] = st;
            B.stream_end[sc.stream0 + m] = en;
            B.stream_sub[sc.stream0 + m] = carry + part[threadIdx.x] - nsub;
        }
        __syncthreads();
        if (threadIdx.x == 255) carry += part[255];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (bad) atomicOr(&B.err[sc.image], BJ_ERR_RST_COUNT);
        if (carry > sc.n_sub_max) atomicOr(&B.err[sc.image], BJ_ERR_SYNC);
    }
}

// ---- speculative pass ------------------------------------------------------------------------------
__global__ void __launch_bounds__(T) spec_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B,
                                                 uint32_t lut_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CtaShared& sh = *reinterpret_cast<CtaShared*>(smem_raw);
    load_scan(sh, scans, scan_first + blockIdx.x, B, lut_cap);
    const uint32_t base = blockIdx.y * T;
    if (base >= sh.scan_nsub) return;
    const uint32_t lscan = base + threadIdx.x;
    SubInfo si = locate(sh, B, lscan);
    if (!si.valid) return;
    GlobalSrc src{B.words, (uint32_t)B.words_len};
    const int z0 = (sh.sc.mode == BJ_MODE_AC_FIRST) ? sh.sc.ss : 0;
    uint64_t st;
    if (si.l == 0) st = pack_state(si.b0, z0, 0);
    else {
        uint64_t ex;
        SubCount k;  // nothing is counted while warming up (own_rel = 0xFFFFFFFF)
        run_sub(sh, B, src, si.b0, 0xFFFFFFFFu, si.own_rel, si.end_rel, pack_state(si.own - kWarm, z0, 0), ex, k);
        st = ex;
    }
    uint64_t ex;
    SubCount k;
    run_sub(sh, B, src, si.b0, si.own_rel, si.stop_rel, si.end_rel, st, ex, k);
    const size_t g = (size_t)sh.sc.sub0 + lscan;
    B.sub_entry[g] = st;
    B.sub_exit[g] = ex;
    reinterpret_cast<uint4*>(B.sub_count)[g] = make_uint4(k.blocks, (uint32_t)k.dc[0], (uint32_t)k.dc[1], (uint32_t)k.dc[2]);
}

// ---- fix-up, stage 1: CTA-local convergence -----------------------------------------------------------
// Each CTA iterates (shared memory) until every subsequence's entry state equals its predecessor's
// exit state, taking the speculative entry of its own first subsequence as given.  Re-decodes are
// COMPACTED: in every round the subsequences whose entry changed are collected into a dense list and
// decoded by the first threads of the CTA, so warps stay full even when few subsequences need work.
// The kernel is latency bound, so it reads the bitstream and the LUTs through L1 instead of staging
// them (7.7 KB of shared memory per CTA -> 16 CTAs per SM).
__global__ void __launch_bounds__(T, 16) fix_local_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B) {
    __shared__ CtaSharedLite sh;
    __shared__ uint64_t s_entry[T], s_exit[T];
    __shared__ uint64_t s_b0[T];
    __shared__ uint32_t s_ownr[T], s_stopr[T], s_endr[T];
    __shared__ uint32_t s_cnt[T][4];
    __shared__ uint16_t s_list[T];
    __shared__ uint32_t s_wcount[T / 32];
    load_scan_header(sh, scans, scan_first + blockIdx.x, B);
    const uint32_t base = blockIdx.y * T;
    if (base >= sh.scan_nsub) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lscan = base + tid;
    SubInfo si = locate(sh, B, lscan);
    GlobalSrc src{B.words, (uint32_t)B.words_len};
    const uint32_t* const glut = B.lut + sh.sc.lut_off;
    const size_t g = (size_t)sh.sc.sub0 + lscan;
    {
        uint64_t entry = 0, ex = 0;
        uint4 c = make_uint4(0, 0, 0, 0);
        if (si.valid) {
            entry = B.sub_entry[g];
            ex = B.sub_exit[g];
            c = reinterpret_cast<const uint4*>(B.sub_count)[g];
        }
        s_entry[tid] = entry;
        s_exit[tid] = ex;
        s_cnt[tid][0] = c.x; s_cnt[tid][1] = c.y; s_cnt[tid][2] = c.z; s_cnt[tid][3] = c.w;
        s_b0[tid] = si.b0; s_ownr[tid] = si.own_rel; s_stopr[tid] = si.stop_rel; s_endr[tid] = si.end_rel;
    }
    const bool head = si.valid && si.l == 0;  // entry state known exactly
    uint32_t changes = 0;
    bool dirty = false;
    __syncthreads();
    for (;;) {
        bool need = false;
        uint64_t want = 0;
        if (si.valid && !head && tid > 0) {  // thread 0's entry stays speculative here (chain_kernel checks it)
            want = s_exit[tid - 1];
            need = s_entry[tid] != want;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, need);
        if (lane == 0) s_wcount[warp] = __popc(bal);
        __syncthreads();
        uint32_t off = 0, total = 0;
#pragma unroll
        for (int w = 0; w < T / 32; w++) {
            uint32_t cw = s_wcount[w];
            if (w < warp) off += cw;
            total += cw;
        }
        if (total == 0) break;
        if (need) {
            s_entry[tid] = want;
            s_list[off + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)tid;
            dirty = true;
        }
        __syncthreads();
        if ((uint32_t)tid < total) {  // dense: item i is decoded by thread i
            const int j = s_list[tid];
            uint64_t ex;
            SubCount k;
            run_sub_core(sh.sc.mode, sh.ctx, glut, src, s_b0[j], s_ownr[j], s_stopr[j], s_endr[j], s_entry[j], ex, k);
            s_exit[j] = ex;
            s_cnt[j][0] = k.blocks; s_cnt[j][1] = (uint32_t)k.dc[0]; s_cnt[j][2] = (uint32_t)k.dc[1]; s_cnt[j][3] = (uint32_t)k.dc[2];
            changes++;
        }
        __syncthreads();
    }
    if (si.valid && dirty) {
        B.sub_entry[g] = s_entry[tid];
        B.sub_exit[g] = s_exit[tid];
        reinterpret_cast<uint4*>(B.sub_count)[g] = make_uint4(s_cnt[tid][0], s_cnt[tid][1], s_cnt[tid][2], s_cnt[tid][3]);
    }
    if (changes && B.sync_changes) atomicAdd(B.sync_changes, changes);
}

// ---- fix-up, stage 2: one CTA per scan --------------------------------------------------------------------
// After stage 1 the only places where an entry state can still differ from its predecessor's exit are the
// CTA boundaries of stage 1 (every T-th subsequence).  Thread i owns boundaries (i + 1) * T + k * kChainThreads
// * T; on a mismatch it re-decodes forward from the corrected state until the exit state matches the stored
// entry of the next subsequence, never beyond its own range of T subsequences (so threads never race); a
// correction that reaches the end of a range is picked up by the owner of the next boundary in the next pass.
// Passes repeat until nothing mismatches.  Then warp 0 computes the segmented exclusive prefix sums (first block
// index and DC predictors per subsequence; segments = streams, their heads marked in a shared-memory bitmap).
// Nothing waits on another CTA: all scans of the batch are repaired concurrently.
constexpr int kChainThreads = 128;

__global__ void __launch_bounds__(kChainThreads) chain_kernel(const bj_scan* __restrict__ scans, int scan_first, int n_scans,
                                                              bj_entropy_buffers B, uint32_t bitmap_words, uint32_t lut_cap) {
    extern __shared__ uint32_t s_heads[];  // bitmap_words words (0: scans with several streams fall back to a binary search)
    uint32_t* const s_lut = s_heads + bitmap_words;  // lut_cap words: the scan's Huffman LUTs when they fit
    __shared__ CtaSharedLite sh;
    const int tid = threadIdx.x, lane = tid & 31;
    if ((int)blockIdx.x >= n_scans) return;
    load_scan_header(sh, scans, scan_first + blockIdx.x, B);
    const uint32_t nsub = sh.scan_nsub;
    const size_t g0 = sh.sc.sub0;
    const uint32_t n_streams = sh.sc.n_streams;
    const bool use_bitmap = n_streams > 1 && (nsub + 31) / 32 <= bitmap_words;
    const bool lut_in_smem = sh.sc.lut_len <= lut_cap;
    if (lut_in_smem)
        for (uint32_t i = tid; i < sh.sc.lut_len; i += kChainThreads) s_lut[i] = __ldg(B.lut + sh.sc.lut_off + i);
    if (use_bitmap) {
        for (uint32_t i = tid; i < (nsub + 31) / 32; i += kChainThreads) s_heads[i] = 0u;
        __syncthreads();
        for (uint32_t m = tid; m < n_streams; m += kChainThreads) {
            const uint32_t l = B.stream_sub[sh.sc.stream0 + m];
            if (l < nsub) atomicOr(&s_heads[l >> 5], 1u << (l & 31));
        }
    }
    __syncthreads();
    {
        GlobalSrc src{B.words, (uint32_t)B.words_len};
        const uint32_t* const glut = B.lut + sh.sc.lut_off;
        uint32_t repairs = 0;
        for (;;) {
            bool any = false;
            for (uint32_t lb0 = T; lb0 < nsub; lb0 += kChainThreads * T) {
                const uint32_t lb = lb0 + tid * T;
                if (lb < nsub) {
                    uint32_t cur = lb;
                    uint64_t st = B.sub_exit[g0 + cur - 1];
                    if (B.sub_entry[g0 + cur] != st) {
                        const uint32_t lim = min(lb + (uint32_t)T, nsub);
                        for (;;) {
                            SubInfo si = locate(sh, B, cur);
                            if (!si.valid || si.l == 0) break;  // a stream head has a known entry state
                            B.sub_entry[g0 + cur] = st;
                            uint64_t ex;
                            SubCount k;
                            if (lut_in_smem) run_sub_core(sh.sc.mode, sh.ctx, s_lut, src, si.b0, si.own_rel, si.stop_rel, si.end_rel, st, ex, k);
                            else run_sub_core(sh.sc.mode, sh.ctx, glut, src, si.b0, si.own_rel, si.stop_rel, si.end_rel, st, ex, k);
                            B.sub_exit[g0 + cur] = ex;
                            reinterpret_cast<uint4*>(B.sub_count)[g0 + cur] =
                                make_uint4(k.blocks, (uint32_t)k.dc[0], (uint32_t)k.dc[1], (uint32_t)k.dc[2]);
                            repairs++;
                            any = true;
                            cur++;
                            if (cur >= lim || B.sub_entry[g0 + cur] == ex) break;
                            st = ex;
                        }
                    }
                }
            }
            __threadfence_block();
            if (!__syncthreads_or(any ? 1 : 0)) break;
        }
        if (repairs && B.sync_changes) atomicAdd(B.sync_changes, repairs);
    }
    __syncthreads();
    // Segmented exclusive prefix sums (segments = streams): every thread owns a contiguous chunk of the scan's
    // subsequences; chunk totals go through shared memory; the chunk is walked a second time to write.
    __shared__ uint32_t s_part[kChainThreads][4];
    __shared__ uint32_t s_seen[kChainThreads];
    auto is_head = [&](uint32_t l) -> bool {
        if (l == 0) return true;
        if (n_streams <= 1) return false;
        if (use_bitmap) return (s_heads[l >> 5] >> (l & 31)) & 1u;
        uint32_t lo = 0, hi = n_streams - 1;  // stream_sub is increasing
        while (lo < hi) {
            uint32_t mid = (lo + hi + 1) >> 1;
            if (B.stream_sub[sh.sc.stream0 + mid] <= l) lo = mid;
            else hi = mid - 1;
        }
        return B.stream_sub[sh.sc.stream0 + lo] == l;
    };
    const uint32_t chunk = (nsub + kChainThreads - 1) / kChainThreads;
    const uint32_t c_lo = min((uint32_t)tid * chunk, nsub), c_hi = min(c_lo + chunk, nsub);
    const uint4* cnt = reinterpret_cast<const uint4*>(B.sub_count) + g0;
    {
        uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0, seen = 0;
        for (uint32_t l = c_lo; l < c_hi; l++) {
            const uint4 c = cnt[l];
            if (is_head(l)) {
                r0 = r1 = r2 = r3 = 0;
                seen = 1;
            }
            r0 += c.x; r1 += c.y; r2 += c.z; r3 += c.w;
        }
        s_part[tid][0] = r0; s_part[tid][1] = r1; s_part[tid][2] = r2; s_part[tid][3] = r3;
        s_seen[tid] = seen;
    }
    __syncthreads();
    uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0;
    for (int p = tid - 1; p >= 0; p--) {  // back to the latest chunk that contains a stream head
        r0 += s_part[p][0]; r1 += s_part[p][1]; r2 += s_part[p][2]; r3 += s_part[p][3];
        if (s_seen[p]) break;
    }
    uint4* pre = reinterpret_cast<uint4*>(B.sub_prefix) + g0;
    for (uint32_t l = c_lo; l < c_hi; l++) {
        const uint4 c = cnt[l];
        if (is_head(l)) r0 = r1 = r2 = r3 = 0;
        pre[l] = make_uint4(r0, r1, r2, r3);
        r0 += c.x; r1 += c.y; r2 += c.z; r3 += c.w;
    }
}

// ---- writing pass ------------------------------------------------------------------------------------
__device__ __forceinline__ size_t block_address(const bj_scan& sc, uint32_t mcu, int slot) {
    if (sc.interleaved) return (size_t)sc.coef_block0 + (size_t)mcu * sc.frame_bpm + sc.slot_frame[slot];
    uint32_t by = mcu / sc.mcus_x, bx = mcu - by * sc.mcus_x;
    uint32_t fm = (by / sc.comp_v) * sc.frame_mcus_x + bx / sc.comp_h;
    return (size_t)sc.coef_block0 + (size_t)fm * sc.frame_bpm + sc.comp_slot0 + (by % sc.comp_v) * sc.comp_h + (bx % sc.comp_h);
}

// Baseline block sink: the thread's block lives in shared memory as 8 chunks of 16 bytes, chunk c of
// thread t at (c * TW + t) * 16: conflict-free 128-bit reads when the block is flushed.
struct SmemBlockSink {
    unsigned char* base;  // buf + tid * 16
    int16_t* coef;
    const bj_scan* sc;
    uint32_t mcu0;
    uint32_t mcu_next;  // MCU of the next block to commit (0xFFFFFFFF: not known yet)
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void put(int z, int16_t v) {
        *reinterpret_cast<int16_t*>(base + (z >> 3) * (TW * 16) + ((z & 7) << 1)) = v;
    }
    __device__ __forceinline__ void commit(uint32_t blk, int slot) {
        // blocks are committed in order: the MCU index is tracked instead of divided out for every block
        if (mcu_next == 0xFFFFFFFFu) mcu_next = mcu0 + blk / sc->nslots;
        const uint32_t mcu = mcu_next;
        if (slot + 1 == (int)sc->nslots) mcu_next++;
        uint4* dst = reinterpret_cast<uint4*>(coef + block_address(*sc, mcu, slot) * 64);
        const uint4 zero = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int c = 0; c < 8; c++) {
            uint4* s = reinterpret_cast<uint4*>(base + c * (TW * 16));
            uint4 v = *s;
            *s = zero;
            dst[c] = v;
        }
    }
};

struct GlobalCoefSink {  // progressive first scans: single coefficient stores
    int16_t* coef;
    const bj_scan* sc;
    uint32_t mcu0;
    __device__ __forceinline__ void store_dc(uint32_t blk, int slot, int16_t v) {
        uint32_t mcu = mcu0 + blk / sc->nslots;
        coef[block_address(*sc, mcu, slot) * 64] = v;
    }
    __device__ __forceinline__ void store(uint32_t blk, int z, int16_t v) {
        coef[block_address(*sc, mcu0 + blk, 0) * 64 + z] = v;
    }
};

__global__ void __launch_bounds__(TW + 32) write_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B,
                                                       uint32_t lut_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CtaShared& sh = *reinterpret_cast<CtaShared*>(smem_raw);
    __shared__ __align__(16) uint32_t s_blocks[TW * 32];
    __shared__ __align__(16) uint32_t s_stage[TW * (kRing * 4 + 2)];
    load_scan(sh, scans, scan_first + blockIdx.x, B, lut_cap);
    const uint32_t base = blockIdx.y * TW;
    if (base >= sh.scan_nsub) return;
    const int tid = threadIdx.x;
    for (int i = tid; i < TW * 32; i += TW + 32) s_blocks[i] = 0u;
    staged_init<TW>(s_stage, tid, TW + 32);
    __syncthreads();
    if (tid >= TW) {  // the producer warp
        staged_producer<TW>(s_stage, B.words, (uint32_t)(B.words_len >> 2) - 1u, tid - TW);
        return;
    }
    typedef StagedSrc<TW> SrcT;
    const SrcT src = staged_src<TW>(s_stage, tid, B.words, (uint32_t)B.words_len);
    const uint32_t lscan = base + tid;
    SubInfo si = locate(sh, B, lscan);
    if (!si.valid) {
        src.done();
        return;
    }
    const size_t g = (size_t)sh.sc.sub0 + lscan;
    const uint64_t st = B.sub_entry[g];
    const uint4 pre = reinterpret_cast<const uint4*>(B.sub_prefix)[g];
    BitReader<SrcT> rd;
    rd.seek(&src, si.b0, (uint32_t)(state_pos(st) - si.b0));
    int z = state_z(st), slot = state_slot(st);
    uint32_t blk = pre.x;
    int pred[3] = {(int)pre.y, (int)pre.z, (int)pre.w};
    uint32_t err = 0;
    const int mode = sh.sc.mode;
    const bool ls = sh.lut_in_smem != 0;
    const uint32_t* glut = B.lut + sh.sc.lut_off;
    if (mode == BJ_MODE_BASELINE) {
        SmemBlockSink sink{reinterpret_cast<unsigned char*>(s_blocks) + tid * 16, B.coef, &sh.sc, si.mcu0, 0xFFFFFFFFu};
        if (ls) err = base_write_run(rd, z, slot, sh.ctx, sh.lut, si.stop_rel, si.end_rel, blk, si.nblk_stream, pred, sink);
        else err = base_write_run(rd, z, slot, sh.ctx, glut, si.stop_rel, si.end_rel, blk, si.nblk_stream, pred, sink);
    } else if (mode == BJ_MODE_DC_FIRST) {
        GlobalCoefSink sink{B.coef, &sh.sc, si.mcu0};
        if (ls) err = dcfirst_write_run(rd, slot, sh.ctx, sh.lut, si.stop_rel, si.end_rel, blk, si.nblk_stream, pred, sink);
        else err = dcfirst_write_run(rd, slot, sh.ctx, glut, si.stop_rel, si.end_rel, blk, si.nblk_stream, pred, sink);
    } else {
        GlobalCoefSink sink{B.coef, &sh.sc, si.mcu0};
        uint32_t adv = 0;
        if (ls) err = acfirst_run<true>(rd, z, sh.ctx, sh.lut, si.own_rel, si.stop_rel, si.end_rel, blk, si.nblk_stream, adv, sink);
        else err = acfirst_run<true>(rd, z, sh.ctx, glut, si.own_rel, si.stop_rel, si.end_rel, blk, si.nblk_stream, adv, sink);
    }
    src.done();
    // the last subsequence of a stream checks that the stream held all its blocks
    if (si.stop == si.b1) {
        uint4 c = reinterpret_cast<const uint4*>(B.sub_count)[g];
        if (pre.x + c.x < si.nblk_stream) err |= BJ_ERR_OVERRUN;
    }
    if (err) atomicOr(&B.err[sh.sc.image], err);
}

// ---- DC refinement (:1036-1043): bit b of a stream belongs to its block b -----------------------------
__global__ void __launch_bounds__(256) dcrefine_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B) {
    const bj_scan& sc = scans[scan_first + blockIdx.y];
    const uint32_t total = sc.n_mcu * sc.nslots;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        uint32_t mcu = i / sc.nslots;
        int slot = (int)(i - mcu * sc.nslots);
        uint32_t m = mcu / sc.ri;
        uint32_t b = i - m * sc.ri * sc.nslots;
        uint64_t bit = B.stream_start[sc.stream0 + m] * 8 + b;
        if (bit >= B.stream_end[sc.stream0 + m] * 8) {
            atomicOr(&B.err[sc.image], BJ_ERR_OVERRUN);
            continue;
        }
        uint32_t v = (__ldg(B.words + (bit >> 5)) >> (31 - (uint32_t)(bit & 31))) & 1u;
        int16_t* c = B.coef + block_address(sc, mcu, slot) * 64;
        *c = (int16_t)(*c | (int16_t)(v << sc.al));
    }
}

// ---- AC refinement: sequential parse per stream + parallel apply per block (see bj_entropy.cuh) ---------
// Non-zero history of a 128-byte block: eight 128-bit loads.
__device__ __forceinline__ void load_block(const int16_t* blk, uint4 (&v)[8]) {
    const uint4* q = reinterpret_cast<const uint4*>(blk);
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = q[i];
}
__device__ __forceinline__ uint64_t block_mask(const uint4 (&v)[8]) {
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t w[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
        uint32_t b = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            b |= ((w[j] & 0xFFFFu) ? 1u : 0u) << (2 * j);
            b |= ((w[j] >> 16) ? 1u : 0u) << (2 * j + 1);
        }
        if (i < 4) lo |= b << (8 * i);
        else hi |= b << (8 * (i - 4));
    }
    return ((uint64_t)hi << 32) | lo;
}

// One warp per stream.  The warp pre-decodes a window of the bitstream (one candidate symbol per bit position, all
// lanes), stages the masks of the next 32 blocks (their loads are issued one chunk ahead), turns them into the
// per-block landing tables, then lane 0 chases the chain through window and tables (bj_entropy.cuh) and all lanes
// store the start positions.  The window is rebuilt whenever the next block could run past its end.
__global__ void __launch_bounds__(32) acrefine_parse_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B,
                                                            uint32_t lut_cap, uint32_t win_bits) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CtaShared& sh = *reinterpret_cast<CtaShared*>(smem_raw);
    // the pre-decoded window follows the LUT in dynamic shared memory: win_bits entries (the host picks a small window
    // for waves with many short streams -- restart intervals -- so that many of these one-warp CTAs fit an SM)
    uint32_t* const s_pre = reinterpret_cast<uint32_t*>(smem_raw + ((sizeof(CtaShared) + sizeof(uint32_t) * lut_cap + 15) & ~(size_t)15));
    __shared__ __align__(4) uint8_t s_tab[32 * BJ_ACR_TAB_STRIDE];
    __shared__ uint32_t s_pos[32];
    __shared__ uint32_t s_state[4];   // pos, eob_run, next block, err (lane 0 -> warp)
    load_scan(sh, scans, scan_first + blockIdx.y, B, lut_cap);
    const bj_scan& sc = sh.sc;
    const uint32_t m = blockIdx.x;
    if (m >= sc.n_streams) return;
    const int lane = threadIdx.x;
    GlobalSrc src{B.words, (uint32_t)B.words_len};
    const uint64_t sb0 = B.stream_start[sc.stream0 + m] * 8, sb1 = B.stream_end[sc.stream0 + m] * 8;
    const uint32_t end_rel = (uint32_t)(sb1 - sb0);
    const uint32_t mcu0 = m * sc.ri;
    const uint32_t nblk = min(sc.ri, sc.n_mcu - mcu0);
    const bool ls = sh.lut_in_smem != 0;  // two call sites: shared-memory loads for the common case, not generic ones
    const uint32_t* gtab = B.lut + sc.lut_off + sh.ctx.ac_tab[0];
    const uint32_t* stab = sh.lut + sh.ctx.ac_tab[0];
    const int ss = sh.ctx.ss, se = sh.ctx.se;
    uint32_t win_base = 0;
    auto build_window = [&](uint32_t base) {
        win_base = base;
        // positions past the end of the stream (+ slack for a corrupt tail) are never visited
        const uint32_t n = min(win_bits, end_rel + 64u > base ? end_rel + 64u - base : 0u);
        if (ls) for (uint32_t k = lane; k < n; k += 32) s_pre[k] = acrefine_predecode(src, sb0 + base + k, stab);
        else for (uint32_t k = lane; k < n; k += 32) s_pre[k] = acrefine_predecode(src, sb0 + base + k, gtab);
        __syncwarp();
    };
    build_window(0);
    uint32_t pos = 0, eob_run = 0;
    uint4 v[8];
    size_t addr = 0, addr_next = 0;
    if ((uint32_t)lane < nblk) {
        addr_next = block_address(sc, mcu0 + lane, 0);
        load_block(B.coef + addr_next * 64, v);
    }
    for (uint32_t cb = 0; cb < nblk; cb += 32) {
        const int nb = (int)min(32u, nblk - cb);
        addr = addr_next;
        if (lane < nb) acrefine_build_table(block_mask(v), ss, se, s_tab + lane * BJ_ACR_TAB_STRIDE);
        if (cb + 32 + lane < nblk) {
            addr_next = block_address(sc, mcu0 + cb + 32 + lane, 0);
            load_block(B.coef + addr_next * 64, v);
        }
        __syncwarp();
        int i = 0;
        uint32_t err = 0;
        while (i < nb) {
            if (pos > win_base + (win_bits - BJ_ACR_WIN_SLACK)) build_window(pos);
            if (lane == 0) {
                uint32_t e = 0;
                const int i2 = acrefine_parse_window(s_pre, win_base, win_base + (win_bits - BJ_ACR_WIN_SLACK), sh.ctx,
                                                     end_rel, s_tab, i, nb, pos, eob_run, s_pos, e);
                s_state[0] = pos; s_state[1] = eob_run; s_state[2] = (uint32_t)i2; s_state[3] = e;
            }
            __syncwarp();
            pos = s_state[0]; eob_run = s_state[1]; i = (int)s_state[2]; err = s_state[3];
            __syncwarp();
            if (err) break;
        }
        if (err) {
            if (lane == 0) atomicOr(&B.err[sc.image], err);
            // blocks that were not reached decode nothing: an end-of-band block at the end of the stream
            for (uint32_t b = cb + lane; b < nblk; b += 32)
                B.blk_pos[block_address(sc, mcu0 + b, 0)] = end_rel | BJ_ACR_IN_EOBRUN;
            return;
        }
        if (lane < nb) B.blk_pos[addr] = s_pos[lane];
        __syncwarp();
    }
}

// T81: the T.81 correction rule (BJ_PHASE_T81_REFINE) instead of the reference's (acrefine_corrections)
template <bool T81>
__global__ void __launch_bounds__(128) acrefine_apply_kernel(const bj_scan* __restrict__ scans, int scan_first, bj_entropy_buffers B,
                                                             uint32_t lut_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CtaShared& sh = *reinterpret_cast<CtaShared*>(smem_raw);
    load_scan(sh, scans, scan_first + blockIdx.y, B, lut_cap);
    const bj_scan& sc = sh.sc;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= sc.n_mcu) return;
    const uint32_t m = i / sc.ri;
    const size_t addr = block_address(sc, i, 0);
    int16_t* p = B.coef + addr * 64;
    uint4 v[8];
    load_block(p, v);
    const uint32_t pos = B.blk_pos[addr];
    const uint64_t sb0 = B.stream_start[sc.stream0 + m] * 8, sb1 = B.stream_end[sc.stream0 + m] * 8;
    GlobalSrc src{B.words, (uint32_t)B.words_len};
    BitReader<GlobalSrc> rd;
    rd.seek(&src, sb0, pos & ~BJ_ACR_IN_EOBRUN);
    uint32_t eob_run = (pos & BJ_ACR_IN_EOBRUN) ? 1u : 0u;
    const uint64_t mask = block_mask(v);
    const uint32_t end_rel = (uint32_t)(sb1 - sb0);
    uint32_t err;
    if (sh.lut_in_smem) err = acrefine_block<true, T81>(rd, sh.ctx, sh.lut + sh.ctx.ac_tab[0], end_rel, mask, eob_run, p);
    else err = acrefine_block<true, T81>(rd, sh.ctx, B.lut + sc.lut_off + sh.ctx.ac_tab[0], end_rel, mask, eob_run, p);
    if (err) atomicOr(&B.err[sc.image], err);
}

size_t cta_smem_bytes(uint32_t lut_cap) { return sizeof(CtaShared) + sizeof(uint32_t) * lut_cap; }

}  // namespace

extern "C" {

static_assert(sizeof(bj_scan) == 144, "bj_scan layout");
static_assert(offsetof(bj_scan, raw_len) == 16 && offsetof(bj_scan, tile0) == 60 && offsetof(bj_scan, frame_mcus_x) == 64 &&
              offsetof(bj_scan, slot_frame) == 78 && offsetof(bj_scan, slot_comp) == 88 && offsetof(bj_scan, slot_dc) == 98 &&
              offsetof(bj_scan, slot_ac) == 118 && offsetof(bj_scan, reserved) == 140, "bj_scan layout");
int bj_sizeof_entropy(int what) {
    return what == 1 ? (int)sizeof(bj_scan) : what == 2 ? (int)sizeof(bj_entropy_buffers) : what == 3 ? BJ_SUBSEQ_BITS : -1;
}

bj_status bj_entropy_plan(const bj_scan* scans, int scan_first, int n_scans, const uint64_t* tile_sum,
                          const bj_entropy_buffers* bufs, void* stream) {
    if (!scans || n_scans <= 0 || !tile_sum || !bufs) return BJ_E_ARG;
    plan_kernel<<<n_scans, 256, 0, (cudaStream_t)stream>>>(scans, scan_first, tile_sum, *bufs);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_entropy_plan");
    return BJ_OK;
}

bj_status bj_entropy_decode(const bj_scan* scans, int scan_first, int n_scans, int mode, uint32_t max_sub,
                            uint32_t max_streams, uint32_t max_blocks, uint32_t max_lut,
                            const bj_entropy_buffers* bufs, uint32_t* chain, int phases, void* stream) {
    if (!scans || n_scans <= 0 || !bufs) return BJ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    const uint32_t lut_cap = max_lut < (uint32_t)kMaxLutSmem ? max_lut : (uint32_t)kMaxLutSmem;
    const size_t smem = cta_smem_bytes(lut_cap);
    if (mode == BJ_MODE_BASELINE || mode == BJ_MODE_DC_FIRST || mode == BJ_MODE_AC_FIRST) {
        (void)chain;
        if (max_sub == 0) return BJ_E_ARG;
        e = cudaFuncSetAttribute(spec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_entropy_decode/attr");
        dim3 grid((unsigned)n_scans, (max_sub + T - 1) / T);
        if (grid.y > 65535) return BJ_E_ARG;
        if (phases & BJ_PHASE_SPEC) {
            spec_kernel<<<grid, T, smem, st>>>(scans, scan_first, *bufs, lut_cap);
        }
        if (phases & BJ_PHASE_FIX) {
            fix_local_kernel<<<grid, T, 0, st>>>(scans, scan_first, *bufs);
            // shared-memory bitmap of stream heads: one bit per subsequence of the largest scan, up to 32 KB
            // (with the 8 KB of LUT and the static arrays this stays below the 48 KB default limit)
            uint32_t bitmap_words = (max_sub + 31) / 32;
            if (bitmap_words > 8192u || (phases & BJ_PHASE_NO_BITMAP)) bitmap_words = 0;
            const uint32_t chain_lut = lut_cap <= 2048u ? lut_cap : 2048u;  // bitmap + LUT stay below the 48 KB default limit
            chain_kernel<<<n_scans, kChainThreads, (bitmap_words + chain_lut) * sizeof(uint32_t), st>>>(scans, scan_first, n_scans, *bufs,
                                                                                                         bitmap_words, chain_lut);
        }
        if (phases & BJ_PHASE_WRITE) {
            write_kernel<<<dim3((unsigned)n_scans, (max_sub + TW - 1) / TW), TW + 32, smem, st>>>(scans, scan_first, *bufs, lut_cap);
        }
    } else if (mode == BJ_MODE_DC_REFINE) {
        unsigned gx = (max_blocks + 255) / 256;
        if (gx == 0) gx = 1;
        if (gx > 4096) gx = 4096;
        // the scan index rides on grid.y (at most 65535): larger waves are launched in slices
        for (int s0 = 0; s0 < n_scans; s0 += 65535) {
            const int ns = n_scans - s0 < 65535 ? n_scans - s0 : 65535;
            dcrefine_kernel<<<dim3(gx, (unsigned)ns), 256, 0, st>>>(scans, scan_first + s0, *bufs);
        }
    } else if (mode == BJ_MODE_AC_REFINE) {
        if (!bufs->blk_pos || max_streams == 0 || max_blocks == 0) return BJ_E_ARG;
        // window of the sequential parse: large for long streams (fewer rebuilds), small when the wave consists of many
        // short streams (restart intervals): their one-warp CTAs then fit an SM by the dozen
        const uint32_t win_bits = max_streams > 32u ? 4096u : (uint32_t)BJ_ACR_WIN_BITS;
        const size_t parse_smem = ((smem + 15) & ~(size_t)15) + sizeof(uint32_t) * win_bits;
        e = cudaFuncSetAttribute(acrefine_parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)parse_smem);
        const bool t81 = (phases & BJ_PHASE_T81_REFINE) != 0;
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(t81 ? acrefine_apply_kernel<true> : acrefine_apply_kernel<false>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_entropy_decode/attr");
        for (int s0 = 0; s0 < n_scans; s0 += 65535) {
            const int ns = n_scans - s0 < 65535 ? n_scans - s0 : 65535;
            acrefine_parse_kernel<<<dim3(max_streams, (unsigned)ns), 32, parse_smem, st>>>(scans, scan_first + s0, *bufs, lut_cap, win_bits);
            if (t81) acrefine_apply_kernel<true><<<dim3((max_blocks + 127) / 128, (unsigned)ns), 128, smem, st>>>(scans, scan_first + s0, *bufs, lut_cap);
            else acrefine_apply_kernel<false><<<dim3((max_blocks + 127) / 128, (unsigned)ns), 128, smem, st>>>(scans, scan_first + s0, *bufs, lut_cap);
        }
    } else {
        return BJ_E_ARG;
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return bj_set_cuda_error(e, "bj_entropy_decode/launch");
    return BJ_OK;
}

}  // extern "C"
