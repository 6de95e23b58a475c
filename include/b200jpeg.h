/*
 * b200jpeg.h -- C ABI of the B200-native JPEG decode hot path (libb200jpeg.so).
 *
 * This is the drop-in boundary for the hot path of tbpaolini/PyJpegDecoder (jpeg_decoder.py):
 * everything between "scan descriptors parsed on the host" and "uint8 RGB pixels".  The reference has
 * no FFI of its own (it is one pure-Python file); each entry point below names the reference
 * function(s) whose work it replaces.  The Python host layer (pyjpegdecoder_b200/) binds these with
 * ctypes; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch/CUDA-runtime types in signatures
 *     (a CUDA stream is passed as void*; NULL = the legacy default stream).
 *   - All buffers are DEVICE pointers owned by the caller unless a name ends in _host.
 *     The library allocates nothing per call; work space sizes come from bj_*_workspace_bytes().
 *   - Every call is asynchronous on the given stream and returns a bj_status (0 = ok) that only
 *     reports launch/argument errors.  Data errors (corrupt entropy data, ...) are written to the
 *     per-image device error words (BJ_ERR_* bits) and mapped by the host to the reference's
 *     exception classes (jpeg_decoder.py:1714-1725).
 *   - Re-entrant per (device, stream); no global mutable state.
 *
 * Data layout in HBM
 *   coefficient buffer  int16, 128-byte blocks of 64 coefficients in ZIG-ZAG order, quantised.
 *                       Per image the blocks are stored MCU-major over the padded MCU grid:
 *                       block index = coef_block0 + mcu * blocks_per_mcu + slot, slots in frame
 *                       component order, h*v blocks per component, row-major inside the MCU
 *                       (the interleaved scan order of jpeg_decoder.py:774-805/:875).
 *   sample buffer       int16, same block indexing, each block 8x8 row-major [y][x] after
 *                       de-zigzag * Q, IDCT, round, +128 (jpeg_decoder.py:869-872).
 *   output              uint8 row-major (H, W, 3) or (H, W); the reference's (W, H, 3) array
 *                       (jpeg_decoder.py:626, :1373-1386) is the transposed VIEW of it.
 */
#ifndef B200JPEG_H
#define B200JPEG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BJ_VERSION 100

typedef int bj_status;
#define BJ_OK 0
#define BJ_E_ARG 1      /* bad argument */
#define BJ_E_CUDA 2     /* CUDA runtime error, see bj_last_cuda_error() */
#define BJ_E_NOGPU 3    /* no CUDA device */

/* per-image device error word bits */
#define BJ_ERR_BAD_CODE 1u      /* no Huffman code within 16 bits   -> CorruptedJpeg (:718-719, :957-958) */
#define BJ_ERR_OVERRUN 2u       /* entropy data ended early          -> IndexError in the reference */
#define BJ_ERR_RST_COUNT 4u     /* fewer restart markers than the MCU count requires */
#define BJ_ERR_SYNC 8u          /* internal: more subsequences than the host reserved slots for (planning bug) */
#define BJ_ERR_COEF_INDEX 16u   /* coefficient index ran past 63 in a progressive scan */

#define BJ_MAX_COMP 3
#define BJ_MAX_SLOTS 10 /* blocks per MCU (T.81 limit) */

/* ---------------------------------------------------------------------------------------------
 * Image geometry for the pixel stages.  Filled by the host from SOF/SOS (jpeg_decoder.py:112-247,
 * :583-632).  72 bytes, 8-byte aligned.
 * ------------------------------------------------------------------------------------------- */
typedef struct bj_image {
    uint64_t coef_block0;  /* first block of this image in the coefficient / sample buffers */
    uint64_t out_offset;   /* offset of pixel (0,0) in the output buffer, in output ELEMENTS (uint8 or int16) */
    uint32_t out_pitch;    /* output elements per row (>= width * channels) */
    uint32_t width, height;
    uint32_t mcus_x, mcus_y;      /* padded MCU grid (interleaved geometry, :609-611) */
    uint32_t qtab[BJ_MAX_COMP];   /* index of each component's table in the qtab buffer (64 int16, zig-zag order) */
    uint8_t ncomp;                /* 1 (greyscale) or 3 (YCbCr) */
    uint8_t hs[BJ_MAX_COMP];      /* sampling factors, 1 or 2 (forced to 1 when ncomp == 1); hmax/hs and
                                     vmax/vs in {1,2}; at most two distinct upsampling kinds per image */
    uint8_t vs[BJ_MAX_COMP];
    uint8_t hmax, vmax;
    uint8_t blocks_per_mcu;
    uint8_t slot0[BJ_MAX_COMP];   /* first block slot of each component inside an MCU */
    uint16_t strip_mcus;          /* MCUs handled by one CTA of the pixel kernels: bj_pixels_fast_strip(layout) for the
                                     specialised layouts, else host-chosen <= 192 / blocks_per_mcu */
    uint16_t strips_per_row;      /* ceil(mcus_x / strip_mcus) */
    uint32_t layout;              /* BJ_LAYOUT_*: selects the specialised pixel kernel (0 = generic) */
} bj_image;

/* ---------------------------------------------------------------------------------------------
 * Entropy stage descriptors.
 *
 * A SCAN is one SOS segment of one image (jpeg_decoder.py:505-652).  Its entropy-coded bytes are
 * split by restart markers into STREAMS (restart intervals, :898-900 / :1050-1053 / :1297-1298);
 * a scan without DRI is one stream.  Every stream is decoded by many threads: it is cut into
 * SUBSEQUENCES of BJ_SUBSEQ_BITS bits that are decoded speculatively and then stitched together
 * (self-synchronising Huffman decode), see DESIGN.md.
 * ------------------------------------------------------------------------------------------- */
#ifndef BJ_SUBSEQ_BITS
#define BJ_SUBSEQ_BITS 8192   /* bj_sizeof_entropy(3) reports the value the library was built with */
#endif
#ifndef BJ_ENTROPY_THREADS
#define BJ_ENTROPY_THREADS 128 /* subsequences per CTA */
#endif
#define BJ_UNSTUFF_TILE 4096   /* raw bytes per CTA of the un-stuffing kernels */

#define BJ_MODE_BASELINE 0  /* baseline_dct_scan           :697-906   */
#define BJ_MODE_DC_FIRST 1  /* progressive DC first        :983-1033  */
#define BJ_MODE_DC_REFINE 2 /* progressive DC refinement   :1036-1043 */
#define BJ_MODE_AC_FIRST 3  /* progressive AC first + EOB runs :1120-1256 */
#define BJ_MODE_AC_REFINE 4 /* progressive AC refinement   :1100-1115, :1183-1198, :1258-1292 */

typedef struct bj_scan {
    uint64_t raw_off;      /* byte offset of the entropy-coded segment in the raw buffer (any alignment; the buffer
                              itself is 16-byte aligned and padded with 32 spare bytes) */
    uint64_t coef_block0;  /* first block of the image in the coefficient buffer */
    uint32_t raw_len;      /* bytes, including stuffed zeros and restart markers */
    uint32_t image;        /* index of the per-image error word */
    uint32_t stream0;      /* first entry of this scan in the stream tables */
    uint32_t n_streams;    /* ceil(n_mcu / ri), or 1 */
    uint32_t ri;           /* MCUs per stream (= n_mcu when there is no DRI) */
    uint32_t n_mcu;        /* MCUs in the scan (:621) */
    uint32_t mcus_x;       /* scan MCU grid width (:609-619) */
    uint32_t sub0;         /* first subsequence slot of this scan in the per-subsequence arrays */
    uint32_t n_sub_max;    /* slots reserved: >= sum over streams of ceil(bits / BJ_SUBSEQ_BITS) */
    uint32_t lut_off;      /* this scan's Huffman tables in the LUT buffer (uint32 entries) */
    uint32_t lut_len;
    uint32_t tile0;        /* first un-stuffing tile of this scan */
    uint16_t frame_mcus_x; /* interleaved MCU grid width of the frame */
    uint8_t frame_bpm;     /* blocks per MCU of the frame (coefficient buffer stride) */
    uint8_t nslots;        /* blocks per MCU of this scan */
    uint8_t mode;          /* BJ_MODE_* */
    uint8_t ss, se, ah, al;
    uint8_t interleaved;   /* 1: block = coef_block0 + mcu*frame_bpm + slot_frame[slot];
                              0: single component, block grid raster (:612-619), see comp_* */
    uint8_t comp_h, comp_v, comp_slot0; /* non-interleaved: the component's h, v and first frame slot */
    uint8_t ncomp_scan;                 /* components in the scan */
    uint8_t slot_frame[BJ_MAX_SLOTS];   /* scan slot -> slot inside the frame MCU */
    uint8_t slot_comp[BJ_MAX_SLOTS];    /* scan slot -> component index within the scan (DC predictor) */
    uint16_t slot_dc[BJ_MAX_SLOTS];     /* scan slot -> DC table offset inside the scan's LUT blob */
    uint16_t slot_ac[BJ_MAX_SLOTS];     /* scan slot -> AC table offset */
    uint32_t reserved;
} bj_scan;

/* Device buffers of the entropy stage (all caller-allocated, see pyjpegdecoder_b200/pipeline.py):
 *   words        un-stuffed bitstream, big-endian 32-bit words (bit 31 of word 0 = first bit)
 *   stream_start byte offset of each stream in `words`; stream_end likewise
 *   stream_sub   first subsequence of each stream, relative to its scan's sub0
 *   sub_entry/sub_exit  packed decoder state at the start / end of each subsequence
 *   sub_count    per subsequence: blocks started + DC difference sums of up to 3 components
 *   sub_prefix   exclusive prefix sums of sub_count (in subsequence order)
 */
typedef struct bj_entropy_buffers {
    const uint32_t* words;  /* 16-byte aligned (write_kernel copies it in 16-byte groups) */
    uint64_t words_len;     /* in 32-bit words, including 64 words of slack at the end */
    uint64_t* stream_start;
    uint64_t* stream_end;
    uint32_t* stream_sub;
    uint64_t* sub_entry;
    uint64_t* sub_exit;
    uint32_t* sub_count;    /* 4 x uint32 per subsequence */
    uint32_t* sub_prefix;   /* 4 x uint32 per subsequence */
    const uint32_t* lut;
    int16_t* coef;
    uint32_t* err;          /* per image error word (BJ_ERR_*) */
    uint32_t* sync_changes; /* optional statistics: subsequences re-decoded by the fix-up pass */
    uint32_t* blk_pos;      /* one per coefficient block; only needed (non-NULL) when the batch has AC
                               refinement scans: where each block's data starts in its stream */
} bj_entropy_buffers;

/*
 * Byte un-stuffing + restart-marker removal for every scan of a batch in one pass
 * (replaces the reader side of bits_generator/get_bits, jpeg_decoder.py:654-695: the byte after
 * 0xFF is dropped (:676-677); restart markers are skipped (:667-669)).
 *   raw         all entropy-coded segments, each starting at scan.raw_off
 *   tile_scan   scan index of every BJ_UNSTUFF_TILE-byte tile; a scan owns
 *               max(1, ceil(((raw_off & 15) + raw_len) / BJ_UNSTUFF_TILE)) consecutive tiles from tile0
 *   tile_sum    workspace, uint64[n_tiles + 1]
 *   words_out   compacted bitstream as big-endian 32-bit words (size >= total raw bytes / 4 + 64)
 *   stream_start/stream_end  filled per stream; missing restart markers leave UINT64_MAX
 */
bj_status bj_unstuff(const uint8_t* raw, const bj_scan* scans, int n_scans, const uint32_t* tile_scan,
                     int n_tiles, uint64_t* tile_sum, uint32_t* words_out, uint64_t* stream_start,
                     uint64_t* stream_end, int n_streams_total, void* stream);

/*
 * Stream planning: after bj_unstuff, computes for every scan the length of each stream, the number of
 * subsequences per stream and the first subsequence of each stream; flags missing restart markers
 * (BJ_ERR_RST_COUNT).  tile_sum is the workspace bj_unstuff filled.
 */
bj_status bj_entropy_plan(const bj_scan* scans, int scan_first, int n_scans, const uint64_t* tile_sum,
                          const bj_entropy_buffers* bufs, void* stream);

/*
 * Entropy decode of scans [scan_first, scan_first + n_scans), all of the same `mode` and independent
 * of each other (one "wave": normally the k-th scan of every image of the batch).  Replaces
 * baseline_dct_scan's entropy part (:709-722, :805-866, :898-900) and progressive_dct_scan
 * (:908-1304); coefficients go straight into the coefficient buffer (zig-zag order, quantised).
 * Progressive images need their coefficient blocks zeroed before the first scan.
 *   max_sub      max over the wave's scans of n_sub_max         (baseline / DC first / AC first)
 *   max_streams  max over the wave's scans of n_streams         (AC refine)
 *   max_blocks   max over the wave's scans of n_mcu * nslots    (DC refine, AC refine)
 *   max_lut      max over the wave's scans of lut_len
 *   chain        reserved (may be NULL)
 *   phases       BJ_PHASE_ALL, or a subset of the three kernels of the speculative modes so that a
 *                caller can time them separately (they must still run in this order)
 */
#define BJ_PHASE_SPEC 1
#define BJ_PHASE_FIX 2
#define BJ_PHASE_WRITE 4
#define BJ_PHASE_ALL 7
#define BJ_PHASE_NO_BITMAP 8 /* testing: the chain step finds stream heads by binary search, the path it takes by
                                itself for a scan of more than 262144 subsequences (128 MB of entropy-coded data) */
#define BJ_PHASE_T81_REFINE 16 /* AC refinement corrections by the T.81 rule (G.1.2.3, libjpeg-turbo's): a correction bit
                                  adds +-(1 << Al) by sign when that bit of the magnitude is clear, instead of the
                                  reference's `coef |= 1 << Al` on the two's-complement value; DC refinement is the same
                                  under both rules */
bj_status bj_entropy_decode(const bj_scan* scans, int scan_first, int n_scans, int mode, uint32_t max_sub,
                            uint32_t max_streams, uint32_t max_blocks, uint32_t max_lut,
                            const bj_entropy_buffers* bufs, uint32_t* chain, int phases, void* stream);

/* Sampling layouts with a specialised pixel kernel (chroma 1x1, luma HxV) */
#define BJ_LAYOUT_GENERIC 0
#define BJ_LAYOUT_420 1  /* luma 2x2 */
#define BJ_LAYOUT_422 2  /* luma 2x1 */
#define BJ_LAYOUT_440 3  /* luma 1x2 */
#define BJ_LAYOUT_444 4  /* luma 1x1 */
#define BJ_LAYOUT_GRAY 5 /* one component */

/* Output selector of bj_pixels(). */
#define BJ_OUT_RGB 0     /* uint8: fused IDCT + upsample + YCbCr->RGB (+ clamp)            */
#define BJ_OUT_SAMPLES 1 /* int16 sample buffer: de-zigzag, dequantise, IDCT, +128 only    */
#define BJ_OUT_CANVAS 2  /* int16 (H, W, ncomp): Y/Cb/Cr after upsampling, before colour   */
/* Input selector */
#define BJ_IN_COEF 0     /* coefficient buffer (zig-zag, quantised) */
#define BJ_IN_SAMPLES 1  /* sample buffer produced by BJ_OUT_SAMPLES */

int bj_version(void);
int bj_sizeof(int what);         /* 0: sizeof(bj_image), 1: sizeof(bj_resize_job), 2: sizeof(bj_scaled_job),
                                    3: sizeof(bj_crop_job), 4: sizeof(bj_resize_pil_job) -- lets a binding verify its
                                    struct mirrors */
int bj_sizeof_entropy(int what); /* 1: sizeof(bj_scan), 2: sizeof(bj_entropy_buffers), 3: BJ_SUBSEQ_BITS */
int bj_pixels_fast_strip(int layout); /* MCUs per CTA the specialised pixel kernel uses for BJ_LAYOUT_* (0: generic) */
const char* bj_last_cuda_error(void);

/*
 * Host-side helpers for the Python marker walk (no GPU involved).
 *   bj_host_find_marker  first p >= pos with data[p] == 0xFF and data[p+1] not 0x00 / RSTn: the end of an
 *                        entropy-coded segment as the reference's main loop sees it (jpeg_decoder.py:93)
 *   bj_host_count_sos    bytes.count(SOS) of jpeg_decoder.py:635-637
 */
uint64_t bj_host_find_marker(const uint8_t* data, uint64_t n, uint64_t pos);
uint32_t bj_host_count_sos(const uint8_t* data, uint64_t n, uint64_t pos);

/* One entry of the byte-level marker walk: a marker segment (payload [start, end), marker = second marker
 * byte) or an entropy-coded run (marker = 0x100).  Offsets are relative to the start of the file. */
typedef struct bj_host_entry {
    uint64_t start, end;
    uint32_t marker;
    uint32_t reserved;
} bj_host_entry;

/* Byte-level marker walk of one file, mirroring the main loop of jpeg_decoder.py:78-110 (segments are
 * located, not interpreted).  Returns the number of entries, -1: not a JPEG, -2: more than max_entries. */
int bj_host_walk(const uint8_t* data, uint64_t n, bj_host_entry* entries, int max_entries);
/* The same for n_files files of one buffer on n_threads host threads (entries: [n_files][max_entries]). */
void bj_host_walk_batch(const uint8_t* raw, const uint64_t* off, const uint64_t* size, int n_files,
                        bj_host_entry* entries, int max_entries, int32_t* counts, int n_threads);

/* bj_host_walk_batch plus a 128-bit hash per file (key_hash[2*i], key_hash[2*i+1]) of everything that determines
 * the parse (marker sequence + payloads of SOFn/DHT/DQT/DRI/SOS/DNL/EOI + one tag per entropy-coded run): files
 * with equal hashes share one parsed template on the host. */
void bj_host_walk_batch_keys(const uint8_t* raw, const uint64_t* off, const uint64_t* size, int n_files,
                             bj_host_entry* entries, int max_entries, int32_t* counts, uint64_t* key_hash, int n_threads);

/* Threaded gather of n_files host buffers into one packed buffer: memcpy(dst + off[i], src[i], size[i]). */
void bj_host_pack(const uint8_t* const* src, const uint64_t* size, const uint64_t* off, int n_files, uint8_t* dst,
                  int n_threads);

/* bj_host_pack + bj_host_walk_batch_keys in one pass (each file is walked right after it was copied, cache-hot). */
void bj_host_pack_walk_keys(const uint8_t* const* src, const uint64_t* size, const uint64_t* off, int n_files, uint8_t* dst,
                            bj_host_entry* entries, int max_entries, int32_t* counts, uint64_t* key_hash, int n_threads);

/* File sizes from host threads: size[i] = bytes of paths[i], or -errno. */
void bj_host_stat_files(const char* const* paths, int n_files, int64_t* size, int n_threads);

/* Read n_files files straight into a packed buffer (dst + off[i], size[i] bytes as measured by bj_host_stat_files)
 * from host threads; with entries != NULL every file is also walked and hashed like bj_host_walk_batch_keys right
 * after it was read.  status[i] = 0 or the errno of the failed open / read.  This is the file-read step in front of
 * the reference's JpegDecoder(Path) (jpeg_decoder.py:32-33) for a whole batch, without intermediate copies. */
void bj_host_read_files(const char* const* paths, const uint64_t* size, const uint64_t* off, int n_files, uint8_t* dst,
                        int32_t* status, bj_host_entry* entries, int max_entries, int32_t* counts, uint64_t* key_hash,
                        int n_threads);

/*
 * Pixel stages.  Replaces, for a whole batch of images in one launch:
 *   undo_zigzag * Q              jpeg_decoder.py:1648-1662, :869, :1347-1348   (int16 product wraps)
 *   InverseDCT.__call__          :1561-1573   (fp64 sum in numpy's pairwise order, round-half-even, +128)
 *   ResizeGrid.__call__          :1588-1626   (griddata piece-wise linear 8->16 on Qhull's triangulation)
 *   YCbCr_to_RGB + clip + crop   :1683-1700, :1372-1386
 * and the loops that drive them (:868-891 baseline, :1306-1366 progressive final stage).
 *
 *   images      device array of n_images bj_image
 *   in          coefficient buffer (BJ_IN_COEF) or sample buffer (BJ_IN_SAMPLES)
 *   total_blocks number of 128-byte blocks in `in` (bounds of the TMA tensor map over the coefficient buffer)
 *   qtabs       int16 quantisation tables, 64 entries each, zig-zag order as in the DQT segment
 *   idct_table_t 4096 doubles [u][v][x][y]: the reference's InverseDCT.idct_table (:1541-1553,
 *               indexed [x][y][u][v] there) TRANSPOSED so that the 64 output samples of one (u,v)
 *               are contiguous; computed by the host with the reference's expression; used only to
 *               resolve samples that the fp32 fast path cannot round safely.
 *   out         BJ_OUT_RGB: uint8 (H, W, 3|1) per image at out_offset/out_pitch;
 *               BJ_OUT_SAMPLES: int16 sample buffer (block indexing as the coefficient buffer);
 *               BJ_OUT_CANVAS: int16 (H, W, ncomp) per image at out_offset/out_pitch (int16 elements)
 *   max_strips  max over images of mcus_y * strips_per_row (grid x size)
 *   layout_mask bit L set: some image has layout L.  For BJ_IN_COEF -> BJ_OUT_RGB the images with a
 *               specialised layout (bits 1..5) run in the layout-specialised kernels and the generic
 *               kernel only handles layout 0; layout_mask == 0 sends every image through the generic
 *               kernel (the other in/out kinds always do).
 *   stats       optional device uint32[4]: [0] blocks recomputed exactly, [1] pixels recomputed exactly
 */
bj_status bj_pixels(const bj_image* images, int n_images, int max_strips, const void* in, int in_kind,
                    uint64_t total_blocks, const int16_t* qtabs, const double* idct_table_t, void* out, int out_kind,
                    uint32_t layout_mask, uint32_t* stats, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Resize + normalise of decoded images into one (N, 3, h, w) batch tensor (data-loader output).
 *
 * Filter: torch.nn.functional.interpolate(mode="bilinear", align_corners=False, antialias=True), separable
 * triangle filter, weights computed in the kernel (csrc/bj_resize_math.cuh), fp32 accumulation.  Value of an
 * output element of channel c: v * a[c] + b[c], v the resized value on the 0..255 scale; uint8 output rounds
 * that to nearest even and clamps to [0, 255].  Greyscale sources give three channels (each with its a/b).
 * ------------------------------------------------------------------------------------------- */
#define BJ_DTYPE_U8 0
#define BJ_DTYPE_F16 1
#define BJ_DTYPE_BF16 2
#define BJ_DTYPE_F32 3

/* One source image: 40 bytes, 8-byte aligned. */
typedef struct bj_resize_job {
    uint64_t src_offset;   /* byte offset of pixel (0,0) in src (bj_image.out_offset of BJ_OUT_RGB); any alignment */
    uint32_t src_pitch;    /* bytes per source row (bj_image.out_pitch) */
    uint32_t channels;     /* 3 (RGB) or 1 (greyscale) */
    uint32_t x0, y0, x1, y1; /* source box [x0, x1) x [y0, y1) in pixels, x0 < x1 <= width, y0 < y1 <= height */
    uint32_t dst_index;    /* image slot n of the output tensor */
    uint32_t reserved;
} bj_resize_job;

typedef struct bj_resize_params {
    uint32_t out_h, out_w;  /* output size, 1..65535 */
    uint32_t dtype;         /* BJ_DTYPE_* */
    uint32_t channels_last; /* 0: NCHW, 1: NHWC storage of the (N, 3, h, w) tensor */
    float a[3], b[3];       /* per-channel scale and offset */
} bj_resize_params;

/*
 *   jobs   DEVICE array of n_jobs bj_resize_job
 *   src    decoded uint8 pixels (the BJ_OUT_RGB buffer of bj_pixels)
 *   dst    output tensor storage, element type dtype, dense NCHW or NHWC
 *   p      HOST pointer; copied into the kernel parameters (the caller may reuse it when the call returns)
 * One launch covers every job (grid: output tiles x jobs; more than 65535 jobs are launched in slices).
 */
bj_status bj_resize(const bj_resize_job* jobs, int n_jobs, const uint8_t* src, void* dst, const bj_resize_params* p,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pillow's resample: PIL.Image.resize((VW, VH), BILINEAR | BICUBIC) of each job's source box, bit for bit, and of that
 * virtual (VH, VW) image only the (out_h, out_w) window at (win_x, win_y) is computed -- torchvision's Resize(r) +
 * CenterCrop(size) without the pixels the crop drops.  Arithmetic (csrc/bj_resize_pil_math.cuh): Resample.c's double
 * coefficients rounded to 22-bit fixed point, the horizontal pass rounded to uint8, then the vertical pass; both
 * in int32 (the header derives the bound).  Every output pixel uses the coefficients of the full (VW, VH) resize.
 * Value of an output element of channel c: v * a[c] + b[c] in fp32, v the uint8 resampled value; uint8 output stores v
 * (a = 1, b = 0 expected).  Greyscale sources give three channels (each with its a/b).
 * ------------------------------------------------------------------------------------------- */
#define BJ_PIL_BILINEAR 0
#define BJ_PIL_BICUBIC 1

typedef struct bj_resize_pil_job {   /* 56 bytes, 8-byte aligned */
    uint64_t src_offset;   /* byte offset of pixel (0,0) in src; any alignment */
    uint32_t src_pitch;    /* bytes per source row */
    uint32_t channels;     /* 3 (RGB) or 1 (greyscale) */
    uint32_t x0, y0, x1, y1; /* source box [x0, x1) x [y0, y1) in pixels: the image Pillow resizes */
    uint32_t dst_index;    /* image slot n of the output tensor */
    uint32_t virt_w, virt_h; /* the size the box is resized to, 1..2^31 - 1 (plain resize: out_w, out_h) */
    uint32_t win_x, win_y; /* the window's offset in the virtual image, win_x + out_w <= virt_w, win_y + out_h <= virt_h
                              (plain resize: 0, 0) */
    uint32_t reserved;
} bj_resize_pil_job;

/*
 *   jobs    DEVICE array of n_jobs bj_resize_pil_job
 *   src     decoded uint8 pixels (bj_pixels' BJ_OUT_RGB buffer or any packed layout of the same form)
 *   dst     output tensor storage, element type p->dtype, dense NCHW or NHWC
 *   p       HOST pointer, as for bj_resize: out_h / out_w are the window's size
 *   filter  BJ_PIL_BILINEAR or BJ_PIL_BICUBIC
 * One launch covers every job (grid: output tiles x jobs; more than 65535 jobs are launched in slices).  The kernel
 * computes the coefficients it needs itself; nothing is allocated.  A job whose box or window is empty or outside the
 * virtual image, or whose virtual size exceeds 2^31 - 1, writes nothing.  Returns BJ_E_ARG for a NULL pointer, n_jobs <= 0, an output size outside 1..65535, an
 * unknown dtype or an unknown filter.
 */
bj_status bj_resize_pil(const bj_resize_pil_job* jobs, int n_jobs, const uint8_t* src, void* dst,
                        const bj_resize_params* p, int filter, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Reduced-size decode: scale 1/s, s = 2, 4 or 8, in the DCT domain (libjpeg's scale_denom, PIL's draft()).
 * Output (ceil(H/s), ceil(W/s), 3) or (ceil(H/s), ceil(W/s)); scaled pixel k covers full pixels [k s, (k+1) s), the
 * encoder's padding included at the right / bottom edge.  Each block of component c gives an NY x NX tile,
 * NX = 8 (hmax / h_c) / s, NY = 8 (vmax / v_c) / s: the 2-D inverse DCT of the block's low-frequency NX x NY corner
 * with the cosine argument of an N-point transform (the 8-point IDCT's normalisation, so the block mean is kept),
 * rounded half to even, + 128; no layout needs chroma upsampling.  Colour: the fp32 rule of the full path, clip,
 * round half to even.  The arithmetic, with its fp32 error bound, is csrc/bj_scaled_math.cuh.
 * ------------------------------------------------------------------------------------------- */
typedef struct bj_scaled_job {   /* 24 bytes */
    uint64_t out_offset;         /* byte offset of scaled pixel (0,0) in out */
    uint32_t out_pitch;          /* bytes per row, >= ceil(width/s) * channels */
    uint32_t image;              /* index into images */
    uint32_t log2_scale;         /* 1, 2 or 3 */
    uint32_t reserved;
} bj_scaled_job;

/*
 *   images      DEVICE array of bj_image, the records bj_pixels reads; out_offset, out_pitch, strip_mcus and
 *               strips_per_row are not used
 *   jobs        DEVICE array of n_jobs bj_scaled_job: any mix of images, layouts and scales
 *   max_strips  max over jobs of mcus_y * ceil(mcus_x / S), S = min(192 / blocks_per_mcu,
 *               6144 / (ncomp * 16 * hmax * vmax)) MCUs per CTA
 *   coef        coefficient buffer (zig-zag, quantised); only the zig-zag prefix each block's corner needs is read
 *   qtabs       as for bj_pixels
 *   out         uint8 pixels at each job's out_offset / out_pitch
 * One launch covers every job (grid: strips x jobs; more than 65535 jobs are launched in slices).
 */
bj_status bj_pixels_scaled(const bj_image* images, const bj_scaled_job* jobs, int n_jobs, int max_strips,
                           const int16_t* coef, const int16_t* qtabs, uint8_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Crop decode: only the MCUs under a pixel box, at scale 1, 2, 4 or 8 (nvJPEG's ROI decode, libjpeg-turbo's
 * jpeg_crop_scanline).  The box [x0, x1) x [y0, y1) is in pixels of the image decoded at 1/s (s = 1 << log2_scale)
 * and lies inside it: x0 < x1 <= ceil(W / s), y0 < y1 <= ceil(H / s).
 * Window rule: with an MCU of mw = 8 hmax / s by mh = 8 vmax / s pixels at that scale, the job decodes the MCUs
 * [x0 / mw, ceil(x1 / mw)) x [y0 / mh, ceil(y1 / mh)) -- every MCU the box touches, no other.  A full-size MCU's
 * chroma interpolation and a scaled block's tile never read outside their own MCU, so the window's pixels are the
 * bytes bj_pixels / bj_pixels_scaled would write there.
 * Output contract: pixel (x, y) of the box goes to out + out_offset + (y - y0) * out_pitch + (x - x0) * channels; nothing
 * else is written.  Rows may start at any byte address.
 * ------------------------------------------------------------------------------------------- */
typedef struct bj_crop_job {   /* 40 bytes */
    uint64_t out_offset;       /* byte offset of box pixel (x0, y0) in out */
    uint32_t out_pitch;        /* bytes per row, >= (x1 - x0) * channels */
    uint32_t image;            /* index into images */
    uint32_t log2_scale;       /* 0, 1, 2 or 3 */
    uint32_t x0, y0, x1, y1;   /* the box, in pixels of the image decoded at 1/s */
    uint32_t reserved;
} bj_crop_job;

#define BJ_CROP_SCALED 8       /* bit of bj_pixels_crop's `kinds`: some job has log2_scale > 0 */

/*
 *   images      DEVICE array of bj_image, the records bj_pixels reads; out_offset and out_pitch are not used
 *   jobs        DEVICE array of n_jobs bj_crop_job: any mix of images, layouts and scales
 *   max_strips  max over jobs of (window rows) * ceil((window columns) / S), S = the image's strip_mcus at s = 1 and
 *               bj_pixels_scaled's MCUs per CTA at s > 1
 *   coef, total_blocks, qtabs, idct_table_t, stats   as for bj_pixels (COEF in, RGB out)
 *   out         uint8 pixels at each job's out_offset / out_pitch
 *   kinds       which kernels have work: bit BJ_LAYOUT_* for the layouts of the jobs at s = 1, bit BJ_CROP_SCALED for
 *               jobs at s > 1 (as bj_pixels' layout_mask, it saves the launches that would find no job)
 * One call covers every job; each specialised layout keeps its own kernel (grid: strips of the job's MCU window x jobs;
 * more than 65535 jobs are launched in slices).
 */
bj_status bj_pixels_crop(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                         const int16_t* coef, uint64_t total_blocks, const int16_t* qtabs, const double* idct_table_t,
                         uint8_t* out, uint32_t kinds, uint32_t* stats, void* stream);

/* ---------------------------------------------------------------------------------------------
 * libjpeg-turbo-exact pixels (compat="libjpeg-turbo"): bit for bit what libjpeg-turbo's default jpeg_read_scanlines
 * writes (JDCT_ISLOW, do_fancy_upsampling = TRUE, no merged upsampling; Pillow's Image.open pixels), from T.81
 * coefficients (bj_entropy_decode with BJ_PHASE_T81_REFINE for progressive files).  Dequantisation as int (no int16
 * wrap), jpeg_idct_islow with its range_limit table, jdsample.c's fancy upsampling -- which reads across MCU
 * boundaries, with edges replicated at each component's real size ceil(W h / hmax) x ceil(H v / vmax) -- and jdcolor.c's
 * table-exact YCbCr -> RGB.  The arithmetic is csrc/bj_ijg_math.cuh.  Full size only: jobs with log2_scale != 0 are
 * skipped (nothing is written).
 *
 * Jobs are bj_crop_job: box [x0, x1) x [y0, y1) in pixels of the image, x0 < x1 <= W, y0 < y1 <= H; a full decode is
 * one job with the box (0, 0, W, H) and the image's out_offset / out_pitch.
 * Output contract: as bj_pixels_crop -- pixel (x, y) of the box goes to out + out_offset + (y - y0) * out_pitch +
 * (x - x0) * channels, nothing else is written, rows may start at any byte.
 * Halo rule (bj::ijg_window): a job decodes the MCUs its box touches, grown to every MCU that holds a sample the fancy
 * upsampling of a box pixel reads: a component at ratio 2 in a direction (h2v1 / h2v2 with downsampled_width > 2, h1v2)
 * reads sample j - 1 for the even pixel 2j (j > 0) and j + 1 for the odd pixel 2j + 1 (j below the last real sample), so
 * the window grows by at most one MCU per side.  Call these MCUs [mx0, mx1) x [my0, my1).
 * Workspace rule: `reserved` of each job holds the byte offset of its planes in `workspace` divided by 256; the
 * job's planes are uint8, component after component, plane c having (mx1 - mx0) * 8 h_c columns and
 * (my1 - my0) * 8 v_c rows, row-major without padding; jobs must not overlap.  The library allocates nothing: the
 * caller sizes the workspace as the sum over jobs of these planes (each job's start rounded up to 256 bytes, see
 * pyjpegdecoder_b200/ijg.py).
 * ------------------------------------------------------------------------------------------- */
#define BJ_IJG_IDCT 1          /* bit of bj_pixels_ijg's `kinds`: run the IDCT launch (coefficients -> planes) */
#define BJ_IJG_COLOUR 2        /* run the upsample + colour launch (planes -> pixels) */
#define BJ_IJG_ALL 3

/*
 *   images      DEVICE array of bj_image, the records bj_pixels reads; out_offset and out_pitch are not used
 *   jobs        DEVICE array of n_jobs bj_crop_job: log2_scale 0, reserved = workspace offset / 256
 *   max_strips  max over jobs of my1 - my0 (grid x of both launches: one CTA per MCU row of the window)
 *   coef        coefficient buffer (zig-zag, quantised, T.81 refinement)
 *   qtabs       as for bj_pixels
 *   workspace   uint8 sample planes (workspace rule above), 256-byte aligned
 *   out         uint8 pixels at each job's out_offset / out_pitch
 *   kinds       BJ_IJG_ALL, or one of its two bits so that a caller can time the launches separately (the IDCT launch
 *               must have run before the colour launch reads the planes)
 * Returns BJ_E_ARG for a NULL buffer, n_jobs <= 0, max_strips <= 0 or a `kinds` outside BJ_IJG_ALL.
 */
bj_status bj_pixels_ijg(const bj_image* images, const bj_crop_job* jobs, int n_jobs, int max_strips,
                        const int16_t* coef, const int16_t* qtabs, uint8_t* workspace, uint8_t* out, uint32_t kinds,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200JPEG_H */
