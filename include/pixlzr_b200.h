/*
 * pixlzr_b200.h — C ABI of the B200-native pixlzr hot path (libpixlzr_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, opaque handles, integer status
 * codes, no C++/torch types.  The reference (crate `pixlzr` v0.3.1) has no FFI of its own; the
 * boundary sits behind its Rust `pub` API, between `Pixlzr::shrink*` / `expand` / `to_image`
 * and their bodies (SURVEY 8b).  Each entry point cites the reference interface it replaces
 * (path:line relative to the reference tree).  INTEGRATION.md shows the Rust `extern "C"`
 * binding a maintainer would add.
 *
 * Ownership: the caller owns every host buffer; the library owns device buffers behind the
 * handles, freed by the matching *_free.  Errors: every call returns a pxz_status (never
 * unwinds or aborts across the boundary — the reference panics instead); the message is
 * available from pxz_last_error().  Threading: a pxz_ctx is bound to one device and one CUDA
 * stream and is not thread-safe — use one per host thread.  All work is stream-ordered on the
 * context's stream; calls that fill host buffers synchronise that stream before returning.
 *
 * There is NO CPU fallback: every compute entry point runs hand-written sm_100a kernels and
 * fails with PXZ_E_CUDA when no such device is usable.
 */
#ifndef PIXLZR_B200_H
#define PIXLZR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PXZ_ABI_VERSION 1

typedef struct pxz_ctx pxz_ctx;         /* device + stream + scratch                          */
typedef struct pxz_image pxz_image;     /* pitched RGB8 / RGBA8 image resident in HBM         */
typedef struct pxz_payload pxz_payload; /* packed block payload + descriptor table in HBM     */

typedef enum {
  PXZ_OK = 0,
  PXZ_E_ARG = -1,         /* invalid argument (the reference would panic or produce garbage) */
  PXZ_E_CUDA = -2,        /* CUDA runtime / launch failure, or no sm_100 device               */
  PXZ_E_OOM = -3,         /* host or device allocation failed                                 */
  PXZ_E_NCCL = -4,        /* NCCL not loadable / collective failed                            */
  PXZ_E_UNSUPPORTED = -5, /* valid in the reference but not covered here (see message)        */
  PXZ_E_FORMAT = -6       /* malformed .pxlzr container / QOI stream                          */
} pxz_status;

/* == FilterType #[repr(u8)], src/data_types/mod.rs:10-30.  Unknown u8 -> Nearest (:110-121). */
typedef enum { PXZ_NEAREST = 0, PXZ_TRIANGLE = 1, PXZ_CATMULLROM = 2, PXZ_GAUSSIAN = 3, PXZ_LANCZOS3 = 4 } pxz_filter;

typedef enum {
  PXZ_METRIC_OKLAB_MAD = 0, /* get_block_variance with |x-avg|, src/operations.rs:26-126      */
  PXZ_METRIC_SOBEL_DIR = 1  /* get_block_variance_directionally, src/operations.rs:192-259    */
} pxz_metric;

/* pxz_shrink flags */
#define PXZ_FLAG_AFTER_IDENTITY 0x1u   /* `after = |x| x` as process() does (process/mod.rs:107-121)
                                          instead of `x * factor * 10` (pixlzr.rs:15,162)            */
#define PXZ_FLAG_NORMALISE_GLOBAL 0x2u /* EXTENSION: v' = (v-min)/(max-min) over all blocks of the
                                          image (all ranks of the communicator) before `after`.  min
                                          and max are the reference-order values of the extreme blocks
                                          in every mode; dims and pixels are bit-exact in every mode  */
#define PXZ_FLAG_EXACT_VALUES 0x4u     /* Oklab-MAD: run the reference-order (sequential f32) path on
                                          EVERY block, so stored values are bit-exact too.  Without
                                          it only blocks whose value lies near a level boundary are
                                          recomputed that way; dims are bit-exact in both modes.    */

/* One block of the reduced image, row-major grid order.  == PixlzrBlockRaw {width, height,
 * block_value, data} (src/data_types/block.rs:76-81) with `data` at payload[offset ..]. */
typedef struct {
  uint64_t offset; /* byte offset of the block's tightly packed pixels in the payload            */
  float value;     /* block_value = hypot(v0, v1) after parse_value (operations.rs:145,154)      */
  uint16_t w, h;   /* reduced size                                                               */
} pxz_block_desc;

/* ---- library / context ---------------------------------------------------------------- */
int pxz_abi_version(void);
/* number of usable CUDA devices (0 if none / no driver) */
int pxz_device_count(void);
/* One context per host thread; it owns one CUDA stream and its scratch.  Environment read at creation (diagnostics only):
 *   PXZ_RESAMPLE_KERNELS=warp|cta  force a resample kernel family (default: by tile count): warp-per-tile (the
 *                                  TMA-fed shrink kernel) or CTA-per-tile. */
pxz_status pxz_ctx_create(int device, pxz_ctx** out);
/* same, but work is ordered on an existing CUDA stream (cudaStream_t / CUstream passed as
 * void*), e.g. torch.cuda.current_stream().cuda_stream.  The stream must outlive the ctx. */
pxz_status pxz_ctx_create_on_stream(int device, void* cuda_stream, pxz_ctx** out);
void pxz_ctx_destroy(pxz_ctx* ctx);
const char* pxz_last_error(const pxz_ctx* ctx);
pxz_status pxz_synchronize(pxz_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t pxz_launch_count(const pxz_ctx* ctx);
/* Resample arithmetic of this context.  0 (default): the reference's order — separate multiply and add, no
 * contraction — resampled pixels are bit-identical to the CPU result.  1: fused multiply-add on the RGBA fast paths;
 * faster, dims / offsets / values unchanged, pixels within +-1 LSB of the reference (the bar BASELINE.json states). */
/* Which branch of PixlzrBlock::resize (src/data_types/block.rs:273-334) the resample kernels compute.
 *   PXZ_RESIZE_IMAGE_RS (default): the `image` crate branch (block.rs:282-290) — f32, vertical pass first; this is the
 *       branch the reference's committed fixtures were produced with, reproduced bit for bit.
 *   PXZ_RESIZE_FIR: the `fast_image_resize` branch (block.rs:292-333 with FilterType::to_fir_resizing_algorithm,
 *       data_types/mod.rs:65-107), the crate's default cargo feature — 16-bit fixed-point convolution, horizontal pass
 *       first into a u8 image, Triangle = Hamming when shrinking / Bilinear when growing, pre-multiplied alpha for RGBA.
 *       Restated from the crate's published algorithm: PARITY UNPINNED (no artefact of the reference was made with it). */
typedef enum { PXZ_RESIZE_IMAGE_RS = 0, PXZ_RESIZE_FIR = 1 } pxz_resize_semantics;
pxz_status pxz_ctx_set_resize_semantics(pxz_ctx* ctx, pxz_resize_semantics semantics);
pxz_status pxz_ctx_set_fast_resample(pxz_ctx* ctx, int on);
/* ---- per-block filter pairs ("strategy"; SURVEY.md §8f N4) --------------------------------------------------
 * The reference's author measured, per bucket of width 1/64 of the value that enters the level quantiser, which
 * (down, up) filter pair reproduces a block best (strategies.txt:1-118, summarised in strategies_by_level.txt:1-12),
 * but the crate never uses the result: `shrink_*` / `expand` take one filter per call.  With a strategy installed,
 * pxz_shrink / pxz_expand* / pxz_payload_upload of this context ignore their filter argument and pick, per block,
 * down[b] / up[b] with b = pxz_strategy_bucket(block value).  The bucket is a function of the value STORED with the
 * block (pxz_block_desc.value = hypot(p0, p1), operations.rs:154; it travels in the container), so a decoder finds the
 * same filter: b = floor(64 * value / sqrt(2)) clamped to [0, 64]; NaN and negatives give 0.  value / sqrt(2) is the
 * quantiser's input p for Oklab-MAD (both axes share it) and the root mean square of (p0, p1) for the Sobel metric.
 * pxz_tree_process keeps its two explicit filters.  NULL removes the strategy.  No reference run exists for this
 * mode: parity is against the oracle's restatement of the same rule on top of the pinned per-block resize. */
#define PXZ_STRATEGY_BUCKETS 65
typedef struct pxz_strategy {
  uint8_t down[PXZ_STRATEGY_BUCKETS]; /* pxz_filter per bucket, used by pxz_shrink        */
  uint8_t up[PXZ_STRATEGY_BUCKETS];   /* pxz_filter per bucket, used by the expand calls  */
} pxz_strategy;
uint32_t pxz_strategy_bucket(float block_value);
/* the table the reference's log arrives at (strategies_by_level.txt:1-12) */
pxz_status pxz_strategy_by_level(pxz_strategy* out);
pxz_status pxz_ctx_set_strategy(pxz_ctx* ctx, const pxz_strategy* strategy);
/* Per-kernel device timing (CUDA events recorded on the context's stream around every kernel
 * launch while enabled).  pxz_profile_read synchronises the stream, returns the accumulated
 * duration and launch count of kernel `kernel_id` since profiling was enabled.  Kernel ids are
 * 0 .. n-1 where pxz_profile_kernel_name(n) == NULL. */
pxz_status pxz_profile_enable(pxz_ctx* ctx, int on);
const char* pxz_profile_kernel_name(int kernel_id);
pxz_status pxz_profile_read(pxz_ctx* ctx, int kernel_id, double* total_ms, uint64_t* launches);
/* pinned host memory for fast H2D / D2H */
pxz_status pxz_host_alloc(size_t bytes, void** out);
void pxz_host_free(void* p);

/* ---- images: Pixlzr::from_image (src/data_types/pixlzr_image.rs:6-22) -------------------
 * The reference materialises one cropped copy per block (split.rs:10-27).  Here a block is an
 * index into the pitched image; `from_image` is just the upload. */
pxz_status pxz_image_upload(pxz_ctx* ctx, const uint8_t* host, uint32_t w, uint32_t h, uint32_t channels /* 3|4 */,
                            size_t host_pitch, pxz_image** out);
pxz_status pxz_image_alloc(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t channels, pxz_image** out);
/* non-owning view of device memory the caller keeps alive (e.g. a torch uint8 tensor) */
pxz_status pxz_image_wrap(pxz_ctx* ctx, void* device_ptr, uint32_t w, uint32_t h, uint32_t channels, size_t pitch,
                          pxz_image** out);
pxz_status pxz_image_info(const pxz_image* img, uint32_t* w, uint32_t* h, uint32_t* channels, size_t* pitch,
                          void** device_ptr);
pxz_status pxz_image_download(pxz_ctx* ctx, const pxz_image* img, uint8_t* host, size_t host_pitch);
void pxz_image_free(pxz_image* img);

/* ---- batches of images (SURVEY.md 8b "batch round-robin entry points"; BASELINE config 5) ------------------------
 * A batch is n_images images of one size stacked in one pitched device allocation (image i at rows
 * [i * h, (i + 1) * h)).  pxz_shrink_batch / pxz_expand_batch run ONE launch per stage over the tiles of all images
 * — what a loop of Pixlzr::from_image(..).shrink_by(..) / to_image(..) over the batch computes (pixlzr.rs:155-185,
 * pixlzr_image.rs:24-74), image by image identical to the single-image calls.  The payload of a batch is one buffer:
 * descriptors in image order, then row-major per image (pxz_payload_info reports cols / rows of ONE image,
 * pxz_payload_batch_count the images), offsets running through the whole batch.  pxz_image_download /
 * pxz_payload_download / pxz_expand take host buffers laid out the same way (images back to back).
 * Not available on a batch: PXZ_FLAG_NORMALISE_GLOBAL (per image by definition), the container stage, tree processing. */
pxz_status pxz_image_alloc_batch(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t channels, uint32_t n_images, pxz_image** out);
pxz_status pxz_image_upload_batch(pxz_ctx* ctx, const uint8_t* host, uint32_t w, uint32_t h, uint32_t channels, size_t host_pitch,
                                  uint32_t n_images, pxz_image** out);
pxz_status pxz_image_wrap_batch(pxz_ctx* ctx, void* device_ptr, uint32_t w, uint32_t h, uint32_t channels, size_t pitch,
                                uint32_t n_images, pxz_image** out);
uint32_t pxz_image_batch_count(const pxz_image* img);
/* block grid: cols = ceil(w/bw), rows = ceil(h/bh) (split.rs:45-46, pixlzr.rs:37-42) */
pxz_status pxz_grid(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t* cols, uint32_t* rows);

/* ---- analysis: get_block_variance / get_block_variance_directionally ---------------------
 * Raw per-block metric (before `after`), row-major; host arrays of cols*rows floats (a batch image:
 * cols*rows*pxz_image_batch_count(img), image after image).
 * OKLAB_MAD fills values_x (values_y, if given, gets a copy); SOBEL_DIR fills (hz, vr).
 * flags: PXZ_FLAG_EXACT_VALUES for reference-order f32 sums. */
pxz_status pxz_analyze(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint32_t flags,
                       float* host_values_x, float* host_values_y /* may be NULL */);

/* ---- encode: Pixlzr::shrink_by (pixlzr.rs:155-185), shrink_directionally (:187-205),
 * reduce_image_section (operations.rs:140-156), PixlzrBlock::resize (block.rs:273-290).
 * One device pass: analysis -> plan (value -> level -> dims -> offsets) -> fused resample
 * writing the packed payload.  Nothing is copied to the host. */
pxz_status pxz_shrink(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                      pxz_filter filter_down, uint32_t flags, pxz_payload** out);

/* EXTENSION (rate control; the reference takes the factor only, src/bin/main.rs `-k`).  k = the largest finite f32 > 0 for
 * which pxz_shrink(ctx, img, bw, bh, metric, k, filter_down, flags) produces at most max_bytes payload bytes
 * (pxz_payload_info's `bytes`; an RGB image counts 3 bytes per pixel).  *out is that payload, byte for byte what
 * pxz_shrink returns for k (descriptors incl. stored values, pixels); *factor_out = k.  k = FLT_MAX when even that fits.
 * The size is monotone in k, so one analysis pass is enough: the device evaluates the size for up to 256 factors per round
 * from the block values alone, and the Oklab fast path checks the two sizes that bracket the budget in reference order
 * (DESIGN.md §3).  Each round reads sizes back to the host, so this call synchronises the stream and cannot be captured
 * in a CUDA graph.
 * PXZ_E_ARG: max_bytes below the payload at the smallest positive factor (the message names that size),
 *            PXZ_FLAG_AFTER_IDENTITY (the factor is unused), unknown filter / metric.
 * PXZ_E_UNSUPPORTED: a batch image; PXZ_FLAG_NORMALISE_GLOBAL on a context with a communicator. */
pxz_status pxz_shrink_to_size(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint64_t max_bytes,
                              pxz_filter filter_down, uint32_t flags, float* factor_out, pxz_payload** out);

/* ---- decode error and strategy fit (EXTENSION: the reference has no error measure; its author's filter-pair experiment,
 * strategies.txt, was run outside the crate) ---------------------------------------------------------------------------
 * Per-block error between two images of one geometry (w, h, channels; not batches) on the block grid (bw, bh) of pxz_grid:
 * sse[b] = sum over the tile's pixels and channels of (a - b)^2 (exact, u64), max[b] = max |a - b| over the same.  Integer
 * arithmetic: the result does not depend on the order of the sums.  Each output may be NULL; *total_sse = sum of sse[b].
 * Host arrays hold cols*rows entries in row-major order.  PSNR = 10 log10(255^2 * w * h * channels / total_sse).
 * PXZ_E_ARG: geometry mismatch, block size 0.  PXZ_E_UNSUPPORTED: a batch image. */
pxz_status pxz_image_error(pxz_ctx* ctx, const pxz_image* a, const pxz_image* b, uint32_t bw, uint32_t bh,
                           uint64_t* host_block_sse, uint8_t* host_block_max, uint64_t* host_total_sse);

#define PXZ_FILTER_PAIRS 25 /* pair index = down * 5 + up */
/* For every (down, up) filter pair: the error of pxz_expand_to_image(pxz_shrink(img, bw, bh, metric, factor, down, flags), up)
 * against img, summed per strategy bucket of the block's stored value.  host_sse[bucket * 25 + pair] (65 * 25 u64),
 * host_blocks[bucket] (65 u32): filled, not accumulated.  A block's shrink + expand depends only on its tile, its dims and its
 * filter pair, so the error of any per-bucket table is the sum of these entries.  The bucket of each block is the one its
 * reference-order stored value gives, in every mode (every bucket edge is resolved in the guard band of the fast Oklab path),
 * so flags 0 and PXZ_FLAG_EXACT_VALUES return identical reports.  The context's strategy is not used and is left installed.
 * One analysis, 5 shrinks, 25 expands and error passes; only the report crosses to the host.
 * PXZ_E_ARG as pxz_shrink (unknown metric, Sobel trailing tile, ...).  PXZ_E_UNSUPPORTED: a batch image,
 * PXZ_FLAG_NORMALISE_GLOBAL on a context with a communicator. */
pxz_status pxz_strategy_measure(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                                uint32_t flags, uint64_t* host_sse, uint32_t* host_blocks);
/* Host: the table that minimises the summed error per bucket.  down[b], up[b] = the pair of least sse[b][*]; on a tie base's
 * pair if it is among the least, else the lowest pair index; a bucket with blocks[b] == 0 keeps base's pair.  base == NULL
 * means pxz_strategy_by_level.  Reports of several images can be added element-wise before this call.
 * Installed with pxz_ctx_set_strategy in the default (reference-order) resample arithmetic, the table's pxz_shrink ->
 * pxz_expand_to_image -> pxz_image_error total is exactly sum over b of sse[b][down[b] * 5 + up[b]], which is <= the total of
 * every uniform pair and of base.  With pxz_ctx_set_fast_resample(1) pixels are within +-1 LSB and that equality does not hold.
 * PXZ_E_ARG: a NULL sse / blocks / out, an unknown filter in base. */
pxz_status pxz_strategy_choose(const uint64_t* sse, const uint32_t* blocks, const pxz_strategy* base, pxz_strategy* out);

/* EXTENSION (rate-distortion).  For one (filter_down, filter_up) pair: every distinct payload pxz_shrink(img, bw, bh, metric, k,
 * filter_down, flags) produces over the finite factors k > 0, in increasing k.  Point i: factor[i] = the SMALLEST f32 k giving that
 * payload geometry (factor[0] = the smallest positive f32), bytes[i] = its payload bytes (pxz_payload_info; an RGB image counts 3
 * per pixel), sse[i] = the total squared error of pxz_expand_to_image(that payload, filter_up) against img (pxz_image_error).
 * bytes is strictly increasing.  n <= 1 + cols*rows*(ceil(log2 bw) + ceil(log2 bh)) (Oklab-MAD: ceil(log2 max(bw, bh))).
 * *n_out is always set; cap < n -> PXZ_E_ARG (message names n), nothing written.  sse is exact in the default resample
 * arithmetic (both resize semantics); with pxz_ctx_set_fast_resample(1) it is not claimed.
 * One reference-order analysis, then one plan + resample + expand + error pass per level pair (Oklab-MAD: 1 + ceil(log2
 * max(bw, bh)) passes, 7 at 64x64; Sobel: (1 + ceil(log2 bw)) * (1 + ceil(log2 bh)), 49 at 64x64), then per block the factors
 * at which its dims change, one sort and one scan (DESIGN.md §3).  Device scratch: passes x blocks x 8 bytes for the error table
 * (about 100 MB for Sobel on a 32768 x 32768 image at 64x64) plus about 100 bytes per possible point.  The host arrays may be
 * NULL when cap = 0.  Synchronises the stream.
 * PXZ_E_ARG and PXZ_E_UNSUPPORTED: as pxz_shrink_to_size, an unknown filter_up; PXZ_E_UNSUPPORTED: a strategy installed on the
 * context (the filter pair would follow the stored value, which moves with k). */
pxz_status pxz_rd_curve(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, pxz_filter filter_down,
                        pxz_filter filter_up, uint32_t flags, float* host_factor, uint64_t* host_bytes, uint64_t* host_sse,
                        size_t cap, size_t* n_out);

/* EXTENSION (rate control by error).  k = the smallest finite f32 > 0 whose decode (filter_up) has total SSE <= max_sse: the first
 * point of pxz_rd_curve within the budget.  Payload size is monotone in k, so this is the smallest payload any factor gives
 * within the budget.  *out = pxz_shrink(k, filter_down, flags) byte for byte (descriptors incl. stored values, pixels);
 * *factor_out = k, *sse_out = its SSE (each may be NULL).  Synchronises the stream.
 * PXZ_E_ARG: no factor reaches max_sse (the message names the least SSE reachable), PXZ_FLAG_AFTER_IDENTITY, unknown filter /
 *            metric.
 * PXZ_E_UNSUPPORTED: a batch image, a strategy installed on the context, PXZ_FLAG_NORMALISE_GLOBAL with a communicator. */
pxz_status pxz_shrink_to_error(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint64_t max_sse,
                               pxz_filter filter_down, pxz_filter filter_up, uint32_t flags, float* factor_out, uint64_t* sse_out,
                               pxz_payload** out);

/* EXTENSION (rate-distortion optimised encode).  A decoder takes each block's dims from its QOI header, so an encoder may give
 * every block any size.  A block's candidates are the dims scaled_dim(tw, lx) x scaled_dim(th, ly) of every level pair
 * 0 <= lx <= ceil(log2 bw), 0 <= ly <= ceil(log2 bh), priced at bytes = w' * h' * (channels; 3 for RGB) and sse = the error of
 * that block's decode (filter_down, then filter_up).  Every payload pxz_shrink gives (any metric, factor, flags) is one choice
 * among them.  The curve: point 0 has every block at 1 x 1; each next point takes the next segment, by falling rate
 * (error removed per byte added, compared exactly), of the blocks' lower convex hulls.  bytes strictly increases, sse strictly
 * decreases, the last point has sse 0, and no choice of sizes has at most a point's bytes and less error than it.
 * n <= 1 + blocks * ((1 + ceil(log2 bw)) * (1 + ceil(log2 bh)) - 1).  *n_out is always set; cap < n -> PXZ_E_ARG (message names
 * n), nothing written.  sse is exact in the default resample arithmetic (both resize semantics); with
 * pxz_ctx_set_fast_resample(1) it is not claimed.  One plan + resample + expand + error pass per level pair (49 at 64x64), then
 * per block its hull, one merge sort and one scan (DESIGN.md §3 "Per-block sizes").  Device scratch: passes x blocks x 8 bytes
 * for the error table plus about 100 bytes per possible event.  The host arrays may be NULL when cap = 0.  Synchronises the
 * stream.
 * PXZ_E_ARG: an unknown filter, a block size of 0.
 * PXZ_E_UNSUPPORTED: a batch image, a strategy installed on the context (its filter pair follows the stored value), more than
 *                    2^31 events. */
pxz_status pxz_rdo_curve(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_filter filter_down, pxz_filter filter_up,
                         uint64_t* host_bytes, uint64_t* host_sse, size_t cap, size_t* n_out);

/* EXTENSION (rate-distortion optimised encode).  The payload of one point of pxz_rdo_curve: to size, the last point with
 * bytes <= max_bytes (the least error within the budget); to error, the first point with sse <= max_sse (the fewest bytes
 * within the budget).  Each block is encoded at its vertex's smallest level pair (lx, ly) with the stored value
 * hypot(2^-lx, 2^-ly) (= pxz_reduce_dims(2^-lx, 2^-ly, tw, th)), so every reader of the format decodes it.  *bytes_out /
 * *sse_out (each may be NULL) = the point's bytes and sse, which the payload's pxz_payload_info bytes and its decode with
 * filter_up (pxz_image_error) equal in the default resample arithmetic.  Against pxz_shrink_to_error with the same filter pair
 * (payload B_A bytes): the first curve point with bytes >= B_A is within max_sse, so pxz_rdo_shrink_to_error's payload is at most
 * one hull segment larger than B_A.  Synchronises the stream.
 * PXZ_E_ARG: as pxz_rdo_curve; max_bytes below the payload with every block at 1 x 1 (the message names that size).
 * PXZ_E_UNSUPPORTED: as pxz_rdo_curve. */
pxz_status pxz_rdo_shrink_to_size(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, uint64_t max_bytes, pxz_filter filter_down,
                                  pxz_filter filter_up, uint64_t* bytes_out, uint64_t* sse_out, pxz_payload** out);
pxz_status pxz_rdo_shrink_to_error(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, uint64_t max_sse, pxz_filter filter_down,
                                   pxz_filter filter_up, uint64_t* bytes_out, uint64_t* sse_out, pxz_payload** out);

/* Scalar part of reduce_image_section (operations.rs:128-156) on the host: (v0, v1) after `after`
 * -> parse_value -> level -> reduced size of a w x h block and the stored block value.  Uses the
 * same threshold table as the device plan kernel. */
pxz_status pxz_reduce_dims(float v0, float v1, uint32_t w, uint32_t h, uint32_t* out_w, uint32_t* out_h, float* stored);

/* Host helper / diagnostic: the tap table the resample kernels apply for one axis, n_in -> n_out samples with
 * `filter` (image 0.25.5 sample loops behind PixlzrBlock::resize, block.rs:282-290): first tap `left[o]`, tap count
 * `count[o]` and normalised f32 weights `weights[o * max_taps + i]` per output o.  Returns the largest tap count
 * (> max_taps means the arrays were too small and nothing was written) or a negative pxz_status. */
int32_t pxz_resample_table(uint32_t n_in, uint32_t n_out, pxz_filter filter, uint32_t* left, uint32_t* count, float* weights,
                           uint32_t max_taps);

/* ---- payload ---------------------------------------------------------------------------- */
pxz_status pxz_payload_info(pxz_ctx* ctx, const pxz_payload* p, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                            uint32_t* cols, uint32_t* rows, uint32_t* channels, uint64_t* bytes);
/* host_descs: cols*rows entries; host_pixels: `bytes` from pxz_payload_info */
pxz_status pxz_payload_download(pxz_ctx* ctx, const pxz_payload* p, pxz_block_desc* host_descs, uint8_t* host_pixels);
/* build a device payload from decoded blocks (what Pixlzr::decode_from_vec yields) */
pxz_status pxz_payload_upload(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels,
                              const pxz_block_desc* descs, const uint8_t* pixels, uint64_t bytes, pxz_payload** out);
void pxz_payload_free(pxz_payload* p);

/* ---- decode: Pixlzr::expand (pixlzr.rs:77-122) + to_image paste (pixlzr_image.rs:24-74) --
 * One kernel: every block is resampled to its tile size and written straight into the
 * pitched output image. */
pxz_status pxz_expand(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, uint8_t* host_out, size_t host_pitch);
pxz_status pxz_expand_to_image(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, pxz_image* out);
/* batch forms (see "batches of images" above): same arguments, the image / payload handles hold n_images images */
pxz_status pxz_shrink_batch(pxz_ctx* ctx, const pxz_image* batch, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                            pxz_filter filter_down, uint32_t flags, pxz_payload** out);
pxz_status pxz_expand_batch(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, pxz_image* out_batch);
pxz_status pxz_payload_upload_batch(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels,
                                    uint32_t n_images, const pxz_block_desc* descs, const uint8_t* pixels, uint64_t bytes,
                                    pxz_payload** out);
uint32_t pxz_payload_batch_count(const pxz_payload* p);


/* ---- quadtree processing: tree::process_custom (src/process/tree.rs:23-83) with before = |x-avg|, after = identity.
 * Blocks whose value is below |threshold| are reduced and re-expanded (filter_down / filter_up); the others are split
 * again with halved block size until the size reaches max(min, 4), where they stay unchanged.  A negative threshold
 * inverts the test at the top level only, as the reference does (the recursion receives |threshold|).  `out` has the
 * geometry of `img` (the reference pastes into an RGBA8 canvas: add alpha 255 for RGB inputs).  Block sizes must stay
 * exact when halved (divisible by 2^(levels-1)), else PXZ_E_UNSUPPORTED. */
pxz_status pxz_tree_process(pxz_ctx* ctx, const pxz_image* img, float threshold, uint32_t bw, uint32_t bh, uint32_t min_bw,
                            uint32_t min_bh, pxz_filter filter_down, pxz_filter filter_up, pxz_image* out);

/* ---- multi-GPU (one process per GPU) ------------------------------------------------------
 * Only PXZ_FLAG_NORMALISE_GLOBAL needs communication: one all-reduce of {min, -max} per
 * metric component over NCCL on the context's stream.  Rank 0 creates the id and shares its
 * 128 bytes (e.g. torch.distributed.broadcast); every rank then calls pxz_comm_init. */
#define PXZ_COMM_ID_BYTES 128
pxz_status pxz_comm_unique_id(uint8_t id[PXZ_COMM_ID_BYTES]);
pxz_status pxz_comm_init(pxz_ctx* ctx, int nranks, int rank, const uint8_t id[PXZ_COMM_ID_BYTES]);
void pxz_comm_destroy(pxz_ctx* ctx);
/* A rank whose shard has no block rows (more ranks than block rows) still has to take part in the exchange of
 * every pxz_shrink(PXZ_FLAG_NORMALISE_GLOBAL) its peers issue: it calls this instead, once per such shrink.
 * (A rank whose pxz_shrink fails before the exchange joins by itself, with an error flag that makes its peers
 * return PXZ_E_NCCL instead of waiting for it.) */
pxz_status pxz_comm_join_empty(pxz_ctx* ctx);

/* ---- host container stage (stays on the host, layout unchanged) ---------------------------
 * Pixlzr::encode_to_vec / decode_from_vec (src/encoding/mod.rs:40-165) with the qoi 0.4.1
 * per-block codec.  `value_present == NULL` means every block has a value. */
int64_t pxz_container_bound(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels, uint64_t payload_bytes);
int64_t pxz_container_encode(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t filter_byte, uint32_t channels,
                             const pxz_block_desc* descs, const uint8_t* pixels, const uint8_t* value_present,
                             uint8_t* out, size_t cap, int nthreads);
/* pass 1: descs == NULL -> header fields, channels and payload byte count.  pass 2: fills both. */
pxz_status pxz_container_decode(const uint8_t* data, size_t len, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                                int32_t* filter_byte /* -1 if absent */, uint32_t* channels, uint64_t* payload_bytes,
                                pxz_block_desc* descs, uint8_t* pixels);

/* The same stage on the device (SURVEY.md §8f N1): the per-block QOI streams are written from / decoded into the
 * device-resident payload, so only the compressed file crosses PCIe.  Output and accepted input are byte-identical to
 * pxz_container_encode / pxz_container_decode (= Pixlzr::encode_to_vec / decode_from_vec, src/encoding/mod.rs:40-165).
 * values_present = 0 writes every block value as 0.0 (block_value == None, :173-178).  host_out: capacity from
 * pxz_container_bound(); *bytes_out = size of the file.  pxz_payload_from_container returns a payload ready for
 * pxz_expand*; *filter_byte as pxz_container_decode. */
pxz_status pxz_payload_to_container(pxz_ctx* ctx, const pxz_payload* p, uint32_t filter_byte, int values_present, uint8_t* host_out,
                                    size_t cap, uint64_t* bytes_out);
pxz_status pxz_payload_from_container(pxz_ctx* ctx, const uint8_t* data, size_t len, int32_t* filter_byte, pxz_payload** out);

/* ---- random access (EXTENSION: the reference always decodes whole images) ------------------------------------------
 * A block's expand depends only on its descriptor, its pixels and its tile size, so a block-aligned window of an image is
 * an ordinary pixlzr image (same trailing-tile rule at its right and bottom edges), and the container's line table lets a
 * reader jump to any block row.  Regions are bit-identical to the same rectangle of the whole decode (DESIGN.md §3).
 *
 * The blocks of columns [c0, c0+nc) x rows [r0, r0+nr) of p, as a payload of the sub-image they tile: width
 * min(W, (c0+nc)*bw) - c0*bw, height likewise, same block size and channels.  Descriptors (value, w, h) are copied, block
 * pixels copied and re-packed densely in row-major window order; per-block expand filters (strategy) and resize tables are
 * kept.  The result is an ordinary payload, independent of p: every call that takes a payload takes it.
 * PXZ_E_ARG: empty or out-of-grid window.  PXZ_E_UNSUPPORTED: a batch payload. */
pxz_status pxz_payload_window(pxz_ctx* ctx, const pxz_payload* p, uint32_t c0, uint32_t r0, uint32_t nc, uint32_t nr,
                              pxz_payload** out);
/* Pixels [x, x+w) x [y, y+h) of the decoded image, bit-identical to that rectangle of pxz_expand_to_image(p, filter_up)
 * (with pxz_ctx_set_fast_resample(1): within +-1 LSB, since a small window may run the other resample kernel family);
 * only the blocks the rectangle touches are read and resampled.  out: w x h, p's channels, not a batch.
 * PXZ_E_ARG: empty rectangle, rectangle outside the image, output geometry mismatch.  PXZ_E_UNSUPPORTED: a batch payload. */
pxz_status pxz_expand_region(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, uint32_t x, uint32_t y, uint32_t w,
                             uint32_t h, pxz_image* out);
/* Header only: dimensions, block size, filter byte (-1 if absent); checks the line table against len.  O(rows). */
pxz_status pxz_container_header(const uint8_t* data, size_t len, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                                int32_t* filter_byte);
/* The .pxlzr file of the block window (c0, r0, nc, nr) of the image in `data`, without decoding: header with the window's
 * size, a new line table, the window's block records copied verbatim.  Reads the header, the line table and the block
 * headers of rows r0 .. r0+nr-1 only; every record of those rows is checked as pxz_container_decode checks it, and each
 * row against its line-table entry.  Consequence: a file that is corrupt only outside the window still crops (and its
 * crop decodes), while pxz_container_decode refuses the whole file.  cap >= len always suffices; out == NULL writes
 * nothing and returns the size of the cropped file.  Byte-identical to the file of the same window written from a payload
 * (pxz_payload_window + pxz_payload_to_container).  Returns the bytes written, or a negative pxz_status: PXZ_E_ARG for an
 * empty or out-of-grid window or a too small `cap`, PXZ_E_FORMAT / PXZ_E_UNSUPPORTED as pxz_container_decode. */
int64_t pxz_container_crop(const uint8_t* data, size_t len, uint32_t c0, uint32_t r0, uint32_t nc, uint32_t nr, uint8_t* out,
                           size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* PIXLZR_B200_H */
