// pxz_internal.h — shared between the host side (abi.cpp, tables.cpp) and the kernels (kernels.cu).
// Not part of the public ABI (that is include/pixlzr_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <tuple>

#include "../../include/pixlzr_b200.h"

namespace pxz {

// One device block cut into typed arrays.  A layout is the list of its arrays, each a pointer to set and an element count;
// the same list gives the block's size (bytes()) and, once the block is allocated, every array's address (place()), so the
// two cannot disagree.  Every array starts at a multiple of kLayoutAlign bytes from the base, as aligned as an allocation of
// its own would be.
constexpr size_t kLayoutAlign = 256;
inline size_t layout_round(size_t bytes) { return (bytes + kLayoutAlign - 1) & ~(kLayoutAlign - 1); }
template <class T>
struct LayoutPart {
  T** ptr;
  size_t n;
  size_t bytes() const { return layout_round(n * sizeof(T)); }
  void place(uint8_t*& at) const {
    *ptr = reinterpret_cast<T*>(at);
    at += bytes();
  }
};
template <class T>
LayoutPart<T> part(T*& ptr, size_t n) { return {&ptr, n}; }
template <class... T>
struct Layout {
  std::tuple<LayoutPart<T>...> parts;
  size_t bytes() const {
    return std::apply([](const auto&... p) { return (size_t{0} + ... + p.bytes()); }, parts);
  }
  void place(void* base) const {
    uint8_t* at = static_cast<uint8_t*>(base);
    std::apply([&](const auto&... p) { (p.place(at), ...); }, parts);
  }
};
template <class... T>
Layout<T...> layout_of(LayoutPart<T>... parts) { return {{parts...}}; }

constexpr int kMaxLevel = 16;              // level exponents 0..16 get their own resample table
constexpr int kLevelsPerClass = kMaxLevel + 1;
constexpr int kThresholds = 41;            // thr[k], k = 0..40: smallest f32 v with round(log2 v) >= -k
constexpr uint32_t kLevelOnePixel = 0xFFu; // "level 0" / below every threshold: 1 px

// One axis of a separable resample: n_in source samples -> n_out outputs.
// Pool layout at `off` (32-bit words): left[n_out] | count[n_out] | weights[n_out * stride] (f32 bits).
// Blocked form at `boff` (outputs in groups of 4, nb = ceil(n_out / 4) groups; pool offset is a multiple of 4 words):
//   w4[rows_total] (float4: the weights of the group's 4 outputs for one source sample, 0 outside an output's
//   window) | lo[nb] | rows[nb] | first[nb] (index of the group's first float4)
// A kernel walks source samples lo .. lo+rows once per group and feeds 4 accumulators, so each accumulator still
// receives its taps in ascending order (adding p * 0 is exact).
//
// Two more forms serve the warp-per-tile kernels (k_shrink_tma / k_expand_warp):
//  * slide2 form at `s2off` (downscale, n_in >= n_out; pool offset and s2words are multiples of 4 words, so one bulk copy
//    stages it): n_in rows of `slots` f32 pairs — pair s of row r holds (w, w), w = the weight of the output o with
//    o % slots == s whose (zero-trimmed) window contains source sample r, else +0; one f32x2 operand whose lanes are two
//    image columns — followed by end[n_out]: the source sample that holds output o's last tap.  One walk over the source
//    samples feeds all live outputs, so every sample is loaded and converted once and no multiply is wasted; each
//    accumulator still sees its taps in ascending order.  slots in {2, 4, 6}; slots = s2words = 0: the table has no
//    slide2 form (more than 6 outputs live at once; k_shrink_warp shrinks those tiles from the blocked form).
//  * gather8 form at `goff` (upscale, every output has <= 7 taps): n_out rows of 8 floats (weights, +0 padded),
//    then left[n_out]; at `gpoff` (multiple of 4 words) ceil(n_out / 2) rows of 8 float pairs
//    (w[2p][i], w[2p+1][i]): two output rows with the same first tap run as the two lanes of one f32x2 operation.
//    goff = 0xFFFFFFFF if an output has more than 7 taps.
//  bpad: upscale tables store every blocked group with bpad (2, 4 or 8) rows; 0 = own lengths.
struct AxisTab {
  uint32_t n_in, n_out, stride, off;
  uint32_t boff, nb, brows_total, bwords;
  uint32_t pad1_, slots, goff, gpoff;
  uint32_t bpad, s2off, s2words, pad2_;  // s2off / s2words: slide2 form (tables.cpp), 0 words = none
};

// fast_image_resize filter kernels (tables.cpp build_axis_table_fir; data_types/mod.rs:65-107 picks them)
enum { PXZ_FIR_NEAREST = 0, PXZ_FIR_BILINEAR = 1, PXZ_FIR_CATMULLROM = 2, PXZ_FIR_GAUSSIAN = 3, PXZ_FIR_LANCZOS3 = 4, PXZ_FIR_HAMMING = 5 };

// Geometry of the block grid over a pitched image.
// A batch is `nimg` images of one size stacked in one pitched allocation, image i at pixel rows [i * img_rows, ...): the
// block grid of the batch is the images' grids one below the other, so `rows` counts the block rows of ALL images
// (cols * rows = blocks of the batch) while H, trail_h and rows_img describe one image.  nimg = 1: a plain image.
struct Geom {
  uint32_t W, H, bw, bh, cols, rows, C;
  uint32_t trail_w, trail_h;  // W % bw, H % bh (0 = no trailing column / row)
  uint32_t rows_img, nimg, img_rows;
};

// How raw metric values become (v0, v1): pixlzr.rs:162 (`x * factor * 10`), :199 (`x * factor`),
// process/mod.rs:110 (identity); optional global normalisation first (extension).
struct ValueMap {
  float factor;
  int mode;       // 0: MAD * factor * 10 | 1: MAD identity | 2: Sobel (hz,vr) * factor
  int normalise;  // 0/1; minmax = {min_x, -max_x, min_y, -max_y} on device
  float extra_thr;  // tree processing: an additional decision threshold on the value (NaN = none), process/tree.rs:56
  // per-block filter strategy: bit k-1 set = the buckets k-1 and k (edge at p = k/64) name different filters, so the
  // fast Oklab-MAD path must resolve that edge exactly as well (guard band)
  unsigned long long bucket_edges = 0;
};

struct LevelThresholds {
  float thr[kThresholds];
};

// Per-block filter pair chosen by the block value (include/pixlzr_b200.h, pxz_strategy; reference: the experiment
// logged in strategies.txt / strategies_by_level.txt).  The bucket is a function of the value STORED with the block
// (sqrt(p0^2 + p1^2), operations.rs:154), so a decoder finds the same filter again: value / sqrt(2) is the quantiser's
// input p when both axes share it (Oklab-MAD), and its root mean square otherwise.
constexpr int kStrategyBuckets = 65;
struct StrategyLut {
  uint32_t on;      // 0: one filter for all blocks
  uint32_t stride;  // tables per filter in the combined table set
  uint8_t down[kStrategyBuckets + 3];
  uint8_t up[kStrategyBuckets + 3];
};
#ifdef __CUDACC__
__host__ __device__
#endif
inline uint32_t strategy_bucket(float value) {
  const float t = value * 45.25483322143555f;  // 64 / sqrt(2), one f32 multiply
  if (!(t > 0.0f)) return 0;                   // zero, negative, NaN
  if (t >= 64.0f) return 64;
  return (uint32_t)t;
}

// Guard band of the fast Oklab-MAD path (DESIGN.md "guard band"): a block is recomputed in reference
// order when its fast value is within the bound of |v_ref - v_fast| of a level threshold.  The bound's
// sequential-summation terms are derived in kernels.cu; `abs_raw` / `rel` cover the fast arithmetic itself.
struct GuardBand {
  float rel;
  float abs_raw;
};

// ---- kernel launchers (kernels.cu) ---------------------------------------------------------
// All return cudaGetLastError() of the launch; *launches is incremented per kernel launched.
// zero_word (may be NULL): a device word the kernel clears — the guard-band list counter launch_analyze_mad_exact
// appends to next (saves a memset launch per image)
cudaError_t launch_analyze_mad_fast(const uint8_t* img, size_t pitch, const Geom& g, float* vx, uint8_t* opaque,
                                    uint32_t* zero_word, cudaStream_t s, int sm_count, uint64_t* launches);
// Reference-order Oklab values.  vx_fast == NULL: every tile.  vx_fast != NULL: the tiles of a list built first from the
// fast values — with vm != NULL the guard band of the level thresholds (k_band_list), with vm == NULL the tiles that can
// hold the minimum or the maximum of the image (k_extreme_list; minmax = {min, -max} of the fast values).  *count must be
// zero when the list is built (launch_analyze_mad_fast's zero_word, or a memset between two lists of one image).
cudaError_t launch_analyze_mad_exact(const uint8_t* img, size_t pitch, const Geom& g, float* vx, const float* vx_fast,
                                     const uint8_t* opaque, const ValueMap* vm, const LevelThresholds* thr, const GuardBand* band,
                                     const float* minmax, uint32_t* list, uint32_t* count, cudaStream_t s, int sm_count,
                                     uint64_t* launches);
cudaError_t launch_analyze_sobel(const uint8_t* img, size_t pitch, const Geom& g, float* vx, float* vy, cudaStream_t s,
                                 int sm_count, uint64_t* launches);
cudaError_t launch_minmax(const float* vx, const float* vy, uint32_t n, float* minmax4, cudaStream_t s,
                          uint64_t* launches);
// mask (may be NULL): blocks with mask[b] == 0 get an empty descriptor (w = h = 0) and are skipped by the resample
cudaError_t launch_plan(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                        const LevelThresholds& thr, const uint8_t* mask, pxz_block_desc* descs, uint32_t* tabidx,
                        uint64_t* total_bytes, void* scan_state, uint32_t* lists, uint32_t cap, cudaStream_t s,
                        uint64_t* launches, const StrategyLut* strategy = nullptr, uint32_t* tabidx_up = nullptr);
// Payload sizes k_plan would compute (mask = NULL) for each of cand.n factors: bytes[i] = sum over blocks of w' * h' * bpp
// with the factor vm.factor replaced by cand.k[i].  bpp: bytes per pixel counted (3 for an RGB image on the RGBA kernels).
constexpr int kMaxSizeCandidates = 256;
struct SizeCandidates {
  uint32_t n;
  float k[kMaxSizeCandidates];
};
cudaError_t launch_size_curve(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                              const LevelThresholds& thr, uint32_t bpp, const SizeCandidates& cand, uint64_t* bytes, cudaStream_t s,
                              int sm_count, uint64_t* launches);
// Work order of the warp-per-tile resample kernels: lists[c * cap + i], c < 8, = the blocks of cost class c (0 = most
// expensive), lists[8 * cap + c] = how many.  launch_plan fills them; this entry point does the same for descriptors
// that came from the host.
constexpr uint32_t kOrderClasses = 8;
#ifdef __CUDACC__
__host__ __device__
#endif
inline size_t order_list_words(size_t cap) { return (size_t)kOrderClasses * cap + kOrderClasses; }
cudaError_t launch_class_lists(const pxz_block_desc* descs, const Geom& g, void* scan_state, uint32_t* lists, uint32_t cap,
                               cudaStream_t s, uint64_t* launches);
// The blocks of columns [c0, c0 + g.cols) x rows [r0, r0 + g.rows) of a payload with pcols columns (descs / meta / pixels of
// capacity pcap) as the payload of geometry g: descriptors with re-packed offsets, table indices (and, with copy_up, the
// expand-side indices), work-order lists, total and pixels, in one launch.  meta: pxz_payload::d_tabidx layout.
// scan_state: window_scan_state_bytes(g.cols * g.rows), zero on entry and on exit (shared with launch_plan).
size_t window_scan_state_bytes(uint32_t nblocks);
cudaError_t launch_payload_window(const pxz_block_desc* pdescs, const uint32_t* pmeta, uint32_t pcap, const uint8_t* ppx, uint32_t pcols,
                                  uint32_t c0, uint32_t r0, const Geom& g, bool copy_up, pxz_block_desc* descs, uint32_t* meta, uint32_t cap,
                                  uint8_t* px, uint64_t* total_bytes, void* scan_state, cudaStream_t s, uint64_t* launches);
// quadtree level (process/tree.rs:47-77): leaf[b] = active && ((v >= thr) ^ positive), recurse[b] = active && !that,
// where active = recurse flag of the parent block one level up (NULL parent = every block is active)
cudaError_t launch_tree_mask(const float* vx, const Geom& g, const uint8_t* parent_recurse, uint32_t parent_cols, float thr,
                             int positive, uint8_t* leaf, uint8_t* recurse, cudaStream_t s, uint64_t* launches);
size_t plan_scan_state_bytes(uint32_t nblocks);
// container stage on the device (qoi_device.cu): per-block QOI streams written from / decoded into the packed payload.
// arena: qoi_arena_bytes(); out: 26 + 4 * rows + arena bytes; *total = bytes of the finished file
size_t qoi_arena_bytes(uint32_t nblocks, uint64_t payload_bytes, uint32_t C);
cudaError_t launch_qoi_encode(const pxz_block_desc* descs, const uint8_t* pixels, const Geom& g, int values_present,
                              uint32_t filter_byte, uint8_t* arena, uint32_t* enc_len, unsigned long long* out_off, uint8_t* out,
                              unsigned long long* total, cudaStream_t s, uint64_t* launches);
cudaError_t launch_qoi_decode(const uint8_t* in, const unsigned long long* in_off, const uint32_t* qlen, const pxz_block_desc* descs,
                              const Geom& g, uint8_t* pixels, int* err, cudaStream_t s, uint64_t* launches);
// per-block error of two images of geometry g (not a batch): sse[b] += sum of (a - b)^2 over the tile, mx[b] = max(mx[b], max |a - b|)
// (mx may be NULL).  Both arrays are zero on entry.
cudaError_t launch_block_error(const uint8_t* a, size_t pa, const uint8_t* b, size_t pb, const Geom& g, uint64_t* sse, uint32_t* mx,
                               cudaStream_t s, int sm_count, uint64_t* launches);
// strategy measure: sse[bucket * kFilterPairs + pair] += block_sse[i] with bucket = strategy_bucket(descs[i].value); count: also
// blocks[bucket] += 1
constexpr uint32_t kFilterPairs = 25;  // pair = down * 5 + up
static_assert(kFilterPairs == PXZ_FILTER_PAIRS, "filter pair count");
cudaError_t launch_bucket_sum(const pxz_block_desc* descs, const uint64_t* block_sse, uint32_t nblocks, uint32_t pair, bool count,
                              uint64_t* sse, uint32_t* blocks, cudaStream_t s, int sm_count, uint64_t* launches);
// Rate-distortion curve (pxz_rd_curve / pxz_shrink_to_error).
// launch_rd_levels: vx[b] = fx, vy[b] = fy for b < n (the forced levels of one error pass).
cudaError_t launch_rd_levels(float* vx, float* vy, uint32_t n, float fx, float fy, cudaStream_t s, int sm_count, uint64_t* launches);
// The error pass of a block at levels (kx, ky): min(kx, cap_x) * stride_x + min(ky, cap_y) * stride_y; block b's error in that
// pass is sse_table[pass * nblocks + b].
struct RdPasses {
  uint32_t cap_x, cap_y, stride_x, stride_y;
};
constexpr uint32_t kRdNoEvent = 0xFFFFFFFFu;  // key of an unused event slot (above every finite factor's bit pattern)
// launch_rd_events: per block, from its raw values (vm.factor ignored) the factors at which its dims change: slot
// b * maxev + i < b * maxev + maxev holds key = the smallest f32 bit pattern with the new dims, dbytes / dsse = the change of
// the block's payload bytes / squared error there (dsse two's complement: it may fall), id = the slot; unused slots have key
// kRdNoEvent and zero changes.  base[0] / base[1] += the bytes / errors of all blocks at pattern 1 (zero on entry).
cudaError_t launch_rd_events(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                             const LevelThresholds& thr, uint32_t bpp, const uint64_t* sse_table, const RdPasses& ps, uint32_t maxev,
                             uint32_t* keys, uint32_t* ids, uint64_t* dbytes, uint64_t* dsse, uint64_t* base, cudaStream_t s,
                             uint64_t* launches);
// launch_rd_curve: the events sorted by key, prefix sums of their changes, one point per distinct key.  Point 0 = pattern 1
// with the base totals; point j = the j-th distinct key with base + the changes up to it.  out: least sse of any point, the
// point count, the first point with sse <= max_sse (0xFFFFFFFF: none).  scratch: rd_curve_scratch_bytes(nev).
struct RdOut {
  unsigned long long least_sse;
  uint32_t count;
  uint32_t first_within;
};
size_t rd_curve_scratch_bytes(uint32_t nev);
cudaError_t launch_rd_curve(const uint32_t* keys, const uint32_t* ids, const uint64_t* dbytes, const uint64_t* dsse, uint32_t nev,
                            const uint64_t* base, uint64_t max_sse, void* scratch, size_t scratch_bytes, uint32_t* pt_key, uint64_t* pt_bytes,
                            uint64_t* pt_sse, RdOut* out, cudaStream_t s, int sm_count, uint64_t* launches);
// Rate-distortion optimised encode (pxz_rdo_*).  The error table has every level pair: block b's error at (lx, ly) is
// sse_table[(lx * (ly_max + 1) + ly) * nblocks + b].  An event is one segment of a block's hull: gain = the error it removes,
// cost = the bytes it adds (both > 0); padding has gain 0, cost 1.
struct RdoEvent {
  unsigned long long gain, cost;
};
// launch_rdo_hull: per block its candidates (one per distinct byte count, from dims scaled_dim(tw, lx) x scaled_dim(th, ly)), the
// lower convex hull of those whose error strictly falls from the 1 x 1 one, and its segments in slots b * maxev + i: ev, the
// pass of the vertex the segment ends at (ev_pass; kRdNoEvent: padding), id = the slot.  pass0[b] = the pass of the first vertex.
// base[0] / base[1] / base[2] += the bytes / errors of all blocks at that vertex / the event count (zero on entry).  maxev + 1
// must bound every tile's distinct byte counts.
cudaError_t launch_rdo_hull(const uint64_t* sse_table, const Geom& g, uint32_t bpp, uint32_t lx_max, uint32_t ly_max, uint32_t maxev, RdoEvent* ev,
                            uint32_t* ids, uint32_t* ev_pass, uint32_t* pass0, uint64_t* base, cudaStream_t s, uint64_t* launches);
// launch_rdo_curve: the events stable-sorted in place by rate gain / cost (descending, exact), rank[slot] = its place in that
// order, and the curve: point 0 = base, point j = base + the first j events (pt_bytes / pt_sse: nev + 1 words).  out: point
// count, the last point with bytes <= max_bytes plus one (0: none), the first with sse <= max_sse (0xFFFFFFFF: none).
// scratch: rdo_curve_scratch_bytes(nev).
struct RdoOut {
  uint32_t count;
  uint32_t best_within;
  uint32_t first_within;
};
size_t rdo_curve_scratch_bytes(uint32_t nev);
cudaError_t launch_rdo_curve(RdoEvent* ev, uint32_t* ids, uint32_t nev, const uint64_t* base, uint64_t max_bytes, uint64_t max_sse, void* scratch,
                             size_t scratch_bytes, uint32_t* rank, uint64_t* pt_bytes, uint64_t* pt_sse, RdoOut* out, cudaStream_t s, int sm_count,
                             uint64_t* launches);
// launch_rdo_levels: vx[b] = 2^-lx, vy[b] = 2^-ly of block b's vertex at curve point j (after its events of rank < j).
cudaError_t launch_rdo_levels(const uint32_t* pass0, const uint32_t* ev_pass, const uint32_t* rank, uint32_t maxev, uint32_t nblocks,
                              uint32_t ly_max, uint32_t j, float* vx, float* vy, cudaStream_t s, int sm_count, uint64_t* launches);
// Which resample kernel family runs (PXZ_RESAMPLE_KERNELS=warp|cta).  Auto: by tile count; Warp: warp-per-tile kernels
// (shrink: k_shrink_tma, then k_shrink_warp for the tiles without a slide2 table; expand: k_expand_warp); Cta: CTA-per-tile
// kernels.  The forced warp family still needs the RGBA fast geometry, tables that have the warp forms and, to shrink, an
// image a tensor map can address; otherwise the CTA-per-tile kernels run.
enum class ResampleKernels { Auto, Warp, Cta };
struct ResampleArgs {
  int direction;  // 0: image tiles -> payload (shrink); 1: payload -> image tiles (expand)
  uint8_t* img;
  size_t pitch;
  Geom g;
  const pxz_block_desc* descs;
  const uint32_t* tabidx;
  uint8_t* payload;
  const AxisTab* tabs;
  const uint32_t* pool;
  uint32_t ntabs;
  uint32_t max_src_px, max_src_dim, max_tmp_px, max_tab_words;  // bounds of the source blocks, intermediate and tables
  uint8_t* scratch;        // non-NULL: global scratch of scratch_per_cta bytes per CTA instead of shared memory (grid CTAs)
  size_t scratch_per_cta;
  int grid;                // CTA-per-tile kernel grid
  bool fused;              // pxz_ctx_set_fast_resample
  const uint8_t* opaque_flags;  // may be NULL: per tile, alpha is 255 everywhere
  uint32_t* tile_counter;  // work counter of the warp-per-tile kernels
  const uint32_t* lists;   // work-order lists of capacity cap (launch_plan)
  uint32_t cap;
  bool warp_tables;        // every table has the forms the warp-per-tile kernels need
  ResampleKernels kernels;
  bool has_noslide;        // shrink: some table has no slide2 form (k_shrink_tma leaves those tiles to k_shrink_warp)
};
cudaError_t launch_resample(const ResampleArgs& a, cudaStream_t s, int sm_count, uint64_t* launches);
size_t resample_smem_bytes(uint32_t max_src_px, uint32_t max_tmp_px, uint32_t C);
// RGB images on the RGBA kernels: widen = 1: RGB rows -> RGBA rows (alpha 255); 0: RGBA rows -> RGB rows
cudaError_t launch_rgb_widen(const uint8_t* src, size_t spitch, uint8_t* dst, size_t dpitch, uint32_t w, uint32_t rows, int widen,
                             cudaStream_t s, int sm_count, uint64_t* launches);
// payload of `sc` channels (descs, pixels, meta = tabidx | order lists | expand-side indices with capacity scap) -> `dc` channels
cudaError_t launch_payload_convert(const pxz_block_desc* sdescs, const uint8_t* spx, const uint32_t* smeta, uint32_t scap,
                                   const uint64_t* stotal, pxz_block_desc* ddescs, uint8_t* dpx, uint32_t* dmeta, uint32_t dcap,
                                   uint64_t* dtotal, uint32_t nblocks, int sc, int dc, cudaStream_t s, int sm_count, uint64_t* launches);
// `fir` resize semantics (integer convolution, horizontal pass first, pre-multiplied alpha): one CTA per block
size_t resample_fir_smem_bytes(uint32_t max_src_px, uint32_t max_tmp_px, uint32_t C);
cudaError_t launch_resample_fir(int direction, uint8_t* img, size_t pitch, const Geom& g, const pxz_block_desc* descs,
                                const uint32_t* tabidx, uint8_t* payload, const AxisTab* tabs, const uint32_t* pool, size_t smem,
                                uint32_t src_cap_bytes, cudaStream_t s, int sm_count, uint64_t* launches);
constexpr uint32_t kFirNearestFlag = 0x100u;  // AxisTab::pad2_ of a fir table: precision | this flag for ResizeAlg::Nearest
int resample_grid(int sm_count, uint32_t nblocks);

}  // namespace pxz
