// abi.cpp — implementation of the C ABI in include/pixlzr_b200.h: context / stream / scratch
// management, resample-table caching, and the stream-ordered pipelines
//
//   pxz_shrink : analyse -> [min/max (+ NCCL)] -> guard-band recompute -> plan (scan) -> resample
//   pxz_expand : resample (payload -> tiles of the pitched image)
//
// which replace the bodies of Pixlzr::shrink_by / shrink_directionally / expand / to_image
// (src/data_types/pixlzr.rs:77-205, pixlzr_image.rs:24-74).  No CPU fallback exists.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <new>
#include <string>
#include <tuple>
#include <vector>

#include "pxz_host.h"

using namespace pxz;

// -------------------------------------------------------------------------------------------------
// objects
// -------------------------------------------------------------------------------------------------
namespace {

// index-aligned list of (reduced size, tile size) pairs that a payload's tabidx refers to
struct TabSpec {
  std::vector<uint32_t> n_small, n_tile;
};

struct TabSet {  // device copy of the axis tables of one (spec, filter, direction)
  AxisTab* d_tabs = nullptr;
  uint32_t* d_pool = nullptr;
  uint32_t max_words = 0;  // largest single table (left | count | weights), in 32-bit words
  uint32_t ntabs = 0;
  bool warp_ok = false;    // every table has the form the warp-per-tile kernels need
  bool has_noslide = false;  // direction 0: some table has no slide2 form (k_shrink_tma leaves those tiles to k_shrink_warp)
};

using TabKey = std::tuple<std::vector<uint32_t>, std::vector<uint32_t>, int, int>;

// K_REGION_COPY times the device-to-device copy of pxz_expand_region out of its staging image (not a kernel)
enum KernelId { K_MAD_FAST = 0, K_MAD_EXACT, K_SOBEL, K_MINMAX, K_PLAN, K_RESAMPLE_DOWN, K_RESAMPLE_UP, K_QOI_ENCODE, K_QOI_DECODE,
                K_PAYLOAD_WINDOW, K_REGION_COPY, K_SIZE_CURVE, K_BLOCK_ERROR, K_BUCKET_SUM, K_RD_LEVELS, K_RD_EVENTS, K_RD_CURVE,
                K_RDO_HULL, K_RDO_CURVE, K_RDO_LEVELS, K_COUNT };
const char* const kKernelNames[K_COUNT] = {"analyze_mad_fast", "mad_exact",      "analyze_sobel", "minmax",
                                           "plan",             "resample_down",  "resample_up",   "qoi_encode",
                                           "qoi_decode",       "payload_window", "region_copy",   "size_curve",
                                           "block_error",      "bucket_sum",     "rd_levels",     "rd_events",
                                           "rd_curve",         "rdo_hull",       "rdo_curve",     "rdo_levels"};
struct ProfRec {
  int id;
  cudaEvent_t a, b;
};

}  // namespace

// device buffers of a released payload, kept by the context for the next pxz_shrink / pxz_payload_upload so that
// steady-state calls neither touch the allocator nor share blocks with other streams' contexts
struct PayloadBufs {
  pxz_block_desc* d_descs = nullptr;
  uint32_t* d_tabidx = nullptr;
  uint8_t* d_pixels = nullptr;
  uint64_t* d_total = nullptr;
  size_t nblocks = 0;
  uint64_t capacity = 0;
};

struct pxz_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  size_t max_smem_optin = 0;
  std::string err;
  uint64_t launches = 0;
  LevelThresholds thr{};
  StrategyLut strategy{};  // on = 0 unless pxz_ctx_set_strategy installed a table
  GuardBand band{};
  // scratch, grown on demand
  float* d_vx = nullptr;
  float* d_vy = nullptr;
  uint8_t* d_opaque = nullptr;
  uint32_t* d_list = nullptr;  // [values_cap + 1]: banded tile indices, last word = count
  size_t values_cap = 0;
  float* d_minmax = nullptr;
  uint32_t* d_tile_counter = nullptr;  // work counter of the warp-per-tile resample kernels (they leave it at 0)
  ResampleKernels resample_kernels = ResampleKernels::Auto;  // PXZ_RESAMPLE_KERNELS
  void* d_scan = nullptr;
  size_t scan_cap = 0;
  uint8_t* d_scratch = nullptr;
  size_t scratch_cap = 0;
  uint64_t* h_total = nullptr;  // pinned
  std::map<TabKey, TabSet> tabs;
  void* comm = nullptr;
  bool fast_resample = false;
  int resize_semantics = PXZ_RESIZE_IMAGE_RS;  // which branch of PixlzrBlock::resize (pxz_ctx_set_resize_semantics)
  std::vector<PayloadBufs> payload_cache;  // at most kPayloadCacheMax entries
  // per-kernel timing
  bool profiling = false;
  std::vector<ProfRec> prof_open;
  std::vector<cudaEvent_t> prof_pool;
  double prof_ms[K_COUNT] = {0};
  uint64_t prof_n[K_COUNT] = {0};
};

struct pxz_image {
  pxz_ctx* ctx;
  uint8_t* d;
  size_t pitch;
  uint32_t w, h, c;
  bool owned;
  uint32_t nimg = 1;  // > 1: a batch, image i at rows [i * h, (i + 1) * h) of the allocation
};

constexpr size_t kPayloadCacheMax = 4;
constexpr size_t kTabCacheMax = 48;  // table sets kept per context (get_tabset)

struct pxz_payload {
  pxz_ctx* ctx;
  Geom g;
  size_t nblocks_cap = 0;
  pxz_block_desc* d_descs = nullptr;
  uint32_t* d_tabidx = nullptr;  // [nblocks_cap] table indices, then the work-order lists (launch_plan) of capacity nblocks_cap
  uint32_t* d_order() const { return d_tabidx + nblocks_cap; }
  uint32_t* d_up() const { return d_order() + order_list_words(nblocks_cap); }  // [nblocks_cap] expand-side indices (strategy)
  // 0: one filter per call | 1: per-block filters, expand indices in d_up() (pxz_shrink) | 2: ... in d_tabidx (upload)
  int strategy = 0;
  uint8_t* d_pixels = nullptr;
  uint64_t capacity = 0;
  uint64_t* d_total = nullptr;
  bool bytes_known = false;
  uint64_t bytes = 0;
  std::shared_ptr<TabSpec> spec;
  uint32_t max_small_px = 0;  // largest reduced block (pixels)
  uint32_t max_small_dim = 0; // largest reduced block side
  uint32_t max_tmp_down = 0;  // largest vertical-pass intermediate when shrinking / expanding (pixels)
  uint32_t max_tmp_up = 0;
};

namespace {

pxz_status fail(pxz_ctx* ctx, pxz_status st, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return st;
}

// A launch or an asynchronous call returned the error e: clear it and report "<what>: <error>" with status st
pxz_status cuda_fail(pxz_ctx* ctx, cudaError_t e, const char* what, pxz_status st = PXZ_E_CUDA) {
  cudaGetLastError();
  return fail(ctx, st, std::string(what) + ": " + cudaGetErrorString(e));
}

#define PXZ_CUDA(ctx, expr)                                                                             \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess) return cuda_fail((ctx), _e, #expr, _e == cudaErrorMemoryAllocation ? PXZ_E_OOM : PXZ_E_CUDA); \
  } while (0)

// records an event pair around one kernel launch while profiling is on
struct ProfScope {
  pxz_ctx* ctx;
  ProfRec rec;
  bool live = false;
  ProfScope(pxz_ctx* c, int id) : ctx(c) {
    if (!c->profiling) return;
    auto take = [&](cudaEvent_t* e) {
      if (!c->prof_pool.empty()) {
        *e = c->prof_pool.back();
        c->prof_pool.pop_back();
        return true;
      }
      return cudaEventCreate(e) == cudaSuccess;
    };
    rec.id = id;
    if (!take(&rec.a)) return;
    if (!take(&rec.b)) { c->prof_pool.push_back(rec.a); return; }
    cudaEventRecord(rec.a, c->stream);
    live = true;
  }
  ~ProfScope() {
    if (!live) return;
    cudaEventRecord(rec.b, ctx->stream);
    ctx->prof_open.push_back(rec);
  }
};

// one launch (`launch()` returns its cudaError_t) timed under the profile id `prof`; a failure is reported as cuda_fail(what)
template <class F>
pxz_status profiled(pxz_ctx* ctx, int prof, const char* what, F&& launch) {
  cudaError_t e;
  {
    ProfScope scope(ctx, prof);
    e = launch();
  }
  return e == cudaSuccess ? PXZ_OK : cuda_fail(ctx, e, what);
}

// the filters of pxz_filter
inline bool known_filter(pxz_filter f) { return (int)f >= 0 && (int)f <= 4; }

inline uint32_t ceil_div_u32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a + b - 1) / b); }

pxz_status make_geom(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t c, uint32_t bw, uint32_t bh, Geom* g, uint32_t nimg = 1) {
  if (w == 0 || h == 0 || nimg == 0) return fail(ctx, PXZ_E_ARG, "empty image");
  if (c != 3 && c != 4) return fail(ctx, PXZ_E_ARG, "channels must be 3 (RGB8) or 4 (RGBA8)");
  if (bw == 0 || bh == 0) return fail(ctx, PXZ_E_ARG, "block size must be >= 1 (the reference divides by it)");
  if (bw > 65535u || bh > 65535u) return fail(ctx, PXZ_E_UNSUPPORTED, "block size above 65535 is not supported");
  g->W = w; g->H = h; g->bw = bw; g->bh = bh; g->C = c;
  g->cols = ceil_div_u32(w, bw);  // == ceil(w as f64 / bw as f64), split.rs:45-46
  g->rows_img = ceil_div_u32(h, bh);
  g->nimg = nimg;
  g->img_rows = h;
  g->trail_w = w % bw;
  g->trail_h = h % bh;
  if ((uint64_t)g->cols * g->rows_img * nimg > 0x7FFFFFFFull) return fail(ctx, PXZ_E_UNSUPPORTED, "more than 2^31 blocks");
  if ((uint64_t)h * nimg > 0xFFFFFFFFull) return fail(ctx, PXZ_E_UNSUPPORTED, "batch taller than 2^32 rows");
  g->rows = g->rows_img * nimg;  // block rows of the whole batch
  return PXZ_OK;
}

pxz_status dev_alloc(pxz_ctx* ctx, void** p, size_t bytes) {
  *p = nullptr;
  PXZ_CUDA(ctx, cudaMallocAsync(p, bytes ? bytes : 16, ctx->stream));
  return PXZ_OK;
}
void dev_free(pxz_ctx* ctx, void* p) {
  if (p) cudaFreeAsync(p, ctx->stream);
}

// the dev_alloc blocks of one call (at most five), freed stream-ordered in allocation order when the owner goes out of scope
struct DevBlocks {
  pxz_ctx* ctx;
  void* blocks[5] = {};
  int n = 0;
  explicit DevBlocks(pxz_ctx* c) : ctx(c) {}
  DevBlocks(const DevBlocks&) = delete;
  DevBlocks& operator=(const DevBlocks&) = delete;
  ~DevBlocks() {
    for (int i = 0; i < n; ++i) dev_free(ctx, blocks[i]);
  }
  template <class T>
  pxz_status alloc(T** out, size_t bytes) {
    void* q = nullptr;
    const pxz_status st = dev_alloc(ctx, &q, bytes);
    if (st != PXZ_OK) return st;
    blocks[n++] = q;
    *out = static_cast<T*>(q);
    return PXZ_OK;
  }
  void keep() { n = 0; }  // the blocks have another owner now
};

// scan_bytes: the scan state the next plan / window launch needs (0: launch_plan's for nblocks)
pxz_status ensure_scratch(pxz_ctx* ctx, uint32_t nblocks, size_t scan_bytes = 0) {
  if (ctx->values_cap < nblocks) {
    dev_free(ctx, ctx->d_vx);
    dev_free(ctx, ctx->d_vy);
    dev_free(ctx, ctx->d_opaque);
    dev_free(ctx, ctx->d_list);
    ctx->d_vx = ctx->d_vy = nullptr;
    ctx->d_opaque = nullptr;
    ctx->d_list = nullptr;
    ctx->values_cap = 0;
    pxz_status st;
    if ((st = dev_alloc(ctx, (void**)&ctx->d_vx, (size_t)nblocks * 4)) != PXZ_OK) return st;
    if ((st = dev_alloc(ctx, (void**)&ctx->d_vy, (size_t)nblocks * 4)) != PXZ_OK) return st;
    if ((st = dev_alloc(ctx, (void**)&ctx->d_opaque, (size_t)nblocks)) != PXZ_OK) return st;
    if ((st = dev_alloc(ctx, (void**)&ctx->d_list, ((size_t)nblocks + 1) * 4)) != PXZ_OK) return st;
    ctx->values_cap = nblocks;
  }
  const size_t need = scan_bytes ? scan_bytes : plan_scan_state_bytes(nblocks);
  if (ctx->scan_cap < need) {
    dev_free(ctx, ctx->d_scan);
    ctx->d_scan = nullptr;
    ctx->scan_cap = 0;
    pxz_status st;
    if ((st = dev_alloc(ctx, &ctx->d_scan, need)) != PXZ_OK) return st;
    // the plan / work-order kernels find this zeroed and leave it zeroed
    PXZ_CUDA(ctx, cudaMemsetAsync(ctx->d_scan, 0, need, ctx->stream));
    ctx->scan_cap = need;
  }
  return PXZ_OK;
}

// table index layout of payloads produced by pxz_shrink: (axis * 2 + trailing) * 17 + level
std::shared_ptr<TabSpec> spec_for_geom(const Geom& g) {
  auto sp = std::make_shared<TabSpec>();
  const uint32_t n_of[4] = {g.bw, g.trail_w ? g.trail_w : g.bw, g.bh, g.trail_h ? g.trail_h : g.bh};
  for (int a = 0; a < 4; ++a) {
    for (int k = 0; k <= kMaxLevel; ++k) {
      const uint32_t n = n_of[a];
      uint32_t nn = (uint32_t)(((uint64_t)n + ((1ull << k) - 1)) >> k);
      if (nn < 1) nn = 1;
      sp->n_small.push_back(nn);
      sp->n_tile.push_back(n);
    }
  }
  return sp;
}

// direction 0: tile -> reduced (filter_down); 1: reduced -> tile (filter_up)
pxz_status get_tabset(pxz_ctx* ctx, const TabSpec& spec, int filter, int direction, TabSet* out) {
  const bool fir = ctx->resize_semantics == PXZ_RESIZE_FIR;
  TabKey key(spec.n_small, spec.n_tile, filter, direction + (fir ? 2 : 0));
  auto it = ctx->tabs.find(key);
  if (it != ctx->tabs.end()) {
    *out = it->second;
    return PXZ_OK;
  }
  // filter < 0: the tables of all five filters one after the other (index = filter * spec size + i), for payloads
  // whose blocks carry their own filter (pxz_ctx_set_strategy)
  const size_t per_filter = spec.n_small.size();
  const int f0 = filter < 0 ? 0 : filter, f1 = filter < 0 ? 4 : filter;
  std::vector<AxisTab> tabs(per_filter * (size_t)(f1 - f0 + 1));
  std::vector<uint32_t> pool;
  for (int f = f0; f <= f1; ++f) {
    std::map<std::pair<uint32_t, uint32_t>, AxisTab> seen;
    for (size_t i = 0; i < per_filter; ++i) {
      AxisTab& t = tabs[(size_t)(f - f0) * per_filter + i];
      const uint32_t n_in = direction == 0 ? spec.n_tile[i] : spec.n_small[i];
      const uint32_t n_out = direction == 0 ? spec.n_small[i] : spec.n_tile[i];
      auto s = seen.find({n_in, n_out});
      if (s != seen.end()) {
        t = s->second;
        continue;
      }
      if (fir) {
        // FilterType::to_fir_resizing_algorithm (data_types/mod.rs:65-107): Triangle is Hamming when a block shrinks and
        // Bilinear when it grows; the other filters keep their kernel, Nearest stays nearest
        const int alg = f == PXZ_NEAREST ? PXZ_FIR_NEAREST : f == PXZ_TRIANGLE ? (direction == 0 ? PXZ_FIR_HAMMING : PXZ_FIR_BILINEAR)
                        : f == PXZ_CATMULLROM ? PXZ_FIR_CATMULLROM : f == PXZ_GAUSSIAN ? PXZ_FIR_GAUSSIAN : PXZ_FIR_LANCZOS3;
        if (!build_axis_table_fir(n_in, n_out, alg, &pool, &t)) return fail(ctx, PXZ_E_ARG, "bad resample table request");
      } else if (!build_axis_table(n_in, n_out, f, &pool, &t)) {
        return fail(ctx, PXZ_E_ARG, "bad resample table request");
      }
      seen[{n_in, n_out}] = t;
    }
  }
  pool.resize(pool.size() + 16, 0u);  // staged copies are rounded up to 16 bytes
  TabSet ts;
  ts.ntabs = (uint32_t)tabs.size();
  ts.warp_ok = true;
  for (const AxisTab& t : tabs) {
    ts.max_words = std::max(ts.max_words, std::max(2 * t.n_out + t.n_out * t.stride, t.bwords));
    if (direction == 1 && t.goff == 0xFFFFFFFFu) ts.warp_ok = false;
    if (direction == 0 && t.s2words == 0) ts.has_noslide = true;
  }
  // the cache is bounded: payloads built from host descriptors (decoded files, PixlzrBlock::resize size pairs) bring
  // their own size sets, and a long-running decoder must not pile their tables up.  Frees are stream-ordered, so kernels
  // already queued on this context's stream keep their tables.
  if (ctx->tabs.size() >= kTabCacheMax) {
    for (auto& kv : ctx->tabs) {
      dev_free(ctx, kv.second.d_tabs);
      dev_free(ctx, kv.second.d_pool);
    }
    ctx->tabs.clear();
  }
  DevBlocks bufs(ctx);
  pxz_status st;
  if ((st = bufs.alloc(&ts.d_tabs, tabs.size() * sizeof(AxisTab))) != PXZ_OK) return st;
  if ((st = bufs.alloc(&ts.d_pool, pool.size() * 4)) != PXZ_OK) return st;
  // pageable -> device copies are staged by the runtime before returning, so the vectors may die
  cudaError_t ce = cudaMemcpyAsync(ts.d_tabs, tabs.data(), tabs.size() * sizeof(AxisTab), cudaMemcpyHostToDevice, ctx->stream);
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(ts.d_pool, pool.data(), pool.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  if (ce != cudaSuccess) return cuda_fail(ctx, ce, "resample table upload");
  bufs.keep();  // the cache owns them
  ctx->tabs[key] = ts;
  *out = ts;
  return PXZ_OK;
}

pxz_status run_resample(pxz_ctx* ctx, int direction, uint8_t* img, size_t pitch, const pxz_payload* p, const TabSet& ts,
                        uint32_t max_src_px, uint32_t max_src_dim, uint32_t max_tmp_px, const uint8_t* opaque_flags = nullptr) {
  const Geom& g = p->g;
  const uint32_t nblocks = g.cols * g.rows;
  if (ctx->resize_semantics == PXZ_RESIZE_FIR) {
    // integer convolution, horizontal pass first: its own kernel (one CTA per block, source + u8 intermediate in smem)
    const uint32_t tmp_px = max_src_dim * std::max(g.bw, max_src_dim);  // source rows x widest destination row
    const size_t fsmem = resample_fir_smem_bytes(max_src_px, tmp_px, g.C);
    if (fsmem > ctx->max_smem_optin) return fail(ctx, PXZ_E_UNSUPPORTED, "blocks too large for the fir resize path");
    ProfScope prof(ctx, direction == 0 ? K_RESAMPLE_DOWN : K_RESAMPLE_UP);
    const uint32_t* tabidx = (direction == 1 && p->strategy == 1) ? p->d_up() : p->d_tabidx;
    PXZ_CUDA(ctx, launch_resample_fir(direction, img, pitch, g, p->d_descs, tabidx, p->d_pixels, ts.d_tabs, ts.d_pool, fsmem,
                                      (uint32_t)(((size_t)max_src_px * g.C + 15) & ~(size_t)15), ctx->stream, ctx->sm_count, &ctx->launches));
    return PXZ_OK;
  }
  size_t smem = resample_smem_bytes(max_src_px, max_tmp_px, g.C);
  int grid = resample_grid(ctx->sm_count, nblocks);
  uint8_t* scratch = nullptr;
  size_t per_cta = 0;
  if (smem > ctx->max_smem_optin) {  // tiles too large for shared memory
    per_cta = (smem + 255) & ~(size_t)255;
    grid = std::min<int>(grid, ctx->sm_count * 2);
    const size_t need = per_cta * (size_t)grid;
    if (ctx->scratch_cap < need) {
      dev_free(ctx, ctx->d_scratch);
      ctx->d_scratch = nullptr;
      ctx->scratch_cap = 0;
      pxz_status st;
      if ((st = dev_alloc(ctx, (void**)&ctx->d_scratch, need)) != PXZ_OK) return st;
      ctx->scratch_cap = need;
    }
    scratch = ctx->d_scratch;
  }
  ResampleArgs a;
  a.direction = direction;
  a.img = img;
  a.pitch = pitch;
  a.g = g;
  a.descs = p->d_descs;
  a.tabidx = (direction == 1 && p->strategy == 1) ? p->d_up() : p->d_tabidx;
  a.payload = p->d_pixels;
  a.tabs = ts.d_tabs;
  a.pool = ts.d_pool;
  a.ntabs = ts.ntabs;
  a.max_src_px = max_src_px;
  a.max_src_dim = max_src_dim;
  a.max_tmp_px = max_tmp_px;
  a.max_tab_words = ts.max_words;
  a.scratch = scratch;
  a.scratch_per_cta = per_cta;
  a.grid = grid;
  a.fused = ctx->fast_resample;
  a.opaque_flags = opaque_flags;
  a.tile_counter = ctx->d_tile_counter;
  a.lists = p->d_order();
  a.cap = (uint32_t)p->nblocks_cap;
  a.warp_tables = ts.warp_ok;
  a.kernels = ctx->resample_kernels;
  a.has_noslide = ts.has_noslide;
  ProfScope prof(ctx, direction == 0 ? K_RESAMPLE_DOWN : K_RESAMPLE_UP);
  PXZ_CUDA(ctx, launch_resample(a, ctx->stream, ctx->sm_count, &ctx->launches));
  return PXZ_OK;
}

void payload_release(pxz_payload* p) {
  if (!p) return;
  pxz_ctx* ctx = p->ctx;
  if (p->d_descs && p->d_tabidx && p->d_pixels && p->d_total && ctx->payload_cache.size() < kPayloadCacheMax) {
    PayloadBufs b;
    b.d_descs = p->d_descs; b.d_tabidx = p->d_tabidx; b.d_pixels = p->d_pixels; b.d_total = p->d_total;
    b.nblocks = p->nblocks_cap; b.capacity = p->capacity;
    ctx->payload_cache.push_back(b);  // stream order makes the reuse safe: later work on this ctx runs after ours
  } else {
    dev_free(ctx, p->d_descs);
    dev_free(ctx, p->d_tabidx);
    dev_free(ctx, p->d_pixels);
    dev_free(ctx, p->d_total);
  }
  delete p;
}

// owners of a payload / an image on the internal paths: released when the owner goes out of scope
struct PayloadRelease {
  void operator()(pxz_payload* p) const { payload_release(p); }
};
using PayloadOwner = std::unique_ptr<pxz_payload, PayloadRelease>;
struct ImageFree {
  void operator()(pxz_image* im) const { pxz_image_free(im); }
};
using ImageOwner = std::unique_ptr<pxz_image, ImageFree>;

pxz_status image_new(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t c, uint32_t nimg, ImageOwner* out) {
  pxz_image* im = nullptr;
  const pxz_status st = pxz_image_alloc_batch(ctx, w, h, c, nimg, &im);
  out->reset(im);
  return st;
}

inline uint32_t pad8(uint32_t v) { return (v + 7u) & ~7u; }  // intermediate rows are padded to 8 columns

// shared-memory bounds of the two resample directions for a payload planned on g (every block at most its tile);
// coupled: both axes share the level (Oklab MAD)
void set_plan_bounds(pxz_payload* p, const Geom& g, bool coupled) {
  p->max_small_px = g.bw * g.bh;
  p->max_small_dim = std::max(g.bw, g.bh);
  if (coupled) {
    p->max_tmp_down = ((g.bh + 1) / 2) * pad8(g.bw);  // dh <= ceil(th/2), sw = tw
    p->max_tmp_up = g.bh * pad8((g.bw + 1) / 2);      // dh = th, sw <= ceil(tw/2)
    // a 1-px-wide/-high trailing tile keeps that axis while the other shrinks: still within the bounds
  } else {
    p->max_tmp_down = g.bh * pad8(g.bw);
    p->max_tmp_up = g.bh * pad8(g.bw);
  }
}

// a payload over the same blocks as src (another channel count, a window): same tables, filters and bounds
void copy_layout(pxz_payload* dst, const pxz_payload* src) {
  dst->spec = src->spec;
  dst->strategy = src->strategy;
  dst->max_small_px = src->max_small_px;
  dst->max_small_dim = src->max_small_dim;
  dst->max_tmp_down = src->max_tmp_down;
  dst->max_tmp_up = src->max_tmp_up;
}

pxz_status ctx_create_common(int device, cudaStream_t stream, bool own, pxz_ctx** out) {
  if (!out) return PXZ_E_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return PXZ_E_CUDA;
  }
  if (device < 0 || device >= n) return PXZ_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return PXZ_E_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PXZ_E_CUDA;
  pxz_ctx* ctx = new (std::nothrow) pxz_ctx();
  if (!ctx) return PXZ_E_OOM;
  ctx->device = device;
  if (prop.major != 10) {
    // the library only carries sm_100a code; refuse loudly instead of failing at the first launch
    fprintf(stderr, "pixlzr_b200: device %d is sm_%d%d, need sm_100 (B200)\n", device, prop.major, prop.minor);
    delete ctx;
    return PXZ_E_CUDA;
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->max_smem_optin = prop.sharedMemPerBlockOptin;
  if (own) {
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return PXZ_E_CUDA; }
    ctx->own_stream = true;
  } else {
    ctx->stream = stream;
  }
  // keep freed blocks in the stream-ordered pool: alloc/free per call must not hit the driver
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thresh = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh);
  }
  build_level_thresholds(&ctx->thr);
  ctx->band.rel = 2.0e-5f;     // fast arithmetic, relative
  ctx->band.abs_raw = 8.0e-6f; // fast arithmetic, absolute (SFU cube roots; measured <= 4e-6)
  if (const char* e = getenv("PXZ_RESAMPLE_KERNELS"))
    ctx->resample_kernels = !strcmp(e, "warp") ? ResampleKernels::Warp
                            : !strcmp(e, "cta") ? ResampleKernels::Cta
                                                : ResampleKernels::Auto;
  if (cudaMalloc((void**)&ctx->d_minmax, 8 * sizeof(float)) != cudaSuccess ||
      cudaMalloc((void**)&ctx->d_tile_counter, 64) != cudaSuccess || cudaMemset(ctx->d_tile_counter, 0, 64) != cudaSuccess ||
      cudaMallocHost((void**)&ctx->h_total, 64) != cudaSuccess) {
    cudaGetLastError();
    delete ctx;
    return PXZ_E_OOM;
  }
  *out = ctx;
  return PXZ_OK;
}

}  // namespace

// -------------------------------------------------------------------------------------------------
// C ABI
// -------------------------------------------------------------------------------------------------
extern "C" {

int pxz_abi_version(void) { return PXZ_ABI_VERSION; }

int pxz_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

pxz_status pxz_ctx_create(int device, pxz_ctx** out) { return ctx_create_common(device, nullptr, true, out); }

pxz_status pxz_ctx_create_on_stream(int device, void* cuda_stream, pxz_ctx** out) {
  return ctx_create_common(device, (cudaStream_t)cuda_stream, false, out);
}

void pxz_ctx_destroy(pxz_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->comm) nccl_comm_destroy(ctx->comm);
  for (auto& b : ctx->payload_cache) {
    dev_free(ctx, b.d_descs); dev_free(ctx, b.d_tabidx); dev_free(ctx, b.d_pixels); dev_free(ctx, b.d_total);
  }
  ctx->payload_cache.clear();
  for (auto& kv : ctx->tabs) {
    dev_free(ctx, kv.second.d_tabs);
    dev_free(ctx, kv.second.d_pool);
  }
  dev_free(ctx, ctx->d_vx);
  dev_free(ctx, ctx->d_vy);
  dev_free(ctx, ctx->d_opaque);
  dev_free(ctx, ctx->d_list);
  dev_free(ctx, ctx->d_scan);
  dev_free(ctx, ctx->d_scratch);
  cudaStreamSynchronize(ctx->stream);
  for (auto& r : ctx->prof_open) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto& e : ctx->prof_pool) cudaEventDestroy(e);
  cudaFree(ctx->d_minmax);
  cudaFree(ctx->d_tile_counter);
  cudaFreeHost(ctx->h_total);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* pxz_last_error(const pxz_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

pxz_status pxz_synchronize(pxz_ctx* ctx) {
  if (!ctx) return PXZ_E_ARG;
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

uint64_t pxz_launch_count(const pxz_ctx* ctx) { return ctx ? ctx->launches : 0; }

pxz_status pxz_ctx_set_resize_semantics(pxz_ctx* ctx, pxz_resize_semantics semantics) {
  if (!ctx) return PXZ_E_ARG;
  if (semantics != PXZ_RESIZE_IMAGE_RS && semantics != PXZ_RESIZE_FIR) return fail(ctx, PXZ_E_ARG, "unknown resize semantics");
  ctx->resize_semantics = (int)semantics;
  return PXZ_OK;
}

pxz_status pxz_ctx_set_fast_resample(pxz_ctx* ctx, int on) {
  if (!ctx) return PXZ_E_ARG;
  ctx->fast_resample = on != 0;
  return PXZ_OK;
}

// ---- per-block filter pairs (strategies.txt / strategies_by_level.txt) ----------------------------------------
uint32_t pxz_strategy_bucket(float block_value) { return strategy_bucket(block_value); }

pxz_status pxz_strategy_by_level(pxz_strategy* out) {
  if (!out) return PXZ_E_ARG;
  // strategies_by_level.txt:1-12 (= strategies.txt, one line per bucket of width 1/64)
  for (int b = 0; b < PXZ_STRATEGY_BUCKETS; ++b) {
    pxz_filter down = PXZ_LANCZOS3, up = PXZ_LANCZOS3;  // v in [0.0625; 0.703125)
    if (b == 0) { down = PXZ_NEAREST; up = PXZ_NEAREST; }            // v < 0.015625
    else if (b == 1) { down = PXZ_TRIANGLE; up = PXZ_NEAREST; }      // [0.015625; 0.03125)
    else if (b == 2) { down = PXZ_CATMULLROM; up = PXZ_LANCZOS3; }   // [0.03125; 0.046875)
    else if (b == 3) { down = PXZ_LANCZOS3; up = PXZ_CATMULLROM; }   // [0.046875; 0.0625)
    else if (b >= 45) { down = PXZ_NEAREST; up = PXZ_NEAREST; }      // v >= 0.703125
    out->down[b] = (uint8_t)down;
    out->up[b] = (uint8_t)up;
  }
  return PXZ_OK;
}

pxz_status pxz_ctx_set_strategy(pxz_ctx* ctx, const pxz_strategy* strategy) {
  if (!ctx) return PXZ_E_ARG;
  if (!strategy) {
    ctx->strategy.on = 0;
    return PXZ_OK;
  }
  for (int b = 0; b < PXZ_STRATEGY_BUCKETS; ++b)
    if (strategy->down[b] > 4 || strategy->up[b] > 4) return fail(ctx, PXZ_E_ARG, "unknown filter in the strategy table");
  static_assert(PXZ_STRATEGY_BUCKETS == kStrategyBuckets, "bucket count");
  memcpy(ctx->strategy.down, strategy->down, PXZ_STRATEGY_BUCKETS);
  memcpy(ctx->strategy.up, strategy->up, PXZ_STRATEGY_BUCKETS);
  ctx->strategy.on = 1;
  return PXZ_OK;
}

static pxz_status prof_drain(pxz_ctx* ctx) {
  if (ctx->prof_open.empty()) return PXZ_OK;
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& r : ctx->prof_open) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ctx->prof_ms[r.id] += ms;
      ctx->prof_n[r.id] += 1;
    }
    ctx->prof_pool.push_back(r.a);
    ctx->prof_pool.push_back(r.b);
  }
  ctx->prof_open.clear();
  return PXZ_OK;
}

pxz_status pxz_profile_enable(pxz_ctx* ctx, int on) {
  if (!ctx) return PXZ_E_ARG;
  pxz_status st = prof_drain(ctx);
  if (st != PXZ_OK) return st;
  if (on) {
    for (int i = 0; i < K_COUNT; ++i) { ctx->prof_ms[i] = 0; ctx->prof_n[i] = 0; }
  }
  ctx->profiling = on != 0;
  return PXZ_OK;
}

const char* pxz_profile_kernel_name(int kernel_id) {
  return (kernel_id >= 0 && kernel_id < K_COUNT) ? kKernelNames[kernel_id] : nullptr;
}

pxz_status pxz_profile_read(pxz_ctx* ctx, int kernel_id, double* total_ms, uint64_t* launches) {
  if (!ctx || kernel_id < 0 || kernel_id >= K_COUNT) return PXZ_E_ARG;
  pxz_status st = prof_drain(ctx);
  if (st != PXZ_OK) return st;
  if (total_ms) *total_ms = ctx->prof_ms[kernel_id];
  if (launches) *launches = ctx->prof_n[kernel_id];
  return PXZ_OK;
}

pxz_status pxz_host_alloc(size_t bytes, void** out) {
  if (!out) return PXZ_E_ARG;
  if (cudaMallocHost(out, bytes ? bytes : 1) != cudaSuccess) {
    cudaGetLastError();
    *out = nullptr;
    return PXZ_E_OOM;
  }
  return PXZ_OK;
}
void pxz_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

pxz_status pxz_grid(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t* cols, uint32_t* rows) {
  if (!cols || !rows || bw == 0 || bh == 0) return PXZ_E_ARG;
  *cols = ceil_div_u32(w, bw);
  *rows = ceil_div_u32(h, bh);
  return PXZ_OK;
}

// ---- images ---------------------------------------------------------------------------------------
pxz_status pxz_image_alloc(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t channels, pxz_image** out) {
  return pxz_image_alloc_batch(ctx, w, h, channels, 1, out);
}

pxz_status pxz_image_alloc_batch(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t channels, uint32_t n_images, pxz_image** out) {
  if (!ctx || !out) return PXZ_E_ARG;
  *out = nullptr;
  if (w == 0 || h == 0 || n_images == 0) return fail(ctx, PXZ_E_ARG, "empty image");
  if ((uint64_t)h * n_images > 0xFFFFFFFFull) return fail(ctx, PXZ_E_UNSUPPORTED, "batch taller than 2^32 rows");
  if (channels != 3 && channels != 4) return fail(ctx, PXZ_E_ARG, "channels must be 3 or 4");
  cudaSetDevice(ctx->device);
  pxz_image* im = new (std::nothrow) pxz_image();
  if (!im) return fail(ctx, PXZ_E_OOM, "host allocation failed");
  im->ctx = ctx; im->w = w; im->h = h; im->c = channels; im->owned = true; im->nimg = n_images;
  im->pitch = (((size_t)w * channels) + 127) & ~(size_t)127;  // 128-byte rows: every tile row starts 16 B aligned for RGBA
  pxz_status st = dev_alloc(ctx, (void**)&im->d, im->pitch * h * n_images);
  if (st != PXZ_OK) { delete im; return st; }
  *out = im;
  return PXZ_OK;
}

pxz_status pxz_image_upload(pxz_ctx* ctx, const uint8_t* host, uint32_t w, uint32_t h, uint32_t channels, size_t host_pitch,
                            pxz_image** out) {
  return pxz_image_upload_batch(ctx, host, w, h, channels, host_pitch, 1, out);
}

pxz_status pxz_image_upload_batch(pxz_ctx* ctx, const uint8_t* host, uint32_t w, uint32_t h, uint32_t channels, size_t host_pitch,
                                  uint32_t n_images, pxz_image** out) {
  if (!ctx || !host || !out) return PXZ_E_ARG;
  if (host_pitch < (size_t)w * channels) return fail(ctx, PXZ_E_ARG, "host pitch smaller than a row");
  pxz_status st = pxz_image_alloc_batch(ctx, w, h, channels, n_images, out);
  if (st != PXZ_OK) return st;
  // the host images follow each other without a gap (image i at host + i * h * host_pitch): one 2-D copy
  cudaError_t e = cudaMemcpy2DAsync((*out)->d, (*out)->pitch, host, host_pitch, (size_t)w * channels, (size_t)h * n_images,
                                    cudaMemcpyHostToDevice, ctx->stream);
  if (e != cudaSuccess) {
    pxz_image_free(*out);
    *out = nullptr;
    return cuda_fail(ctx, e, "cudaMemcpy2DAsync");
  }
  return PXZ_OK;
}

pxz_status pxz_image_wrap(pxz_ctx* ctx, void* device_ptr, uint32_t w, uint32_t h, uint32_t channels, size_t pitch,
                          pxz_image** out) {
  return pxz_image_wrap_batch(ctx, device_ptr, w, h, channels, pitch, 1, out);
}

pxz_status pxz_image_wrap_batch(pxz_ctx* ctx, void* device_ptr, uint32_t w, uint32_t h, uint32_t channels, size_t pitch,
                                uint32_t n_images, pxz_image** out) {
  if (!ctx || !device_ptr || !out) return PXZ_E_ARG;
  if (w == 0 || h == 0 || n_images == 0 || (channels != 3 && channels != 4) || pitch < (size_t)w * channels ||
      (uint64_t)h * n_images > 0xFFFFFFFFull)
    return fail(ctx, PXZ_E_ARG, "bad image geometry");
  pxz_image* im = new (std::nothrow) pxz_image();
  if (!im) return fail(ctx, PXZ_E_OOM, "host allocation failed");
  im->ctx = ctx; im->d = (uint8_t*)device_ptr; im->pitch = pitch; im->w = w; im->h = h; im->c = channels; im->owned = false;
  im->nimg = n_images;
  *out = im;
  return PXZ_OK;
}

pxz_status pxz_image_info(const pxz_image* img, uint32_t* w, uint32_t* h, uint32_t* channels, size_t* pitch, void** device_ptr) {
  if (!img) return PXZ_E_ARG;
  if (w) *w = img->w;
  if (h) *h = img->h;
  if (channels) *channels = img->c;
  if (pitch) *pitch = img->pitch;
  if (device_ptr) *device_ptr = img->d;
  return PXZ_OK;
}

pxz_status pxz_image_download(pxz_ctx* ctx, const pxz_image* img, uint8_t* host, size_t host_pitch) {
  if (!ctx || !img || !host) return PXZ_E_ARG;
  if (host_pitch < (size_t)img->w * img->c) return fail(ctx, PXZ_E_ARG, "host pitch smaller than a row");
  PXZ_CUDA(ctx, cudaMemcpy2DAsync(host, host_pitch, img->d, img->pitch, (size_t)img->w * img->c, (size_t)img->h * img->nimg,
                                  cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

void pxz_image_free(pxz_image* img) {
  if (!img) return;
  if (img->owned) dev_free(img->ctx, img->d);
  delete img;
}

// ---- analysis -----------------------------------------------------------------------------------------
static pxz_status run_analysis(pxz_ctx* ctx, const pxz_image* img, const Geom& g, pxz_metric metric, bool exact_all,
                               const ValueMap* vm_for_band) {
  const uint32_t nblocks = g.cols * g.rows;
  pxz_status st = ensure_scratch(ctx, nblocks);
  if (st != PXZ_OK) return st;
  if (metric == PXZ_METRIC_OKLAB_MAD) {
    if (exact_all) {
      ProfScope prof(ctx, K_MAD_EXACT);
      PXZ_CUDA(ctx, launch_analyze_mad_exact(img->d, img->pitch, g, ctx->d_vx, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                             ctx->d_list, ctx->d_list + nblocks, ctx->stream, ctx->sm_count, &ctx->launches));
    } else {
      {
        ProfScope prof(ctx, K_MAD_FAST);
        PXZ_CUDA(ctx, launch_analyze_mad_fast(img->d, img->pitch, g, ctx->d_vx, ctx->d_opaque, ctx->d_list + nblocks, ctx->stream,
                                              ctx->sm_count, &ctx->launches));
      }
      if (vm_for_band) {
        // recompute, in reference order, the tiles whose level could differ from the CPU result
        ProfScope prof(ctx, K_MAD_EXACT);
        PXZ_CUDA(ctx, launch_analyze_mad_exact(img->d, img->pitch, g, ctx->d_vx, ctx->d_vx, ctx->d_opaque, vm_for_band, &ctx->thr,
                                               &ctx->band, ctx->d_minmax, ctx->d_list, ctx->d_list + nblocks, ctx->stream,
                                               ctx->sm_count, &ctx->launches));
      }
    }
  } else if (metric == PXZ_METRIC_SOBEL_DIR) {
    // operations.rs:220-221: `height - 2` / `width - 2` underflow -> the reference panics
    const uint32_t min_w = g.trail_w ? std::min(g.bw, g.trail_w) : std::min(g.bw, g.W);
    const uint32_t min_h = g.trail_h ? std::min(g.bh, g.trail_h) : std::min(g.bh, g.H);
    if (min_w < 2 || min_h < 2)
      return fail(ctx, PXZ_E_ARG, "directional metric needs every block to be at least 2x2 (the reference panics)");
    ProfScope prof(ctx, K_SOBEL);
    PXZ_CUDA(ctx, launch_analyze_sobel(img->d, img->pitch, g, ctx->d_vx, ctx->d_vy, ctx->stream, ctx->sm_count, &ctx->launches));
  } else {
    return fail(ctx, PXZ_E_ARG, "unknown metric");
  }
  return PXZ_OK;
}

pxz_status pxz_analyze(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint32_t flags,
                       float* host_values_x, float* host_values_y) {
  if (!ctx || !img || !host_values_x) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g, img->nimg);
  if (st != PXZ_OK) return st;
  st = run_analysis(ctx, img, g, metric, (flags & PXZ_FLAG_EXACT_VALUES) != 0, nullptr);
  if (st != PXZ_OK) return st;
  const size_t n = (size_t)g.cols * g.rows;
  PXZ_CUDA(ctx, cudaMemcpyAsync(host_values_x, ctx->d_vx, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (host_values_y) {
    const float* src = metric == PXZ_METRIC_SOBEL_DIR ? ctx->d_vy : ctx->d_vx;
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_values_y, src, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

// ---- encode -------------------------------------------------------------------------------------------
static pxz_status payload_new(pxz_ctx* ctx, const Geom& g, uint64_t capacity, PayloadOwner* out) {
  PayloadOwner p(new (std::nothrow) pxz_payload());
  if (!p) return fail(ctx, PXZ_E_OOM, "host allocation failed");
  p->ctx = ctx;
  p->g = g;
  const size_t nblocks = (size_t)g.cols * g.rows;
  // a cached set that is large enough (smallest fit)
  int best = -1;
  for (size_t i = 0; i < ctx->payload_cache.size(); ++i) {
    const PayloadBufs& b = ctx->payload_cache[i];
    if (b.nblocks >= nblocks && b.capacity >= capacity && (best < 0 || b.capacity < ctx->payload_cache[best].capacity)) best = (int)i;
  }
  if (best >= 0) {
    const PayloadBufs b = ctx->payload_cache[best];
    ctx->payload_cache.erase(ctx->payload_cache.begin() + best);
    p->d_descs = b.d_descs; p->d_tabidx = b.d_tabidx; p->d_pixels = b.d_pixels; p->d_total = b.d_total;
    p->nblocks_cap = b.nblocks; p->capacity = b.capacity;
    *out = std::move(p);
    return PXZ_OK;
  }
  p->capacity = capacity;
  p->nblocks_cap = nblocks;
  pxz_status st;
  if ((st = dev_alloc(ctx, (void**)&p->d_descs, nblocks * sizeof(pxz_block_desc))) != PXZ_OK ||
      (st = dev_alloc(ctx, (void**)&p->d_tabidx, (2 * nblocks + order_list_words(nblocks)) * 4)) != PXZ_OK ||  // table indices | work order lists | expand-side indices
      (st = dev_alloc(ctx, (void**)&p->d_pixels, capacity)) != PXZ_OK ||
      (st = dev_alloc(ctx, (void**)&p->d_total, 8)) != PXZ_OK)
    return st;  // payload_release frees a partial set: only complete sets enter the cache
  *out = std::move(p);
  return PXZ_OK;
}

// The one exchange of the path (PXZ_FLAG_NORMALISE_GLOBAL with a communicator): ncclMin over {min_x, -max_x, min_y, -max_y,
// ok}.  `ok` is 0 on a healthy rank and -1 on a rank that failed before it got here — such a rank still joins, with
// neutral values, so that its peers do not wait in the all-reduce forever; everybody then learns that a rank failed.
// `local_ok == false`: this rank contributes nothing (an error before the exchange, or a shard without rows).
static pxz_status exchange_minmax(pxz_ctx* ctx, bool local_ok, bool* peers_ok) {
  *peers_ok = true;
  if (!ctx->comm) return PXZ_OK;
  if (local_ok) {
    PXZ_CUDA(ctx, cudaMemsetAsync(ctx->d_minmax + 4, 0, sizeof(float), ctx->stream));
  } else {
    static const float neutral[5] = {INFINITY, INFINITY, INFINITY, INFINITY, -1.0f};
    PXZ_CUDA(ctx, cudaMemcpyAsync(ctx->d_minmax, neutral, sizeof(neutral), cudaMemcpyHostToDevice, ctx->stream));
  }
  std::string err;
  if (nccl_allreduce_min_f32(ctx->comm, ctx->d_minmax, 5, ctx->stream, &err) != 0) return fail(ctx, PXZ_E_NCCL, err);
  float flag = 0.f;
  PXZ_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_minmax + 4, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *peers_ok = !(flag < 0.f);
  return PXZ_OK;
}

pxz_status pxz_comm_join_empty(pxz_ctx* ctx) {
  if (!ctx) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (!ctx->comm) return fail(ctx, PXZ_E_ARG, "no communicator (pxz_comm_init)");
  // a rank whose shard has no rows: neutral values, but a healthy flag
  static const float neutral[5] = {INFINITY, INFINITY, INFINITY, INFINITY, 0.0f};
  PXZ_CUDA(ctx, cudaMemcpyAsync(ctx->d_minmax, neutral, sizeof(neutral), cudaMemcpyHostToDevice, ctx->stream));
  std::string err;
  if (nccl_allreduce_min_f32(ctx->comm, ctx->d_minmax, 5, ctx->stream, &err) != 0) return fail(ctx, PXZ_E_NCCL, err);
  float flag = 0.f;
  PXZ_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_minmax + 4, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (flag < 0.f) return fail(ctx, PXZ_E_NCCL, "another rank failed before the min/max exchange");
  return PXZ_OK;
}

// RGB images whose geometry suits the RGBA fast kernels run on them (kernels.cu "RGB images on the RGBA fast kernels")
static bool rgb_on_rgba(const pxz_ctx* ctx, uint32_t w, uint32_t c, uint32_t bw, uint32_t bh) {
  return c == 3 && ctx->resize_semantics == PXZ_RESIZE_IMAGE_RS && bw <= 64 && bh <= 64 && bw % 4 == 0 && w % 4 == 0;
}

// payload of the other channel count (3 <-> 4) with the same blocks, tables and work order
static pxz_status payload_rechannel(pxz_ctx* ctx, const pxz_payload* src, uint32_t dc, PayloadOwner* out) {
  Geom g = src->g;
  const uint32_t sc = g.C;
  g.C = dc;
  const uint32_t nblocks = g.cols * g.rows;
  // k_payload_convert writes each block at offset / sc * dc.  Uploaded payloads may hold blocks larger than their tiles, so
  // W * H * dc does not bound that; every block lies inside src->capacity (payload_from_descs checks it).
  const uint64_t cap = std::max<uint64_t>((uint64_t)g.W * g.H * dc * g.nimg, (src->capacity + sc - 1) / sc * dc);
  PayloadOwner p;
  pxz_status st = payload_new(ctx, g, cap, &p);
  if (st != PXZ_OK) return st;
  copy_layout(p.get(), src);
  if (src->bytes_known) { p->bytes = src->bytes / sc * dc; p->bytes_known = true; }
  cudaError_t e = launch_payload_convert(src->d_descs, src->d_pixels, src->d_tabidx, (uint32_t)src->nblocks_cap, src->d_total, p->d_descs,
                                         p->d_pixels, p->d_tabidx, (uint32_t)p->nblocks_cap, p->d_total, nblocks, (int)sc, (int)dc,
                                         ctx->stream, ctx->sm_count, &ctx->launches);
  if (e != cudaSuccess) return cuda_fail(ctx, e, "payload convert");
  *out = std::move(p);
  return PXZ_OK;
}

// An RGB image on the RGBA fast kernels: widen it to RGBA (alpha 255: its metric term is exactly +0 and the opaque resample
// path never touches it), run `encode` on the 4-channel image, narrow the payload back
extern "C++" {  // a template inside the extern "C" block
static pxz_status rgb_widened(pxz_ctx* ctx, const pxz_image* img, ImageOwner* wide) {
  pxz_status st = image_new(ctx, img->w, img->h, 4, img->nimg, wide);
  if (st != PXZ_OK) return st;
  cudaError_t e = launch_rgb_widen(img->d, img->pitch, (*wide)->d, (*wide)->pitch, img->w, img->h * img->nimg, 1, ctx->stream, ctx->sm_count,
                                   &ctx->launches);
  return e == cudaSuccess ? PXZ_OK : cuda_fail(ctx, e, "rgb widen");
}
template <class F>
static pxz_status encode_via_rgba(pxz_ctx* ctx, const pxz_image* img, F&& encode, pxz_payload** out) {
  ImageOwner wide;
  pxz_status st = rgb_widened(ctx, img, &wide);
  if (st != PXZ_OK) return st;
  pxz_payload* raw = nullptr;
  st = encode(wide.get(), &raw);
  wide.reset();  // stream-ordered: the kernels queued above keep it
  const PayloadOwner p4(raw);
  if (st != PXZ_OK) return st;
  PayloadOwner p3;
  st = payload_rechannel(ctx, p4.get(), 3, &p3);
  *out = p3.release();
  return st;
}
}  // extern "C++"

static ValueMap shrink_value_map(const pxz_ctx* ctx, pxz_metric metric, uint32_t flags, float factor) {
  ValueMap vm;
  vm.factor = factor;
  vm.mode = (metric == PXZ_METRIC_SOBEL_DIR) ? 2 : ((flags & PXZ_FLAG_AFTER_IDENTITY) ? 1 : 0);
  vm.normalise = (flags & PXZ_FLAG_NORMALISE_GLOBAL) ? 1 : 0;
  vm.extra_thr = NAN;
  if (ctx->strategy.on)
    for (int k = 1; k < kStrategyBuckets; ++k)
      if (ctx->strategy.down[k] != ctx->strategy.down[k - 1] || ctx->strategy.up[k] != ctx->strategy.up[k - 1])
        vm.bucket_edges |= 1ull << (k - 1);
  return vm;
}

// min / max of the values in ctx->d_vx (and d_vy) into ctx->d_minmax
static pxz_status run_minmax(pxz_ctx* ctx, pxz_metric metric, uint32_t nblocks) {
  return profiled(ctx, K_MINMAX, "minmax", [&] {
    return launch_minmax(ctx->d_vx, metric == PXZ_METRIC_SOBEL_DIR ? ctx->d_vy : nullptr, nblocks, ctx->d_minmax, ctx->stream, &ctx->launches);
  });
}

// Global normalisation on the fast Oklab path, first half: the exact extremes come from the few tiles that can hold them
// (their reference-order values patched into ctx->d_vx), then a second min / max over the patched values
static pxz_status run_exact_extremes(pxz_ctx* ctx, const pxz_image* img, const Geom& g, uint32_t nblocks) {
  const pxz_status st = profiled(ctx, K_MAD_EXACT, "extremes", [&] {
    return launch_analyze_mad_exact(img->d, img->pitch, g, ctx->d_vx, ctx->d_vx, ctx->d_opaque, nullptr, &ctx->thr, &ctx->band, ctx->d_minmax,
                                    ctx->d_list, ctx->d_list + nblocks, ctx->stream, ctx->sm_count, &ctx->launches);
  });
  return st != PXZ_OK ? st : run_minmax(ctx, PXZ_METRIC_OKLAB_MAD, nblocks);
}

// Guard band of the fast Oklab path for the factor of `vm`: the tiles listed from the fast values `vx_fast` get their
// reference-order value in `vx` (in place when vx == vx_fast, as pxz_shrink does)
static pxz_status run_guard_band(pxz_ctx* ctx, const pxz_image* img, const Geom& g, const ValueMap& vm, float* vx, const float* vx_fast) {
  const uint32_t nblocks = g.cols * g.rows;
  return profiled(ctx, K_MAD_EXACT, "guard band", [&] {
    const cudaError_t e = cudaMemsetAsync(ctx->d_list + nblocks, 0, sizeof(uint32_t), ctx->stream);  // the list counter
    return e != cudaSuccess ? e
                            : launch_analyze_mad_exact(img->d, img->pitch, g, vx, vx_fast, ctx->d_opaque, &vm, &ctx->thr, &ctx->band, ctx->d_minmax,
                                                       ctx->d_list, ctx->d_list + nblocks, ctx->stream, ctx->sm_count, &ctx->launches);
  });
}

// The analysis of pxz_shrink before the min / max exchange: the values into ctx->d_vx / d_vy, then with global normalisation
// their min / max and, on the fast Oklab path, the exact extremes.  band_vm (may be NULL): the value map whose guard band the
// fast Oklab path resolves in the same pass; with global normalisation the band waits for the exchanged range.
static pxz_status run_shrink_analysis(pxz_ctx* ctx, const pxz_image* img, const Geom& g, pxz_metric metric, uint32_t flags,
                                      const ValueMap* band_vm) {
  const bool normalise = (flags & PXZ_FLAG_NORMALISE_GLOBAL) != 0;
  const bool exact_all = (flags & PXZ_FLAG_EXACT_VALUES) != 0;
  const uint32_t nblocks = g.cols * g.rows;
  pxz_status st = run_analysis(ctx, img, g, metric, exact_all, normalise ? nullptr : band_vm);
  if (st != PXZ_OK || !normalise) return st;
  if ((st = run_minmax(ctx, metric, nblocks)) != PXZ_OK) return st;
  return metric == PXZ_METRIC_OKLAB_MAD && !exact_all ? run_exact_extremes(ctx, img, g, nblocks) : PXZ_OK;
}

// The part of pxz_shrink after the analysis: plan (value -> level -> dims -> offsets) from ctx->d_vx / d_vy, then the
// resample into a new payload
static pxz_status plan_and_resample(pxz_ctx* ctx, const pxz_image* img, const Geom& g, pxz_metric metric, const ValueMap& vm,
                                    pxz_filter filter_down, bool exact_all, pxz_payload** out) {
  PayloadOwner p;
  pxz_status st = payload_new(ctx, g, (uint64_t)g.W * g.H * g.C * g.nimg, &p);
  if (st != PXZ_OK) return st;
  p->spec = spec_for_geom(g);
  set_plan_bounds(p.get(), g, metric == PXZ_METRIC_OKLAB_MAD);
  StrategyLut lut = ctx->strategy;
  lut.stride = (uint32_t)p->spec->n_small.size();
  p->strategy = lut.on ? 1 : 0;
  st = profiled(ctx, K_PLAN, "plan", [&] {
    return launch_plan(ctx->d_vx, metric == PXZ_METRIC_SOBEL_DIR ? ctx->d_vy : nullptr, g, vm, ctx->d_minmax, ctx->thr, nullptr, p->d_descs,
                       p->d_tabidx, p->d_total, ctx->d_scan, p->d_order(), (uint32_t)p->nblocks_cap, ctx->stream, &ctx->launches, &lut, p->d_up());
  });
  if (st != PXZ_OK) return st;
  TabSet ts;
  if ((st = get_tabset(ctx, *p->spec, p->strategy ? -1 : (int)filter_down, 0, &ts)) != PXZ_OK) return st;
  // the fast Oklab-MAD pass also told which tiles are fully opaque: their alpha channel needs no arithmetic
  const uint8_t* opaque_flags = (metric == PXZ_METRIC_OKLAB_MAD && !exact_all) ? ctx->d_opaque : nullptr;
  if ((st = run_resample(ctx, 0, img->d, img->pitch, p.get(), ts, g.bw * g.bh, std::max(g.bw, g.bh), p->max_tmp_down, opaque_flags)) != PXZ_OK)
    return st;
  *out = p.release();
  return PXZ_OK;
}

pxz_status pxz_shrink(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                      pxz_filter filter_down, uint32_t flags, pxz_payload** out) {
  if (!ctx || !img || !out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  if (rgb_on_rgba(ctx, img->w, img->c, bw, bh))
    return encode_via_rgba(
        ctx, img, [&](const pxz_image* wide, pxz_payload** p4) { return pxz_shrink(ctx, wide, bw, bh, metric, factor, filter_down, flags, p4); },
        out);
  const bool normalise = (flags & PXZ_FLAG_NORMALISE_GLOBAL) != 0;
  // Every rank of a communicator must reach the min/max exchange, whatever happens to it before: a rank-local failure
  // (an unknown filter, a trailing block the Sobel metric cannot take, no memory) joins with neutral values and an
  // error flag instead of leaving its peers in the collective.
  auto bail = [&](pxz_status why) -> pxz_status {
    if (normalise && ctx->comm) {
      const std::string msg = ctx->err;
      bool peers_ok = true;
      exchange_minmax(ctx, false, &peers_ok);
      ctx->err = msg;
    }
    return why;
  };
  if (!known_filter(filter_down)) return bail(fail(ctx, PXZ_E_ARG, "unknown filter"));
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g, img->nimg);
  if (st != PXZ_OK) return bail(st);
  if (normalise && img->nimg > 1) return bail(fail(ctx, PXZ_E_UNSUPPORTED, "global normalisation is per image: not available on a batch"));

  const ValueMap vm = shrink_value_map(ctx, metric, flags, factor);

  // with global normalisation every value depends on the exact min and max, so the Oklab path
  // runs in reference order for all blocks (DESIGN.md)
  const bool exact_all = (flags & PXZ_FLAG_EXACT_VALUES) != 0;
  // Global normalisation of the Oklab values on the fast path: the exact extremes come from the few tiles that can hold
  // them, and the guard band (scaled by 1 / range) then decides as in the default mode which tiles need their
  // reference-order value; with PXZ_FLAG_EXACT_VALUES every tile is computed in reference order as before.
  const bool fast_norm = normalise && metric == PXZ_METRIC_OKLAB_MAD && !exact_all;
  st = run_shrink_analysis(ctx, img, g, metric, flags, &vm);
  if (st != PXZ_OK) return bail(st);

  if (normalise) {
    bool peers_ok = true;
    st = exchange_minmax(ctx, true, &peers_ok);
    if (st != PXZ_OK) return st;
    if (!peers_ok) return fail(ctx, PXZ_E_NCCL, "another rank failed before the min/max exchange");
    if (fast_norm && (st = run_guard_band(ctx, img, g, vm, ctx->d_vx, ctx->d_vx)) != PXZ_OK) return st;
  }
  return plan_and_resample(ctx, img, g, metric, vm, filter_down, exact_all, out);
}

// Rate control (pxz_shrink_to_size).  bpp: bytes per pixel the budget counts (3 for an RGB image on the RGBA kernels).
static pxz_status shrink_to_size(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint64_t max_bytes,
                                 pxz_filter filter_down, uint32_t flags, uint32_t bpp, float* factor_out, pxz_payload** out) {
  if (rgb_on_rgba(ctx, img->w, img->c, bw, bh))
    return encode_via_rgba(
        ctx, img,
        [&](const pxz_image* wide, pxz_payload** p4) {
          return shrink_to_size(ctx, wide, bw, bh, metric, max_bytes, filter_down, flags, 3, factor_out, p4);
        },
        out);
  if (!known_filter(filter_down)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (metric != PXZ_METRIC_OKLAB_MAD && metric != PXZ_METRIC_SOBEL_DIR) return fail(ctx, PXZ_E_ARG, "unknown metric");
  if (flags & PXZ_FLAG_AFTER_IDENTITY) return fail(ctx, PXZ_E_ARG, "PXZ_FLAG_AFTER_IDENTITY ignores the factor: no size to choose");
  if (img->nimg > 1) return fail(ctx, PXZ_E_UNSUPPORTED, "a size budget is per image: not available on a batch");
  const bool normalise = (flags & PXZ_FLAG_NORMALISE_GLOBAL) != 0;
  if (normalise && ctx->comm)
    return fail(ctx, PXZ_E_UNSUPPORTED, "a size budget with global normalisation over a communicator is not available");
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g, img->nimg);
  if (st != PXZ_OK) return st;
  const uint32_t nblocks = g.cols * g.rows;
  ValueMap vm = shrink_value_map(ctx, metric, flags, 1.0f);
  const bool exact_all = (flags & PXZ_FLAG_EXACT_VALUES) != 0;
  // fast Oklab values: sizes found on them are checked against the guard band before they are trusted
  const bool fast = metric == PXZ_METRIC_OKLAB_MAD && !exact_all;

  // analysis as pxz_shrink runs it, without the guard band (it depends on the factor)
  if ((st = run_shrink_analysis(ctx, img, g, metric, flags, nullptr)) != PXZ_OK) return st;

  // scratch: the sizes of one round, and on the fast path the copy of the values the search runs on
  DevBlocks bufs(ctx);
  uint8_t* scratch = nullptr;
  const size_t sizes_bytes = (size_t)kMaxSizeCandidates * sizeof(uint64_t);
  if ((st = bufs.alloc(&scratch, sizes_bytes + (fast ? (size_t)nblocks * 4 : 0))) != PXZ_OK) return st;
  uint64_t* d_sizes = reinterpret_cast<uint64_t*>(scratch);
  float* d_search = fast ? reinterpret_cast<float*>(scratch + sizes_bytes) : ctx->d_vx;
  const float* d_search_y = metric == PXZ_METRIC_SOBEL_DIR ? ctx->d_vy : nullptr;
  if (fast) PXZ_CUDA(ctx, cudaMemcpyAsync(d_search, ctx->d_vx, (size_t)nblocks * 4, cudaMemcpyDeviceToDevice, ctx->stream));

  constexpr uint32_t kMaxPattern = 0x7F7FFFFFu;  // FLT_MAX; patterns 1 .. kMaxPattern are the finite factors > 0
  auto factor_of = [](uint32_t bits) {
    float f;
    memcpy(&f, &bits, 4);
    return f;
  };
  uint64_t size_at_min = 0;  // payload at the smallest positive factor (pattern 1), once evaluated
  std::vector<uint64_t> sizes(kMaxSizeCandidates);
  auto evaluate = [&](const std::vector<uint32_t>& pats) -> pxz_status {
    SizeCandidates cand;
    cand.n = (uint32_t)pats.size();
    for (size_t i = 0; i < pats.size(); ++i) cand.k[i] = factor_of(pats[i]);
    {
      ProfScope prof(ctx, K_SIZE_CURVE);
      PXZ_CUDA(ctx, launch_size_curve(d_search, d_search_y, g, vm, ctx->d_minmax, ctx->thr, bpp, cand, d_sizes, ctx->stream, ctx->sm_count,
                                      &ctx->launches));
    }
    PXZ_CUDA(ctx, cudaMemcpyAsync(sizes.data(), d_sizes, pats.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < pats.size(); ++i)
      if (pats[i] == 1u) size_at_min = sizes[i];
    return PXZ_OK;
  };
  // The size is monotone in the factor (DESIGN.md §3), so the bit patterns that fit are a prefix of [1, kMaxPattern].
  // lo fits (0: none known to), hi does not (kMaxPattern + 1: none known not to); each round evaluates up to 256 evenly
  // spaced patterns strictly between them.
  uint32_t k_bits = 0;
  auto search = [&]() -> pxz_status {
    uint32_t lo = 0, hi = kMaxPattern + 1;
    while (hi - lo > 1) {
      const uint32_t inner = hi - lo - 1;
      const uint32_t n = std::min<uint32_t>(inner, kMaxSizeCandidates);
      std::vector<uint32_t> pats(n);
      for (uint32_t i = 0; i < n; ++i) pats[i] = lo + 1 + (n > 1 ? (uint32_t)((uint64_t)i * (inner - 1) / (n - 1)) : 0u);
      if ((st = evaluate(pats)) != PXZ_OK) return st;
      uint32_t new_lo = lo, new_hi = hi;
      for (uint32_t i = 0; i < n; ++i) {
        if (sizes[i] <= max_bytes) new_lo = pats[i];
        else { new_hi = pats[i]; break; }
      }
      lo = new_lo;
      hi = new_hi;
    }
    k_bits = lo;
    return PXZ_OK;
  };
  for (;;) {
    if ((st = search()) != PXZ_OK) return st;
    if (!fast) break;
    // The search ran on fast values.  Recompute, in reference order, the guard band of k and of the next factor up (band
    // list from the untouched fast values, exact values into the search copy): both sizes are then exact.  When they do not
    // bracket the budget, search again on the corrected copy — each failure replaced at least one value by its exact one.
    std::vector<uint32_t> pats;
    if (k_bits >= 1u) pats.push_back(k_bits);
    if (k_bits < kMaxPattern) pats.push_back(k_bits + 1);
    for (uint32_t bits : pats) {
      ValueMap v = vm;
      v.factor = factor_of(bits);
      if ((st = run_guard_band(ctx, img, g, v, d_search, ctx->d_vx)) != PXZ_OK) return st;
    }
    if ((st = evaluate(pats)) != PXZ_OK) return st;
    const bool fits = k_bits < 1u || sizes[0] <= max_bytes;
    const bool next_over = k_bits >= kMaxPattern || sizes[pats.size() - 1] > max_bytes;
    if (fits && next_over) break;
  }
  if (k_bits == 0)
    return fail(ctx, PXZ_E_ARG, "max_bytes " + std::to_string(max_bytes) + " is below the payload at the smallest positive factor (" +
                                    std::to_string(size_at_min) + " bytes)");
  const float k = factor_of(k_bits);
  // encode at k exactly as pxz_shrink does, from the fast values
  vm.factor = k;
  if (fast && (st = run_guard_band(ctx, img, g, vm, ctx->d_vx, ctx->d_vx)) != PXZ_OK) return st;
  st = plan_and_resample(ctx, img, g, metric, vm, filter_down, exact_all, out);
  if (st == PXZ_OK) *factor_out = k;
  return st;
}

pxz_status pxz_shrink_to_size(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint64_t max_bytes,
                              pxz_filter filter_down, uint32_t flags, float* factor_out, pxz_payload** out) {
  if (!ctx || !img || !out || !factor_out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  return shrink_to_size(ctx, img, bw, bh, metric, max_bytes, filter_down, flags, img->c, factor_out, out);
}

// ---- decode error and strategy fit (extension) -------------------------------------------------------------------
// per-block error of a against b on the grid g into d_sse (and d_max, if given): both cleared first
static pxz_status run_block_error(pxz_ctx* ctx, const pxz_image* a, const pxz_image* b, const Geom& g, uint64_t* d_sse, uint32_t* d_max) {
  const size_t nblocks = (size_t)g.cols * g.rows;
  PXZ_CUDA(ctx, cudaMemsetAsync(d_sse, 0, nblocks * sizeof(uint64_t), ctx->stream));
  if (d_max) PXZ_CUDA(ctx, cudaMemsetAsync(d_max, 0, nblocks * sizeof(uint32_t), ctx->stream));
  ProfScope prof(ctx, K_BLOCK_ERROR);
  PXZ_CUDA(ctx, launch_block_error(a->d, a->pitch, b->d, b->pitch, g, d_sse, d_max, ctx->stream, ctx->sm_count, &ctx->launches));
  return PXZ_OK;
}

pxz_status pxz_image_error(pxz_ctx* ctx, const pxz_image* a, const pxz_image* b, uint32_t bw, uint32_t bh, uint64_t* host_block_sse,
                           uint8_t* host_block_max, uint64_t* host_total_sse) {
  if (!ctx || !a || !b) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (a->nimg != 1 || b->nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "the error of a batch image is not supported");
  if (a->w != b->w || a->h != b->h || a->c != b->c) return fail(ctx, PXZ_E_ARG, "image geometry mismatch");
  Geom g;
  pxz_status st = make_geom(ctx, a->w, a->h, a->c, bw, bh, &g);
  if (st != PXZ_OK) return st;
  const size_t nblocks = (size_t)g.cols * g.rows;
  DevBlocks bufs(ctx);
  uint8_t* buf = nullptr;
  if ((st = bufs.alloc(&buf, nblocks * (sizeof(uint64_t) + sizeof(uint32_t)))) != PXZ_OK) return st;
  uint64_t* d_sse = reinterpret_cast<uint64_t*>(buf);
  uint32_t* d_max = reinterpret_cast<uint32_t*>(buf + nblocks * sizeof(uint64_t));
  if ((st = run_block_error(ctx, a, b, g, d_sse, host_block_max ? d_max : nullptr)) != PXZ_OK) return st;
  // the total is summed on the host from the block sums (cols * rows words; the grid is what the caller asked for)
  std::vector<uint64_t> sse(nblocks);
  std::vector<uint32_t> mx(host_block_max ? nblocks : 0);
  PXZ_CUDA(ctx, cudaMemcpyAsync(sse.data(), d_sse, nblocks * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (host_block_max) PXZ_CUDA(ctx, cudaMemcpyAsync(mx.data(), d_max, nblocks * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  uint64_t total = 0;
  for (size_t i = 0; i < nblocks; ++i) total += sse[i];
  if (host_block_sse) memcpy(host_block_sse, sse.data(), nblocks * sizeof(uint64_t));
  if (host_block_max)
    for (size_t i = 0; i < nblocks; ++i) host_block_max[i] = (uint8_t)mx[i];
  if (host_total_sse) *host_total_sse = total;
  return PXZ_OK;
}

// pxz_strategy_measure after the checks, with the context's strategy cleared: one analysis, then for each down filter the plan
// + resample of pxz_shrink and for each up filter an expand into one scratch image and the error / bucket passes
static pxz_status strategy_measure(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                                   uint32_t flags, uint64_t* host_sse, uint32_t* host_blocks) {
  // An RGB image that pxz_shrink runs on the RGBA kernels is measured as its RGBA widening: the payloads are then the 4-channel
  // payloads pxz_shrink narrows, and the decodes those pxz_expand_to_image narrows.  The alpha channel is 255 in the source and
  // in every decode, so it adds 0 to every sum and the report equals that of the 3-channel image.
  if (rgb_on_rgba(ctx, img->w, img->c, bw, bh)) {
    ImageOwner wide;
    pxz_status st = rgb_widened(ctx, img, &wide);
    if (st != PXZ_OK) return st;
    return strategy_measure(ctx, wide.get(), bw, bh, metric, factor, flags, host_sse, host_blocks);
  }
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g);
  if (st != PXZ_OK) return st;
  const uint32_t nblocks = g.cols * g.rows;
  // Every bucket edge is resolved in the guard band, so the bucket of every block is the one its reference-order value gives
  // (DESIGN.md §3); the dims are those of pxz_shrink in every mode
  ValueMap vm = shrink_value_map(ctx, metric, flags, factor);
  vm.bucket_edges = ~0ull;
  const bool exact_all = (flags & PXZ_FLAG_EXACT_VALUES) != 0;
  const bool fast_norm = (flags & PXZ_FLAG_NORMALISE_GLOBAL) && metric == PXZ_METRIC_OKLAB_MAD && !exact_all;
  if ((st = run_shrink_analysis(ctx, img, g, metric, flags, &vm)) != PXZ_OK) return st;
  if (fast_norm && (st = run_guard_band(ctx, img, g, vm, ctx->d_vx, ctx->d_vx)) != PXZ_OK) return st;
  // device scratch: the report (65 x 25 sums, 65 counts), the block errors of one pair
  const size_t report_sse = (size_t)kStrategyBuckets * kFilterPairs * sizeof(uint64_t);
  const size_t report_bytes = report_sse + kStrategyBuckets * sizeof(uint32_t);
  const size_t block_sse_off = (report_bytes + 7) & ~(size_t)7;
  DevBlocks bufs(ctx);
  uint8_t* buf = nullptr;
  if ((st = bufs.alloc(&buf, block_sse_off + (size_t)nblocks * sizeof(uint64_t))) != PXZ_OK) return st;
  uint64_t* d_sse = reinterpret_cast<uint64_t*>(buf);
  uint32_t* d_blocks = reinterpret_cast<uint32_t*>(buf + report_sse);
  uint64_t* d_block_sse = reinterpret_cast<uint64_t*>(buf + block_sse_off);
  PXZ_CUDA(ctx, cudaMemsetAsync(buf, 0, report_bytes, ctx->stream));
  ImageOwner dec;
  if ((st = image_new(ctx, img->w, img->h, img->c, 1, &dec)) != PXZ_OK) return st;
  // down outer, up inner: one payload and one decode alive at a time.  The dims do not depend on the filter, so the five
  // payloads have the same descriptors and the bucket of a block is the same in all 25 passes.
  for (uint32_t down = 0; down < 5; ++down) {
    pxz_payload* raw = nullptr;
    if ((st = plan_and_resample(ctx, img, g, metric, vm, (pxz_filter)down, exact_all, &raw)) != PXZ_OK) return st;
    const PayloadOwner p(raw);
    for (uint32_t up = 0; up < 5; ++up) {
      const uint32_t pair = down * 5 + up;
      if ((st = pxz_expand_to_image(ctx, p.get(), (pxz_filter)up, dec.get())) != PXZ_OK) return st;
      if ((st = run_block_error(ctx, img, dec.get(), g, d_block_sse, nullptr)) != PXZ_OK) return st;
      st = profiled(ctx, K_BUCKET_SUM, "bucket sum", [&] {
        return launch_bucket_sum(p->d_descs, d_block_sse, nblocks, pair, pair == 0, d_sse, d_blocks, ctx->stream, ctx->sm_count, &ctx->launches);
      });
      if (st != PXZ_OK) return st;
    }
  }
  PXZ_CUDA(ctx, cudaMemcpyAsync(host_sse, d_sse, report_sse, cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaMemcpyAsync(host_blocks, d_blocks, kStrategyBuckets * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

pxz_status pxz_strategy_measure(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                                uint32_t flags, uint64_t* host_sse, uint32_t* host_blocks) {
  if (!ctx || !img || !host_sse || !host_blocks) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (img->nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "a strategy measure is per image: not available on a batch");
  if ((flags & PXZ_FLAG_NORMALISE_GLOBAL) && ctx->comm)
    return fail(ctx, PXZ_E_UNSUPPORTED, "a strategy measure with global normalisation over a communicator is not available");
  // the installed strategy would pick one pair per block: cleared for the call, restored on every return path
  struct StrategyOff {
    pxz_ctx* c;
    StrategyLut saved;
    explicit StrategyOff(pxz_ctx* cc) : c(cc), saved(cc->strategy) { c->strategy.on = 0; }
    ~StrategyOff() { c->strategy = saved; }
  } off(ctx);
  return strategy_measure(ctx, img, bw, bh, metric, factor, flags, host_sse, host_blocks);
}

// ---- rate-distortion curve (extension) ---------------------------------------------------------------------------
// What pxz_rd_curve and pxz_shrink_to_error refuse: pxz_shrink_to_size's refusals, plus an installed strategy (its filter pair
// follows the stored value, which moves with the factor) and an unknown up filter
static pxz_status rd_refusal(pxz_ctx* ctx, const pxz_image* img, pxz_metric metric, pxz_filter filter_down, pxz_filter filter_up, uint32_t flags) {
  if (!known_filter(filter_down) || !known_filter(filter_up)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (metric != PXZ_METRIC_OKLAB_MAD && metric != PXZ_METRIC_SOBEL_DIR) return fail(ctx, PXZ_E_ARG, "unknown metric");
  if (flags & PXZ_FLAG_AFTER_IDENTITY) return fail(ctx, PXZ_E_ARG, "PXZ_FLAG_AFTER_IDENTITY ignores the factor: no curve over it");
  if (img->nimg > 1) return fail(ctx, PXZ_E_UNSUPPORTED, "a rate-distortion curve is per image: not available on a batch");
  if ((flags & PXZ_FLAG_NORMALISE_GLOBAL) && ctx->comm)
    return fail(ctx, PXZ_E_UNSUPPORTED, "a rate-distortion curve with global normalisation over a communicator is not available");
  if (ctx->strategy.on)
    return fail(ctx, PXZ_E_UNSUPPORTED, "a rate-distortion curve with a strategy installed is not available (the filter pair moves with the factor)");
  return PXZ_OK;
}

// What one curve computation returns to the host besides the points
struct RdSummary {
  uint32_t n = 0;                  // curve points
  uint32_t first = 0xFFFFFFFFu;    // first point with sse <= max_sse (0xFFFFFFFF: none)
  uint32_t first_bits = 0;         // its factor's bit pattern
  uint64_t first_sse = 0;
  uint64_t least_sse = 0;          // least sse of any point
};

static uint32_t ceil_log2(uint32_t n) { return n <= 1 ? 0u : 32u - (uint32_t)__builtin_clz(n - 1); }

// The error table of the rate-distortion curves: per level pair (lx, ly) the plan + resample of pxz_shrink with every block
// forced to it — values 2^-lx / 2^-ly under the directional map at factor 1, no normalisation — then the decode with filter_up
// and its per-block error into table + pass * nblocks, pass = lx * ps.stride_x + ly * ps.stride_y.  diagonal: the pairs (l, l)
// for l <= lx_max, else every pair up to (lx_max, ly_max).  Overwrites ctx->d_vx / d_vy.
static pxz_status rd_error_table(pxz_ctx* ctx, const pxz_image* img, const Geom& g, pxz_filter filter_down, pxz_filter filter_up, bool diagonal,
                                 uint32_t lx_max, uint32_t ly_max, const RdPasses& ps, uint64_t* table) {
  const size_t nblocks = (size_t)g.cols * g.rows;
  ImageOwner dec;
  pxz_status st = image_new(ctx, img->w, img->h, img->c, 1, &dec);
  if (st != PXZ_OK) return st;
  const ValueMap forced = shrink_value_map(ctx, PXZ_METRIC_SOBEL_DIR, 0, 1.0f);
  for (uint32_t lx = 0; lx <= lx_max; ++lx) {
    for (uint32_t ly = diagonal ? lx : 0; ly <= (diagonal ? lx : ly_max); ++ly) {
      const float fx = ldexpf(1.0f, -(int)lx), fy = ldexpf(1.0f, -(int)ly);
      uint32_t w = 0, h = 0;  // level_k(2^-l) = l: the plan sees exactly these levels
      pxz_reduce_dims(fx, fy, g.bw, g.bh, &w, &h, nullptr);
      if (w != std::max(1u, ceil_div_u32(g.bw, 1u << lx)) || h != std::max(1u, ceil_div_u32(g.bh, 1u << ly)))
        return fail(ctx, PXZ_E_CUDA, "level table does not map 2^-l to level l");
      st = profiled(ctx, K_RD_LEVELS, "rd levels", [&] {
        return launch_rd_levels(ctx->d_vx, ctx->d_vy, (uint32_t)nblocks, fx, fy, ctx->stream, ctx->sm_count, &ctx->launches);
      });
      if (st != PXZ_OK) return st;
      pxz_payload* raw = nullptr;
      if ((st = plan_and_resample(ctx, img, g, PXZ_METRIC_SOBEL_DIR, forced, filter_down, true, &raw)) != PXZ_OK) return st;
      const PayloadOwner p(raw);
      if ((st = pxz_expand_to_image(ctx, p.get(), filter_up, dec.get())) != PXZ_OK) return st;
      const uint32_t pass = lx * ps.stride_x + ly * ps.stride_y;
      if ((st = run_block_error(ctx, img, dec.get(), g, table + (size_t)pass * nblocks, nullptr)) != PXZ_OK) return st;
    }
  }
  return PXZ_OK;
}

// The curve of pxz_rd_curve after the checks (DESIGN.md §3).  bpp: bytes per pixel counted (3 for an RGB image on the RGBA
// kernels).  The points are copied to the host arrays when cap >= n.
static pxz_status rd_curve(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, pxz_filter filter_down,
                           pxz_filter filter_up, uint32_t flags, uint32_t bpp, uint64_t max_sse, float* host_factor, uint64_t* host_bytes,
                           uint64_t* host_sse, size_t cap, RdSummary* sum) {
  // An RGB image that pxz_shrink runs on the RGBA kernels is measured as its RGBA widening, as in strategy_measure: alpha is 255
  // in the source and in every decode and adds 0
  if (rgb_on_rgba(ctx, img->w, img->c, bw, bh)) {
    ImageOwner wide;
    pxz_status st = rgb_widened(ctx, img, &wide);
    if (st != PXZ_OK) return st;
    return rd_curve(ctx, wide.get(), bw, bh, metric, filter_down, filter_up, flags, 3, max_sse, host_factor, host_bytes, host_sse, cap, sum);
  }
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g);
  if (st != PXZ_OK) return st;
  const size_t nblocks = (size_t)g.cols * g.rows;
  const bool sobel = metric == PXZ_METRIC_SOBEL_DIR;
  // Error passes: Oklab-MAD has one level for both axes (the diagonal), Sobel every (lx, ly) pair.  A level above Lx (Ly) gives
  // the dims of Lx (Ly), so those passes cover every level a block can reach.
  const uint32_t lx_max = ceil_log2(bw), ly_max = ceil_log2(bh), l_max = std::max(lx_max, ly_max);
  const RdPasses ps = sobel ? RdPasses{lx_max, ly_max, ly_max + 1, 1} : RdPasses{l_max, l_max, 1, 0};
  const uint32_t npass = sobel ? (lx_max + 1) * (ly_max + 1) : l_max + 1;
  const uint32_t maxev = sobel ? lx_max + ly_max : l_max;  // dims changes per block
  const uint64_t nev64 = (uint64_t)nblocks * maxev;
  if (nev64 > 0x7FFFFFFFull) return fail(ctx, PXZ_E_UNSUPPORTED, "more than 2^31 curve events (blocks x levels)");
  const uint32_t nev = (uint32_t)nev64;

  // 1. reference-order values (their dims are pxz_shrink's in every mode), the min / max as pxz_shrink takes it, and a copy
  if ((st = run_shrink_analysis(ctx, img, g, metric, flags | PXZ_FLAG_EXACT_VALUES, nullptr)) != PXZ_OK) return st;
  DevBlocks bufs(ctx);
  float* vals = nullptr;
  uint64_t* table = nullptr;  // [npass][nblocks] block errors
  uint8_t* ev = nullptr;      // events: keys | ids | dbytes | dsse | base[2] | points: key | bytes | sse | RdOut
  void* scratch = nullptr;
  const size_t scratch_bytes = rd_curve_scratch_bytes(nev);
  const size_t npt = (size_t)nev + 1;
  const size_t ev_bytes = (size_t)nev * 24 + 16 + npt * 20 + sizeof(RdOut) + 64;
  if ((st = bufs.alloc(&vals, nblocks * 4 * (sobel ? 2 : 1))) != PXZ_OK || (st = bufs.alloc(&table, (size_t)npass * nblocks * 8)) != PXZ_OK ||
      (st = bufs.alloc(&ev, ev_bytes)) != PXZ_OK || (st = bufs.alloc(&scratch, scratch_bytes)) != PXZ_OK)
    return st;
  // 8-byte words first
  uint64_t* dbytes = reinterpret_cast<uint64_t*>(ev);
  uint64_t* dsse = dbytes + nev;
  uint64_t* base = dsse + nev;
  uint64_t* pt_bytes = base + 2;
  uint64_t* pt_sse = pt_bytes + npt;
  RdOut* d_out = reinterpret_cast<RdOut*>(pt_sse + npt);
  uint32_t* keys = reinterpret_cast<uint32_t*>(d_out + 1);
  uint32_t* ids = keys + nev;
  uint32_t* pt_key = ids + nev;
  PXZ_CUDA(ctx, cudaMemcpyAsync(vals, ctx->d_vx, nblocks * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  if (sobel) PXZ_CUDA(ctx, cudaMemcpyAsync(vals + nblocks, ctx->d_vy, nblocks * 4, cudaMemcpyDeviceToDevice, ctx->stream));

  // 2. error table
  if ((st = rd_error_table(ctx, img, g, filter_down, filter_up, !sobel, sobel ? lx_max : l_max, sobel ? ly_max : l_max, ps, table)) != PXZ_OK)
    return st;

  // 3. events of every block, 4. the curve
  const ValueMap vm = shrink_value_map(ctx, metric, flags & PXZ_FLAG_NORMALISE_GLOBAL, 1.0f);
  PXZ_CUDA(ctx, cudaMemsetAsync(base, 0, 2 * sizeof(uint64_t), ctx->stream));
  st = profiled(ctx, K_RD_EVENTS, "rd events", [&] {
    return launch_rd_events(vals, sobel ? vals + nblocks : nullptr, g, vm, ctx->d_minmax, ctx->thr, bpp, table, ps, maxev, keys, ids, dbytes, dsse,
                            base, ctx->stream, &ctx->launches);
  });
  if (st != PXZ_OK) return st;
  st = profiled(ctx, K_RD_CURVE, "rd curve", [&] {
    return launch_rd_curve(keys, ids, dbytes, dsse, nev, base, max_sse, scratch, scratch_bytes, pt_key, pt_bytes, pt_sse, d_out, ctx->stream,
                           ctx->sm_count, &ctx->launches);
  });
  if (st != PXZ_OK) return st;

  // 5. to the host: the summary, the first point within max_sse, and the points when they fit
  RdOut o;
  PXZ_CUDA(ctx, cudaMemcpyAsync(&o, d_out, sizeof(o), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  sum->n = o.count;
  sum->first = o.first_within;
  sum->least_sse = o.least_sse;
  if (o.first_within < o.count) {
    PXZ_CUDA(ctx, cudaMemcpyAsync(&sum->first_bits, pt_key + o.first_within, 4, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaMemcpyAsync(&sum->first_sse, pt_sse + o.first_within, 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (cap >= o.count && host_factor && host_bytes && host_sse) {
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_factor, pt_key, (size_t)o.count * 4, cudaMemcpyDeviceToHost, ctx->stream));  // f32 bits
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_bytes, pt_bytes, (size_t)o.count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_sse, pt_sse, (size_t)o.count * 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

pxz_status pxz_rd_curve(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, pxz_filter filter_down,
                        pxz_filter filter_up, uint32_t flags, float* host_factor, uint64_t* host_bytes, uint64_t* host_sse, size_t cap,
                        size_t* n_out) {
  if (n_out) *n_out = 0;
  if (!ctx || !img || !n_out || (cap > 0 && (!host_factor || !host_bytes || !host_sse))) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  pxz_status st = rd_refusal(ctx, img, metric, filter_down, filter_up, flags);
  if (st != PXZ_OK) return st;
  RdSummary sum;
  st = rd_curve(ctx, img, bw, bh, metric, filter_down, filter_up, flags, img->c, 0, host_factor, host_bytes, host_sse, cap, &sum);
  if (st != PXZ_OK) return st;
  *n_out = sum.n;
  if (cap < sum.n) return fail(ctx, PXZ_E_ARG, "cap " + std::to_string(cap) + " is below the curve's " + std::to_string(sum.n) + " points");
  return PXZ_OK;
}

pxz_status pxz_shrink_to_error(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_metric metric, uint64_t max_sse,
                               pxz_filter filter_down, pxz_filter filter_up, uint32_t flags, float* factor_out, uint64_t* sse_out,
                               pxz_payload** out) {
  if (!ctx || !img || !out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  pxz_status st = rd_refusal(ctx, img, metric, filter_down, filter_up, flags);
  if (st != PXZ_OK) return st;
  RdSummary sum;
  st = rd_curve(ctx, img, bw, bh, metric, filter_down, filter_up, flags, img->c, max_sse, nullptr, nullptr, nullptr, 0, &sum);
  if (st != PXZ_OK) return st;
  if (sum.first >= sum.n)
    return fail(ctx, PXZ_E_ARG, "max_sse " + std::to_string(max_sse) + " is below the least squared error any factor reaches (" +
                                    std::to_string(sum.least_sse) + ")");
  float k;
  memcpy(&k, &sum.first_bits, 4);
  // the curve's point is the payload of pxz_shrink(k): encode it exactly so
  if ((st = pxz_shrink(ctx, img, bw, bh, metric, k, filter_down, flags, out)) != PXZ_OK) return st;
  if (factor_out) *factor_out = k;
  if (sse_out) *sse_out = sum.first_sse;
  return PXZ_OK;
}

// ---- rate-distortion optimised encode (extension) ----------------------------------------------------------------
// No metric, flags or factor: every block takes the dims of any level pair (DESIGN.md §3 "Per-block sizes")
static pxz_status rdo_refusal(pxz_ctx* ctx, const pxz_image* img, pxz_filter filter_down, pxz_filter filter_up) {
  if (!known_filter(filter_down) || !known_filter(filter_up)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (img->nimg > 1) return fail(ctx, PXZ_E_UNSUPPORTED, "an optimised encode is per image: not available on a batch");
  if (ctx->strategy.on)
    return fail(ctx, PXZ_E_UNSUPPORTED, "an optimised encode with a strategy installed is not available (its filter pair follows the stored value)");
  return PXZ_OK;
}

// Most events a block can have: its distinct byte counts over every level pair, less one, over the (up to four) tile shapes
static uint32_t rdo_max_events(const Geom& g) {
  const uint32_t lx_max = ceil_log2(g.bw), ly_max = ceil_log2(g.bh);
  uint32_t most = 0;
  for (uint32_t tw : {g.bw, g.trail_w ? g.trail_w : g.bw}) {
    for (uint32_t th : {g.bh, g.trail_h ? g.trail_h : g.bh}) {
      std::vector<uint64_t> sizes;
      for (uint32_t lx = 0; lx <= lx_max; ++lx)
        for (uint32_t ly = 0; ly <= ly_max; ++ly)
          sizes.push_back((uint64_t)std::max(1u, ceil_div_u32(tw, 1u << lx)) * std::max(1u, ceil_div_u32(th, 1u << ly)));
      std::sort(sizes.begin(), sizes.end());
      most = std::max(most, (uint32_t)(std::unique(sizes.begin(), sizes.end()) - sizes.begin()) - 1);
    }
  }
  return most;
}

enum class RdoPick { None, Size, Error };

// What one optimised curve returns to the host besides the points
struct RdoSummary {
  uint32_t n = 0;       // curve points
  uint64_t bytes0 = 0;  // payload bytes with every block at 1 x 1 (point 0)
  uint64_t bytes = 0;   // the chosen point's bytes and sse
  uint64_t sse = 0;
};

// The optimised curve after the checks, and with pick != None the payload of the point a budget picks (to size: the last with
// bytes <= budget; to error: the first with sse <= budget) into *out.  bpp: bytes per pixel counted (3 for an RGB image on the
// RGBA kernels).  The points are copied to the host arrays when cap >= n.
static pxz_status rdo(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_filter filter_down, pxz_filter filter_up, uint32_t bpp,
                      RdoPick pick, uint64_t budget, uint64_t* host_bytes, uint64_t* host_sse, size_t cap, RdoSummary* sum, pxz_payload** out) {
  // An RGB image that pxz_shrink runs on the RGBA kernels is measured and encoded as its RGBA widening (alpha is 255 in the
  // source and every decode and adds 0); the payload is narrowed back as pxz_shrink narrows it
  if (rgb_on_rgba(ctx, img->w, img->c, bw, bh)) {
    auto wide_rdo = [&](const pxz_image* wide, pxz_payload** p4) {
      return rdo(ctx, wide, bw, bh, filter_down, filter_up, 3, pick, budget, host_bytes, host_sse, cap, sum, p4);
    };
    if (pick != RdoPick::None) return encode_via_rgba(ctx, img, wide_rdo, out);
    ImageOwner wide;
    pxz_status st = rgb_widened(ctx, img, &wide);
    return st != PXZ_OK ? st : wide_rdo(wide.get(), nullptr);
  }
  Geom g;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw, bh, &g);
  if (st != PXZ_OK) return st;
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t lx_max = ceil_log2(bw), ly_max = ceil_log2(bh);
  const uint32_t npass = (lx_max + 1) * (ly_max + 1);
  const uint32_t maxev = rdo_max_events(g);
  const uint64_t nev64 = (uint64_t)nblocks * maxev;
  if (nev64 > 0x7FFFFFFFull) return fail(ctx, PXZ_E_UNSUPPORTED, "more than 2^31 optimised curve events (blocks x sizes)");
  const uint32_t nev = (uint32_t)nev64;
  if ((st = ensure_scratch(ctx, nblocks)) != PXZ_OK) return st;

  DevBlocks bufs(ctx);
  uint64_t* table = nullptr;  // [npass][nblocks] block errors
  uint8_t* ev = nullptr;      // events | base[3] | points: bytes | sse | ids | ev_pass | rank | pass0 | RdoOut
  void* scratch = nullptr;
  const size_t scratch_bytes = rdo_curve_scratch_bytes(nev);
  const size_t npt = (size_t)nev + 1;
  const size_t ev_bytes = (size_t)nev * (sizeof(RdoEvent) + 12) + 24 + npt * 16 + (size_t)nblocks * 4 + sizeof(RdoOut);
  if ((st = bufs.alloc(&table, (size_t)npass * nblocks * 8)) != PXZ_OK || (st = bufs.alloc(&ev, ev_bytes)) != PXZ_OK ||
      (st = bufs.alloc(&scratch, scratch_bytes)) != PXZ_OK)
    return st;
  RdoEvent* events = reinterpret_cast<RdoEvent*>(ev);
  uint64_t* base = reinterpret_cast<uint64_t*>(events + nev);
  uint64_t* pt_bytes = base + 3;
  uint64_t* pt_sse = pt_bytes + npt;
  uint32_t* ids = reinterpret_cast<uint32_t*>(pt_sse + npt);
  uint32_t* ev_pass = ids + nev;
  uint32_t* rank = ev_pass + nev;
  uint32_t* pass0 = rank + nev;
  RdoOut* d_out = reinterpret_cast<RdoOut*>(pass0 + nblocks);

  // 1. error table over every level pair, 2. per-block hulls, 3. the curve
  const RdPasses ps{lx_max, ly_max, ly_max + 1, 1};
  if ((st = rd_error_table(ctx, img, g, filter_down, filter_up, false, lx_max, ly_max, ps, table)) != PXZ_OK) return st;
  PXZ_CUDA(ctx, cudaMemsetAsync(base, 0, 3 * sizeof(uint64_t), ctx->stream));
  st = profiled(ctx, K_RDO_HULL, "rdo hull", [&] {
    return launch_rdo_hull(table, g, bpp, lx_max, ly_max, maxev, events, ids, ev_pass, pass0, base, ctx->stream, &ctx->launches);
  });
  if (st != PXZ_OK) return st;
  st = profiled(ctx, K_RDO_CURVE, "rdo curve", [&] {
    return launch_rdo_curve(events, ids, nev, base, pick == RdoPick::Size ? budget : 0, pick == RdoPick::Error ? budget : 0, scratch, scratch_bytes,
                            rank, pt_bytes, pt_sse, d_out, ctx->stream, ctx->sm_count, &ctx->launches);
  });
  if (st != PXZ_OK) return st;

  // 4. to the host: the summary, the chosen point, and the points when they fit
  RdoOut o;
  PXZ_CUDA(ctx, cudaMemcpyAsync(&o, d_out, sizeof(o), cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaMemcpyAsync(&sum->bytes0, pt_bytes, 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  sum->n = o.count;
  if (cap >= o.count && host_bytes && host_sse) {
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_bytes, pt_bytes, (size_t)o.count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaMemcpyAsync(host_sse, pt_sse, (size_t)o.count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if (pick == RdoPick::None) return PXZ_OK;
  const uint32_t j = pick == RdoPick::Size ? o.best_within - 1 : o.first_within;
  if (pick == RdoPick::Size && o.best_within == 0)
    return fail(ctx, PXZ_E_ARG, "max_bytes " + std::to_string(budget) + " is below the payload with every block at 1 x 1 (" +
                                    std::to_string(sum->bytes0) + " bytes)");
  if (j >= o.count) {  // the last point has sse 0 in the default resample arithmetic; with the fused one it may not
    uint64_t least = 0;
    PXZ_CUDA(ctx, cudaMemcpyAsync(&least, pt_sse + o.count - 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return fail(ctx, PXZ_E_ARG, "max_sse " + std::to_string(budget) + " is below the least squared error of any point (" + std::to_string(least) + ")");
  }

  // 5. the payload: every block forced to its vertex at point j, planned and resampled as the error table's passes are
  st = profiled(ctx, K_RDO_LEVELS, "rdo levels", [&] {
    return launch_rdo_levels(pass0, ev_pass, rank, maxev, nblocks, ly_max, j, ctx->d_vx, ctx->d_vy, ctx->stream, ctx->sm_count, &ctx->launches);
  });
  if (st != PXZ_OK) return st;
  if ((st = plan_and_resample(ctx, img, g, PXZ_METRIC_SOBEL_DIR, shrink_value_map(ctx, PXZ_METRIC_SOBEL_DIR, 0, 1.0f), filter_down, true, out)) !=
      PXZ_OK)
    return st;
  PXZ_CUDA(ctx, cudaMemcpyAsync(&sum->bytes, pt_bytes + j, 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaMemcpyAsync(&sum->sse, pt_sse + j, 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

pxz_status pxz_rdo_curve(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, pxz_filter filter_down, pxz_filter filter_up,
                         uint64_t* host_bytes, uint64_t* host_sse, size_t cap, size_t* n_out) {
  if (n_out) *n_out = 0;
  if (!ctx || !img || !n_out || (cap > 0 && (!host_bytes || !host_sse))) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  pxz_status st = rdo_refusal(ctx, img, filter_down, filter_up);
  if (st != PXZ_OK) return st;
  RdoSummary sum;
  st = rdo(ctx, img, bw, bh, filter_down, filter_up, img->c, RdoPick::None, 0, host_bytes, host_sse, cap, &sum, nullptr);
  if (st != PXZ_OK) return st;
  *n_out = sum.n;
  if (cap < sum.n) return fail(ctx, PXZ_E_ARG, "cap " + std::to_string(cap) + " is below the curve's " + std::to_string(sum.n) + " points");
  return PXZ_OK;
}

static pxz_status rdo_shrink(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, RdoPick pick, uint64_t budget, pxz_filter filter_down,
                             pxz_filter filter_up, uint64_t* bytes_out, uint64_t* sse_out, pxz_payload** out) {
  if (!ctx || !img || !out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  pxz_status st = rdo_refusal(ctx, img, filter_down, filter_up);
  if (st != PXZ_OK) return st;
  RdoSummary sum;
  st = rdo(ctx, img, bw, bh, filter_down, filter_up, img->c, pick, budget, nullptr, nullptr, 0, &sum, out);
  if (st != PXZ_OK) return st;
  if (bytes_out) *bytes_out = sum.bytes;
  if (sse_out) *sse_out = sum.sse;
  return PXZ_OK;
}

pxz_status pxz_rdo_shrink_to_size(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, uint64_t max_bytes, pxz_filter filter_down,
                                  pxz_filter filter_up, uint64_t* bytes_out, uint64_t* sse_out, pxz_payload** out) {
  return rdo_shrink(ctx, img, bw, bh, RdoPick::Size, max_bytes, filter_down, filter_up, bytes_out, sse_out, out);
}

pxz_status pxz_rdo_shrink_to_error(pxz_ctx* ctx, const pxz_image* img, uint32_t bw, uint32_t bh, uint64_t max_sse, pxz_filter filter_down,
                                   pxz_filter filter_up, uint64_t* bytes_out, uint64_t* sse_out, pxz_payload** out) {
  return rdo_shrink(ctx, img, bw, bh, RdoPick::Error, max_sse, filter_down, filter_up, bytes_out, sse_out, out);
}

pxz_status pxz_strategy_choose(const uint64_t* sse, const uint32_t* blocks, const pxz_strategy* base, pxz_strategy* out) {
  if (!sse || !blocks || !out) return PXZ_E_ARG;
  pxz_strategy b;
  if (base) {
    for (int k = 0; k < PXZ_STRATEGY_BUCKETS; ++k)
      if (base->down[k] > 4 || base->up[k] > 4) return PXZ_E_ARG;
    b = *base;
  } else {
    pxz_strategy_by_level(&b);
  }
  for (int k = 0; k < PXZ_STRATEGY_BUCKETS; ++k) {
    const uint64_t* row = sse + (size_t)k * PXZ_FILTER_PAIRS;
    const uint32_t own = (uint32_t)b.down[k] * 5u + b.up[k];
    uint32_t pick = own;
    if (blocks[k] != 0) {
      uint64_t least = row[0];
      for (uint32_t q = 1; q < PXZ_FILTER_PAIRS; ++q) least = std::min(least, row[q]);
      if (row[own] != least) {
        pick = 0;
        while (row[pick] != least) ++pick;
      }
    }
    out->down[k] = (uint8_t)(pick / 5u);
    out->up[k] = (uint8_t)(pick % 5u);
  }
  return PXZ_OK;
}

// host restatement of the plan kernel's scalar path (same threshold table)
pxz_status pxz_reduce_dims(float v0, float v1, uint32_t w, uint32_t h, uint32_t* out_w, uint32_t* out_h, float* stored) {
  if (!out_w || !out_h || w == 0 || h == 0) return PXZ_E_ARG;
  static const LevelThresholds thr = [] {  // function-local static: initialised once, thread-safe
    LevelThresholds t;
    build_level_thresholds(&t);
    return t;
  }();
  auto parse = [](float v) -> float {  // operations.rs:128-138
    if (!signbit(v)) return v;
    float x = 1.0f + v;
    return (x != x) ? 0.0f : (x > 0.0f ? x : 0.0f);
  };
  auto level = [&](float pv) -> uint32_t {
    if (pv != pv) return 0;
    if (pv >= thr.thr[0]) return 0;
    for (int k = 1; k < kThresholds; ++k)
      if (pv >= thr.thr[k]) return (uint32_t)k;
    return kLevelOnePixel;
  };
  auto dim = [](uint32_t n, uint32_t k) -> uint32_t {
    if (k >= 32) return 1;
    uint32_t d = (uint32_t)(((uint64_t)n + ((1ull << k) - 1)) >> k);
    return d < 1 ? 1 : d;
  };
  const float p0 = parse(v0), p1 = parse(v1);
  *out_w = dim(w, level(p0));
  *out_h = dim(h, level(p1));
  if (stored) *stored = (isinf(p0) || isinf(p1)) ? INFINITY : (float)sqrt((double)p0 * (double)p0 + (double)p1 * (double)p1);
  return PXZ_OK;
}

int32_t pxz_resample_table(uint32_t n_in, uint32_t n_out, pxz_filter filter, uint32_t* left, uint32_t* count, float* weights,
                           uint32_t max_taps) {
  if (!left || !count || !weights || n_in == 0 || n_out == 0) return PXZ_E_ARG;
  std::vector<uint32_t> pool;
  AxisTab t;
  if (!build_axis_table(n_in, n_out, (int)filter, &pool, &t)) return PXZ_E_ARG;
  if (t.stride > max_taps) return (int32_t)t.stride;
  for (uint32_t o = 0; o < n_out; ++o) {
    left[o] = pool[t.off + o];
    count[o] = pool[t.off + n_out + o];
    for (uint32_t i = 0; i < max_taps; ++i) {
      uint32_t bits = i < t.stride ? pool[t.off + 2 * n_out + (size_t)o * t.stride + i] : 0u;
      memcpy(&weights[(size_t)o * max_taps + i], &bits, 4);
    }
  }
  return (int32_t)t.stride;
}

// ---- payload ------------------------------------------------------------------------------------------
static pxz_status payload_bytes(pxz_ctx* ctx, const pxz_payload* cp, uint64_t* bytes) {
  pxz_payload* p = const_cast<pxz_payload*>(cp);
  if (!p->bytes_known) {
    PXZ_CUDA(ctx, cudaMemcpyAsync(ctx->h_total, p->d_total, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    p->bytes = *ctx->h_total;
    p->bytes_known = true;
  }
  *bytes = p->bytes;
  return PXZ_OK;
}

pxz_status pxz_payload_info(pxz_ctx* ctx, const pxz_payload* p, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                            uint32_t* cols, uint32_t* rows, uint32_t* channels, uint64_t* bytes) {
  if (!ctx || !p) return PXZ_E_ARG;
  if (w) *w = p->g.W;
  if (h) *h = p->g.H;
  if (bw) *bw = p->g.bw;
  if (bh) *bh = p->g.bh;
  if (cols) *cols = p->g.cols;
  if (rows) *rows = p->g.rows_img;  /* per image; pxz_payload_batch_count() images */
  if (channels) *channels = p->g.C;
  if (bytes) return payload_bytes(ctx, p, bytes);
  return PXZ_OK;
}

pxz_status pxz_payload_download(pxz_ctx* ctx, const pxz_payload* p, pxz_block_desc* host_descs, uint8_t* host_pixels) {
  if (!ctx || !p || !host_descs || !host_pixels) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  uint64_t bytes = 0;
  pxz_status st = payload_bytes(ctx, p, &bytes);
  if (st != PXZ_OK) return st;
  const size_t nblocks = (size_t)p->g.cols * p->g.rows;
  PXZ_CUDA(ctx, cudaMemcpyAsync(host_descs, p->d_descs, nblocks * sizeof(pxz_block_desc), cudaMemcpyDeviceToHost, ctx->stream));
  if (bytes) PXZ_CUDA(ctx, cudaMemcpyAsync(host_pixels, p->d_pixels, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  PXZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PXZ_OK;
}

// pixels == NULL with copy_pixels == false: the caller fills p->d_pixels on the device (pxz_payload_from_container)
static pxz_status payload_from_descs(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels,
                                     const pxz_block_desc* descs, const uint8_t* pixels, bool copy_pixels, uint64_t bytes,
                                     pxz_payload** out, uint32_t nimg = 1) {
  *out = nullptr;
  cudaSetDevice(ctx->device);
  Geom g;
  pxz_status st = make_geom(ctx, w, h, channels, bw, bh, &g, nimg);
  if (st != PXZ_OK) return st;
  // the decoder sizes the grid in f32 (encoding/mod.rs:118-119); identical to the integer ceil below 2^24
  const size_t nblocks = (size_t)g.cols * g.rows;
  // distinct (reduced, tile) size pairs -> table indices
  auto spec = std::make_shared<TabSpec>();
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> index;
  std::vector<uint32_t> tabidx(nblocks);
  std::vector<uint8_t> filt(ctx->strategy.on ? nblocks : 0);  // per-block expand filter (pxz_ctx_set_strategy)
  uint32_t max_small = 1, max_tmp_up = 1, max_tmp_down = 1, max_dim = 1;
  auto idx_of = [&](uint32_t small, uint32_t tile) -> uint32_t {
    auto it = index.find({small, tile});
    if (it != index.end()) return it->second;
    const uint32_t id = (uint32_t)spec->n_small.size();
    spec->n_small.push_back(small);
    spec->n_tile.push_back(tile);
    index[{small, tile}] = id;
    return id;
  };
  for (size_t b = 0; b < nblocks; ++b) {
    const uint32_t by = (uint32_t)((b / g.cols) % g.rows_img), bx = (uint32_t)(b % g.cols);
    // target size as Pixlzr::expand computes it (pixlzr.rs:92-107)
    const uint32_t tw = (bx == g.cols - 1 && g.trail_w) ? g.trail_w : g.bw;
    const uint32_t th = (by == g.rows_img - 1 && g.trail_h) ? g.trail_h : g.bh;
    const pxz_block_desc& d = descs[b];
    if (d.w == 0 || d.h == 0) return fail(ctx, PXZ_E_ARG, "block with zero size");
    const uint64_t sz = (uint64_t)d.w * d.h * channels;
    if (d.offset > bytes || sz > bytes - d.offset) return fail(ctx, PXZ_E_ARG, "block descriptor points outside the payload");
    if (channels == 4 && (d.offset & 3u)) return fail(ctx, PXZ_E_ARG, "RGBA block offsets must be 4-byte aligned");
    const uint32_t ix = idx_of(d.w, tw), iy = idx_of(d.h, th);
    if (ix > 0xFFFFu || iy > 0xFFFFu) return fail(ctx, PXZ_E_UNSUPPORTED, "more than 65536 distinct block sizes");
    tabidx[b] = ix | (iy << 16);
    if (ctx->strategy.on) filt[b] = ctx->strategy.up[strategy_bucket(d.value)];
    max_small = std::max(max_small, (uint32_t)d.w * d.h);
    max_dim = std::max(max_dim, (uint32_t)std::max(d.w, d.h));
    max_tmp_up = std::max(max_tmp_up, th * pad8(d.w));
    max_tmp_down = std::max(max_tmp_down, (uint32_t)d.h * pad8(tw));
  }
  PayloadOwner p;
  st = payload_new(ctx, g, bytes, &p);
  if (st != PXZ_OK) return st;
  p->spec = spec;
  if (ctx->strategy.on) {
    const uint32_t per_filter = (uint32_t)spec->n_small.size();
    if (per_filter * 5u > 0x10000u) return fail(ctx, PXZ_E_UNSUPPORTED, "too many distinct block sizes for per-block filters");
    for (size_t b = 0; b < nblocks; ++b) tabidx[b] += (filt[b] * per_filter) * 0x10001u;
    p->strategy = 2;
  }
  p->max_small_px = max_small;
  p->max_small_dim = max_dim;
  p->max_tmp_up = max_tmp_up;
  p->max_tmp_down = max_tmp_down;
  p->bytes = bytes;
  p->bytes_known = true;
  cudaError_t e = cudaMemcpyAsync(p->d_descs, descs, nblocks * sizeof(pxz_block_desc), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_tabidx, tabidx.data(), nblocks * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && bytes && copy_pixels) e = cudaMemcpyAsync(p->d_pixels, pixels, bytes, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_total, &p->bytes, 8, cudaMemcpyHostToDevice, ctx->stream);
  // work order of the expand kernel (blocks by cost class)
  if (e == cudaSuccess && ensure_scratch(ctx, (uint32_t)nblocks) != PXZ_OK) e = cudaErrorMemoryAllocation;
  if (e == cudaSuccess) e = launch_class_lists(p->d_descs, g, ctx->d_scan, p->d_order(), (uint32_t)p->nblocks_cap, ctx->stream, &ctx->launches);
  // tabidx is a pageable temporary and `pixels` may be reused by the caller right away
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return cuda_fail(ctx, e, "payload upload");
  *out = p.release();
  return PXZ_OK;
}

pxz_status pxz_payload_upload(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels,
                              const pxz_block_desc* descs, const uint8_t* pixels, uint64_t bytes, pxz_payload** out) {
  if (!ctx || !descs || (!pixels && bytes) || !out) return PXZ_E_ARG;
  return payload_from_descs(ctx, w, h, bw, bh, channels, descs, pixels, true, bytes, out);
}

pxz_status pxz_payload_upload_batch(pxz_ctx* ctx, uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels,
                                    uint32_t n_images, const pxz_block_desc* descs, const uint8_t* pixels, uint64_t bytes,
                                    pxz_payload** out) {
  if (!ctx || !descs || (!pixels && bytes) || !out || n_images == 0) return PXZ_E_ARG;
  return payload_from_descs(ctx, w, h, bw, bh, channels, descs, pixels, true, bytes, out, n_images);
}

uint32_t pxz_image_batch_count(const pxz_image* img) { return img ? img->nimg : 0; }
uint32_t pxz_payload_batch_count(const pxz_payload* p) { return p ? p->g.nimg : 0; }

pxz_status pxz_shrink_batch(pxz_ctx* ctx, const pxz_image* batch, uint32_t bw, uint32_t bh, pxz_metric metric, float factor,
                            pxz_filter filter_down, uint32_t flags, pxz_payload** out) {
  // one launch per stage over the tiles of all images: the batch is one block grid (pxz_internal.h, Geom)
  return pxz_shrink(ctx, batch, bw, bh, metric, factor, filter_down, flags, out);
}

pxz_status pxz_expand_batch(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, pxz_image* out_batch) {
  return pxz_expand_to_image(ctx, p, filter_up, out_batch);
}

// ---- container stage on the device (qoi_device.cu) ------------------------------------------------------------
pxz_status pxz_payload_to_container(pxz_ctx* ctx, const pxz_payload* p, uint32_t filter_byte, int values_present, uint8_t* host_out,
                                    size_t cap, uint64_t* bytes_out) {
  if (!ctx || !p || !host_out || !bytes_out) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (p->g.nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "a container holds one image: not available on a batch");
  uint64_t bytes = 0;
  pxz_status st = payload_bytes(ctx, p, &bytes);
  if (st != PXZ_OK) return st;
  const Geom& g = p->g;
  const uint32_t nblocks = g.cols * g.rows;
  const size_t arena_bytes = qoi_arena_bytes(nblocks, bytes, g.C);
  const size_t out_cap = 26 + (size_t)4 * g.rows + arena_bytes;
  DevBlocks bufs(ctx);
  uint8_t *d_arena = nullptr, *d_out = nullptr;
  uint32_t* d_len = nullptr;
  unsigned long long *d_off = nullptr, *d_total = nullptr;
  if ((st = bufs.alloc(&d_arena, arena_bytes)) != PXZ_OK || (st = bufs.alloc(&d_out, out_cap)) != PXZ_OK ||
      (st = bufs.alloc(&d_len, (size_t)nblocks * 4)) != PXZ_OK || (st = bufs.alloc(&d_off, (size_t)nblocks * 8)) != PXZ_OK ||
      (st = bufs.alloc(&d_total, 8)) != PXZ_OK)
    return st;
  st = profiled(ctx, K_QOI_ENCODE, "container encode", [&] {
    return launch_qoi_encode(p->d_descs, p->d_pixels, g, values_present, filter_byte, d_arena, d_len, d_off, d_out, d_total, ctx->stream,
                             &ctx->launches);
  });
  if (st != PXZ_OK) return st;
  unsigned long long total = 0;
  cudaError_t e = cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess && total <= cap) {
    e = cudaMemcpyAsync(host_out, d_out, total, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  if (e != cudaSuccess) return cuda_fail(ctx, e, "container encode");
  *bytes_out = total;
  if (total > cap) return fail(ctx, PXZ_E_ARG, "output buffer too small (size it with pxz_container_bound)");
  return PXZ_OK;
}

pxz_status pxz_payload_from_container(pxz_ctx* ctx, const uint8_t* data, size_t len, int32_t* filter_byte, pxz_payload** out) {
  if (!ctx || !data || !out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  uint32_t w, h, bw, bh, ch;
  int32_t filt = -1;
  uint64_t bytes = 0;
  // the host walks the headers (a few bytes per block); the streams themselves are decoded on the device
  pxz_status st = pxz_container_decode(data, len, &w, &h, &bw, &bh, &filt, &ch, &bytes, nullptr, nullptr);
  if (st != PXZ_OK) return fail(ctx, st, "malformed .pxlzr container");
  Geom g;
  if ((st = make_geom(ctx, w, h, ch, bw, bh, &g)) != PXZ_OK) return st;
  const size_t nblocks = (size_t)g.cols * g.rows;  // == the decoder's f32 grid: pxz_container_decode refuses files where they differ
  std::vector<pxz_block_desc> descs(nblocks);
  st = pxz_container_decode(data, len, &w, &h, &bw, &bh, &filt, &ch, &bytes, descs.data(), nullptr);
  if (st != PXZ_OK) return fail(ctx, st, "malformed .pxlzr container");
  std::vector<unsigned long long> in_off(nblocks);
  std::vector<uint32_t> qlen(nblocks);
  {
    size_t q = 26 + (size_t)4 * g.rows;  // constants.rs:19-20 + the line table; validated by the walk above
    for (size_t b = 0; b < nblocks; ++b) {
      if (q + 13 > len) return fail(ctx, PXZ_E_FORMAT, "malformed .pxlzr container");  // cannot happen after the walk above
      const uint8_t* hd = data + q + 9;
      qlen[b] = (uint32_t)hd[0] << 24 | (uint32_t)hd[1] << 16 | (uint32_t)hd[2] << 8 | hd[3];
      in_off[b] = q + 13;
      q += 13 + (size_t)qlen[b];
      if (q > len) return fail(ctx, PXZ_E_FORMAT, "malformed .pxlzr container");
    }
  }
  for (size_t b = 0; b < nblocks; ++b)
    if (ch == 4 && (descs[b].offset & 3u)) return fail(ctx, PXZ_E_UNSUPPORTED, "unaligned RGBA block");  // cannot happen: w*h*4
  pxz_payload* raw = nullptr;
  st = payload_from_descs(ctx, w, h, bw, bh, ch, descs.data(), nullptr, false, bytes, &raw);
  if (st != PXZ_OK) return st;
  PayloadOwner p(raw);
  DevBlocks bufs(ctx);
  uint8_t* d_in = nullptr;
  unsigned long long* d_off = nullptr;
  uint32_t* d_len = nullptr;
  int* d_err = nullptr;
  if ((st = bufs.alloc(&d_in, len)) != PXZ_OK || (st = bufs.alloc(&d_off, nblocks * 8)) != PXZ_OK ||
      (st = bufs.alloc(&d_len, nblocks * 4)) != PXZ_OK || (st = bufs.alloc(&d_err, 4)) != PXZ_OK)
    return st;
  int err = 0;
  cudaError_t e = cudaMemcpyAsync(d_in, data, len, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, in_off.data(), nblocks * 8, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_len, qlen.data(), nblocks * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_err, 0, 4, ctx->stream);
  if (e == cudaSuccess) {
    ProfScope prof(ctx, K_QOI_DECODE);
    e = launch_qoi_decode(d_in, d_off, d_len, p->d_descs, g, p->d_pixels, d_err, ctx->stream, &ctx->launches);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return cuda_fail(ctx, e, "container decode");
  if (err) return fail(ctx, PXZ_E_FORMAT, "truncated QOI stream");
  if (filter_byte) *filter_byte = filt;
  *out = p.release();
  return PXZ_OK;
}

void pxz_payload_free(pxz_payload* p) { payload_release(p); }

// ---- decode -------------------------------------------------------------------------------------------
pxz_status pxz_expand_to_image(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, pxz_image* out) {
  if (!ctx || !p || !out) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (!known_filter(filter_up)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (out->w != p->g.W || out->h != p->g.H || out->c != p->g.C || out->nimg != p->g.nimg)
    return fail(ctx, PXZ_E_ARG, "output image geometry mismatch");
  if (rgb_on_rgba(ctx, p->g.W, p->g.C, p->g.bw, p->g.bh) && p->max_small_dim <= 64) {
    PayloadOwner p4;
    pxz_status st = payload_rechannel(ctx, p, 4, &p4);
    if (st != PXZ_OK) return st;
    ImageOwner wide;
    if ((st = image_new(ctx, out->w, out->h, 4, out->nimg, &wide)) != PXZ_OK) return st;
    if ((st = pxz_expand_to_image(ctx, p4.get(), filter_up, wide.get())) != PXZ_OK) return st;
    cudaError_t e = launch_rgb_widen(wide->d, wide->pitch, out->d, out->pitch, out->w, out->h * out->nimg, 0, ctx->stream, ctx->sm_count,
                                     &ctx->launches);
    return e == cudaSuccess ? PXZ_OK : cuda_fail(ctx, e, "rgb narrow");
  }
  TabSet ts;
  pxz_status st = get_tabset(ctx, *p->spec, p->strategy ? -1 : (int)filter_up, 1, &ts);
  if (st != PXZ_OK) return st;
  return run_resample(ctx, 1, out->d, out->pitch, p, ts, p->max_small_px, p->max_small_dim, p->max_tmp_up);
}

pxz_status pxz_expand(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, uint8_t* host_out, size_t host_pitch) {
  if (!ctx || !p || !host_out) return PXZ_E_ARG;
  ImageOwner im;
  pxz_status st = image_new(ctx, p->g.W, p->g.H, p->g.C, p->g.nimg, &im);
  if (st != PXZ_OK) return st;
  st = pxz_expand_to_image(ctx, p, filter_up, im.get());
  return st != PXZ_OK ? st : pxz_image_download(ctx, im.get(), host_out, host_pitch);
}

// ---- random access (extension) ------------------------------------------------------------------------------------
// A block's expand reads only its descriptor, its pixels and its tile size, so the blocks of a window, given the tile
// sizes they have in the whole image, are an ordinary payload whose expand is that window of the whole expand.
pxz_status pxz_payload_window(pxz_ctx* ctx, const pxz_payload* p, uint32_t c0, uint32_t r0, uint32_t nc, uint32_t nr,
                              pxz_payload** out) {
  if (!ctx || !p || !out) return PXZ_E_ARG;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  const Geom& pg = p->g;
  if (pg.nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "windows of a batch payload are not supported");
  if (nc == 0 || nr == 0 || c0 >= pg.cols || r0 >= pg.rows || nc > pg.cols - c0 || nr > pg.rows - r0)
    return fail(ctx, PXZ_E_ARG, "empty or out-of-grid window");
  const uint32_t w = (uint32_t)(std::min<uint64_t>(pg.W, (uint64_t)(c0 + nc) * pg.bw) - (uint64_t)c0 * pg.bw);
  const uint32_t h = (uint32_t)(std::min<uint64_t>(pg.H, (uint64_t)(r0 + nr) * pg.bh) - (uint64_t)r0 * pg.bh);
  Geom g;
  pxz_status st = make_geom(ctx, w, h, pg.C, pg.bw, pg.bh, &g);
  if (st != PXZ_OK) return st;
  const uint32_t nblocks = nc * nr;
  if ((st = ensure_scratch(ctx, nblocks, window_scan_state_bytes(nblocks))) != PXZ_OK) return st;
  // max_small_px bounds every block of p, whatever made it (uploads may hold blocks larger than their tiles); the parent's
  // capacity alone could be the whole gigapixel frame
  const uint64_t capacity = std::min<uint64_t>(p->capacity, (uint64_t)nblocks * p->max_small_px * pg.C);
  PayloadOwner wp;
  if ((st = payload_new(ctx, g, capacity, &wp)) != PXZ_OK) return st;
  copy_layout(wp.get(), p);  // the window's table indices are the parent's: same spec, same bounds, same kernel family
  st = profiled(ctx, K_PAYLOAD_WINDOW, "payload window", [&] {
    return launch_payload_window(p->d_descs, p->d_tabidx, (uint32_t)p->nblocks_cap, p->d_pixels, pg.cols, c0, r0, g, p->strategy == 1, wp->d_descs,
                                 wp->d_tabidx, (uint32_t)wp->nblocks_cap, wp->d_pixels, wp->d_total, ctx->d_scan, ctx->stream, &ctx->launches);
  });
  if (st != PXZ_OK) return st;
  *out = wp.release();
  return PXZ_OK;
}

pxz_status pxz_expand_region(pxz_ctx* ctx, const pxz_payload* p, pxz_filter filter_up, uint32_t x, uint32_t y, uint32_t w,
                             uint32_t h, pxz_image* out) {
  if (!ctx || !p || !out) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  const Geom& pg = p->g;
  if (pg.nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "regions of a batch payload are not supported");
  if (!known_filter(filter_up)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (w == 0 || h == 0) return fail(ctx, PXZ_E_ARG, "empty rectangle");
  if (x >= pg.W || y >= pg.H || w > pg.W - x || h > pg.H - y) return fail(ctx, PXZ_E_ARG, "rectangle outside the image");
  if (out->w != w || out->h != h || out->c != pg.C || out->nimg != 1) return fail(ctx, PXZ_E_ARG, "output image geometry mismatch");
  if (x == 0 && y == 0 && w == pg.W && h == pg.H) return pxz_expand_to_image(ctx, p, filter_up, out);
  const uint32_t c0 = x / pg.bw, r0 = y / pg.bh;
  const uint32_t nc = (x + w - 1) / pg.bw - c0 + 1, nr = (y + h - 1) / pg.bh - r0 + 1;
  pxz_payload* raw = nullptr;
  pxz_status st = pxz_payload_window(ctx, p, c0, r0, nc, nr, &raw);
  if (st != PXZ_OK) return st;
  const PayloadOwner wp(raw);
  const uint32_t dx = x - c0 * pg.bw, dy = y - r0 * pg.bh;
  if (dx == 0 && dy == 0 && w == wp->g.W && h == wp->g.H) return pxz_expand_to_image(ctx, wp.get(), filter_up, out);  // no staging
  ImageOwner stage;  // freed stream-ordered: the copy queued below keeps it
  if ((st = image_new(ctx, wp->g.W, wp->g.H, pg.C, 1, &stage)) != PXZ_OK) return st;
  if ((st = pxz_expand_to_image(ctx, wp.get(), filter_up, stage.get())) != PXZ_OK) return st;
  return profiled(ctx, K_REGION_COPY, "region copy", [&] {
    return cudaMemcpy2DAsync(out->d, out->pitch, stage->d + (size_t)dy * stage->pitch + (size_t)dx * pg.C, stage->pitch, (size_t)w * pg.C, h,
                             cudaMemcpyDeviceToDevice, ctx->stream);
  });
}

// ---- quadtree processing (process/tree.rs:23-109) ---------------------------------------------------------
pxz_status pxz_tree_process(pxz_ctx* ctx, const pxz_image* img, float threshold, uint32_t bw, uint32_t bh, uint32_t min_bw,
                            uint32_t min_bh, pxz_filter filter_down, pxz_filter filter_up, pxz_image* out) {
  if (!ctx || !img || !out) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (!known_filter(filter_down) || !known_filter(filter_up)) return fail(ctx, PXZ_E_ARG, "unknown filter");
  if (out->w != img->w || out->h != img->h || out->c != img->c) return fail(ctx, PXZ_E_ARG, "output image geometry mismatch");
  if (img->nimg != 1 || out->nimg != 1) return fail(ctx, PXZ_E_UNSUPPORTED, "tree processing takes one image at a time");
  if (bw == 0 || bh == 0) return fail(ctx, PXZ_E_ARG, "block size must be >= 1");
  // unchanged pixels (blocks that reach the minimum size, tree.rs:35-37) come straight from the source
  PXZ_CUDA(ctx, cudaMemcpy2DAsync(out->d, out->pitch, img->d, img->pitch, (size_t)img->w * img->c, img->h, cudaMemcpyDeviceToDevice,
                                  ctx->stream));
  const uint32_t mbw = std::max(min_bw, 4u), mbh = std::max(min_bh, 4u);  // :33-34
  int levels = 0;
  while ((bw >> levels) > mbw && (bh >> levels) > mbh) ++levels;
  if (levels == 0) return PXZ_OK;  // :35-37: image.clone()
  // the reference splits every block relative to its own origin; the levels form global grids only when the halved
  // sizes stay exact, which is what the accelerated path covers
  if ((bw & ((1u << (levels - 1)) - 1)) || (bh & ((1u << (levels - 1)) - 1)))
    return fail(ctx, PXZ_E_UNSUPPORTED, "tree processing needs block sizes divisible by 2^(levels-1)");
  const bool positive = threshold >= 0.0f;  // :38
  const float thr = fabsf(threshold);       // :39

  DevBlocks bufs(ctx);
  uint8_t* d_leaf = nullptr;
  uint8_t* d_rec[2] = {nullptr, nullptr};
  Geom gl;
  pxz_status st = make_geom(ctx, img->w, img->h, img->c, bw >> (levels - 1), bh >> (levels - 1), &gl);
  if (st != PXZ_OK) return st;
  const size_t max_blocks = (size_t)gl.cols * gl.rows;
  if ((st = bufs.alloc(&d_leaf, max_blocks)) != PXZ_OK || (st = bufs.alloc(&d_rec[0], max_blocks)) != PXZ_OK ||
      (st = bufs.alloc(&d_rec[1], max_blocks)) != PXZ_OK)
    return st;
  uint32_t parent_cols = 0;
  for (int lv = 0; lv < levels; ++lv) {
    Geom g;
    if ((st = make_geom(ctx, img->w, img->h, img->c, bw >> lv, bh >> lv, &g)) != PXZ_OK) return st;
    ValueMap vm;
    vm.factor = 1.0f; vm.mode = 1; vm.normalise = 0;  // after = identity (tree.rs:97)
    vm.extra_thr = thr;
    if ((st = run_analysis(ctx, img, g, PXZ_METRIC_OKLAB_MAD, false, &vm)) != PXZ_OK) return st;
    cudaError_t e = launch_tree_mask(ctx->d_vx, g, lv == 0 ? nullptr : d_rec[(lv - 1) & 1], parent_cols, thr,
                                     (lv == 0 ? positive : true) ? 1 : 0,  // the recursion receives |threshold| (:70)
                                     d_leaf, d_rec[lv & 1], ctx->stream, &ctx->launches);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "tree mask");
    parent_cols = g.cols;
    PayloadOwner p;
    if ((st = payload_new(ctx, g, (uint64_t)g.W * g.H * g.C, &p)) != PXZ_OK) return st;
    p->spec = spec_for_geom(g);
    set_plan_bounds(p.get(), g, true);
    vm.extra_thr = NAN;
    e = launch_plan(ctx->d_vx, nullptr, g, vm, ctx->d_minmax, ctx->thr, d_leaf, p->d_descs, p->d_tabidx, p->d_total, ctx->d_scan, p->d_order(),
                    (uint32_t)p->nblocks_cap, ctx->stream, &ctx->launches);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "plan");
    TabSet ts;
    if ((st = get_tabset(ctx, *p->spec, (int)filter_down, 0, &ts)) != PXZ_OK) return st;
    if ((st = run_resample(ctx, 0, img->d, img->pitch, p.get(), ts, g.bw * g.bh, std::max(g.bw, g.bh), p->max_tmp_down)) != PXZ_OK) return st;
    if ((st = get_tabset(ctx, *p->spec, (int)filter_up, 1, &ts)) != PXZ_OK) return st;
    if ((st = run_resample(ctx, 1, out->d, out->pitch, p.get(), ts, p->max_small_px, p->max_small_dim, p->max_tmp_up)) != PXZ_OK) return st;
  }
  return PXZ_OK;
}

// ---- multi-GPU ----------------------------------------------------------------------------------------
pxz_status pxz_comm_unique_id(uint8_t id[PXZ_COMM_ID_BYTES]) {
  if (!id) return PXZ_E_ARG;
  std::string err;
  if (nccl_get_unique_id(id, &err) != 0) {
    fprintf(stderr, "pixlzr_b200: %s\n", err.c_str());
    return PXZ_E_NCCL;
  }
  return PXZ_OK;
}

pxz_status pxz_comm_init(pxz_ctx* ctx, int nranks, int rank, const uint8_t id[PXZ_COMM_ID_BYTES]) {
  if (!ctx || !id || nranks < 1 || rank < 0 || rank >= nranks) return PXZ_E_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->comm) {
    nccl_comm_destroy(ctx->comm);
    ctx->comm = nullptr;
  }
  std::string err;
  if (nccl_comm_init(&ctx->comm, nranks, rank, id, &err) != 0) return fail(ctx, PXZ_E_NCCL, err);
  return PXZ_OK;
}

void pxz_comm_destroy(pxz_ctx* ctx) {
  if (ctx && ctx->comm) {
    nccl_comm_destroy(ctx->comm);
    ctx->comm = nullptr;
  }
}

}  // extern "C"
