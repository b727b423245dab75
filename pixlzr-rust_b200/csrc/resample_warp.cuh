// resample_warp.cuh — warp-per-tile resample kernels for RGBA8 tiles up to 64x64 (included by kernels.cu, namespace pxz).
//
// Every warp owns one tile at a time (tiles are handed out through an atomic counter), so there is no CTA barrier
// anywhere and a light tile never idles the threads of a heavy one:
//   * shrink (k_shrink_warp): the tiles k_shrink_tma (resample_tma.cuh) leaves, those whose vertical table has no slide2
//     form (more than 6 outputs live at once).  Lane = columns 2x and 2x + 1; every group of 4 output rows walks its
//     source rows straight from global memory / L1 (blocked table form) into an 8-row strip of f32 intermediates in
//     shared memory; whenever the strip is full the warp runs the horizontal pass over it and writes the packed payload
//     pixels.
//   * expand: the (small) source block is streamed once through a 7-row register window of converted samples; two
//     rows of intermediates at a time go through shared memory to the horizontal pass, which writes the image tile
//     (the paste is fused: 16-byte stores into the pitched image).
// Arithmetic order per output is the reference's (ascending taps, product and sum rounded separately), on the packed
// f32x2 pipe (Acc4 / mac2 in kernels.cu).
#pragma once

#ifndef PXZ_SHRINK_WARPS
#define PXZ_SHRINK_WARPS 4
#endif
constexpr int kWarpCtaThreads = 128;  // expand: 4 warps per CTA
constexpr int kWarpsPerCta = kWarpCtaThreads / 32;
constexpr int kShrinkWarps = PXZ_SHRINK_WARPS;
constexpr int kShrinkCtaThreads = kShrinkWarps * 32;
constexpr int kStripRows = 8;         // shrink: rows of intermediates per horizontal batch
constexpr int kStripStride = 65;      // float4 per strip row: 64 + 1, so 8 rows of one column sit in 8 different banks
constexpr int kHTabWords = 512;       // shrink: per-warp copy of the tile's horizontal table (2 KB), else read via L1
constexpr int kShrinkWarpBytes = kStripRows * kStripStride * 16 + kHTabWords * 4;
constexpr int kExpandRow1 = 68;       // expand: second strip row starts at 64 + pad (pad chosen per tile, <= 4)
constexpr int kExpandPairPx = kExpandRow1 + 64 + 8;  // one pair of strip rows (second row at 64 + pad), + the walk's overrun
constexpr int kExpandWarpBytes = 2 * kExpandPairPx * 16;  // two pairs: blocks at most 16 wide run two row pairs per vertical pass

// v-th block in cost order (lists: see launch_plan); nullptr = natural order
struct TileOrder {
  const uint32_t* lists;
  uint32_t cap;
  uint32_t end[8];  // running class totals
  __device__ __forceinline__ void init(const uint32_t* l, uint32_t c) {
    lists = l; cap = c;
    uint32_t run = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      run += l ? __ldg(l + (size_t)8 * c + i) : 0u;
      end[i] = run;
    }
  }
  __device__ __forceinline__ uint32_t at(uint32_t v) const {
    if (lists == nullptr) return v;
    uint32_t c = 0, start = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i)
      if (v >= end[i]) { c = i + 1; start = end[i]; }
    return __ldg(lists + (size_t)c * cap + (v - start));
  }
};

// lane 0 only: position in the order list, or 0xFFFFFFFF when every tile has been handed out; `n_drawn` = draws before this one.
// The draw count is the 64-bit word at `counter`; n_drawn adds its two halves (the high half stays zero).  Reading the low
// half alone would give the same values but changes the generated code of the three warp-per-tile kernels.
__device__ __forceinline__ uint32_t draw_position(uint32_t* counter, uint32_t ntiles, uint32_t& n_drawn) {
  const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long*>(counter), 1ull);
  const uint32_t f = (uint32_t)old;
  n_drawn = f + (uint32_t)(old >> 32);
  return n_drawn < ntiles ? f : 0xFFFFFFFFu;
}

// next tile of this warp (lane 0 asks, everybody gets the answer).  Every warp draws exactly one position past the end;
// the warp that draws the very last one puts the counter back to zero for the next launch on this stream.
__device__ __forceinline__ uint32_t next_tile(uint32_t* counter, uint32_t ntiles, uint32_t total_warps) {
  uint32_t v = 0;
  if ((threadIdx.x & 31u) == 0) {
    uint32_t n;
    v = draw_position(counter, ntiles, n);
    if (n == ntiles + total_warps - 1) *reinterpret_cast<unsigned long long*>(counter) = 0ull;
  }
  return __shfl_sync(0xffffffffu, v, 0);
}

// ---- shrink ------------------------------------------------------------------------------------------------------
constexpr uint32_t kBlockedFrom = 8;  // outputs per row from which the horizontal pass walks groups of 4 (else scalar chains)
// The horizontal table of a tile as the pass reads it: from kBlockedFrom outputs the blocked form (w4 rows | lo | rows | first), else the
// per-output form (left | count | weights).  `tab` points at a per-warp shared-memory copy when it fits, else at the pool.
struct HTab {
  const uint32_t* tab;
  uint32_t nb, brows_total, stride;
};
__device__ __forceinline__ HTab stage_htab(const AxisTab& tx, uint32_t dw, const uint32_t* __restrict__ pool, uint32_t* smem_tab) {
  const uint32_t lane = threadIdx.x & 31u;
  HTab h;
  h.nb = tx.nb; h.brows_total = tx.brows_total; h.stride = tx.stride;
  const uint32_t* src = dw >= kBlockedFrom ? pool + tx.boff : pool + tx.off;
  const uint32_t words = dw >= kBlockedFrom ? tx.bwords : 2 * dw + dw * tx.stride;
  if (words <= (uint32_t)kHTabWords) {
    for (uint32_t i = lane; i < words; i += 32) smem_tab[i] = __ldg(src + i);
    h.tab = smem_tab;
  } else {
    h.tab = src;
  }
  return h;
}

// horizontal pass over `nrows` strip rows (output rows row0 .. row0 + nrows - 1) -> payload block at dst
template <int MODE>
__device__ __forceinline__ void shrink_horizontal(const float4* strip, uint32_t row0, uint32_t nrows, uint32_t dw, const HTab& ht,
                                                  uint32_t* dst, const TapK& k) {
  const uint32_t lane = threadIdx.x & 31u;
  if (dw >= kBlockedFrom) {
    // groups of 4 outputs share one walk (blocked table form); item = (strip row, group): the 8 lanes of a
    // shared-memory phase read the same column of 8 different rows = 8 different banks (row stride 65)
    const ulonglong2* w4 = reinterpret_cast<const ulonglong2*>(ht.tab);
    const uint32_t* lo = ht.tab + 4 * ht.brows_total;
    const uint32_t* rows = lo + ht.nb;
    const uint32_t* first = rows + ht.nb;
    for (uint32_t i = lane; i < ht.nb * kStripRows; i += 32) {
      const uint32_t r = i & (kStripRows - 1), ob = i / kStripRows;
      if (r >= nrows) continue;
      const uint32_t n = rows[ob];
      const ulonglong2* wp = w4 + first[ob];
      const float4* tp = strip + r * kStripStride + lo[ob];
      Acc4<MODE> acc;
      uint32_t c = n;
      for (; c >= 2; c -= 2) {
        const float4 p0 = tp[0], p1 = tp[1];
        const ulonglong2 w0 = wp[0], w1 = wp[1];
        acc.step(p0, w0, k);
        acc.step(p1, w1, k);
        tp += 2;
        wp += 2;
      }
      if (c) acc.step(tp[0], wp[0], k);
      const uint32_t ox = ob * 4, nvalid = min(4u, dw - ox);
      uint32_t* o = dst + (size_t)(row0 + r) * dw + ox;
      const uint4 pk = acc.pack4();
      o[0] = pk.x;
      if (nvalid > 1) o[1] = pk.y;
      if (nvalid > 2) o[2] = pk.z;
      if (nvalid > 3) o[3] = pk.w;
    }
  } else {
    // few outputs: one scalar chain per (row, output, channel)
    const uint32_t* left = ht.tab;
    const uint32_t* cnt = left + dw;
    const float* w = reinterpret_cast<const float*>(left + 2 * dw);
    const uint32_t total = nrows * dw * 4;
    for (uint32_t i = lane; i < total; i += 32) {
      const uint32_t c = i & 3u, j = i >> 2, r = j / dw, ox = j - r * dw;
      uint32_t byte = 0xFFu;
      if ((MODE & 1) || c < 3) {
        const uint32_t n = cnt[ox];
        const float* wr = w + ox * ht.stride;
        const float* tp = reinterpret_cast<const float*>(strip + r * kStripStride + left[ox]) + c;
        float a = 0.f;
        uint32_t t = 0;
        for (; t + 4 <= n; t += 4) {
          const float p0 = tp[0], p1 = tp[4], p2 = tp[8], p3 = tp[12];
          const float w0 = wr[t], w1 = wr[t + 1], w2 = wr[t + 2], w3 = wr[t + 3];
          a = mac1<MODE>(a, p0, w0); a = mac1<MODE>(a, p1, w1); a = mac1<MODE>(a, p2, w2); a = mac1<MODE>(a, p3, w3);
          tp += 16;
        }
        for (; t < n; ++t) {
          a = mac1<MODE>(a, tp[0], wr[t]);
          tp += 4;
        }
        byte = to_u8_fast(a);
      }
      reinterpret_cast<uint8_t*>(dst)[((size_t)(row0 + r) * dw + ox) * 4 + c] = (uint8_t)byte;
    }
  }
}

// Vertical pass from the blocked table (two groups of 4 output rows per strip, each walking its source rows straight from
// global memory / L1), then the horizontal pass over the strip.
template <int MODE>
__device__ __forceinline__ void shrink_tile_warp(const uint8_t* __restrict__ img, size_t pitch, const Tile& t,
                                                 const pxz_block_desc& d, const HTab& ht, const AxisTab& ty,
                                                 const uint32_t* __restrict__ pool, float4* strip,
                                                 uint8_t* __restrict__ payload, const TapK& k) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t dw = d.w, dh = d.h;
  const bool has = 2 * lane < t.tw;  // tile widths are multiples of 4 here
  const uint8_t* col0 = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4 + (size_t)lane * 8;
  uint32_t* dst = reinterpret_cast<uint32_t*>(payload + d.offset);
  const ulonglong2* w4 = reinterpret_cast<const ulonglong2*>(pool + ty.boff);
  const uint32_t* lo = pool + ty.boff + 4 * ty.brows_total;
  const uint32_t* rows = lo + ty.nb;
  const uint32_t* first = rows + ty.nb;
  for (uint32_t batch0 = 0, ob = 0; batch0 < dh; batch0 += kStripRows) {
    for (uint32_t j = 0; j < 2 && ob < ty.nb; ++j, ++ob) {
      const uint32_t n = __ldg(rows + ob), r0 = __ldg(lo + ob);
      const ulonglong2* wp = w4 + __ldg(first + ob);
      Acc4<MODE> a0, a1;
      for (uint32_t r = 0; r < n; ++r) {
        const uint2 px = has ? __ldg(reinterpret_cast<const uint2*>(col0 + (size_t)(r0 + r) * pitch)) : make_uint2(0u, 0u);
        const ulonglong2 w = __ldg(wp + r);
        a0.step(px_to_f4<MODE>(px.x), w, k);
        a1.step(px_to_f4<MODE>(px.y), w, k);
      }
      float4* srow = strip + (j * 4) * kStripStride + 2 * lane;
      srow[0] = a0.out(0); srow[1] = a1.out(0);
      srow[kStripStride] = a0.out(1); srow[kStripStride + 1] = a1.out(1);
      srow[2 * kStripStride] = a0.out(2); srow[2 * kStripStride + 1] = a1.out(2);
      srow[3 * kStripStride] = a0.out(3); srow[3 * kStripStride + 1] = a1.out(3);
    }
    __syncwarp();
    shrink_horizontal<MODE>(strip, batch0, min((uint32_t)kStripRows, dh - batch0), dw, ht, dst, k);
    __syncwarp();
  }
}

template <bool FUSED>
__global__ void __launch_bounds__(kShrinkCtaThreads, PXZ_SHRINK_WARP_CTAS) k_shrink_warp(
    const uint8_t* __restrict__ img, size_t pitch, Geom g, const pxz_block_desc* __restrict__ descs,
    const uint32_t* __restrict__ tabidx, const uint32_t* __restrict__ lists, uint32_t cap, const uint8_t* __restrict__ opaque_flags,
    uint8_t* __restrict__ payload,
    const AxisTab* __restrict__ tabs, const uint32_t* __restrict__ pool, uint32_t* counter, float rt_one, float rt_negzero) {
  extern __shared__ float4 s_warp[];
  float4* strip = s_warp + (threadIdx.x >> 5) * (kShrinkWarpBytes / 16);
  uint32_t* htab_smem = reinterpret_cast<uint32_t*>(strip + kStripRows * kStripStride);
  const TapK k = make_tapk(rt_one, rt_negzero);
  pdl_wait();
  pdl_trigger();
  const uint32_t ntiles = g.cols * g.rows, total_warps = gridDim.x * kShrinkWarps;
  constexpr int F = FUSED ? 2 : 0;
  uint32_t last_tx = 0xFFFFFFFFu, last_ty = 0xFFFFFFFFu;
  AxisTab ty{};
  HTab ht{};
  auto process = [&](uint32_t b, const pxz_block_desc& d, uint32_t ti) {
    const Tile t = tile_of(g, b);
    if (d.w == 0 || d.h == 0) return;  // masked out (quadtree levels)
    // launched behind k_shrink_tma, which copies the full-size blocks and shrinks every tile whose vertical table has a
    // slide2 form
    if ((d.w == t.tw && d.h == t.th) || tabs[ti >> 16].s2words != 0) return;
    // tiles come in cost order, so a warp's consecutive tiles mostly share their tables: keep them
    if ((ti >> 16) != last_ty) {
      ty = tabs[ti >> 16];
      last_ty = ti >> 16;
    }
    if ((ti & 0xFFFFu) != last_tx) {
      __syncwarp();  // the previous tile's horizontal pass is done with the table copy
      ht = stage_htab(tabs[ti & 0xFFFFu], d.w, pool, htab_smem);
      __syncwarp();
      last_tx = ti & 0xFFFFu;
    }
    const bool opaque = opaque_flags != nullptr && opaque_flags[b] != 0;
    if (opaque) shrink_tile_warp<F>(img, pitch, t, d, ht, ty, pool, strip, payload, k);
    else shrink_tile_warp<F | 1>(img, pitch, t, d, ht, ty, pool, strip, payload, k);
  };
  // Tiles are drawn in the order of the `order` list (most expensive first, so the kernel does not end on a few warps
  // that drew a 20-microsecond tile last); the next tile's index, descriptor and table indices are requested while the
  // current tile is processed.
  TileOrder ord;
  ord.init(lists, cap);
  uint32_t v = next_tile(counter, ntiles, total_warps);
  uint32_t b = 0, ti = 0;
  pxz_block_desc d{};
  if (v < ntiles) { b = ord.at(v); d = descs[b]; ti = tabidx[b]; }
  while (v < ntiles) {
    const uint32_t vn = next_tile(counter, ntiles, total_warps);
    uint32_t bn = 0, tin = 0;
    pxz_block_desc dn{};
    if (vn < ntiles) { bn = ord.at(vn); dn = descs[bn]; tin = tabidx[bn]; }
    process(b, d, ti);
    v = vn; b = bn; d = dn; ti = tin;
  }
}

// ---- expand ------------------------------------------------------------------------------------------------------
// fixed-length walk of the horizontal pass (the table stores every group with STEPS rows, +0 weights beyond its own)
template <int MODE, int STEPS>
__device__ __forceinline__ void expand_walk(Acc4<MODE>& acc, const float4* tp, const ulonglong2 (&w)[8], const TapK& k) {
#pragma unroll
  for (int c = 0; c < STEPS; ++c) acc.step(tp[c], w[c], k);
}

template <int MODE>
__device__ __forceinline__ void expand_tile_warp(uint8_t* __restrict__ img, size_t pitch, const Tile& t, const pxz_block_desc& d,
                                                 const AxisTab& tx, const AxisTab& ty, const uint32_t* __restrict__ pool,
                                                 float4* strip, const uint8_t* __restrict__ payload, const TapK& k) {
  constexpr int NC = (MODE & 1) ? 4 : 3;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t sw = d.w, sh = d.h, dw = t.tw, dh = t.th;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(payload + d.offset);
  uint8_t* dst = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
  const float4* g8 = reinterpret_cast<const float4*>(pool + ty.goff);
  const uint32_t* gleft = pool + ty.goff + 8 * ty.n_out;
  const ulonglong2* gp = reinterpret_cast<const ulonglong2*>(pool + ty.gpoff);
  // second strip row: offset so that the 8 lanes of a shared-memory phase (4 groups x 2 rows) hit 8 different banks:
  // a 2x upscale reads every other column (odd offset), wider ratios read adjacent columns (offset 4)
  const uint32_t row1 = 64 + ((tx.n_out == 2 * tx.n_in) ? 1u : 4u);
  // one intermediate sample of strip row `r1` (0 / 1) of pair `pr`, column x
  auto put = [&](uint32_t pr, uint32_t r1, uint32_t x, const float (&v)[4]) {
    strip[pr * kExpandPairPx + (r1 ? row1 : 0u) + x] = make_float4(v[0], v[1], v[2], v[3]);
  };

  // horizontal: lane = (group of 4 outputs, strip row); fixed for the whole tile
  const uint32_t hr = lane & 1u, ob = lane >> 1;
  const bool hact = ob < tx.nb;
  const uint32_t* blo = pool + tx.boff + 4 * tx.brows_total;
  const uint32_t hn = hact ? __ldg(blo + tx.nb + ob) : 0u;
  const uint32_t hlo = hact ? __ldg(blo + ob) : 0u;
  const float4* htp = strip + hr * row1 + hlo;
  const ulonglong2* hw = reinterpret_cast<const ulonglong2*>(pool + tx.boff) + (hact ? __ldg(blo + 2 * tx.nb + ob) : 0u);
  const uint32_t hox = ob * 4, hvalid = hact ? min(4u, dw - hox) : 0u;
  const uint32_t bpad = tx.bpad;
  // the walk of this lane's group is the same for every row of the tile: its weights stay in registers
  ulonglong2 hwr[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) hwr[c] = (hact && (uint32_t)c < bpad) ? __ldg(hw + c) : make_ulonglong2(0ull, 0ull);
  auto horizontal = [&](uint32_t oy0, uint32_t nrows, const float4* tp) {  // tp: this lane's first sample of the row pair
    if (hact && hr < nrows) {
      Acc4<MODE> acc;
      if (bpad == 8) expand_walk<MODE, 8>(acc, tp, hwr, k);
      else if (bpad == 4) expand_walk<MODE, 4>(acc, tp, hwr, k);
      else if (bpad == 2) expand_walk<MODE, 2>(acc, tp, hwr, k);
      else
        for (uint32_t c = 0; c < hn; ++c) acc.step(tp[c], __ldg(hw + c), k);
      uint32_t* o = reinterpret_cast<uint32_t*>(dst + (size_t)(oy0 + hr) * pitch) + hox;
      const uint4 pk = acc.pack4();
      const uint32_t p0 = pk.x, p1 = pk.y, p2 = pk.z, p3 = pk.w;
      if (hvalid == 4) {
        *reinterpret_cast<uint4*>(o) = make_uint4(p0, p1, p2, p3);  // tile rows are 16-byte aligned
      } else {
        o[0] = p0;
        if (hvalid > 1) o[1] = p1;
        if (hvalid > 2) o[2] = p2;
      }
    }
  };

  if (sw <= 4 && sh <= 4) {
    // Tiny source (a block reduced to at most 4 x 4: three of the eight classes of the bench frame).  The whole vertical
    // pass is done at once — lane = output rows 2 lane, 2 lane + 1 (the two lanes of the f32x2 operations), one source
    // column at a time, every tap of the column (taps before a row's first one get weight +0, which leaves the sum as it
    // is) — into a compact [row][4] array of intermediates; the horizontal pass then runs down the tile without the
    // per-pair window / table-request bookkeeping of the general path (6.4 K -> 3 K instructions per tile).
    const uint32_t y0 = 2 * lane;
    u64 wp[4];  // (weight of row y0, weight of row y0 + 1) for source rows 0..3
    {
      float wa[2][4];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const uint32_t y = min(y0 + r, dh - 1);
        const float4 w4 = __ldg(g8 + 2 * y);
        const uint32_t l = __ldg(gleft + y);
        const float w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float v = 0.f;
#pragma unroll
          for (int t = 0; t <= j; ++t) v = (l + t == (uint32_t)j) ? w[t] : v;
          wa[r][j] = v;
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) wp[j] = pk2(wa[0][j], wa[1][j]);
    }
    for (uint32_t x = 0; x < sw; ++x) {
      u64 a[NC];
#pragma unroll
      for (int c = 0; c < NC; ++c) a[c] = 0ull;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if ((uint32_t)j < sh) {
          const float4 pf = px_to_f4<MODE>(__ldg(src + (size_t)j * sw + x));
          const float pc[4] = {pf.x, pf.y, pf.z, pf.w};
#pragma unroll
          for (int c = 0; c < NC; ++c) mac2_acc<MODE>(a[c], pk2(pc[c], pc[c]), wp[j], k);
        }
      }
      float lo_[4] = {0.f, 0.f, 0.f, 0.f}, hi_[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < NC; ++c) unpk2(a[c], lo_[c], hi_[c]);
      if (y0 < dh) strip[y0 * 4 + x] = make_float4(lo_[0], lo_[1], lo_[2], lo_[3]);
      if (y0 + 1 < dh) strip[(y0 + 1) * 4 + x] = make_float4(hi_[0], hi_[1], hi_[2], hi_[3]);
    }
    __syncwarp();
    const float4* tp = strip + hr * 4 + hlo;  // the lane's first sample as in the general path, rows 4 samples apart
    for (uint32_t oy0 = 0; oy0 < dh; oy0 += 2, tp += 8) horizontal(oy0, min(2u, dh - oy0), tp);
    __syncwarp();
  } else if (sw <= 32) {
    // vertical: lane = source column; a 7-row window of converted samples lives in registers and moves down with the
    // outputs' first tap.  Two output rows with the same first tap are the two lanes of one f32x2 accumulator.  Blocks
    // at most 16 wide use the upper half warp for the next pair of rows (own window, own table rows): 4 rows per pass.
    const uint32_t nh = sw <= 16 ? 2u : 1u;
    const uint32_t half = nh == 2 ? lane >> 4 : 0u, x = nh == 2 ? (lane & 15u) : lane;
    const bool vact = x < sw;
    float win[7][NC];
    auto conv = [&](uint32_t word, float(&o)[NC]) {
      const float4 p = px_to_f4<MODE>(word);
      o[0] = p.x; o[1] = p.y; o[2] = p.z;
      if (NC > 3) o[NC > 3 ? 3 : 0] = p.w;
    };
#pragma unroll
    for (int j = 0; j < 7; ++j) conv((vact && (uint32_t)j < sh) ? __ldg(src + (size_t)j * sw + x) : 0u, win[j]);
    uint32_t L = 0;
    uint32_t nextpx = (vact && 7 < sh) ? __ldg(src + (size_t)7 * sw + x) : 0u;
    auto advance = [&](uint32_t left) {
      while (L < left) {
#pragma unroll
        for (int j = 0; j < 6; ++j)
#pragma unroll
          for (int c = 0; c < NC; ++c) win[j][c] = win[j + 1][c];
        conv(nextpx, win[6]);
        ++L;
        nextpx = (vact && L + 7 < sh) ? __ldg(src + (size_t)(L + 7) * sw + x) : 0u;
      }
    };
    auto vrow_solo = [&](uint32_t oy, uint32_t r1) {
      advance(__ldg(gleft + oy));
      const float4 wa = __ldg(g8 + 2 * oy), wb = __ldg(g8 + 2 * oy + 1);
      const float w[7] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z};
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 7; ++j)
#pragma unroll
        for (int c = 0; c < NC; ++c) a[c] = mac1<MODE>(a[c], win[j][c], w[j]);
      if (vact) put(half, r1, x, a);
    };
    // The table rows of a pair of output rows are requested right after the vertical pass of the previous pair (into
    // the same registers: they are dead by then), one horizontal pass before they are used.
    ulonglong2 w01 = make_ulonglong2(0ull, 0ull), w23 = w01, w45 = w01, w67 = w01;
    uint32_t la = 0, lb = 0;
    auto request = [&](uint32_t oy) {  // table rows of the pair (oy, oy + 1)
      if (oy < dh) {
        const ulonglong2* wn = gp + 4 * (oy >> 1);
        w01 = __ldg(wn); w23 = __ldg(wn + 1); w45 = __ldg(wn + 2); w67 = __ldg(wn + 3);
        la = __ldg(gleft + oy);
        lb = oy + 1 < dh ? __ldg(gleft + oy + 1) : la;
      }
    };
    request(2 * half);
    for (uint32_t oy0 = 0; oy0 < dh; oy0 += 2 * nh) {
      const uint32_t my = oy0 + 2 * half;  // this lane's pair of output rows
      if (my >= dh) {
        // no rows left for the upper half warp
      } else if (la == lb) {
        advance(la);
        const u64 w[7] = {w01.x, w01.y, w23.x, w23.y, w45.x, w45.y, w67.x};
        u64 a[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) a[c] = 0ull;
        // blocks of at most 2 / 4 rows have at most that many taps (the table rows are +0 beyond them)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int c = 0; c < NC; ++c) mac2_acc<MODE>(a[c], pk2(win[j][c], win[j][c]), w[j], k);
        if (sh > 2) {
#pragma unroll
          for (int j = 2; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < NC; ++c) mac2_acc<MODE>(a[c], pk2(win[j][c], win[j][c]), w[j], k);
          if (sh > 4) {
#pragma unroll
            for (int j = 4; j < 7; ++j)
#pragma unroll
              for (int c = 0; c < NC; ++c) mac2_acc<MODE>(a[c], pk2(win[j][c], win[j][c]), w[j], k);
          }
        }
        if (vact) {
          float lo_[4] = {0.f, 0.f, 0.f, 0.f}, hi_[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int c = 0; c < NC; ++c) unpk2(a[c], lo_[c], hi_[c]);
          put(half, 0u, x, lo_);
          put(half, 1u, x, hi_);
        }
      } else {
        vrow_solo(my, 0u);
        vrow_solo(my + 1, 1u);
      }
      request(my + 2 * nh);
      __syncwarp();
      horizontal(oy0, min(2u, dh - oy0), htp);
      if (nh == 2 && oy0 + 2 < dh) horizontal(oy0 + 2, min(2u, dh - oy0 - 2), htp + kExpandPairPx);
      __syncwarp();
    }
  } else {
    // wide source (only one axis was reduced): every tap is read and converted where it is used
    const bool has0 = lane < sw, has1 = lane + 32 < sw;
    const uint32_t* lcnt = pool + ty.off + ty.n_out;
    for (uint32_t oy0 = 0; oy0 < dh; oy0 += 2) {
      const uint32_t nrows = min(2u, dh - oy0);
      for (uint32_t r = 0; r < nrows; ++r) {
        const uint32_t oy = oy0 + r, left = __ldg(gleft + oy), n = __ldg(lcnt + oy);
        const float* w = reinterpret_cast<const float*>(g8 + 2 * oy);
        float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
        for (uint32_t j = 0; j < n; ++j) {
          const float wj = __ldg(w + j);
          const float4 p0 = px_to_f4<MODE>(has0 ? __ldg(src + (size_t)(left + j) * sw + lane) : 0u);
          const float4 p1 = px_to_f4<MODE>(has1 ? __ldg(src + (size_t)(left + j) * sw + lane + 32) : 0u);
          const float c0[4] = {p0.x, p0.y, p0.z, p0.w}, c1[4] = {p1.x, p1.y, p1.z, p1.w};
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            a0[c] = mac1<MODE>(a0[c], c0[c], wj);
            a1[c] = mac1<MODE>(a1[c], c1[c], wj);
          }
        }
        if (has0) put(0u, r, lane, a0);
        if (has1) put(0u, r, lane + 32, a1);
      }
      __syncwarp();
      horizontal(oy0, nrows, htp);
      __syncwarp();
    }
  }
}

template <bool FUSED>
__global__ void __launch_bounds__(kWarpCtaThreads, PXZ_EXPAND_WARP_CTAS) k_expand_warp(
    uint8_t* __restrict__ img, size_t pitch, Geom g, const pxz_block_desc* __restrict__ descs,
    const uint32_t* __restrict__ tabidx, const uint32_t* __restrict__ lists, uint32_t cap, const uint8_t* __restrict__ payload,
    const AxisTab* __restrict__ tabs,
    const uint32_t* __restrict__ pool, uint32_t* counter, float rt_one, float rt_negzero) {
  extern __shared__ float4 s_warp[];
  float4* strip = s_warp + (threadIdx.x >> 5) * (kExpandWarpBytes / 16);
  const TapK k = make_tapk(rt_one, rt_negzero);
  const uint32_t lane = threadIdx.x & 31u;
  // the fixed-length walks read up to 7 strip entries past a group's own window: keep them finite (w = +0 there)
  for (uint32_t i = lane; i < kExpandWarpBytes / 16; i += 32) strip[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  pdl_wait();
  pdl_trigger();
  const uint32_t ntiles = g.cols * g.rows, total_warps = gridDim.x * kWarpsPerCta;
  constexpr int F = FUSED ? 2 : 0;
  auto process = [&](uint32_t b, const pxz_block_desc& d, uint32_t ti) {
    const Tile t = tile_of(g, b);
    const uint32_t sw = d.w, sh = d.h, dw = t.tw, dh = t.th;
    if (sw == 0 || sh == 0) return;  // masked out: the tile keeps what the output image already holds
    uint8_t* dst = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(payload + d.offset);
    if (sw == dw && sh == dh) {
      const bool has = 2 * lane < dw;
      for (uint32_t r0 = 0; r0 < dh; r0 += 8) {
        uint32_t v0[8], v1[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v0[j] = (r0 + j < dh && has) ? __ldcs(src + (size_t)(r0 + j) * dw + 2 * lane) : 0u;
          v1[j] = (r0 + j < dh && has) ? __ldcs(src + (size_t)(r0 + j) * dw + 2 * lane + 1) : 0u;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (r0 + j < dh && has) *reinterpret_cast<uint2*>(dst + (size_t)(r0 + j) * pitch + lane * 8) = make_uint2(v0[j], v1[j]);
      }
      return;
    }
    if (sw == 1 && sh == 1) {
      // every output has one tap of normalised weight w / w = 1.0 in both passes: the tile is the source pixel
      const uint32_t p = __ldg(src);
      const uint4 v = make_uint4(p, p, p, p);
      // lane = (row of a pair, group of 4 pixels): two rows of 16 groups per pass, no division in the loop
      const uint32_t x = (lane & 15u) << 2;
      if (x < dw) {
        uint8_t* o = dst + (size_t)(lane >> 4) * pitch + (size_t)x * 4;
        if (x + 4 <= dw) {
          for (uint32_t y = lane >> 4; y < dh; y += 2, o += 2 * pitch) *reinterpret_cast<uint4*>(o) = v;
        } else {
          for (uint32_t y = lane >> 4; y < dh; y += 2, o += 2 * pitch)
            for (uint32_t i = 0; x + i < dw; ++i) reinterpret_cast<uint32_t*>(o)[i] = p;
        }
      }
      return;
    }
    const AxisTab tx = tabs[ti & 0xFFFFu], ty = tabs[ti >> 16];
    uint32_t aand = 0xFF000000u;
    for (uint32_t i = lane; i < sw * sh; i += 32) aand &= __ldg(src + i);
    const bool opaque = __all_sync(0xffffffffu, (aand & 0xFF000000u) == 0xFF000000u) != 0;
    if (opaque) expand_tile_warp<F>(img, pitch, t, d, tx, ty, pool, strip, payload, k);
    else expand_tile_warp<F | 1>(img, pitch, t, d, tx, ty, pool, strip, payload, k);
  };
  // Tiles are drawn in the order of the `order` list (most expensive first, so the kernel does not end on a few warps
  // that drew a 20-microsecond tile last); the next tile's index, descriptor and table indices are requested while the
  // current tile is processed.
  TileOrder ord;
  ord.init(lists, cap);
  uint32_t v = next_tile(counter, ntiles, total_warps);
  uint32_t b = 0, ti = 0;
  pxz_block_desc d{};
  if (v < ntiles) { b = ord.at(v); d = descs[b]; ti = tabidx[b]; }
  while (v < ntiles) {
    const uint32_t vn = next_tile(counter, ntiles, total_warps);
    uint32_t bn = 0, tin = 0;
    pxz_block_desc dn{};
    if (vn < ntiles) { bn = ord.at(vn); dn = descs[bn]; tin = tabidx[bn]; }
    process(b, d, ti);
    v = vn; b = bn; d = dn; ti = tin;
  }
}
