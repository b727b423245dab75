// resample_tma.cuh — TMA-fed warp-per-tile shrink kernel for RGBA8 tiles up to 64x64 (included by kernels.cu after
// resample_warp.cuh, namespace pxz).  Replaces the body of PixlzrBlock::resize on the encode side
// (src/data_types/block.rs:273-290, image-crate branch) for whole images at once.
//
// Every warp owns one tile at a time (tiles come from an atomic counter in cost order, next tile one ahead):
//   * the source tile is streamed from the pitched image with 2-D tensor copies (cp.async.bulk.tensor, one elected
//     lane, 64 px x 4 rows = 1 KB per box) into a 5-slot ring with one mbarrier per slot; the stream runs on into the
//     warp's NEXT tile, so a warp never starts a tile with an empty pipe;
//   * the tile's two tables (vertical: slide2 form, horizontal: blocked / per-output form) are staged into the warp's
//     shared memory with 1-D bulk copies, only when they differ from the previous tile's (tiles arrive in cost order);
//   * vertical pass: lane = image columns 2x, 2x + 1 — the two lanes of every f32x2 operation — so a pixel pair is
//     converted with two byte permutes and one packed add, and the weights come as (w, w) pairs straight from shared
//     memory (no register moves); every source row feeds the <= 6 live output rows, finished rows go to an 8-row strip
//     (even columns in the first half of a strip row, odd ones in the second: conflict-free 16-byte stores);
//   * horizontal pass per strip: item = (strip row, group of 4 outputs) on the blocked table.
// Arithmetic order per output is the reference's (ascending taps, product and sum rounded separately).
#pragma once

#include <cuda.h>  // CUtensorMap (types only: the encode entry point is fetched through cudaGetDriverEntryPoint)

#ifndef PXZ_TMA_WARPS
#define PXZ_TMA_WARPS 4
#endif
#ifndef PXZ_TMA_BOXROWS
#define PXZ_TMA_BOXROWS 4
#endif
#ifndef PXZ_TMA_SLOTS
#define PXZ_TMA_SLOTS 5
#endif
constexpr int kTWarps = PXZ_TMA_WARPS;         // warps (= tiles in flight) per CTA
constexpr int kTBoxRows = PXZ_TMA_BOXROWS;     // source rows per tensor copy
constexpr int kTSlots = PXZ_TMA_SLOTS;         // ring slots per warp
constexpr int kTBoxBytes = kTBoxRows * 64 * 4; // 1 KB
#ifndef PXZ_TMA_STRIPROWS
#define PXZ_TMA_STRIPROWS 8
#endif
constexpr int kTStripRows = PXZ_TMA_STRIPROWS;  // output rows per horizontal batch (a power of two)
constexpr int kTStripStride = 65;              // float4 per strip row
constexpr int kTVtabWords = 64 * 12 + 64;      // slide2 table of a 64-sample axis with 6 slots + end[64]
constexpr int kTHtabWords = 512;
constexpr int kTRingOff = 0;
constexpr int kTStripOff = kTRingOff + kTSlots * kTBoxBytes;
constexpr int kTVtabOff = kTStripOff + kTStripRows * kTStripStride * 16;
constexpr int kTHtabOff = kTVtabOff + kTVtabWords * 4;
constexpr int kTBarOff = kTHtabOff + kTHtabWords * 4;
constexpr int kTWarpBytes = ((kTBarOff + 8 * (kTSlots + 1)) + 127) & ~127;
static_assert(kTStripOff % 128 == 0 && kTVtabOff % 16 == 0 && kTHtabOff % 16 == 0 && kTBarOff % 8 == 0, "smem layout");

// ---- mbarrier / bulk-copy PTX ------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // labels inside a PTX block are local to it, so inlined copies do not clash
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PXZ_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra PXZ_DONE;\n"
      "bra PXZ_WAIT;\n"
      "PXZ_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t x, uint32_t y, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(tm), "r"(x), "r"(y), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- the warp's tile queue ------------------------------------------------------------------------------------------
// A tile's descriptor is three dependent trips to L2 away (work counter -> order list -> descriptor).  The chain for
// the tile AFTER the next one runs while the current tile is processed: the atomic is issued when the tile starts, the
// list entry is requested a few boxes later, the descriptor a few boxes after that (tq_tick, called at every box
// boundary), so no step waits for the one before it.
struct TDesc {
  uint32_t b, ti, op;
  pxz_block_desc d;
  bool valid;
};
struct TQueue {
  const pxz_block_desc* descs;
  const uint32_t* tabidx;
  const uint8_t* opaque;
  uint32_t* counter;
  uint32_t ntiles;
  TileOrder ord;
  uint32_t raw;        // lane 0: the drawn position (atomic in flight)
  bool drawing;        // this warp has not yet drawn an index >= ntiles
  TDesc q;             // the tile being fetched
  uint32_t step;       // 0: drawn | 1: list entry requested | 2: descriptor requested
  uint32_t tick, next_at;
};
__device__ __forceinline__ void tq_start(TQueue& q) {
  q.raw = 0xFFFFFFFFu;
  if (q.drawing && (threadIdx.x & 31u) == 0) {
    uint32_t n;
    q.raw = draw_position(q.counter, q.ntiles, n);
  }
  q.step = 0; q.tick = 0; q.next_at = 4;
}
__device__ __forceinline__ void tq_advance(TQueue& q) {
  if (q.step == 0) {
    const uint32_t v = __shfl_sync(0xffffffffu, q.raw, 0);
    q.drawing = v < q.ntiles;
    q.q.valid = q.drawing;
    q.q.b = q.q.valid ? q.ord.at(v) : 0u;
    q.step = 1;
  } else if (q.step == 1) {
    q.q.ti = 0; q.q.op = 0; q.q.d = pxz_block_desc{};
    if (q.q.valid) {
      q.q.d = q.descs[q.q.b];
      q.q.ti = q.tabidx[q.q.b];
      q.q.op = q.opaque != nullptr ? (uint32_t)q.opaque[q.q.b] : 0u;
    }
    q.step = 2;
  }
}
__device__ __forceinline__ void tq_tick(TQueue& q) {
  if (++q.tick == q.next_at) {
    tq_advance(q);
    q.next_at += 5;
  }
}
__device__ __forceinline__ TDesc tq_finish(TQueue& q) {
  while (q.step < 2) tq_advance(q);
  return q.q;
}

// ---- the warp's source stream -------------------------------------------------------------------------------------
// Boxes are issued and consumed in one global order (this tile's boxes, then the next tile's), slot = order % kTSlots.
struct TFeed {
  uint32_t ring, bars;         // shared-space byte addresses (ring slot 0, barrier 0)
  uint32_t inflight;           // boxes issued and not yet released
  uint32_t islot;              // slot of the next box to issue
  uint32_t rslot, rpar;        // slot / phase parity of the next box to wait for
  uint32_t cx, cy, cnb, cpb;   // current tile: origin (pixels), boxes, boxes issued
  uint32_t nx, ny, nnb, npb;   // next tile
};

__device__ __forceinline__ void tfeed_pump(TFeed& f, const CUtensorMap* tm) {
  const bool leader = (threadIdx.x & 31u) == 0;
  while (f.inflight < (uint32_t)kTSlots) {
    uint32_t x, y;
    if (f.cpb < f.cnb) { x = f.cx; y = f.cy + f.cpb * kTBoxRows; ++f.cpb; }
    else if (f.npb < f.nnb) { x = f.nx; y = f.ny + f.npb * kTBoxRows; ++f.npb; }
    else break;
    if (leader) {
      const uint32_t bar = f.bars + 8u * f.islot;
      mbar_expect_tx(bar, kTBoxBytes);
      tma_load_2d(f.ring + f.islot * kTBoxBytes, tm, x, y, bar);
    }
    f.islot = f.islot + 1 == (uint32_t)kTSlots ? 0u : f.islot + 1;
    ++f.inflight;
  }
}
// blocks until the next box of the stream has landed; returns its shared-space address
__device__ __forceinline__ uint32_t tfeed_wait(TFeed& f) {
  mbar_wait(f.bars + 8u * f.rslot, f.rpar);
  const uint32_t addr = f.ring + f.rslot * kTBoxBytes;
  if (f.rslot + 1 == (uint32_t)kTSlots) { f.rslot = 0; f.rpar ^= 1u; }
  else ++f.rslot;
  return addr;
}
// the oldest box has been read by every lane: its slot takes the next box of the stream
__device__ __forceinline__ void tfeed_release(TFeed& f, const CUtensorMap* tm, TQueue& q) {
  __syncwarp();
  --f.inflight;
  tfeed_pump(f, tm);
  tq_tick(q);
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds_u32x2(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ ulonglong2 lds_u64x2(uint32_t addr) {
  ulonglong2 v;
  asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "r"(addr));
  return v;
}

// swizzled strip column: even columns in [0, 32), odd ones in [32, 64)
__device__ __forceinline__ uint32_t strip_col(uint32_t c) { return (c >> 1) + ((c & 1u) << 5); }

// ---- horizontal pass over `nrows` strip rows (output rows row0 .. row0 + nrows - 1) -> payload block at dst ------
template <int MODE>
__device__ __forceinline__ void tma_horizontal_body(const float4* strip, uint32_t row0, uint32_t nrows, uint32_t dw, const HTab& ht,
                                                    uint32_t* dst, const TapK& k) {
  const uint32_t lane = threadIdx.x & 31u;
  if (dw >= kBlockedFrom) {
    const ulonglong2* w4 = reinterpret_cast<const ulonglong2*>(ht.tab);
    const uint32_t* lo = ht.tab + 4 * ht.brows_total;
    const uint32_t* rows = lo + ht.nb;
    const uint32_t* first = rows + ht.nb;
    for (uint32_t i = lane; i < ht.nb * kTStripRows; i += 32) {
      const uint32_t r = i & (kTStripRows - 1), ob = i / kTStripRows;
      if (r >= nrows) continue;
      const uint32_t n = rows[ob], c0 = lo[ob];
      const ulonglong2* wp = w4 + first[ob];
      const float4* row = strip + r * kTStripStride;
      const float4* pa = row + strip_col(c0);       // columns c0, c0 + 2, ...
      const float4* pb = row + strip_col(c0 + 1);   // columns c0 + 1, c0 + 3, ...
      Acc4<MODE> acc;
      uint32_t c = n;
      for (; c >= 2; c -= 2) {
        const float4 p0 = pa[0], p1 = pb[0];
        const ulonglong2 w0 = wp[0], w1 = wp[1];
        acc.step(p0, w0, k);
        acc.step(p1, w1, k);
        ++pa; ++pb;
        wp += 2;
      }
      if (c) acc.step(pa[0], wp[0], k);
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
        const uint32_t n = cnt[ox], l0 = left[ox];
        const float* wr = w + ox * ht.stride;
        const float* row = reinterpret_cast<const float*>(strip + r * kTStripStride) + c;
        float a = 0.f;
        uint32_t t = 0;
        for (; t + 4 <= n; t += 4) {
          const float p0 = row[strip_col(l0 + t) * 4], p1 = row[strip_col(l0 + t + 1) * 4];
          const float p2 = row[strip_col(l0 + t + 2) * 4], p3 = row[strip_col(l0 + t + 3) * 4];
          const float w0 = wr[t], w1 = wr[t + 1], w2 = wr[t + 2], w3 = wr[t + 3];
          a = mac1<MODE>(a, p0, w0); a = mac1<MODE>(a, p1, w1); a = mac1<MODE>(a, p2, w2); a = mac1<MODE>(a, p3, w3);
        }
        for (; t < n; ++t) a = mac1<MODE>(a, row[strip_col(l0 + t) * 4], wr[t]);
        byte = to_u8_fast(a);
      }
      reinterpret_cast<uint8_t*>(dst)[((size_t)(row0 + r) * dw + ox) * 4 + c] = (uint8_t)byte;
    }
  }
}

// A real call for the vertical variants that are not worth their own copy of the pass (2- and 4-slot tables with more
// output rows than slots: filters other than Lanczos3 / Gaussian); the Lanczos3 path and the short tiles inline it.
template <int MODE>
__device__ __noinline__ void tma_horizontal_call(const float4* strip, uint32_t row0, uint32_t nrows, uint32_t dw, const HTab ht,
                                                 uint32_t* dst, float rt_one, float rt_negzero) {
  const TapK k = make_tapk(rt_one, rt_negzero);
  tma_horizontal_body<MODE>(strip, row0, nrows, dw, ht, dst, k);
}
template <int MODE, bool INLINE>
__device__ __forceinline__ void tma_horizontal(const float4* strip, uint32_t row0, uint32_t nrows, uint32_t dw, const HTab& ht,
                                               uint32_t* dst, const TapK& k) {
  if (INLINE) tma_horizontal_body<MODE>(strip, row0, nrows, dw, ht, dst, k);
  else tma_horizontal_call<MODE>(strip, row0, nrows, dw, ht, dst, k.one, k.nz);
}

// ---- tiles whose output rows all fit the accumulators (dh <= A) ------------------------------------------------------
// Every output row keeps its own accumulator for the whole walk and nothing is emitted on the way: the loop is one
// box per iteration, its rows unrolled (loads of the whole box first).  TS = slot pairs per table row; A <= TS.
__device__ __forceinline__ u64 lds_u64(uint32_t addr) {
  u64 v;
  asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
  return v;
}
template <int MODE>
__device__ __forceinline__ void px_pair_to_f32x2(const uint2& px, u64 (&pp)[(MODE & 1) ? 4 : 3]) {
  constexpr int NC = (MODE & 1) ? 4 : 3;
  const u64 magic = pk2(-8388608.0f, -8388608.0f);
  pp[0] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7440)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7440))), magic);
  pp[1] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7441)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7441))), magic);
  pp[2] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7442)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7442))), magic);
  if (NC > 3) pp[NC > 3 ? 3 : 0] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7443)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7443))), magic);
}
template <int MODE, int A, int TS>
__device__ __forceinline__ void tma_shrink_tile_simple(TFeed& f, TQueue& q, const CUtensorMap* tm, uint32_t sh, uint32_t dw, uint32_t dh,
                                                       uint32_t vtab, float4* strip, const HTab& ht, uint32_t* dst, const TapK& k) {
  constexpr int NC = (MODE & 1) ? 4 : 3;
  constexpr int R = kTBoxRows;
  const uint32_t lane = threadIdx.x & 31u;
  u64 acc[A][NC];
#pragma unroll
  for (int s = 0; s < A; ++s)
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[s][c] = 0ull;
  auto load_w = [&](uint32_t wrow, u64(&w)[A]) {
    if (A == 1) {
      w[0] = lds_u64(wrow);
    } else {
#pragma unroll
      for (int s = 0; s < A; s += 2) {
        const ulonglong2 t = lds_u64x2(wrow + s * 8);
        w[s] = t.x;
        w[s + 1 < A ? s + 1 : s] = t.y;
      }
    }
  };
  const uint32_t nbox = (sh + R - 1) / R;
  uint32_t wrow = vtab;
  for (uint32_t bx = 0; bx < nbox; ++bx) {
    const uint32_t box = tfeed_wait(f) + lane * 8;
    const uint32_t nr = min((uint32_t)R, sh - bx * R);
    if (nr == (uint32_t)R) {
      uint2 px[R];
      u64 w[R][A];
#pragma unroll
      for (int j = 0; j < R; ++j) px[j] = lds_u32x2(box + j * 256);
#pragma unroll
      for (int j = 0; j < R; ++j) load_w(wrow + j * (TS * 8), w[j]);
#pragma unroll
      for (int j = 0; j < R; ++j) {
        u64 pp[NC];
        px_pair_to_f32x2<MODE>(px[j], pp);
#pragma unroll
        for (int s = 0; s < A; ++s)
#pragma unroll
          for (int c = 0; c < NC; ++c) mac2_acc<MODE>(acc[s][c], pp[c], w[j][s], k);
      }
    } else {
      for (uint32_t j = 0; j < nr; ++j) {
        const uint2 px = lds_u32x2(box + j * 256);
        u64 w[A], pp[NC];
        load_w(wrow + j * (TS * 8), w);
        px_pair_to_f32x2<MODE>(px, pp);
#pragma unroll
        for (int s = 0; s < A; ++s)
#pragma unroll
          for (int c = 0; c < NC; ++c) mac2_acc<MODE>(acc[s][c], pp[c], w[s], k);
      }
    }
    wrow += R * TS * 8;
    tfeed_release(f, tm, q);
  }
#pragma unroll
  for (int o = 0; o < A; ++o) {
    if ((uint32_t)o < dh) {
      float4* srow = strip + o * kTStripStride + lane;
      srow[0] = make_float4(lo2(acc[o][0]), lo2(acc[o][1]), lo2(acc[o][2]), NC > 3 ? lo2(acc[o][NC > 3 ? 3 : 0]) : 0.f);
      srow[32] = make_float4(hi2(acc[o][0]), hi2(acc[o][1]), hi2(acc[o][2]), NC > 3 ? hi2(acc[o][NC > 3 ? 3 : 0]) : 0.f);
    }
  }
}

// ---- vertical pass + horizontal batches of one tile -----------------------------------------------------------------
// A = accumulator slots of the tile's slide2 table (2, 4, 6); the stream has this tile's boxes next.
template <int MODE, int A>
__device__ __forceinline__ void tma_shrink_tile(TFeed& f, TQueue& q, const CUtensorMap* tm, uint32_t sh, uint32_t dw, uint32_t dh, uint32_t vtab,
                                                float4* strip, const HTab& ht, uint32_t* dst, const TapK& k) {
  constexpr int NC = (MODE & 1) ? 4 : 3;
  const uint32_t lane = threadIdx.x & 31u;
  u64 acc[A][NC];
#pragma unroll
  for (int s = 0; s < A; ++s)
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[s][c] = 0ull;
  // shared-space address of this lane's column of the strip, made opaque: derived from the thread index, the compiler
  // would otherwise rebuild it (two S2R and an IMAD) for every finished row
  uint32_t strip_lane_sa = (uint32_t)__cvta_generic_to_shared(strip + lane);
  asm volatile("mov.u32 %0, %0;" : "+r"(strip_lane_sa));
  const u64 magic = pk2(-8388608.0f, -8388608.0f);
  const uint32_t endp = vtab + sh * (A * 8);  // end[o], after the table rows
  // row 0: pixels and weights
  uint32_t box = tfeed_wait(f) + lane * 8;  // this lane's two pixels of the box's first row
  uint32_t boxes_read = 1, rib = 0;         // rows of the current box already loaded
  uint2 px = lds_u32x2(box);
  uint32_t wrow = vtab;
  ulonglong2 w01 = lds_u64x2(wrow), w23 = make_ulonglong2(0ull, 0ull), w45 = w23;
  if (A > 2) w23 = lds_u64x2(wrow + 16);
  if (A > 4) w45 = lds_u64x2(wrow + 32);
  uint32_t r = 0, o = 0, slot = 0, batch0 = 0;
  uint32_t e = lds_u32(endp);
  const uint32_t nbox = (sh + kTBoxRows - 1) / kTBoxRows;
  // one source row: its taps into the live accumulators, then the next row's operands
  auto one_row = [&]() {
    // this row's operands
    u64 pp[NC];
    pp[0] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7440)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7440))), magic);
    pp[1] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7441)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7441))), magic);
    pp[2] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7442)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7442))), magic);
    if (NC > 3) pp[NC > 3 ? 3 : 0] = add2(pk2(__uint_as_float(__byte_perm(px.x, 0x4B000000u, 0x7443)), __uint_as_float(__byte_perm(px.y, 0x4B000000u, 0x7443))), magic);
    {
      const u64 w[6] = {w01.x, w01.y, w23.x, w23.y, w45.x, w45.y};
#pragma unroll
      for (int s = 0; s < A; ++s)
#pragma unroll
        for (int c = 0; c < NC; ++c) mac2_acc<MODE>(acc[s][c], pp[c], w[s], k);
    }
    // next row's operands, into the registers this row's just left (the pixels of row r are converted: a box whose
    // last row that was is free)
    ++r;
    ++rib;
    if (r < sh) {
      if (rib == (uint32_t)kTBoxRows) {
        tfeed_release(f, tm, q);
        box = tfeed_wait(f) + lane * 8;
        ++boxes_read;
        rib = 0;
      }
      px = lds_u32x2(box + rib * 256);
      wrow += A * 8;
      w01 = lds_u64x2(wrow);
      if (A > 2) w23 = lds_u64x2(wrow + 16);
      if (A > 4) w45 = lds_u64x2(wrow + 32);
    }
  };
  for (;;) {
    while (r <= e) one_row();  // (two rows per trip: no gain per level, and the larger code cost 5 us on the mixed frame)
    // output row o is complete in accumulator slot `slot`: to the strip, slot cleared
    {
      // one short block per slot behind a real branch: the stores and the clears are volatile asm, so the compiler cannot
      // turn the switch into selects over all six slots (it did: 88 instructions per finished row)
      const uint32_t sa = strip_lane_sa + (o - batch0) * (kTStripStride * 16);
#define PXZ_TAKE(S)                                                                                                   \
  case S:                                                                                                             \
    if (S < A) {                                                                                                      \
      constexpr int S_ = S < A ? S : 0;                                                                               \
      asm volatile("{\n.reg .f32 l<4>, h<4>;\nmov.b64 {l0, h0}, %1;\nmov.b64 {l1, h1}, %2;\nmov.b64 {l2, h2}, %3;\nmov.b64 {l3, h3}, %4;\n" \
                   "st.shared.v4.f32 [%0], {l0, l1, l2, l3};\nst.shared.v4.f32 [%0 + 512], {h0, h1, h2, h3};\n}"    \
                   ::"r"(sa), "l"(acc[S_][0]), "l"(acc[S_][1]), "l"(acc[S_][2]), "l"(NC > 3 ? acc[S_][NC > 3 ? 3 : 0] : 0ull) : "memory"); \
      _Pragma("unroll") for (int c = 0; c < NC; ++c) asm volatile("mov.b64 %0, 0;" : "=l"(acc[S_][c]));               \
    }                                                                                                                 \
    break;
      switch (slot) {
        PXZ_TAKE(0)
        PXZ_TAKE(1)
        PXZ_TAKE(2)
        PXZ_TAKE(3)
        PXZ_TAKE(4)
        default:
          PXZ_TAKE(5)
      }
#undef PXZ_TAKE
    }
    ++o;
    slot = slot + 1 == (uint32_t)A ? 0u : slot + 1;
    if (o < dh) e = lds_u32(endp + 4 * o);
    if (o - batch0 == (uint32_t)kTStripRows || o == dh) {
      __syncwarp();
      tma_horizontal<MODE, A == 6>(strip, batch0, o - batch0, dw, ht, dst, k);
      __syncwarp();
      batch0 = o;
      if (o == dh) break;
    }
  }
  // rows behind the last tap (weights exactly zero) are never read, but their boxes are part of the stream
  tfeed_release(f, tm, q);
  for (; boxes_read < nbox; ++boxes_read) {
    tfeed_wait(f);
    tfeed_release(f, tm, q);
  }
}

template <bool FUSED>
__global__ void __launch_bounds__(kTWarps * 32, PXZ_SHRINK_TMA_CTAS) k_shrink_tma(
    const __grid_constant__ CUtensorMap tm, Geom g, const pxz_block_desc* __restrict__ descs, const uint32_t* __restrict__ tabidx,
    const uint32_t* __restrict__ lists, uint32_t cap, const uint8_t* __restrict__ opaque_flags, uint8_t* __restrict__ payload,
    const AxisTab* __restrict__ tabs, uint32_t ntabs, const uint32_t* __restrict__ pool, uint32_t* counter, float rt_one,
    float rt_negzero) {
  extern __shared__ __align__(128) uint8_t s_tma[];
  __shared__ uint8_t s_noslide[kFastMaxTabs];  // table has no slide2 form
  uint8_t* wbase = s_tma + (threadIdx.x >> 5) * kTWarpBytes;
  float4* strip = reinterpret_cast<float4*>(wbase + kTStripOff);
  uint32_t* htab_smem = reinterpret_cast<uint32_t*>(wbase + kTHtabOff);
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(wbase);
  const uint32_t vtab = sbase + kTVtabOff;
  const uint32_t bars = sbase + kTBarOff;                 // kTSlots ring barriers, then the table barrier
  const uint32_t tbar = bars + 8u * kTSlots;
  const uint32_t lane = threadIdx.x & 31u;
  const TapK k = make_tapk(rt_one, rt_negzero);
  if (lane == 0) {
    for (int i = 0; i <= kTSlots; ++i) mbar_init(bars + 8u * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_proxy_async();
  __syncwarp();
  pdl_wait();
  pdl_trigger();
  for (uint32_t i = threadIdx.x; i < ntabs; i += kTWarps * 32) s_noslide[i] = tabs[i].s2words == 0 ? 1 : 0;
  __syncthreads();
  const uint32_t ntiles = g.cols * g.rows, total_warps = gridDim.x * kTWarps;
  constexpr int F = FUSED ? 2 : 0;
  TFeed f;
  f.ring = sbase + kTRingOff; f.bars = bars;
  f.inflight = 0; f.islot = 0; f.rslot = 0; f.rpar = 0;
  f.cx = f.cy = f.cnb = f.cpb = 0; f.nx = f.ny = f.nnb = f.npb = 0;
  uint32_t tpar = 0;                                      // phase parity of the table barrier
  uint32_t last_tx = 0xFFFFFFFFu, last_ty = 0xFFFFFFFFu;
  AxisTab ty{};
  HTab ht{};
  // does a block stream its source tile?  masked-out blocks (quadtree levels) and tiles whose vertical table has no
  // slide2 form (left to k_shrink_warp by the launcher) do not
  auto boxes_of = [&](const Tile& t, const pxz_block_desc& d, uint32_t ti) -> uint32_t {
    if (d.w == 0 || d.h == 0) return 0u;
    if (!(d.w == t.tw && d.h == t.th) && s_noslide[ti >> 16]) return 0u;
    return (t.th + kTBoxRows - 1) / kTBoxRows;
  };
  // P0: the tile being processed | P1: the next one (complete: the source stream runs on into it) | q: the one after
  TQueue q;
  q.descs = descs; q.tabidx = tabidx; q.opaque = opaque_flags; q.counter = counter; q.ntiles = ntiles;
  q.ord.init(lists, cap);
  q.drawing = true;
  tq_start(q);
  TDesc P0 = tq_finish(q);
  tq_start(q);
  TDesc P1 = tq_finish(q);
  {
    const Tile t = tile_of(g, P0.b);
    f.cx = t.x0; f.cy = t.y0; f.cnb = P0.valid ? boxes_of(t, P0.d, P0.ti) : 0u; f.cpb = 0;
  }
  while (P0.valid) {
    tq_start(q);
    f.nnb = 0; f.npb = 0;
    if (P1.valid) {
      const Tile tn = tile_of(g, P1.b);
      f.nx = tn.x0; f.ny = tn.y0; f.nnb = boxes_of(tn, P1.d, P1.ti);
    }
    const uint32_t b = P0.b, ti = P0.ti;
    const pxz_block_desc d = P0.d;
    const Tile t = tile_of(g, b);
    if (f.cnb != 0) {
      tfeed_pump(f, &tm);
      uint32_t* dst = reinterpret_cast<uint32_t*>(payload + d.offset);
      if (d.w == t.tw && d.h == t.th) {
        // block.rs:279-281: clone.  The block is contiguous in the payload (4-byte aligned only): words in lane order.
        for (uint32_t bx = 0; bx < f.cnb; ++bx) {
          const uint32_t box = tfeed_wait(f);
          const uint32_t nr = min((uint32_t)kTBoxRows, t.th - bx * kTBoxRows);
          uint32_t* o = dst + (size_t)bx * kTBoxRows * t.tw;
          if (t.tw == 64 && (d.offset & 15u) == 0 && nr == (uint32_t)kTBoxRows) {
            // 16 bytes per lane: two instructions per row pair
            uint4 v[kTBoxRows / 2];
#pragma unroll
            for (int i = 0; i < kTBoxRows / 2; ++i)
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[i].x), "=r"(v[i].y), "=r"(v[i].z), "=r"(v[i].w) : "r"(box + (i * 32 + lane) * 16));
#pragma unroll
            for (int i = 0; i < kTBoxRows / 2; ++i) reinterpret_cast<uint4*>(o)[i * 32 + lane] = v[i];
          } else if (t.tw == 64) {
#pragma unroll
            for (uint32_t i = 0; i < (uint32_t)kTBoxRows * 2; ++i)
              if (i < nr * 2) o[i * 32 + lane] = lds_u32(box + (i * 32 + lane) * 4);
          } else {
            for (uint32_t rr = 0; rr < nr; ++rr)
              for (uint32_t x = lane; x < t.tw; x += 32) o[rr * t.tw + x] = lds_u32(box + (rr * 64 + x) * 4);
          }
          tfeed_release(f, &tm, q);
        }
      } else {
        // stage the tile's tables when they change: one expect_tx for both, then the bulk copies
        const bool new_ty = (ti >> 16) != last_ty, new_tx = (ti & 0xFFFFu) != last_tx;
        if (new_ty | new_tx) {
          uint32_t staged = 0, hwords = 0;
          const uint32_t* hsrc = nullptr;
          if (new_ty) {
            ty = tabs[ti >> 16];
            last_ty = ti >> 16;
            staged += ty.s2words * 4;
          }
          if (new_tx) {
            const AxisTab tx = tabs[ti & 0xFFFFu];
            last_tx = ti & 0xFFFFu;
            ht.nb = tx.nb; ht.brows_total = tx.brows_total; ht.stride = tx.stride;
            const uint32_t off = d.w >= kBlockedFrom ? tx.boff : tx.off;
            hsrc = pool + off;
            hwords = ((d.w >= kBlockedFrom ? tx.bwords : 2 * d.w + d.w * tx.stride) + 3u) & ~3u;
            if (hwords <= (uint32_t)kTHtabWords && (off & 3u) == 0) {
              staged += hwords * 4;
              ht.tab = htab_smem;
            } else {
              ht.tab = hsrc;  // too large or unaligned: read through L1 / L2
              hwords = 0;
            }
          }
          if (staged) {
            fence_proxy_async();  // the previous tile's reads of the table buffers come before the async-proxy writes
            if (lane == 0) {
              mbar_expect_tx(tbar, staged);
              if (new_ty) bulk_load(vtab, pool + ty.s2off, ty.s2words * 4, tbar);
              if (hwords) bulk_load((uint32_t)__cvta_generic_to_shared(htab_smem), hsrc, hwords * 4, tbar);
            }
            mbar_wait(tbar, tpar);
            tpar ^= 1u;
          }
        }
        const bool opaque = P0.op != 0;
        const uint32_t slots = ty.slots;
        // dh <= slots: every output row keeps its accumulator (a zero-trimmed window never starts before an earlier
        // output's, so output o sits in slot o)
#define PXZ_TMA_TILE(M)                                                                                              \
  do {                                                                                                               \
    bool simple = true;                                                                                              \
    if (slots == 2 && d.h == 1) tma_shrink_tile_simple<M, 1, 2>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k);  \
    else if (slots == 2 && d.h == 2) tma_shrink_tile_simple<M, 2, 2>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k); \
    else if (slots == 4 && d.h <= 4) tma_shrink_tile_simple<M, 4, 4>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k); \
    else {                                                                                                           \
      simple = false;                                                                                                \
      if (slots == 2) tma_shrink_tile<M, 2>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k);                    \
      else if (slots == 4) tma_shrink_tile<M, 4>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k);               \
      else tma_shrink_tile<M, 6>(f, q, &tm, t.th, d.w, d.h, vtab, strip, ht, dst, k);                               \
    }                                                                                                                \
    if (simple) { /* the strip holds the whole block: one shared copy of the pass */                                 \
      __syncwarp();                                                                                                  \
      tma_horizontal<M, true>(strip, 0, d.h, d.w, ht, dst, k);                                                       \
      __syncwarp();                                                                                                  \
    }                                                                                                                \
  } while (0)
        if (opaque) PXZ_TMA_TILE(F);
        else PXZ_TMA_TILE(F | 1);
#undef PXZ_TMA_TILE
      }
    }
    P0 = P1;
    P1 = tq_finish(q);
    f.cx = f.nx; f.cy = f.ny; f.cnb = f.nnb; f.cpb = f.npb;
    f.nnb = 0; f.npb = 0;
  }
  // the last warp out puts the draw counts (one 64-bit word) and the exit count back for the next launch on this stream
  if (lane == 0) {
    if (atomicAdd(counter + 2, 1u) == total_warps - 1) {
      counter[0] = 0u;
      counter[1] = 0u;
      counter[2] = 0u;
    }
  }
}
