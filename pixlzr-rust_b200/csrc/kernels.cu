// kernels.cu — hand-written sm_100a kernels of the pixlzr hot path.
//
//   k_analyze_mad_rgba   Oklab mean-absolute-deviation per tile, fast arithmetic (operations.rs:26-126)
//   k_analyze_mad_any    same, any channel count / alignment
//   k_mad_exact          reference-order (sequential f32, no fma, glibc cbrtf) recomputation of the
//                        tiles whose fast value lies in the guard band of a level threshold
//   k_analyze_sobel      directional Sobel metric, integer exact (operations.rs:192-259)
//   k_minmax             global min / -max of the raw values (normalise extension)
//   k_plan               value -> parse_value -> level -> dims -> payload offsets (single-pass scan)
//                        (operations.rs:128-156)
//   k_resample           per-block separable resample, image-crate order (block.rs:273-290):
//                        image tiles -> packed payload (shrink) or payload -> image tiles (expand+paste)
//   k_block_error        per-block squared error and largest difference of two images (integer, exact)
//   k_bucket_sum         block errors summed per strategy bucket of the stored block value (strategy measure)
//   k_rd_levels          forced levels of one error pass of the rate-distortion curve
//   k_rd_events          per block, the factors at which its dims change and what that changes (rate-distortion curve)
//   k_rd_gather / k_rd_compact   sorted events -> scan input -> curve points (around CUB's radix sort and scan)
//   k_rdo_hull           per block, the lower convex hull of its (bytes, error) over every level pair (optimised encode)
//   k_rdo_gather / k_rdo_points  events sorted by rate -> scan input -> curve points (around CUB's merge sort and scan)
//   k_rdo_levels         per block, the levels of one point of the optimised curve
//
// Nothing here is a dense contraction, so no tensor cores: the kernels are HBM / FP32-pipe work with
// 16-byte coalesced loads, shared-memory staging and warp-shuffle reductions (DESIGN.md).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <cub/device/device_merge_sort.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "pxz_internal.h"

namespace pxz {

// ------------------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------------------
__constant__ float c_srgb_lut[256] = {
#include "srgb_lut.inc"
};

// palette 0.7.6 Oklab matrices (linear sRGB -> LMS, LMS' -> Lab), f32
#define M1_00 0.4122214708f
#define M1_01 0.5363325363f
#define M1_02 0.0514459929f
#define M1_10 0.2119034982f
#define M1_11 0.6806995451f
#define M1_12 0.1073969566f
#define M1_20 0.0883024619f
#define M1_21 0.2817188376f
#define M1_22 0.6299787005f
#define M2_00 0.2104542553f
#define M2_01 0.7936177850f
#define M2_02 (-0.0040720468f)
#define M2_10 1.9779984951f
#define M2_11 (-2.4285922050f)
#define M2_12 0.4505937099f
#define M2_20 0.0259040371f
#define M2_21 0.7827717662f
#define M2_22 (-0.8086757660f)

constexpr float kInv255 = (float)(1.0 / 255.0);
constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// Programmatic dependent launch: a kernel launched with launch_pdl() may become resident while the kernel before it
// on the stream is still draining.  pdl_wait() blocks until that kernel has completed and its writes are visible —
// every kernel calls it before it touches global memory that another kernel writes or reads — and pdl_trigger() lets
// the kernel behind this one start being scheduled as soon as SM resources free up.  Without the launch attribute
// both are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// x >= 0.  cube root through the SFU: 2^(log2(x)/3); ~4e-7 relative error (fast path only).
__device__ __forceinline__ float cbrt_fast(float x) {
  float l, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(x));
  l *= 0.333333343f;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(l));
  return r;
}

// u8 -> f32 without the conversion pipe: splice the byte into the mantissa of 2^23.
template <int BYTE>
__device__ __forceinline__ float byte_to_float(uint32_t word) {
  uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7440 | BYTE);  // {b, 0, 0, 0x4B}
  return __uint_as_float(bits) - 8388608.0f;
}

// ---- packed f32x2 arithmetic (sm_100a FFMA2: two f32 lanes per issue slot) ---------------------------------------
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpk2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ float lo2(u64 v) { float a, b; unpk2(v, a, b); return a; }
__device__ __forceinline__ float hi2(u64 v) { float a, b; unpk2(v, a, b); return b; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
  u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// tile geometry of block index b
struct Tile {
  uint32_t x0, y0, tw, th;
};
__device__ __forceinline__ Tile tile_of(const Geom& g, uint32_t b) {
  Tile t;
  uint32_t by = b / g.cols, bx = b - by * g.cols;
  uint32_t base = 0;
  if (g.nimg > 1) {  // stacked batch: block row -> (image, block row of that image)
    const uint32_t im = by / g.rows_img;
    by -= im * g.rows_img;
    base = im * g.img_rows;
  }
  t.x0 = bx * g.bw;
  t.tw = min(g.bw, g.W - t.x0);  // split.rs:18-19
  t.th = min(g.bh, g.H - by * g.bh);
  t.y0 = base + by * g.bh;
  return t;
}

// ------------------------------------------------------------------------------------------------
// Oklab MAD, fast path.
// One group of G threads per tile, 256/G tiles per CTA iteration, persistent CTAs (grid-stride over
// tiles) so the 32 KB bank-conflict-free sRGB table is built once per CTA.  Each thread keeps the
// cube-rooted LMS of its <= 16 pixels in registers, so pass 2 (|c - mean|) does not redo the cube
// roots the reference computes twice (operations.rs:75-84 / 111-119).
// ------------------------------------------------------------------------------------------------
struct OklabFast {
  float l, m, s;  // cube-rooted LMS
};

__device__ __forceinline__ OklabFast lms_fast(uint32_t px, const float* lut_lane) {
  // lut_lane = s_lut + lane; entry v at lut_lane[v * 32] -> bank == lane, conflict free
  const float r = lut_lane[(px & 0xFFu) << 5];
  const float g = lut_lane[((px >> 8) & 0xFFu) << 5];
  const float b = lut_lane[((px >> 16) & 0xFFu) << 5];
  OklabFast o;
  o.l = cbrt_fast(fmaf(M1_02, b, fmaf(M1_01, g, M1_00 * r)));
  o.m = cbrt_fast(fmaf(M1_12, b, fmaf(M1_11, g, M1_10 * r)));
  o.s = cbrt_fast(fmaf(M1_22, b, fmaf(M1_21, g, M1_20 * r)));
  return o;
}

// cube-rooted LMS of one packed RGBA pixel.  lut_lane_addr = shared-space byte address of s_lut[lane];
// entry v lives at +v*128 bytes, so the bank is always the lane: no conflicts for arbitrary pixel data.
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float r;
  asm("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr));
  return r;
}
__device__ __forceinline__ OklabFast lms_fast_addr(uint32_t px, uint32_t lut_lane_addr) {
  const float r = lds_f32(lut_lane_addr + (__byte_perm(px, 0, 0x4440) << 7));
  const float g = lds_f32(lut_lane_addr + (__byte_perm(px, 0, 0x4441) << 7));
  const float b = lds_f32(lut_lane_addr + (__byte_perm(px, 0, 0x4442) << 7));
  OklabFast o;
  o.l = cbrt_fast(fmaf(M1_02, b, fmaf(M1_01, g, M1_00 * r)));
  o.m = cbrt_fast(fmaf(M1_12, b, fmaf(M1_11, g, M1_10 * r)));
  o.s = cbrt_fast(fmaf(M1_22, b, fmaf(M1_21, g, M1_20 * r)));
  return o;
}

// two pixels at once: the 3x3 products run as f32x2 FMAs (each lane is the same IEEE fma as the scalar form, so the
// values — and the guard band derived for them — do not change; only the issue slots halve)
__device__ __forceinline__ void lms_fast_pair(uint32_t px0, uint32_t px1, uint32_t lut_lane_addr, OklabFast& o0, OklabFast& o1) {
  const u64 r = pk2(lds_f32(lut_lane_addr + (__byte_perm(px0, 0, 0x4440) << 7)), lds_f32(lut_lane_addr + (__byte_perm(px1, 0, 0x4440) << 7)));
  const u64 g = pk2(lds_f32(lut_lane_addr + (__byte_perm(px0, 0, 0x4441) << 7)), lds_f32(lut_lane_addr + (__byte_perm(px1, 0, 0x4441) << 7)));
  const u64 b = pk2(lds_f32(lut_lane_addr + (__byte_perm(px0, 0, 0x4442) << 7)), lds_f32(lut_lane_addr + (__byte_perm(px1, 0, 0x4442) << 7)));
#define PXZ_ROW2(c0, c1, c2) fma2(pk2(c2, c2), b, fma2(pk2(c1, c1), g, mul2(pk2(c0, c0), r)))
  const u64 l = PXZ_ROW2(M1_00, M1_01, M1_02), m = PXZ_ROW2(M1_10, M1_11, M1_12), q = PXZ_ROW2(M1_20, M1_21, M1_22);
#undef PXZ_ROW2
  o0.l = cbrt_fast(lo2(l)); o1.l = cbrt_fast(hi2(l));
  o0.m = cbrt_fast(lo2(m)); o1.m = cbrt_fast(hi2(m));
  o0.s = cbrt_fast(lo2(q)); o1.s = cbrt_fast(hi2(q));
}
// the same with the results left as pairs (l', m', s' of the two pixels)
__device__ __forceinline__ u64 cbrt_fast2(u64 x) {
  float a, b, la, lb;
  unpk2(x, a, b);
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(la) : "f"(a));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lb) : "f"(b));
  const u64 t = mul2(pk2(la, lb), pk2(0.333333343f, 0.333333343f));
  unpk2(t, la, lb);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(a) : "f"(la));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(b) : "f"(lb));
  return pk2(a, b);
}
struct OklabFast2 {
  u64 l, m, s;
};
#ifndef PXZ_MAD_LUT_STRIDE
#define PXZ_MAD_LUT_STRIDE 64  // floats per table entry: 64 = one byte permute builds the whole offset, 32 = half the shared memory
#endif
constexpr int kMadLutStride = PXZ_MAD_LUT_STRIDE;
// offset of entry `byte BYTE of px` in this lane's column of the table.  With 256-byte entries the offset is
// {lane * 4, value, 0, 0} as bytes: one PRMT, and the table base rides in a uniform register (LDS [R + UR]).
template <int BYTE>
__device__ __forceinline__ float lut_fetch(uint32_t px, uint32_t lut_base, uint32_t lane4) {
  if (kMadLutStride == 64) return lds_f32(lut_base + __byte_perm(px, lane4, 0x7704 | (BYTE << 4)));
  return lds_f32(lut_base + lane4 + (__byte_perm(px, 0, 0x4440 | BYTE) << 7));
}
__device__ __forceinline__ OklabFast2 lms_fast_pair2(uint32_t px0, uint32_t px1, uint32_t lut_base, uint32_t lane4) {
  const u64 r = pk2(lut_fetch<0>(px0, lut_base, lane4), lut_fetch<0>(px1, lut_base, lane4));
  const u64 g = pk2(lut_fetch<1>(px0, lut_base, lane4), lut_fetch<1>(px1, lut_base, lane4));
  const u64 b = pk2(lut_fetch<2>(px0, lut_base, lane4), lut_fetch<2>(px1, lut_base, lane4));
#define PXZ_ROW2(c0, c1, c2) fma2(pk2(c2, c2), b, fma2(pk2(c1, c1), g, mul2(pk2(c0, c0), r)))
  OklabFast2 o;
  o.l = cbrt_fast2(PXZ_ROW2(M1_00, M1_01, M1_02));
  o.m = cbrt_fast2(PXZ_ROW2(M1_10, M1_11, M1_12));
  o.s = cbrt_fast2(PXZ_ROW2(M1_20, M1_21, M1_22));
#undef PXZ_ROW2
  return o;
}

#ifndef PXZ_MAD_MINBLOCKS
#define PXZ_MAD_MINBLOCKS 2
#endif
template <int G, int QPT>
__global__ void __launch_bounds__(kThreads, PXZ_MAD_MINBLOCKS) k_analyze_mad_rgba(const uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                                  float* __restrict__ vx, uint8_t* __restrict__ opaque,
                                                                  uint32_t* __restrict__ zero_word) {
  constexpr int TPC = kThreads / G;  // tiles per CTA iteration
  constexpr int WPG = G / 32;        // warps per group
  extern __shared__ float s_lut[];   // [256][kMadLutStride], columns 0..31 used: bank == lane for any pixel data
  __shared__ float s_r1[2][kThreads / 32][4];
  __shared__ float s_r2[2][kThreads / 32];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int grp = tid / G, gt = tid % G, gwarp0 = grp * WPG;
  for (int i = tid; i < 256 * 32; i += kThreads) s_lut[(i >> 5) * kMadLutStride + (i & 31)] = c_srgb_lut[i >> 5];
  __syncthreads();
  const uint32_t lut_base = (uint32_t)__cvta_generic_to_shared(s_lut), lane4 = (uint32_t)lane * 4u;

  const uint32_t ntiles = g.cols * g.rows;
  const uint32_t qpr = g.bw >> 2;  // quads (4 px = 16 B) per full tile row
  // this thread's quads: the (row, column) mapping does not depend on the tile
  uint32_t qrc[QPT];   // row << 16 | first column
  uint32_t qoff[QPT];  // byte offset inside the tile ((bh - 1) * pitch + bw * 4 < 2^32, checked by the launcher)
  bool all_in = true;  // every quad of this thread lies inside a FULL tile
#pragma unroll
  for (int j = 0; j < QPT; ++j) {
    const uint32_t q = gt + j * G;
    const uint32_t row = q / qpr, col = (q - row * qpr) * 4;
    qrc[j] = (row << 16) | col;
    qoff[j] = (uint32_t)((size_t)row * pitch + (size_t)col * 4);
    all_in = all_in && (row < g.bh);
  }
#define QROW(j) (qrc[j] >> 16)
#define QCOL(j) (qrc[j] & 0xFFFFu)
  const bool cta_all_in = __syncthreads_and(all_in) != 0;
  // everything above (the 32 KB table, the quad mapping) may run while the previous kernel on the stream drains
  pdl_wait();
  pdl_trigger();
  if (zero_word != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero_word = 0u;  // the guard-band list counter of the next kernel

  auto load_tile = [&](uint32_t tile, uint4(&v)[QPT]) {
    if (tile < ntiles) {
      const Tile t = tile_of(g, tile);
      const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
#pragma unroll
      for (int j = 0; j < QPT; ++j)
        v[j] = (QROW(j) < t.th && QCOL(j) < t.tw) ? ldg_nc_v4(base + qoff[j]) : make_uint4(0, 0, 0, 0);
    }
  };

  // one tile; MASK = false when every pixel of every thread is inside the tile (interior tiles)
  auto process = [&](auto mask_tag, const Tile& t, bool valid, uint4(&cur)[QPT], uint4(&nxt)[QPT], uint32_t next_tile,
                     uint32_t tile, int buf) {
    constexpr bool MASK = decltype(mask_tag)::value;
    OklabFast2 c[QPT * 2];  // pixel pairs
    u64 sl2 = 0ull, sm2 = 0ull, ss2 = 0ull;
    uint32_t asum = 0;  // integer sum of the alpha bytes (exact)
#pragma unroll
    for (int j = 0; j < QPT; ++j) {
      const bool inq = !MASK || (valid && QROW(j) < t.th && QCOL(j) < t.tw);
      const uint32_t w4[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
#pragma unroll
      for (int k = 0; k < 4; k += 2) {
        OklabFast2 o = lms_fast_pair2(w4[k], w4[k + 1], lut_base, lane4);
        if (MASK && !inq) { o.l = 0ull; o.m = 0ull; o.s = 0ull; }
        c[j * 2 + (k >> 1)] = o;
        sl2 = add2(sl2, o.l); sm2 = add2(sm2, o.m); ss2 = add2(ss2, o.s);
        asum = __dp4a(w4[k], 0x01000000u, asum);  // out-of-tile quads were loaded as zeros
        asum = __dp4a(w4[k + 1], 0x01000000u, asum);
      }
#ifdef PXZ_MAD_SCHED_FENCE
      asm volatile("" ::: "memory");  // keep the quads' LDS / MUFU bursts apart (MIO queue pressure)
#endif
    }
    // the source quads are dead now: fetch the next tile while pass 2 and the reductions run
#pragma unroll
    for (int j = 0; j < QPT; ++j) nxt[j] = make_uint4(0, 0, 0, 0);
    load_tile(next_tile, nxt);
    // ---- group reduction 1 ----
    float sl = lo2(sl2) + hi2(sl2), sm = lo2(sm2) + hi2(sm2), ss = lo2(ss2) + hi2(ss2);
    // the alpha bytes are summed as integers: one REDUX instead of five shuffle / add steps
    float sa = (float)__reduce_add_sync(0xffffffffu, asum);
    sl = warp_sum(sl); sm = warp_sum(sm); ss = warp_sum(ss);
    if (WPG > 1) {
      if (lane == 0) { s_r1[buf][warp][0] = sl; s_r1[buf][warp][1] = sm; s_r1[buf][warp][2] = ss; s_r1[buf][warp][3] = sa; }
      __syncthreads();
      sl = sm = ss = sa = 0.f;
#pragma unroll
      for (int w = 0; w < WPG; ++w) {
        sl += s_r1[buf][gwarp0 + w][0]; sm += s_r1[buf][gwarp0 + w][1];
        ss += s_r1[buf][gwarp0 + w][2]; sa += s_r1[buf][gwarp0 + w][3];
      }
    }
    const float count = (float)(t.tw * t.th);
    const float inv = valid ? 1.0f / count : 0.f;
    // byte sums of <= 4096 pixels are exact in f32: the tile is opaque iff the sum is 255 * count
    const bool is_opaque = (sa == 255.0f * count);
    sl *= inv; sm *= inv; ss *= inv;
    const float mean_alpha = sa * inv * kInv255;
    // the Lab transform is linear: mean(Lab) = M2 * mean(l', m', s')
    const float nL = -(M2_00 * sl + M2_01 * sm + M2_02 * ss);
    const float nA = -(M2_10 * sl + M2_11 * sm + M2_12 * ss);
    const float nB = -(M2_20 * sl + M2_21 * sm + M2_22 * ss);
    float d = 0.f;
    float dp[4] = {0.f, 0.f, 0.f, 0.f};
    const u64 nL2 = pk2(nL, nL), nA2 = pk2(nA, nA), nB2 = pk2(nB, nB);
#pragma unroll
    for (int i = 0; i < QPT * 4; i += 2) {
      const u64 ol = c[i >> 1].l, om = c[i >> 1].m, os = c[i >> 1].s;
#define PXZ_ROW2(c0, c1, c2, bias) fma2(pk2(c2, c2), os, fma2(pk2(c1, c1), om, fma2(pk2(c0, c0), ol, bias)))
      const u64 dL2 = PXZ_ROW2(M2_00, M2_01, M2_02, nL2), dA2 = PXZ_ROW2(M2_10, M2_11, M2_12, nA2), dB2 = PXZ_ROW2(M2_20, M2_21, M2_22, nB2);
#undef PXZ_ROW2
      const float e0 = (fabsf(lo2(dA2)) + fabsf(lo2(dB2))) + fabsf(lo2(dL2));
      const float e1 = (fabsf(hi2(dA2)) + fabsf(hi2(dB2))) + fabsf(hi2(dL2));
      if (MASK) {
        const int j = i >> 2, k = i & 3;
        const bool rowin = valid && QROW(j) < t.th;
        d += (rowin && (QCOL(j) + k) < t.tw) ? e0 : 0.f;
        d += (rowin && (QCOL(j) + k + 1) < t.tw) ? e1 : 0.f;
      } else {
        dp[i & 3] += e0;
        dp[(i + 1) & 3] += e1;
      }
    }
    if (!MASK) d = (dp[0] + dp[1]) + (dp[2] + dp[3]);
    if (!is_opaque) {
      // rare: per-pixel alpha deviations; the quads are re-read (L1/L2 hot) instead of being kept in registers
      if (valid) {
        const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
#pragma unroll
        for (int j = 0; j < QPT; ++j) {
          if (QROW(j) < t.th && QCOL(j) < t.tw) {
            const uint4 q = ldg_nc_v4(base + qoff[j]);
            d += fabsf(byte_to_float<3>(q.x) * kInv255 - mean_alpha) + fabsf(byte_to_float<3>(q.y) * kInv255 - mean_alpha);
            d += fabsf(byte_to_float<3>(q.z) * kInv255 - mean_alpha) + fabsf(byte_to_float<3>(q.w) * kInv255 - mean_alpha);
          }
        }
      }
    }
    d = warp_sum(d);
    if (WPG > 1) {
      if (lane == 0) s_r2[buf][warp] = d;
      __syncthreads();
      d = 0.f;
#pragma unroll
      for (int w = 0; w < WPG; ++w) d += s_r2[buf][gwarp0 + w];
    }
    if (valid && gt == 0) {
      vx[tile] = d * inv;
      opaque[tile] = (uint8_t)(is_opaque ? 1 : 0);
    }
  };

  uint4 cur[QPT], nxt[QPT];
  uint32_t base_tile = blockIdx.x * TPC;
  uint32_t it = 0;
#pragma unroll
  for (int j = 0; j < QPT; ++j) cur[j] = make_uint4(0, 0, 0, 0);
  load_tile(base_tile + grp, cur);
  for (; base_tile < ntiles; base_tile += gridDim.x * TPC, ++it) {
    const uint32_t tile = base_tile + grp;
    const bool valid = tile < ntiles;
    const Tile t = valid ? tile_of(g, tile) : Tile{0, 0, 0, 0};
    const uint32_t next_tile = tile + gridDim.x * TPC;
    // interior tiles of a fully populated CTA skip every bounds predicate (CTA-uniform choice when TPC == 1)
    const bool full = cta_all_in && valid && t.tw == g.bw && t.th == g.bh;
    const bool full_all = (TPC == 1) ? full : (__syncthreads_and(full) != 0);
    if (full_all) process(std::false_type{}, t, valid, cur, nxt, next_tile, tile, it & 1);
    else process(std::true_type{}, t, valid, cur, nxt, next_tile, tile, it & 1);
#pragma unroll
    for (int j = 0; j < QPT; ++j) cur[j] = nxt[j];
  }
}
#undef QROW
#undef QCOL

// Any channel count / alignment / tile size: one CTA per tile (grid-stride), byte loads, same fast
// arithmetic.  The first 16 pixels of every thread stay in registers; a tile with more than
// 16 * 256 pixels recomputes the rest in pass 2.
template <int C>
__global__ void __launch_bounds__(kThreads) k_analyze_mad_any(const uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                              float* __restrict__ vx, uint8_t* __restrict__ opaque,
                                                              uint32_t* __restrict__ zero_word) {
  pdl_wait();
  pdl_trigger();
  if (zero_word != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero_word = 0u;
  extern __shared__ float s_lut[];
  __shared__ float s_r1[kThreads / 32][4];
  __shared__ float s_r2[kThreads / 32];
  __shared__ int s_opq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 256 * 32; i += kThreads) s_lut[i] = c_srgb_lut[i >> 5];
  __syncthreads();
  const float* lut_lane = s_lut + lane;
  constexpr int KEEP = 16;
  const uint32_t ntiles = g.cols * g.rows;
  for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const Tile t = tile_of(g, tile);
    const uint32_t npx = t.tw * t.th;
    const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
    if (tid == 0) s_opq = 1;
    bool all255 = true;
    auto fetch = [&](uint32_t idx, float& a) -> OklabFast {
      uint32_t y = idx / t.tw, x = idx - y * t.tw;
      const uint8_t* p = base + (size_t)y * pitch + (size_t)x * C;
      uint32_t px = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
      if (C == 4) {
        a = (float)p[3] * kInv255;
        all255 = all255 && (p[3] == 255);
      } else {
        a = 0.f;
      }
      return lms_fast(px, lut_lane);
    };
    OklabFast c[KEEP];
    float al[KEEP];
    float sl = 0.f, sm = 0.f, ss = 0.f, sa = 0.f;
#pragma unroll
    for (int k = 0; k < KEEP; ++k) {
      uint32_t idx = tid + k * kThreads;
      if (idx < npx) {
        c[k] = fetch(idx, al[k]);
        sl += c[k].l; sm += c[k].m; ss += c[k].s; sa += al[k];
      }
    }
    for (uint32_t idx = tid + KEEP * kThreads; idx < npx; idx += kThreads) {
      float a;
      OklabFast o = fetch(idx, a);
      sl += o.l; sm += o.m; ss += o.s; sa += a;
    }
    sl = warp_sum(sl); sm = warp_sum(sm); ss = warp_sum(ss); sa = warp_sum(sa);
    if (lane == 0) { s_r1[warp][0] = sl; s_r1[warp][1] = sm; s_r1[warp][2] = ss; s_r1[warp][3] = sa; }
    if (C == 4 && !all255) s_opq = 0;  // benign race: everyone writes the same value
    __syncthreads();
    sl = sm = ss = sa = 0.f;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) { sl += s_r1[w][0]; sm += s_r1[w][1]; ss += s_r1[w][2]; sa += s_r1[w][3]; }
    const float inv = 1.0f / (float)npx;
    sl *= inv; sm *= inv; ss *= inv; sa *= inv;
    const float nL = -(M2_00 * sl + M2_01 * sm + M2_02 * ss);
    const float nA = -(M2_10 * sl + M2_11 * sm + M2_12 * ss);
    const float nB = -(M2_20 * sl + M2_21 * sm + M2_22 * ss);
    auto dev = [&](const OklabFast& o, float a) -> float {
      const float dL = fmaf(M2_02, o.s, fmaf(M2_01, o.m, fmaf(M2_00, o.l, nL)));
      const float dA = fmaf(M2_12, o.s, fmaf(M2_11, o.m, fmaf(M2_10, o.l, nA)));
      const float dB = fmaf(M2_22, o.s, fmaf(M2_21, o.m, fmaf(M2_20, o.l, nB)));
      float e = (fabsf(dA) + fabsf(dB)) + fabsf(dL);
      if (C == 4) e += fabsf(a - sa);
      return e;
    };
    float d = 0.f;
#pragma unroll
    for (int k = 0; k < KEEP; ++k) {
      uint32_t idx = tid + k * kThreads;
      if (idx < npx) d += dev(c[k], al[k]);
    }
    for (uint32_t idx = tid + KEEP * kThreads; idx < npx; idx += kThreads) {
      float a;
      OklabFast o = fetch(idx, a);
      d += dev(o, a);
    }
    d = warp_sum(d);
    if (lane == 0) s_r2[warp] = d;
    __syncthreads();
    if (tid == 0) {
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) tot += s_r2[w];
      vx[tile] = tot * inv;
      opaque[tile] = (uint8_t)((C == 3 || s_opq) ? 1 : 0);
    }
    __syncthreads();  // s_r1 / s_r2 reuse
  }
}

// ------------------------------------------------------------------------------------------------
// value -> level (operations.rs:128-148), shared by the guard-band test and the plan kernel
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float parse_value_dev(float value) {  // operations.rs:128-138
  if (!signbit(value)) return value;
  float v = __fadd_rn(1.0f, value);
  v = (v != v) ? 0.0f : (v > 0.0f ? v : 0.0f);  // f32::max(NaN, 0) = 0; -0 -> +0
  return v;
}

// k such that level = 2^-k; kLevelOnePixel when level * n < 1 for every n < 2^40.
__device__ __forceinline__ uint32_t level_k(float pv, const LevelThresholds& thr) {
  if (pv != pv) return 0;           // NaN.min(0) = 0 -> exp2(0) = 1
  if (pv >= thr.thr[0]) return 0;   // includes +inf
  if (!(pv >= thr.thr[kThresholds - 1])) return kLevelOnePixel;  // 0, denormals, tiny
  // thr is decreasing in k; the answer is within one of the binade estimate
  int e = (int)((__float_as_uint(pv) >> 23) & 0xFF) - 127;  // floor(log2 pv) for normals
  int k = -e - 1;                                             // candidate: round(log2) in {e, e+1}
  if (k < 0) k = 0;
  if (k > kThresholds - 1) k = kThresholds - 1;
  while (k > 0 && pv >= thr.thr[k - 1]) --k;
  while (k < kThresholds - 1 && !(pv >= thr.thr[k])) ++k;
  return (uint32_t)k;
}

__device__ __forceinline__ uint32_t scaled_dim(uint32_t n, uint32_t k) {  // operations.rs:150-151
  if (k >= 32) return 1;
  uint32_t d = (uint32_t)(((uint64_t)n + ((1ull << k) - 1)) >> k);
  return d < 1 ? 1 : d;
}

// a * b as the reference's host computes it: a NaN operand comes back as it is (x86 returns the first NaN operand,
// sign included), where the GPU would produce the canonical positive NaN.  The sign matters: the Sobel metric of a
// block without interior pixels is 0/0 = the *negative* default NaN, which parse_value sends through `1 + v` to 0
// (operations.rs:128-138), i.e. to a 1-pixel block, while a positive NaN keeps the block at full size.
__device__ __forceinline__ float mul_host(float a, float b) {
  if (a != a) return a;
  if (b != b) return b;
  return __fmul_rn(a, b);
}

__device__ __forceinline__ void map_values(const ValueMap& vm, const float* minmax, float rx, float ry, float& v0,
                                           float& v1) {
  if (vm.normalise) {
    // extension: v' = (v - min) / (max - min), 0 when the range is empty
    const float mnx = minmax[0], mxx = -minmax[1];
    const float rgx = __fsub_rn(mxx, mnx);
    rx = (rgx > 0.f) ? (rx == rx ? __fdiv_rn(__fsub_rn(rx, mnx), rgx) : rx) : 0.f;  // a NaN value stays the NaN it is (host arithmetic)
    if (vm.mode == 2) {
      const float mny = minmax[2], mxy = -minmax[3];
      const float rgy = __fsub_rn(mxy, mny);
      ry = (rgy > 0.f) ? (ry == ry ? __fdiv_rn(__fsub_rn(ry, mny), rgy) : ry) : 0.f;
    }
  }
  if (vm.mode == 0) {
    v0 = v1 = mul_host(mul_host(rx, vm.factor), 10.0f);  // pixlzr.rs:162
  } else if (vm.mode == 1) {
    v0 = v1 = rx;  // process/mod.rs:110
  } else {
    v0 = mul_host(rx, vm.factor);  // pixlzr.rs:199
    v1 = mul_host(ry, vm.factor);
  }
}

// ------------------------------------------------------------------------------------------------
// Oklab MAD, reference-order path: plain IEEE f32 evaluated exactly as the reference does —
// no fma, pre-2.41 glibc cbrtf (double polynomial + one Halley step), sequential running sums in
// block scan order — so the value is bit-identical to the CPU result.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float cbrtf_ref(float x) {  // x >= 0, finite
  if (x == 0.0f) return 0.0f;
  int xe;
  float xm;
  const uint32_t xb = __float_as_uint(x);
  if (xb >= 0x00800000u && xb < 0x7F800000u) {  // normal: frexp is a field split (mantissa in [0.5, 1))
    xe = (int)(xb >> 23) - 126;
    xm = __uint_as_float((xb & 0x007FFFFFu) | 0x3F000000u);
  } else {
    xm = frexpf(x, &xe);
  }
  const double dxm = (double)xm;
  const float u = __double2float_rn(__dadd_rn(
      0.492659620528969547, __dmul_rn(__dsub_rn(0.697570460207922770, __dmul_rn(0.191502161678719066, dxm)), dxm)));
  const float t2 = __fmul_rn(__fmul_rn(u, u), u);
  const double dt2 = (double)t2;
  const int rem = xe % 3;  // C truncation, as glibc
  const double factor = rem == -2 ? 0.62996052494743658238361
                      : rem == -1 ? 0.79370052598409973737585
                      : rem == 0  ? 1.0
                      : rem == 1  ? 1.2599210498948731647672
                                  : 1.5874010519681994747517;
  const double num = __dmul_rn((double)u, __dadd_rn(dt2, __dmul_rn(2.0, dxm)));
  const double den = __dadd_rn(__dmul_rn(2.0, dt2), dxm);
  const float ym = __double2float_rn(__dmul_rn(__ddiv_rn(num, den), factor));
  // ldexpf(ym, xe / 3): ym is in [0.5, 2) and |xe / 3| <= 50, so the product with the power of two is exact
  return __fmul_rn(ym, __uint_as_float((uint32_t)(xe / 3 + 127) << 23));
}

__device__ __forceinline__ void oklab_ref(const float* lut, uint32_t r8, uint32_t g8, uint32_t b8, float& L, float& A,
                                          float& B) {
  const float r = lut[r8], g = lut[g8], b = lut[b8];
  const float l = __fadd_rn(__fadd_rn(__fmul_rn(M1_00, r), __fmul_rn(M1_01, g)), __fmul_rn(M1_02, b));
  const float m = __fadd_rn(__fadd_rn(__fmul_rn(M1_10, r), __fmul_rn(M1_11, g)), __fmul_rn(M1_12, b));
  const float s = __fadd_rn(__fadd_rn(__fmul_rn(M1_20, r), __fmul_rn(M1_21, g)), __fmul_rn(M1_22, b));
  const float l_ = cbrtf_ref(l), m_ = cbrtf_ref(m), s_ = cbrtf_ref(s);
  // `a*x + b*y - c*z` in the reference's source; the negative constants are written as subtractions
  L = __fsub_rn(__fadd_rn(__fmul_rn(M2_00, l_), __fmul_rn(M2_01, m_)), __fmul_rn(0.0040720468f, s_));
  A = __fadd_rn(__fsub_rn(__fmul_rn(M2_10, l_), __fmul_rn(2.4285922050f, m_)), __fmul_rn(M2_12, s_));
  B = __fsub_rn(__fadd_rn(__fmul_rn(M2_20, l_), __fmul_rn(M2_21, m_)), __fmul_rn(0.8086757660f, s_));
}

#ifndef PXZ_EXACT_PIPELINE
#define PXZ_EXACT_PIPELINE 1
#endif
constexpr int kExactChunk = 4096;             // pixels staged per pass
constexpr int kExactStride = kExactChunk + 4; // +4 floats: 16-byte aligned rows, and the 4 channel lanes hit different banks

// the sequential f32 sum of the reference over p[0..n), continuing from s; p is 16-byte aligned.  Loads run one batch
// of 16 ahead of the dependent adds.
__device__ __forceinline__ float chain_sum(const float* __restrict__ p, uint32_t n, float s) {
  const float4* p4 = reinterpret_cast<const float4*>(p);
  const uint32_t nb = n >> 4;
#define PXZ_ADD16(q0, q1, q2, q3)                                                                       \
  s = __fadd_rn(s, q0.x); s = __fadd_rn(s, q0.y); s = __fadd_rn(s, q0.z); s = __fadd_rn(s, q0.w);        \
  s = __fadd_rn(s, q1.x); s = __fadd_rn(s, q1.y); s = __fadd_rn(s, q1.z); s = __fadd_rn(s, q1.w);        \
  s = __fadd_rn(s, q2.x); s = __fadd_rn(s, q2.y); s = __fadd_rn(s, q2.z); s = __fadd_rn(s, q2.w);        \
  s = __fadd_rn(s, q3.x); s = __fadd_rn(s, q3.y); s = __fadd_rn(s, q3.z); s = __fadd_rn(s, q3.w);
  if (nb) {
    float4 a0 = p4[0], a1 = p4[1], a2 = p4[2], a3 = p4[3];
    for (uint32_t bi = 1; bi < nb; ++bi) {
      const float4 c0 = p4[4 * bi], c1 = p4[4 * bi + 1], c2 = p4[4 * bi + 2], c3 = p4[4 * bi + 3];
      PXZ_ADD16(a0, a1, a2, a3)
      a0 = c0; a1 = c1; a2 = c2; a3 = c3;
    }
    PXZ_ADD16(a0, a1, a2, a3)
  }
#undef PXZ_ADD16
  for (uint32_t i = nb << 4; i < n; ++i) s = __fadd_rn(s, p[i]);
  return s;
}

template <int C>
__device__ __forceinline__ void stage_exact_px(const uint8_t* __restrict__ base, size_t pitch, const Tile& t, uint32_t idx, uint32_t slot,
                                               float* s_val, const float* s_lut256) {
  const uint32_t y = idx / t.tw, x = idx - y * t.tw;
  const uint8_t* p = base + (size_t)y * pitch + (size_t)x * C;
  float L, A, B;
  oklab_ref(s_lut256, p[0], p[1], p[2], L, A, B);
  s_val[0 * kExactStride + slot] = A;
  s_val[1 * kExactStride + slot] = B;
  s_val[2 * kExactStride + slot] = L;
  if (C == 4) s_val[3 * kExactStride + slot] = __fmul_rn((float)p[3], kInv255);
}

template <int C>
__device__ __forceinline__ void stage_exact_px2(const uint8_t* __restrict__ base, size_t pitch, const Tile& t, uint32_t idx0, uint32_t idx1,
                                                uint32_t slot0, uint32_t slot1, float* s_val, const float* s_lut256) {
  const uint32_t y0 = idx0 / t.tw, x0 = idx0 - y0 * t.tw, y1 = idx1 / t.tw, x1 = idx1 - y1 * t.tw;
  const uint8_t* p0 = base + (size_t)y0 * pitch + (size_t)x0 * C;
  const uint8_t* p1 = base + (size_t)y1 * pitch + (size_t)x1 * C;
  float L0, A0, B0, L1, A1, B1;
  oklab_ref(s_lut256, p0[0], p0[1], p0[2], L0, A0, B0);
  oklab_ref(s_lut256, p1[0], p1[1], p1[2], L1, A1, B1);
  s_val[0 * kExactStride + slot0] = A0;
  s_val[1 * kExactStride + slot0] = B0;
  s_val[2 * kExactStride + slot0] = L0;
  s_val[0 * kExactStride + slot1] = A1;
  s_val[1 * kExactStride + slot1] = B1;
  s_val[2 * kExactStride + slot1] = L1;
  if (C == 4) {
    s_val[3 * kExactStride + slot0] = __fmul_rn((float)p0[3], kInv255);
    s_val[3 * kExactStride + slot1] = __fmul_rn((float)p1[3], kInv255);
  }
}

template <int C>
__device__ float mad_exact_tile(const uint8_t* __restrict__ img, size_t pitch, const Tile& t, float* s_val /*[4][stride]*/,
                                const float* s_lut256, float* s_avg /*[4]*/) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t npx = t.tw * t.th;
  const float count = (float)npx;
  const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
  float run = 0.0f;  // lane c of warp 0 carries channel c: 0 = a, 1 = b, 2 = l, 3 = alpha
  for (int pass = 0; pass < 2; ++pass) {
    run = 0.0f;
#if PXZ_EXACT_PIPELINE
    if (pass == 0 && npx <= (uint32_t)kExactChunk && blockDim.x >= 128) {
      // The first pass in quarters of the tile: while warp 0 runs the sequential sums of quarter k, the other warps convert
      // quarter k + 1 (the conversion is bound by the FP64 pipe, the sums by the latency of dependent adds; with a
      // 384-thread CTA the adding warp shares its scheduler with two converting warps only).  Same values, same order.
      constexpr uint32_t kSub = 1024;
      auto stage = [&](uint32_t s0, uint32_t cnt, uint32_t first, uint32_t nthr) {
        if ((uint32_t)tid >= first) {
          uint32_t i = (uint32_t)tid - first;
          for (; i + nthr < cnt; i += 2 * nthr) stage_exact_px2<C>(base, pitch, t, s0 + i, s0 + i + nthr, s0 + i, s0 + i + nthr, s_val, s_lut256);
          if (i < cnt) stage_exact_px<C>(base, pitch, t, s0 + i, s0 + i, s_val, s_lut256);
        }
      };
      stage(0, min(kSub, npx), 0, blockDim.x);
      __syncthreads();
      for (uint32_t s0 = 0; s0 < npx; s0 += kSub) {
        const uint32_t cnt = min(kSub, npx - s0);
        if (s0 + kSub < npx) stage(s0 + kSub, min(kSub, npx - s0 - kSub), 32, blockDim.x - 32);
        if (warp == 0 && lane < C) run = chain_sum(s_val + lane * kExactStride + s0, cnt, run);
        __syncthreads();
      }
    } else
#endif
    for (uint32_t c0 = 0; c0 < npx; c0 += kExactChunk) {
      const uint32_t n = min((uint32_t)kExactChunk, npx - c0);
      // stage the chunk (skipped in pass 2 when the whole tile is still resident)
      if (pass == 0 || npx > (uint32_t)kExactChunk) {
        // two pixels per iteration: the conversion is a long dependent chain (double-precision divide), so a thread
        // keeps six cube roots in flight instead of three
        uint32_t i = tid;
        for (; i + blockDim.x < n; i += 2 * blockDim.x) stage_exact_px2<C>(base, pitch, t, c0 + i, c0 + i + blockDim.x, i, i + blockDim.x, s_val, s_lut256);
        if (i < n) stage_exact_px<C>(base, pitch, t, c0 + i, i, s_val, s_lut256);
        __syncthreads();
      }
      if (pass == 1) {
        for (uint32_t i = tid; i < n; i += blockDim.x) {
#pragma unroll
          for (int c = 0; c < C; ++c) s_val[c * kExactStride + i] = fabsf(__fsub_rn(s_val[c * kExactStride + i], s_avg[c]));
        }
        __syncthreads();
      }
      if (warp == 0 && lane < C) run = chain_sum(s_val + lane * kExactStride, n, run);
      __syncthreads();
    }
    if (pass == 0) {
      if (warp == 0 && lane < C) s_avg[lane] = __fdiv_rn(run, count);  // operations.rs:65-68
      __syncthreads();
    }
  }
  // operations.rs:89 / :124  (d_a + d_b + d_l [+ d_alpha]) / count, left to right
  float result = 0.f;
  if (warp == 0) {
    const float d0 = __shfl_sync(0xffffffffu, run, 0), d1 = __shfl_sync(0xffffffffu, run, 1);
    const float d2 = __shfl_sync(0xffffffffu, run, 2), d3 = __shfl_sync(0xffffffffu, run, 3);
    float tot = __fadd_rn(__fadd_rn(d0, d1), d2);
    if (C == 4) tot = __fadd_rn(tot, d3);
    result = __fdiv_rn(tot, count);
  }
  return result;  // valid in warp 0
}

// Could the reference-order value of this tile land on the other side of a level threshold?
// Bound of |v_ref - v_fast| in raw-metric units for a tile of n pixels (DESIGN.md "guard band"):
//   sequential f32 mean of channel c : |delta_c| <= 0.375 * n * 2^-24 * max|x_c|   (0.375 = 3/4 * 1/2: partial
//                                      sums grow at most linearly, ulp(s) <= 3/4 * 2^-23 s on average over the ramp)
//   with max L <= 1, max|a| <= 0.276, max|b| <= 0.312 over the sRGB gamut, max alpha <= 1 (0 if the tile is opaque:
//   its alpha sum is exact);  shifting a mean by delta moves that channel's MAD by at most |delta|;
//   sequential f32 sum of the deviations: relative n * 2^-24;  fast arithmetic (SFU cube roots, tree sums): band.abs_raw.
// bound of |reference-order value - fast value| of a tile of npx pixels, raw-metric units
__device__ __forceinline__ float guard_tol_raw(float raw, bool opaque, int C, uint32_t npx, const GuardBand& band) {
  const float nu = (float)npx * 5.9604645e-8f;  // n * 2^-24
  const float gamut = (C == 4 && !opaque) ? 2.588f : 1.588f;
  return 0.375f * nu * gamut + (nu + band.rel) * fabsf(raw) + band.abs_raw;
}

__device__ __forceinline__ bool in_guard_band(float raw, bool opaque, int C, const Tile& t, const ValueMap& vm,
                                              const LevelThresholds& thr, const GuardBand& band, const float* minmax) {
  float v0, v1;
  map_values(vm, minmax, raw, raw, v0, v1);
  const float pv = parse_value_dev(v0);
  if (pv != pv) return true;
  const float tol_raw = guard_tol_raw(raw, opaque, C, t.tw * t.th, band);
  float scale = (vm.mode == 0) ? fabsf(vm.factor) * 10.0f : 1.0f;
  float slack = 1e-30f;
  if (vm.normalise) {
    // v' = (v - min) / (max - min) with the EXACT min and max (k_extreme_list + recompute): an error of the raw value is
    // divided by the range; the subtraction, the division and the two products of the map round once each
    const float rg = __fsub_rn(-minmax[1], minmax[0]);
    if (!(rg > 0.f)) return false;  // empty range: every value maps to 0
    scale /= rg;
    slack += 5e-7f * fabsf(pv);
  }
  const float tol = tol_raw * scale * 1.0001f + slack;
  // only thresholds that change the size of this tile matter
  uint32_t nmax = max(t.tw, t.th);
  int kmax = 0;
  while ((1u << kmax) < nmax) ++kmax;  // dims are 1 for every k >= ceil(log2 n)
  if (kmax > kThresholds - 1) kmax = kThresholds - 1;
  for (int k = 0; k < kmax; ++k) {  // thr[k] separates level k+1 (below) from k (at or above)
    if (fabsf(pv - thr.thr[k]) <= tol) return true;
  }
  if (vm.extra_thr == vm.extra_thr && fabsf(v0 - vm.extra_thr) <= tol) return true;  // quadtree split decision
  if (vm.bucket_edges != 0ull) {  // filter strategy: the bucket of sqrt(2) * pv / sqrt(2) changes at pv = k / 64
    const float kq = rintf(pv * 64.0f);
    if (kq >= 1.0f && kq <= 64.0f && ((vm.bucket_edges >> ((int)kq - 1)) & 1ull) &&
        fabsf(pv - kq * 0.015625f) <= tol + 2e-6f * pv)  // + the roundings of hypot and of the bucket product
      return true;
  }
  // the kink of parse_value at v = -1 (1 + v = 0) maps to 1 px on both sides
  return false;
}

// compact list of the tiles inside the guard band (order is irrelevant)
__global__ void __launch_bounds__(kThreads) k_band_list(const float* __restrict__ vx_fast, const uint8_t* __restrict__ opaque,
                                                        Geom g, int C, ValueMap vm, LevelThresholds thr, GuardBand band,
                                                        const float* minmax, uint32_t* __restrict__ list,
                                                        uint32_t* __restrict__ count) {
  pdl_wait();
  pdl_trigger();
  const uint32_t ntiles = g.cols * g.rows;
  const uint32_t tile = blockIdx.x * kThreads + threadIdx.x;
  if (tile >= ntiles) return;
  const Tile t = tile_of(g, tile);
  if (in_guard_band(vx_fast[tile], opaque[tile] != 0, C, t, vm, thr, band, minmax)) list[atomicAdd(count, 1u)] = tile;
}

// Global normalisation on the fast path: the tiles whose reference-order value could be the minimum or the maximum of the
// image.  minmax = {min, -max} of the FAST values.  The exact minimum is at most fast_min + T (T = the bound at the
// minimum, taken for a full non-opaque tile), so a tile with raw - tol > fast_min + T cannot hold it — and its fast value
// stays above the exact minimum, so a second k_minmax over the patched values returns the exact extremes.
__global__ void __launch_bounds__(kThreads) k_extreme_list(const float* __restrict__ vx_fast, const uint8_t* __restrict__ opaque,
                                                           Geom g, int C, GuardBand band, const float* __restrict__ minmax,
                                                           uint32_t* __restrict__ list, uint32_t* __restrict__ count) {
  pdl_wait();
  pdl_trigger();
  const uint32_t ntiles = g.cols * g.rows;
  const uint32_t tile = blockIdx.x * kThreads + threadIdx.x;
  if (tile >= ntiles) return;
  const Tile t = tile_of(g, tile);
  const float raw = vx_fast[tile];
  if (raw != raw) return;  // NaNs are ignored by the extension
  const float mn = minmax[0], mx = -minmax[1];
  const float tol = guard_tol_raw(raw, opaque[tile] != 0, C, t.tw * t.th, band) * 1.0001f;
  const float t_min = guard_tol_raw(mn, false, C, g.bw * g.bh, band) * 1.0001f;
  const float t_max = guard_tol_raw(mx, false, C, g.bw * g.bh, band) * 1.0001f;
  if (raw - tol <= mn + t_min || raw + tol >= mx - t_max) list[atomicAdd(count, 1u)] = tile;
}

// list == nullptr: every tile (PXZ_FLAG_EXACT_VALUES); else the *count tiles of the list, one per CTA round-robin
// Threads of the CTA that recomputes one guard-band tile.  The per-pixel conversion is parallel and bound by the FP64 pipe,
// the sums are a sequential chain on four lanes, so the CTA mostly waits — and while it does, a 1024-thread CTA holds a whole
// SM's registers against the kernels of the other streams.  Measured on the bench (4 streams): 1024 threads 132.6 GP/s /
// 48.2 us single-stream, 512: 138.0 / 41.4, 384: 139.9 / 44.2, 256: 139.2 / 50.6, 128: 136.2 / 70.0.
#ifndef PXZ_EXACT_THREADS
#define PXZ_EXACT_THREADS 384
#endif
constexpr int kExactThreads = PXZ_EXACT_THREADS;
template <int C>
__global__ void __launch_bounds__(kExactThreads) k_mad_exact(const uint8_t* __restrict__ img, size_t pitch, Geom g, float* vx,
                                                             const uint32_t* __restrict__ list, const uint32_t* __restrict__ count) {
  extern __shared__ float s_dyn[];
  float* s_val = s_dyn;  // 4 * kExactStride
  __shared__ float s_lut256[256];
  __shared__ float s_avg[4];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut256[i] = c_srgb_lut[i];
  pdl_wait();
  pdl_trigger();
  const uint32_t n = list ? *count : g.cols * g.rows;
  if (blockIdx.x >= n) return;
  __syncthreads();
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const uint32_t tile = list ? list[i] : i;
    const Tile t = tile_of(g, tile);
    const float v = mad_exact_tile<C>(img, pitch, t, s_val, s_lut256, s_avg);
    if (threadIdx.x == 0) vx[tile] = v;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Directional Sobel metric (operations.rs:192-259): integer sums, one f64 divide.  Alpha ignored.
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kThreads) k_analyze_sobel(const uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                            float* __restrict__ vx, float* __restrict__ vy) {
  __shared__ unsigned long long s_red[kThreads / 32][2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t ntiles = g.cols * g.rows;
  for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const Tile t = tile_of(g, tile);
    const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
    unsigned long long shz = 0, svr = 0;
    if (t.tw >= 3 && t.th >= 3) {
      const uint32_t ww = t.tw - 2, wh = t.th - 2;
      // one thread per window column, walking down: the three rows are kept in registers
      for (uint32_t x = tid; x < ww; x += kThreads) {
        int r0[3][3], r1[3][3];  // [dx][channel] of rows y, y+1
        const uint8_t* p = base + (size_t)x * C;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx)
#pragma unroll
          for (int c = 0; c < 3; ++c) { r0[dx][c] = p[dx * C + c]; r1[dx][c] = p[pitch + dx * C + c]; }
        uint32_t ahz = 0, avr = 0;
        for (uint32_t y = 0; y < wh; ++y) {
          const uint8_t* q = p + (size_t)(y + 2) * pitch;
          int r2[3][3];
#pragma unroll
          for (int dx = 0; dx < 3; ++dx)
#pragma unroll
            for (int c = 0; c < 3; ++c) r2[dx][c] = q[dx * C + c];
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const int hz = -r0[0][c] - 2 * r0[1][c] - r0[2][c] + r2[0][c] + 2 * r2[1][c] + r2[2][c];  // :240-241
            const int vr = -r0[0][c] - 2 * r1[0][c] - r2[0][c] + r0[2][c] + 2 * r1[2][c] + r2[2][c];  // :244-245
            ahz += (uint32_t)abs(hz);
            avr += (uint32_t)abs(vr);
          }
#pragma unroll
          for (int dx = 0; dx < 3; ++dx)
#pragma unroll
            for (int c = 0; c < 3; ++c) { r0[dx][c] = r1[dx][c]; r1[dx][c] = r2[dx][c]; }
          if ((y & 1023u) == 1023u) { shz += ahz; svr += avr; ahz = avr = 0; }  // u32 cannot overflow in 1024 rows
        }
        shz += ahz;
        svr += avr;
      }
    }
    shz = warp_sum_u64(shz);
    svr = warp_sum_u64(svr);
    if (lane == 0) { s_red[warp][0] = shz; s_red[warp][1] = svr; }
    __syncthreads();
    if (tid == 0) {
      unsigned long long a = 0, b = 0;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) { a += s_red[w][0]; b += s_red[w][1]; }
      const unsigned long long f = (unsigned long long)(t.tw - 2) * (unsigned long long)(t.th - 2) * 4096ull;  // :158,:253-254
      if (t.tw < 3 || t.th < 3 || f == 0) {
        // width or height == 2: the reference divides 0/0 (x86: negative quiet NaN)
        vx[tile] = __uint_as_float(0xFFC00000u);
        vy[tile] = __uint_as_float(0xFFC00000u);
      } else {
        vx[tile] = __double2float_rn(__ddiv_rn((double)a, (double)f));
        vy[tile] = __double2float_rn(__ddiv_rn((double)b, (double)f));
      }
    }
    __syncthreads();
  }
}

// Tiles up to 64x64: the tile is staged once in shared memory as one u32 per pixel; thread (column, row band)
// walks its band keeping the separable partial sums of the two previous rows in registers:
//   h(y) = v(x,y) + 2 v(x+1,y) + v(x+2,y)   ->  hz = h(y+2) - h(y)
//   g(y) = v(x+2,y) - v(x,y)                ->  vr = g(y) + 2 g(y+1) + g(y+2)
// |.| + accumulate is one VABSDIFF each.  Integer arithmetic throughout: bit-exact by construction.
template <int C>
__global__ void __launch_bounds__(kThreads) k_analyze_sobel_tile64(const uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                                   float* __restrict__ vx, float* __restrict__ vy) {
  __shared__ uint32_t s_px[64 * 64];
  __shared__ unsigned long long s_red[kThreads / 32][2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t ntiles = g.cols * g.rows;
  for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const Tile t = tile_of(g, tile);
    const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
    const uint32_t npx = t.tw * t.th;
    for (uint32_t i = tid; i < npx; i += kThreads) {
      const uint32_t y = i / t.tw, x = i - y * t.tw;
      const uint8_t* p = base + (size_t)y * pitch + (size_t)x * C;
      s_px[y * 64 + x] = (C == 4) ? *reinterpret_cast<const uint32_t*>(p)
                                  : ((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16));
    }
    __syncthreads();
    uint32_t ahz = 0, avr = 0;
    if (t.tw >= 3 && t.th >= 3) {
      const uint32_t ww = t.tw - 2, wh = t.th - 2;
      const uint32_t x = tid & 63u, band = tid >> 6;  // 4 bands of window rows
      const uint32_t rows_per = (wh + 3) >> 2;
      const uint32_t y_lo = band * rows_per, y_hi = min(wh, y_lo + rows_per);
      if (x < ww && y_lo < y_hi) {
        int h0[3], h1[3], g0[3], g1[3];
        auto row_terms = [&](uint32_t y, int(&h)[3], int(&gd)[3]) {
          const uint32_t* r = s_px + y * 64 + x;
          const uint32_t p0 = r[0], p1 = r[1], p2 = r[2];
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const int a = (int)((p0 >> (8 * c)) & 0xFFu), b = (int)((p1 >> (8 * c)) & 0xFFu), d = (int)((p2 >> (8 * c)) & 0xFFu);
            h[c] = a + 2 * b + d;
            gd[c] = d - a;
          }
        };
        row_terms(y_lo, h0, g0);
        row_terms(y_lo + 1, h1, g1);
#pragma unroll 2
        for (uint32_t y = y_lo; y < y_hi; ++y) {
          int h2[3], g2[3];
          row_terms(y + 2, h2, g2);
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            ahz = __sad(h2[c], h0[c], ahz);                  // |hz|, operations.rs:240-241,247
            avr = __sad(g0[c] + 2 * g1[c] + g2[c], 0, avr);  // |vr|, operations.rs:244-245,248
            h0[c] = h1[c]; h1[c] = h2[c];
            g0[c] = g1[c]; g1[c] = g2[c];
          }
        }
      }
    }
    unsigned long long shz = warp_sum_u64(ahz), svr = warp_sum_u64(avr);  // per thread <= 16 rows * 3 * 1020 each
    if (lane == 0) { s_red[warp][0] = shz; s_red[warp][1] = svr; }
    __syncthreads();
    if (tid == 0) {
      unsigned long long a = 0, b = 0;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) { a += s_red[w][0]; b += s_red[w][1]; }
      const unsigned long long f = (unsigned long long)(t.tw - 2) * (unsigned long long)(t.th - 2) * 4096ull;  // :158,:253-254
      if (t.tw < 3 || t.th < 3 || f == 0) {
        vx[tile] = __uint_as_float(0xFFC00000u);  // 0/0 in the reference (x86: negative quiet NaN)
        vy[tile] = __uint_as_float(0xFFC00000u);
      } else {
        vx[tile] = __double2float_rn(__ddiv_rn((double)a, (double)f));
        vy[tile] = __double2float_rn(__ddiv_rn((double)b, (double)f));
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// min / -max of the raw values (normalise extension).  out = {min_x, -max_x, min_y, -max_y}, so a
// single ncclMin all-reduce of 4 floats finishes the job across ranks.  NaNs are ignored.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_minmax(const float* __restrict__ vx, const float* __restrict__ vy, uint32_t n,
                                                 float* __restrict__ out4) {
  __shared__ float s[32][4];
  float m[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float a = vx[i], b = vy ? vy[i] : a;
    if (a == a) { m[0] = fminf(m[0], a); m[1] = fminf(m[1], -a); }
    if (b == b) { m[2] = fminf(m[2], b); m[3] = fminf(m[3], -b); }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m[k] = fminf(m[k], __shfl_xor_sync(0xffffffffu, m[k], o));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0)
    for (int k = 0; k < 4; ++k) s[warp][k] = m[k];
  __syncthreads();
  if (threadIdx.x < 4) {
    float r = INFINITY;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r = fminf(r, s[w][threadIdx.x]);
    out4[threadIdx.x] = r;
  }
}

// ------------------------------------------------------------------------------------------------
// plan: reduce_image_section minus the resize (operations.rs:140-156) + exclusive scan of the
// payload sizes (single pass, decoupled look-back), producing the descriptor table.
// ------------------------------------------------------------------------------------------------
// Cost class of a block for the resample kernels' work order (0 = most expensive): by the larger reduced side, then
// plain copies, then blocks a quadtree level masked out.
constexpr int kCostClasses = 8;
__device__ __forceinline__ uint32_t cost_class(uint32_t w, uint32_t h, uint32_t tw, uint32_t th) {
  if (w == 0 || h == 0) return 7u;
  if (w == tw && h == th) return 6u;
  const uint32_t k = 31u - __clz(max(w, h));  // 0..6 for sides 1..64
  return k >= 5u ? 0u : 5u - k;
}

constexpr int kPlanItems = 1;
constexpr int kPlanTile = kThreads * kPlanItems;

// All of it is zero between launches: the CTA that finishes last puts it back (no memset per call).
struct ScanState {
  unsigned int ticket;
  unsigned int done;             // CTAs that are through with the shared state
  unsigned long long status[1];  // [num_tiles]: flag << 62 | value ; flag 1 = aggregate, 2 = inclusive prefix
};

// Decoupled look-back for tile `tile` (tiles taken in ticket order) whose own sum is `agg`; called by all 32 lanes of one
// warp, returns the tile's exclusive prefix to every lane and publishes its inclusive prefix.  One window of 32
// predecessors per step: every lane waits for its own predecessor's status, the window is summed back to the nearest
// inclusive prefix (tiles are ticket-ordered, so predecessors always arrive).
__device__ __forceinline__ unsigned long long lookback_prefix(ScanState* st, uint32_t tile, unsigned long long agg, int lane) {
  constexpr unsigned long long kValue = (1ull << 62) - 1;
  unsigned long long prefix = 0;
  volatile unsigned long long* status = st->status;
  if (tile == 0) {
    if (lane == 0) {
      __threadfence();
      status[0] = (2ull << 62) | agg;
    }
  } else {
    if (lane == 0) {
      status[tile] = (1ull << 62) | agg;
      __threadfence();
    }
    int base = (int)tile - 1;
    while (true) {
      const int idx = base - lane;
      unsigned long long sv = 2ull << 62;  // before tile 0: an inclusive prefix of zero
      if (idx >= 0) {
        do { sv = status[idx]; } while ((sv >> 62) == 0ull);
      }
      const unsigned incl = __ballot_sync(0xffffffffu, (sv >> 62) == 2ull);
      const int stop = incl ? __ffs((int)incl) - 1 : 31;  // nearest inclusive prefix in this window
      unsigned long long v = lane <= stop ? (sv & kValue) : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      prefix += v;
      if (incl) break;
      base -= 32;
    }
    if (lane == 0) {
      __threadfence();
      status[tile] = (2ull << 62) | (prefix + agg);
    }
  }
  return prefix;
}

template <bool STRATEGY>
__global__ void __launch_bounds__(kThreads) k_plan(const float* __restrict__ vx, const float* __restrict__ vy, Geom g,
                                                   ValueMap vm, const float* __restrict__ minmax, LevelThresholds thr,
                                                   const uint8_t* __restrict__ mask, pxz_block_desc* __restrict__ descs,
                                                   uint32_t* __restrict__ tabidx,
                                                   unsigned long long* __restrict__ total, ScanState* st,
                                                   uint32_t* __restrict__ cursor, uint32_t* __restrict__ lists, uint32_t cap,
                                                   StrategyLut strat, uint32_t* __restrict__ tabidx_up) {
  __shared__ unsigned int s_tile;
  __shared__ uint32_t s_hist[kCostClasses], s_base[kCostClasses];
  if (threadIdx.x < kCostClasses) s_hist[threadIdx.x] = 0;
  __shared__ unsigned long long s_warp[kThreads / 32];
  __shared__ unsigned long long s_prefix;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_wait();
  pdl_trigger();
  if (tid == 0) s_tile = atomicAdd(&st->ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t first = tile * kPlanTile + tid * kPlanItems;

  uint32_t dw[kPlanItems], dh[kPlanItems], tix[kPlanItems], tix_up[kPlanItems];
  float val[kPlanItems];
  unsigned long long sz[kPlanItems];
  unsigned long long tsum = 0;
#pragma unroll
  for (int j = 0; j < kPlanItems; ++j) {
    const uint32_t b = first + j;
    sz[j] = 0;
    if (b < nblocks) {
      const Tile t = tile_of(g, b);
      float v0, v1;
      map_values(vm, minmax, vx[b], vy ? vy[b] : vx[b], v0, v1);
      const float p0 = parse_value_dev(v0), p1 = parse_value_dev(v1);
      const uint32_t k0 = level_k(p0, thr), k1 = level_k(p1, thr);
      dw[j] = scaled_dim(t.tw, k0);
      dh[j] = scaled_dim(t.th, k1);
      // f32::hypot (operations.rs:154)
      val[j] = (isinf(p0) || isinf(p1)) ? INFINITY
                                        : __double2float_rn(sqrt(__dadd_rn(__dmul_rn((double)p0, (double)p0),
                                                                           __dmul_rn((double)p1, (double)p1))));
      const uint32_t cx = (t.tw != g.bw) ? 1u : 0u, cy = (t.th != g.bh) ? 1u : 0u;
      const uint32_t ix = (0u * 2u + cx) * kLevelsPerClass + min(k0, (uint32_t)kMaxLevel);
      const uint32_t iy = (1u * 2u + cy) * kLevelsPerClass + min(k1, (uint32_t)kMaxLevel);
      tix[j] = ix | (iy << 16);
      if (STRATEGY) {  // the block's filter pair: the same tables, `stride` entries further per filter
        const uint32_t bucket = strategy_bucket(val[j]);
        const uint32_t fd = strat.down[bucket] * strat.stride, fu = strat.up[bucket] * strat.stride;
        tix_up[j] = (ix + fu) | ((iy + fu) << 16);
        tix[j] = (ix + fd) | ((iy + fd) << 16);
      }
      if (mask != nullptr && mask[b] == 0) { dw[j] = 0; dh[j] = 0; }  // not a leaf of this quadtree level
      sz[j] = (unsigned long long)dw[j] * dh[j] * g.C;
      tsum += sz[j];
    }
  }
  __syncthreads();
  // work order of the resample kernels: per cost class a list of block indices (lists[c * cap ...]); a block's slot is
  // the class cursor this CTA reserved plus its rank inside the CTA.  Order inside a class does not matter.
  uint32_t cls[kPlanItems], rank[kPlanItems];
#pragma unroll
  for (int j = 0; j < kPlanItems; ++j) {
    const uint32_t b = first + j;
    cls[j] = 0; rank[j] = 0;
    if (b < nblocks) {
      const Tile t = tile_of(g, b);
      cls[j] = cost_class(dw[j], dh[j], t.tw, t.th);
      rank[j] = atomicAdd(&s_hist[cls[j]], 1u);
    }
  }
  __syncthreads();
  if (tid < kCostClasses) {
    s_base[tid] = s_hist[tid] ? atomicAdd(&cursor[tid], s_hist[tid]) : 0u;
    __threadfence();  // reserved before this CTA's scan status is published (the last CTA reads the final cursors)
  }
  // block-wide exclusive scan of tsum
  unsigned long long inc = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long n = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += n;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  unsigned long long wbase = 0, agg = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    if (w < warp) wbase += s_warp[w];
    agg += s_warp[w];
  }
  unsigned long long excl = wbase + inc - tsum;

  if (warp == 0) {
    const unsigned long long prefix = lookback_prefix(st, tile, agg, lane);
    if (lane == 0) s_prefix = prefix;
    if ((tile + 1) * (uint32_t)kPlanTile >= nblocks) {
      if (lane == 0) *total = prefix + agg;
      // every other CTA has published its status, hence reserved its slots: the cursors are final
      __syncwarp();
      __threadfence();
      if (lane < kCostClasses) lists[(size_t)kCostClasses * cap + lane] = atomicAdd(&cursor[lane], 0u);
    }
  }
  __syncthreads();
  excl += s_prefix;
#pragma unroll
  for (int j = 0; j < kPlanItems; ++j) {
    const uint32_t b = first + j;
    if (b < nblocks) {
      pxz_block_desc d;
      d.offset = excl;
      d.value = val[j];
      d.w = (uint16_t)dw[j];
      d.h = (uint16_t)dh[j];
      descs[b] = d;
      tabidx[b] = tix[j];
      if (STRATEGY) tabidx_up[b] = tix_up[j];
      lists[(size_t)cls[j] * cap + s_base[cls[j]] + rank[j]] = b;
      excl += sz[j];
    }
  }
  // the CTA that finishes last leaves ticket, status and cursors zeroed for the next launch on this stream
  __shared__ bool s_last;
  if (tid == 0) {
    __threadfence();
    s_last = atomicAdd(&st->done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {
    for (uint32_t i = tid; i < gridDim.x; i += kThreads) st->status[i] = 0ull;
    if (tid < 2 * kCostClasses) cursor[tid] = 0u;
    if (tid == 0) { st->ticket = 0u; st->done = 0u; }
  }
}

// ------------------------------------------------------------------------------------------------
// size curve (rate control, pxz_shrink_to_size): for each of M candidate factors, the payload size k_plan would compute
// from one set of raw values, through the same value -> dims helpers (map_values, parse_value_dev, level_k, scaled_dim).  A thread keeps kSizeItems blocks' values and tile sizes in registers and walks the
// candidates of its CTA (blockIdx.y splits them when the image has too few blocks to fill the device); per candidate a
// warp sum, the warps' partial sums in shared memory, then one 64-bit atomicAdd per CTA and candidate.  Integer sums: the
// result does not depend on the order of the additions.  bytes[] is zero on entry.
// ------------------------------------------------------------------------------------------------
constexpr int kSizeItems = 4;
__global__ void __launch_bounds__(kThreads) k_size_curve(const float* __restrict__ vx, const float* __restrict__ vy, Geom g,
                                                         ValueMap vm, const float* __restrict__ minmax, LevelThresholds thr,
                                                         uint32_t bpp, SizeCandidates cand, unsigned long long* __restrict__ bytes) {
  __shared__ float s_k[kMaxSizeCandidates];
  __shared__ unsigned long long s_part[kThreads / 32][kMaxSizeCandidates];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t per = (cand.n + gridDim.y - 1) / gridDim.y;
  const uint32_t c0 = blockIdx.y * per, c1 = min(cand.n, c0 + per);
  for (uint32_t c = c0 + tid; c < c1; c += kThreads) s_k[c - c0] = cand.k[c];
  float mm[4] = {0.f, 0.f, 0.f, 0.f};
  if (vm.normalise)
#pragma unroll
    for (int i = 0; i < 4; ++i) mm[i] = minmax[i];
  const uint32_t nblocks = g.cols * g.rows;
  float rx[kSizeItems], ry[kSizeItems];
  uint32_t tw[kSizeItems], th[kSizeItems];
#pragma unroll
  for (int j = 0; j < kSizeItems; ++j) {
    const uint32_t b = (blockIdx.x * kSizeItems + j) * kThreads + tid;
    tw[j] = th[j] = 0u;  // no block: contributes nothing
    rx[j] = ry[j] = 0.f;
    if (b < nblocks) {
      const Tile t = tile_of(g, b);
      tw[j] = t.tw;
      th[j] = t.th;
      rx[j] = vx[b];
      ry[j] = vy ? vy[b] : rx[j];
    }
  }
  __syncthreads();
  for (uint32_t c = c0; c < c1; ++c) {
    ValueMap v = vm;
    v.factor = s_k[c - c0];
    unsigned long long px = 0;
#pragma unroll
    for (int j = 0; j < kSizeItems; ++j) {
      float v0, v1;
      map_values(v, mm, rx[j], ry[j], v0, v1);
      const uint32_t dw = scaled_dim(tw[j], level_k(parse_value_dev(v0), thr));
      const uint32_t dh = scaled_dim(th[j], level_k(parse_value_dev(v1), thr));
      if (tw[j] != 0u) px += (unsigned long long)dw * dh;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) px += __shfl_xor_sync(0xffffffffu, px, o);
    if (lane == 0) s_part[warp][c - c0] = px;
  }
  __syncthreads();
  for (uint32_t c = c0 + tid; c < c1; c += kThreads) {
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += s_part[w][c - c0];
    if (s != 0ull) atomicAdd(&bytes[c], s * bpp);
  }
}

// ------------------------------------------------------------------------------------------------
// rate-distortion curve (pxz_rd_curve, pxz_shrink_to_error; DESIGN.md §3).  A block's dims at factor k follow from its raw
// values through the helpers k_plan uses, and they grow monotonically with k (raw values are >= +0 or NaN), so each block
// steps through its few distinct dims at exact f32 bit patterns.  k_rd_events finds them by bisection over the patterns and
// prices each step with the block's error at the new dims, read from the per-pass error table.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kMaxPattern = 0x7F7FFFFFu;  // FLT_MAX; patterns 1 .. kMaxPattern are the finite factors > 0

__global__ void __launch_bounds__(kThreads) k_rd_levels(float* __restrict__ vx, float* __restrict__ vy, uint32_t n, float fx, float fy) {
  for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
    vx[i] = fx;
    vy[i] = fy;
  }
}

// dims and error pass of a block with raw values (rx, ry) and tile (tw, th) at the factor with bit pattern `bits`
struct RdAt {
  uint32_t dw, dh, pass;
};
__device__ __forceinline__ RdAt rd_at(const ValueMap& vm, const float* minmax, const LevelThresholds& thr, const RdPasses& ps, float rx, float ry,
                                      uint32_t tw, uint32_t th, uint32_t bits) {
  ValueMap v = vm;
  v.factor = __uint_as_float(bits);
  float v0, v1;
  map_values(v, minmax, rx, ry, v0, v1);
  const uint32_t kx = level_k(parse_value_dev(v0), thr), ky = level_k(parse_value_dev(v1), thr);
  return RdAt{scaled_dim(tw, kx), scaled_dim(th, ky), min(kx, ps.cap_x) * ps.stride_x + min(ky, ps.cap_y) * ps.stride_y};
}

__global__ void __launch_bounds__(kThreads) k_rd_events(const float* __restrict__ vx, const float* __restrict__ vy, Geom g, ValueMap vm,
                                                        const float* __restrict__ minmax, LevelThresholds thr, uint32_t bpp,
                                                        const unsigned long long* __restrict__ sse_table, RdPasses ps, uint32_t maxev,
                                                        uint32_t* __restrict__ keys, uint32_t* __restrict__ ids,
                                                        unsigned long long* __restrict__ dbytes, unsigned long long* __restrict__ dsse,
                                                        unsigned long long* __restrict__ base) {
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t b = blockIdx.x * kThreads + threadIdx.x;
  unsigned long long bytes0 = 0, sse0 = 0;
  if (b < nblocks) {
    const Tile t = tile_of(g, b);
    // the global normalisation does not depend on the factor: applied once here (the directional map at factor 1 returns the
    // normalised values exactly), then every pattern maps the normalised values
    float rx, ry;
    {
      ValueMap n = vm;
      n.mode = 2;
      n.factor = 1.0f;
      map_values(n, minmax, vx[b], vy ? vy[b] : vx[b], rx, ry);
      vm.normalise = 0;
    }
    RdAt cur = rd_at(vm, minmax, thr, ps, rx, ry, t.tw, t.th, 1u);
    const RdAt end = rd_at(vm, minmax, thr, ps, rx, ry, t.tw, t.th, kMaxPattern);
    unsigned long long sse = sse_table[(size_t)cur.pass * nblocks + b];
    bytes0 = (unsigned long long)cur.dw * cur.dh * bpp;
    sse0 = sse;
    uint32_t p = 1u, n = 0;
    for (; n < maxev && (cur.dw != end.dw || cur.dh != end.dh); ++n) {
      // the smallest pattern above p whose dims differ from cur's: dims(lo) == cur, dims(hi) != cur
      uint32_t lo = p, hi = kMaxPattern;
      while (hi - lo > 1u) {
        const uint32_t mid = lo + (hi - lo) / 2u;
        const RdAt m = rd_at(vm, minmax, thr, ps, rx, ry, t.tw, t.th, mid);
        if (m.dw == cur.dw && m.dh == cur.dh) lo = mid; else hi = mid;
      }
      const RdAt next = rd_at(vm, minmax, thr, ps, rx, ry, t.tw, t.th, hi);
      const unsigned long long nsse = sse_table[(size_t)next.pass * nblocks + b];
      const size_t slot = (size_t)b * maxev + n;
      keys[slot] = hi;
      ids[slot] = (uint32_t)slot;
      dbytes[slot] = ((unsigned long long)next.dw * next.dh - (unsigned long long)cur.dw * cur.dh) * bpp;
      dsse[slot] = nsse - sse;  // mod 2^64: the scan's sums are exact
      cur = next;
      sse = nsse;
      p = hi;
    }
    for (; n < maxev; ++n) {
      const size_t slot = (size_t)b * maxev + n;
      keys[slot] = kRdNoEvent;
      ids[slot] = (uint32_t)slot;
      dbytes[slot] = 0ull;
      dsse[slot] = 0ull;
    }
  }
  bytes0 = warp_sum_u64(bytes0);
  sse0 = warp_sum_u64(sse0);
  if ((threadIdx.x & 31) == 0) {
    if (bytes0) atomicAdd(&base[0], bytes0);
    if (sse0) atomicAdd(&base[1], sse0);
  }
}

// running sums of the sorted events: payload bytes and squared error (mod 2^64); the curve points (last event of each key) are
// counted by a second scan over u32 flags, which keeps the 16-byte scan free of spills
struct RdAcc {
  unsigned long long bytes, sse;
};
struct RdAccSum {
  __host__ __device__ RdAcc operator()(const RdAcc& a, const RdAcc& b) const { return {a.bytes + b.bytes, a.sse + b.sse}; }
};

__device__ __forceinline__ bool rd_last_of_key(const uint32_t* keys, uint32_t i, uint32_t nev) {
  const uint32_t k = keys[i];
  return k != kRdNoEvent && (i + 1 == nev || keys[i + 1] != k);
}

__global__ void __launch_bounds__(kThreads) k_rd_gather(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ ids,
                                                        const unsigned long long* __restrict__ dbytes,
                                                        const unsigned long long* __restrict__ dsse, uint32_t nev, RdAcc* __restrict__ acc,
                                                        uint32_t* __restrict__ last) {
  for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < nev; i += gridDim.x * kThreads) {
    const uint32_t id = ids[i];
    acc[i] = RdAcc{dbytes[id], dsse[id]};
    last[i] = rd_last_of_key(keys, i, nev) ? 1u : 0u;
  }
}

__device__ __forceinline__ void rd_point(uint32_t j, uint32_t key, unsigned long long bytes, unsigned long long sse, unsigned long long max_sse,
                                         uint32_t* pt_key, unsigned long long* pt_bytes, unsigned long long* pt_sse, RdOut* out) {
  pt_key[j] = key;
  pt_bytes[j] = bytes;
  pt_sse[j] = sse;
  atomicMin(&out->least_sse, sse);
  if (sse <= max_sse) atomicMin(&out->first_within, j);
}

// out is all ones on entry (least = first = max)
__global__ void __launch_bounds__(kThreads) k_rd_compact(const uint32_t* __restrict__ keys, const RdAcc* __restrict__ acc,
                                                         const uint32_t* __restrict__ points, uint32_t nev,
                                                         const unsigned long long* __restrict__ base, unsigned long long max_sse,
                                                         uint32_t* __restrict__ pt_key, unsigned long long* __restrict__ pt_bytes,
                                                         unsigned long long* __restrict__ pt_sse, RdOut* __restrict__ out) {
  const uint32_t first = blockIdx.x * kThreads + threadIdx.x;
  if (first == 0) {
    rd_point(0, 1u, base[0], base[1], max_sse, pt_key, pt_bytes, pt_sse, out);
    if (nev == 0) out->count = 1;
  }
  for (uint32_t i = first; i < nev; i += gridDim.x * kThreads) {
    const uint32_t j = points[i];
    if (rd_last_of_key(keys, i, nev)) {
      const RdAcc a = acc[i];
      rd_point(j, keys[i], base[0] + a.bytes, base[1] + a.sse, max_sse, pt_key, pt_bytes, pt_sse, out);
    }
    if (i + 1 == nev) out->count = j + 1;
  }
}

// ------------------------------------------------------------------------------------------------
// rate-distortion optimised encode (pxz_rdo_curve, pxz_rdo_shrink_to_size / _to_error; DESIGN.md §3 "Per-block sizes").  Each
// block may take the dims of any level pair; the error table holds its decode error at every pair.  k_rdo_hull turns a
// block's candidates into the segments of their lower convex hull (the events), the events sorted by rate gain / cost and
// summed in that order give the curve, and k_rdo_levels forces the levels of one curve point for the encode.
// ------------------------------------------------------------------------------------------------
constexpr int kRdoHullThreads = 128;

// gain_a / cost_a > gain_b / cost_b, exactly (costs > 0): the 128-bit products gain_a * cost_b and gain_b * cost_a.  Errors and
// bytes of u16 blocks reach 2^50 and 2^34, so 64-bit products overflow and an f64 rate cannot tell close rates apart.
__device__ __forceinline__ bool rdo_rate_above(unsigned long long ga, unsigned long long ca, unsigned long long gb, unsigned long long cb) {
  const unsigned long long ha = __umul64hi(ga, cb), hb = __umul64hi(gb, ca);
  return ha != hb ? ha > hb : ga * cb > gb * ca;
}

// the merge sort's order: rate descending (padding, gain 0 and cost 1, has rate 0 and sorts after every event)
struct RdoRateDesc {
  __device__ bool operator()(const RdoEvent& a, const RdoEvent& b) const { return rdo_rate_above(a.gain, a.cost, b.gain, b.cost); }
};

// One thread per block; its candidates live in shared memory, column `threadIdx.x` of ncand rows (ncand * 20 bytes per thread).
// The shared memory, not registers, bounds the CTAs per SM: the minimum of one block keeps ptxas from spilling to reach more.
// Candidates, sorted by bytes: one per distinct byte count, the least error, on a tie the lower pass (a block's decode at equal
// dims is the same, so this also keeps the smallest level pair of each dims).  Then from the fewest bytes (1 x 1) the points
// whose error strictly falls, reduced to their lower convex hull in place (a point strictly above the chord of its neighbours
// goes; collinear points stay).
__global__ void __launch_bounds__(kRdoHullThreads, 1) k_rdo_hull(const unsigned long long* __restrict__ sse_table, Geom g, uint32_t bpp,
                                                                 uint32_t lx_max, uint32_t ly_max, uint32_t maxev, RdoEvent* __restrict__ ev,
                                                                 uint32_t* __restrict__ ids, uint32_t* __restrict__ ev_pass,
                                                                 uint32_t* __restrict__ pass0, unsigned long long* __restrict__ base) {
  extern __shared__ __align__(16) uint8_t smem_rdo[];
  const uint32_t ncand = maxev + 1, T = blockDim.x;
  unsigned long long* cb = reinterpret_cast<unsigned long long*>(smem_rdo) + threadIdx.x;  // bytes, row stride T
  unsigned long long* cs = cb + (size_t)ncand * T;                                         // error
  uint32_t* cp = reinterpret_cast<uint32_t*>(smem_rdo + (size_t)ncand * T * 16) + threadIdx.x;  // pass
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t b = blockIdx.x * T + threadIdx.x;
  unsigned long long bytes0 = 0, sse0 = 0, events = 0;
  if (b < nblocks) {
    const Tile t = tile_of(g, b);
    uint32_t n = 0;
    for (uint32_t lx = 0; lx <= lx_max; ++lx) {
      const unsigned long long w = scaled_dim(t.tw, lx);
      for (uint32_t ly = 0; ly <= ly_max; ++ly) {
        const uint32_t pass = lx * (ly_max + 1) + ly;
        const unsigned long long bytes = w * scaled_dim(t.th, ly) * bpp;
        const unsigned long long sse = sse_table[(size_t)pass * nblocks + b];
        uint32_t i = n;
        while (i > 0 && cb[(i - 1) * T] > bytes) --i;
        if (i > 0 && cb[(i - 1) * T] == bytes) {
          if (sse < cs[(i - 1) * T]) {
            cs[(i - 1) * T] = sse;
            cp[(i - 1) * T] = pass;
          }
          continue;
        }
        if (n == ncand) continue;  // not reached: ncand bounds the distinct byte counts of every tile
        for (uint32_t j = n; j > i; --j) {
          cb[j * T] = cb[(j - 1) * T];
          cs[j * T] = cs[(j - 1) * T];
          cp[j * T] = cp[(j - 1) * T];
        }
        cb[i * T] = bytes;
        cs[i * T] = sse;
        cp[i * T] = pass;
        ++n;
      }
    }
    uint32_t top = 0;  // the hull is rows 0 .. top
    for (uint32_t i = 1; i < n; ++i) {
      const unsigned long long pb = cb[i * T], ps = cs[i * T];
      if (ps >= cs[top * T]) continue;  // no less error than a point with fewer bytes
      while (top > 0) {
        const unsigned long long ob = cb[(top - 1) * T], os = cs[(top - 1) * T];
        // the middle point goes when the chord from the point before it falls faster than the step to it
        if (!rdo_rate_above(os - ps, pb - ob, os - cs[top * T], cb[top * T] - ob)) break;
        --top;
      }
      ++top;
      cb[top * T] = pb;
      cs[top * T] = ps;
      cp[top * T] = cp[i * T];
    }
    bytes0 = cb[0];
    sse0 = cs[0];
    events = top;
    pass0[b] = cp[0];
    for (uint32_t k = 0; k < maxev; ++k) {
      const size_t slot = (size_t)b * maxev + k;
      ids[slot] = (uint32_t)slot;
      if (k < top) {
        ev[slot] = RdoEvent{cs[k * T] - cs[(k + 1) * T], cb[(k + 1) * T] - cb[k * T]};
        ev_pass[slot] = cp[(k + 1) * T];
      } else {
        ev[slot] = RdoEvent{0ull, 1ull};
        ev_pass[slot] = kRdNoEvent;
      }
    }
  }
  bytes0 = warp_sum_u64(bytes0);
  sse0 = warp_sum_u64(sse0);
  events = warp_sum_u64(events);
  if ((threadIdx.x & 31) == 0) {
    if (bytes0) atomicAdd(&base[0], bytes0);
    if (sse0) atomicAdd(&base[1], sse0);
    if (events) atomicAdd(&base[2], events);
  }
}

// after the sort: the scan input (bytes up, error down, mod 2^64; padding adds nothing) and each slot's rank in rate order
__global__ void __launch_bounds__(kThreads) k_rdo_gather(const RdoEvent* __restrict__ ev, const uint32_t* __restrict__ ids, uint32_t nev,
                                                         RdAcc* __restrict__ acc, uint32_t* __restrict__ rank) {
  for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < nev; i += gridDim.x * kThreads) {
    const RdoEvent e = ev[i];
    acc[i] = e.gain ? RdAcc{e.cost, 0ull - e.gain} : RdAcc{0ull, 0ull};
    rank[ids[i]] = i;
  }
}

// point 0 = the base totals, point i + 1 = base + the first i + 1 sorted events.  out: count, the last point with bytes <=
// max_bytes plus one (0 on entry: none) and the first with sse <= max_sse (all ones on entry: none)
__global__ void __launch_bounds__(kThreads) k_rdo_points(const RdoEvent* __restrict__ ev, const RdAcc* __restrict__ sums, uint32_t nev,
                                                         const unsigned long long* __restrict__ base, unsigned long long max_bytes,
                                                         unsigned long long max_sse, unsigned long long* __restrict__ pt_bytes,
                                                         unsigned long long* __restrict__ pt_sse, RdoOut* __restrict__ out) {
  const uint32_t first = blockIdx.x * kThreads + threadIdx.x;
  for (uint32_t j = first; j <= nev; j += gridDim.x * kThreads) {
    if (j > 0 && ev[j - 1].gain == 0) break;  // padding: sorted after every event
    unsigned long long bytes = base[0], sse = base[1];
    if (j > 0) {
      const RdAcc a = sums[j - 1];
      bytes += a.bytes;
      sse += a.sse;
    }
    pt_bytes[j] = bytes;
    pt_sse[j] = sse;
    if (bytes <= max_bytes) atomicMax(&out->best_within, j + 1);
    if (sse <= max_sse) atomicMin(&out->first_within, j);
  }
  if (first == 0) out->count = (uint32_t)base[2] + 1;
}

// levels of curve point j: per block the vertex after its events of rank < j (a block's events are ranked in hull order)
__global__ void __launch_bounds__(kThreads) k_rdo_levels(const uint32_t* __restrict__ pass0, const uint32_t* __restrict__ ev_pass,
                                                         const uint32_t* __restrict__ rank, uint32_t maxev, uint32_t nblocks, uint32_t ly_max,
                                                         uint32_t j, float* __restrict__ vx, float* __restrict__ vy) {
  for (uint32_t b = blockIdx.x * kThreads + threadIdx.x; b < nblocks; b += gridDim.x * kThreads) {
    uint32_t pass = pass0[b];
    for (uint32_t k = 0; k < maxev; ++k) {
      const size_t slot = (size_t)b * maxev + k;
      const uint32_t p = ev_pass[slot];
      if (p == kRdNoEvent || rank[slot] >= j) break;
      pass = p;
    }
    const uint32_t lx = pass / (ly_max + 1), ly = pass - lx * (ly_max + 1);
    vx[b] = __uint_as_float((127u - lx) << 23);  // 2^-lx
    vy[b] = __uint_as_float((127u - ly) << 23);
  }
}

// ------------------------------------------------------------------------------------------------
// window of a payload (random access): the blocks of columns [c0, c0 + g.cols) x rows [r0, r0 + g.rows) of a parent payload
// with `pcols` columns, as the payload of the sub-image they tile (geometry g).  One lane of warp 0 per window block takes
// the parent's descriptor and table indices, the block sizes are scanned as in k_plan (same look-back, same work-order
// lists; 32-block tiles, see window_scan_state_bytes), then every warp of the CTA copies whole blocks to their re-packed
// offsets.  Tiles of 32 blocks rather than k_plan's 256: the copy, not the scan, is the work, and with 256 blocks per CTA
// a window of a few hundred blocks ran on one or two SMs, each warp copying 32 blocks in turn (50 us for 256 blocks).  A
// block's tile size in the window is its tile size in the parent, so the parent's table indices stay valid.
// meta / pmeta: tabidx [cap] | order lists | expand-side indices [cap] (pxz_payload::d_tabidx); copy_up: take the latter too
// ------------------------------------------------------------------------------------------------
constexpr int kWindowTile = 32;  // window blocks per CTA: one warp scans them, all 8 warps copy them (4 blocks per warp)
__global__ void __launch_bounds__(kThreads) k_payload_window(const pxz_block_desc* __restrict__ pdescs, const uint32_t* __restrict__ pmeta,
                                                             uint32_t pcap, const uint8_t* __restrict__ ppx, uint32_t pcols, uint32_t c0,
                                                             uint32_t r0, Geom g, int copy_up, pxz_block_desc* __restrict__ descs,
                                                             uint32_t* __restrict__ meta, uint32_t cap, uint8_t* __restrict__ px,
                                                             unsigned long long* __restrict__ total, ScanState* st, uint32_t* __restrict__ cursor) {
  __shared__ unsigned int s_tile;
  __shared__ uint32_t s_hist[kCostClasses], s_base[kCostClasses];
  __shared__ unsigned long long s_src[kWindowTile], s_dst[kWindowTile];
  __shared__ uint32_t s_len[kWindowTile];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < kCostClasses) s_hist[tid] = 0;
  if (tid == 0) s_tile = atomicAdd(&st->ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t nblocks = g.cols * g.rows;
  if (warp == 0) {
    const uint32_t b = tile * kWindowTile + lane;
    uint32_t pb = 0, cls = 0, rank = 0;
    pxz_block_desc d = {};
    unsigned long long sz = 0;
    if (b < nblocks) {
      const uint32_t j = b / g.cols, i = b - j * g.cols;
      pb = (r0 + j) * pcols + c0 + i;
      d = pdescs[pb];
      sz = (unsigned long long)d.w * d.h * g.C;
      const Tile t = tile_of(g, b);
      cls = cost_class(d.w, d.h, t.tw, t.th);
      rank = atomicAdd(&s_hist[cls], 1u);
    }
    __syncwarp();
    if (lane < kCostClasses) {
      s_base[lane] = s_hist[lane] ? atomicAdd(&cursor[lane], s_hist[lane]) : 0u;
      __threadfence();  // reserved before this CTA's scan status is published (the last CTA reads the final cursors)
    }
    __syncwarp();
    unsigned long long inc = sz;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      unsigned long long n = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += n;
    }
    const unsigned long long agg = __shfl_sync(0xffffffffu, inc, 31);
    const unsigned long long prefix = lookback_prefix(st, tile, agg, lane);
    if ((tile + 1) * (uint32_t)kWindowTile >= nblocks) {
      if (lane == 0) *total = prefix + agg;
      // every other CTA has published its status, hence reserved its slots: the cursors are final
      __syncwarp();
      __threadfence();
      if (lane < kCostClasses) meta[(size_t)cap + (size_t)kCostClasses * cap + lane] = atomicAdd(&cursor[lane], 0u);
    }
    if (b < nblocks) {
      const unsigned long long off = prefix + inc - sz;
      s_src[lane] = d.offset;
      s_dst[lane] = off;
      s_len[lane] = (uint32_t)sz;
      d.offset = off;
      descs[b] = d;
      meta[b] = pmeta[pb];
      if (copy_up) meta[(size_t)cap + order_list_words(cap) + b] = pmeta[(size_t)pcap + order_list_words(pcap) + pb];
      meta[(size_t)cap + (size_t)cls * cap + s_base[cls] + rank] = b;
    }
  }
  __syncthreads();
  // block pixels: a warp per block, in 16-byte words when both offsets and the length allow, else 4-byte words (every RGBA
  // block), else bytes
  const uint32_t nhere = min((uint32_t)kWindowTile, nblocks - min(nblocks, tile * (uint32_t)kWindowTile));
  for (uint32_t k = (uint32_t)warp; k < nhere; k += kThreads / 32) {
    const uint8_t* s = ppx + s_src[k];
    uint8_t* o = px + s_dst[k];
    const uint32_t n = s_len[k];
    const unsigned long long a = s_src[k] | s_dst[k] | n;
    if ((a & 15u) == 0) {
#pragma unroll 4
      for (uint32_t q = lane; q < n / 16; q += 32) reinterpret_cast<uint4*>(o)[q] = ldg_nc_v4(s + (size_t)q * 16);
    } else if ((a & 3u) == 0) {
#pragma unroll 4
      for (uint32_t q = lane; q < n / 4; q += 32) reinterpret_cast<uint32_t*>(o)[q] = __ldg(reinterpret_cast<const uint32_t*>(s) + q);
    } else {
      for (uint32_t q = lane; q < n; q += 32) o[q] = __ldg(s + q);
    }
  }
  // the CTA that finishes last leaves ticket, status and cursors zeroed for the next launch on this stream
  __shared__ bool s_last;
  if (tid == 0) {
    __threadfence();
    s_last = atomicAdd(&st->done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {
    for (uint32_t i = tid; i < gridDim.x; i += kThreads) st->status[i] = 0ull;
    if (tid < 2 * kCostClasses) cursor[tid] = 0u;
    if (tid == 0) { st->ticket = 0u; st->done = 0u; }
  }
}

// ------------------------------------------------------------------------------------------------
// resample: image 0.25.5 imageops::resize restated for one block — vertical pass into an unrounded
// f32 intermediate, then horizontal pass, sequential f32 accumulation (no fma) with host-built
// normalised weights, clamp + round half away from zero.  Same-size blocks are copied
// (block.rs:279-281).  direction 0: tile of the image -> payload; 1: payload -> tile of the image.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t to_u8(float t) {
  t = fminf(fmaxf(t, 0.0f), 255.0f);
  const int r = (int)t;
  return (uint32_t)(r + ((t - (float)r) >= 0.5f ? 1 : 0));
}

template <int C>
__device__ __forceinline__ void load_px(const uint8_t* p, float (&f)[C]) {
  if (C == 4) {
    const uint32_t w = *reinterpret_cast<const uint32_t*>(p);
    f[0] = byte_to_float<0>(w);
    f[1] = byte_to_float<1>(w);
    f[2] = byte_to_float<2>(w);
    f[3] = byte_to_float<3>(w);
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) f[c] = (float)p[c];
  }
}

template <int C>
__global__ void __launch_bounds__(kThreads) k_resample(int direction, uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                       const pxz_block_desc* __restrict__ descs,
                                                       const uint32_t* __restrict__ tabidx, uint8_t* __restrict__ payload,
                                                       const AxisTab* __restrict__ tabs, const uint32_t* __restrict__ pool,
                                                       uint32_t max_src_px, uint32_t max_tmp_px, uint8_t* scratch,
                                                       size_t scratch_per_cta) {
  extern __shared__ float s_dyn[];
  float* s_src;
  float* s_tmp;
  if (scratch != nullptr) {  // tiles too large for shared memory: per-CTA global scratch
    s_src = reinterpret_cast<float*>(scratch + (size_t)blockIdx.x * scratch_per_cta);
    s_tmp = s_src + (size_t)max_src_px * C;
  } else {
    s_src = s_dyn;
    s_tmp = s_dyn + (size_t)max_src_px * C;
  }
  const int tid = threadIdx.x;
  const uint32_t nblocks = g.cols * g.rows;
  for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
    const Tile t = tile_of(g, b);
    const pxz_block_desc d = descs[b];
    if (d.w == 0 || d.h == 0) continue;  // masked out (quadtree levels)
    uint8_t* tile_ptr = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
    uint8_t* blk_ptr = payload + d.offset;
    const uint8_t* src;
    uint8_t* dst;
    size_t spitch, dpitch;
    uint32_t sw, sh, dw, dh;
    if (direction == 0) {
      src = tile_ptr; spitch = pitch; sw = t.tw; sh = t.th;
      dst = blk_ptr; dpitch = (size_t)d.w * C; dw = d.w; dh = d.h;
    } else {
      src = blk_ptr; spitch = (size_t)d.w * C; sw = d.w; sh = d.h;
      dst = tile_ptr; dpitch = pitch; dw = t.tw; dh = t.th;
    }
    if (sw == dw && sh == dh) {  // block.rs:279-281
      if (C == 4) {
        for (uint32_t i = tid; i < sw * sh; i += kThreads) {
          const uint32_t y = i / sw, x = i - y * sw;
          *reinterpret_cast<uint32_t*>(dst + (size_t)y * dpitch + (size_t)x * 4) =
              *reinterpret_cast<const uint32_t*>(src + (size_t)y * spitch + (size_t)x * 4);
        }
      } else {
        const uint32_t rb = sw * C;
        for (uint32_t i = tid; i < rb * sh; i += kThreads) {
          const uint32_t y = i / rb, x = i - y * rb;
          dst[(size_t)y * dpitch + x] = src[(size_t)y * spitch + x];
        }
      }
      continue;
    }
    const uint32_t ti = tabidx[b];
    const AxisTab tx = tabs[ti & 0xFFFFu], ty = tabs[ti >> 16];
    const uint32_t* ly = pool + ty.off;
    const uint32_t* cy = ly + ty.n_out;
    const float* wy = reinterpret_cast<const float*>(cy + ty.n_out);
    const uint32_t* lx = pool + tx.off;
    const uint32_t* cx = lx + tx.n_out;
    const float* wx = reinterpret_cast<const float*>(cx + tx.n_out);

    // phase 0: stage the source block as f32
    for (uint32_t i = tid; i < sw * sh; i += kThreads) {
      const uint32_t y = i / sw, x = i - y * sw;
      float f[C];
      load_px<C>(src + (size_t)y * spitch + (size_t)x * C, f);
#pragma unroll
      for (int c = 0; c < C; ++c) s_src[(size_t)i * C + c] = f[c];
    }
    __syncthreads();
    // phase 1: vertical_sample -> f32 [dh][sw]
    for (uint32_t i = tid; i < dh * sw; i += kThreads) {
      const uint32_t oy = i / sw, x = i - oy * sw;
      const uint32_t left = ly[oy], cnt = cy[oy];
      const float* w = wy + (size_t)oy * ty.stride;
      float acc[C];
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c] = 0.0f;
      const float* sp = s_src + ((size_t)left * sw + x) * C;
      for (uint32_t k = 0; k < cnt; ++k) {
        const float wk = w[k];
#pragma unroll
        for (int c = 0; c < C; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(sp[c], wk));
        sp += (size_t)sw * C;
      }
#pragma unroll
      for (int c = 0; c < C; ++c) s_tmp[(size_t)i * C + c] = acc[c];
    }
    __syncthreads();
    // phase 2: horizontal_sample -> u8 [dh][dw]
    for (uint32_t i = tid; i < dh * dw; i += kThreads) {
      const uint32_t oy = i / dw, ox = i - oy * dw;
      const uint32_t left = lx[ox], cnt = cx[ox];
      const float* w = wx + (size_t)ox * tx.stride;
      float acc[C];
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c] = 0.0f;
      const float* sp = s_tmp + ((size_t)oy * sw + left) * C;
      for (uint32_t k = 0; k < cnt; ++k) {
        const float wk = w[k];
#pragma unroll
        for (int c = 0; c < C; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(sp[c], wk));
        sp += C;
      }
      uint8_t* o = dst + (size_t)oy * dpitch + (size_t)ox * C;
      if (C == 4) {
        *reinterpret_cast<uint32_t*>(o) = to_u8(acc[0]) | (to_u8(acc[1]) << 8) | (to_u8(acc[2]) << 16) | (to_u8(acc[3]) << 24);
      } else {
#pragma unroll
        for (int c = 0; c < C; ++c) o[c] = (uint8_t)to_u8(acc[c]);
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// RGBA fast paths of the resample: blocks of at most 64x64 (4096 px), 16-byte aligned tile rows.
// Same arithmetic and accumulation order as k_resample (so the pixels stay bit-identical), but
//   * the next block's source is prefetched into registers while the current one is resampled
//     (persistent CTAs, grid-stride), so global-load latency is off the critical path;
//   * the source block stays packed RGBA8 in shared memory (16 KB, row stride 64 px) and is converted to f32 as it
//     is read by the vertical pass, which keeps three CTAs resident per SM;
//   * outputs are produced in groups of 4 that share one walk over the source samples (blocked tap
//     tables, AxisTab::boff): one 16-byte source load + one broadcast 16-byte weight load feed 16
//     multiply-adds, so the kernel is bound by the FP32 pipe and not by shared-memory bandwidth;
//   * when every alpha of the block is 255 the alpha channel is not computed (it resamples to 255);
//   * rounding to u8 avoids the conversion pipe;
//   * descriptors, table indices and the tap tables themselves run one block ahead (cp.async into a second
//     shared-memory table buffer), so no dependent global load sits between two blocks.
// ------------------------------------------------------------------------------------------------
#ifndef PXZ_RESAMPLE_MINBLOCKS
#define PXZ_RESAMPLE_MINBLOCKS 3
#endif
constexpr int kFastMaxPx = 4096;
constexpr int kFastMaxTabWords = 768;   // one staged table section (checked on the host: max_tab_words)
constexpr int kFastMaxTabs = 128;       // AxisTab entries cached in shared memory (checked on the host)
constexpr int kSrcStride = 64;          // pixels (u32) per source row in shared memory

struct FastSmem {
  uint32_t* src;      // [64][64] packed RGBA8
  float4* tmp;        // [dh][ts], ts = sw rounded up to 8, column index XORed with (row & 7)
  uint32_t* tab;      // [2 buffers][2 axes (y, x)][kFastMaxTabWords]
  AxisTab* atab;      // [kFastMaxTabs]
  uint32_t* taby;     // current buffer, set per block
  uint32_t* tabx;
};

__host__ __device__ constexpr size_t fast_smem_bytes(uint32_t max_tmp_px) {
  return (size_t)kFastMaxPx * 4 + (size_t)max_tmp_px * 16 + 4 * (size_t)kFastMaxTabWords * 4 + (size_t)kFastMaxTabs * sizeof(AxisTab);
}

__device__ __forceinline__ FastSmem carve_fast_smem(float* base, uint32_t max_tmp_px) {
  FastSmem s;
  s.src = reinterpret_cast<uint32_t*>(base);
  s.tmp = reinterpret_cast<float4*>(s.src + kFastMaxPx);
  s.tab = reinterpret_cast<uint32_t*>(s.tmp + max_tmp_px);
  s.atab = reinterpret_cast<AxisTab*>(s.tab + 4 * kFastMaxTabWords);
  s.taby = s.tab;
  s.tabx = s.tab + kFastMaxTabWords;
  return s;
}

__device__ __forceinline__ void cp_async_4(uint32_t* smem_dst, const uint32_t* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
__device__ __forceinline__ void cp_async_wait_keep1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// asynchronous staging of one axis table (blocked or per-output form) into a shared-memory table buffer
__device__ __forceinline__ void stage_axis_async(const AxisTab& t, bool blocked, const uint32_t* __restrict__ pool, uint32_t* dst) {
  const uint32_t* src = pool + (blocked ? t.boff : t.off);
  const uint32_t words = blocked ? t.bwords : 2 * t.n_out + t.n_out * t.stride;
  for (uint32_t i = threadIdx.x; i < words; i += kThreads) cp_async_4(dst + i, src + i);
}
// which table forms a (sw x sh) -> (dw x dh) block uses
__device__ __forceinline__ bool y_blocked(uint32_t dh) { return dh >= 8; }
__device__ __forceinline__ bool x_blocked(uint32_t dw, uint32_t dh) { return dw >= 8 && dh >= 8; }

template <int MODE>
__device__ __forceinline__ float4 px_to_f4(uint32_t w) {
  return make_float4(byte_to_float<0>(w), byte_to_float<1>(w), byte_to_float<2>(w), (MODE & 1) ? byte_to_float<3>(w) : 0.f);
}

// NumCast::from(FloatNearest(clamp(t, 0, 255))): round half away from zero, without F2I/I2F.  For t >= 0 that is
// floor(t + 0.5): both additions round toward zero, so t + 0.5 never crosses an integer upwards and adding 2^23
// drops the fraction; the integer sits in the low mantissa bits.  Returns the float whose low byte is the result.
__device__ __forceinline__ uint32_t to_u8_bits(float t) {
  t = fminf(fmaxf(t, 0.0f), 255.0f);
  return __float_as_uint(__fadd_rz(__fadd_rz(t, 0.5f), 8388608.0f));
}
__device__ __forceinline__ uint32_t to_u8_fast(float t) { return to_u8_bits(t) & 0xFFu; }


// 1.0 and -0.0 as *run-time* values (kernel arguments).  The reference rounds the product and the sum of a tap
// separately (t += p * w without contraction); written as fma(p, w, -0) and fma(product, 1, t) those are two
// exactly-rounded operations in the packed pipe, and because ptxas cannot know the two constants it can neither fold
// them away nor contract the pair into one FFMA2 (it does both when they are literals, even across asm volatile).
struct TapK {
  u64 one2, nz2;
  float one, nz;
};
__device__ __forceinline__ TapK make_tapk(float rt_one, float rt_negzero) {
  TapK k;
  k.one = rt_one; k.nz = rt_negzero;
  k.one2 = pk2(rt_one, rt_one);
  k.nz2 = pk2(rt_negzero, rt_negzero);
  return k;
}

// MODE bit 0: the alpha channel is computed; bit 1: fused multiply-add (PXZ "fast resample": not bit-exact,
// pixels stay within +-1 LSB of the reference order)
template <int MODE>
__device__ __forceinline__ u64 mac2(u64 acc, u64 p, u64 w, const TapK& k) {
  if (MODE & 2) return fma2(p, w, acc);
  return fma2(fma2(p, w, k.nz2), k.one2, acc);
}
// the same with the accumulator updated in place (one register pair in and out: no copies in loop-carried chains)
template <int MODE>
__device__ __forceinline__ void mac2_acc(u64& acc, u64 p, u64 w, const TapK& k) {
  if (MODE & 2) {
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(p), "l"(w));
  } else {
    asm("{\n.reg .b64 t;\nfma.rn.f32x2 t, %1, %2, %3;\nfma.rn.f32x2 %0, t, %4, %0;\n}" : "+l"(acc) : "l"(p), "l"(w), "l"(k.nz2), "l"(k.one2));
  }
}
template <int MODE>
__device__ __forceinline__ float mac1(float acc, float p, float w) {
  if (MODE & 2) return fmaf(p, w, acc);
  return __fadd_rn(acc, __fmul_rn(p, w));
}
__device__ __forceinline__ uint32_t pack_bits(uint32_t r, uint32_t g, uint32_t b, uint32_t a) {
  // byte 0 of each rounded channel, gathered with byte permutes
  return __byte_perm(__byte_perm(r, g, 0x0040), __byte_perm(b, a, 0x0040), 0x5410);
}

__device__ __forceinline__ uint32_t pack_sat_u8x2(int32_t hi_byte, int32_t lo_byte, uint32_t upper16) {
  uint32_t d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(hi_byte), "r"(lo_byte), "r"(upper16));
  return d;
}
// Round-half-away + clamp of two values per instruction.  For t >= 0 the reference's rounding is floor(t + 0.5): the sum
// is rounded toward zero (it never crosses an integer upwards), then the product with 2^-149, again toward zero, is the
// subnormal whose BIT PATTERN is that integer (one ulp of a subnormal is 2^-149; the packed pipe does not flush).  A
// negative sum comes out with the sign bit set, i.e. as a negative s32, so cvt.pack.sat sends it to 0 and anything
// above 255 to 255: two packed FP32 instructions per channel PAIR instead of three scalar ones per channel.
__device__ __forceinline__ u64 round_away_bits2(u64 t2) {
  u64 h, d;
  asm("add.rz.f32x2 %0, %1, %2;" : "=l"(h) : "l"(t2), "l"(0x3f0000003f000000ull));  // + (0.5, 0.5)
  asm("mul.rz.f32x2 %0, %1, %2;" : "=l"(d) : "l"(h), "l"(0x0000000100000001ull));   // * (2^-149, 2^-149)
  return d;
}

// Four outputs that share one walk over the source samples: per channel the accumulators of outputs (0,1) and (2,3)
// sit in one f32x2 register pair each, the sample is broadcast and the weights of the four outputs arrive as one
// 16-byte row — 2 FFMA2 issue slots per channel and sample in fused mode, 4 in exact mode (8 scalar before).
template <int MODE>
struct Acc4 {
  static constexpr int NC = (MODE & 1) ? 4 : 3;
  u64 a01[NC], a23[NC];
  __device__ __forceinline__ Acc4() {
#pragma unroll
    for (int c = 0; c < NC; ++c) a01[c] = a23[c] = 0ull;
  }
  __device__ __forceinline__ void step(const float4& p, const ulonglong2& w, const TapK& k) {
    const float pc[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const u64 pp = pk2(pc[c], pc[c]);
      mac2_acc<MODE>(a01[c], pp, w.x, k);  // in place: no copies of the accumulators in unrolled walks
      mac2_acc<MODE>(a23[c], pp, w.y, k);
    }
  }
  __device__ __forceinline__ float4 out(int j) const {  // j is a compile-time constant at every call site
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const u64 q = (j < 2) ? a01[c] : a23[c];
      v[c] = (j & 1) ? hi2(q) : lo2(q);
    }
    return make_float4(v[0], v[1], v[2], v[3]);
  }
  // the four outputs as packed RGBA8 pixels (alpha 255 when it is not computed)
  __device__ __forceinline__ uint4 pack4() const {
    u64 q01[NC], q23[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) { q01[c] = round_away_bits2(a01[c]); q23[c] = round_away_bits2(a23[c]); }
    auto px = [&](const u64 (&q)[NC], bool hi) -> uint32_t {
      const int32_t r = (int32_t)(hi ? (uint32_t)(q[0] >> 32) : (uint32_t)q[0]), g = (int32_t)(hi ? (uint32_t)(q[1] >> 32) : (uint32_t)q[1]);
      const int32_t b = (int32_t)(hi ? (uint32_t)(q[2] >> 32) : (uint32_t)q[2]);
      const int32_t a = (NC > 3) ? (int32_t)(hi ? (uint32_t)(q[NC > 3 ? 3 : 0] >> 32) : (uint32_t)q[NC > 3 ? 3 : 0]) : 255;
      return pack_sat_u8x2(g, r, pack_sat_u8x2(a, b, 0u));
    };
    return make_uint4(px(q01, false), px(q01, true), px(q23, false), px(q23, true));
  }
};

// One output: channels paired as (r, g) and (b, a); without alpha the blue channel stays scalar.
template <int MODE>
struct Acc1 {
  u64 rg, ba;
  float b;
  __device__ __forceinline__ Acc1() : rg(0ull), ba(0ull), b(0.f) {}
  __device__ __forceinline__ void step(u64 prg, u64 pba, float pb, float w, const TapK& k) {
    const u64 ww = pk2(w, w);
    rg = mac2<MODE>(rg, prg, ww, k);
    if (MODE & 1) ba = mac2<MODE>(ba, pba, ww, k);
    else b = mac1<MODE>(b, pb, w);
  }
  __device__ __forceinline__ float4 out() const {
    float r, g, bb, a;
    unpk2(rg, r, g);
    if (MODE & 1) unpk2(ba, bb, a);
    else { bb = b; a = 0.f; }
    return make_float4(r, g, bb, a);
  }
};

// The same rounding with the clamp left to the pack instruction: 1.5 * 2^23 keeps the exponent fixed on both sides of
// zero, so the bits of the sum are 0x4B400000 + n with n = floor(t + 0.5) for t >= 0 and some negative integer for
// t < -0.5; cvt.pack.sat clamps n to [0, 255] and packs two channels per instruction (|t| < 2^22 here).
__device__ __forceinline__ int32_t round_away_int(float t) {
  return (int32_t)(__float_as_uint(__fadd_rz(__fadd_rz(t, 0.5f), 12582912.0f)) - 0x4B400000u);
}
template <int MODE>
__device__ __forceinline__ uint32_t pack_px(const float4& a) {
  const uint32_t ba = pack_sat_u8x2((MODE & 1) ? round_away_int(a.w) : 255, round_away_int(a.z), 0u);  // {b, a, 0, 0}
  return pack_sat_u8x2(round_away_int(a.y), round_away_int(a.x), ba);                                  // {r, g, b, a}
}

// ---- vertical_sample: src [sh][64] -> tmp [dh][ts] ---------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ void vertical_blocked(const uint32_t* src, float4* tmp, uint32_t sw, uint32_t ts, uint32_t dh,
                                                 const AxisTab& ty, const uint32_t* taby, const TapK& k) {
  const uint32_t lshift = sw <= 1 ? 0 : 32 - __clz(sw - 1);  // lanes per row = next power of two >= sw
  const uint32_t x = threadIdx.x & ((1u << lshift) - 1), grp = threadIdx.x >> lshift, ngrp = kThreads >> lshift;
  if (x >= sw) return;
  const ulonglong2* w4 = reinterpret_cast<const ulonglong2*>(taby);
  const uint32_t* lo = taby + 4 * ty.brows_total;
  const uint32_t* rows = lo + ty.nb;
  const uint32_t* first = rows + ty.nb;
  for (uint32_t ob = grp; ob < ty.nb; ob += ngrp) {
    const uint32_t n = rows[ob];
    const ulonglong2* wp = w4 + first[ob];
    const uint32_t* sp = src + lo[ob] * kSrcStride + x;
    Acc4<MODE> acc;
    uint32_t r = 0;
    for (; r + 2 <= n; r += 2) {
      const float4 p0 = px_to_f4<MODE>(sp[0]), p1 = px_to_f4<MODE>(sp[kSrcStride]);
      const ulonglong2 w0 = wp[r], w1 = wp[r + 1];
      acc.step(p0, w0, k);
      acc.step(p1, w1, k);
      sp += 2 * kSrcStride;
    }
    if (r < n) acc.step(px_to_f4<MODE>(sp[0]), wp[r], k);
    const uint32_t oy = ob * 4;
    tmp[(oy + 0) * ts + (x ^ ((oy + 0) & 7u))] = acc.out(0);
    if (oy + 1 < dh) tmp[(oy + 1) * ts + (x ^ ((oy + 1) & 7u))] = acc.out(1);
    if (oy + 2 < dh) tmp[(oy + 2) * ts + (x ^ ((oy + 2) & 7u))] = acc.out(2);
    if (oy + 3 < dh) tmp[(oy + 3) * ts + (x ^ ((oy + 3) & 7u))] = acc.out(3);
  }
}

template <int MODE>
__device__ __forceinline__ void vertical_plain(const uint32_t* src, float4* tmp, uint32_t sw, uint32_t ts, uint32_t dh,
                                               const AxisTab& ty, const uint32_t* taby, const TapK& k) {
  const uint32_t lshift = sw <= 1 ? 0 : 32 - __clz(sw - 1);
  const uint32_t x = threadIdx.x & ((1u << lshift) - 1), grp = threadIdx.x >> lshift, ngrp = kThreads >> lshift;
  if (x >= sw) return;
  const uint32_t* left = taby;
  const uint32_t* cnt = taby + dh;
  const float* w = reinterpret_cast<const float*>(taby + 2 * dh);
  for (uint32_t oy = grp; oy < dh; oy += ngrp) {
    const uint32_t n = cnt[oy];
    const float* wr = w + oy * ty.stride;
    const uint32_t* sp = src + left[oy] * kSrcStride + x;
    Acc1<MODE> acc;
    auto tap = [&](uint32_t word, float wk) {
      const float4 p = px_to_f4<MODE>(word);
      acc.step(pk2(p.x, p.y), pk2(p.z, p.w), p.z, wk, k);
    };
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) {
      const uint32_t q0 = sp[0], q1 = sp[kSrcStride], q2 = sp[2 * kSrcStride], q3 = sp[3 * kSrcStride];
      const float w0 = wr[i], w1 = wr[i + 1], w2 = wr[i + 2], w3 = wr[i + 3];
      tap(q0, w0); tap(q1, w1); tap(q2, w2); tap(q3, w3);
      sp += 4 * kSrcStride;
    }
    for (; i < n; ++i) {
      tap(sp[0], wr[i]);
      sp += kSrcStride;
    }
    tmp[oy * ts + (x ^ (oy & 7u))] = acc.out();
  }
}

// ---- horizontal_sample: tmp [dh][ts] -> packed RGBA pixels, written through `put(oy, ox, n, px[4])` ------------------
template <int MODE, typename Put>
__device__ __forceinline__ void horizontal_blocked(const float4* tmp, uint32_t ts, uint32_t dw, uint32_t dh, const AxisTab& tx,
                                                   const uint32_t* tabx, const TapK& k, Put put) {
  const ulonglong2* w4 = reinterpret_cast<const ulonglong2*>(tabx);
  const uint32_t* lo = tabx + 4 * tx.brows_total;
  const uint32_t* rows = lo + tx.nb;
  const uint32_t* first = rows + tx.nb;
  const uint32_t hshift = dh <= 1 ? 0 : 32 - __clz(dh - 1);  // lanes = consecutive output rows
  const uint32_t items = tx.nb << hshift;
  for (uint32_t i = threadIdx.x; i < items; i += kThreads) {
    const uint32_t oy = i & ((1u << hshift) - 1), ob = i >> hshift;
    if (oy >= dh) continue;
    const uint32_t n = rows[ob], c0 = lo[ob], s7 = oy & 7u;
    const ulonglong2* wp = w4 + first[ob];
    const float4* trow = tmp + oy * ts;
    Acc4<MODE> acc;
    uint32_t c = 0;
    for (; c + 2 <= n; c += 2) {
      const float4 p0 = trow[(c0 + c) ^ s7], p1 = trow[(c0 + c + 1) ^ s7];
      const ulonglong2 w0 = wp[c], w1 = wp[c + 1];
      acc.step(p0, w0, k);
      acc.step(p1, w1, k);
    }
    if (c < n) acc.step(trow[(c0 + c) ^ s7], wp[c], k);
    const uint32_t ox = ob * 4;
    const uint32_t nvalid = min(4u, dw - ox);
    const uint4 pk = acc.pack4();
    uint32_t px[4] = {pk.x, pk.y, pk.z, pk.w};
    put(oy, ox, nvalid, px);
  }
}

template <int MODE, typename Put>
__device__ __forceinline__ void horizontal_plain(const float4* tmp, uint32_t ts, uint32_t dw, uint32_t dh, const AxisTab& tx,
                                                 const uint32_t* tabx, const TapK& k, Put put) {
  const uint32_t* left = tabx;
  const uint32_t* cnt = tabx + dw;
  const float* w = reinterpret_cast<const float*>(tabx + 2 * dw);
  for (uint32_t i = threadIdx.x; i < dw * dh; i += kThreads) {
    const uint32_t oy = i / dw, ox = i - oy * dw, s7 = oy & 7u;
    const uint32_t n = cnt[ox], c0 = left[ox];
    const float* wr = w + ox * tx.stride;
    const ulonglong2* trow = reinterpret_cast<const ulonglong2*>(tmp + oy * ts);
    Acc1<MODE> acc;
    for (uint32_t t = 0; t < n; ++t) {
      const ulonglong2 p = trow[(c0 + t) ^ s7];
      acc.step(p.x, p.y, lo2(p.y), wr[t], k);
    }
    uint32_t px[4] = {pack_px<MODE>(acc.out()), 0, 0, 0};
    put(oy, ox, 1u, px);
  }
}

// the two passes for one staged block; `put` writes up to 4 horizontally adjacent output pixels
template <int MODE, typename Put>
__device__ __forceinline__ void resample_staged(const FastSmem& sm, uint32_t sw, uint32_t dw, uint32_t dh, const AxisTab& tx,
                                                const AxisTab& ty, bool yblocked, bool xblocked, const TapK& k, Put put) {
  const uint32_t ts = (sw + 7u) & ~7u;
  if (yblocked) vertical_blocked<MODE>(sm.src, sm.tmp, sw, ts, dh, ty, sm.taby, k);
  else vertical_plain<MODE>(sm.src, sm.tmp, sw, ts, dh, ty, sm.taby, k);
  __syncthreads();
  if (xblocked) horizontal_blocked<MODE>(sm.tmp, ts, dw, dh, tx, sm.tabx, k, put);
  else horizontal_plain<MODE>(sm.tmp, ts, dw, dh, tx, sm.tabx, k, put);
}

// ---- encode side: 64x64-or-smaller tiles of the pitched image -> packed payload -----------------------------
template <bool FUSED>
__global__ void __launch_bounds__(kThreads, PXZ_RESAMPLE_MINBLOCKS) k_shrink_rgba(const uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                             const pxz_block_desc* __restrict__ descs,
                                                             const uint32_t* __restrict__ tabidx, uint8_t* __restrict__ payload,
                                                             const AxisTab* __restrict__ tabs, uint32_t ntabs,
                                                             const uint32_t* __restrict__ pool, uint32_t max_tmp_px, float rt_one, float rt_negzero) {
  extern __shared__ float s_dyn[];
  FastSmem sm = carve_fast_smem(s_dyn, max_tmp_px);
  const TapK tapk = make_tapk(rt_one, rt_negzero);
  const uint32_t tid = threadIdx.x;
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t qpr = g.bw >> 2;  // 16-byte quads per full tile row
  uint32_t qrow[4], qcol[4];       // this thread's four quads: fixed for the whole launch
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t q = tid + j * kThreads;
    qrow[j] = q / qpr;
    qcol[j] = (q - qrow[j] * qpr) * 4;
  }
  for (uint32_t i = tid; i < ntabs * (sizeof(AxisTab) / 4); i += kThreads)
    reinterpret_cast<uint32_t*>(sm.atab)[i] = __ldg(reinterpret_cast<const uint32_t*>(tabs) + i);
  __syncthreads();

  auto prefetch = [&](uint32_t b, uint4(&v)[4]) {
    if (b >= nblocks) return;
    const Tile t = tile_of(g, b);
    const uint8_t* base = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      v[j] = (qrow[j] < t.th && qcol[j] < t.tw) ? ldg_nc_v4(base + (size_t)qrow[j] * pitch + (size_t)qcol[j] * 4)
                                                 : make_uint4(0xFF000000u, 0xFF000000u, 0xFF000000u, 0xFF000000u);
  };
  // tables of block `b` (descriptor d, table indices ti) -> table buffer `buf`; always commits one cp.async group
  auto stage_tables = [&](uint32_t b, const pxz_block_desc& d, uint32_t ti, uint32_t buf) {
    if (b < nblocks) {
      const Tile t = tile_of(g, b);
      if (d.w != 0 && d.h != 0 && !(t.tw == d.w && t.th == d.h)) {
        uint32_t* dst = sm.tab + buf * 2 * kFastMaxTabWords;
        stage_axis_async(sm.atab[ti >> 16], y_blocked(d.h), pool, dst);
        stage_axis_async(sm.atab[ti & 0xFFFFu], x_blocked(d.w, d.h), pool, dst + kFastMaxTabWords);
      }
    }
    cp_async_commit();
  };

  uint32_t b = blockIdx.x;
  uint4 cur[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) cur[j] = make_uint4(0, 0, 0, 0);
  prefetch(b, cur);
  pxz_block_desc dcur{}, dnxt{};
  uint32_t ticur = 0, tinxt = 0;
  if (b < nblocks) { dcur = descs[b]; ticur = tabidx[b]; }
  if (b + gridDim.x < nblocks) { dnxt = descs[b + gridDim.x]; tinxt = tabidx[b + gridDim.x]; }
  stage_tables(b, dcur, ticur, 0);
  for (uint32_t it = 0; b < nblocks; b += gridDim.x, ++it) {
    const uint32_t buf = it & 1;
    const Tile t = tile_of(g, b);
    const pxz_block_desc d = dcur;
    const uint32_t ti = ticur;
    // everything the next block needs is requested now and consumed one iteration later
    uint4 nxt[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) nxt[j] = make_uint4(0, 0, 0, 0);
    prefetch(b + gridDim.x, nxt);
    pxz_block_desc dnn{};
    uint32_t tinn = 0;
    if (b + 2 * gridDim.x < nblocks) { dnn = descs[b + 2 * gridDim.x]; tinn = tabidx[b + 2 * gridDim.x]; }
    stage_tables(b + gridDim.x, dnxt, tinxt, buf ^ 1);

    uint32_t* dst = reinterpret_cast<uint32_t*>(payload + d.offset);
    const uint32_t sw = t.tw, sh = t.th, dw = d.w, dh = d.h;
    if (dw == 0 || dh == 0) {
      // masked out (quadtree levels): nothing to write
    } else if (sw == dw && sh == dh) {
      // block.rs:279-281: clone.  The tile is contiguous in the payload (4-byte aligned only).
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (qrow[j] < sh && qcol[j] < sw) {
          uint32_t* o = dst + (size_t)qrow[j] * sw + qcol[j];
          o[0] = cur[j].x; o[1] = cur[j].y; o[2] = cur[j].z; o[3] = cur[j].w;
        }
      }
    } else {
      const AxisTab tx = sm.atab[ti & 0xFFFFu], ty = sm.atab[ti >> 16];
      const bool yb = y_blocked(dh), xb = x_blocked(dw, dh);
      sm.taby = sm.tab + buf * 2 * kFastMaxTabWords;
      sm.tabx = sm.taby + kFastMaxTabWords;
      uint32_t aand = 0xFF000000u;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        aand &= (cur[j].x & cur[j].y) & (cur[j].z & cur[j].w);  // out-of-tile quads were filled with alpha 255
        if (qrow[j] < sh && qcol[j] < sw) *reinterpret_cast<uint4*>(sm.src + qrow[j] * kSrcStride + qcol[j]) = cur[j];
      }
      cp_async_wait_keep1();  // this block's tables (requested one iteration ago) have landed
      const bool opaque = __syncthreads_and(aand == 0xFF000000u) != 0;  // also the barrier after staging
      auto put = [&](uint32_t oy, uint32_t ox, uint32_t n, const uint32_t(&px)[4]) {
        uint32_t* o = dst + (size_t)oy * dw + ox;
        o[0] = px[0];
        if (n > 1) o[1] = px[1];
        if (n > 2) o[2] = px[2];
        if (n > 3) o[3] = px[3];
      };
      if (opaque) resample_staged<(FUSED ? 2 : 0)>(sm, sw, dw, dh, tx, ty, yb, xb, tapk, put);
      else resample_staged<(FUSED ? 3 : 1)>(sm, sw, dw, dh, tx, ty, yb, xb, tapk, put);
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) cur[j] = nxt[j];
    dcur = dnxt; ticur = tinxt;
    dnxt = dnn; tinxt = tinn;
  }
}

// ---- decode side: packed payload blocks -> 64x64-or-smaller tiles of the pitched image (expand + paste) ------
template <bool FUSED>
__global__ void __launch_bounds__(kThreads, PXZ_RESAMPLE_MINBLOCKS) k_expand_rgba(uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                             const pxz_block_desc* __restrict__ descs,
                                                             const uint32_t* __restrict__ tabidx,
                                                             const uint8_t* __restrict__ payload,
                                                             const AxisTab* __restrict__ tabs, uint32_t ntabs,
                                                             const uint32_t* __restrict__ pool, uint32_t max_tmp_px, float rt_one, float rt_negzero) {
  extern __shared__ float s_dyn[];
  FastSmem sm = carve_fast_smem(s_dyn, max_tmp_px);
  const TapK tapk = make_tapk(rt_one, rt_negzero);
  const uint32_t tid = threadIdx.x;
  const uint32_t nblocks = g.cols * g.rows;
  for (uint32_t i = tid; i < ntabs * (sizeof(AxisTab) / 4); i += kThreads)
    reinterpret_cast<uint32_t*>(sm.atab)[i] = __ldg(reinterpret_cast<const uint32_t*>(tabs) + i);
  __syncthreads();

  auto prefetch = [&](uint32_t b, uint32_t(&v)[16], const pxz_block_desc& d) {
    if (b >= nblocks) return;
    const uint32_t n = (uint32_t)d.w * d.h;
    const uint32_t* p = reinterpret_cast<const uint32_t*>(payload + d.offset);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const uint32_t i = tid + j * kThreads;
      v[j] = i < n ? __ldg(p + i) : 0xFF000000u;
    }
  };
  auto stage_tables = [&](uint32_t b, const pxz_block_desc& d, uint32_t ti, uint32_t buf) {
    if (b < nblocks) {
      const Tile t = tile_of(g, b);
      if (d.w != 0 && d.h != 0 && !(t.tw == d.w && t.th == d.h)) {
        uint32_t* dst = sm.tab + buf * 2 * kFastMaxTabWords;
        stage_axis_async(sm.atab[ti >> 16], y_blocked(t.th), pool, dst);
        stage_axis_async(sm.atab[ti & 0xFFFFu], x_blocked(t.tw, t.th), pool, dst + kFastMaxTabWords);
      }
    }
    cp_async_commit();
  };

  // descriptors run two blocks ahead: the pixel prefetch of the next block needs its descriptor
  uint32_t b = blockIdx.x;
  pxz_block_desc dcur{}, dnxt{};
  uint32_t ticur = 0, tinxt = 0;
  if (b < nblocks) { dcur = descs[b]; ticur = tabidx[b]; }
  if (b + gridDim.x < nblocks) { dnxt = descs[b + gridDim.x]; tinxt = tabidx[b + gridDim.x]; }
  uint32_t cur[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) cur[j] = 0xFF000000u;
  prefetch(b, cur, dcur);
  stage_tables(b, dcur, ticur, 0);
  for (uint32_t it = 0; b < nblocks; b += gridDim.x, ++it) {
    const uint32_t buf = it & 1;
    const Tile t = tile_of(g, b);
    const pxz_block_desc d = dcur;
    const uint32_t ti = ticur;
    uint32_t nxt[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) nxt[j] = 0xFF000000u;
    prefetch(b + gridDim.x, nxt, dnxt);
    pxz_block_desc dnn{};
    uint32_t tinn = 0;
    if (b + 2 * gridDim.x < nblocks) { dnn = descs[b + 2 * gridDim.x]; tinn = tabidx[b + 2 * gridDim.x]; }
    stage_tables(b + gridDim.x, dnxt, tinxt, buf ^ 1);

    uint8_t* dst = img + (size_t)t.y0 * pitch + (size_t)t.x0 * 4;
    const uint32_t sw = d.w, sh = d.h, dw = t.tw, dh = t.th;
    const bool pow2 = (sw & (sw - 1)) == 0;
    const uint32_t sshift = 31 - __clz(sw | 1u);
    if (sw == 0 || sh == 0) {
      // masked out (quadtree levels): the tile keeps what the output image already holds
    } else if (sw == dw && sh == dh) {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const uint32_t i = tid + j * kThreads;
        if (i < sw * sh) {
          const uint32_t y = pow2 ? (i >> sshift) : (i / sw), x = i - y * sw;
          *reinterpret_cast<uint32_t*>(dst + (size_t)y * pitch + (size_t)x * 4) = cur[j];
        }
      }
    } else if (sw == 1 && sh == 1) {
      // a 1x1 block: every output has exactly one tap whose normalised weight is w / w = 1.0 in both passes, so the
      // tile is the source pixel replicated — for every filter.  16-byte stores, no staging, no barrier.
      const uint32_t p = __ldg(reinterpret_cast<const uint32_t*>(payload + d.offset));
      const uint4 v = make_uint4(p, p, p, p);
      const uint32_t qpr = (dw + 3) >> 2;
      for (uint32_t q = tid; q < qpr * dh; q += kThreads) {
        const uint32_t y = q / qpr, x = (q - y * qpr) << 2;
        uint8_t* o = dst + (size_t)y * pitch + (size_t)x * 4;
        if (x + 4 <= dw) *reinterpret_cast<uint4*>(o) = v;
        else for (uint32_t k = x; k < dw; ++k) reinterpret_cast<uint32_t*>(dst + (size_t)y * pitch)[k] = p;
      }
    } else {
      const AxisTab tx = sm.atab[ti & 0xFFFFu], ty = sm.atab[ti >> 16];
      const bool yb = y_blocked(dh), xb = x_blocked(dw, dh);
      sm.taby = sm.tab + buf * 2 * kFastMaxTabWords;
      sm.tabx = sm.taby + kFastMaxTabWords;
      uint32_t aand = 0xFF000000u;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const uint32_t i = tid + j * kThreads;
        aand &= cur[j];
        if (i < sw * sh) {
          const uint32_t y = pow2 ? (i >> sshift) : (i / sw), x = i - y * sw;
          sm.src[y * kSrcStride + x] = cur[j];
        }
      }
      cp_async_wait_keep1();
      const bool opaque = __syncthreads_and((aand & 0xFF000000u) == 0xFF000000u) != 0;
      auto put = [&](uint32_t oy, uint32_t ox, uint32_t n, const uint32_t(&px)[4]) {
        uint32_t* o = reinterpret_cast<uint32_t*>(dst + (size_t)oy * pitch) + ox;
        if (n == 4) {
          *reinterpret_cast<uint4*>(o) = make_uint4(px[0], px[1], px[2], px[3]);  // tile rows are 16-byte aligned
        } else {
          o[0] = px[0];
          if (n > 1) o[1] = px[1];
          if (n > 2) o[2] = px[2];
        }
      };
      if (opaque) resample_staged<(FUSED ? 2 : 0)>(sm, sw, dw, dh, tx, ty, yb, xb, tapk, put);
      else resample_staged<(FUSED ? 3 : 1)>(sm, sw, dw, dh, tx, ty, yb, xb, tapk, put);
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) cur[j] = nxt[j];
    dcur = dnxt; ticur = tinxt;
    dnxt = dnn; tinxt = tinn;
  }
}

// ---- work order of the warp-per-tile resample kernels for descriptors that came from the host (k_plan does the same
// for its own): cursor[0..7] class cursors, cursor[8] = CTAs done; all zero on entry
__global__ void __launch_bounds__(kThreads) k_class_lists(const pxz_block_desc* __restrict__ descs, Geom g, uint32_t* __restrict__ cursor,
                                                          uint32_t* __restrict__ lists, uint32_t cap) {
  __shared__ uint32_t s_hist[kCostClasses], s_base[kCostClasses];
  const uint32_t tid = threadIdx.x;
  const uint32_t nblocks = g.cols * g.rows;
  if (tid < kCostClasses) s_hist[tid] = 0;
  __syncthreads();
  const uint32_t b = blockIdx.x * kThreads + tid;
  uint32_t cls = 0, rank = 0;
  if (b < nblocks) {
    const Tile t = tile_of(g, b);
    const pxz_block_desc d = descs[b];
    cls = cost_class(d.w, d.h, t.tw, t.th);
    rank = atomicAdd(&s_hist[cls], 1u);
  }
  __syncthreads();
  if (tid < kCostClasses) s_base[tid] = s_hist[tid] ? atomicAdd(&cursor[tid], s_hist[tid]) : 0u;
  __syncthreads();
  if (b < nblocks) lists[(size_t)cls * cap + s_base[cls] + rank] = b;
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&cursor[kCostClasses], 1u) == gridDim.x - 1) {
      for (int c = 0; c < kCostClasses; ++c) lists[(size_t)kCostClasses * cap + c] = atomicAdd(&cursor[c], 0u);
      for (int c = 0; c <= kCostClasses; ++c) cursor[c] = 0u;  // zero again for the next launch (k_plan shares the words)
    }
  }
}

// quadtree level decision (process/tree.rs:47-77)
__global__ void __launch_bounds__(kThreads) k_tree_mask(const float* __restrict__ vx, Geom g, const uint8_t* __restrict__ parent_recurse,
                                                        uint32_t parent_cols, float thr, int positive, uint8_t* __restrict__ leaf,
                                                        uint8_t* __restrict__ recurse) {
  const uint32_t b = blockIdx.x * kThreads + threadIdx.x;
  if (b >= g.cols * g.rows) return;
  const uint32_t by = b / g.cols, bx = b - by * g.cols;
  const bool active = parent_recurse == nullptr || parent_recurse[(by >> 1) * parent_cols + (bx >> 1)] != 0;
  const bool reduce = (vx[b] >= thr) != (positive != 0);  // (value >= threshold) ^ is_positive; NaN >= thr is false
  leaf[b] = (uint8_t)(active && reduce);
  recurse[b] = (uint8_t)(active && !reduce);
}

// ------------------------------------------------------------------------------------------------
// `fir` resize semantics (PixlzrBlock::resize with the fast_image_resize feature, block.rs:292-333): integer
// convolution with 16-bit coefficients (tables.cpp build_axis_table_fir), HORIZONTAL pass first into a u8 image, then the
// vertical pass; an axis that keeps its size is not convolved; RGBA with a non-nearest algorithm runs on alpha
// pre-multiplied samples.  One CTA per block, source and intermediate in shared memory.  Bit-exact against the oracle's
// restatement by construction (integer arithmetic); "parity unpinned" against the crate itself.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mul_div_255_dev(uint32_t a, uint32_t b) {
  const uint32_t t = a * b + 128u;
  return ((t >> 8) + t) >> 8;
}
template <int C>
__global__ void __launch_bounds__(kThreads) k_resample_fir(int direction, uint8_t* __restrict__ img, size_t pitch, Geom g,
                                                           const pxz_block_desc* __restrict__ descs, const uint32_t* __restrict__ tabidx,
                                                           uint8_t* __restrict__ payload, const AxisTab* __restrict__ tabs,
                                                           const uint32_t* __restrict__ pool, uint32_t src_cap_bytes) {
  extern __shared__ uint8_t s_fir[];
  uint8_t* s_src = s_fir;
  uint8_t* s_tmp = s_fir + src_cap_bytes;
  const uint32_t nblocks = g.cols * g.rows;
  for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
    const pxz_block_desc d = descs[b];
    if (d.w == 0 || d.h == 0) continue;  // masked out
    const Tile t = tile_of(g, b);
    uint8_t* tile0 = img + (size_t)t.y0 * pitch + (size_t)t.x0 * C;
    uint8_t* blk = payload + d.offset;
    const uint32_t sw = direction == 0 ? t.tw : d.w, sh = direction == 0 ? t.th : d.h;
    const uint32_t dw = direction == 0 ? d.w : t.tw, dh = direction == 0 ? d.h : t.th;
    const uint8_t* src = direction == 0 ? tile0 : blk;
    const size_t sstride = direction == 0 ? pitch : (size_t)sw * C;
    uint8_t* dst = direction == 0 ? blk : tile0;
    const size_t dstride = direction == 0 ? (size_t)dw * C : pitch;
    if (sw == dw && sh == dh) {  // block.rs:279-281: clone
      for (uint32_t i = threadIdx.x; i < sh * sw * C; i += kThreads) {
        const uint32_t y = i / (sw * C), x = i - y * (sw * C);
        dst[(size_t)y * dstride + x] = src[(size_t)y * sstride + x];
      }
      continue;
    }
    const uint32_t ti = tabidx[b];
    const AxisTab tx = tabs[ti & 0xFFFFu], ty = tabs[ti >> 16];
    const bool premul = C == 4 && !(tx.pad2_ & kFirNearestFlag);
    __syncthreads();  // the previous block's passes are done with the buffers
    for (uint32_t i = threadIdx.x; i < sw * sh; i += kThreads) {
      const uint32_t y = i / sw, x = i - y * sw;
      const uint8_t* p = src + (size_t)y * sstride + (size_t)x * C;
      uint32_t c0 = p[0], c1 = p[1], c2 = p[2];
      if (C == 4) {
        const uint32_t a = p[3];
        if (premul) { c0 = mul_div_255_dev(c0, a); c1 = mul_div_255_dev(c1, a); c2 = mul_div_255_dev(c2, a); }
        s_src[(size_t)i * 4 + 3] = (uint8_t)a;
      }
      s_src[(size_t)i * C] = (uint8_t)c0; s_src[(size_t)i * C + 1] = (uint8_t)c1; s_src[(size_t)i * C + 2] = (uint8_t)c2;
    }
    __syncthreads();
    const uint8_t* hsrc = s_src;  // [sh][dw] after the horizontal pass
    if (sw != dw) {
      const uint32_t* left = pool + tx.off;
      const uint32_t* cnt = left + dw;
      const int32_t* kk = reinterpret_cast<const int32_t*>(cnt + dw);
      const int p = (int)(tx.pad2_ & 0xFFu);
      for (uint32_t i = threadIdx.x; i < sh * dw; i += kThreads) {
        const uint32_t y = i / dw, x = i - y * dw;
        const uint32_t l = left[x], n = cnt[x];
        const int32_t* kr = kk + (size_t)x * tx.stride;
        int32_t ss[C];
#pragma unroll
        for (int c = 0; c < C; ++c) ss[c] = 1 << (p - 1);
        const uint8_t* q = s_src + ((size_t)y * sw + l) * C;
        for (uint32_t j = 0; j < n; ++j) {
          const int32_t k = kr[j];
#pragma unroll
          for (int c = 0; c < C; ++c) ss[c] += (int32_t)q[j * C + c] * k;
        }
#pragma unroll
        for (int c = 0; c < C; ++c) s_tmp[(size_t)i * C + c] = (uint8_t)min(255, max(0, ss[c] >> p));
      }
      hsrc = s_tmp;
      __syncthreads();
    }
    {
      const uint32_t* left = pool + ty.off;
      const uint32_t* cnt = left + dh;
      const int32_t* kk = reinterpret_cast<const int32_t*>(cnt + dh);
      const int p = (int)(ty.pad2_ & 0xFFu);
      const bool vert = sh != dh;
      for (uint32_t i = threadIdx.x; i < dh * dw; i += kThreads) {
        const uint32_t y = i / dw, x = i - y * dw;
        uint32_t o[4] = {0, 0, 0, 255};
        if (vert) {
          const uint32_t l = left[y], n = cnt[y];
          const int32_t* kr = kk + (size_t)y * ty.stride;
          int32_t ss[C];
#pragma unroll
          for (int c = 0; c < C; ++c) ss[c] = 1 << (p - 1);
          for (uint32_t j = 0; j < n; ++j) {
            const int32_t k = kr[j];
            const uint8_t* q = hsrc + ((size_t)(l + j) * dw + x) * C;
#pragma unroll
            for (int c = 0; c < C; ++c) ss[c] += (int32_t)q[c] * k;
          }
#pragma unroll
          for (int c = 0; c < C; ++c) o[c] = (uint32_t)min(255, max(0, ss[c] >> p));
        } else {
#pragma unroll
          for (int c = 0; c < C; ++c) o[c] = hsrc[((size_t)y * dw + x) * C + c];
        }
        if (premul) {
          const uint32_t a = o[3];
#pragma unroll
          for (int c = 0; c < 3; ++c) o[c] = a == 0 ? 0u : min(255u, (o[c] * 255u + a / 2) / a);
        }
        uint8_t* out = dst + (size_t)y * dstride + (size_t)x * C;
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = (uint8_t)o[c];
      }
    }
  }
}

#ifndef PXZ_SHRINK_WARP_CTAS
#define PXZ_SHRINK_WARP_CTAS 3
#endif
#ifndef PXZ_EXPAND_WARP_CTAS
#define PXZ_EXPAND_WARP_CTAS 4
#endif
#ifndef PXZ_SHRINK_TMA_CTAS
#define PXZ_SHRINK_TMA_CTAS 3
#endif
#include "resample_warp.cuh"
#include "resample_tma.cuh"
#include "analyze_sobel_tma.cuh"

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static inline int clamp_grid(long long want, long long cap) { return (int)(want < 1 ? 1 : (want > cap ? cap : want)); }

template <typename K>
static cudaError_t set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return cudaSuccess;
}

// Both launchers raise the kernel's dynamic shared memory limit when `smem` is above the default 48 KB and return
// cudaGetLastError() of the launch.
// launch_pdl: programmatic stream serialization (see pdl_wait): the kernel may be scheduled while its predecessor drains
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaError_t e = set_smem(kernel, smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  const cudaError_t last = cudaGetLastError();
  return e != cudaSuccess ? e : last;
}
// launch: an ordinary stream-ordered launch
template <typename... KArgs, typename... Args>
static cudaError_t launch(void (*kernel)(KArgs...), dim3 grid, int block, size_t smem, cudaStream_t s, Args&&... args) {
  const cudaError_t e = set_smem(kernel, smem);
  if (e != cudaSuccess) return e;
  kernel<<<grid, block, smem, s>>>(KArgs(args)...);
  return cudaGetLastError();
}

cudaError_t launch_analyze_mad_fast(const uint8_t* img, size_t pitch, const Geom& g, float* vx, uint8_t* opaque,
                                    uint32_t* zero_word, cudaStream_t s, int sm_count, uint64_t* launches) {
  const uint32_t ntiles = g.cols * g.rows;
  const bool aligned = g.C == 4 && (g.bw % 4 == 0) && (g.W % 4 == 0) && (pitch % 16 == 0) &&
                       ((reinterpret_cast<uintptr_t>(img) & 15u) == 0);
  const uint32_t quads = (g.bw / 4) * g.bh;
  // k_analyze_mad_rgba keeps in-tile byte offsets in 32 bits; a wider tile (a view into a very wide tensor) takes
  // k_analyze_mad_any, which addresses with size_t
  const bool offsets32 = (size_t)(g.bh - 1) * pitch + (size_t)g.bw * 4 <= 0xFFFFFFFFull;
  ++*launches;
  if (aligned && offsets32 && quads <= 1024) {
    // G threads per tile, <= 4 quads (16 px) per thread; 256 / G tiles per CTA
    struct Variant {
      void (*kernel)(const uint8_t*, size_t, Geom, float*, uint8_t*, uint32_t*);
      uint32_t tiles_per_cta;
    };
    const Variant v = quads > 512   ? Variant{k_analyze_mad_rgba<256, 4>, 1}
                      : quads > 256 ? Variant{k_analyze_mad_rgba<128, 4>, 2}
                      : quads > 128 ? Variant{k_analyze_mad_rgba<64, 4>, 4}
                                    : Variant{k_analyze_mad_rgba<32, 4>, 8};
    return launch_pdl(v.kernel, clamp_grid((ntiles + v.tiles_per_cta - 1) / v.tiles_per_cta, sm_count * PXZ_MAD_MINBLOCKS), kThreads,
                      256 * kMadLutStride * sizeof(float), s, img, pitch, g, vx, opaque, zero_word);
  }
  return launch_pdl(g.C == 4 ? k_analyze_mad_any<4> : k_analyze_mad_any<3>, clamp_grid(ntiles, sm_count * 3), kThreads,
                    256 * 32 * sizeof(float), s, img, pitch, g, vx, opaque, zero_word);
}

cudaError_t launch_analyze_mad_exact(const uint8_t* img, size_t pitch, const Geom& g, float* vx, const float* vx_fast,
                                     const uint8_t* opaque, const ValueMap* vm, const LevelThresholds* thr, const GuardBand* band,
                                     const float* minmax, uint32_t* list, uint32_t* count, cudaStream_t s, int sm_count,
                                     uint64_t* launches) {
  const uint32_t ntiles = g.cols * g.rows;
  const bool banded = vx_fast != nullptr;
  if (banded) {
    // *count was zeroed by the fast analysis kernel that produced vx_fast (launch_analyze_mad_fast's zero_word), or by the
    // caller between two lists of one image
    ++*launches;
    const int lgrid = (ntiles + kThreads - 1) / kThreads;
    const cudaError_t e =
        vm == nullptr  // candidates for the image's extremes (global normalisation on the fast path)
            ? launch_pdl(k_extreme_list, lgrid, kThreads, 0, s, vx_fast, opaque, g, (int)g.C, *band, minmax, list, count)
            : launch_pdl(k_band_list, lgrid, kThreads, 0, s, vx_fast, opaque, g, (int)g.C, *vm, *thr, *band, minmax, list, count);
    if (e != cudaSuccess) return e;
  }
  ++*launches;
  // few listed tiles: one CTA per tile (latency); every tile: three narrow CTAs per SM (throughput).  A list can hold
  // anything between a handful and all tiles (an image whose values all sit at the extremes): the grid covers both.
  const int threads = banded ? kExactThreads : kThreads;
  const int grid = clamp_grid(ntiles, (long long)sm_count * (banded ? 2 : 3));
  return launch_pdl(g.C == 4 ? k_mad_exact<4> : k_mad_exact<3>, grid, threads, (size_t)4 * kExactStride * sizeof(float), s, img, pitch, g, vx,
                    banded ? list : nullptr, count);
}

// cuTensorMapEncodeTiled through the runtime (the library links cudart statically and has no libcuda dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// the pitched RGBA8 image as a 2-D tensor of 32-bit pixels, box = 64 px x box_rows rows
static bool make_image_tmap(const uint8_t* img, size_t pitch, uint32_t W, uint32_t H, CUtensorMap* tm, uint32_t box_rows = kTBoxRows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t dims[2] = {W, H};
  const cuuint64_t strides[1] = {pitch};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<uint8_t*>(img), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t launch_analyze_sobel(const uint8_t* img, size_t pitch, const Geom& g, float* vx, float* vy, cudaStream_t s,
                                 int sm_count, uint64_t* launches) {
  const uint32_t ntiles = g.cols * g.rows;
  ++*launches;
  // RGBA, 64x64 tiles, rows a tensor copy can address: tiles streamed by TMA, dp4a row terms (analyze_sobel_tma.cuh)
  if (g.C == 4 && g.bw == 64 && g.bh == 64 && (pitch % 16 == 0) && ((reinterpret_cast<uintptr_t>(img) & 15u) == 0)) {
    CUtensorMap tm;
    if (make_image_tmap(img, pitch, g.W, g.nimg > 1 ? (g.nimg - 1) * g.img_rows + g.H : g.H, &tm, 64))
      return launch(k_analyze_sobel_tma, clamp_grid(ntiles, (long long)sm_count * PXZ_SOBEL_CTAS), 256, kSobSmemBytes, s, tm, g, vx, vy);
  }
  const bool small = g.bw <= 64 && g.bh <= 64 && (g.C == 3 || ((pitch & 3u) == 0 && (reinterpret_cast<uintptr_t>(img) & 3u) == 0));
  const auto k = small ? (g.C == 4 ? k_analyze_sobel_tile64<4> : k_analyze_sobel_tile64<3>) : (g.C == 4 ? k_analyze_sobel<4> : k_analyze_sobel<3>);
  return launch(k, clamp_grid(ntiles, sm_count * 8), kThreads, 0, s, img, pitch, g, vx, vy);
}

cudaError_t launch_tree_mask(const float* vx, const Geom& g, const uint8_t* parent_recurse, uint32_t parent_cols, float thr,
                             int positive, uint8_t* leaf, uint8_t* recurse, cudaStream_t s, uint64_t* launches) {
  const uint32_t n = g.cols * g.rows;
  ++*launches;
  return launch(k_tree_mask, (n + kThreads - 1) / kThreads, kThreads, 0, s, vx, g, parent_recurse, parent_cols, thr, positive, leaf, recurse);
}

cudaError_t launch_minmax(const float* vx, const float* vy, uint32_t n, float* minmax4, cudaStream_t s, uint64_t* launches) {
  ++*launches;
  return launch(k_minmax, 1, 1024, 0, s, vx, vy, n, minmax4);
}

// layout: class_hist[16] | ScanState
constexpr size_t kClassHistBytes = 2 * kCostClasses * sizeof(uint32_t);
size_t plan_scan_state_bytes(uint32_t nblocks) {
  const uint32_t tiles = (nblocks + kPlanTile - 1) / kPlanTile;
  return kClassHistBytes + sizeof(ScanState) + (size_t)tiles * sizeof(unsigned long long);
}

cudaError_t launch_plan(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                        const LevelThresholds& thr, const uint8_t* mask, pxz_block_desc* descs, uint32_t* tabidx,
                        uint64_t* total_bytes, void* scan_state, uint32_t* lists, uint32_t cap, cudaStream_t s, uint64_t* launches,
                        const StrategyLut* strategy, uint32_t* tabidx_up) {
  const uint32_t nblocks = g.cols * g.rows;
  const uint32_t tiles = (nblocks + kPlanTile - 1) / kPlanTile;
  const bool adaptive = strategy != nullptr && strategy->on != 0 && tabidx_up != nullptr;
  StrategyLut lut = {};
  if (adaptive) lut = *strategy;
  // scan_state is zero on entry and on exit (ensure_scratch clears it once)
  ++*launches;
  uint32_t* cursor = reinterpret_cast<uint32_t*>(scan_state);
  ScanState* st = reinterpret_cast<ScanState*>(reinterpret_cast<uint8_t*>(scan_state) + kClassHistBytes);
  return launch_pdl(adaptive ? k_plan<true> : k_plan<false>, tiles, kThreads, 0, s, vx, vy, g, vm, minmax, thr, mask, descs, tabidx,
                    reinterpret_cast<unsigned long long*>(total_bytes), st, cursor, lists, cap, lut, tabidx_up);
}

cudaError_t launch_size_curve(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                              const LevelThresholds& thr, uint32_t bpp, const SizeCandidates& cand, uint64_t* bytes, cudaStream_t s,
                              int sm_count, uint64_t* launches) {
  if (cand.n == 0 || cand.n > (uint32_t)kMaxSizeCandidates) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(bytes, 0, (size_t)cand.n * sizeof(uint64_t), s);
  if (e != cudaSuccess) return e;
  const uint32_t nblocks = g.cols * g.rows;
  const int gx = clamp_grid(((long long)nblocks + kThreads * kSizeItems - 1) / (kThreads * kSizeItems), 1ll << 30);
  // few blocks: split the candidates over more CTAs (at least 8 candidates per CTA) to fill the SMs
  const int gy = clamp_grid(std::min<long long>((long long)sm_count * 2 / gx, cand.n / 8), 32);
  ++*launches;
  return launch(k_size_curve, dim3(gx, gy), kThreads, 0, s, vx, vy, g, vm, minmax, thr, bpp, cand, reinterpret_cast<unsigned long long*>(bytes));
}

size_t window_scan_state_bytes(uint32_t nblocks) {
  const uint32_t tiles = (nblocks + kWindowTile - 1) / kWindowTile;
  return kClassHistBytes + sizeof(ScanState) + (size_t)tiles * sizeof(unsigned long long);
}

cudaError_t launch_payload_window(const pxz_block_desc* pdescs, const uint32_t* pmeta, uint32_t pcap, const uint8_t* ppx, uint32_t pcols,
                                  uint32_t c0, uint32_t r0, const Geom& g, bool copy_up, pxz_block_desc* descs, uint32_t* meta, uint32_t cap,
                                  uint8_t* px, uint64_t* total_bytes, void* scan_state, cudaStream_t s, uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  uint32_t* cursor = reinterpret_cast<uint32_t*>(scan_state);  // zero on entry and on exit
  ScanState* st = reinterpret_cast<ScanState*>(reinterpret_cast<uint8_t*>(scan_state) + kClassHistBytes);
  ++*launches;
  return launch(k_payload_window, (nblocks + kWindowTile - 1) / kWindowTile, kThreads, 0, s, pdescs, pmeta, pcap, ppx, pcols, c0, r0, g,
                copy_up ? 1 : 0, descs, meta, cap, px, reinterpret_cast<unsigned long long*>(total_bytes), st, cursor);
}

cudaError_t launch_class_lists(const pxz_block_desc* descs, const Geom& g, void* scan_state, uint32_t* lists, uint32_t cap,
                               cudaStream_t s, uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  uint32_t* cursor = reinterpret_cast<uint32_t*>(scan_state);  // zero on entry and on exit
  ++*launches;
  return launch(k_class_lists, (nblocks + kThreads - 1) / kThreads, kThreads, 0, s, descs, g, cursor, lists, cap);
}

size_t resample_smem_bytes(uint32_t max_src_px, uint32_t max_tmp_px, uint32_t C) {
  return ((size_t)max_src_px + max_tmp_px) * C * sizeof(float);
}

int resample_grid(int sm_count, uint32_t nblocks) { return clamp_grid(nblocks, (long long)sm_count * 8); }

cudaError_t launch_resample(const ResampleArgs& a, cudaStream_t s, int sm_count, uint64_t* launches) {
  const Geom& g = a.g;
  ++*launches;
  // RGBA fast paths: tiles <= 64x64 with 16-byte aligned rows
  const bool fast = g.C == 4 && g.bw <= 64 && g.bh <= 64 && (g.bw % 4 == 0) && (g.W % 4 == 0) && (a.pitch % 16 == 0) &&
                    ((reinterpret_cast<uintptr_t>(a.img) & 15u) == 0) && a.max_src_px <= (uint32_t)kFastMaxPx && a.max_src_dim <= 64u &&
                    a.max_tmp_px <= (uint32_t)kFastMaxPx && a.max_tab_words <= (uint32_t)kFastMaxTabWords &&
                    a.ntabs <= (uint32_t)kFastMaxTabs && a.scratch == nullptr;
  // warp-per-tile kernels (resample_warp.cuh, resample_tma.cuh) once there are enough tiles to keep every warp slot of
  // the GPU busy for a few tiles; below that one tile's latency (15-40 us on one warp) decides and 8 warps per tile
  // finish sooner.  a.kernels forces a family (ResampleKernels).
  const long long ntiles = (long long)g.cols * g.rows;
  if (fast && a.warp_tables && a.kernels != ResampleKernels::Cta &&
      (a.kernels == ResampleKernels::Warp || ntiles >= (long long)sm_count * 16)) {
    if (a.direction == 1) {
      const int wgrid = clamp_grid((ntiles + kWarpsPerCta - 1) / kWarpsPerCta, (long long)sm_count * PXZ_EXPAND_WARP_CTAS);
      return launch_pdl(a.fused ? k_expand_warp<true> : k_expand_warp<false>, wgrid, kWarpCtaThreads, (size_t)kWarpsPerCta * kExpandWarpBytes,
                        s, a.img, a.pitch, g, a.descs, a.tabidx, a.lists, a.cap, a.payload, a.tabs, a.pool, a.tile_counter, 1.0f, -0.0f);
    }
    // an image no tensor map can address (driver entry point missing, beyond the tensor-map limits) takes the
    // CTA-per-tile kernel below
    CUtensorMap tm;
    if (make_image_tmap(a.img, a.pitch, g.W, g.nimg > 1 ? (g.nimg - 1) * g.img_rows + g.H : g.H, &tm)) {
      const int tgrid = clamp_grid((ntiles + kTWarps - 1) / kTWarps, (long long)sm_count * PXZ_SHRINK_TMA_CTAS);
      const cudaError_t e = launch_pdl(a.fused ? k_shrink_tma<true> : k_shrink_tma<false>, tgrid, kTWarps * 32, (size_t)kTWarps * kTWarpBytes, s, tm,
                                       g, a.descs, a.tabidx, a.lists, a.cap, a.opaque_flags, a.payload, a.tabs, a.ntabs, a.pool, a.tile_counter,
                                       1.0f, -0.0f);
      if (e != cudaSuccess || !a.has_noslide) return e;
      ++*launches;  // the tiles whose vertical table has no slide2 form
      const int wgrid = clamp_grid((ntiles + kShrinkWarps - 1) / kShrinkWarps, (long long)sm_count * PXZ_SHRINK_WARP_CTAS);
      return launch_pdl(a.fused ? k_shrink_warp<true> : k_shrink_warp<false>, wgrid, kShrinkCtaThreads, (size_t)kShrinkWarps * kShrinkWarpBytes, s,
                        a.img, a.pitch, g, a.descs, a.tabidx, a.lists, a.cap, a.opaque_flags, a.payload, a.tabs, a.pool, a.tile_counter, 1.0f, -0.0f);
    }
  }
  if (fast) {
    const int fgrid = clamp_grid(ntiles, (long long)sm_count * PXZ_RESAMPLE_MINBLOCKS);
    const size_t smem = fast_smem_bytes(a.max_tmp_px);
    if (a.direction == 0)
      return launch(a.fused ? k_shrink_rgba<true> : k_shrink_rgba<false>, fgrid, kThreads, smem, s, a.img, a.pitch, g, a.descs, a.tabidx, a.payload,
                    a.tabs, a.ntabs, a.pool, a.max_tmp_px, 1.0f, -0.0f);
    return launch(a.fused ? k_expand_rgba<true> : k_expand_rgba<false>, fgrid, kThreads, smem, s, a.img, a.pitch, g, a.descs, a.tabidx, a.payload,
                  a.tabs, a.ntabs, a.pool, a.max_tmp_px, 1.0f, -0.0f);
  }
  const size_t smem = a.scratch ? 0 : resample_smem_bytes(a.max_src_px, a.max_tmp_px, g.C);
  return launch(g.C == 4 ? k_resample<4> : k_resample<3>, a.grid, kThreads, smem, s, a.direction, a.img, a.pitch, g, a.descs, a.tabidx, a.payload,
                a.tabs, a.pool, a.max_src_px, a.max_tmp_px, a.scratch, a.scratch_per_cta);
}

// ------------------------------------------------------------------------------------------------
// RGB (3-channel) images on the RGBA fast kernels: an RGB image is widened to RGBA with alpha 255 (the 4-channel
// metric's alpha term is then exactly +0 and the opaque resample path never touches alpha, so every value and pixel is
// bit-identical to the 3-channel computation), processed, and the payload narrowed back.  Three streaming kernels.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_rgb_to_rgba(const uint8_t* __restrict__ src, size_t spitch, uint8_t* __restrict__ dst,
                                                          size_t dpitch, uint32_t w, uint32_t rows) {
  // 4 pixels per thread: 12 bytes in, 16 bytes out
  const uint32_t quads = (w + 3) / 4;
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < (size_t)quads * rows; i += (size_t)gridDim.x * kThreads) {
    const uint32_t y = (uint32_t)(i / quads), q = (uint32_t)(i - (size_t)y * quads);
    const uint8_t* s = src + (size_t)y * spitch + (size_t)q * 12;
    uint32_t* d = reinterpret_cast<uint32_t*>(dst + (size_t)y * dpitch) + (size_t)q * 4;
    const uint32_t n = min(4u, w - q * 4);
    for (uint32_t k = 0; k < n; ++k) d[k] = (uint32_t)s[3 * k] | ((uint32_t)s[3 * k + 1] << 8) | ((uint32_t)s[3 * k + 2] << 16) | 0xFF000000u;
  }
}
__global__ void __launch_bounds__(kThreads) k_rgba_to_rgb(const uint8_t* __restrict__ src, size_t spitch, uint8_t* __restrict__ dst,
                                                          size_t dpitch, uint32_t w, uint32_t rows) {
  const uint32_t quads = (w + 3) / 4;
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < (size_t)quads * rows; i += (size_t)gridDim.x * kThreads) {
    const uint32_t y = (uint32_t)(i / quads), q = (uint32_t)(i - (size_t)y * quads);
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src + (size_t)y * spitch) + (size_t)q * 4;
    uint8_t* d = dst + (size_t)y * dpitch + (size_t)q * 12;
    const uint32_t n = min(4u, w - q * 4);
    for (uint32_t k = 0; k < n; ++k) {
      const uint32_t p = s[k];
      d[3 * k] = (uint8_t)p; d[3 * k + 1] = (uint8_t)(p >> 8); d[3 * k + 2] = (uint8_t)(p >> 16);
    }
  }
}
// payload + metadata of one channel count -> the other: block pixels (a warp per block), descriptors with rescaled
// offsets (a block's offset is a multiple of its channel count), table indices, work-order lists, total
__global__ void __launch_bounds__(kThreads) k_payload_convert(const pxz_block_desc* __restrict__ sdescs, const uint8_t* __restrict__ spx,
                                                              const uint32_t* __restrict__ smeta, uint32_t scap, const unsigned long long* stotal,
                                                              pxz_block_desc* __restrict__ ddescs, uint8_t* __restrict__ dpx,
                                                              uint32_t* __restrict__ dmeta, uint32_t dcap, unsigned long long* dtotal,
                                                              uint32_t nblocks, int sc, int dc) {
  const uint32_t lane = threadIdx.x & 31u, wpc = kThreads / 32;
  for (uint32_t b = blockIdx.x * wpc + (threadIdx.x >> 5); b < nblocks; b += gridDim.x * wpc) {
    const pxz_block_desc d = sdescs[b];
    const unsigned long long doff = d.offset / (unsigned)sc * (unsigned)dc;
    if (lane == 0) {
      pxz_block_desc o = d;
      o.offset = doff;
      ddescs[b] = o;
      dmeta[b] = smeta[b];                                                         // tabidx
      dmeta[(size_t)dcap + order_list_words(dcap) + b] = smeta[(size_t)scap + order_list_words(scap) + b];  // expand-side indices
    }
    const uint32_t npx = (uint32_t)d.w * d.h;
    const uint8_t* s = spx + d.offset;
    uint8_t* o = dpx + doff;
    if (sc == 4) {
      for (uint32_t i = lane; i < npx; i += 32) {
        const uint32_t p = reinterpret_cast<const uint32_t*>(s)[i];
        o[3 * i] = (uint8_t)p; o[3 * i + 1] = (uint8_t)(p >> 8); o[3 * i + 2] = (uint8_t)(p >> 16);
      }
    } else {
      for (uint32_t i = lane; i < npx; i += 32)
        reinterpret_cast<uint32_t*>(o)[i] = (uint32_t)s[3 * i] | ((uint32_t)s[3 * i + 1] << 8) | ((uint32_t)s[3 * i + 2] << 16) | 0xFF000000u;
    }
  }
  // work-order lists: lists[c * cap + i], then the 8 class counts
  const uint32_t* sl = smeta + scap;
  uint32_t* dl = dmeta + dcap;
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < (size_t)kOrderClasses * nblocks + kOrderClasses; i += (size_t)gridDim.x * kThreads) {
    if (i < (size_t)kOrderClasses * nblocks) {
      const uint32_t c = (uint32_t)(i / nblocks), k = (uint32_t)(i - (size_t)c * nblocks);
      dl[(size_t)c * dcap + k] = sl[(size_t)c * scap + k];
    } else {
      const uint32_t c = (uint32_t)(i - (size_t)kOrderClasses * nblocks);
      dl[(size_t)kOrderClasses * dcap + c] = sl[(size_t)kOrderClasses * scap + c];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *dtotal = *stotal / (unsigned)sc * (unsigned)dc;
}

// ------------------------------------------------------------------------------------------------
// per-block error of two images of one geometry (pxz_image_error, pxz_strategy_measure).  Integer arithmetic only: per 4 bytes
// one VABSDIFF4 (|a - b| per byte) and one IDP.4A (sum of the four squares), __vmaxu4 for the largest difference.  A work item is
// a band of at most kErrRows rows inside one block row times kThreads consecutive units of a row; a thread keeps the same unit
// in every row of its band, so its byte range maps to the same block column(s) and it sums in registers (u32: at most
// 32 rows x 16 bytes x 255^2 < 2^32).  Units: 16 aligned bytes (kVec: both images' rows start 16-byte aligned and a block
// row is >= 16 bytes, so a unit straddles at most one block-column edge) or one pixel (any pitch, any block width).  The
// thread's sums go to shared per-column slots, then one 64-bit atomicAdd per block column and work item: integer sums, so the
// result does not depend on the order.  sse[] / mx[] are zero on entry; trailing tiles count their real pixels only.
// ------------------------------------------------------------------------------------------------
constexpr int kErrRows = 32;
constexpr int kErrCols = kThreads + 2;  // block columns one work item can touch (units of >= 16 bytes or one pixel)

// the 16 bytes at p (only the first n when n < 16: the unit at the end of a row must not read past it), as 4 words
__device__ __forceinline__ uint4 load_unit(const uint8_t* p, uint32_t n) {
  if (n == 16) return ldg_nc_v4(p);
  uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
  for (uint32_t i = 0; i < 16; ++i)  // unrolled: the words stay in registers
    if (i < n) w[i >> 2] |= (uint32_t)__ldg(p + i) << (8 * (i & 3));
  return make_uint4(w[0], w[1], w[2], w[3]);
}
// bytes [0, k) of a 16-byte unit as 4 word masks' word i
__device__ __forceinline__ uint32_t lead_mask(uint32_t k, int i) {
  const int n = (int)k - 4 * i;
  return n <= 0 ? 0u : (n >= 4 ? 0xFFFFFFFFu : (1u << (8 * n)) - 1u);
}

template <bool kVec>
__global__ void __launch_bounds__(kThreads) k_block_error(const uint8_t* __restrict__ a, size_t pa, const uint8_t* __restrict__ b, size_t pb,
                                                          Geom g, uint32_t units, uint32_t ux, uint32_t bands_per_row,
                                                          unsigned long long nwork, unsigned long long* __restrict__ sse,
                                                          uint32_t* __restrict__ mx) {
  __shared__ unsigned long long s_sse[kErrCols];
  __shared__ uint32_t s_max[kErrCols];
  const uint32_t tid = threadIdx.x;
  const uint32_t rowb = g.W * g.C, bwc = g.bw * g.C;
  for (unsigned long long w = blockIdx.x; w < nwork; w += gridDim.x) {
    const uint32_t cx = (uint32_t)(w % ux);
    const unsigned long long band = w / ux;
    const uint32_t by = (uint32_t)(band / bands_per_row), k = (uint32_t)(band - (unsigned long long)by * bands_per_row);
    const unsigned long long ytop = (unsigned long long)by * g.bh;
    const unsigned long long y0 = ytop + (unsigned long long)k * kErrRows;
    const unsigned long long y1 = min(min(y0 + kErrRows, ytop + g.bh), (unsigned long long)g.H);
    if (y0 >= y1) continue;  // the last band of a trailing block row: uniform over the CTA
    const uint32_t u0 = cx * kThreads;
    const uint32_t bc_first = (kVec ? u0 * 16u : u0 * g.C) / bwc;
    for (uint32_t i = tid; i < kErrCols; i += kThreads) {
      s_sse[i] = 0ull;
      s_max[i] = 0u;
    }
    __syncthreads();
    const uint32_t u = u0 + tid;
    if (u < units) {
      const uint32_t xb = kVec ? u * 16u : u * g.C;
      const uint32_t bc = xb / bwc;
      const uint8_t* pa0 = a + (size_t)y0 * pa + xb;
      const uint8_t* pb0 = b + (size_t)y0 * pb + xb;
      const uint32_t nrows = (uint32_t)(y1 - y0);
      uint32_t acc = 0u, m = 0u, acc2 = 0u, m2 = 0u;  // second column: the bytes of a 16-byte unit past a block-column edge
      uint32_t split = 16u;
      if (kVec) {
        const uint32_t n = min(16u, rowb - xb);
        split = min((bc + 1u) * bwc - xb, n);  // bytes of the unit in column bc
        if (n == 16u && split == 16u) {
#pragma unroll 4
          for (uint32_t r = 0; r < nrows; ++r) {
            const uint4 va = ldg_nc_v4(pa0 + (size_t)r * pa), vb = ldg_nc_v4(pb0 + (size_t)r * pb);
            const uint32_t d0 = __vabsdiffu4(va.x, vb.x), d1 = __vabsdiffu4(va.y, vb.y);
            const uint32_t d2 = __vabsdiffu4(va.z, vb.z), d3 = __vabsdiffu4(va.w, vb.w);
            acc = __dp4a(d0, d0, acc);
            acc = __dp4a(d1, d1, acc);
            acc = __dp4a(d2, d2, acc);
            acc = __dp4a(d3, d3, acc);
            m = __vmaxu4(m, __vmaxu4(__vmaxu4(d0, d1), __vmaxu4(d2, d3)));
          }
        } else {  // the unit at the end of a row or across a block-column edge
          uint32_t lo[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) lo[i] = lead_mask(split, i);
          for (uint32_t r = 0; r < nrows; ++r) {
            const uint4 va = load_unit(pa0 + (size_t)r * pa, n), vb = load_unit(pb0 + (size_t)r * pb, n);
            const uint32_t d[4] = {__vabsdiffu4(va.x, vb.x), __vabsdiffu4(va.y, vb.y), __vabsdiffu4(va.z, vb.z), __vabsdiffu4(va.w, vb.w)};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t dl = d[i] & lo[i], dh = d[i] & ~lo[i];
              acc = __dp4a(dl, dl, acc);
              acc2 = __dp4a(dh, dh, acc2);
              m = __vmaxu4(m, dl);
              m2 = __vmaxu4(m2, dh);
            }
          }
        }
      } else {
        const uint32_t C = g.C;
        for (uint32_t r = 0; r < nrows; ++r) {
          const uint8_t* qa = pa0 + (size_t)r * pa;
          const uint8_t* qb = pb0 + (size_t)r * pb;
          uint32_t wa = 0u, wb = 0u;
          for (uint32_t c = 0; c < C; ++c) {
            wa |= (uint32_t)__ldg(qa + c) << (8 * c);
            wb |= (uint32_t)__ldg(qb + c) << (8 * c);
          }
          const uint32_t d = __vabsdiffu4(wa, wb);
          acc = __dp4a(d, d, acc);
          m = __vmaxu4(m, d);
        }
      }
      auto bytes_max = [](uint32_t v) { return max(max(v & 0xFFu, (v >> 8) & 0xFFu), max((v >> 16) & 0xFFu, v >> 24)); };
      if (acc) atomicAdd(&s_sse[bc - bc_first], (unsigned long long)acc);
      if (m) atomicMax(&s_max[bc - bc_first], bytes_max(m));
      if (acc2) atomicAdd(&s_sse[bc + 1u - bc_first], (unsigned long long)acc2);
      if (m2) atomicMax(&s_max[bc + 1u - bc_first], bytes_max(m2));
    }
    __syncthreads();
    const uint32_t u_end = min(u0 + (uint32_t)kThreads, units);
    const uint32_t last_byte = (kVec ? min(u_end * 16u, rowb) : u_end * g.C) - 1u;
    const uint32_t ncols = last_byte / bwc - bc_first + 1u;
    for (uint32_t i = tid; i < ncols; i += kThreads) {
      const size_t blk = (size_t)by * g.cols + bc_first + i;
      if (s_sse[i]) atomicAdd(&sse[blk], s_sse[i]);
      if (mx && s_max[i]) atomicMax(&mx[blk], s_max[i]);
    }
    __syncthreads();  // the slots are cleared for the next work item
  }
}

// strategy measure: the block errors of one (down, up) pair added into sse[bucket * kFilterPairs + pair], the bucket taken from
// the value the plan stored in the block's descriptor; count: also the block histogram.  A shared histogram per CTA, then one
// global add per bucket.
__global__ void __launch_bounds__(kThreads) k_bucket_sum(const pxz_block_desc* __restrict__ descs, const unsigned long long* __restrict__ block_sse,
                                                         uint32_t nblocks, uint32_t pair, int count, unsigned long long* __restrict__ sse,
                                                         uint32_t* __restrict__ blocks) {
  __shared__ unsigned long long s_sse[kStrategyBuckets];
  __shared__ uint32_t s_n[kStrategyBuckets];
  for (int i = threadIdx.x; i < kStrategyBuckets; i += kThreads) {
    s_sse[i] = 0ull;
    s_n[i] = 0u;
  }
  __syncthreads();
  for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < nblocks; i += gridDim.x * kThreads) {
    const uint32_t k = strategy_bucket(descs[i].value);
    const unsigned long long e = block_sse[i];
    if (e) atomicAdd(&s_sse[k], e);
    if (count) atomicAdd(&s_n[k], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kStrategyBuckets; i += kThreads) {
    if (s_sse[i]) atomicAdd(&sse[(size_t)i * kFilterPairs + pair], s_sse[i]);
    if (count && s_n[i]) atomicAdd(&blocks[i], s_n[i]);
  }
}

cudaError_t launch_block_error(const uint8_t* a, size_t pa, const uint8_t* b, size_t pb, const Geom& g, uint64_t* sse, uint32_t* mx,
                               cudaStream_t s, int sm_count, uint64_t* launches) {
  const bool vec = (((uintptr_t)a | (uintptr_t)b | pa | pb) & 15u) == 0 && g.bw * g.C >= 16u;
  const uint32_t units = vec ? (g.W * g.C + 15u) / 16u : g.W;
  const uint32_t ux = (units + kThreads - 1) / kThreads;
  const uint32_t bands_per_row = (g.bh + kErrRows - 1) / kErrRows;
  const unsigned long long nwork = (unsigned long long)g.rows * bands_per_row * ux;
  const int grid = clamp_grid((long long)std::min<unsigned long long>(nwork, 1ull << 30), (long long)sm_count * 16);
  ++*launches;
  return launch(vec ? k_block_error<true> : k_block_error<false>, grid, kThreads, 0, s, a, pa, b, pb, g, units, ux, bands_per_row, nwork,
                reinterpret_cast<unsigned long long*>(sse), mx);
}

cudaError_t launch_bucket_sum(const pxz_block_desc* descs, const uint64_t* block_sse, uint32_t nblocks, uint32_t pair, bool count,
                              uint64_t* sse, uint32_t* blocks, cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const int grid = clamp_grid(((long long)nblocks + kThreads - 1) / kThreads, (long long)sm_count * 2);
  return launch(k_bucket_sum, grid, kThreads, 0, s, descs, reinterpret_cast<const unsigned long long*>(block_sse), nblocks, pair, count ? 1 : 0,
                reinterpret_cast<unsigned long long*>(sse), blocks);
}

cudaError_t launch_rgb_widen(const uint8_t* src, size_t spitch, uint8_t* dst, size_t dpitch, uint32_t w, uint32_t rows, int widen,
                             cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const long long quads = (long long)((w + 3) / 4) * rows;
  const int grid = clamp_grid((quads + kThreads - 1) / kThreads, (long long)sm_count * 8);
  return launch(widen ? k_rgb_to_rgba : k_rgba_to_rgb, grid, kThreads, 0, s, src, spitch, dst, dpitch, w, rows);
}

cudaError_t launch_payload_convert(const pxz_block_desc* sdescs, const uint8_t* spx, const uint32_t* smeta, uint32_t scap,
                                   const uint64_t* stotal, pxz_block_desc* ddescs, uint8_t* dpx, uint32_t* dmeta, uint32_t dcap,
                                   uint64_t* dtotal, uint32_t nblocks, int sc, int dc, cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const int grid = clamp_grid(((long long)nblocks + 7) / 8, (long long)sm_count * 8);
  return launch(k_payload_convert, grid, kThreads, 0, s, sdescs, spx, smeta, scap, reinterpret_cast<const unsigned long long*>(stotal), ddescs, dpx,
                dmeta, dcap, reinterpret_cast<unsigned long long*>(dtotal), nblocks, sc, dc);
}

cudaError_t launch_rd_levels(float* vx, float* vy, uint32_t n, float fx, float fy, cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const int grid = clamp_grid(((long long)n + kThreads - 1) / kThreads, (long long)sm_count * 8);
  return launch(k_rd_levels, grid, kThreads, 0, s, vx, vy, n, fx, fy);
}

cudaError_t launch_rd_events(const float* vx, const float* vy, const Geom& g, const ValueMap& vm, const float* minmax,
                             const LevelThresholds& thr, uint32_t bpp, const uint64_t* sse_table, const RdPasses& ps, uint32_t maxev,
                             uint32_t* keys, uint32_t* ids, uint64_t* dbytes, uint64_t* dsse, uint64_t* base, cudaStream_t s,
                             uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  ++*launches;
  return launch(k_rd_events, (nblocks + kThreads - 1) / kThreads, kThreads, 0, s, vx, vy, g, vm, minmax, thr, bpp,
                reinterpret_cast<const unsigned long long*>(sse_table), ps, maxev, keys, ids, reinterpret_cast<unsigned long long*>(dbytes),
                reinterpret_cast<unsigned long long*>(dsse), reinterpret_cast<unsigned long long*>(base));
}

// scratch of launch_rd_curve: sorted keys | sorted ids | last-of-key flags | point indices | scan input | scan output | CUB's
// temporary storage
static size_t rd_cub_bytes(uint32_t nev) {
  size_t sort = 0, scan = 0, count = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (int)nev, 0, 32);
  cub::DeviceScan::InclusiveScan(nullptr, scan, (const RdAcc*)nullptr, (RdAcc*)nullptr, RdAccSum(), (int)nev);
  cub::DeviceScan::InclusiveSum(nullptr, count, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)nev);
  return std::max(sort, std::max(scan, count));
}
struct RdCurveScratch {
  uint32_t *skeys = nullptr, *sids = nullptr, *last = nullptr, *points = nullptr;
  RdAcc *acc = nullptr, *sums = nullptr;
  uint8_t* cub = nullptr;
  size_t cub_bytes = 0;
};
static auto rd_curve_layout(uint32_t nev, RdCurveScratch& sc) {
  sc.cub_bytes = rd_cub_bytes(nev);
  return layout_of(part(sc.skeys, nev), part(sc.sids, nev), part(sc.last, nev), part(sc.points, nev), part(sc.acc, nev), part(sc.sums, nev),
                   part(sc.cub, sc.cub_bytes));
}
size_t rd_curve_scratch_bytes(uint32_t nev) {
  RdCurveScratch sc;
  return rd_curve_layout(nev, sc).bytes();
}

cudaError_t launch_rd_curve(const uint32_t* keys, const uint32_t* ids, const uint64_t* dbytes, const uint64_t* dsse, uint32_t nev,
                            const uint64_t* base, uint64_t max_sse, void* scratch, size_t scratch_bytes, uint32_t* pt_key, uint64_t* pt_bytes,
                            uint64_t* pt_sse, RdOut* out, cudaStream_t s, int sm_count, uint64_t* launches) {
  RdCurveScratch sc;
  const auto lay = rd_curve_layout(nev, sc);
  if (scratch_bytes < lay.bytes() || nev > 0x7FFFFFFFu) return cudaErrorInvalidValue;
  lay.place(scratch);
  size_t cub_bytes = sc.cub_bytes;
  cudaError_t e = cudaMemsetAsync(out, 0xFF, sizeof(RdOut), s);
  const int grid = clamp_grid(((long long)nev + kThreads - 1) / kThreads, (long long)sm_count * 8);
  if (e == cudaSuccess && nev > 0) {
    // sort, gather, two scans: CUB's sort and scans launch several kernels each and count as one launch here
    *launches += 4;
    e = cub::DeviceRadixSort::SortPairs(sc.cub, cub_bytes, keys, sc.skeys, ids, sc.sids, (int)nev, 0, 32, s);
    if (e == cudaSuccess) e = launch(k_rd_gather, grid, kThreads, 0, s, sc.skeys, sc.sids, reinterpret_cast<const unsigned long long*>(dbytes),
                                     reinterpret_cast<const unsigned long long*>(dsse), nev, sc.acc, sc.last);
    if (e == cudaSuccess) {
      cub_bytes = sc.cub_bytes;
      e = cub::DeviceScan::InclusiveScan(sc.cub, cub_bytes, sc.acc, sc.sums, RdAccSum(), (int)nev, s);
    }
    if (e == cudaSuccess) {
      cub_bytes = sc.cub_bytes;
      e = cub::DeviceScan::InclusiveSum(sc.cub, cub_bytes, sc.last, sc.points, (int)nev, s);
    }
  }
  if (e != cudaSuccess) return e;
  ++*launches;
  return launch(k_rd_compact, grid, kThreads, 0, s, sc.skeys, sc.sums, sc.points, nev, reinterpret_cast<const unsigned long long*>(base),
                (unsigned long long)max_sse, pt_key, reinterpret_cast<unsigned long long*>(pt_bytes), reinterpret_cast<unsigned long long*>(pt_sse),
                out);
}

cudaError_t launch_rdo_hull(const uint64_t* sse_table, const Geom& g, uint32_t bpp, uint32_t lx_max, uint32_t ly_max, uint32_t maxev, RdoEvent* ev,
                            uint32_t* ids, uint32_t* ev_pass, uint32_t* pass0, uint64_t* base, cudaStream_t s, uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  // 20 bytes per candidate and thread: 128 threads while that fits 96 KB (13 candidates at 64 x 64), fewer for very large blocks
  const size_t per_thread = (size_t)(maxev + 1) * 20;
  int threads = kRdoHullThreads;
  while (threads > 32 && per_thread * threads > 96 * 1024) threads /= 2;
  if (per_thread * threads > 200 * 1024) return cudaErrorInvalidValue;
  ++*launches;
  return launch(k_rdo_hull, (nblocks + threads - 1) / threads, threads, per_thread * threads, s,
                reinterpret_cast<const unsigned long long*>(sse_table), g, bpp, lx_max, ly_max, maxev, ev, ids, ev_pass, pass0,
                reinterpret_cast<unsigned long long*>(base));
}

// scratch of launch_rdo_curve: scan input | scan output | CUB's temporary storage (merge sort or scan)
static size_t rdo_cub_bytes(uint32_t nev) {
  size_t sort = 0, scan = 0;
  cub::DeviceMergeSort::StableSortPairs(nullptr, sort, (RdoEvent*)nullptr, (uint32_t*)nullptr, (int)nev, RdoRateDesc());
  cub::DeviceScan::InclusiveScan(nullptr, scan, (const RdAcc*)nullptr, (RdAcc*)nullptr, RdAccSum(), (int)nev);
  return std::max(sort, scan);
}
struct RdoCurveScratch {
  RdAcc *acc = nullptr, *sums = nullptr;
  uint8_t* cub = nullptr;
  size_t cub_bytes = 0;
};
static auto rdo_curve_layout(uint32_t nev, RdoCurveScratch& sc) {
  sc.cub_bytes = rdo_cub_bytes(nev);
  return layout_of(part(sc.acc, nev), part(sc.sums, nev), part(sc.cub, sc.cub_bytes));
}
size_t rdo_curve_scratch_bytes(uint32_t nev) {
  RdoCurveScratch sc;
  return rdo_curve_layout(nev, sc).bytes();
}

cudaError_t launch_rdo_curve(RdoEvent* ev, uint32_t* ids, uint32_t nev, const uint64_t* base, uint64_t max_bytes, uint64_t max_sse, void* scratch,
                             size_t scratch_bytes, uint32_t* rank, uint64_t* pt_bytes, uint64_t* pt_sse, RdoOut* out, cudaStream_t s, int sm_count,
                             uint64_t* launches) {
  RdoCurveScratch sc;
  const auto lay = rdo_curve_layout(nev, sc);
  if (scratch_bytes < lay.bytes() || nev > 0x7FFFFFFFu) return cudaErrorInvalidValue;
  lay.place(scratch);
  size_t cub_bytes = sc.cub_bytes;
  // best_within = 0 (none), first_within = all ones (none)
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(RdoOut), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(&out->first_within, 0xFF, sizeof(uint32_t), s);
  const int grid = clamp_grid(((long long)nev + kThreads) / kThreads, (long long)sm_count * 8);
  if (e == cudaSuccess && nev > 0) {
    // sort, gather, scan: CUB's sort and scan launch several kernels each and count as one launch here
    *launches += 3;
    e = cub::DeviceMergeSort::StableSortPairs(sc.cub, cub_bytes, ev, ids, (int)nev, RdoRateDesc(), s);
    if (e == cudaSuccess) e = launch(k_rdo_gather, grid, kThreads, 0, s, ev, ids, nev, sc.acc, rank);
    if (e == cudaSuccess) {
      cub_bytes = sc.cub_bytes;
      e = cub::DeviceScan::InclusiveScan(sc.cub, cub_bytes, sc.acc, sc.sums, RdAccSum(), (int)nev, s);
    }
  }
  if (e != cudaSuccess) return e;
  ++*launches;
  return launch(k_rdo_points, grid, kThreads, 0, s, ev, sc.sums, nev, reinterpret_cast<const unsigned long long*>(base),
                (unsigned long long)max_bytes, (unsigned long long)max_sse, reinterpret_cast<unsigned long long*>(pt_bytes),
                reinterpret_cast<unsigned long long*>(pt_sse), out);
}

cudaError_t launch_rdo_levels(const uint32_t* pass0, const uint32_t* ev_pass, const uint32_t* rank, uint32_t maxev, uint32_t nblocks,
                              uint32_t ly_max, uint32_t j, float* vx, float* vy, cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const int grid = clamp_grid(((long long)nblocks + kThreads - 1) / kThreads, (long long)sm_count * 8);
  return launch(k_rdo_levels, grid, kThreads, 0, s, pass0, ev_pass, rank, maxev, nblocks, ly_max, j, vx, vy);
}

size_t resample_fir_smem_bytes(uint32_t max_src_px, uint32_t max_tmp_px, uint32_t C) {
  return (((size_t)max_src_px * C + 15) & ~(size_t)15) + (size_t)max_tmp_px * C;
}

cudaError_t launch_resample_fir(int direction, uint8_t* img, size_t pitch, const Geom& g, const pxz_block_desc* descs,
                                const uint32_t* tabidx, uint8_t* payload, const AxisTab* tabs, const uint32_t* pool, size_t smem,
                                uint32_t src_cap_bytes, cudaStream_t s, int sm_count, uint64_t* launches) {
  ++*launches;
  const int grid = clamp_grid((long long)g.cols * g.rows, (long long)sm_count * 8);
  return launch(g.C == 4 ? k_resample_fir<4> : k_resample_fir<3>, grid, kThreads, smem, s, direction, img, pitch, g, descs, tabidx, payload, tabs,
                pool, src_cap_bytes);
}

}  // namespace pxz
