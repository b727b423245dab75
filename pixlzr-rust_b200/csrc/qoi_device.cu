// qoi_device.cu — the container stage on the device (SURVEY.md §8f N1, second half): the per-block QOI streams of a
// .pxlzr file are written / read by the GPU straight from / into the packed payload, so that only the compressed bytes
// cross PCIe.  Byte-identical to the host stage (container.cpp), which restates src/encoding/mod.rs:40-242 and the
// qoi crate 0.4.1 (incl. its habit of writing a finished run of one pixel as QOI_OP_INDEX).
//
// QOI is sequential inside a block (running 64-entry colour table, previous pixel, run length) and blocks are small
// (<= 64 KB) and independent: one thread per block, 64-thread CTAs, the colour tables in shared memory (entry * 64 +
// thread: conflict free), output bytes gathered into aligned 32-bit words.  Encoding goes through worst-case slots
// (offset derived from the block's payload offset, no extra scan), a single-CTA scan turns the encoded lengths into
// file offsets and the per-row length table, and one warp per block moves the bytes to their place.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "pxz_internal.h"

namespace pxz {
namespace {

constexpr int kQoiThreads = 64;
constexpr uint32_t OP_INDEX = 0x00, OP_DIFF = 0x40, OP_LUMA = 0x80, OP_RUN = 0xC0, OP_RGB = 0xFE, OP_RGBA = 0xFF;
constexpr uint32_t kBlockHeader = 13;  // "block" + value f32 BE + qoi_len u32 BE (encoding/mod.rs:167-192)
constexpr uint32_t kQoiHeader = 10;    // width, height u32 BE, channels, colour space (no magic, :189-191)
constexpr uint32_t kFileHeader = 26;   // constants.rs:19-20

// worst case of one encoded block: 13 + 10 + (C + 1) bytes per pixel + 8 = 31 + npx * (C + 1); slots start 4-byte aligned
__host__ __device__ inline size_t slot_offset(uint64_t payload_off, uint32_t b, uint32_t C) {
  return (size_t)36 * b + (size_t)(((payload_off / C) * (C + 1)) & ~(uint64_t)3);
}

__device__ __forceinline__ uint32_t qoi_hash(uint32_t px) {
  return ((px & 255u) * 3u + ((px >> 8) & 255u) * 5u + ((px >> 16) & 255u) * 7u + (px >> 24) * 11u) & 63u;
}

struct WordWriter {  // appends bytes to a 4-byte aligned stream, one aligned store per word
  uint32_t* p;
  uint32_t acc = 0, n = 0;
  __device__ __forceinline__ void put(uint32_t v) {
    acc |= (v & 255u) << (8u * (n & 3u));
    if ((++n & 3u) == 0u) {
      p[(n >> 2) - 1u] = acc;
      acc = 0;
    }
  }
  __device__ __forceinline__ void put_be32(uint32_t v) { put(v >> 24); put(v >> 16); put(v >> 8); put(v); }
  __device__ __forceinline__ void flush() { if (n & 3u) p[n >> 2] = acc; }
};

template <int C>
__global__ void __launch_bounds__(kQoiThreads) k_qoi_encode(const pxz_block_desc* __restrict__ descs, const uint8_t* __restrict__ pixels,
                                                            uint32_t nblocks, int values_present, uint8_t* __restrict__ arena,
                                                            uint32_t* __restrict__ enc_len) {
  __shared__ uint32_t s_tab[64 * kQoiThreads];
  const int tid = threadIdx.x;
  for (int i = tid; i < 64 * kQoiThreads; i += kQoiThreads) s_tab[i] = 0u;
  __syncthreads();
  const uint32_t b = blockIdx.x * kQoiThreads + tid;
  if (b >= nblocks) return;
  const pxz_block_desc d = descs[b];
  uint8_t* slot = arena + slot_offset(d.offset, b, C);
  WordWriter w{reinterpret_cast<uint32_t*>(slot)};
  w.put('b'); w.put('l'); w.put('o'); w.put('c'); w.put('k');
  w.put_be32(values_present ? __float_as_uint(d.value) : 0u);  // encoding/mod.rs:173-178: None is written as 0.0
  w.put_be32(0u);                                             // qoi_len, patched below
  w.put_be32(d.w);
  w.put_be32(d.h);
  w.put(C);
  w.put(0);  // sRGB with linear alpha
  uint32_t* tab = s_tab + tid;  // entry e at tab[e * kQoiThreads]
  uint32_t last = 0xFF000000u, last_slot = qoi_hash(last), run = 0;
  bool seen_literal = false;
  const uint32_t npx = (uint32_t)d.w * d.h;
  const uint8_t* p = pixels + d.offset;
  // pixels are fetched eight at a time: the loop body is one long dependent chain, a load per iteration would add its
  // full latency to every pixel
  constexpr uint32_t kBatch = 8;
  uint32_t buf[kBatch];
  for (uint32_t i = 0; i < npx; ++i) {
    if ((i & (kBatch - 1)) == 0) {
#pragma unroll
      for (uint32_t j = 0; j < kBatch; ++j) {
        const uint32_t k = min(i + j, npx - 1);
        if (C == 4) buf[j] = reinterpret_cast<const uint32_t*>(p)[k];
        else buf[j] = (uint32_t)p[3 * k] | ((uint32_t)p[3 * k + 1] << 8) | ((uint32_t)p[3 * k + 2] << 16) | 0xFF000000u;
      }
    }
    uint32_t cur = buf[0];
#pragma unroll
    for (uint32_t j = 0; j < kBatch - 1; ++j) buf[j] = buf[j + 1];  // register shift: no dynamic indexing
    if (cur == last) {
      if (++run == 62u || i + 1u == npx) {
        w.put(OP_RUN | (run - 1u));
        run = 0;
      }
      continue;
    }
    if (run) {
      w.put((run == 1u && seen_literal) ? (OP_INDEX | last_slot) : (OP_RUN | (run - 1u)));
      run = 0;
    }
    seen_literal = true;
    last_slot = qoi_hash(cur);
    if (tab[last_slot * kQoiThreads] == cur) {
      w.put(OP_INDEX | last_slot);
    } else {
      tab[last_slot * kQoiThreads] = cur;
      const uint32_t r = cur & 255u, g = (cur >> 8) & 255u, bl = (cur >> 16) & 255u;
      if ((cur >> 24) != (last >> 24)) {
        w.put(OP_RGBA); w.put(r); w.put(g); w.put(bl); w.put(cur >> 24);
      } else {
        const int dr = (int)(int8_t)(r - (last & 255u)), dg = (int)(int8_t)(g - ((last >> 8) & 255u));
        const int db = (int)(int8_t)(bl - ((last >> 16) & 255u));
        const int dgr = (int)(int8_t)(dr - dg), dgb = (int)(int8_t)(db - dg);
        if (dr >= -2 && dr <= 1 && dg >= -2 && dg <= 1 && db >= -2 && db <= 1) {
          w.put(OP_DIFF | ((dr + 2) << 4) | ((dg + 2) << 2) | (db + 2));
        } else if (dg >= -32 && dg <= 31 && dgr >= -8 && dgr <= 7 && dgb >= -8 && dgb <= 7) {
          w.put(OP_LUMA | (dg + 32));
          w.put(((dgr + 8) << 4) | (dgb + 8));
        } else {
          w.put(OP_RGB); w.put(r); w.put(g); w.put(bl);
        }
      }
    }
    last = cur;
  }
  for (int i = 0; i < 7; ++i) w.put(0);
  w.put(1);
  w.flush();
  const uint32_t qlen = w.n - kBlockHeader;
  slot[9] = (uint8_t)(qlen >> 24); slot[10] = (uint8_t)(qlen >> 16); slot[11] = (uint8_t)(qlen >> 8); slot[12] = (uint8_t)qlen;
  enc_len[b] = w.n;
}

// One CTA: exclusive scan of the encoded lengths -> offsets behind the file header and line table; line table; header.
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) k_qoi_layout(const uint32_t* __restrict__ enc_len, Geom g, uint32_t filter_byte,
                                                             unsigned long long* __restrict__ out_off, uint8_t* __restrict__ out,
                                                             unsigned long long* __restrict__ total) {
  __shared__ unsigned long long s_warp[kScanThreads / 32];
  __shared__ unsigned long long s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t nblocks = g.cols * g.rows;
  const unsigned long long base = kFileHeader + 4ull * g.rows;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t c0 = 0; c0 < nblocks; c0 += kScanThreads) {
    const uint32_t b = c0 + tid;
    const unsigned long long v = b < nblocks ? enc_len[b] : 0ull;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long n = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += n;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    unsigned long long wbase = 0, agg = 0;
    for (int w = 0; w < kScanThreads / 32; ++w) {
      if (w < warp) wbase += s_warp[w];
      agg += s_warp[w];
    }
    const unsigned long long carry = s_carry;
    if (b < nblocks) out_off[b] = base + carry + wbase + inc - v;
    __syncthreads();
    if (tid == 0) s_carry = carry + agg;
    __syncthreads();
  }
  const unsigned long long end = base + s_carry;
  if (tid == 0) {
    *total = end;
    const uint8_t hdr[10] = {'P', 'I', 'X', 'L', 'Z', 'R', 0, 0, 2, (uint8_t)filter_byte};
    for (int i = 0; i < 10; ++i) out[i] = hdr[i];
    const uint32_t f[4] = {g.W, g.H, g.bw, g.bh};
    for (int k = 0; k < 4; ++k)
      for (int i = 0; i < 4; ++i) out[10 + 4 * k + i] = (uint8_t)(f[k] >> (24 - 8 * i));
  }
  // bytes of every block row (encoding/mod.rs:60-75); out_off was written by this CTA: visible after the barrier above
  for (uint32_t r = tid; r < g.rows; r += kScanThreads) {
    const unsigned long long lo = out_off[(size_t)r * g.cols];
    const unsigned long long hi = (r + 1 < g.rows) ? out_off[(size_t)(r + 1) * g.cols] : end;
    const uint32_t len = (uint32_t)(hi - lo);
    uint8_t* o = out + kFileHeader + 4ull * r;
    o[0] = (uint8_t)(len >> 24); o[1] = (uint8_t)(len >> 16); o[2] = (uint8_t)(len >> 8); o[3] = (uint8_t)len;
  }
}

// one warp per block: slot -> final position
__global__ void __launch_bounds__(256) k_qoi_compact(const pxz_block_desc* __restrict__ descs, const uint8_t* __restrict__ arena,
                                                     const uint32_t* __restrict__ enc_len, const unsigned long long* __restrict__ out_off,
                                                     uint32_t nblocks, uint32_t C, uint8_t* __restrict__ out) {
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  for (uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < nblocks; b += warps) {
    const uint8_t* src = arena + slot_offset(descs[b].offset, b, C);
    uint8_t* dst = out + out_off[b];
    const uint32_t n = enc_len[b];
    for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
  }
}

// thread per block: QOI body at in + in_off[b] (length qlen[b]) -> payload pixels.  err: set to 1 on a truncated stream.
template <int C>
__global__ void __launch_bounds__(kQoiThreads) k_qoi_decode(const uint8_t* __restrict__ in, const unsigned long long* __restrict__ in_off,
                                                            const uint32_t* __restrict__ qlen, const pxz_block_desc* __restrict__ descs,
                                                            uint32_t nblocks, uint8_t* __restrict__ pixels, int* __restrict__ err) {
  __shared__ uint32_t s_tab[64 * kQoiThreads];
  const int tid = threadIdx.x;
  for (int i = tid; i < 64 * kQoiThreads; i += kQoiThreads) s_tab[i] = 0u;
  __syncthreads();
  const uint32_t b = blockIdx.x * kQoiThreads + tid;
  if (b >= nblocks) return;
  const pxz_block_desc d = descs[b];
  const uint32_t len = qlen[b];
  const uint8_t* p = in + in_off[b] + kQoiHeader;
  const uint8_t* end = in + in_off[b] + len - 8;
  uint32_t* tab = s_tab + tid;
  uint32_t cur = 0xFF000000u, run = 0;
  const uint32_t npx = (uint32_t)d.w * d.h;
  uint8_t* o = pixels + d.offset;
  bool bad = false;
  for (uint32_t i = 0; i < npx; ++i) {
    if (run) {
      --run;
    } else {
      if (p >= end) { bad = true; break; }  // the stream ends before the block is full
      const uint32_t op = *p++;
      if (op == OP_RGB) {
        if (p + 3 > end) { bad = true; break; }
        cur = (cur & 0xFF000000u) | p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
        p += 3;
      } else if (op == OP_RGBA) {
        if (p + 4 > end) { bad = true; break; }
        cur = p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
        p += 4;
      } else if ((op & 0xC0u) == OP_INDEX) {
        cur = tab[(op & 63u) * kQoiThreads];
      } else if ((op & 0xC0u) == OP_DIFF) {
        const uint32_t r = (cur + ((op >> 4) & 3u) - 2u) & 255u, g = ((cur >> 8) + ((op >> 2) & 3u) - 2u) & 255u;
        const uint32_t bl = ((cur >> 16) + (op & 3u) - 2u) & 255u;
        cur = (cur & 0xFF000000u) | r | (g << 8) | (bl << 16);
      } else if ((op & 0xC0u) == OP_LUMA) {
        if (p >= end) { bad = true; break; }
        const uint32_t x = *p++;
        const uint32_t dg = (op & 63u) - 32u;
        const uint32_t r = (cur + dg - 8u + (x >> 4)) & 255u, g = ((cur >> 8) + dg) & 255u;
        const uint32_t bl = ((cur >> 16) + dg - 8u + (x & 15u)) & 255u;
        cur = (cur & 0xFF000000u) | r | (g << 8) | (bl << 16);
      } else {
        run = op & 63u;  // OP_RUN
      }
      tab[qoi_hash(cur) * kQoiThreads] = cur;
    }
    if (C == 4) {
      reinterpret_cast<uint32_t*>(o)[i] = cur;
    } else {
      o[3 * i] = (uint8_t)cur; o[3 * i + 1] = (uint8_t)(cur >> 8); o[3 * i + 2] = (uint8_t)(cur >> 16);
    }
  }
  if (bad) atomicExch(err, 1);
}

}  // namespace

size_t qoi_arena_bytes(uint32_t nblocks, uint64_t payload_bytes, uint32_t C) {
  return (size_t)36 * nblocks + (size_t)(payload_bytes / C) * (C + 1) + 8;
}

cudaError_t launch_qoi_encode(const pxz_block_desc* descs, const uint8_t* pixels, const Geom& g, int values_present,
                              uint32_t filter_byte, uint8_t* arena, uint32_t* enc_len, unsigned long long* out_off, uint8_t* out,
                              unsigned long long* total, cudaStream_t s, uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  const int grid = (int)((nblocks + kQoiThreads - 1) / kQoiThreads);
  *launches += 3;
  const auto encode = g.C == 4 ? k_qoi_encode<4> : k_qoi_encode<3>;
  encode<<<grid, kQoiThreads, 0, s>>>(descs, pixels, nblocks, values_present, arena, enc_len);
  k_qoi_layout<<<1, kScanThreads, 0, s>>>(enc_len, g, filter_byte, out_off, out, total);
  const int cgrid = (int)std::min<uint32_t>((nblocks + 7) / 8, 148u * 8u);
  k_qoi_compact<<<cgrid, 256, 0, s>>>(descs, arena, enc_len, out_off, nblocks, g.C, out);
  return cudaGetLastError();
}

cudaError_t launch_qoi_decode(const uint8_t* in, const unsigned long long* in_off, const uint32_t* qlen, const pxz_block_desc* descs,
                              const Geom& g, uint8_t* pixels, int* err, cudaStream_t s, uint64_t* launches) {
  const uint32_t nblocks = g.cols * g.rows;
  const int grid = (int)((nblocks + kQoiThreads - 1) / kQoiThreads);
  ++*launches;
  const auto decode = g.C == 4 ? k_qoi_decode<4> : k_qoi_decode<3>;
  decode<<<grid, kQoiThreads, 0, s>>>(in, in_off, qlen, descs, nblocks, pixels, err);
  return cudaGetLastError();
}

}  // namespace pxz
