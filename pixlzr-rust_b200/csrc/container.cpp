// container.cpp — the host stage either side of the device path: the .pxlzr / .pix container
// (version 0.0.2) and its per-block QOI streams.  It stays on the host and keeps the file layout
// byte-identical to the reference (src/encoding/mod.rs:40-242, src/constants.rs, qoi crate 0.4.1):
//
//   "PIXLZR" | 0,0,2 | filter u8 | width, height, block_w, block_h (u32 BE)
//   | one u32 BE per block row: bytes of that row's encoded blocks
//   | blocks, row-major: "block" | value f32 BE | qoi_len u32 BE | QOI stream minus its "qoif" magic
//
// Block rows are encoded in parallel (the reference uses rayon over block rows, encoding/mod.rs:60-75)
// straight out of the packed payload the device produced — no per-block allocations.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>

#include "pxz_host.h"

namespace {

struct Rgba {
  uint8_t r, g, b, a;
  bool operator==(const Rgba& o) const { return r == o.r && g == o.g && b == o.b && a == o.a; }
  uint32_t slot() const { return (r * 3u + g * 5u + b * 7u + a * 11u) & 63u; }
};

constexpr uint8_t OP_INDEX = 0x00, OP_DIFF = 0x40, OP_LUMA = 0x80, OP_RUN = 0xC0, OP_RGB = 0xFE, OP_RGBA = 0xFF;

inline void be32(uint8_t* p, uint32_t v) {
  p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }

// worst case of one QOI body (without magic): header 10 + (channels + 1) bytes per pixel + 8
inline size_t qoi_body_bound(size_t npx, uint32_t ch) { return 10 + npx * (ch + 1) + 8; }

// Encodes one block as a QOI stream WITHOUT the 4-byte magic (encoding/mod.rs:189-191).
// qoi 0.4.1 encode_impl: the spec's op order, plus that crate's habit of emitting a finished run
// of exactly one pixel as QOI_OP_INDEX of the previous pixel's slot once any non-run pixel was seen.
size_t qoi_body_encode(const uint8_t* px, uint32_t w, uint32_t h, uint32_t ch, uint8_t* out) {
  uint8_t* o = out;
  be32(o, w); be32(o + 4, h);
  o[8] = (uint8_t)ch;
  o[9] = 0;  // sRGB with linear alpha
  o += 10;
  Rgba table[64];
  memset(table, 0, sizeof(table));
  Rgba last{0, 0, 0, 255};
  uint32_t last_slot = last.slot();
  uint32_t run = 0;
  bool seen_literal = false;
  const size_t npx = (size_t)w * h;
  const uint8_t* p = px;
  for (size_t i = 0; i < npx; ++i, p += ch) {
    const Rgba cur{p[0], p[1], p[2], ch == 4 ? p[3] : (uint8_t)255};
    if (cur == last) {
      if (++run == 62 || i + 1 == npx) {
        *o++ = (uint8_t)(OP_RUN | (run - 1));
        run = 0;
      }
      continue;
    }
    if (run) {
      *o++ = (run == 1 && seen_literal) ? (uint8_t)(OP_INDEX | last_slot) : (uint8_t)(OP_RUN | (run - 1));
      run = 0;
    }
    seen_literal = true;
    last_slot = cur.slot();
    if (table[last_slot] == cur) {
      *o++ = (uint8_t)(OP_INDEX | last_slot);
    } else {
      table[last_slot] = cur;
      if (cur.a != last.a) {
        *o++ = OP_RGBA; *o++ = cur.r; *o++ = cur.g; *o++ = cur.b; *o++ = cur.a;
      } else {
        const int8_t dr = (int8_t)(cur.r - last.r), dg = (int8_t)(cur.g - last.g), db = (int8_t)(cur.b - last.b);
        const int8_t dgr = (int8_t)(dr - dg), dgb = (int8_t)(db - dg);
        if (dr >= -2 && dr <= 1 && dg >= -2 && dg <= 1 && db >= -2 && db <= 1) {
          *o++ = (uint8_t)(OP_DIFF | ((dr + 2) << 4) | ((dg + 2) << 2) | (db + 2));
        } else if (dg >= -32 && dg <= 31 && dgr >= -8 && dgr <= 7 && dgb >= -8 && dgb <= 7) {
          *o++ = (uint8_t)(OP_LUMA | (dg + 32));
          *o++ = (uint8_t)(((dgr + 8) << 4) | (dgb + 8));
        } else {
          *o++ = OP_RGB; *o++ = cur.r; *o++ = cur.g; *o++ = cur.b;
        }
      }
    }
    last = cur;
  }
  static const uint8_t tail[8] = {0, 0, 0, 0, 0, 0, 0, 1};
  memcpy(o, tail, 8);
  return (size_t)(o + 8 - out);
}

// Decodes a QOI body (no magic).  Returns false on a truncated / inconsistent stream.
bool qoi_body_decode(const uint8_t* in, size_t len, uint32_t ch_expected, uint8_t* out, size_t out_px) {
  if (len < 10 + 8) return false;
  const uint32_t ch = in[8];
  if (ch != ch_expected) return false;
  const uint8_t* p = in + 10;
  const uint8_t* end = in + len - 8;
  Rgba table[64];
  memset(table, 0, sizeof(table));
  Rgba cur{0, 0, 0, 255};
  uint32_t run = 0;
  for (size_t i = 0; i < out_px; ++i) {
    if (run) {
      --run;
    } else {
      if (p >= end) return false;  // the stream ends before the block is full (qoi 0.4.1: UnexpectedBufferEnd)
      const uint8_t op = *p++;
      if (op == OP_RGB) {
        if (p + 3 > end) return false;
        cur.r = p[0]; cur.g = p[1]; cur.b = p[2]; p += 3;
      } else if (op == OP_RGBA) {
        if (p + 4 > end) return false;
        cur.r = p[0]; cur.g = p[1]; cur.b = p[2]; cur.a = p[3]; p += 4;
      } else {
        switch (op & 0xC0) {
          case OP_INDEX: cur = table[op & 63]; break;
          case OP_DIFF:
            cur.r = (uint8_t)(cur.r + ((op >> 4) & 3) - 2);
            cur.g = (uint8_t)(cur.g + ((op >> 2) & 3) - 2);
            cur.b = (uint8_t)(cur.b + (op & 3) - 2);
            break;
          case OP_LUMA: {
            if (p >= end) return false;
            const uint8_t x = *p++;
            const int dg = (op & 63) - 32;
            cur.r = (uint8_t)(cur.r + dg - 8 + (x >> 4));
            cur.g = (uint8_t)(cur.g + dg);
            cur.b = (uint8_t)(cur.b + dg - 8 + (x & 15));
            break;
          }
          default: run = op & 63; break;  // OP_RUN
        }
      }
      table[cur.slot()] = cur;
    }
    uint8_t* o = out + i * ch;
    o[0] = cur.r; o[1] = cur.g; o[2] = cur.b;
    if (ch == 4) o[3] = cur.a;
  }
  return true;
}

inline uint32_t grid_f32(uint32_t n, uint32_t b) {  // pixlzr.rs:37-42, encoding/mod.rs:118-119
  return (uint32_t)ceilf((float)n / (float)b);
}

constexpr size_t kHeader = 26;      // constants.rs:19-20
constexpr size_t kBlockHeader = 13; // "block" + f32 + u32

struct FileHeader {
  uint32_t w, h, bw, bh, cols, rows;
  int32_t filt;       // -1 if absent
  size_t line_table;  // offset of the line table
  size_t body;        // offset of the first block record
};

// The file header and the line table's total (encoding/mod.rs:95-141): O(rows), no block record is read.
pxz_status read_header(const uint8_t* data, size_t len, FileHeader* hd) {
  if (len < 9 || memcmp(data, "PIXLZR", 6) != 0) return PXZ_E_FORMAT;  // encoding/mod.rs:99-104
  const uint32_t version = (uint32_t)data[6] << 16 | (uint32_t)data[7] << 8 | data[8];
  size_t p = 9;
  hd->filt = -1;
  if (version >= 1) {  // "filter" since 0.0.1 (encoding/mod.rs:16-19,109-111)
    if (len < p + 1) return PXZ_E_FORMAT;
    hd->filt = data[p++];
  }
  if (version < 2) return PXZ_E_UNSUPPORTED;  // "line-sizes" since 0.0.2; the reference cannot read older files either
  if (len < p + 16) return PXZ_E_FORMAT;
  hd->w = rd32(data + p); hd->h = rd32(data + p + 4); hd->bw = rd32(data + p + 8); hd->bh = rd32(data + p + 12);
  p += 16;
  if (hd->bw == 0 || hd->bh == 0 || hd->w == 0 || hd->h == 0) return PXZ_E_FORMAT;
  hd->cols = grid_f32(hd->w, hd->bw);
  hd->rows = grid_f32(hd->h, hd->bh);
  // the reference sizes the grid in f32 (encoding/mod.rs:118-119), the device side in integers: the two agree below
  // 2^24; a file for which they differ is refused instead of being walked with two different block counts
  if ((uint64_t)hd->cols != ((uint64_t)hd->w + hd->bw - 1) / hd->bw || (uint64_t)hd->rows != ((uint64_t)hd->h + hd->bh - 1) / hd->bh)
    return PXZ_E_UNSUPPORTED;
  if ((uint64_t)hd->cols * hd->rows > 0x7FFFFFFFull) return PXZ_E_UNSUPPORTED;
  if (len < p + (size_t)hd->rows * 4) return PXZ_E_FORMAT;
  hd->line_table = p;
  uint64_t body = 0;
  for (uint32_t r = 0; r < hd->rows; ++r) body += rd32(data + p + (size_t)r * 4);
  hd->body = p + (size_t)hd->rows * 4;
  if (hd->body + body != len) return PXZ_E_FORMAT;  // assert_eq!(reader.data.len(), ...), encoding/mod.rs:141
  return PXZ_OK;
}

struct BlockRecord {
  float value;
  uint32_t qlen, qw, qh;  // QOI body length (after the 13-byte record header) and size
};

// Checks the block record at data[p] ("block" | value | qoi_len | QOI stream minus its magic): magic, lengths, the QOI
// header and hostile sizes.  *ch: the file's channel count, 0 until the first record sets it.
pxz_status read_block_record(const uint8_t* data, size_t len, size_t p, uint32_t* ch, BlockRecord* rec) {
  if (p + kBlockHeader + 10 > len || memcmp(data + p, "block", 5) != 0) return PXZ_E_FORMAT;
  const uint32_t bits = rd32(data + p + 5);
  memcpy(&rec->value, &bits, 4);
  rec->qlen = rd32(data + p + 9);
  p += kBlockHeader;
  if (p + rec->qlen > len || rec->qlen < 18) return PXZ_E_FORMAT;
  rec->qw = rd32(data + p);
  rec->qh = rd32(data + p + 4);
  const uint32_t qc = data[p + 8];
  if (qc != 3 && qc != 4) return PXZ_E_FORMAT;
  if (*ch == 0) *ch = qc;
  if (qc != *ch) return PXZ_E_UNSUPPORTED;  // mixed RGB / RGBA blocks in one file
  if (rec->qw > 65535 || rec->qh > 65535 || rec->qw == 0 || rec->qh == 0) return PXZ_E_UNSUPPORTED;
  // hostile headers: the qoi crate refuses more than 400 M pixels, and an op byte yields at most 62 pixels (a run),
  // so a stream of qlen bytes cannot fill more than 62 * qlen of them — checked before anything is allocated
  if ((uint64_t)rec->qw * rec->qh > 400000000ull || (uint64_t)rec->qw * rec->qh > 62ull * rec->qlen) return PXZ_E_FORMAT;
  return PXZ_OK;
}

}  // namespace

extern "C" {

int64_t pxz_container_bound(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t channels, uint64_t payload_bytes) {
  if (bw == 0 || bh == 0 || (channels != 3 && channels != 4)) return PXZ_E_ARG;
  const uint64_t cols = grid_f32(w, bw), rows = grid_f32(h, bh);
  const uint64_t npx = payload_bytes / channels;
  return (int64_t)(kHeader + rows * 4 + cols * rows * (kBlockHeader + 18) + npx * (channels + 1));
}

int64_t pxz_container_encode(uint32_t w, uint32_t h, uint32_t bw, uint32_t bh, uint32_t filter_byte, uint32_t channels,
                             const pxz_block_desc* descs, const uint8_t* pixels, const uint8_t* value_present,
                             uint8_t* out, size_t cap, int nthreads) {
  if (!descs || !pixels || !out || bw == 0 || bh == 0 || (channels != 3 && channels != 4)) return PXZ_E_ARG;
  const uint32_t cols = grid_f32(w, bw), rows = grid_f32(h, bh);
  // every block row is encoded into its own worst-case slice of a scratch arena, then the rows are
  // concatenated behind the line-length table
  std::vector<size_t> row_cap(rows), row_off(rows + 1, 0), row_len(rows, 0);
  for (uint32_t r = 0; r < rows; ++r) {
    size_t c = 0;
    for (uint32_t x = 0; x < cols; ++x) {
      const pxz_block_desc& d = descs[(size_t)r * cols + x];
      c += kBlockHeader + qoi_body_bound((size_t)d.w * d.h, channels);
    }
    row_cap[r] = c;
    row_off[r + 1] = row_off[r] + c;
  }
  std::vector<uint8_t> arena(row_off[rows]);
  std::atomic<uint32_t> next{0};
  auto work = [&]() {
    for (uint32_t r = next.fetch_add(1); r < rows; r = next.fetch_add(1)) {
      uint8_t* o = arena.data() + row_off[r];
      for (uint32_t x = 0; x < cols; ++x) {
        const size_t bi = (size_t)r * cols + x;
        const pxz_block_desc& d = descs[bi];
        memcpy(o, "block", 5);
        const float v = (value_present && !value_present[bi]) ? 0.0f : d.value;  // encoding/mod.rs:173-178
        uint32_t bits;
        memcpy(&bits, &v, 4);
        be32(o + 5, bits);
        const size_t n = qoi_body_encode(pixels + d.offset, d.w, d.h, channels, o + kBlockHeader);
        be32(o + 9, (uint32_t)n);
        o += kBlockHeader + n;
      }
      row_len[r] = (size_t)(o - (arena.data() + row_off[r]));
    }
  };
  int nt = std::max(1, std::min<int>(nthreads, (int)rows));
  std::vector<std::thread> pool;
  for (int i = 1; i < nt; ++i) pool.emplace_back(work);
  work();
  for (auto& t : pool) t.join();

  size_t total = kHeader + (size_t)rows * 4;
  for (uint32_t r = 0; r < rows; ++r) total += row_len[r];
  if (total > cap) return PXZ_E_ARG;  // size `out` with pxz_container_bound()
  memcpy(out, "PIXLZR", 6);
  out[6] = 0; out[7] = 0; out[8] = 2;
  out[9] = (uint8_t)filter_byte;
  be32(out + 10, w); be32(out + 14, h); be32(out + 18, bw); be32(out + 22, bh);
  uint8_t* o = out + kHeader;
  for (uint32_t r = 0; r < rows; ++r, o += 4) be32(o, (uint32_t)row_len[r]);
  for (uint32_t r = 0; r < rows; ++r) {
    memcpy(o, arena.data() + row_off[r], row_len[r]);
    o += row_len[r];
  }
  return (int64_t)total;
}

pxz_status pxz_container_decode(const uint8_t* data, size_t len, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                                int32_t* filter_byte, uint32_t* channels, uint64_t* payload_bytes, pxz_block_desc* descs,
                                uint8_t* pixels) {
  if (!data || !w || !h || !bw || !bh || !channels || !payload_bytes) return PXZ_E_ARG;
  FileHeader hd;
  pxz_status st = read_header(data, len, &hd);
  if (st != PXZ_OK) return st;
  *w = hd.w; *h = hd.h; *bw = hd.bw; *bh = hd.bh;
  if (filter_byte) *filter_byte = hd.filt;
  const uint32_t cols = hd.cols, rows = hd.rows;
  size_t p = hd.body;
  uint64_t off = 0;
  uint32_t ch = 0;
  size_t row_start = p;
  for (size_t bi = 0; bi < (size_t)cols * rows; ++bi) {
    if (bi && bi % cols == 0) {
      // every block row fills exactly its entry of the line table (encoding/mod.rs:142-155 slices the rows by it)
      if (p - row_start != rd32(data + hd.line_table + (bi / cols - 1) * 4)) return PXZ_E_FORMAT;
      row_start = p;
    }
    BlockRecord rec;
    if ((st = read_block_record(data, len, p, &ch, &rec)) != PXZ_OK) return st;
    p += kBlockHeader;
    if (descs) {
      descs[bi].offset = off;
      descs[bi].value = rec.value;
      descs[bi].w = (uint16_t)rec.qw;
      descs[bi].h = (uint16_t)rec.qh;
      if (pixels && !qoi_body_decode(data + p, rec.qlen, ch, pixels + off, (size_t)rec.qw * rec.qh)) return PXZ_E_FORMAT;
    }
    off += (uint64_t)rec.qw * rec.qh * ch;
    p += rec.qlen;
  }
  if (p - row_start != rd32(data + hd.line_table + (size_t)(rows - 1) * 4)) return PXZ_E_FORMAT;
  *channels = ch;
  *payload_bytes = off;
  return PXZ_OK;
}

pxz_status pxz_container_header(const uint8_t* data, size_t len, uint32_t* w, uint32_t* h, uint32_t* bw, uint32_t* bh,
                                int32_t* filter_byte) {
  if (!data || !w || !h || !bw || !bh) return PXZ_E_ARG;
  FileHeader hd;
  const pxz_status st = read_header(data, len, &hd);
  if (st != PXZ_OK) return st;
  *w = hd.w; *h = hd.h; *bw = hd.bw; *bh = hd.bh;
  if (filter_byte) *filter_byte = hd.filt;
  return PXZ_OK;
}

int64_t pxz_container_crop(const uint8_t* data, size_t len, uint32_t c0, uint32_t r0, uint32_t nc, uint32_t nr, uint8_t* out,
                           size_t cap) {
  if (!data) return PXZ_E_ARG;
  FileHeader hd;
  pxz_status st = read_header(data, len, &hd);
  if (st != PXZ_OK) return st;
  if (nc == 0 || nr == 0 || c0 >= hd.cols || r0 >= hd.rows || nc > hd.cols - c0 || nr > hd.rows - r0) return PXZ_E_ARG;
  // rows before the window are skipped by their line-table entries; the rows of the window are walked record by record
  size_t p = hd.body;
  for (uint32_t r = 0; r < r0; ++r) p += rd32(data + hd.line_table + (size_t)r * 4);
  const size_t head = kHeader + (size_t)nr * 4;
  if (out && head > cap) return PXZ_E_ARG;
  size_t o = head;
  uint32_t ch = 0;
  for (uint32_t r = r0; r < r0 + nr; ++r) {
    const size_t row_start = p;
    size_t sel0 = p, sel1 = p;  // bytes of the records c0 .. c0 + nc - 1
    for (uint32_t c = 0; c < hd.cols; ++c) {
      if (c == c0) sel0 = p;
      BlockRecord rec;
      if ((st = read_block_record(data, len, p, &ch, &rec)) != PXZ_OK) return st;
      p += kBlockHeader + rec.qlen;
      if (c + 1 == c0 + nc) sel1 = p;
    }
    if (p - row_start != rd32(data + hd.line_table + (size_t)r * 4)) return PXZ_E_FORMAT;
    const size_t n = sel1 - sel0;
    if (out) {
      if (o + n > cap) return PXZ_E_ARG;
      memcpy(out + o, data + sel0, n);
      be32(out + kHeader + (size_t)(r - r0) * 4, (uint32_t)n);
    }
    o += n;
  }
  if (out) {
    memcpy(out, "PIXLZR", 6);
    out[6] = 0; out[7] = 0; out[8] = 2;
    out[9] = (uint8_t)hd.filt;  // present from version 0.0.1 on
    be32(out + 10, (uint32_t)(std::min<uint64_t>(hd.w, (uint64_t)(c0 + nc) * hd.bw) - (uint64_t)c0 * hd.bw));
    be32(out + 14, (uint32_t)(std::min<uint64_t>(hd.h, (uint64_t)(r0 + nr) * hd.bh) - (uint64_t)r0 * hd.bh));
    be32(out + 18, hd.bw);
    be32(out + 22, hd.bh);
  }
  return (int64_t)o;
}

}  // extern "C"
