// tables.cpp — host-side parameter setup for the kernels (O(block size) work, no pixel data):
//   * per-axis resample tables (tap ranges + normalised f32 weights) for the `image`-crate
//     semantics of PixlzrBlock::resize (src/data_types/block.rs:282-290 -> image 0.25.5
//     imageops::sample::{vertical_sample, horizontal_sample});
//   * the value -> level thresholds of reduce_image_section (src/operations.rs:147-148).
// The kernels apply these tables in the reference's accumulation order, which is what makes the
// resampled pixels bit-identical to the CPU result.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "pxz_host.h"

namespace pxz {

namespace {

const float kPi = 3.14159274101257324219f;  // f32::consts::PI

// image 0.25.5 imageops/sample.rs kernels, evaluated in f32
struct KernelFn {
  float support;
  float (*eval)(float);
};

float eval_box(float) { return 1.0f; }
float eval_triangle(float x) {
  const float a = fabsf(x);
  return a < 1.0f ? 1.0f - a : 0.0f;
}
float eval_catmullrom(float x) {  // bc_cubic_spline(x, 0.0, 0.5)
  const float a = fabsf(x);
  float k = 0.0f;
  if (a < 1.0f) {
    const float a2 = a * a, a3 = a2 * a;
    k = 9.0f * a3 + -15.0f * a2 + 6.0f;
  } else if (a < 2.0f) {
    const float a2 = a * a, a3 = a2 * a;
    k = -3.0f * a3 + 15.0f * a2 + -24.0f * a + 12.0f;
  }
  return k / 6.0f;
}
float eval_gaussian(float x) {  // gaussian(x, 0.5)
  const float r = 0.5f;
  const float scale = 1.0f / (sqrtf(2.0f * kPi) * r);
  return scale * expf(-(x * x) / (2.0f * (r * r)));
}
float sinc_f32(float t) {
  const float a = t * kPi;
  return t == 0.0f ? 1.0f : sinf(a) / a;
}
float eval_lanczos3(float x) { return fabsf(x) < 3.0f ? sinc_f32(x) * sinc_f32(x / 3.0f) : 0.0f; }

bool kernel_of(int filter, KernelFn* k) {
  switch (filter) {
    case PXZ_NEAREST: *k = {0.0f, eval_box}; return true;
    case PXZ_TRIANGLE: *k = {1.0f, eval_triangle}; return true;
    case PXZ_CATMULLROM: *k = {2.0f, eval_catmullrom}; return true;
    case PXZ_GAUSSIAN: *k = {3.0f, eval_gaussian}; return true;
    case PXZ_LANCZOS3: *k = {3.0f, eval_lanczos3}; return true;
  }
  return false;
}

}  // namespace

bool build_axis_table(uint32_t n_in, uint32_t n_out, int filter, std::vector<uint32_t>* pool, AxisTab* tab) {
  KernelFn kf;
  if (!kernel_of(filter, &kf) || n_in == 0 || n_out == 0) return false;
  const float ratio = (float)n_in / (float)n_out;
  const float sratio = ratio < 1.0f ? 1.0f : ratio;
  const float reach = kf.support * sratio;

  // first sweep: tap ranges, to size the weight rows
  std::vector<uint32_t> lefts(n_out), counts(n_out);
  uint32_t stride = 1;
  for (uint32_t o = 0; o < n_out; ++o) {
    const float centre = ((float)o + 0.5f) * ratio;
    long long lo = (long long)floorf(centre - reach);
    if (lo < 0) lo = 0;
    if (lo > (long long)n_in - 1) lo = (long long)n_in - 1;
    long long hi = (long long)ceilf(centre + reach);
    if (hi < lo + 1) hi = lo + 1;
    if (hi > (long long)n_in) hi = (long long)n_in;
    lefts[o] = (uint32_t)lo;
    counts[o] = (uint32_t)(hi - lo);
    if (counts[o] > stride) stride = counts[o];
  }
  tab->n_in = n_in;
  tab->n_out = n_out;
  tab->stride = stride;
  tab->off = (uint32_t)pool->size();
  pool->insert(pool->end(), lefts.begin(), lefts.end());
  pool->insert(pool->end(), counts.begin(), counts.end());
  const size_t wbase = pool->size();
  pool->resize(wbase + (size_t)n_out * stride, 0u);
  // second sweep: weights, normalised by their sequential f32 sum
  std::vector<float> row(stride);
  for (uint32_t o = 0; o < n_out; ++o) {
    const float centre = ((float)o + 0.5f) * ratio - 0.5f;
    float total = 0.0f;
    for (uint32_t i = 0; i < counts[o]; ++i) {
      const float w = kf.eval(((float)(lefts[o] + i) - centre) / sratio);
      row[i] = w;
      total += w;
    }
    for (uint32_t i = 0; i < counts[o]; ++i) {
      const float w = row[i] / total;
      memcpy(&(*pool)[wbase + (size_t)o * stride + i], &w, sizeof(float));
    }
  }
  // blocked form: groups of 4 consecutive outputs share one walk over the source samples.  Groups with identical
  // weight rows (the interior groups of an integer ratio) share one copy, so most lanes of a warp read one address.
  while (pool->size() % 4) pool->push_back(0u);
  const uint32_t nb = (n_out + 3) / 4;
  std::vector<uint32_t> lo(nb), rows(nb), first(nb);
  std::vector<uint32_t> w4;  // unique groups, 4 words per source sample
  // upscale tables: every group is stored with the same number of rows (2, 4 or 8; +0 weights beyond its own), so the
  // expand kernel runs a fixed, fully unrolled walk.  bpad = 0: groups keep their own length.
  uint32_t bpad = 0;
  if (n_in <= n_out) {
    uint32_t longest = 0;
    for (uint32_t b = 0; b < nb; ++b) {
      uint32_t l = lefts[4 * b], h = 0;
      for (uint32_t j = 0; j < 4 && 4 * b + j < n_out; ++j) {
        l = std::min(l, lefts[4 * b + j]);
        h = std::max(h, lefts[4 * b + j] + counts[4 * b + j]);
      }
      longest = std::max(longest, h - l);
    }
    bpad = longest <= 2 ? 2u : longest <= 4 ? 4u : longest <= 8 ? 8u : 0u;
  }
  for (uint32_t b = 0; b < nb; ++b) {
    uint32_t l = lefts[4 * b], h = 0;
    for (uint32_t j = 0; j < 4 && 4 * b + j < n_out; ++j) {
      l = std::min(l, lefts[4 * b + j]);
      h = std::max(h, lefts[4 * b + j] + counts[4 * b + j]);
    }
    lo[b] = l;
    rows[b] = h - l;
    std::vector<uint32_t> grp((size_t)std::max(rows[b], bpad) * 4, 0u);  // +0.0f everywhere
    for (uint32_t j = 0; j < 4 && 4 * b + j < n_out; ++j) {
      const uint32_t o = 4 * b + j;
      for (uint32_t i = 0; i < counts[o]; ++i) grp[(size_t)(lefts[o] + i - l) * 4 + j] = (*pool)[wbase + (size_t)o * stride + i];
    }
    bool found = false;
    for (uint32_t p = 0; p < b && !found; ++p) {
      if (std::max(rows[p], bpad) == std::max(rows[b], bpad) && std::equal(grp.begin(), grp.end(), w4.begin() + (size_t)first[p] * 4)) {
        first[b] = first[p];
        found = true;
      }
    }
    if (!found) {
      first[b] = (uint32_t)(w4.size() / 4);
      w4.insert(w4.end(), grp.begin(), grp.end());
    }
  }
  tab->boff = (uint32_t)pool->size();
  tab->nb = nb;
  tab->brows_total = (uint32_t)(w4.size() / 4);
  const size_t w4base = pool->size();
  pool->insert(pool->end(), w4.begin(), w4.end());
  pool->insert(pool->end(), lo.begin(), lo.end());
  pool->insert(pool->end(), rows.begin(), rows.end());
  pool->insert(pool->end(), first.begin(), first.end());
  tab->bwords = (uint32_t)(pool->size() - w4base);

  // ---- slide2 form (see pxz_internal.h) ----
  tab->pad1_ = 0;
  tab->slots = 0;
  tab->goff = 0xFFFFFFFFu;
  tab->gpoff = 0;
  tab->bpad = bpad;
  tab->s2off = tab->s2words = 0;
  tab->pad2_ = 0;
  auto weight_of = [&](uint32_t o, uint32_t i) {
    float w;
    memcpy(&w, &(*pool)[wbase + (size_t)o * stride + i], sizeof(float));
    return w;
  };
  if (n_in >= n_out) {
    // zero-trimmed windows: a tap whose weight is exactly 0 adds p * 0 = +-0 to an accumulator that is never -0
    std::vector<uint32_t> tl(n_out), tr(n_out);
    bool ok = true;
    for (uint32_t o = 0; o < n_out; ++o) {
      uint32_t a = 0, b = counts[o];
      while (a < b && weight_of(o, a) == 0.0f) ++a;
      while (b > a && weight_of(o, b - 1) == 0.0f) --b;
      if (a == b) { a = 0; b = 1; }  // all-zero row cannot happen (the weights sum to 1); keep one tap
      tl[o] = lefts[o] + a;
      tr[o] = lefts[o] + b;
      if (o > 0 && (tl[o] < tl[o - 1] || tr[o] < tr[o - 1])) ok = false;  // outputs must start and finish in order
    }
    uint32_t max_live = 0;
    if (ok) {
      for (uint32_t r = 0; r < n_in; ++r) {
        uint32_t live = 0;
        for (uint32_t o = 0; o < n_out; ++o) live += (tl[o] <= r && r < tr[o]) ? 1u : 0u;
        max_live = std::max(max_live, live);
      }
    }
    const uint32_t slots = max_live <= 2 ? 2u : max_live <= 4 ? 4u : max_live <= 6 ? 6u : 0u;
    if (ok && slots) {
      // with windows ordered on both ends the live outputs at any sample are consecutive, so o % slots never collides
      while (pool->size() % 4) pool->push_back(0u);
      const size_t s2 = pool->size();
      pool->resize(s2 + (size_t)n_in * slots * 2, 0u);
      for (uint32_t o = 0; o < n_out; ++o)
        for (uint32_t r = tl[o]; r < tr[o]; ++r) {
          const size_t at = s2 + ((size_t)r * slots + o % slots) * 2;
          (*pool)[at] = (*pool)[at + 1] = (*pool)[wbase + (size_t)o * stride + (r - lefts[o])];
        }
      for (uint32_t o = 0; o < n_out; ++o) pool->push_back(tr[o] - 1);
      while (pool->size() % 4) pool->push_back(0u);
      tab->slots = slots;
      tab->s2off = (uint32_t)s2;
      tab->s2words = (uint32_t)(pool->size() - s2);
    }
  }
  // ---- gather8 form ----
  if (n_in <= n_out && stride <= 7) {  // the expand kernel keeps a 7-sample window
    while (pool->size() % 4) pool->push_back(0u);
    const size_t gbase = pool->size();
    const uint32_t npairs = (n_out + 1) / 2;
    const uint32_t lpad = (4u - (n_out % 4u)) % 4u;  // keep the pair rows 16-byte aligned
    const size_t pbase = gbase + (size_t)n_out * 8 + n_out + lpad;
    pool->resize(pbase + (size_t)npairs * 16, 0u);
    for (uint32_t o = 0; o < n_out; ++o) {
      for (uint32_t i = 0; i < counts[o]; ++i) {
        const uint32_t wbits = (*pool)[wbase + (size_t)o * stride + i];
        (*pool)[gbase + (size_t)o * 8 + i] = wbits;
        (*pool)[pbase + (size_t)(o / 2) * 16 + 2 * i + (o & 1u)] = wbits;  // pair rows: (w_even[i], w_odd[i])
      }
      (*pool)[gbase + (size_t)n_out * 8 + o] = lefts[o];
    }
    tab->goff = (uint32_t)gbase;
    tab->gpoff = (uint32_t)pbase;
  }
  return true;
}

// ---- fast_image_resize 4.2.1 semantics (PixlzrBlock::resize, `fir` branch, block.rs:292-333) -----------------------
// The crate is not in the reference tree (Cargo.lock pins it): this follows its published algorithm — f64 weights,
// radius = support * max(scale, 1), taps [floor(centre - radius), ceil(centre + radius)) clamped to the axis, weights
// normalised to sum 1 and converted to 16-bit fixed point with the largest precision p < 22 for which
// round(max_w * 2^(p+1)) < 2^15.  "parity unpinned": no artefact of the reference was produced with this branch.
// Table at `off`: left[n_out] | count[n_out] | coefficient[n_out * stride] (i16 values in 32-bit words); tab->pad2_ = p.
namespace {
double fir_sinc(double x) { return x == 0.0 ? 1.0 : sin(x * M_PI) / (x * M_PI); }
double fir_eval(int alg, double x) {
  switch (alg) {
    case PXZ_FIR_BILINEAR: x = fabs(x); return x < 1.0 ? 1.0 - x : 0.0;
    case PXZ_FIR_HAMMING:
      x = fabs(x);
      if (x == 0.0) return 1.0;
      if (x >= 1.0) return 0.0;
      x *= M_PI;
      return (0.54 + 0.46 * cos(x)) * sin(x) / x;
    case PXZ_FIR_CATMULLROM: {
      const double a = -0.5;
      x = fabs(x);
      if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0;
      if (x < 2.0) return (((x - 5.0) * x + 8.0) * x - 4.0) * a;
      return 0.0;
    }
    case PXZ_FIR_GAUSSIAN: {
      if (fabs(x) >= 3.0) return 0.0;
      const double r = 0.5;
      return exp(-(x * x) / (2.0 * r * r)) / (sqrt(2.0 * M_PI) * r);
    }
    case PXZ_FIR_LANCZOS3: return (x >= -3.0 && x < 3.0) ? fir_sinc(x) * fir_sinc(x / 3.0) : 0.0;
  }
  return 0.0;
}
}  // namespace

bool build_axis_table_fir(uint32_t n_in, uint32_t n_out, int alg, std::vector<uint32_t>* pool, AxisTab* tab) {
  if (n_in == 0 || n_out == 0 || alg < PXZ_FIR_NEAREST || alg > PXZ_FIR_HAMMING) return false;
  memset(tab, 0, sizeof(*tab));
  tab->n_in = n_in;
  tab->n_out = n_out;
  tab->goff = 0xFFFFFFFFu;
  std::vector<uint32_t> lefts(n_out), counts(n_out);
  std::vector<std::vector<double>> w(n_out);
  const double scale = (double)n_in / (double)n_out;
  double maxw = 0.0;
  uint32_t stride = 1;
  if (alg == PXZ_FIR_NEAREST) {
    // ResizeAlg::Nearest: source sample (scale / 2 + scale * o) truncated; one tap of weight 1
    for (uint32_t o = 0; o < n_out; ++o) {
      uint32_t x = (uint32_t)(scale * 0.5 + scale * (double)o);
      if (x > n_in - 1) x = n_in - 1;
      lefts[o] = x; counts[o] = 1; w[o].assign(1, 1.0);
    }
    maxw = 1.0;
  } else {
    const double support = alg == PXZ_FIR_CATMULLROM ? 2.0 : (alg == PXZ_FIR_GAUSSIAN || alg == PXZ_FIR_LANCZOS3) ? 3.0 : 1.0;
    const double fscale = scale > 1.0 ? scale : 1.0, radius = support * fscale;
    for (uint32_t o = 0; o < n_out; ++o) {
      const double centre = ((double)o + 0.5) * scale;
      double lo = floor(centre - radius), hi = ceil(centre + radius);
      if (lo < 0.0) lo = 0.0;
      if (hi > (double)n_in) hi = (double)n_in;
      const uint32_t x0 = (uint32_t)lo, x1 = (uint32_t)hi;
      double ww = 0.0;
      for (uint32_t x = x0; x < x1; ++x) {
        const double v = fir_eval(alg, ((double)x + 0.5 - centre) / fscale);
        w[o].push_back(v);
        ww += v;
      }
      if (ww != 0.0)
        for (double& v : w[o]) v /= ww;
      for (double v : w[o]) maxw = std::max(maxw, v);
      lefts[o] = x0; counts[o] = x1 - x0;
      stride = std::max(stride, x1 - x0);
    }
  }
  int p = 0;
  for (p = 0; p < 22; ++p)
    if ((int)lround(maxw * (double)(1 << (p + 1))) >= (1 << 15)) break;
  tab->stride = stride;
  tab->pad2_ = (uint32_t)p | (alg == PXZ_FIR_NEAREST ? kFirNearestFlag : 0u);
  tab->off = (uint32_t)pool->size();
  pool->insert(pool->end(), lefts.begin(), lefts.end());
  pool->insert(pool->end(), counts.begin(), counts.end());
  const size_t kbase = pool->size();
  pool->resize(kbase + (size_t)n_out * stride, 0u);
  for (uint32_t o = 0; o < n_out; ++o)
    for (size_t i = 0; i < w[o].size(); ++i) (*pool)[kbase + (size_t)o * stride + i] = (uint32_t)(int32_t)lround(w[o][i] * (double)(1 << p));
  return true;
}

// thr[k] = smallest positive f32 v with round(log2f(v)) >= -k  (round = half away from zero).
// Built with the host libm exactly as the reference evaluates `value.log2().round()`, so the
// device-side comparison `v >= thr[k]` reproduces the CPU decision for every f32 input.
static inline int rounded_log2(float v) { return (int)roundf(log2f(v)); }

void build_level_thresholds(LevelThresholds* out) {
  for (int k = 0; k < kThresholds; ++k) {
    // the switch happens between 2^(-k-1) (round(log2) = -k-1) and 2^-k (round(log2) = -k)
    uint32_t lo, hi;
    float flo = ldexpf(1.0f, -k - 1), fhi = ldexpf(1.0f, -k);
    memcpy(&lo, &flo, 4);
    memcpy(&hi, &fhi, 4);
    while (hi - lo > 1) {
      const uint32_t mid = lo + (hi - lo) / 2;
      float fm;
      memcpy(&fm, &mid, 4);
      if (rounded_log2(fm) >= -k) hi = mid; else lo = mid;
    }
    // (tests/test_host_logic.py checks +-4096 ulps around every threshold against log2f itself)
    memcpy(&out->thr[k], &hi, 4);
  }
}

}  // namespace pxz
