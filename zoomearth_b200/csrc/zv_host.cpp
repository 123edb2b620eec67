// Host-side (CPU, integer / fp64) part of libzoomvit: zoom geometry, Pillow coefficient tables, the
// normalisation LUT and the per-batch plan.  Everything here must be BIT-EXACT against the reference's
// Python arithmetic, so the translation unit is compiled with -ffp-contract=off and written in the same
// evaluation order as the code it replaces:
//   cut_box        reference src/eval/infer.py:41-76
//   resize_dims    reference src/eval/infer.py:78-85
//   smart_resize   HF models/qwen2_vl/image_processing_pil_qwen2_vl.py:57-83
//   coefficients   Pillow ImagingResample (precompute_coeffs + normalize_coeffs_8bpc), bicubic a=-0.5; or torch's
//                  uint8 antialiased bicubic (aten UpSampleKernel.cpp, int16 taps), what torchvision's resize runs
//   plan           HF models/qwen2_5_vl/modeling_qwen2_5_vl.py:382-451,470-496
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>

#include "zv_common.h"

namespace zv {

static thread_local std::string g_err;
static thread_local int64_t g_launches = 0;

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
void count_launch(int64_t n) { g_launches += n; }
void reset_launch_count() { g_launches = 0; }

// Python's int(x) for a double: truncation toward zero.
static inline int64_t py_int(double x) { return (int64_t)x; }
// Python's a // b for ints (floor division).
static inline int64_t floordiv(int64_t a, int64_t b) {
  int64_t q = a / b, r = a % b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}

static inline double bicubic(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

int32_t resample_ksize(int32_t in_size, int32_t out_size) {
  if (in_size == out_size) return 1;              // Pillow skips the pass: identity tap
  double scale = (double)in_size / out_size;
  double fs = scale < 1.0 ? 1.0 : scale;
  return (int32_t)std::ceil(2.0 * fs) * 2 + 1;
}

int check_resample_kind(int32_t kind, const char* who) {
  if (kind == ZV_RESAMPLE_PIL || kind == ZV_RESAMPLE_TORCHVISION || kind == ZV_RESAMPLE_TORCHVISION_CUDA) return ZV_OK;
  return fail(ZV_EINVAL, "%s: resample_kind %d (0 ZV_RESAMPLE_PIL, 1 ZV_RESAMPLE_TORCHVISION, 2 ZV_RESAMPLE_TORCHVISION_CUDA)",
              who, kind);
}

static void resample_coeffs_pil(int32_t in_size, int32_t out_size, AxisCoeffs* c) {
  const double scale = (double)in_size / out_size;
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * fs;
  const double ss = 1.0 / fs;
  std::vector<double> w(c->ksize);
  for (int32_t xx = 0; xx < out_size; ++xx) {
    double center = 0 + (xx + 0.5) * scale;
    int32_t xmin = (int32_t)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int32_t xmax = (int32_t)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    double ww = 0.0;
    for (int32_t x = 0; x < xmax; ++x) {
      double v = bicubic((x + xmin - center + 0.5) * ss);
      w[x] = v;
      ww += v;
    }
    int32_t* k = &c->kk[(size_t)xx * c->ksize];
    for (int32_t x = 0; x < xmax; ++x) {
      double v = w[x];
      if (ww != 0.0) v /= ww;
      k[x] = v < 0 ? (int32_t)(-0.5 + v * (double)(1 << 22)) : (int32_t)(0.5 + v * (double)(1 << 22));
    }
    c->bounds[2 * xx] = xmin;
    c->bounds[2 * xx + 1] = xmax;
  }
}

// torch's taps: Pillow's windows (clamped to ksize) and fp64 weights, rounded to int16 at ONE precision p for the whole
// axis - the first p < 22 at which the largest weight would need 16 bits one bit further - then moved to 22 bits.  A tap
// t 2^(22-p) makes the kernels' (acc + 2^21) >> 22 equal to torch's (acc_p + 2^(p-1)) >> p, so every K1 route runs them.
static void resample_coeffs_tv(int32_t in_size, int32_t out_size, AxisCoeffs* c) {
  const double scale = (double)in_size / out_size;
  const double support = scale >= 1.0 ? 2.0 * scale : 2.0;
  const double invscale = scale >= 1.0 ? 1.0 / scale : 1.0;
  const int32_t ks = c->ksize;
  std::vector<double> w((size_t)out_size * ks, 0.0);
  double w_max = 0.0;
  for (int32_t xx = 0; xx < out_size; ++xx) {
    const double center = scale * (xx + 0.5);
    const int32_t xmin = std::max((int32_t)(center - support + 0.5), 0);
    const int32_t xsize = std::min(std::max(std::min((int32_t)(center + support + 0.5), in_size) - xmin, 0), ks);
    double* wx = &w[(size_t)xx * ks];
    double total = 0.0;
    for (int32_t j = 0; j < xsize; ++j) {
      wx[j] = bicubic((j + xmin - center + 0.5) * invscale);
      total += wx[j];
    }
    if (total != 0.0)
      for (int32_t j = 0; j < xsize; ++j) {
        wx[j] /= total;
        w_max = std::max(w_max, wx[j]);
      }
    c->bounds[2 * xx] = xmin;
    c->bounds[2 * xx + 1] = xsize;
  }
  int32_t p = 0;
  while (p < 22 && (int32_t)(0.5 + w_max * (double)(1 << (p + 1))) < (1 << 15)) ++p;
  c->precision = p;
  for (size_t i = 0; i < w.size(); ++i) {
    const double v = w[i] * (double)(1 << p);
    c->kk[i] = (v < 0 ? (int32_t)(-0.5 + v) : (int32_t)(0.5 + v)) * (1 << (22 - p));
  }
}

// torch's fp32 antialiased bicubic on a CUDA device (aten upsample_gen2d_aa_out_frame<float, float, BicubicFilterFunctor>,
// upsample_antialias::_compute_weights_span / _compute_weights), operation for operation as its sm_100 SASS runs them: the
// centre scale (i + 0.5) is never rounded on its own - it is folded into FFMAs for the window ends and for xmin - centre -
// the filter's Horner steps are FFMAs, everything else is a separately rounded fp32 add, multiply or IEEE divide.  The
// host compiles with -ffp-contract=off, so each std::fma below is the one FFMA and nothing else is fused.  kk holds the
// weights' fp32 bits.  torch's xsize never exceeds its interp_size = ceilf(support) 2 + 1, which never exceeds Pillow's
// ksize for the same axis (fl32(in / out) <= k / 2 whenever in / out <= k / 2), so the weights fit Pillow's tap slots.
static float bicubic_f32(float x) {
  if (x < 0.0f) x = -x;
  if (x < 1.0f) return std::fma(x, x * std::fma(x, 1.5f, -2.5f), 1.0f);
  if (x < 2.0f) return std::fma(x, std::fma(x, x - 5.0f, 8.0f), -4.0f) * -0.5f;
  return 0.0f;
}

static void resample_coeffs_f32(int32_t in_size, int32_t out_size, AxisCoeffs* c) {
  const float scale = (float)in_size / (float)out_size;
  const float support = scale >= 1.0f ? scale + scale : 2.0f;
  const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
  const int32_t ks = c->ksize;
  std::vector<float> w(ks);
  for (int32_t xx = 0; xx < out_size; ++xx) {
    const float ci = (float)xx + 0.5f;
    const int32_t xmin = std::max((int32_t)(std::fma(ci, scale, -support) + 0.5f), 0);
    const int32_t xsize = std::min(std::min((int32_t)(std::fma(ci, scale, support) + 0.5f), in_size) - xmin, ks);
    const float xmin_m_center = std::fma(-ci, scale, (float)xmin);
    float total = 0.0f;
    for (int32_t j = 0; j < xsize; ++j) {
      w[j] = bicubic_f32(((float)j + xmin_m_center + 0.5f) * invscale);
      total += w[j];
    }
    int32_t* k = &c->kk[(size_t)xx * ks];
    for (int32_t j = 0; j < xsize; ++j) {
      const float v = total != 0.0f ? w[j] / total : w[j];
      std::memcpy(&k[j], &v, sizeof(v));
    }
    c->bounds[2 * xx] = xmin;
    c->bounds[2 * xx + 1] = xsize;
  }
}

void resample_coeffs(int32_t kind, int32_t in_size, int32_t out_size, AxisCoeffs* c) {
  c->in_size = in_size;
  c->out_size = out_size;
  c->ksize = resample_ksize(in_size, out_size);
  c->bounds.assign((size_t)out_size * 2, 0);
  c->kk.assign((size_t)out_size * c->ksize, 0);
  c->precision = 22;
  // same size: both libraries skip the pass, expressed as one exact tap.  torch's fp32 path does run a same-size axis when
  // the other one is resized, but with scale 1 its taps are (-0, 1, -0, 0) at integer offsets: every output is its
  // input exactly, the one fp32 tap 1.0f below (up to the sign of a zero, which the final rounding to uint8 drops)
  if (in_size == out_size) {
    const float one = 1.0f;
    for (int32_t xx = 0; xx < out_size; ++xx) {
      c->bounds[2 * xx] = xx;
      c->bounds[2 * xx + 1] = 1;
      if (kind == ZV_RESAMPLE_TORCHVISION_CUDA) std::memcpy(&c->kk[xx], &one, sizeof(float));
      else c->kk[xx] = 1 << 22;
    }
    return;
  }
  if (kind == ZV_RESAMPLE_TORCHVISION_CUDA) resample_coeffs_f32(in_size, out_size, c);
  else if (kind == ZV_RESAMPLE_TORCHVISION) resample_coeffs_tv(in_size, out_size, c);
  else resample_coeffs_pil(in_size, out_size, c);
}

// Row blocks of the tcgen05 window-attention kernel: windows (segments of cu, each <= max_rows) in order, as many whole
// consecutive ones per block as fit in max_rows rows.  4 ints per block: (row0, n_rows, 0, 0).
void build_window_blocks(const std::vector<int32_t>& cu, int32_t max_rows, std::vector<int32_t>* blocks) {
  blocks->clear();
  int32_t row0 = cu.empty() ? 0 : cu[0], rows = 0;
  for (size_t s = 0; s + 1 < cu.size(); ++s) {
    const int32_t len = cu[s + 1] - cu[s];
    if (rows > 0 && rows + len > max_rows) {
      blocks->insert(blocks->end(), {row0, rows, 0, 0});
      row0 = cu[s]; rows = 0;
    }
    rows += len;
  }
  if (rows > 0) blocks->insert(blocks->end(), {row0, rows, 0, 0});
}
// bounds[row] = (first row, end row) of the segment that holds `row`
void fill_window_bounds(const std::vector<int32_t>& cu, int32_t* bounds) {
  for (size_t s = 0; s + 1 < cu.size(); ++s)
    for (int32_t r = cu[s]; r < cu[s + 1]; ++r) { bounds[2 * r] = cu[s]; bounds[2 * r + 1] = cu[s + 1]; }
}

void normalize_lut(const zv_cfg* cfg, float* lut) {
  // both torchvision conventions: HF builds the same fp32 mean / std tensors and divides with IEEE fp32 on either device
  if (cfg->resample_kind == ZV_RESAMPLE_TORCHVISION || cfg->resample_kind == ZV_RESAMPLE_TORCHVISION_CUDA) {
    // TorchvisionBackend.rescale_and_normalize: mean' = f32(mean) * f32(1 / rescale), std' likewise, (f32(v) - mean') / std'
    const float inv = (float)(1.0 / cfg->rescale);
    for (int c = 0; c < 3; ++c) {
      const float m = cfg->mean[c] * inv, s = cfg->std[c] * inv;
      for (int v = 0; v < 256; ++v) lut[c * 256 + v] = ((float)v - m) / s;
    }
    return;
  }
  for (int c = 0; c < 3; ++c)
    for (int v = 0; v < 256; ++v) {
      float x = (float)((double)v * cfg->rescale);      // rescale: f64 product, then cast to f32
      lut[c * 256 + v] = (x - cfg->mean[c]) / cfg->std[c];  // normalize: f32 subtract, f32 divide
    }
}

}  // namespace zv

using namespace zv;

extern "C" {

const char* zv_version(void) { return "zoomvit-b200 0.3 (sm_100a)"; }
const char* zv_last_error(void) { return g_err.c_str(); }
int64_t zv_last_launch_count(void) { return g_launches; }

void zv_default_cfg(zv_cfg* c) {
  std::memset(c, 0, sizeof *c);
  c->patch = 14; c->merge = 2; c->temporal = 2; c->window = 112; c->min_size = 512;
  c->depth = 32; c->hidden = 1280; c->heads = 16; c->inter = 3420; c->out_hidden = 2048;
  c->fullatt_mask_lo = (int32_t)((1u << 7) | (1u << 15) | (1u << 23) | (1u << 31));
  c->min_pixels = 56 * 56; c->max_pixels = 28 * 28 * 1280;
  c->rescale = 1.0 / 255;
  c->mean[0] = 0.48145466f; c->mean[1] = 0.4578275f; c->mean[2] = 0.40821073f;
  c->std[0] = 0.26862954f; c->std[1] = 0.26130258f; c->std[2] = 0.27577711f;
  c->eps = 1e-6f;
  c->op_dtype = ZV_F16;      // the dtype the reference's eval loop runs in (infer.py:149); bf16 operands are opt-in
}

int zv_cut_box(int32_t img_w, int32_t img_h, const double* b, int32_t min_size, int32_t* out) {
  if (!b || !out) return fail(ZV_EINVAL, "zv_cut_box: null argument");
  int64_t x1 = py_int(b[0]), y1 = py_int(b[1]), x2 = py_int(b[2]), y2 = py_int(b[3]);
  int64_t width = x2 - x1, height = y2 - y1;
  if (width < min_size || height < min_size) {
    int64_t cx = floordiv(x1 + x2, 2), cy = floordiv(y1 + y2, 2);
    int64_t nx1 = cx - min_size / 2, ny1 = cy - min_size / 2;
    int64_t nx2 = nx1 + min_size, ny2 = ny1 + min_size;
    if (nx1 < 0) { nx2 += -nx1; nx1 = 0; }
    if (ny1 < 0) { ny2 += -ny1; ny1 = 0; }
    if (nx2 > img_w) { nx1 -= nx2 - img_w; nx2 = img_w; }
    if (ny2 > img_h) { ny1 -= ny2 - img_h; ny2 = img_h; }
    nx1 = std::max<int64_t>(0, nx1);
    ny1 = std::max<int64_t>(0, ny1);
    nx2 = std::min<int64_t>(img_w, nx1 + min_size);
    ny2 = std::min<int64_t>(img_h, ny1 + min_size);
    x1 = nx1; y1 = ny1; x2 = nx2; y2 = ny2;
  }
  out[0] = (int32_t)x1; out[1] = (int32_t)y1; out[2] = (int32_t)x2; out[3] = (int32_t)y2;
  return ZV_OK;
}

int zv_resize_dims(int32_t w, int32_t h, int32_t max_size, int32_t* wh, double* inv_scale) {
  if (!wh) return fail(ZV_EINVAL, "zv_resize_dims: null argument");
  double scale = (double)max_size / (double)std::max(w, h);
  if (scale < 1) {
    wh[0] = (int32_t)((double)w * scale);
    wh[1] = (int32_t)((double)h * scale);
  } else {
    wh[0] = w; wh[1] = h;
  }
  if (inv_scale) *inv_scale = 1 / scale;
  return ZV_OK;
}

// resize_image() variants of the reference: 0 infer.py:78-85 / demo.py:86-93, 1 SFT.py:76-81, 2 customized_funcs.py:76-85
int zv_resize_dims_ex(int32_t w, int32_t h, int32_t max_size, int32_t mode, int32_t* wh, double* inv_scale) {
  if (!wh || w <= 0 || h <= 0 || max_size <= 0) return fail(ZV_EINVAL, "zv_resize_dims_ex: bad argument");
  if (mode < 0 || mode > 2) return fail(ZV_EINVAL, "zv_resize_dims_ex: mode %d (0 infer/demo, 1 SFT, 2 customized_funcs)", mode);
  double scale = (double)max_size / (double)std::max(w, h);
  if (mode == 2) {
    const double min_scale = 30.0 / (double)std::min(w, h);      // customized_funcs.py:79-80
    scale = std::max(min_scale, scale);
  }
  if (mode == 1 || scale < 1) {                                   // SFT.py resizes unconditionally (may upscale)
    wh[0] = (int32_t)((double)w * scale);
    wh[1] = (int32_t)((double)h * scale);
  } else {
    wh[0] = w; wh[1] = h;
  }
  if (inv_scale) *inv_scale = 1 / scale;
  return ZV_OK;
}

// SFT.py:83-125 cut_image: small boxes take the 512-square rule of infer.py; boxes with both sides >= min_size are cropped,
// resized so that the shorter side is min_size, and centre-cropped to min_size x min_size.
int zv_cut_box_sft(int32_t img_w, int32_t img_h, const double* b, int32_t min_size, int32_t* box, int32_t* resized_wh,
                   int32_t* center_box) {
  if (!b || !box || !resized_wh || !center_box) return fail(ZV_EINVAL, "zv_cut_box_sft: null argument");
  int rc = zv_cut_box(img_w, img_h, b, min_size, box);
  if (rc) return rc;
  const int64_t x1 = py_int(b[0]), y1 = py_int(b[1]), x2 = py_int(b[2]), y2 = py_int(b[3]);
  resized_wh[0] = resized_wh[1] = 0;
  center_box[0] = center_box[1] = center_box[2] = center_box[3] = 0;
  if (x2 - x1 < min_size || y2 - y1 < min_size) return ZV_OK;   // the square branch: the crop is the result
  const int32_t w = box[2] - box[0], h = box[3] - box[1];
  const double scale = (double)min_size / (double)std::min(w, h);
  const int32_t nw = (int32_t)((double)w * scale), nh = (int32_t)((double)h * scale);
  resized_wh[0] = nw; resized_wh[1] = nh;
  const int32_t left = (int32_t)floordiv(nw - min_size, 2), top = (int32_t)floordiv(nh - min_size, 2);
  center_box[0] = left; center_box[1] = top; center_box[2] = left + min_size; center_box[3] = top + min_size;
  return ZV_OK;
}

int zv_smart_resize(int32_t height, int32_t width, int32_t factor, int64_t min_pixels, int64_t max_pixels,
                    int32_t* out) {
  if (!out || height <= 0 || width <= 0 || factor <= 0)
    return fail(ZV_EINVAL, "zv_smart_resize: bad argument (h=%d w=%d factor=%d)", height, width, factor);
  double ar = (double)std::max(height, width) / (double)std::min(height, width);
  if (ar > 200)
    return fail(ZV_EINVAL_ASPECT, "absolute aspect ratio must be smaller than 200, got %.17g", ar);
  // Python round(): half to even == nearbyint under the default rounding mode
  int64_t h_bar = (int64_t)std::nearbyint((double)height / factor) * factor;
  int64_t w_bar = (int64_t)std::nearbyint((double)width / factor) * factor;
  if (h_bar * w_bar > max_pixels) {
    double beta = std::sqrt((double)((int64_t)height * width) / (double)max_pixels);
    h_bar = std::max<int64_t>(factor, (int64_t)std::floor((double)height / beta / factor) * factor);
    w_bar = std::max<int64_t>(factor, (int64_t)std::floor((double)width / beta / factor) * factor);
  } else if (h_bar * w_bar < min_pixels) {
    double beta = std::sqrt((double)min_pixels / (double)((int64_t)height * width));
    h_bar = (int64_t)std::ceil((double)height * beta / factor) * factor;
    w_bar = (int64_t)std::ceil((double)width * beta / factor) * factor;
  }
  out[0] = (int32_t)h_bar; out[1] = (int32_t)w_bar;
  return ZV_OK;
}

int zv_geometry(const zv_cfg* cfg, int32_t n, const int32_t* img_hw, const double* bbox, int32_t* crop_box,
                int32_t* resized_hw, int64_t* grid_thw) {
  if (!cfg || n < 0 || !img_hw || !crop_box || !resized_hw || !grid_thw)
    return fail(ZV_EINVAL, "zv_geometry: null argument");
  const int32_t factor = cfg->patch * cfg->merge;
  for (int32_t i = 0; i < n; ++i) {
    int32_t h = img_hw[2 * i], w = img_hw[2 * i + 1];
    int32_t* box = crop_box + 4 * i;
    if (bbox && cfg->min_size < 0) {            // boxes are final crop boxes (Image.crop semantics, int())
      for (int k = 0; k < 4; ++k) box[k] = (int32_t)py_int(bbox[4 * i + k]);
    } else if (bbox) {
      int rc = zv_cut_box(w, h, bbox + 4 * i, cfg->min_size, box);
      if (rc) return rc;
    } else {
      box[0] = 0; box[1] = 0; box[2] = w; box[3] = h;
    }
    if (box[2] < box[0]) return fail(ZV_EINVAL_BOX, "Coordinate 'right' is less than 'left'");
    if (box[3] < box[1]) return fail(ZV_EINVAL_BOX, "Coordinate 'lower' is less than 'upper'");
    int32_t cw = box[2] - box[0], ch = box[3] - box[1];
    if (cw == 0 || ch == 0) return fail(ZV_EINVAL, "zv_geometry: crop %d is empty (%dx%d)", i, cw, ch);
    int rc = zv_smart_resize(ch, cw, factor, cfg->min_pixels, cfg->max_pixels, resized_hw + 2 * i);
    if (rc) return rc;
    grid_thw[3 * i] = 1;
    grid_thw[3 * i + 1] = resized_hw[2 * i] / cfg->patch;
    grid_thw[3 * i + 2] = resized_hw[2 * i + 1] / cfg->patch;
  }
  return ZV_OK;
}

int32_t zv_resample_ksize(int32_t in_size, int32_t out_size) {
  if (in_size <= 0 || out_size <= 0) return fail(ZV_EINVAL, "zv_resample_ksize: bad size");
  return resample_ksize(in_size, out_size);
}

int zv_resample_coeffs(int32_t in_size, int32_t out_size, int32_t* bounds, int32_t* kk) {
  if (in_size <= 0 || out_size <= 0 || !bounds || !kk) return fail(ZV_EINVAL, "zv_resample_coeffs: bad argument");
  return zv_resample_coeffs_ex(ZV_RESAMPLE_PIL, in_size, out_size, bounds, kk, nullptr);
}

int zv_resample_coeffs_ex(int32_t kind, int32_t in_size, int32_t out_size, int32_t* bounds, int32_t* kk, int32_t* precision) {
  if (in_size <= 0 || out_size <= 0 || !bounds || !kk) return fail(ZV_EINVAL, "zv_resample_coeffs_ex: bad argument");
  int rc = check_resample_kind(kind, "zv_resample_coeffs_ex");
  if (rc) return rc;
  if (kind == ZV_RESAMPLE_TORCHVISION_CUDA)
    return fail(ZV_EINVAL, "zv_resample_coeffs_ex: resample_kind 2 (ZV_RESAMPLE_TORCHVISION_CUDA) resamples in fp32 and has no "
                           "integer taps");
  AxisCoeffs c;
  resample_coeffs(kind, in_size, out_size, &c);
  std::memcpy(bounds, c.bounds.data(), c.bounds.size() * sizeof(int32_t));
  std::memcpy(kk, c.kk.data(), c.kk.size() * sizeof(int32_t));
  if (precision) *precision = c.precision;
  return ZV_OK;
}

int zv_normalize_lut(const zv_cfg* cfg, float* lut) {
  if (!cfg || !lut) return fail(ZV_EINVAL, "zv_normalize_lut: null argument");
  int rc = check_resample_kind(cfg->resample_kind, "zv_normalize_lut");
  if (rc) return rc;
  normalize_lut(cfg, lut);
  return ZV_OK;
}

// ------------------------------------------------------------------------------------------------ plan
static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

int zv_plan_create(const zv_cfg* cfg, int32_t n, const int64_t* grid, zv_plan** out) {
  if (!cfg || n <= 0 || !grid || !out) return fail(ZV_EINVAL, "zv_plan_create: bad argument");
  const int32_t m = cfg->merge, unit = m * m;
  const int32_t ws = cfg->window / cfg->merge / cfg->patch;   // 4 merged tokens per window side
  if (ws <= 0) return fail(ZV_EINVAL, "zv_plan_create: window smaller than a merge group");
  zv_plan* p = new zv_plan();
  p->cfg = *cfg;
  p->n_images = n;
  p->grid_thw.assign(grid, grid + 3 * (size_t)n);
  int64_t S = 0;
  for (int32_t i = 0; i < n; ++i) {
    int64_t t = grid[3 * i], gh = grid[3 * i + 1], gw = grid[3 * i + 2];
    if (t <= 0 || gh <= 0 || gw <= 0 || gh % m || gw % m) {
      delete p;
      return fail(ZV_EINVAL, "zv_plan_create: grid_thw[%d] = (%lld,%lld,%lld) not positive multiples of merge", i,
                  (long long)t, (long long)gh, (long long)gw);
    }
    S += t * gh * gw;
  }
  if (S > (int64_t)1 << 30) { delete p; return fail(ZV_EINVAL, "zv_plan_create: too many patches"); }
  p->S = S;
  p->T = S / unit;
  p->pos_ids.resize((size_t)S * 2);
  p->window_index.reserve(p->T);
  p->cu_window_raw.push_back(0);
  p->cu_full.push_back(0);
  int64_t row = 0, tok_base = 0;
  for (int32_t i = 0; i < n; ++i) {
    const int64_t t = grid[3 * i], gh = grid[3 * i + 1], gw = grid[3 * i + 2];
    const int64_t lh = gh / m, lw = gw / m;
    // rot_pos_emb ids (HF :382-401): merge-group raster order, repeated t times
    for (int64_t tt = 0; tt < t; ++tt)
      for (int64_t bh = 0; bh < lh; ++bh)
        for (int64_t bw = 0; bw < lw; ++bw)
          for (int32_t mh = 0; mh < m; ++mh)
            for (int32_t mw = 0; mw < m; ++mw) {
              p->pos_ids[2 * row] = (int32_t)(bh * m + mh);
              p->pos_ids[2 * row + 1] = (int32_t)(bw * m + mw);
              ++row;
            }
    // get_window_index (HF :411-451): pad is a FULL extra window when the grid is already divisible
    const int64_t pad_h = ws - lh % ws, pad_w = ws - lw % ws;
    const int64_t nwh = (lh + pad_h) / ws, nww = (lw + pad_w) / ws;
    for (int64_t tt = 0; tt < t; ++tt)
      for (int64_t wy = 0; wy < nwh; ++wy)
        for (int64_t wx = 0; wx < nww; ++wx) {
          int32_t cnt = 0;
          for (int64_t a = 0; a < ws; ++a)
            for (int64_t b = 0; b < ws; ++b) {
              int64_t y = wy * ws + a, x = wx * ws + b;
              if (y < lh && x < lw) {
                p->window_index.push_back(tok_base + tt * lh * lw + y * lw + x);
                ++cnt;
              }
            }
          p->cu_window_raw.push_back(p->cu_window_raw.back() + cnt * unit);
        }
    tok_base += t * lh * lw;
    for (int64_t tt = 0; tt < t; ++tt) p->cu_full.push_back(p->cu_full.back() + (int32_t)(gh * gw));
  }
  // torch.unique_consecutive (HF :476)
  for (int32_t v : p->cu_window_raw)
    if (p->cu_window.empty() || p->cu_window.back() != v) p->cu_window.push_back(v);
  p->reverse_index.resize(p->T);
  for (int64_t i = 0; i < p->T; ++i) p->reverse_index[p->window_index[i]] = i;

  // full layers (tcgen05 kernel): 128-row q tiles inside one whole-image segment: (q0, q_len, seg_begin, seg_end)
  for (size_t s = 0; s + 1 < p->cu_full.size(); ++s)
    for (int32_t q0 = p->cu_full[s]; q0 < p->cu_full[s + 1]; q0 += 128) {
      p->full_tiles.push_back(q0);
      p->full_tiles.push_back(std::min(128, p->cu_full[s + 1] - q0));
      p->full_tiles.push_back(p->cu_full[s]);
      p->full_tiles.push_back(p->cu_full[s + 1]);
    }
  // window layers (tcgen05 kernel): consecutive whole windows packed greedily into row blocks of <= 128 rows
  build_window_blocks(p->cu_window, 128, &p->win_blocks);
  p->n_win_blocks = (int32_t)(p->win_blocks.size() / 4);
  p->n_full_tiles = (int32_t)(p->full_tiles.size() / 4);

  int32_t max_pos = 0;
  for (int32_t i = 0; i < n; ++i)
    max_pos = std::max<int32_t>(max_pos, (int32_t)std::max(grid[3 * i + 1], grid[3 * i + 2]));
  zv::PlanDeviceLayout& d = p->dev;
  int64_t off = 0;
  const int32_t half_rot = cfg->hidden / cfg->heads / 4;                                   // 20
  d.max_pos = max_pos;
  d.off_pos = off; off = align_up(off + (int64_t)S * 2 * sizeof(int32_t), 256);
  d.off_rope = off; off = align_up(off + (int64_t)max_pos * half_rot * 2 * sizeof(float), 256);
  d.off_widx = off; off = align_up(off + p->T * (int64_t)sizeof(int32_t), 256);
  d.off_full_tiles = off; off = align_up(off + (int64_t)p->full_tiles.size() * sizeof(int32_t), 256);
  d.off_win_blocks = off; off = align_up(off + (int64_t)p->win_blocks.size() * sizeof(int32_t), 256);
  d.off_win_bounds = off; off = align_up(off + (int64_t)(S + 136) * 2 * sizeof(int32_t), 256);   // + a block of zero padding: the kernel bulk-copies 130 rows from any block start
  d.bytes = off;
  *out = p;
  return ZV_OK;
}

void zv_plan_free(zv_plan* p) { delete p; }
}  // extern "C"

// Byte image of the device-side tables, laid out per PlanDeviceLayout.
void zv::plan_device_image(const zv_plan* p, std::vector<uint8_t>* image) {
  const zv::PlanDeviceLayout& d = p->dev;
  image->assign((size_t)d.bytes, 0);
  uint8_t* base = image->data();
  const int32_t unit = p->cfg.merge * p->cfg.merge;
  int32_t* pos = reinterpret_cast<int32_t*>(base + d.off_pos);
  int32_t* widx = reinterpret_cast<int32_t*>(base + d.off_widx);
  for (int64_t i = 0; i < p->T; ++i) {
    const int64_t g = p->window_index[i];
    widx[i] = (int32_t)g;
    std::memcpy(pos + 2 * unit * i, p->pos_ids.data() + 2 * unit * g, sizeof(int32_t) * 2 * unit);
  }
  // rotary table (HF :117-130): inv_freq_j = 1 / 10000^(2j/dim) with dim = head_dim/2, angle = pos * inv_freq_j
  // in fp32; cos/sin taken in double of that fp32 angle and rounded once.
  const int32_t dim = p->cfg.hidden / p->cfg.heads / 2, half_rot = dim / 2;
  float* rope = reinterpret_cast<float*>(base + d.off_rope);
  for (int32_t ps = 0; ps < d.max_pos; ++ps)
    for (int32_t j = 0; j < half_rot; ++j) {
      const float inv_freq = 1.0f / std::pow(10000.0f, (float)(2 * j) / (float)dim);
      const float ang = (float)ps * inv_freq;
      rope[((size_t)ps * half_rot + j) * 2] = (float)std::cos((double)ang);
      rope[((size_t)ps * half_rot + j) * 2 + 1] = (float)std::sin((double)ang);
    }
  std::memcpy(base + d.off_full_tiles, p->full_tiles.data(), p->full_tiles.size() * sizeof(int32_t));
  std::memcpy(base + d.off_win_blocks, p->win_blocks.data(), p->win_blocks.size() * sizeof(int32_t));
  fill_window_bounds(p->cu_window, reinterpret_cast<int32_t*>(base + d.off_win_bounds));
}

extern "C" {
int64_t zv_plan_num_patches(const zv_plan* p) { return p ? p->S : 0; }
int64_t zv_plan_num_tokens(const zv_plan* p) { return p ? p->T : 0; }
const int64_t* zv_plan_window_index(const zv_plan* p) { return p->window_index.data(); }
const int64_t* zv_plan_reverse_index(const zv_plan* p) { return p->reverse_index.data(); }
const int32_t* zv_plan_cu_window(const zv_plan* p, int32_t* n) { if (n) *n = (int32_t)p->cu_window.size(); return p->cu_window.data(); }
const int32_t* zv_plan_cu_window_raw(const zv_plan* p, int32_t* n) { if (n) *n = (int32_t)p->cu_window_raw.size(); return p->cu_window_raw.data(); }
const int32_t* zv_plan_cu_full(const zv_plan* p, int32_t* n) { if (n) *n = (int32_t)p->cu_full.size(); return p->cu_full.data(); }
const int32_t* zv_plan_pos_ids(const zv_plan* p) { return p->pos_ids.data(); }
int64_t zv_plan_device_bytes(const zv_plan* p) { return p ? p->dev.bytes : 0; }

}  // extern "C"
