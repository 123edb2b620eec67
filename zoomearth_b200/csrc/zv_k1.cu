// K1: fused crop -> Pillow-exact bicubic resize -> rescale/normalize (LUT) -> patchify-permute.
//
// Replaces, as one device pass over uint8 pixels:
//   PIL.Image.crop               reference src/eval/infer.py:72,75   (zero fill outside the image)
//   PIL.Image.resize(BICUBIC)    reference src/eval/infer.py:84, HF image_transforms.py:368
//                                (Pillow ImagingResample, 8 bpc: horizontal pass -> uint8 -> vertical pass)
//   rescale + normalize          HF image_transforms.py:89-124, 384-442   (exact 768-entry LUT)
//   patchify                     HF models/qwen2_vl/image_processing_pil_qwen2_vl.py:186-214
//
// The two resample passes cannot be merged (the intermediate is rounded to uint8), so the data flow is
//   source u8 (HWC) --hpass--> tmp u8 (only the rows the vertical pass needs) --vpass+LUT+permute--> patches.
// Integer arithmetic only, bit-identical to Pillow: 22-bit fixed-point taps computed on the host in fp64
// (zv_host.cpp), int32 sums.
//
// Main route (zv_k1_tc.cuh; row pitch a multiple of 4, downscales up to ~10x): both passes run as ONE transposing
// tcgen05 kernel (TMA -> kind::i8 UMMA -> TMEM epilogue), source -> T (transposed) -> U (the finished uint8 image), and a
// small kernel turns U into normalised patches.  The kernels below serve what that route declines: other row pitches,
// larger downscales.
//
// Fallback fast path (taps <= 45 per axis, 4-byte aligned image rows): the work is instruction-bound on the integer pipes
// (4 multiply-adds per source byte), so both passes run on dp4a.  Each 23-bit tap is split into three byte limbs
// (k = l0 + 256 l1 + 65536 l2, l2 signed); the host emits, per output index, a word-aligned tap window whose limb
// bytes are packed four taps to a word, so one dp4a does four taps of one limb and no per-thread realignment of the
// pixels is needed:
//   hpass_fast  a CTA stages 8 source rows x the span of 128 output columns into shared memory (16-byte cp.async of
//               the raw bytes, then a byte-permute pass to R/G/B planes); a thread owns one output column with its limb
//               words in registers, runs 4 rows x 3 channels, and writes tmp packed 4 rows to a word.
//   vpass_fast  tmp's row-quad words are directly dp4a operands along y; a warp owns output rows with their limb words
//               in registers and sweeps the columns coalesced; the CTA assembles two merge groups' patch rows in shared
//               memory and streams them out with 16-byte stores.
// Everything else (huge downscales, unaligned pitches) takes the plain per-tap kernels k1_hpass / k1_vpass.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <vector>

#include "zv_common.h"
#include "zv_gemm.h"
#include "zv_ptx.cuh"

namespace {

constexpr int kPrecisionBits = 22;
constexpr int kPatchElems = 1176;   // 3 * 2 * 14 * 14
constexpr int kMaxNW = 12;          // fast path: taps <= 4 * kMaxNW - 3 = 45 (5000 px -> 512 px is 41 taps)
constexpr int kHRows = 8;           // hpass_fast: source rows per CTA (two row quads)
constexpr int kHCols = 128;         // hpass_fast: output columns per CTA

struct K1Crop {
  const uint8_t* src;      // image base (device)
  int64_t pitch;           // bytes per image row
  int64_t tmp_off;         // byte offset of this crop's intermediate in the workspace
  int64_t out_row0;        // first patch row of this crop in the output
  int32_t src_h, src_w;
  int32_t x0, y0;          // crop origin in image coordinates (may be negative / extend outside)
  int32_t cw, ch;          // crop extent
  int32_t ow, oh;          // resized extent (multiples of 28)
  int32_t ksh, ksv;        // taps per output column / row
  int32_t ybox0, nrows;    // crop rows [ybox0, ybox0 + nrows) feed the vertical pass (fast path: ybox0 % 4 == 0)
  int32_t off_bh, off_kh, off_bv, off_kv;  // int32 offsets into the coefficient area (bounds, taps)
  int32_t off_lh, off_lv;  // int32 offsets of the dp4a limb tables (fast path)
  int32_t nwh, nwv;        // words per tap window (fast path), 0 = generic path
  int32_t lh, lw;          // merge-group grid (gh/2, gw/2)
  int32_t fast;            // 1: tmp is row-quad packed (fast path), 0: plain rows
  int32_t ks_mma;          // horizontal pass on IMMA: 32-byte K steps per 8-column block (1..4), 0 = dp4a kernel
  int32_t off_mh;          // int32 offset of the IMMA fragment table of the horizontal axis
  int32_t tc;               // 1: both passes on the tensor cores (k1_resample_tc), the kernels below are not used
  uint8_t* dst;            // uint8 output mode (zv_resize_u8): (oh, ow, 3) image, row pitch dst_pitch bytes
  int64_t dst_pitch;
};

// Block -> (crop, local block) through the launch's own prefix array (crops of one kernel class only).
__device__ __forceinline__ int find_slot(const int32_t* __restrict__ blk0, int n, int blk) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (blk0[mid] <= blk) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ int clip8(int v) { return min(255, max(0, v)); }
__device__ __forceinline__ int dp4a_uu(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {   // a unsigned bytes, b signed bytes
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// sum_t px_t * k_t from the three limb sums, rounded like Pillow's 8bpc passes (not yet clipped)
__device__ __forceinline__ int finish_raw(int a0, int a1, int a2) {
  return (a2 * 65536 + (a1 * 256 + (a0 + (1 << (kPrecisionBits - 1))))) >> kPrecisionBits;
}
__device__ __forceinline__ int finish8(int a0, int a1, int a2) { return clip8(finish_raw(a0, a1, a2)); }
// four rounded sums -> four bytes, each saturated to [0, 255] (Pillow's clip8), v0 in the low byte
__device__ __forceinline__ uint32_t pack4_sat(int v0, int v1, int v2, int v3) {
  uint32_t hi, d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi) : "r"(v3), "r"(v2), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(v1), "r"(v0), "r"(hi));
  return d;
}

// Position of merge group (my, mx) in the tower's window order (closed form of argsort(window_index),
// HF modeling_qwen2_5_vl.py:411-451): windows of ws x ws merge groups, row-major over windows, row-major inside.
__host__ __device__ __forceinline__ int window_pos(int my, int mx, int lh, int lw, int ws) {
  // ws = 4 for every Qwen2.5-VL tower (window 112 / merge 2 / patch 14): shifts instead of two runtime divisions
  const int wy = ws == 4 ? my >> 2 : my / ws, wx = ws == 4 ? mx >> 2 : mx / ws;
  const int bh = ws < lh - wy * ws ? ws : lh - wy * ws, bw = ws < lw - wx * ws ? ws : lw - wx * ws;
  return wy * ws * lw + wx * ws * bh + (my - wy * ws) * bw + (mx - wx * ws);
}

template <typename OutT> __device__ __forceinline__ OutT to_out(float v) {
  if constexpr (std::is_same<OutT, __nv_bfloat16>::value) return __float2bfloat16_rn(v);
  else if constexpr (std::is_same<OutT, __half>::value) return __float2half_rn(v);
  else return v;
}

// ------------------------------------------------------------------------------------------------ generic path
// Horizontal pass.  One thread = one (tmp row, output column), all 3 channels.
__global__ void __launch_bounds__(256) k1_hpass(const K1Crop* __restrict__ crops, const int32_t* __restrict__ ids,
                                                const int32_t* __restrict__ blk0, int n_cls,
                                                const int32_t* __restrict__ coef, uint8_t* __restrict__ ws) {
  zv::ptx::pdl_wait();
  const int slot = find_slot(blk0, n_cls, blockIdx.x);
  const K1Crop c = crops[ids[slot]];
  const int64_t item = (int64_t)(blockIdx.x - blk0[slot]) * blockDim.x + threadIdx.x;
  if (item >= (int64_t)c.nrows * c.ow) return;
  const int r = (int)(item / c.ow), xx = (int)(item % c.ow);
  const int y_img = c.y0 + c.ybox0 + r;
  const int xmin = coef[c.off_bh + 2 * xx], cnt = coef[c.off_bh + 2 * xx + 1];
  const int32_t* __restrict__ k = coef + c.off_kh + (int64_t)xx * c.ksh;
  int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
  if (y_img >= 0 && y_img < c.src_h) {
    const uint8_t* __restrict__ row = c.src + (int64_t)y_img * c.pitch;
    for (int t = 0; t < cnt; ++t) {
      const int x_img = c.x0 + xmin + t;
      if (x_img >= 0 && x_img < c.src_w) {
        const int kv = __ldg(k + t);
        const uint8_t* px = row + 3 * (int64_t)x_img;
        a0 += (int)__ldg(px) * kv;
        a1 += (int)__ldg(px + 1) * kv;
        a2 += (int)__ldg(px + 2) * kv;
      }
    }
  }
  uint8_t* o = ws + c.tmp_off + ((int64_t)r * c.ow + xx) * 3;
  o[0] = (uint8_t)clip8(a0 >> kPrecisionBits);
  o[1] = (uint8_t)clip8(a1 >> kPrecisionBits);
  o[2] = (uint8_t)clip8(a2 >> kPrecisionBits);
}

// Vertical pass + LUT normalise + patchify.  One block = one 2x2 merge group (28 x 28 pixels, 4 patch rows).
template <typename OutT>
__global__ void __launch_bounds__(256) k1_vpass(const K1Crop* __restrict__ crops, const int32_t* __restrict__ ids,
                                                const int32_t* __restrict__ blk0, int n_cls,
                                                const int32_t* __restrict__ coef, const uint8_t* __restrict__ ws,
                                                const float* __restrict__ lut, OutT* __restrict__ out, int row_order,
                                                int wsz) {
  __shared__ __align__(16) OutT stage[4 * kPatchElems];
  __shared__ float s_lut[768];
  zv::ptx::pdl_wait();
  const int slot = find_slot(blk0, n_cls, blockIdx.x);
  const K1Crop c = crops[ids[slot]];
  const int g = blockIdx.x - blk0[slot];        // merge group, raster order inside the crop
  const int my = g / c.lw, mx = g % c.lw;
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = lut[i];
  __syncthreads();
  const uint8_t* __restrict__ tmp = ws + c.tmp_off;
  const int64_t tpitch = (int64_t)c.ow * 3;
  for (int item = threadIdx.x; item < 28 * 84; item += blockDim.x) {
    const int yl = item / 84, col = item % 84;             // col = xl * 3 + ch
    const int xl = col / 3, ch = col % 3;
    const int yy = my * 28 + yl;
    const int ymin = coef[c.off_bv + 2 * yy] - c.ybox0, cnt = coef[c.off_bv + 2 * yy + 1];
    const int32_t* __restrict__ k = coef + c.off_kv + (int64_t)yy * c.ksv;
    const uint8_t* __restrict__ p = tmp + (int64_t)ymin * tpitch + (int64_t)(mx * 28) * 3 + col;
    int acc = 1 << (kPrecisionBits - 1);
    for (int t = 0; t < cnt; ++t) acc += (int)__ldg(p + (int64_t)t * tpitch) * __ldg(k + t);
    const float v = s_lut[ch * 256 + clip8(acc >> kPrecisionBits)];
    const int j = (yl / 14) * 2 + (xl / 14);
    const int e = j * kPatchElems + ch * 392 + (yl % 14) * 14 + (xl % 14);
    const OutT o = to_out<OutT>(v);
    stage[e] = o;            // temporal frame 0
    stage[e + 196] = o;      // temporal frame 1 = the repeated frame (HF :189-193)
  }
  __syncthreads();
  const int pos = row_order == ZV_ORDER_WINDOW ? window_pos(my, mx, c.lh, c.lw, wsz) : g;
  uint4* dst = reinterpret_cast<uint4*>(out + (c.out_row0 + 4 * (int64_t)pos) * kPatchElems);
  const uint4* srcv = reinterpret_cast<const uint4*>(stage);
  constexpr int kVec = 4 * kPatchElems * (int)sizeof(OutT) / 16;
  for (int i = threadIdx.x; i < kVec; i += blockDim.x) dst[i] = srcv[i];
}

// ------------------------------------------------------------------------------------------------ fast path
// Limb table of one axis: per output index, (1 + 3 NW) ints: first word of the tap window (in 4-sample words from the
// axis origin), then NW words of limb 0, NW of limb 1, NW of limb 2 (signed bytes); taps outside the window are 0.

// Both fast kernels are persistent: the grid is a few CTAs per SM and every CTA walks a host-built work list
// (int4 items) with a stride of gridDim.x.  An item fixes everything that needs dependent global loads (crop
// descriptor, tap tables of the item's columns / rows) and then covers several units of streaming work, whose loads
// are double-buffered with cp.async so that the copy of unit u+1 runs under the dp4a loop of unit u.

// Horizontal pass on dp4a.  Item = (crop, 128-column chunk, first strip, strips): the CTA keeps the chunk's limb words
// in registers (thread = output column x row quad) and streams 8-row strips of the source through shared memory.
template <int NW>
__global__ void __launch_bounds__(256, NW <= 2 ? 4 : 3) k1_hpass_fast(const K1Crop* __restrict__ crops, const int4* __restrict__ items,
                                                     int n_items, const int32_t* __restrict__ coef,
                                                     uint8_t* __restrict__ ws, int seg_words_max) {
  extern __shared__ uint32_t planes[];            // [8 rows][3 planes][seg_words_max], then raw[2][8][raw_pitch]
  const int raw_pitch = (seg_words_max * 12 + 32 + 15) & ~15;
  uint8_t* raw = reinterpret_cast<uint8_t*>(planes + kHRows * 3 * seg_words_max);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kStride = 1 + 3 * NW;
  zv::ptx::pdl_wait();                // the source may be the previous kernel's output (zv_resize_u8 -> zv_preprocess)

  for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
    const int4 item = __ldg(items + it);
    const K1Crop& c = crops[item.x];
    const uint8_t* __restrict__ src = c.src;
    const int64_t pitch = c.pitch;
    const int src_h = c.src_h, ow = c.ow, nq = (c.nrows + 3) >> 2;
    const int y_base = c.y0 + c.ybox0;
    const int64_t row_bytes = 3 * (int64_t)c.src_w;
    const int32_t* __restrict__ lt = coef + c.off_lh;
    const int xx0 = item.y * kHCols, xx1 = min(ow, xx0 + kHCols);
    const int w_first = __ldg(lt + (int64_t)xx0 * kStride);               // window starts are monotone in xx
    const int seg_words = min(seg_words_max, __ldg(lt + (int64_t)(xx1 - 1) * kStride) + NW - w_first);
    const int64_t b0 = 3 * (int64_t)(c.x0 + w_first * 4);                 // first byte of the segment in a row (may be < 0)
    // this thread's output column: tap window start and limb words stay in registers for the whole item
    const int xx = xx0 + (threadIdx.x & (kHCols - 1));
    const int quad = threadIdx.x >> 7;                                    // 0, 1
    const bool col_ok = xx < xx1;
    int w0 = 0;
    uint32_t l0[NW], l1[NW], l2[NW];
    if (col_ok) {
      const int32_t* __restrict__ e = lt + (int64_t)xx * kStride;
      w0 = __ldg(e) - w_first;
#pragma unroll
      for (int k = 0; k < NW; ++k) { l0[k] = __ldg(e + 1 + k); l1[k] = __ldg(e + 1 + NW + k); l2[k] = __ldg(e + 1 + 2 * NW + k); }
    } else {
#pragma unroll
      for (int k = 0; k < NW; ++k) { l0[k] = 0; l1[k] = 0; l2[k] = 0; }
    }
    uint32_t* __restrict__ tmp_base = reinterpret_cast<uint32_t*>(ws + c.tmp_off);

    // stage A of strip s: raw bytes of its 8 row segments -> raw[buf] with 16-byte cp.async (warp w = row w); bytes
    // outside the image (box beyond the border) are zeros (Image.crop semantics).  Returns (rowp + b0) mod 16.
    auto issue = [&](const int strip, const int buf) -> int {
      const int y_img = y_base + strip * kHRows + warp;
      const bool row_ok = y_img >= 0 && y_img < src_h;
      const uint8_t* rowp = src + (int64_t)(row_ok ? y_img : 0) * pitch;
      const int delta = (int)((reinterpret_cast<uintptr_t>(rowp) + (uintptr_t)(b0 & 15) + 16) & 15);
      const int64_t g0 = b0 - delta;                                      // row byte offset of raw[0]; rowp + g0 is 16-aligned
      const int n_chunks = (delta + seg_words * 12 + 15) >> 4;
      uint8_t* rraw = raw + (buf * kHRows + warp) * raw_pitch;
      // chunks [ck_lo, ck_hi) lie wholly inside the image row: plain 16-byte async copies; the few others (box beyond
      // the left / right border, or the whole row outside the image) are assembled byte by byte with zero fill
      int ck_lo = 0, ck_hi = 0;
      if (row_ok) {
        ck_lo = g0 >= 0 ? 0 : (int)((-g0 + 15) >> 4);
        ck_hi = (int)min((int64_t)n_chunks, (row_bytes - g0) >> 4);
        ck_lo = min(ck_lo, n_chunks);
        ck_hi = max(ck_hi, ck_lo);
      }
      const uint32_t dst0 = (uint32_t)__cvta_generic_to_shared(rraw);
      const uint8_t* src0 = rowp + g0;
      for (int ck = lane; ck < n_chunks; ck += 32) {
        if (ck >= ck_lo && ck < ck_hi) {
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + 16 * ck), "l"(src0 + 16 * (int64_t)ck) : "memory");
        } else {
          const int64_t o = g0 + 16 * (int64_t)ck;
          uint32_t wv[4] = {0u, 0u, 0u, 0u};
          if (row_ok && o + 16 > 0 && o < row_bytes) {
#pragma unroll
            for (int k = 0; k < 16; ++k)
              if (o + k >= 0 && o + k < row_bytes) wv[k >> 2] |= (uint32_t)__ldg(rowp + o + k) << (8 * (k & 3));
          }
          *reinterpret_cast<uint4*>(rraw + 16 * ck) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      return delta;
    };

    int delta_cur = issue(item.z, 0);
    for (int s = 0; s < item.w; ++s) {
      const int strip = item.z + s;
      int delta_next = 0;
      if (s + 1 < item.w) {
        delta_next = issue(strip + 1, (s + 1) & 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();              // every warp is done with the planes of the previous strip; this strip's raw rows landed
      // ---- stage B: de-interleave this warp's row, 4 pixels (12 bytes) per lane step: RGBRGBRGBRGB -> R4 | G4 | B4
      {
        const uint8_t* rraw = raw + ((s & 1) * kHRows + warp) * raw_pitch;
        const uint32_t sh = (uint32_t)(delta_cur & 3) * 8;
        const uint32_t* wsrc = reinterpret_cast<const uint32_t*>(rraw + (delta_cur & ~3));
        uint32_t* p = planes + (warp * 3) * seg_words_max;
        if (sh == 0) {
          for (int wq = lane; wq < seg_words; wq += 32) {
            const uint32_t v0 = wsrc[3 * wq], v1 = wsrc[3 * wq + 1], v2 = wsrc[3 * wq + 2];
            p[wq] = __byte_perm(__byte_perm(v0, v1, 0x0630), v2, 0x5210);
            p[seg_words_max + wq] = __byte_perm(__byte_perm(v0, v1, 0x0741), v2, 0x6210);
            p[2 * seg_words_max + wq] = __byte_perm(__byte_perm(v0, v1, 0x0052), v2, 0x7410);
          }
        } else {
          for (int wq = lane; wq < seg_words; wq += 32) {
            const uint32_t x0 = wsrc[3 * wq], x1 = wsrc[3 * wq + 1], x2 = wsrc[3 * wq + 2], x3 = wsrc[3 * wq + 3];
            const uint32_t v0 = __funnelshift_r(x0, x1, sh), v1 = __funnelshift_r(x1, x2, sh), v2 = __funnelshift_r(x2, x3, sh);
            p[wq] = __byte_perm(__byte_perm(v0, v1, 0x0630), v2, 0x5210);
            p[seg_words_max + wq] = __byte_perm(__byte_perm(v0, v1, 0x0741), v2, 0x6210);
            p[2 * seg_words_max + wq] = __byte_perm(__byte_perm(v0, v1, 0x0052), v2, 0x7410);
          }
        }
      }
      delta_cur = delta_next;
      __syncthreads();
      // ---- compute: thread = (output column, row quad)
      const int q = strip * 2 + quad;
      if (col_ok && q < nq) {
        uint32_t* __restrict__ tmp4 = tmp_base + ((int64_t)q * ow + xx) * 3;
        const uint32_t* __restrict__ prow = planes + quad * 12 * seg_words_max + w0;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          int val[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            const uint32_t* __restrict__ p = prow + (r * 3 + ch) * seg_words_max;
            int a0 = 0, a1 = 0, a2 = 0;
#pragma unroll
            for (int k = 0; k < NW; ++k) {
              const uint32_t v = p[k];
              a0 = dp4a_uu(v, l0[k], a0);
              a1 = dp4a_uu(v, l1[k], a1);
              a2 = dp4a_us(v, l2[k], a2);
            }
            val[r] = finish_raw(a0, a1, a2);
          }
          tmp4[ch] = pack4_sat(val[0], val[1], val[2], val[3]);      // rows 4q..4q+3 of (xx, ch)
        }
      }
    }
    __syncthreads();                // the next item's first copy may land in raw[0] / its planes pass follows a barrier
  }
  zv::ptx::pdl_trigger();
}

// Horizontal pass on the tensor cores (mma.sync m16n8k32, u8 x u8 / u8 x s8 -> s32: exact).  dp4a retires 256 int8 MACs per
// clock per SM, IMMA.16832 2048 (measured, tools/micro/imma_rate.cu), and a Pillow-exact pass is 3 limb products per tap, so
// the dp4a kernel is bound by its dp4a pipe.  Here D[16 rows x 8 output columns] = A[16 rows x 32 KS source bytes] (one colour
// plane of the staged strip, row-major: a fragment register is one 32-bit shared load) x B[32 KS x 8] (one limb of the
// columns' taps, zero outside each column's window; packed per lane by the host, resident in registers for the whole item),
// one accumulator set per limb.  A warp owns two 8-column blocks of the item's 128-column chunk; strips are 16 rows.  The
// finished bytes are regrouped across the four lanes of a row group into the row-quad words the vertical pass reads.
// Fragment table of an axis: per 8-column block 1 + 192 KS ints: first word of the block's source window, then
// [k step][limb][lane][2] fragment words.
__device__ __forceinline__ void imma_uu(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void imma_us(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
constexpr int kMRows = 16;          // hpass_mma: source rows per strip (four row quads)

template <int KS>
__global__ void __launch_bounds__(256, 2) k1_hpass_mma(const K1Crop* __restrict__ crops, const int4* __restrict__ items,
                                                       int n_items, const int32_t* __restrict__ coef,
                                                       uint8_t* __restrict__ ws, int plane_pitch) {
  extern __shared__ uint32_t planes[];            // [16 rows][3 planes][plane_pitch], then raw[2][16][raw_pitch]
  const int raw_pitch = (plane_pitch * 12 + 32 + 15) & ~15;
  uint8_t* raw = reinterpret_cast<uint8_t*>(planes + kMRows * 3 * plane_pitch);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  constexpr int kStride = 1 + 192 * KS;
  zv::ptx::pdl_wait();

  for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
    const int4 item = __ldg(items + it);
    const K1Crop& c = crops[item.x];
    const uint8_t* __restrict__ src = c.src;
    const int64_t pitch = c.pitch;
    const int src_h = c.src_h, ow = c.ow, nq = (c.nrows + 3) >> 2;
    const int y_base = c.y0 + c.ybox0;
    const int64_t row_bytes = 3 * (int64_t)c.src_w;
    const int32_t* __restrict__ lt = coef + c.off_mh;
    const int xx0 = item.y * kHCols;
    const int nb0 = xx0 >> 3, nblocks = min(kHCols / 8, (ow - xx0 + 7) >> 3);
    const int w_first = __ldg(lt + (int64_t)nb0 * kStride);                // window starts are monotone in the block index
    const int seg_words = min(plane_pitch, __ldg(lt + (int64_t)(nb0 + nblocks - 1) * kStride) + 8 * KS - w_first);
    const int64_t b0 = 3 * (int64_t)(c.x0 + w_first * 4);                  // first byte of the segment in a row (may be < 0)
    // this warp's two column blocks: window start and B fragments stay in registers for the whole item
    int wq0[2];
    bool blk_ok[2];
    uint32_t bf[2][KS][3][2];
#pragma unroll
    for (int sblk = 0; sblk < 2; ++sblk) {
      const int nb = warp + 8 * sblk;
      blk_ok[sblk] = nb < nblocks;
      const int32_t* __restrict__ e = lt + (int64_t)(nb0 + (blk_ok[sblk] ? nb : 0)) * kStride;
      wq0[sblk] = __ldg(e) - w_first;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
#pragma unroll
        for (int l = 0; l < 3; ++l) {
          const int32_t* f = e + 1 + ((ks * 3 + l) * 32 + lane) * 2;       // (the table is only 4-byte aligned)
          bf[sblk][ks][l][0] = (uint32_t)__ldg(f); bf[sblk][ks][l][1] = (uint32_t)__ldg(f + 1);
        }
    }
    uint32_t* __restrict__ tmp_base = reinterpret_cast<uint32_t*>(ws + c.tmp_off);

    // stage A of strip s: raw bytes of its 16 row segments -> raw[buf] (warp w = rows 2w, 2w + 1); see k1_hpass_fast
    auto issue = [&](const int strip, const int buf, int (&delta)[2]) {
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int rl = 2 * warp + rr;
        const int y_img = y_base + strip * kMRows + rl;
        const bool row_ok = y_img >= 0 && y_img < src_h;
        const uint8_t* rowp = src + (int64_t)(row_ok ? y_img : 0) * pitch;
        const int dl = (int)((reinterpret_cast<uintptr_t>(rowp) + (uintptr_t)(b0 & 15) + 16) & 15);
        const int64_t g0 = b0 - dl;
        const int n_chunks = (dl + seg_words * 12 + 15) >> 4;
        uint8_t* rraw = raw + (buf * kMRows + rl) * raw_pitch;
        int ck_lo = 0, ck_hi = 0;
        if (row_ok) {
          ck_lo = g0 >= 0 ? 0 : (int)((-g0 + 15) >> 4);
          ck_hi = (int)min((int64_t)n_chunks, (row_bytes - g0) >> 4);
          ck_lo = min(ck_lo, n_chunks);
          ck_hi = max(ck_hi, ck_lo);
        }
        const uint32_t dst0 = (uint32_t)__cvta_generic_to_shared(rraw);
        const uint8_t* src0 = rowp + g0;
        for (int ck = lane; ck < n_chunks; ck += 32) {
          if (ck >= ck_lo && ck < ck_hi) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + 16 * ck), "l"(src0 + 16 * (int64_t)ck) : "memory");
          } else {
            const int64_t o = g0 + 16 * (int64_t)ck;
            uint32_t wv[4] = {0u, 0u, 0u, 0u};
            if (row_ok && o + 16 > 0 && o < row_bytes) {
#pragma unroll
              for (int k = 0; k < 16; ++k)
                if (o + k >= 0 && o + k < row_bytes) wv[k >> 2] |= (uint32_t)__ldg(rowp + o + k) << (8 * (k & 3));
            }
            *reinterpret_cast<uint4*>(rraw + 16 * ck) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
          }
        }
        delta[rr] = dl;
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };

    int delta_cur[2], delta_next[2] = {0, 0};
    issue(item.z, 0, delta_cur);
    for (int s = 0; s < item.w; ++s) {
      const int strip = item.z + s;
      if (s + 1 < item.w) {
        issue(strip + 1, (s + 1) & 1, delta_next);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();              // every warp is done with the planes of the previous strip; this strip's raw rows landed
      // ---- stage B: de-interleave this warp's two rows, 4 pixels (12 bytes) per lane step: RGBRGBRGBRGB -> R4 | G4 | B4
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int rl = 2 * warp + rr;
        const uint8_t* rraw = raw + ((s & 1) * kMRows + rl) * raw_pitch;
        const uint32_t sh = (uint32_t)(delta_cur[rr] & 3) * 8;
        const uint32_t* wsrc = reinterpret_cast<const uint32_t*>(rraw + (delta_cur[rr] & ~3));
        uint32_t* p = planes + (rl * 3) * plane_pitch;
        if (sh == 0) {
          for (int wq = lane; wq < seg_words; wq += 32) {
            const uint32_t v0 = wsrc[3 * wq], v1 = wsrc[3 * wq + 1], v2 = wsrc[3 * wq + 2];
            p[wq] = __byte_perm(__byte_perm(v0, v1, 0x0630), v2, 0x5210);
            p[plane_pitch + wq] = __byte_perm(__byte_perm(v0, v1, 0x0741), v2, 0x6210);
            p[2 * plane_pitch + wq] = __byte_perm(__byte_perm(v0, v1, 0x0052), v2, 0x7410);
          }
        } else {
          for (int wq = lane; wq < seg_words; wq += 32) {
            const uint32_t x0 = wsrc[3 * wq], x1 = wsrc[3 * wq + 1], x2 = wsrc[3 * wq + 2], x3 = wsrc[3 * wq + 3];
            const uint32_t v0 = __funnelshift_r(x0, x1, sh), v1 = __funnelshift_r(x1, x2, sh), v2 = __funnelshift_r(x2, x3, sh);
            p[wq] = __byte_perm(__byte_perm(v0, v1, 0x0630), v2, 0x5210);
            p[plane_pitch + wq] = __byte_perm(__byte_perm(v0, v1, 0x0741), v2, 0x6210);
            p[2 * plane_pitch + wq] = __byte_perm(__byte_perm(v0, v1, 0x0052), v2, 0x7410);
          }
        }
      }
      delta_cur[0] = delta_next[0]; delta_cur[1] = delta_next[1];
      __syncthreads();
      // ---- compute: warp = two 8-column blocks x 3 channels x 16 rows
#pragma unroll
      for (int sblk = 0; sblk < 2; ++sblk) {
        if (!blk_ok[sblk]) continue;
        const int col = xx0 + 8 * (warp + 8 * sblk) + 2 * t + ((g & 1));          // this lane's output column after the regroup
        const int quad = strip * 4 + (g >> 2) + (g & 2);                         // ... and its row quad (g & 2: rows 8-15)
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          int a0c[4] = {0, 0, 0, 0}, a1c[4] = {0, 0, 0, 0}, a2c[4] = {0, 0, 0, 0};
          const uint32_t* __restrict__ pa = planes + (g * 3 + ch) * plane_pitch + wq0[sblk] + t;
          const uint32_t* __restrict__ pb = pa + 8 * 3 * plane_pitch;
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t x0 = pa[8 * ks], x1 = pb[8 * ks], x2 = pa[8 * ks + 4], x3 = pb[8 * ks + 4];
            imma_uu(a0c, x0, x1, x2, x3, bf[sblk][ks][0][0], bf[sblk][ks][0][1]);
            imma_uu(a1c, x0, x1, x2, x3, bf[sblk][ks][1][0], bf[sblk][ks][1][1]);
            imma_us(a2c, x0, x1, x2, x3, bf[sblk][ks][2][0], bf[sblk][ks][2][1]);
          }
          // bytes of this lane: (row g, col 2t), (row g, col 2t + 1), (row g + 8, col 2t), (row g + 8, col 2t + 1)
          const uint32_t mine = pack4_sat(finish_raw(a0c[0], a1c[0], a2c[0]), finish_raw(a0c[1], a1c[1], a2c[1]),
                                          finish_raw(a0c[2], a1c[2], a2c[2]), finish_raw(a0c[3], a1c[3], a2c[3]));
          // regroup across the four lanes of a row quad (same t, g = 4q .. 4q + 3): lane r = g & 3 collects byte r of each
          const int base_lane = lane & ~12;
          const uint32_t y0 = __shfl_sync(0xffffffffu, mine, base_lane), y1 = __shfl_sync(0xffffffffu, mine, base_lane | 4);
          const uint32_t y2 = __shfl_sync(0xffffffffu, mine, base_lane | 8), y3 = __shfl_sync(0xffffffffu, mine, base_lane | 12);
          const uint32_t r4 = (uint32_t)(g & 3), sel = r4 | ((4u + r4) << 4);
          const uint32_t word = __byte_perm(__byte_perm(y0, y1, sel), __byte_perm(y2, y3, sel), 0x5410);   // rows 4q .. 4q + 3
          if (col < ow && quad < nq) tmp_base[((int64_t)quad * ow + col) * 3 + ch] = word;
        }
      }
    }
    __syncthreads();                // the next item's first copy may land in raw[0] / its planes pass follows a barrier
  }
  zv::ptx::pdl_trigger();
}

// Vertical pass on dp4a + LUT + patchify.  Item = (crop, merge-group row, first pair, pairs): the 28 output rows' limb
// tables are parked in shared memory once per item; a unit is two merge groups (28 rows x 56 pixels) whose row quads of
// the intermediate arrive by 16-byte cp.async (double-buffered), the CTA assembles the two groups' 1176-element patch
// rows in shared memory and streams them out with 16-byte stores, straight at their window-order position.
template <int NW, typename OutT>
__global__ void __launch_bounds__(256) k1_vpass_fast(const K1Crop* __restrict__ crops, const int4* __restrict__ items,
                                                     int n_items, const int32_t* __restrict__ coef,
                                                     const uint8_t* __restrict__ ws, const float* __restrict__ lut,
                                                     OutT* __restrict__ out, int row_order, int wsz, int tile_quads_max) {
  extern __shared__ __align__(16) uint8_t vsm[];
  constexpr int kStride = 1 + 3 * NW;
  uint32_t* tile = reinterpret_cast<uint32_t*>(vsm);                                   // [2][tile_quads_max][168]
  OutT* stage = reinterpret_cast<OutT*>(vsm + (size_t)2 * tile_quads_max * 168 * 4);   // [2][4][1176]
  float* s_lut = reinterpret_cast<float*>(stage + 2 * 4 * kPatchElems);                // [768]
  int32_t* s_coef = reinterpret_cast<int32_t*>(s_lut + 768);                           // [28][kStride]
  zv::ptx::pdl_wait();                // the intermediate is the horizontal pass's output
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = lut[i];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per-lane column decomposition, hoisted out of every loop: stage offset and LUT base of columns lane + 32 i
  int eoff[6], lbase[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int col = lane + 32 * i;
    const int xl = col / 3, ch = col - xl * 3;                           // xl in [0, 56)
    const int grp = xl / 28, xg = xl - grp * 28;
    eoff[i] = (grp * 4 + xg / 14) * kPatchElems + ch * 392 + (xg % 14);
    lbase[i] = ch * 256;
  }

  for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
    const int4 item = __ldg(items + it);
    const K1Crop& c = crops[item.x];
    const int my = item.y, lh = c.lh, lw = c.lw;
    const int qpitch = c.ow * 3;                                         // words per row quad
    const int q_origin = c.ybox0 >> 2;                                   // tmp quads are counted from ybox0 (multiple of 4)
    const int64_t out_row0 = c.out_row0;
    const uint32_t* __restrict__ tmp = reinterpret_cast<const uint32_t*>(ws + c.tmp_off);
    const int32_t* __restrict__ lt = coef + c.off_lv + (int64_t)(my * 28) * kStride;
    __syncthreads();                // previous item: every warp is past its tap loop (s_coef, tile) and its stores (stage)
    for (int i = threadIdx.x; i < 28 * kStride; i += blockDim.x) s_coef[i] = __ldg(lt + i);
    __syncthreads();
    const int q_lo = s_coef[0] - q_origin;                               // window starts are monotone in yy
    const int nq = min(tile_quads_max, s_coef[27 * kStride] + NW - q_origin - q_lo);

    auto issue = [&](const int pair, const int buf) {
      const int mx0 = pair * 2;
      const int chunks = (min(2, lw - mx0) * 84) >> 2;                   // 16-byte chunks per quad row (21 or 42)
      const uint32_t* __restrict__ g = tmp + (int64_t)q_lo * qpitch + mx0 * 84;
      uint32_t* t = tile + buf * tile_quads_max * 168;
      const int ck = threadIdx.x & 63;                                   // 64 threads per quad row, 4 rows per sweep
      if (ck < chunks)
        for (int r = threadIdx.x >> 6; r < nq; r += 4)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(t + r * 168 + ck * 4)),
                       "l"(g + (int64_t)r * qpitch + ck * 4) : "memory");
      asm volatile("cp.async.commit_group;" ::: "memory");
    };

    issue(item.z, 0);
    for (int u = 0; u < item.w; ++u) {
      const int mx0 = (item.z + u) * 2;
      const int ngroups = min(2, lw - mx0);
      const int ncols = ngroups * 84;                                    // (pixel, channel) columns of this unit
      if (u + 1 < item.w) {
        issue(item.z + u + 1, (u + 1) & 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();              // this unit's tile landed; the previous unit's patch rows have left `stage`
      const uint32_t* __restrict__ tl = tile + (u & 1) * tile_quads_max * 168;
      for (int yl = warp; yl < 28; yl += 8) {
        const int32_t* e = s_coef + yl * kStride;
        const int q0 = e[0] - q_origin - q_lo;
        uint32_t l0[NW], l1[NW], l2[NW];
#pragma unroll
        for (int k = 0; k < NW; ++k) { l0[k] = e[1 + k]; l1[k] = e[1 + NW + k]; l2[k] = e[1 + 2 * NW + k]; }
        const uint32_t* __restrict__ base = tl + q0 * 168 + lane;
        const int rowoff = (yl / 14) * 2 * kPatchElems + (yl % 14) * 14;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          if (lane + 32 * i < ncols) {
            int a0 = 0, a1 = 0, a2 = 0;
#pragma unroll
            for (int k = 0; k < NW; ++k) {
              const uint32_t v = base[k * 168 + 32 * i];
              a0 = dp4a_uu(v, l0[k], a0);
              a1 = dp4a_uu(v, l1[k], a1);
              a2 = dp4a_us(v, l2[k], a2);
            }
            const OutT o = to_out<OutT>(s_lut[lbase[i] + finish8(a0, a1, a2)]);
            stage[eoff[i] + rowoff] = o;
            stage[eoff[i] + rowoff + 196] = o;
          }
        }
      }
      __syncthreads();
      constexpr int kVec = 4 * kPatchElems * (int)sizeof(OutT) / 16;
      for (int gi = 0; gi < ngroups; ++gi) {
        const int mx = mx0 + gi;
        const int pos = row_order == ZV_ORDER_WINDOW ? window_pos(my, mx, lh, lw, wsz) : my * lw + mx;
        uint4* dst = reinterpret_cast<uint4*>(out + (out_row0 + 4 * (int64_t)pos) * kPatchElems);
        const uint4* srcv = reinterpret_cast<const uint4*>(stage + gi * 4 * kPatchElems);
        for (int i = threadIdx.x; i < kVec; i += blockDim.x) dst[i] = srcv[i];
      }
    }
  }
  zv::ptx::pdl_trigger();
}

// ------------------------------------------------------------------------------------------------ uint8 output
// zv_resize_u8: the vertical pass writes a plain (oh, ow, 3) uint8 image instead of normalised patches - the device form
// of the reference's resize_image() (PIL.Image.resize(BICUBIC), infer.py:78-85), whose result feeds K1 as a source image.
// Fast layout: item = (crop, first output row, rows <= 8); a warp owns one output row with its limb words in registers
// and sweeps the row's (pixel, channel) columns; the row-quad words of the intermediate are dp4a operands as they lie.
// The output is small next to the source (a 5000 x 5000 image becomes 512 x 512), so no staging is needed.
template <int NW>
__global__ void __launch_bounds__(256) k1_vpass_u8_fast(const K1Crop* __restrict__ crops, const int4* __restrict__ items,
                                                        int n_items, const int32_t* __restrict__ coef,
                                                        const uint8_t* __restrict__ ws) {
  constexpr int kStride = 1 + 3 * NW;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  zv::ptx::pdl_wait();
  for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
    const int4 item = __ldg(items + it);
    if (warp >= item.z) continue;
    const K1Crop& c = crops[item.x];
    const int yy = item.y + warp;
    const int qpitch = c.ow * 3;                                         // words per row quad = bytes per output row
    const uint32_t* __restrict__ tmp = reinterpret_cast<const uint32_t*>(ws + c.tmp_off);
    const int32_t* __restrict__ e = coef + c.off_lv + (int64_t)yy * kStride;
    const int q0 = __ldg(e) - (c.ybox0 >> 2);
    uint32_t l0[NW], l1[NW], l2[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) { l0[k] = __ldg(e + 1 + k); l1[k] = __ldg(e + 1 + NW + k); l2[k] = __ldg(e + 1 + 2 * NW + k); }
    const uint32_t* __restrict__ base = tmp + (int64_t)q0 * qpitch;
    uint8_t* __restrict__ drow = c.dst + (int64_t)yy * c.dst_pitch;
#pragma unroll 2
    for (int col = lane; col < qpitch; col += 32) {
      int a0 = 0, a1 = 0, a2 = 0;
#pragma unroll
      for (int k = 0; k < NW; ++k) {
        const uint32_t v = __ldg(base + (int64_t)k * qpitch + col);
        a0 = dp4a_uu(v, l0[k], a0);
        a1 = dp4a_uu(v, l1[k], a1);
        a2 = dp4a_us(v, l2[k], a2);
      }
      drow[col] = (uint8_t)finish8(a0, a1, a2);
    }
  }
}

// Per-tap form over the plain-row intermediate (more than 45 taps, or unaligned source rows): one thread = one output byte.
__global__ void __launch_bounds__(256) k1_vpass_u8(const K1Crop* __restrict__ crops, const int32_t* __restrict__ ids,
                                                   const int32_t* __restrict__ blk0, int n_cls,
                                                   const int32_t* __restrict__ coef, const uint8_t* __restrict__ ws) {
  zv::ptx::pdl_wait();
  const int slot = find_slot(blk0, n_cls, blockIdx.x);
  const K1Crop c = crops[ids[slot]];
  const int64_t tpitch = (int64_t)c.ow * 3;
  const int64_t item = (int64_t)(blockIdx.x - blk0[slot]) * blockDim.x + threadIdx.x;
  if (item >= (int64_t)c.oh * tpitch) return;
  const int yy = (int)(item / tpitch), col = (int)(item % tpitch);
  const int ymin = coef[c.off_bv + 2 * yy] - c.ybox0, cnt = coef[c.off_bv + 2 * yy + 1];
  const int32_t* __restrict__ k = coef + c.off_kv + (int64_t)yy * c.ksv;
  const uint8_t* __restrict__ p = ws + c.tmp_off + (int64_t)ymin * tpitch + col;
  int acc = 1 << (kPrecisionBits - 1);
  for (int t = 0; t < cnt; ++t) acc += (int)__ldg(p + (int64_t)t * tpitch) * __ldg(k + t);
  c.dst[(int64_t)yy * c.dst_pitch + col] = (uint8_t)clip8(acc >> kPrecisionBits);
}

#include "zv_k1_tc.cuh"

// ------------------------------------------------------------------------------------------------ host side
inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }
inline int nw_class(int ksize) {                   // words per tap window (<= 3 samples of misalignment + ksize taps)
  const int need = (ksize + 3 + 3) / 4;
  for (int c : {2, 3, 4, 5, 7, 10, 12}) if (need <= c) return c;
  return 0;
}

struct AxisTables { int32_t off_bounds = 0, off_kk = 0, off_limbs = 0, ksize = 0, nw = 0, seg_words = 0, tile_quads = 0;
                    int32_t off_mma = 0, ks_mma = 0, pitch_mma = 0;
                    int32_t nkb3 = 0, nkb1 = 0; };      // tensor-core route: 128-byte K blocks per 32-byte chunk, 3 channels / 1 channel
// 32-byte K steps the IMMA horizontal pass needs per 8-column block, from the geometry alone (so that the workspace size
// does not depend on the tables): 8 neighbouring outputs span at most floor(7 scale) + 2 source samples between their first
// taps, + ksize taps, + 3 samples of word alignment.  0 = more than 4 steps (the dp4a kernel handles those).
inline int32_t mma_ksteps(int32_t in_size, int32_t out_size, int32_t ksize) {
  const double scale = (double)in_size / out_size;
  const int32_t span = (int32_t)(7.0 * scale) + 2 + ksize + 3;
  const int32_t ks = (span + 31) / 32;
  return ks <= 4 ? ks : 0;
}
struct Layout {
  int64_t off_desc = 0, off_lut = 0, off_coef = 0, off_lists = 0, off_tmp = 0, bytes = 0;
  int64_t off_tmaps = 0, off_jobs = 0, off_pjobs = 0;     // tensor-core route: 3 tensor maps, 3 RJob and 1 PJob per crop
  std::vector<int64_t> u_off;                // per crop, relative to off_tmp: the finished uint8 image (zv_preprocess only)
  std::vector<int64_t> t_pitch;              // per crop: bytes per row of the transposed intermediate T
  int64_t item_cap_tc = 0;
  std::vector<int64_t> tmp_off;              // per crop, relative to off_tmp
  std::vector<int32_t> ybox0, nrows;
  std::map<std::pair<int32_t, int32_t>, AxisTables> axis;   // (in, out) -> table offsets
  std::vector<int32_t> coef;                 // concatenated int32 tables
  int64_t list_ints = 0;
  // persistent fast kernels: strips per hpass item / pairs per vpass item (chosen from the batch's total work so that
  // small batches still spread over the whole GPU), and the capacity of the two work lists (int4 items)
  int32_t strips_per_item = 1, pairs_per_item = 1;
  int64_t item_cap_h = 0, item_cap_v = 0;
};
constexpr int kItemsTarget = 148 * 8;        // aim for at least this many work items per launch
struct AxisCache { std::vector<int32_t> ints; int32_t seg_words = 0, tile_quads = 0, pitch_mma = 0, nkb3 = 0, nkb1 = 0; };
// K blocks (128 input bytes) the widest 32-output-byte chunk of an axis needs when its samples are `ch` bytes apart
inline int32_t tc_k_blocks(const zv::AxisCoeffs& ac, int32_t n_out, int32_t ch) {
  int32_t span = 0;
  const int32_t n_bytes = n_out * ch;
  for (int32_t b0 = 0; b0 < n_bytes; b0 += kTcCols) {
    const int32_t o0 = b0 / ch, o1 = std::min(n_out - 1, (b0 + kTcCols - 1) / ch);
    int32_t end = 0;
    for (int32_t o = o0; o <= o1; ++o) end = std::max(end, ac.bounds[2 * o] + ac.bounds[2 * o + 1]);
    span = std::max(span, ch * (end - ac.bounds[2 * o0]));
  }
  return (span + 15 + 127) / 128;            // + up to 15 bytes between the 16-byte aligned TMA box start and the window
}
// B variants of an input with this row pitch: distinct values of (q pitch) mod 16 over the four row phases
inline int32_t tc_variants(int64_t pitch) { return (pitch & 15) == 0 ? 1 : (pitch & 7) == 0 ? 2 : 4; }
std::mutex g_axis_mu;
std::map<std::tuple<int32_t, int32_t, int32_t>, std::shared_ptr<const AxisCache>> g_axis_cache;   // (resample kind, in, out)

// Workspace layout shared by zv_preprocess_workspace_bytes and zv_preprocess.
// u8_out: the vertical pass writes plain uint8 images (zv_resize_u8): any positive output size, row-group work items.
// kind (ZV_RESAMPLE_*) selects the taps; the layout itself depends on the geometry alone.
int build_layout(int32_t n, const int32_t* crop_box, const int32_t* resized_hw, Layout* L, bool fill, bool u8_out = false,
                 int32_t kind = ZV_RESAMPLE_PIL) {
  L->tmp_off.resize(n); L->ybox0.resize(n); L->nrows.resize(n); L->u_off.resize(n); L->t_pitch.resize(n);
  int64_t coef_ints = 0, tmp_bytes = 0;
  for (int32_t i = 0; i < n; ++i) {
    const int32_t cw = crop_box[4 * i + 2] - crop_box[4 * i], ch = crop_box[4 * i + 3] - crop_box[4 * i + 1];
    const int32_t oh = resized_hw[2 * i], ow = resized_hw[2 * i + 1];
    if (cw <= 0 || ch <= 0 || oh <= 0 || ow <= 0 || (!u8_out && (oh % 28 || ow % 28)))
      return zv::fail(ZV_EINVAL, "%s: crop %d has extent %dx%d -> %dx%d (need >0%s)", u8_out ? "zv_resize_u8" : "zv_preprocess",
                      i, cw, ch, ow, oh, u8_out ? "" : " and multiples of 28");
    const std::pair<int32_t, int32_t> keys[2] = {{cw, ow}, {ch, oh}};
    for (const auto& key : keys) {
      if (L->axis.count(key)) continue;
      AxisTables t;
      t.ksize = zv::resample_ksize(key.first, key.second);
      t.nw = nw_class(t.ksize);
      t.off_bounds = (int32_t)coef_ints;
      t.off_kk = (int32_t)(coef_ints + 2 * (int64_t)key.second);
      t.off_limbs = (int32_t)(coef_ints + 2 * (int64_t)key.second + (int64_t)key.second * t.ksize);
      t.ks_mma = t.nw > 0 ? mma_ksteps(key.first, key.second, t.ksize) : 0;
      const int64_t n_blk8 = (key.second + 7) / 8;
      t.off_mma = (int32_t)(coef_ints + 2 * (int64_t)key.second + (int64_t)key.second * t.ksize + (int64_t)key.second * (1 + 3 * t.nw));
      const int64_t ints = 2 * (int64_t)key.second + (int64_t)key.second * t.ksize + (int64_t)key.second * (1 + 3 * t.nw) +
                           (t.ks_mma ? n_blk8 * (1 + 192 * t.ks_mma) : 0);
      // the tables of an axis depend on (kind, in, out) alone: built once per process and geometry, then copied - a zoom
      // loop asks for the same few sizes over and over and the fp64 tap generation would otherwise pace every small call
      const std::tuple<int32_t, int32_t, int32_t> ckey{kind, key.first, key.second};
      std::shared_ptr<const AxisCache> hit;
      if (fill) {
        std::lock_guard<std::mutex> lock(g_axis_mu);
        auto itc = g_axis_cache.find(ckey);
        if (itc != g_axis_cache.end()) hit = itc->second;
      }
      if (fill && hit) {
        L->coef.insert(L->coef.end(), hit->ints.begin(), hit->ints.end());
        t.seg_words = hit->seg_words; t.tile_quads = hit->tile_quads; t.pitch_mma = hit->pitch_mma;
        t.nkb3 = hit->nkb3; t.nkb1 = hit->nkb1;
      } else if (fill) {
        const size_t coef_start = L->coef.size();
        zv::AxisCoeffs ac;
        zv::resample_coeffs(kind, key.first, key.second, &ac);
        L->coef.insert(L->coef.end(), ac.bounds.begin(), ac.bounds.end());
        L->coef.insert(L->coef.end(), ac.kk.begin(), ac.kk.end());
        // dp4a limb table: the window starts at the first tap rounded down to 4 samples
        std::vector<int32_t> w0(key.second);
        for (int32_t o = 0; o < key.second; ++o) {
          const int32_t xmin = ac.bounds[2 * o], cnt = ac.bounds[2 * o + 1];
          const int32_t a = xmin & ~3;
          w0[o] = a >> 2;
          L->coef.push_back(a >> 2);
          for (int limb = 0; limb < 3; ++limb)
            for (int w = 0; w < t.nw; ++w) {
              uint32_t word = 0;
              for (int b = 0; b < 4; ++b) {
                const int32_t tap = a + 4 * w + b - xmin;
                const int32_t k = (tap >= 0 && tap < cnt) ? ac.kk[(size_t)o * ac.ksize + tap] : 0;
                const uint32_t byte = limb == 0 ? (uint32_t)(k & 255) : limb == 1 ? (uint32_t)((k >> 8) & 255)
                                                                                  : (uint32_t)((k >> 16) & 255);
                word |= byte << (8 * b);
              }
              L->coef.push_back((int32_t)word);
            }
        }
        // widest source span (in words) any 128-column chunk of this axis needs (horizontal use), and the most row
        // quads any 28-row merge-group row needs (vertical use)
        for (int32_t o0 = 0; o0 < key.second; o0 += kHCols) {
          const int32_t o1 = std::min(key.second, o0 + kHCols) - 1;
          t.seg_words = std::max(t.seg_words, w0[o1] + t.nw - w0[o0]);
        }
        for (int32_t o0 = 0; o0 + 27 < key.second; o0 += 28) t.tile_quads = std::max(t.tile_quads, w0[o0 + 27] + t.nw - w0[o0]);
        if (t.tile_quads == 0) t.tile_quads = 1;            // outputs shorter than 28 (uint8 mode only)
        if (t.ks_mma) {
          // IMMA fragment table: per 8-column block the first word of its source window, then, per (k step, limb, lane),
          // the two B-fragment registers of mma.m16n8k32: b0 = taps k 4t .. 4t + 3, b1 = k 16 + 4t .. of output column g
          const int32_t KS = t.ks_mma;
          std::vector<int32_t> bw0((size_t)n_blk8);
          bool fits = true;
          for (int64_t nb = 0; nb < n_blk8; ++nb) {
            const int32_t o0 = (int32_t)(8 * nb), o1 = std::min<int32_t>(key.second, o0 + 8);
            const int32_t a = ac.bounds[2 * o0] & ~3;
            bw0[nb] = a >> 2;
            for (int32_t o = o0; o < o1; ++o) fits = fits && ac.bounds[2 * o] + ac.bounds[2 * o + 1] - a <= 32 * KS;
          }
          if (!fits) return zv::fail(ZV_EINVAL, "zv_preprocess: internal: IMMA window bound violated for %d -> %d", key.first, key.second);
          for (int64_t nb = 0; nb < n_blk8; ++nb) {
            const int32_t a = bw0[nb] * 4;
            L->coef.push_back(bw0[nb]);
            for (int ks = 0; ks < KS; ++ks)
              for (int limb = 0; limb < 3; ++limb)
                for (int lane = 0; lane < 32; ++lane) {
                  const int32_t o = (int32_t)(8 * nb) + (lane >> 2), tq = lane & 3;
                  for (int half = 0; half < 2; ++half) {
                    uint32_t word = 0;
                    for (int b = 0; b < 4; ++b) {
                      int32_t kv = 0;
                      if (o < key.second) {
                        const int32_t tap = a + 32 * ks + 16 * half + 4 * tq + b - ac.bounds[2 * o];
                        if (tap >= 0 && tap < ac.bounds[2 * o + 1]) kv = ac.kk[(size_t)o * ac.ksize + tap];
                      }
                      const uint32_t byte = limb == 0 ? (uint32_t)(kv & 255) : limb == 1 ? (uint32_t)((kv >> 8) & 255)
                                                                                           : (uint32_t)((kv >> 16) & 255);
                      word |= byte << (8 * b);
                    }
                    L->coef.push_back((int32_t)word);
                  }
                }
          }
          // widest source span (in words) of a 128-column chunk, as the shared-memory plane pitch: = 4 (mod 8) words, so
          // that the A-fragment loads of a warp (8 rows x 4 words, rows 3 pitch apart) hit 32 different banks
          int32_t span = 0;
          for (int64_t nb = 0; nb < n_blk8; nb += kHCols / 8) {
            const int64_t last = std::min<int64_t>(n_blk8, nb + kHCols / 8) - 1;
            span = std::max(span, bw0[last] + 8 * KS - bw0[nb]);
          }
          t.pitch_mma = span + ((4 - span % 8) + 8) % 8;
        }
        t.nkb3 = tc_k_blocks(ac, key.second, 3);
        t.nkb1 = tc_k_blocks(ac, key.second, 1);
        auto entry = std::make_shared<AxisCache>();
        entry->ints.assign(L->coef.begin() + coef_start, L->coef.end());
        entry->seg_words = t.seg_words; entry->tile_quads = t.tile_quads; entry->pitch_mma = t.pitch_mma;
        entry->nkb3 = t.nkb3; entry->nkb1 = t.nkb1;
        std::lock_guard<std::mutex> lock(g_axis_mu);
        if (g_axis_cache.size() >= 512) g_axis_cache.clear();              // bounded: a few hundred KB per entry at most
        g_axis_cache[ckey] = entry;
      }
      L->axis[key] = t;
      coef_ints += ints;
      if (coef_ints > INT32_MAX) return zv::fail(ZV_EINVAL, "zv_preprocess: coefficient tables exceed 2^31 entries");
    }
    // rows of the crop the vertical pass reads: [first tap of row 0, last tap of the last row]
    int32_t y_first, y_last;
    if (ch == oh) { y_first = 0; y_last = ch; }
    else {
      const double scale = (double)ch / oh, fs = scale < 1.0 ? 1.0 : scale, support = 2.0 * fs;
      double c0 = 0 + (0 + 0.5) * scale, c1 = 0 + ((oh - 1) + 0.5) * scale;
      y_first = std::max<int32_t>(0, (int32_t)(c0 - support + 0.5));
      y_last = std::min<int32_t>(ch, (int32_t)(c1 + support + 0.5));
    }
    L->ybox0[i] = y_first;
    L->nrows[i] = y_last - y_first;
    L->tmp_off[i] = tmp_bytes;
    // fast path: 4 rows per word, quads counted from ybox0 rounded down to 4, spare quads for zero-tap window padding
    const int64_t quads = (int64_t)((y_last + 3) / 4 - y_first / 4) + kMaxNW + 1;
    // tensor-core route: T[3 ow rounded up to 4][t_pitch], one byte per (output column byte, crop row from ybox0 & ~3)
    L->t_pitch[i] = align_up(4 * (int64_t)((y_last + 3) / 4 - y_first / 4), 16);
    const int64_t t_bytes = align_up(3 * (int64_t)ow, 4) * L->t_pitch[i];
    tmp_bytes += align_up(std::max<int64_t>(std::max<int64_t>((int64_t)L->nrows[i] * ow * 3, quads * ow * 3 * 4), t_bytes), 256);
    if (!u8_out) {                        // ... and the finished uint8 image the patchify kernel reads
      L->u_off[i] = tmp_bytes;
      tmp_bytes += align_up((int64_t)oh * ow * 3, 256);
    }
    const int64_t tiles1 = ((y_last + 3) / 4 - y_first / 4 + 127) / 128, tiles2 = ((3 * (int64_t)ow + 3) / 4 + 127) / 128;
    L->item_cap_tc += ((3 * (int64_t)ow + kTcCols - 1) / kTcCols) * (tiles1 + 1) + (((int64_t)oh + kTcCols - 1) / kTcCols) * tiles2;   // + 1: the tail tile
  }
  // work-list sizing (geometry only, so that the workspace size does not depend on the tables)
  int64_t units_h = 0, units_v = 0;
  for (int32_t i = 0; i < n; ++i) {
    const int32_t oh = resized_hw[2 * i], ow = resized_hw[2 * i + 1];
    const int64_t rows = L->nrows[i] + (L->ybox0[i] & 3);
    units_h += ((rows + kHRows - 1) / kHRows) * ((ow + kHCols - 1) / kHCols);
    units_v += u8_out ? (oh + 7) / 8 : (int64_t)(oh / 28) * ((ow / 28 + 1) / 2);
  }
  L->strips_per_item = (int32_t)std::min<int64_t>(16, std::max<int64_t>(1, units_h / kItemsTarget));
  L->pairs_per_item = (int32_t)std::min<int64_t>(8, std::max<int64_t>(1, units_v / kItemsTarget));
  for (int32_t i = 0; i < n; ++i) {
    const int32_t oh = resized_hw[2 * i], ow = resized_hw[2 * i + 1];
    const int64_t rows = L->nrows[i] + (L->ybox0[i] & 3);
    const int64_t strips = (rows + kHRows - 1) / kHRows, pairs = (ow / 28 + 1) / 2;
    const int64_t strips16 = (rows + kMRows - 1) / kMRows, per16 = std::max<int64_t>(1, L->strips_per_item / 2);   // IMMA kernel: 16-row strips
    L->item_cap_h += ((ow + kHCols - 1) / kHCols) * std::max((strips + L->strips_per_item - 1) / L->strips_per_item, (strips16 + per16 - 1) / per16);
    L->item_cap_v += u8_out ? (oh + 7) / 8 : (int64_t)(oh / 28) * ((pairs + L->pairs_per_item - 1) / L->pairs_per_item);
  }
  if (L->item_cap_h > INT32_MAX / 8 || L->item_cap_v > INT32_MAX / 8 || L->item_cap_tc > INT32_MAX / 8) return zv::fail(ZV_EINVAL, "zv_preprocess: batch too large for one launch");
  int64_t off = 0;
  L->off_desc = off; off = align_up(off + (int64_t)n * sizeof(K1Crop), 256);
  L->off_lut = off; off = align_up(off + 768 * sizeof(float), 256);
  L->off_coef = off; off = align_up(off + coef_ints * (int64_t)sizeof(int32_t), 256);
  // work lists of the fast kernels (int4 items) first, then, for the per-tap kernels, crop ids + block prefix per pass
  L->list_ints = 4 * (L->item_cap_h + L->item_cap_v + L->item_cap_tc) + 4 * ((int64_t)n + 16);
  L->off_lists = off; off = align_up(off + L->list_ints * (int64_t)sizeof(int32_t), 256);
  L->off_tmaps = off; off = align_up(off + 3 * (int64_t)n * (int64_t)sizeof(CUtensorMap), 256);
  L->off_jobs = off; off = align_up(off + 3 * (int64_t)n * (int64_t)sizeof(RJob), 256);
  L->off_pjobs = off; off = align_up(off + (int64_t)n * (int64_t)sizeof(PJob), 256);
  L->off_tmp = off; off += tmp_bytes;
  L->bytes = off;
  return ZV_OK;
}

// grid of a persistent kernel: every CTA slot of the GPU, or one CTA per item when there are fewer items
template <typename K>
int persistent_grid(K kernel, int smem, int64_t n_items) {
  int per_sm = 1;
  const int sms = zv::num_sms();
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  return (int)std::min<int64_t>(n_items, (int64_t)sms * per_sm);
}
template <int NW>
void launch_hfast(int n_items, cudaStream_t s, const K1Crop* d, const int4* items, const int32_t* coef, uint8_t* ws, int seg_words) {
  const int smem = kHRows * 3 * seg_words * 4 + 2 * kHRows * ((seg_words * 12 + 32 + 15) & ~15);
  static std::atomic<uint64_t> attr{0};
  const int dev = zv::current_device();
  if (zv::device_needs_setup(attr, dev)) { cudaFuncSetAttribute(k1_hpass_fast<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); zv::mark_device(attr, dev); }
  zv::launch_pdl(k1_hpass_fast<NW>, dim3((unsigned)persistent_grid(k1_hpass_fast<NW>, smem, n_items)), dim3(256), smem, s, 1,
                 d, items, n_items, coef, ws, seg_words);
}
template <int KS>
void launch_hmma(int n_items, cudaStream_t s, const K1Crop* d, const int4* items, const int32_t* coef, uint8_t* ws, int plane_pitch) {
  const int smem = kMRows * 3 * plane_pitch * 4 + 2 * kMRows * ((plane_pitch * 12 + 32 + 15) & ~15);
  static std::atomic<uint64_t> attr{0};
  const int dev = zv::current_device();
  if (zv::device_needs_setup(attr, dev)) { cudaFuncSetAttribute(k1_hpass_mma<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024); zv::mark_device(attr, dev); }
  zv::launch_pdl(k1_hpass_mma<KS>, dim3((unsigned)persistent_grid(k1_hpass_mma<KS>, smem, n_items)), dim3(256), smem, s, 1,
                 d, items, n_items, coef, ws, plane_pitch);
}
inline int vfast_smem(int nw, int tile_quads, int out_bytes) {
  return 2 * tile_quads * 168 * 4 + 2 * 4 * kPatchElems * out_bytes + 768 * 4 + 28 * (1 + 3 * nw) * 4;
}
template <int NW, typename OutT>
void launch_vfast(int n_items, cudaStream_t s, const K1Crop* d, const int4* items, const int32_t* coef, const uint8_t* ws,
                  const float* lut, OutT* out, int row_order, int wsz, int tile_quads) {
  const int smem = vfast_smem(NW, tile_quads, (int)sizeof(OutT));
  static std::atomic<uint64_t> attr{0};
  const int dev = zv::current_device();
  if (zv::device_needs_setup(attr, dev)) { cudaFuncSetAttribute(k1_vpass_fast<NW, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); zv::mark_device(attr, dev); }
  zv::launch_pdl(k1_vpass_fast<NW, OutT>, dim3((unsigned)persistent_grid(k1_vpass_fast<NW, OutT>, smem, n_items)), dim3(256), smem, s, 1,
                 d, items, n_items, coef, ws, lut, out, row_order, wsz, tile_quads);
}
template <typename OutT>
void launch_vpass(int nw, int count, cudaStream_t s, const K1Crop* d, const int32_t* list, const int32_t* blk0, int ncls,
                  const int32_t* coef, const uint8_t* ws, const float* lut, void* out_, int row_order, int wsz, int tile_quads) {
  OutT* out = static_cast<OutT*>(out_);
  const int4* items = reinterpret_cast<const int4*>(list);
  switch (nw) {
    case 0: zv::launch_pdl(k1_vpass<OutT>, dim3((unsigned)count), dim3(256), 0, s, 1, d, list, blk0, ncls, coef, ws, lut, out, row_order, wsz); break;
    case 2: launch_vfast<2, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    case 3: launch_vfast<3, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    case 4: launch_vfast<4, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    case 5: launch_vfast<5, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    case 7: launch_vfast<7, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    case 10: launch_vfast<10, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
    default: launch_vfast<12, OutT>(count, s, d, items, coef, ws, lut, out, row_order, wsz, tile_quads); break;
  }
}

// Tensor-core route, pass 1: the image is read through super-rows of four rows counted from row 0, which cover rows
// [0, 4 floor(H / 4)).  A crop that also needs the last H mod 4 rows gets a second job for its last row quads, read
// through a tensor map whose super-rows are counted from row H mod 4 (so that they end with the image).  -> quads of the
// first job, first image row of the second (rows_end when there is none); false when the split is impossible.
inline bool tc_split_rows(int64_t row0, int64_t nrows, int64_t y_hi, int32_t src_h, int64_t* nq_a, int64_t* r_b) {
  const int64_t nq = (nrows + 3) / 4, limit = (int64_t)(src_h / 4) * 4;
  if (y_hi <= limit || row0 >= src_h) { *nq_a = nq; *r_b = row0 + 4 * nq; return true; }   // (rows past the image are zero either way)
  const int64_t k = row0 >= limit ? 0 : (limit - row0) / 4;
  *nq_a = std::min(nq, k);
  *r_b = row0 + 4 * *nq_a;
  return *r_b >= (src_h & 3);
}

// Both device entry points: the two resample passes over n crops.  u8_dst == nullptr: patches (LUT + patchify) into out_dev;
// else plain uint8 images into u8_dst[i] (row pitch u8_pitch[i]).
int k1_run(const char* who, const zv_cfg* cfg, int32_t n, const uint8_t* const* src_dev, const int32_t* src_hw,
           const int64_t* src_pitch, const int32_t* crop_box, const int32_t* resized_hw, const int64_t* row_off,
           void* out_dev, int32_t out_dtype, int32_t row_order, uint8_t* const* u8_dst, const int64_t* u8_pitch,
           void* workspace_dev, int64_t workspace_bytes, void* stream_, int32_t* emulate_tc = nullptr) {
  // emulate_tc != nullptr (zv_debug_k1_tc_host, CPU tests): every pointer is HOST memory; nothing is launched, the
  // tensor-core route's kernels are emulated on the CPU over the very tables built here and emulate_tc[i] tells which
  // crops took that route (the others are left untouched).
  const bool u8_out = u8_dst != nullptr;
  // zv_resize_u8 passes no cfg: it is the reference's Pillow resize_image
  const int32_t kind = cfg ? cfg->resample_kind : ZV_RESAMPLE_PIL;
  int rc = zv::check_resample_kind(kind, who);
  if (rc) return rc;
  int ndev = 0;
  if (!emulate_tc && (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)) return zv::fail(ZV_ENODEV, "%s: no CUDA device", who);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  Layout L;
  rc = build_layout(n, crop_box, resized_hw, &L, true, u8_out, kind);
  if (rc) return rc;
  if (workspace_bytes < L.bytes)
    return zv::fail(ZV_ENOMEM, "%s: workspace %lld B < required %lld B", who, (long long)workspace_bytes, (long long)L.bytes);

  // host image of [descriptors | LUT | coefficient tables | launch lists]
  std::vector<uint8_t> host((size_t)L.off_tmp, 0);
  K1Crop* d = reinterpret_cast<K1Crop*>(host.data() + L.off_desc);
#ifdef ZV_DEBUG_K1_GENERIC              // compile-time debug build: force the per-tap kernels
  const bool generic_only = true;
#else
  const bool generic_only = false;
#endif
  std::vector<int32_t> seg_h(n, 0), tq_v(n, 0), pitch_m(n, 0);
#ifdef ZV_DEBUG_K1_NO_TC                // compile-time debug build: keep every crop on the IMMA / dp4a kernels
  const bool tc_enabled = false;
#else
  const bool tc_enabled = !generic_only;
#endif
  int32_t n_tc = 0;
  int64_t row = 0;
  for (int32_t i = 0; i < n; ++i) {
    K1Crop& c = d[i];
    c.src = src_dev[i]; c.pitch = src_pitch[i];
    c.src_h = src_hw[2 * i]; c.src_w = src_hw[2 * i + 1];
    c.x0 = crop_box[4 * i]; c.y0 = crop_box[4 * i + 1];
    c.cw = crop_box[4 * i + 2] - c.x0; c.ch = crop_box[4 * i + 3] - c.y0;
    c.oh = resized_hw[2 * i]; c.ow = resized_hw[2 * i + 1];
    if (!c.src || c.pitch < 3 * (int64_t)c.src_w) return zv::fail(ZV_EINVAL, "%s: image %d has a null pointer or short pitch", who, i);
    if (u8_out) {
      c.dst = u8_dst[i]; c.dst_pitch = u8_pitch[i];
      if (!c.dst || c.dst_pitch < 3 * (int64_t)c.ow) return zv::fail(ZV_EINVAL, "%s: output %d has a null pointer or short pitch", who, i);
    }
    const AxisTables& h = L.axis[{c.cw, c.ow}];
    const AxisTables& v = L.axis[{c.ch, c.oh}];
    c.ksh = h.ksize; c.ksv = v.ksize;
    c.off_bh = h.off_bounds; c.off_kh = h.off_kk; c.off_bv = v.off_bounds; c.off_kv = v.off_kk;
    c.off_lh = h.off_limbs; c.off_lv = v.off_limbs;
    const bool aligned = (reinterpret_cast<uintptr_t>(c.src) & 3) == 0 && (c.pitch & 3) == 0;
    c.fast = (!generic_only && aligned && h.nw > 0 && v.nw > 0 &&
              kHRows * 3 * h.seg_words * 4 + 2 * kHRows * ((h.seg_words * 12 + 32 + 15) & ~15) <= 200 * 1024 &&
              vfast_smem(v.nw, v.tile_quads, 4) <= 200 * 1024) ? 1 : 0;
    c.nwh = c.fast ? h.nw : 0; c.nwv = c.fast ? v.nw : 0;
    const int mma_smem = kMRows * 3 * h.pitch_mma * 4 + 2 * kMRows * ((h.pitch_mma * 12 + 32 + 15) & ~15);
    c.ks_mma = (c.fast && h.ks_mma > 0 && mma_smem <= 110 * 1024) ? h.ks_mma : 0;
    c.off_mh = h.off_mma;
    pitch_m[i] = h.pitch_mma;
    seg_h[i] = h.seg_words;
    tq_v[i] = v.tile_quads;
    c.ybox0 = L.ybox0[i]; c.nrows = L.nrows[i];
    // Tensor-core route (k1_resample_tc): the row pitch is a
    // multiple of 4 bytes (four image rows = one TMA row with a 16-byte-multiple stride), the rows the pass reads lie in complete
    // groups of four image rows counted from the top or from the bottom (tc_split_rows), and a 32-byte chunk of either axis spans at most kTcMaxNkb K blocks (and its B variants fit 96 KB).  A base
    // that is not 16-byte aligned (a cropped view) is rounded down and the difference added to the byte offset, which
    // works as long as the four-row group still fits its pitch.
    {
      const int64_t delta = (int64_t)(reinterpret_cast<uintptr_t>(c.src) & 15);
      const int64_t y_lo = (int64_t)c.y0 + (c.ybox0 & ~3), y_hi = (int64_t)c.y0 + c.ybox0 + c.nrows;
      // (a box that leaves the image is fine: rows above / below are zero-filled by the TMA unit, taps left / right of the
      // image are left out of B - Image.crop's zero fill)
      bool inside = c.src_h >= 8;
      if (inside && y_hi > (int64_t)(c.src_h / 4) * 4 && y_lo < c.src_h) {   // the last rows come through the end-aligned tensor map (tc_split_rows)
        int64_t nq_a, r_b;
        const int64_t delta_b = (int64_t)((reinterpret_cast<uintptr_t>(c.src) + (uintptr_t)((c.src_h & 3) * c.pitch)) & 15);
        inside = tc_split_rows(y_lo, y_hi - y_lo, y_hi, c.src_h, &nq_a, &r_b) && (delta_b == 0 || 3 * (int64_t)c.src_w + delta_b <= c.pitch);
      }
      c.tc = (tc_enabled && inside && (c.pitch & 3) == 0 && (delta == 0 || 3 * (int64_t)c.src_w + delta <= c.pitch) &&
              4 * c.pitch < (int64_t)1 << 30 && h.nkb3 >= 1 && h.nkb3 <= kTcMaxNkb &&
              h.nkb3 * tc_variants(c.pitch) <= kTcMaxBBlocks && v.nkb1 >= 1 && v.nkb1 <= kTcMaxNkb) ? 1 : 0;
      if (c.tc) { c.fast = 0; c.nwh = -1; c.nwv = -1; c.ks_mma = 0; ++n_tc; }
    }
    if (c.fast || c.tc) {               // row quads are counted from ybox0 rounded down to 4
      const int32_t al = c.ybox0 & ~3;
      c.nrows += c.ybox0 - al; c.ybox0 = al;
    }
    c.tmp_off = L.off_tmp + L.tmp_off[i];
    c.lh = c.oh / 28; c.lw = c.ow / 28;
    c.out_row0 = row_off ? row_off[i] : row;
    row += (int64_t)(c.oh / 14) * (c.ow / 14);
  }
  if (!u8_out) zv::normalize_lut(cfg, reinterpret_cast<float*>(host.data() + L.off_lut));
  std::memcpy(host.data() + L.off_coef, L.coef.data(), L.coef.size() * sizeof(int32_t));

  // launch lists, crops grouped by kernel class.  Fast classes: a work list of int4 items - hpass (crop, 128-column
  // chunk, first strip, strips), ordered strip-major so that the CTAs running together read neighbouring row segments;
  // vpass (crop, merge-group row, first pair, pairs).  Per-tap class (nw 0): crop ids + a block prefix.
  struct Launch { int nw; int64_t list_off, blk_off; int32_t ncls; int64_t count; int seg_words; int tile_quads; };
  std::vector<Launch> hl, vl;
  int32_t* lists = reinterpret_cast<int32_t*>(host.data() + L.off_lists);
  int64_t cur = 0;                                    // in ints; items are appended first, so they stay 16-byte aligned
  // kernel class of a crop's horizontal pass: 100 + KS = IMMA kernel, else the dp4a window class (0 = per-tap kernel)
  auto hclass = [&](const K1Crop& c) { return c.ks_mma ? 100 + c.ks_mma : c.nwh; };
  auto build = [&](bool vpass, std::vector<Launch>* outl) -> int {
    for (int nw : {101, 102, 103, 104, 2, 3, 4, 5, 7, 10, 12}) {
      if (vpass && nw > 100) continue;
      Launch l{};
      l.nw = nw; l.list_off = cur;
      for (int32_t i = 0; i < n; ++i) {
        const K1Crop& c = d[i];
        if ((vpass ? c.nwv : hclass(c)) != nw) continue;
        if (vpass && u8_out) {
          for (int y0 = 0; y0 < c.oh; y0 += 8) {
            lists[cur++] = i; lists[cur++] = y0; lists[cur++] = std::min(8, c.oh - y0); lists[cur++] = 0;
          }
        } else if (vpass) {
          const int pairs = (c.lw + 1) / 2;
          for (int my = 0; my < c.lh; ++my)
            for (int p0 = 0; p0 < pairs; p0 += L.pairs_per_item) {
              lists[cur++] = i; lists[cur++] = my; lists[cur++] = p0; lists[cur++] = std::min(L.pairs_per_item, pairs - p0);
            }
          l.tile_quads = std::max(l.tile_quads, tq_v[i]);
        } else if (nw > 100) {                      // IMMA kernel: 16-row strips
          const int strips = (c.nrows + kMRows - 1) / kMRows, chunks = (c.ow + kHCols - 1) / kHCols;
          const int per = std::max(1, L.strips_per_item / 2);
          for (int s0 = 0; s0 < strips; s0 += per)
            for (int ck = 0; ck < chunks; ++ck) {
              lists[cur++] = i; lists[cur++] = ck; lists[cur++] = s0; lists[cur++] = std::min(per, strips - s0);
            }
          l.seg_words = std::max(l.seg_words, pitch_m[i]);
        } else {
          const int strips = (c.nrows + kHRows - 1) / kHRows, chunks = (c.ow + kHCols - 1) / kHCols;
          for (int s0 = 0; s0 < strips; s0 += L.strips_per_item)
            for (int ck = 0; ck < chunks; ++ck) {
              lists[cur++] = i; lists[cur++] = ck; lists[cur++] = s0; lists[cur++] = std::min(L.strips_per_item, strips - s0);
            }
          l.seg_words = std::max(l.seg_words, seg_h[i]);
        }
      }
      l.count = (cur - l.list_off) / 4;
      if (l.count) outl->push_back(l);
    }
    return ZV_OK;
  };
  auto build_generic = [&](bool vpass, std::vector<Launch>* outl) -> int {
    std::vector<int32_t> ids;
    for (int32_t i = 0; i < n; ++i) if ((vpass ? d[i].nwv : hclass(d[i])) == 0) ids.push_back(i);
    if (ids.empty()) return ZV_OK;
    Launch l{};
    l.nw = 0; l.ncls = (int32_t)ids.size();
    l.list_off = cur;
    for (int32_t id : ids) lists[cur++] = id;
    l.blk_off = cur;
    int64_t blocks = 0;
    for (int32_t id : ids) {
      const K1Crop& c = d[id];
      lists[cur++] = (int32_t)blocks;
      blocks += !vpass ? ((int64_t)c.nrows * c.ow + 255) / 256 : u8_out ? ((int64_t)c.oh * c.ow * 3 + 255) / 256 : (int64_t)c.lh * c.lw;
      if (blocks > INT32_MAX) return zv::fail(ZV_EINVAL, "zv_preprocess: batch too large for one launch");
    }
    l.count = blocks;
    outl->push_back(l);
    return ZV_OK;
  };
  rc = build(false, &hl);
  if (!rc) rc = build(true, &vl);
  // tensor-core route: job descriptors, tensor maps and the two work lists (job, 32-byte chunk, first tile, tiles)
  // pass 1 is launched per B-variant class (1, 2, 4 variants: the shared-memory split depends on it), pass 2 has one
  struct TcLaunch { int64_t list_off = 0, count = 0; int nkb = 1, nvar = 1; } tcl[4];      // [0..2]: pass 1 with 1 / 2 / 4 variants, [3]: pass 2
  auto tc_class = [](int nvar) { return nvar == 1 ? 0 : nvar == 2 ? 1 : 2; };
  int32_t n_pjobs = 0;
  int64_t patch_blocks = 0;
  if (!rc && n_tc) {
    RJob* jobs = reinterpret_cast<RJob*>(host.data() + L.off_jobs);
    PJob* pjobs = reinterpret_cast<PJob*>(host.data() + L.off_pjobs);
    uint8_t* tmaps = host.data() + L.off_tmaps;
    uint8_t* ws_dev = static_cast<uint8_t*>(workspace_dev);
    int64_t tile_units = 0;
    for (int32_t i = 0; i < n && !rc; ++i) {
      const K1Crop& c = d[i];
      if (!c.tc) continue;
      const AxisTables& h = L.axis[{c.cw, c.ow}];
      const AxisTables& v = L.axis[{c.ch, c.oh}];
      const int64_t t_pitch = L.t_pitch[i];
      uint8_t* t_dev = ws_dev + c.tmp_off;
      RJob& j1 = jobs[3 * i];
      const int64_t delta = (int64_t)(reinterpret_cast<uintptr_t>(c.src) & 15);
      j1.x_off = 3 * (int64_t)c.x0 + delta; j1.in_pitch = c.pitch; j1.out = t_dev; j1.out_pitch = t_pitch;
      j1.row0 = c.y0 + c.ybox0; j1.n_rows = c.nrows; j1.n_out = c.ow; j1.ch = 3;
      j1.off_b = c.off_bh; j1.off_k = c.off_kh; j1.ksize = c.ksh; j1.origin = 0; j1.tmap = 3 * i; j1.nkb = h.nkb3;
      j1.in_base = c.src - delta; j1.in_dim0 = 3 * c.pitch + 3 * (int64_t)c.src_w + delta; j1.in_dim1 = c.src_h / 4;
      j1.nvar = tc_variants(c.pitch);
      j1.lo = -c.x0; j1.hi = c.src_w - c.x0;                          // crop columns that exist in the image
      // rows past the image's last multiple-of-4 row: a second job over the end-aligned tensor map (tc_split_rows)
      RJob& j3 = jobs[3 * i + 2];
      int64_t nq_a, r_b;
      tc_split_rows(j1.row0, c.nrows, (int64_t)c.y0 + L.ybox0[i] + L.nrows[i], c.src_h, &nq_a, &r_b);
      j3 = j1;
      j3.n_rows = (int32_t)std::max<int64_t>(0, c.nrows - 4 * nq_a);  // 0: no tail job
      j1.n_rows = (int32_t)std::min<int64_t>(c.nrows, 4 * nq_a);
      if (j3.n_rows > 0) {
        const int32_t sft = c.src_h & 3;
        const uint8_t* base_b = c.src + (int64_t)sft * c.pitch;
        const int64_t delta_b = (int64_t)(reinterpret_cast<uintptr_t>(base_b) & 15);
        j3.x_off = 3 * (int64_t)c.x0 + delta_b; j3.row0 = (int32_t)(r_b - sft); j3.out = t_dev + 4 * nq_a; j3.tmap = 3 * i + 2;
        j3.in_base = base_b - delta_b; j3.in_dim0 = 3 * c.pitch + 3 * (int64_t)c.src_w + delta_b; j3.in_dim1 = (c.src_h - sft) / 4;
      }
      RJob& j2 = jobs[3 * i + 1];
      j2.x_off = 0; j2.in_pitch = t_pitch;
      j2.out = u8_out ? c.dst : ws_dev + L.off_tmp + L.u_off[i];
      j2.out_pitch = u8_out ? c.dst_pitch : 3 * (int64_t)c.ow;
      j2.row0 = 0; j2.n_rows = 3 * c.ow; j2.n_out = c.oh; j2.ch = 1;
      j2.off_b = c.off_bv; j2.off_k = c.off_kv; j2.ksize = c.ksv; j2.origin = c.ybox0; j2.tmap = 3 * i + 1; j2.nkb = v.nkb1;
      j2.in_base = t_dev; j2.in_dim0 = 4 * t_pitch; j2.in_dim1 = (3 * c.ow + 3) / 4;
      j2.nvar = 1;                          // t_pitch is a multiple of 16
      j2.lo = INT32_MIN / 2; j2.hi = INT32_MAX / 2;
      TcLaunch& l1 = tcl[tc_class(j1.nvar)];
      l1.nvar = j1.nvar; l1.nkb = std::max(l1.nkb, h.nkb3); tcl[3].nkb = std::max(tcl[3].nkb, v.nkb1);
      // source: super-rows of four image rows (the last image row's padding is not touched); T likewise
      if (!emulate_tc) {
        CUtensorMap tm;
        rc = zv::make_tmap_u8(&tm, j1.in_base, (uint64_t)j1.in_dim0, (uint64_t)j1.in_dim1, 4 * (uint64_t)j1.in_pitch, 128, 128);
        if (rc) break;
        std::memcpy(tmaps + (size_t)(3 * i) * sizeof(CUtensorMap), &tm, sizeof(tm));
        rc = zv::make_tmap_u8(&tm, j2.in_base, (uint64_t)j2.in_dim0, (uint64_t)j2.in_dim1, 4 * (uint64_t)j2.in_pitch, 128, 128);
        if (rc) break;
        std::memcpy(tmaps + (size_t)(3 * i + 1) * sizeof(CUtensorMap), &tm, sizeof(tm));
        if (j3.n_rows > 0) {
          rc = zv::make_tmap_u8(&tm, j3.in_base, (uint64_t)j3.in_dim0, (uint64_t)j3.in_dim1, 4 * (uint64_t)j3.in_pitch, 128, 128);
          if (rc) break;
          std::memcpy(tmaps + (size_t)(3 * i + 2) * sizeof(CUtensorMap), &tm, sizeof(tm));
        }
      }
      if (!u8_out) {
        PJob& pj = pjobs[n_pjobs++];
        pj.u = j2.out; pj.u_pitch = j2.out_pitch; pj.out_row0 = c.out_row0; pj.lh = c.lh; pj.lw = c.lw;
        pj.blk0 = (int32_t)patch_blocks;
        patch_blocks += (int64_t)c.lh * c.lw;
        if (patch_blocks > INT32_MAX) rc = zv::fail(ZV_EINVAL, "zv_preprocess: batch too large for one launch");
      }
      tile_units += (((int64_t)3 * c.ow + kTcCols - 1) / kTcCols) * (((c.nrows + 3) / 4 + 127) / 128);
    }
    // tiles per item: whole columns when the batch is large (the B operand of a chunk is built once per item),
    // single tiles when it is small (spread over every SM)
    const int per = (int)std::min<int64_t>(16, std::max<int64_t>(1, tile_units / (std::max(1, emulate_tc ? 148 : zv::num_sms()) * 4)));
    for (int cls = 0; cls < 4 && !rc; ++cls) {
      TcLaunch& tl = tcl[cls];
      const int pass = cls == 3;
      tl.list_off = cur;
      for (int32_t i = 0; i < n; ++i) {
        const K1Crop& c = d[i];
        if (!c.tc || (!pass && tc_class(jobs[3 * i].nvar) != cls)) continue;
        const int chunks = pass ? (c.oh + kTcCols - 1) / kTcCols : (3 * c.ow + kTcCols - 1) / kTcCols;
        for (int part = 0; part < (pass ? 1 : 2); ++part) {           // pass 1: the job over the top-aligned map, then the tail job
          const int job = pass ? 3 * i + 1 : 3 * i + 2 * part;
          const int tiles = ((jobs[job].n_rows + 3) / 4 + 127) / 128;
          for (int t0 = 0; t0 < tiles; t0 += per)
            for (int ck = 0; ck < chunks; ++ck) {
              lists[cur++] = job; lists[cur++] = ck; lists[cur++] = t0; lists[cur++] = std::min(per, tiles - t0);
            }
        }
      }
      tl.count = (cur - tl.list_off) / 4;
    }
  }
  if (!rc) rc = build_generic(false, &hl);
  if (!rc) rc = build_generic(true, &vl);
  if (rc) return rc;
  if (cur > L.list_ints) return zv::fail(ZV_EINVAL, "zv_preprocess: launch lists overflow");

  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  if (emulate_tc) {
    std::memcpy(ws, host.data(), host.size());
    for (int32_t i = 0; i < n; ++i) emulate_tc[i] = d[i].tc;
    if (!n_tc) return ZV_OK;
    const RJob* jobs = reinterpret_cast<const RJob*>(ws + L.off_jobs);
    const int32_t* coef = reinterpret_cast<const int32_t*>(ws + L.off_coef);
    const int4* items = reinterpret_cast<const int4*>(reinterpret_cast<const int32_t*>(ws + L.off_lists));
    for (const TcLaunch& tl : tcl)
      if (tl.count) tc_emulate_resample(jobs, items + tl.list_off / 4, (int)tl.count, coef);
    if (!u8_out) {
      if (out_dtype != ZV_F32) return zv::fail(ZV_EINVAL, "%s: the host emulation writes fp32 patches only", who);
      tc_emulate_patchify<float>(reinterpret_cast<const PJob*>(ws + L.off_pjobs), n_pjobs, reinterpret_cast<const float*>(ws + L.off_lut),
                                 static_cast<float*>(out_dev), row_order, cfg->window / cfg->merge / cfg->patch, &window_pos);
    }
    return ZV_OK;
  }
  cudaError_t e = cudaMemcpyAsync(ws, host.data(), host.size(), cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return zv::fail(ZV_ECUDA, "%s: table upload: %s", who, cudaGetErrorString(e));
  const K1Crop* dcrops = reinterpret_cast<const K1Crop*>(ws + L.off_desc);
  const int32_t* dcoef = reinterpret_cast<const int32_t*>(ws + L.off_coef);
  const int32_t* dlists = reinterpret_cast<const int32_t*>(ws + L.off_lists);
  const float* dlut = reinterpret_cast<const float*>(ws + L.off_lut);
  const int wsz = u8_out ? 0 : cfg->window / cfg->merge / cfg->patch;
  {
    zv::KernelTimer timer(zv::KC_K1_HPASS, stream);
    for (const Launch& l : hl) {
      const int32_t* list = dlists + l.list_off;
      const int4* items = reinterpret_cast<const int4*>(list);
      const int ni = (int)l.count;
      switch (l.nw) {
        case 0: zv::launch_pdl(k1_hpass, dim3((unsigned)l.count), dim3(256), 0, stream, 1, dcrops, list, dlists + l.blk_off, l.ncls, dcoef, ws); break;
        case 101: launch_hmma<1>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 102: launch_hmma<2>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 103: launch_hmma<3>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 104: launch_hmma<4>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 2: launch_hfast<2>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 3: launch_hfast<3>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 4: launch_hfast<4>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 5: launch_hfast<5>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 7: launch_hfast<7>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        case 10: launch_hfast<10>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
        default: launch_hfast<12>(ni, stream, dcrops, items, dcoef, ws, l.seg_words); break;
      }
      zv::count_launch();
    }
  }
  {
    zv::KernelTimer timer(zv::KC_K1_VPASS, stream);
    for (const Launch& l : vl) {
      const int32_t* list = dlists + l.list_off;
      const int32_t* blk0 = dlists + l.blk_off;
      const int cnt = (int)l.count;
      if (u8_out) {
        const int4* items = reinterpret_cast<const int4*>(list);
        const int grid = (int)std::min<int64_t>(cnt, (int64_t)zv::num_sms() * 8);
        switch (l.nw) {
          case 0: zv::launch_pdl(k1_vpass_u8, dim3((unsigned)cnt), dim3(256), 0, stream, 1, dcrops, list, blk0, l.ncls, dcoef, (const uint8_t*)ws); break;
          case 2: zv::launch_pdl(k1_vpass_u8_fast<2>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          case 3: zv::launch_pdl(k1_vpass_u8_fast<3>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          case 4: zv::launch_pdl(k1_vpass_u8_fast<4>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          case 5: zv::launch_pdl(k1_vpass_u8_fast<5>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          case 7: zv::launch_pdl(k1_vpass_u8_fast<7>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          case 10: zv::launch_pdl(k1_vpass_u8_fast<10>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
          default: zv::launch_pdl(k1_vpass_u8_fast<12>, dim3((unsigned)grid), dim3(256), 0, stream, 1, dcrops, items, cnt, dcoef, (const uint8_t*)ws); break;
        }
      } else if (out_dtype == ZV_BF16) launch_vpass<__nv_bfloat16>(l.nw, cnt, stream, dcrops, list, blk0, l.ncls, dcoef, ws, dlut, out_dev, row_order, wsz, l.tile_quads);
      else if (out_dtype == ZV_F16) launch_vpass<__half>(l.nw, cnt, stream, dcrops, list, blk0, l.ncls, dcoef, ws, dlut, out_dev, row_order, wsz, l.tile_quads);
      else launch_vpass<float>(l.nw, cnt, stream, dcrops, list, blk0, l.ncls, dcoef, ws, dlut, out_dev, row_order, wsz, l.tile_quads);
      zv::count_launch();
    }
  }
  if (n_tc) {
    const RJob* djobs = reinterpret_cast<const RJob*>(ws + L.off_jobs);
    const CUtensorMap* dtmaps = reinterpret_cast<const CUtensorMap*>(ws + L.off_tmaps);
    static std::atomic<uint64_t> attr{0};
    const int dev = zv::current_device();
    if (zv::device_needs_setup(attr, dev)) {
      cudaFuncSetAttribute(k1_resample_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      zv::mark_device(attr, dev);
    }
    auto launch_tc = [&](const TcLaunch& tl) {
      if (!tl.count) return;
      const int nbuf = tc_b_buffers(tl.nvar, tl.nkb), b_blocks = nbuf * tl.nvar * tl.nkb;
      const int stages = tc_stages(b_blocks);
      const int grid = (int)std::min<int64_t>(tl.count, zv::num_sms());
      zv::launch_pdl(k1_resample_tc, dim3((unsigned)grid), dim3(kTcThreads), (size_t)tc_smem_bytes(stages, b_blocks), stream, 1,
                     djobs, reinterpret_cast<const int4*>(dlists + tl.list_off), (int)tl.count, dcoef, dtmaps, stages, tl.nkb,
                     tl.nvar, nbuf);
      zv::count_launch();
    };
    {
      zv::KernelTimer timer(zv::KC_K1_HPASS, stream);
      for (int cls = 0; cls < 3; ++cls) launch_tc(tcl[cls]);
    }
    {
      zv::KernelTimer timer(zv::KC_K1_VPASS, stream);
      launch_tc(tcl[3]);
      if (!u8_out) {
        const PJob* dpj = reinterpret_cast<const PJob*>(ws + L.off_pjobs);
        const int groups = (int)patch_blocks;
        const unsigned blocks = (unsigned)std::min<int64_t>(patch_blocks, (int64_t)zv::num_sms() * 8);
        if (out_dtype == ZV_BF16) zv::launch_pdl(k1_patchify_u8<__nv_bfloat16>, dim3(blocks), dim3(256), 0, stream, 1, dpj, (int)n_pjobs, groups, dlut, static_cast<__nv_bfloat16*>(out_dev), (int)row_order, wsz);
        else if (out_dtype == ZV_F16) zv::launch_pdl(k1_patchify_u8<__half>, dim3(blocks), dim3(256), 0, stream, 1, dpj, (int)n_pjobs, groups, dlut, static_cast<__half*>(out_dev), (int)row_order, wsz);
        else zv::launch_pdl(k1_patchify_u8<float>, dim3(blocks), dim3(256), 0, stream, 1, dpj, (int)n_pjobs, groups, dlut, static_cast<float*>(out_dev), (int)row_order, wsz);
        zv::count_launch();
      }
    }
  }
  e = cudaGetLastError();
  if (e != cudaSuccess) return zv::fail(ZV_ECUDA, "%s: launch: %s", who, cudaGetErrorString(e));
  return ZV_OK;
}

}  // namespace

extern "C" {

int64_t zv_preprocess_workspace_bytes(int32_t n, const int32_t* crop_box, const int32_t* resized_hw) {
  if (n <= 0 || !crop_box || !resized_hw) return zv::fail(ZV_EINVAL, "zv_preprocess_workspace_bytes: bad argument");
  Layout L;
  int rc = build_layout(n, crop_box, resized_hw, &L, false);
  return rc ? rc : L.bytes;
}

int zv_preprocess(const zv_cfg* cfg, int32_t n, const uint8_t* const* src_dev, const int32_t* src_hw,
                  const int64_t* src_pitch, const int32_t* crop_box, const int32_t* resized_hw,
                  const int64_t* row_off, void* out_dev, int32_t out_dtype, int32_t row_order, void* workspace_dev,
                  int64_t workspace_bytes, void* stream_) {
  zv::reset_launch_count();
  zv::NvtxRange nvtx_k1("zv:K1 crop+resize+normalize+patchify");
  if (!cfg || n <= 0 || !src_dev || !src_hw || !src_pitch || !crop_box || !resized_hw || !out_dev || !workspace_dev)
    return zv::fail(ZV_EINVAL, "zv_preprocess: null argument");
  if (cfg->patch != 14 || cfg->merge != 2 || cfg->temporal != 2)
    return zv::fail(ZV_EINVAL, "zv_preprocess: only patch=14, merge=2, temporal=2 is built");
  if (out_dtype != ZV_F32 && out_dtype != ZV_BF16 && out_dtype != ZV_F16) return zv::fail(ZV_EINVAL, "zv_preprocess: bad out_dtype");
  if (row_order != ZV_ORDER_HF && row_order != ZV_ORDER_WINDOW) return zv::fail(ZV_EINVAL, "zv_preprocess: bad row_order");
  return k1_run("zv_preprocess", cfg, n, src_dev, src_hw, src_pitch, crop_box, resized_hw, row_off, out_dev, out_dtype, row_order,
                nullptr, nullptr, workspace_dev, workspace_bytes, stream_);
}

int zv_debug_k1_tc_host(const zv_cfg* cfg, int32_t n, const uint8_t* const* src_host, const int32_t* src_hw,
                        const int64_t* src_pitch, const int32_t* crop_box, const int32_t* resized_hw, float* out_host,
                        int32_t row_order, uint8_t* const* u8_dst_host, const int64_t* u8_pitch, void* workspace_host,
                        int64_t workspace_bytes, int32_t* took_tc) {
  if (n <= 0 || !src_host || !src_hw || !src_pitch || !crop_box || !resized_hw || !workspace_host || !took_tc)
    return zv::fail(ZV_EINVAL, "zv_debug_k1_tc_host: null argument");
  if (!u8_dst_host && (!cfg || !out_host)) return zv::fail(ZV_EINVAL, "zv_debug_k1_tc_host: patch mode needs cfg and out_host");
  return k1_run("zv_debug_k1_tc_host", cfg, n, src_host, src_hw, src_pitch, crop_box, resized_hw, nullptr, out_host, ZV_F32, row_order,
                u8_dst_host, u8_pitch, workspace_host, workspace_bytes, nullptr, took_tc);
}

int64_t zv_resize_u8_workspace_bytes(int32_t n, const int32_t* crop_box, const int32_t* out_hw) {
  if (n <= 0 || !crop_box || !out_hw) return zv::fail(ZV_EINVAL, "zv_resize_u8_workspace_bytes: bad argument");
  Layout L;
  int rc = build_layout(n, crop_box, out_hw, &L, false, true);
  return rc ? rc : L.bytes;
}

int zv_resize_u8(int32_t n, const uint8_t* const* src_dev, const int32_t* src_hw, const int64_t* src_pitch,
                 const int32_t* crop_box, const int32_t* out_hw, uint8_t* const* dst_dev, const int64_t* dst_pitch,
                 void* workspace_dev, int64_t workspace_bytes, void* stream_) {
  zv::reset_launch_count();
  zv::NvtxRange nvtx_k1("zv:K1 crop+resize (uint8)");
  if (n <= 0 || !src_dev || !src_hw || !src_pitch || !crop_box || !out_hw || !dst_dev || !dst_pitch || !workspace_dev)
    return zv::fail(ZV_EINVAL, "zv_resize_u8: null argument");
  return k1_run("zv_resize_u8", nullptr, n, src_dev, src_hw, src_pitch, crop_box, out_hw, nullptr, nullptr, 0, 0, dst_dev, dst_pitch,
                workspace_dev, workspace_bytes, stream_);
}

}  // extern "C"
