// Tower assembly: weight packing, plan upload, and the forward pass of the Qwen2.5-VL vision tower
// (HF modeling_qwen2_5_vl.py:455-518) as a fixed sequence of libzoomvit kernels on the caller's stream.
//
// Precision policy (SURVEY 0.3): residual stream X stays fp32; RMSNorm, rotary, softmax and every
// accumulation are fp32; only GEMM / attention operands are rounded to bf16.
//
// Per block (HF :290-321), with both RMSNorms folded into the GEMMs around them - rmsnorm(x) W^T =
// (x (W diag(g))^T) / rms(x): the gain g is multiplied into the weight columns at pack time, the residual GEMM that
// produces x also emits x as 16-bit operands (X16) and per-row partial sums of squares (SS), and the consumer GEMM
// scales its accumulator rows by 1/rms in the epilogue.  No separate norm pass reads X back from HBM.
//                            QKV = rope((X16 Wqkv'^T) / rms + b)      zv_gemm.cu   EPI_QKV_ROPE
//                            A = attention(QKV)                       zv_attn_win_tc.cu / zv_attn_tc.cu
//                            X += A Wo^T + b ; X16, SS                zv_gemm.cu   EPI_RESID
//                            H = silu((X16 Wg'^T)/rms+b)*((X16 Wu'^T)/rms+b)       EPI_SWIGLU (gate/up rows interleaved)
//                            X += H Wd^T + b ; X16, SS                             EPI_RESID
// Merger (HF :133-146):      Z = rmsnorm(X) viewed (T, 4H); G = gelu(Z W1^T + b); out[widx[i]] = G W2^T + b.
//
// Qwen2-VL tower (cfg->tower_kind = ZV_TOWER_QWEN2, HF models/qwen2_vl/modeling_qwen2_vl.py): LayerNorm with gain g and
// bias beta, folded the same way - LN(x) W^T + b = r (x W'^T) - r mu c + b' with W' = W diag(g) (16-bit), c_n = sum_k W'[n][k]
// of those rounded weights, b' = b + W beta (fp32, from the fp32 source weights), r = rsqrt(var + eps).  The producers emit
// per-64-column-slot (mean, M2) (LNS) instead of sums of squares; every block is full attention:
//                            QKV = rope(r (X16 Wqkv'^T - mu c) + b')   EPI_QKV_ROPE_LN
//                            A = attention(QKV)                        zv_attn_tc.cu
//                            X += A Wo^T + b ; X16, LNS                EPI_RESID_LN
//                            H = quick_gelu(r (X16 W1'^T - mu c) + b') EPI_QGELU   (S, 5120) 16-bit
//                            X += H W2^T + b ; X16, LNS                EPI_RESID_LN
// Merger:                    Z = layernorm(X) viewed (T, 4H); then as above.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "zv_common.h"
#include "zv_gemm.h"
#include "zv_ptx.cuh"

namespace zv {
namespace {

constexpr int kPatchK = 1176;

__device__ __forceinline__ uint32_t pack2(float a, float b, bool f16) {
  if (f16) { __half2 v = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }
inline int ipad(const zv_cfg* c) { return (c->inter + 127) / 128 * 128; }

// ------------------------------------------------------------------------------------------------ small kernels
// One warp per row.  y = w * (x * rsqrt(mean(x^2) + eps)), fp32 math, bf16 out.
__global__ void __launch_bounds__(256) rmsnorm_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                      uint16_t* __restrict__ y, bool f16, int64_t rows, int hidden, float eps) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * hidden);
  const int nv = hidden / 4;
  float4 v[10];                      // hidden <= 1280
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      v[i] = xr[idx];
      ss += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float r = rsqrtf(ss / (float)hidden + eps);
  const float4* wr = reinterpret_cast<const float4*>(w);
  uint2* yr = reinterpret_cast<uint2*>(y + row * hidden);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      const float4 g = __ldg(wr + idx);
      yr[idx] = make_uint2(pack2(g.x * (v[i].x * r), g.y * (v[i].y * r), f16), pack2(g.z * (v[i].z * r), g.w * (v[i].w * r), f16));
    }
  }
}

// One warp per row: 16-bit copy of the row + its sum of squares (producer side of the folded RMSNorm for the patch-embed
// output, which no residual GEMM has touched yet).
__global__ void __launch_bounds__(256) cast_rows_ss_kernel(const float* __restrict__ x, uint16_t* __restrict__ y, bool f16,
                                                           float* __restrict__ ss, int64_t rows, int hidden) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * hidden);
  uint2* yr = reinterpret_cast<uint2*>(y + row * hidden);
  const int nv = hidden / 4;
  float s = 0.f;
  for (int idx = lane; idx < nv; idx += 32) {
    const float4 v = xr[idx];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    yr[idx] = make_uint2(pack2(v.x, v.y, f16), pack2(v.z, v.w, f16));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane < kSsParts) ss[row * kSsParts + lane] = lane == 0 ? s : 0.f;
}

// One warp per row: 16-bit copy of the row + per 64-column slot its (mean, M2), two-pass (producer side of the folded
// LayerNorm for the patch-embed output).  Lanes 0-15 hold slot 2j, lanes 16-31 slot 2j+1 of the j-th 128 columns.
__global__ void __launch_bounds__(256) cast_rows_ln_kernel(const float* __restrict__ x, uint16_t* __restrict__ y, bool f16,
                                                           float2* __restrict__ ln, int64_t rows, int hidden) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * hidden);
  uint2* yr = reinterpret_cast<uint2*>(y + row * hidden);
  for (int j = 0; j < hidden / 128; ++j) {
    const int idx = 32 * j + lane;
    const float4 v = xr[idx];
    yr[idx] = make_uint2(pack2(v.x, v.y, f16), pack2(v.z, v.w, f16));
    float s = (v.x + v.y) + (v.z + v.w);
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.f / 64.f);
    const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
    float m2 = (dx * dx + dy * dy) + (dz * dz + dw * dw);
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
    if ((lane & 15) == 0) ln[row * kSsParts + 2 * j + (lane >> 4)] = make_float2(mean, m2);
  }
}

// One warp per row.  y = (x - mean) * rsqrt(var + eps) * w + b (torch.nn.LayerNorm), two-pass fp32 statistics, 16-bit out.
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ b, uint16_t* __restrict__ y, bool f16,
                                                        int64_t rows, int hidden, float eps) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * hidden);
  const int nv = hidden / 4;
  float4 v[10];                      // hidden <= 1280
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) { v[i] = xr[idx]; s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)hidden;
  float m2 = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
      m2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
  const float r = rsqrtf(m2 / (float)hidden + eps);
  const float4* wr = reinterpret_cast<const float4*>(w);
  const float4* br = reinterpret_cast<const float4*>(b);
  uint2* yr = reinterpret_cast<uint2*>(y + row * hidden);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      const float4 g = __ldg(wr + idx), c = __ldg(br + idx);
      yr[idx] = make_uint2(pack2(fmaf((v[i].x - mean) * r, g.x, c.x), fmaf((v[i].y - mean) * r, g.y, c.y), f16),
                           pack2(fmaf((v[i].z - mean) * r, g.z, c.z), fmaf((v[i].w - mean) * r, g.w, c.w), f16));
    }
  }
}

// Folded LayerNorm, weight side.  One warp per output row n of a consumer GEMM: bias[n] += sum_k W[n][k] beta[k] (fp32 from
// the source weights W) and csum[n] = sum_k W'[n][k] of the packed 16-bit weights (the numbers the MMA multiplies).
template <typename SrcT, typename PkT>
__global__ void __launch_bounds__(256) ln_fold_kernel(const SrcT* __restrict__ w, const PkT* __restrict__ wp,
                                                      const float* __restrict__ beta, float* __restrict__ bias,
                                                      float* __restrict__ csum, int64_t rows, int64_t cols) {
  const int64_t n = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (n >= rows) return;
  const int lane = threadIdx.x & 31;
  float wb = 0.f, cs = 0.f;
  for (int64_t k = lane; k < cols; k += 32) {
    float v;
    if constexpr (std::is_same<SrcT, float>::value) v = w[n * cols + k];
    else if constexpr (std::is_same<SrcT, __half>::value) v = __half2float(w[n * cols + k]);
    else v = __bfloat162float(w[n * cols + k]);
    wb = fmaf(v, beta[k], wb);
    if constexpr (std::is_same<PkT, __half>::value) cs += __half2float(wp[n * cols + k]);
    else cs += __bfloat162float(wp[n * cols + k]);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) { wb += __shfl_xor_sync(0xffffffffu, wb, o); cs += __shfl_xor_sync(0xffffffffu, cs, o); }
  if (lane == 0) { bias[n] += wb; csum[n] = cs; }
}

// dst group i (unit rows x cols, 16-bit operand type) <- src group widx[i] (f32, or already the operand type).
template <typename SrcT>
__global__ void __launch_bounds__(256) gather_kernel(const SrcT* __restrict__ src, uint16_t* __restrict__ dst, bool f16,
                                                     const int32_t* __restrict__ widx, int group_elems) {
  const int64_t gi = blockIdx.x;
  ptx::pdl_wait();
  const SrcT* s = src + (int64_t)widx[gi] * group_elems;
  uint16_t* d = dst + gi * group_elems;
  for (int i = threadIdx.x * 4; i < group_elems; i += blockDim.x * 4) {
    float f[4];
    if constexpr (sizeof(SrcT) == 4) {
      const float4 t = *reinterpret_cast<const float4*>(s + i);
      f[0] = t.x; f[1] = t.y; f[2] = t.z; f[3] = t.w;
      *reinterpret_cast<uint2*>(d + i) = make_uint2(pack2(f[0], f[1], f16), pack2(f[2], f[3], f16));
    } else {
      *reinterpret_cast<uint2*>(d + i) = *reinterpret_cast<const uint2*>(s + i);
    }
  }
}

// LM hand-off: comp[i] = dest[widx[i]] - the inputs_embeds row of the embedding the merger computes at window
// position i (widx: window position -> HF merge-group index; dest: HF embedding index -> placeholder row).
// A destination outside [0, rows) becomes -1: the scatter epilogue drops that row instead of storing out of bounds.
__global__ void __launch_bounds__(256) compose_rows_kernel(const int64_t* __restrict__ dest, const int32_t* __restrict__ widx,
                                                           int32_t* __restrict__ comp, int64_t n, int64_t rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  ptx::pdl_wait();
  if (i < n) {
    const int64_t d = dest[widx[i]];
    comp[i] = (d >= 0 && d < rows) ? (int32_t)d : -1;
  }
}

// Weight import: dst[row_map(r)][c] = src[r][c] (to bf16 or f32).  mode 0 identity, 1 gate, 2 up
// (gate/up rows interleaved in blocks of 128 so one 256-wide GEMM tile holds both halves of 128 outputs).
// `colscale` (fp32 [cols], may be null): the RMSNorm gain folded into the weight columns.
template <typename SrcT, typename DstT>
__global__ void pack_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t rows, int64_t cols,
                            int64_t dst_ld, int mode, const float* __restrict__ colscale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int64_t r = i / cols, c = i % cols;
  int64_t dr = r;
  if (mode == 1) dr = (r / 128) * 256 + r % 128;
  if (mode == 2) dr = (r / 128) * 256 + 128 + r % 128;
  float v;
  if constexpr (std::is_same<SrcT, float>::value) v = src[i];
  else if constexpr (std::is_same<SrcT, __half>::value) v = __half2float(src[i]);
  else v = __bfloat162float(src[i]);
  if (colscale) v *= colscale[c];
  if constexpr (std::is_same<DstT, float>::value) dst[dr * dst_ld + c] = v;
  else if constexpr (std::is_same<DstT, __half>::value) dst[dr * dst_ld + c] = __float2half_rn(v);
  else dst[dr * dst_ld + c] = __float2bfloat16_rn(v);
}

// ------------------------------------------------------------------------------------------------ weight layout
// Qwen2-VL (kind 1): wgu / bgu hold fc1 (inter x H) and its folded bias, wd / bd fc2; n1b / n2b / ln_qb the LayerNorm biases,
// cqkv / cfc1 the column sums c of the folded weights.
struct LayerOff { int64_t n1, n2, wqkv, bqkv, wo, bo, wgu, bgu, wd, bd, n1b, n2b, cqkv, cfc1; };
struct WeightLayout {
  int64_t wpe = 0;
  std::vector<LayerOff> layers;
  int64_t ln_q = 0, w1 = 0, b1 = 0, w2 = 0, b2 = 0, ln_qb = 0, bytes = 0;
};
bool qwen2(const zv_cfg* c) { return c->tower_kind == ZV_TOWER_QWEN2; }

WeightLayout weight_layout(const zv_cfg* c) {
  WeightLayout L;
  const int64_t H = c->hidden, I = ipad(c), O = c->out_hidden;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { int64_t o = off; off = align_up(off + bytes, 256); return o; };
  L.wpe = take(H * kPatchK * 2);
  L.layers.resize(c->depth);
  if (qwen2(c)) {
    for (auto& l : L.layers) {
      l.n1 = take(H * 4); l.n1b = take(H * 4); l.n2 = take(H * 4); l.n2b = take(H * 4);
      l.wqkv = take(3 * H * H * 2); l.bqkv = take(3 * H * 4); l.cqkv = take(3 * H * 4);
      l.wo = take(H * H * 2); l.bo = take(H * 4);
      l.wgu = take(I * H * 2); l.bgu = take(I * 4); l.cfc1 = take(I * 4);
      l.wd = take(H * I * 2); l.bd = take(H * 4);
    }
    L.ln_q = take(H * 4); L.ln_qb = take(H * 4);
    L.w1 = take(16 * H * H * 2); L.b1 = take(4 * H * 4);
    L.w2 = take(O * 4 * H * 2); L.b2 = take(O * 4);
    L.bytes = off;
    return L;
  }
  for (auto& l : L.layers) {
    l.n1 = take(H * 4); l.n2 = take(H * 4);
    l.wqkv = take(3 * H * H * 2); l.bqkv = take(3 * H * 4);
    l.wo = take(H * H * 2); l.bo = take(H * 4);
    l.wgu = take(2 * I * H * 2); l.bgu = take(2 * I * 4);
    l.wd = take(H * I * 2); l.bd = take(H * 4);
  }
  L.ln_q = take(H * 4);
  L.w1 = take(16 * H * H * 2); L.b1 = take(4 * H * 4);
  L.w2 = take(O * 4 * H * 2); L.b2 = take(O * 4);
  L.bytes = off;
  return L;
}

int check_cfg(const zv_cfg* c, const char* who) {
  if (!c) return fail(ZV_EINVAL, "%s: null cfg", who);
  if (c->hidden != 1280 || c->heads != 16 || c->out_hidden % 256 || c->patch != 14 || c->merge != 2 || c->temporal != 2 ||
      c->depth < 1 || c->depth > 32 || c->inter <= 0)
    return fail(ZV_EINVAL, "%s: this build covers hidden=1280, heads=16 (head_dim 80), patch=14, merge=2, temporal=2, depth<=32", who);
  if (c->tower_kind != ZV_TOWER_QWEN25 && c->tower_kind != ZV_TOWER_QWEN2)
    return fail(ZV_EINVAL, "%s: tower_kind=%d (0 Qwen2.5-VL, 1 Qwen2-VL)", who, c->tower_kind);
  if (qwen2(c)) {
    const uint32_t all = c->depth == 32 ? 0xffffffffu : (1u << c->depth) - 1u;
    if (((uint32_t)c->fullatt_mask_lo & all) != all)
      return fail(ZV_EINVAL, "%s: tower_kind=1 (Qwen2-VL) has full attention in every block, but fullatt_mask_lo=0x%08x "
                  "leaves window blocks among the %d", who, (uint32_t)c->fullatt_mask_lo, c->depth);
    if (c->inter != 5120)
      return fail(ZV_EINVAL, "%s: tower_kind=1 (Qwen2-VL) needs inter=5120 (fc1 1280 -> 5120), got inter=%d", who, c->inter);
  }
  return ZV_OK;
}

int check_device(const char* who) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(ZV_ENODEV, "%s: no CUDA device", who);
  int dev = 0, major = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail(ZV_EARCH, "%s: device compute capability %d.x is not sm_100 (no fallback path exists)", who, major);
  return ZV_OK;
}

template <typename DstT>
int pack_one(const zv_tensor* t, DstT* dst, int64_t rows, int64_t cols, int64_t dst_ld, int mode, cudaStream_t s,
             const float* colscale = nullptr) {
  int64_t numel = 1;
  for (int i = 0; i < t->ndim; ++i) numel *= t->shape[i];
  if (numel != rows * cols)
    return fail(ZV_EINVAL, "zv_weights_pack: %s has %lld elements, expected %lld x %lld", t->name, (long long)numel,
                (long long)rows, (long long)cols);
  const unsigned blocks = (unsigned)((numel + 255) / 256);
  if (t->dtype == ZV_F32)
    pack_kernel<float, DstT><<<blocks, 256, 0, s>>>(static_cast<const float*>(t->data), dst, rows, cols, dst_ld, mode, colscale);
  else if (t->dtype == ZV_BF16)
    pack_kernel<__nv_bfloat16, DstT><<<blocks, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(t->data), dst, rows, cols, dst_ld, mode, colscale);
  else if (t->dtype == ZV_F16)
    pack_kernel<__half, DstT><<<blocks, 256, 0, s>>>(static_cast<const __half*>(t->data), dst, rows, cols, dst_ld, mode, colscale);
  else
    return fail(ZV_EINVAL, "zv_weights_pack: %s has unsupported dtype %d", t->name, t->dtype);
  count_launch();
  return ZV_OK;
}

// Folded LayerNorm bias and column sums of one consumer GEMM (ln_fold_kernel); wp = its packed 16-bit weights.
int ln_fold(const zv_tensor* t, const void* wp, bool f16, const float* beta, float* bias, float* csum, int64_t rows,
            int64_t cols, cudaStream_t s) {
  const unsigned blocks = (unsigned)((rows + 7) / 8);
#define ZV_FOLD(SRC)                                                                                                     \
  do {                                                                                                                   \
    const SRC* w_ = static_cast<const SRC*>(t->data);                                                                   \
    if (f16) ln_fold_kernel<SRC, __half><<<blocks, 256, 0, s>>>(w_, static_cast<const __half*>(wp), beta, bias, csum, rows, cols); \
    else ln_fold_kernel<SRC, __nv_bfloat16><<<blocks, 256, 0, s>>>(w_, static_cast<const __nv_bfloat16*>(wp), beta, bias, csum, rows, cols); \
  } while (0)
  if (t->dtype == ZV_F32) ZV_FOLD(float);
  else if (t->dtype == ZV_BF16) ZV_FOLD(__nv_bfloat16);
  else if (t->dtype == ZV_F16) ZV_FOLD(__half);
  else return fail(ZV_EINVAL, "zv_weights_pack: %s has unsupported dtype %d", t->name, t->dtype);
#undef ZV_FOLD
  count_launch();
  return ZV_OK;
}

// Every tensor of the Qwen2-VL tower's state dict (HF names relative to the tower), in packing order.
std::vector<std::string> qwen2_tensor_names(const zv_cfg* c) {
  std::vector<std::string> v{"patch_embed.proj.weight"};
  for (int l = 0; l < c->depth; ++l) {
    const std::string p = "blocks." + std::to_string(l) + ".";
    for (const char* n : {"norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "attn.qkv.weight", "attn.qkv.bias",
                          "attn.proj.weight", "attn.proj.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias"})
      v.push_back(p + n);
  }
  for (const char* n : {"merger.ln_q.weight", "merger.ln_q.bias", "merger.mlp.0.weight", "merger.mlp.0.bias",
                        "merger.mlp.2.weight", "merger.mlp.2.bias"})
    v.push_back(n);
  return v;
}

}  // namespace

int rmsnorm(const float* x, const float* w, void* y, int y_f16, int64_t rows, int hidden, float eps, void* stream) {
  if (hidden % 4 || hidden > 1280) return fail(ZV_EINVAL, "rmsnorm: hidden=%d unsupported", hidden);
  {
    KernelTimer timer(KC_RMSNORM, stream);
    launch_pdl(rmsnorm_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
               x, w, static_cast<uint16_t*>(y), y_f16 != 0, rows, hidden, eps);
  }
  count_launch();
  return ZV_OK;
}

int cast_rows_ss(const float* x, void* x16, int x16_f16, float* ss, int64_t rows, int hidden, void* stream) {
  if (hidden % 4) return fail(ZV_EINVAL, "cast_rows_ss: hidden=%d unsupported", hidden);
  {
    KernelTimer timer(KC_RMSNORM, stream);
    launch_pdl(cast_rows_ss_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
               x, static_cast<uint16_t*>(x16), x16_f16 != 0, ss, rows, hidden);
  }
  count_launch();
  return ZV_OK;
}

int cast_rows_ln(const float* x, void* x16, int x16_f16, float2* ln, int64_t rows, int hidden, void* stream) {
  if (hidden != 64 * kSsParts) return fail(ZV_EINVAL, "cast_rows_ln: hidden=%d unsupported", hidden);
  {
    KernelTimer timer(KC_RMSNORM, stream);
    launch_pdl(cast_rows_ln_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
               x, static_cast<uint16_t*>(x16), x16_f16 != 0, ln, rows, hidden);
  }
  count_launch();
  return ZV_OK;
}

int layernorm(const float* x, const float* w, const float* b, void* y, int y_f16, int64_t rows, int hidden, float eps,
              void* stream) {
  if (hidden % 4 || hidden > 1280) return fail(ZV_EINVAL, "layernorm: hidden=%d unsupported", hidden);
  {
    KernelTimer timer(KC_RMSNORM, stream);
    launch_pdl(layernorm_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
               x, w, b, static_cast<uint16_t*>(y), y_f16 != 0, rows, hidden, eps);
  }
  count_launch();
  return ZV_OK;
}

int gather_rows(const void* src, int src_dtype, void* dst, int dst_f16, const int32_t* widx, int64_t n_groups, int unit,
                int cols, void* stream) {
  const int ge = unit * cols;
  if (ge % 4) return fail(ZV_EINVAL, "gather_rows: group size must be a multiple of 4 elements");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  KernelTimer timer(KC_GATHER, stream);
  if (src_dtype == ZV_F32)
    launch_pdl(gather_kernel<float>, dim3((unsigned)n_groups), dim3(256), 0, s, 1, static_cast<const float*>(src),
               static_cast<uint16_t*>(dst), dst_f16 != 0, widx, ge);
  else   // already the 16-bit operand type: plain row move
    launch_pdl(gather_kernel<uint16_t>, dim3((unsigned)n_groups), dim3(256), 0, s, 1, static_cast<const uint16_t*>(src),
               static_cast<uint16_t*>(dst), dst_f16 != 0, widx, ge);
  count_launch();
  return ZV_OK;
}

}  // namespace zv

using namespace zv;

extern "C" {

int zv_plan_upload(zv_plan* p, void* plan_dev, int64_t bytes, void* stream) {
  if (!p || !plan_dev) return fail(ZV_EINVAL, "zv_plan_upload: null argument");
  if (bytes < p->dev.bytes) return fail(ZV_ENOMEM, "zv_plan_upload: buffer %lld B < required %lld B", (long long)bytes, (long long)p->dev.bytes);
  std::vector<uint8_t> image;
  plan_device_image(p, &image);
  cudaError_t e = cudaMemcpyAsync(plan_dev, image.data(), image.size(), cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_plan_upload: %s", cudaGetErrorString(e));
  return ZV_OK;
}

int64_t zv_weights_bytes(const zv_cfg* cfg) {
  int rc = check_cfg(cfg, "zv_weights_bytes");
  if (rc) return rc;
  return weight_layout(cfg).bytes;
}

int zv_weights_pack(const zv_cfg* cfg, const zv_tensor* tensors, int32_t n, void* packed_dev, int64_t packed_bytes,
                    void* stream_) {
  reset_launch_count();
  int rc = check_cfg(cfg, "zv_weights_pack");
  if (rc) return rc;
  if (!tensors || !packed_dev) return fail(ZV_EINVAL, "zv_weights_pack: null argument");
  std::map<std::string, const zv_tensor*> by_name;
  for (int32_t i = 0; i < n; ++i) {
    std::string nm = tensors[i].name ? tensors[i].name : "";
    for (const char* pre : {"model.visual.", "visual."})
      if (nm.rfind(pre, 0) == 0) { nm = nm.substr(std::strlen(pre)); break; }
    by_name[nm] = &tensors[i];
  }
  if (qwen2(cfg)) {                  // the whole state dict is checked before any device work: missing and extra tensors
    const std::vector<std::string> names = qwen2_tensor_names(cfg);
    for (const std::string& nm : names)
      if (!by_name.count(nm)) return fail(ZV_EINVAL, "zv_weights_pack: missing tensor %s", nm.c_str());
    for (const auto& kv : by_name)
      if (std::find(names.begin(), names.end(), kv.first) == names.end())
        return fail(ZV_EINVAL, "zv_weights_pack: unexpected tensor %s (not part of the Qwen2-VL tower of depth %d)",
                    kv.first.c_str(), cfg->depth);
  }
  rc = check_device("zv_weights_pack");
  if (rc) return rc;
  const WeightLayout L = weight_layout(cfg);
  if (packed_bytes < L.bytes) return fail(ZV_ENOMEM, "zv_weights_pack: buffer %lld B < required %lld B", (long long)packed_bytes, (long long)L.bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream_);
  auto get = [&](const std::string& nm) -> const zv_tensor* {
    auto it = by_name.find(nm);
    return it == by_name.end() ? nullptr : it->second;
  };
  cudaError_t e = cudaMemsetAsync(packed_dev, 0, (size_t)L.bytes, s);   // zero padding rows / columns
  if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_weights_pack: memset: %s", cudaGetErrorString(e));
  uint8_t* base = static_cast<uint8_t*>(packed_dev);
  const int64_t H = cfg->hidden, I = cfg->inter, IP = ipad(cfg), O = cfg->out_hidden;
  const bool f16 = cfg->op_dtype == ZV_F16;
#define ZV_TRY_PACK(expr) do { rc = (expr); if (rc) return rc; } while (0)
#define ZV_PACK_S(NAME, TYPE, OFF, ROWS, COLS, LD, MODE, SCALE)                                            \
  do {                                                                                                      \
    const zv_tensor* t_ = get(NAME);                                                                        \
    if (!t_) return fail(ZV_EINVAL, "zv_weights_pack: missing tensor %s", std::string(NAME).c_str());      \
    if (std::is_same<TYPE, __nv_bfloat16>::value && f16)                                                    \
      rc = pack_one<__half>(t_, reinterpret_cast<__half*>(base + (OFF)), ROWS, COLS, LD, MODE, s, SCALE);   \
    else                                                                                                    \
      rc = pack_one<TYPE>(t_, reinterpret_cast<TYPE*>(base + (OFF)), ROWS, COLS, LD, MODE, s, SCALE);       \
    if (rc) return rc;                                                                                      \
  } while (0)
#define ZV_PACK(NAME, TYPE, OFF, ROWS, COLS, LD, MODE) ZV_PACK_S(NAME, TYPE, OFF, ROWS, COLS, LD, MODE, nullptr)
  ZV_PACK("patch_embed.proj.weight", __nv_bfloat16, L.wpe, H, kPatchK, kPatchK, 0);
  auto fl = [&](size_t off) { return reinterpret_cast<float*>(base + off); };
  for (int l = 0; qwen2(cfg) && l < cfg->depth; ++l) {
    const std::string p = "blocks." + std::to_string(l) + ".";
    const LayerOff& o = L.layers[l];
    ZV_PACK(p + "norm1.weight", float, o.n1, 1, H, H, 0);
    ZV_PACK(p + "norm1.bias", float, o.n1b, 1, H, H, 0);
    ZV_PACK(p + "norm2.weight", float, o.n2, 1, H, H, 0);
    ZV_PACK(p + "norm2.bias", float, o.n2b, 1, H, H, 0);
    // gains into the weight columns as above; then b' = b + W beta and c = column sums of the packed W'
    ZV_PACK_S(p + "attn.qkv.weight", __nv_bfloat16, o.wqkv, 3 * H, H, H, 0, fl(o.n1));
    ZV_PACK(p + "attn.qkv.bias", float, o.bqkv, 1, 3 * H, 3 * H, 0);
    ZV_TRY_PACK(ln_fold(get(p + "attn.qkv.weight"), base + o.wqkv, f16, fl(o.n1b), fl(o.bqkv), fl(o.cqkv), 3 * H, H, s));
    ZV_PACK(p + "attn.proj.weight", __nv_bfloat16, o.wo, H, H, H, 0);
    ZV_PACK(p + "attn.proj.bias", float, o.bo, 1, H, H, 0);
    ZV_PACK_S(p + "mlp.fc1.weight", __nv_bfloat16, o.wgu, I, H, H, 0, fl(o.n2));
    ZV_PACK(p + "mlp.fc1.bias", float, o.bgu, 1, I, I, 0);
    ZV_TRY_PACK(ln_fold(get(p + "mlp.fc1.weight"), base + o.wgu, f16, fl(o.n2b), fl(o.bgu), fl(o.cfc1), I, H, s));
    ZV_PACK(p + "mlp.fc2.weight", __nv_bfloat16, o.wd, H, I, I, 0);
    ZV_PACK(p + "mlp.fc2.bias", float, o.bd, 1, H, H, 0);
  }
  if (qwen2(cfg)) ZV_PACK("merger.ln_q.bias", float, L.ln_qb, 1, H, H, 0);
  for (int l = 0; !qwen2(cfg) && l < cfg->depth; ++l) {
    const std::string p = "blocks." + std::to_string(l) + ".";
    const LayerOff& o = L.layers[l];
    ZV_PACK(p + "norm1.weight", float, o.n1, 1, H, H, 0);
    ZV_PACK(p + "norm2.weight", float, o.n2, 1, H, H, 0);
    // norm1 / norm2 gains (fp32, packed just above on the same stream) are folded into the columns of the GEMM that
    // consumes the normalised rows: W' = W diag(g), rounded once to the operand type
    const float* g1 = reinterpret_cast<const float*>(base + o.n1);
    const float* g2 = reinterpret_cast<const float*>(base + o.n2);
    ZV_PACK_S(p + "attn.qkv.weight", __nv_bfloat16, o.wqkv, 3 * H, H, H, 0, g1);
    ZV_PACK(p + "attn.qkv.bias", float, o.bqkv, 1, 3 * H, 3 * H, 0);
    ZV_PACK(p + "attn.proj.weight", __nv_bfloat16, o.wo, H, H, H, 0);
    ZV_PACK(p + "attn.proj.bias", float, o.bo, 1, H, H, 0);
    ZV_PACK_S(p + "mlp.gate_proj.weight", __nv_bfloat16, o.wgu, I, H, H, 1, g2);
    ZV_PACK_S(p + "mlp.up_proj.weight", __nv_bfloat16, o.wgu, I, H, H, 2, g2);
    ZV_PACK(p + "mlp.gate_proj.bias", float, o.bgu, I, 1, 1, 1);
    ZV_PACK(p + "mlp.up_proj.bias", float, o.bgu, I, 1, 1, 2);
    ZV_PACK(p + "mlp.down_proj.weight", __nv_bfloat16, o.wd, H, I, IP, 0);
    ZV_PACK(p + "mlp.down_proj.bias", float, o.bd, 1, H, H, 0);
  }
  ZV_PACK("merger.ln_q.weight", float, L.ln_q, 1, H, H, 0);
  ZV_PACK("merger.mlp.0.weight", __nv_bfloat16, L.w1, 4 * H, 4 * H, 4 * H, 0);
  ZV_PACK("merger.mlp.0.bias", float, L.b1, 1, 4 * H, 4 * H, 0);
  ZV_PACK("merger.mlp.2.weight", __nv_bfloat16, L.w2, O, 4 * H, 4 * H, 0);
  ZV_PACK("merger.mlp.2.bias", float, L.b2, 1, O, O, 0);
#undef ZV_PACK
#undef ZV_PACK_S
#undef ZV_TRY_PACK
  e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_weights_pack: %s", cudaGetErrorString(e));
  return ZV_OK;
}

namespace {
struct Workspace { int64_t p = 0, x = 0, y = 0, x16 = 0, ss = 0, big = 0, comp = 0, ln = 0, bytes = 0; };
Workspace workspace_layout(const zv_cfg* c, int64_t S) {
  Workspace w;
  const int64_t H = c->hidden;
  const int64_t wide = std::max<int64_t>(3 * H, ipad(c));
  int64_t off = 0;
  auto take = [&](int64_t bytes) { int64_t o = off; off = align_up(off + bytes, 1024); return o; };
  w.p = take(S * kPatchK * 2);
  w.x = take(S * H * 4);
  w.y = take(S * H * 2);
  w.x16 = take(S * H * 2);               // 16-bit copy of the residual stream (A operand of the QKV / gate-up GEMMs)
  w.ss = take(S * kSsParts * 4);         // per-row partial sums of squares of X (folded RMSNorm)
  w.big = take(S * wide * 2);
  w.comp = take((S / 4 + 1) * 4);        // int32 [T]: composed scatter rows of zv_visual_forward_into
  if (qwen2(c)) w.ln = take(S * kSsParts * 8);   // float2 [S][kSsParts]: per-slot (mean, M2) of X (folded LayerNorm)
  w.bytes = off;
  return w;
}
}  // namespace

int64_t zv_visual_workspace_bytes(const zv_cfg* cfg, const zv_plan* p) {
  int rc = check_cfg(cfg, "zv_visual_workspace_bytes");
  if (rc) return rc;
  if (!p) return fail(ZV_EINVAL, "zv_visual_workspace_bytes: null plan");
  return workspace_layout(cfg, p->S).bytes;
}

namespace {
int visual_forward_impl(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                        const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                        int32_t out_dtype, void* hidden_out_dev, void* workspace_dev, int64_t workspace_bytes,
                        void* const* peer_out_dev, int32_t n_peers, int64_t peer_row_off, const int64_t* dest_rows_dev,
                        int64_t dest_rows_limit, void* stream);
}

int zv_visual_forward(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                      const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                      int32_t out_dtype, void* hidden_out_dev, void* workspace_dev, int64_t workspace_bytes,
                      void* stream) {
  return visual_forward_impl(cfg, weights_dev, p, plan_dev, patches_dev, in_dtype, in_order, merged_out_dev, out_dtype,
                             hidden_out_dev, workspace_dev, workspace_bytes, nullptr, 0, 0, nullptr, 0, stream);
}

int zv_visual_forward_into(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                           const void* patches_dev, int32_t in_dtype, int32_t in_order, void* embeds_dev,
                           int64_t embeds_rows, int32_t embeds_dtype, const int64_t* dest_rows_dev, void* workspace_dev,
                           int64_t workspace_bytes, void* stream) {
  if (!dest_rows_dev || !embeds_dev) return fail(ZV_EINVAL, "zv_visual_forward_into: null argument");
  if (embeds_rows <= 0 || embeds_rows > INT32_MAX) return fail(ZV_EINVAL, "zv_visual_forward_into: inputs_embeds has %lld rows (1 .. 2^31-1 supported)", (long long)embeds_rows);
  return visual_forward_impl(cfg, weights_dev, p, plan_dev, patches_dev, in_dtype, in_order, embeds_dev, embeds_dtype,
                             nullptr, workspace_dev, workspace_bytes, nullptr, 0, 0, dest_rows_dev, embeds_rows, stream);
}

int zv_visual_forward_gather(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                             const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                             int32_t out_dtype, void* workspace_dev, int64_t workspace_bytes, void* const* peer_out_dev,
                             int32_t n_peers, int64_t peer_row_off, void* stream) {
  if (n_peers < 0 || n_peers > 8 || (n_peers > 0 && !peer_out_dev)) return fail(ZV_EINVAL, "zv_visual_forward_gather: bad peer list");
  if (n_peers > 0 && out_dtype == ZV_F32) return fail(ZV_EINVAL, "zv_visual_forward_gather: the fused gather writes 16-bit embeddings");
  return visual_forward_impl(cfg, weights_dev, p, plan_dev, patches_dev, in_dtype, in_order, merged_out_dev, out_dtype,
                             nullptr, workspace_dev, workspace_bytes, peer_out_dev, n_peers, peer_row_off, nullptr, 0, stream);
}

int zv_visual_forward_gather_rows(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                                  const void* patches_dev, int32_t in_dtype, int32_t in_order, void* gather_local_dev,
                                  int64_t gather_rows, int32_t out_dtype, const int64_t* dest_rows_dev, void* workspace_dev,
                                  int64_t workspace_bytes, void* const* peer_out_dev, int32_t n_peers, void* stream) {
  if (!dest_rows_dev || !gather_local_dev) return fail(ZV_EINVAL, "zv_visual_forward_gather_rows: null argument");
  if (gather_rows <= 0 || gather_rows > INT32_MAX) return fail(ZV_EINVAL, "zv_visual_forward_gather_rows: gather buffer has %lld rows (1 .. 2^31-1 supported)", (long long)gather_rows);
  if (n_peers < 0 || n_peers > 8 || (n_peers > 0 && !peer_out_dev)) return fail(ZV_EINVAL, "zv_visual_forward_gather_rows: bad peer list");
  if (out_dtype == ZV_F32) return fail(ZV_EINVAL, "zv_visual_forward_gather_rows: the fused gather writes 16-bit embeddings");
  return visual_forward_impl(cfg, weights_dev, p, plan_dev, patches_dev, in_dtype, in_order, gather_local_dev, out_dtype,
                             nullptr, workspace_dev, workspace_bytes, peer_out_dev, n_peers, 0, dest_rows_dev, gather_rows, stream);
}

namespace {
int visual_forward_impl(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                        const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                        int32_t out_dtype, void* hidden_out_dev, void* workspace_dev, int64_t workspace_bytes,
                        void* const* peer_out_dev, int32_t n_peers, int64_t peer_row_off, const int64_t* dest_rows_dev,
                        int64_t dest_rows_limit, void* stream) {
  reset_launch_count();
  NvtxRange nvtx_tower("zv:tower");
  int rc = check_cfg(cfg, "zv_visual_forward");
  if (rc) return rc;
  if (!weights_dev || !p || !plan_dev || !patches_dev || !merged_out_dev || !workspace_dev)
    return fail(ZV_EINVAL, "zv_visual_forward: null argument");
  const int op = cfg->op_dtype == ZV_F16 ? ZV_F16 : ZV_BF16;
  const int f16 = op == ZV_F16;
  if ((in_dtype != ZV_F32 && in_dtype != op) || (out_dtype != ZV_F32 && out_dtype != ZV_BF16 && out_dtype != ZV_F16))
    return fail(ZV_EINVAL, "zv_visual_forward: bad dtype (16-bit patches must be the operand type %s)", f16 ? "fp16" : "bf16");
  rc = check_device("zv_visual_forward");
  if (rc) return rc;
  const int64_t S = p->S, T = p->T, H = cfg->hidden, IP = ipad(cfg), O = cfg->out_hidden;
  const Workspace W = workspace_layout(cfg, S);
  if (workspace_bytes < W.bytes)
    return fail(ZV_ENOMEM, "zv_visual_forward: workspace %lld B < required %lld B", (long long)workspace_bytes, (long long)W.bytes);
  const WeightLayout L = weight_layout(cfg);
  const uint8_t* wb = static_cast<const uint8_t*>(weights_dev);
  const uint8_t* pd = static_cast<const uint8_t*>(plan_dev);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  const int32_t* d_pos = reinterpret_cast<const int32_t*>(pd + p->dev.off_pos);
  const float2* d_rope = reinterpret_cast<const float2*>(pd + p->dev.off_rope);
  const int32_t* d_widx = reinterpret_cast<const int32_t*>(pd + p->dev.off_widx);
  const int32_t* d_full = reinterpret_cast<const int32_t*>(pd + p->dev.off_full_tiles);
  const int32_t* d_wblk = reinterpret_cast<const int32_t*>(pd + p->dev.off_win_blocks);
  const int32_t* d_wbnd = reinterpret_cast<const int32_t*>(pd + p->dev.off_win_bounds);
  float* X = reinterpret_cast<float*>(ws + W.x);
  void* Y = ws + W.y;
  void* BIG = ws + W.big;
#define ZV_TRY(expr) do { rc = (expr); if (rc) return rc; } while (0)

  // patches -> bf16, window order
  const void* P = patches_dev;
  if (in_order == ZV_ORDER_HF) {
    ZV_TRY(gather_rows(patches_dev, in_dtype, ws + W.p, f16, d_widx, T, cfg->merge * cfg->merge, kPatchK, stream));
    P = ws + W.p;
  } else if (in_dtype == ZV_F32) {
    return fail(ZV_EINVAL, "zv_visual_forward: window-ordered input must be the 16-bit operand type (the fused zv_preprocess output)");
  }
  // patch embed (HF :113): X = P Wpe^T, fp32
  GemmArgs g{};
  g.op_f16 = f16;
  g.M = (int)S; g.N = (int)H; g.K = kPatchK; g.out = X; g.ldo = H; g.out_dtype = ZV_F32; g.bias = nullptr;
  ZV_TRY(gemm(EPI_STORE, g, P, kPatchK, wb + L.wpe, kPatchK, stream));

  void* X16 = ws + W.x16;
  float* SS = reinterpret_cast<float*>(ws + W.ss);
  if (qwen2(cfg)) {
    float2* LNS = reinterpret_cast<float2*>(ws + W.ln);
    ZV_TRY(cast_rows_ln(X, X16, f16, LNS, S, (int)H, stream));
    for (int l = 0; l < cfg->depth; ++l) {
      const LayerOff& o = L.layers[l];
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)(3 * H); g.K = (int)H; g.out = BIG; g.ldo = 3 * H; g.out_dtype = op;
      g.bias = reinterpret_cast<const float*>(wb + o.bqkv); g.pos = d_pos; g.rope = d_rope; g.heads = cfg->heads;
      g.row_ln = LNS; g.colsum = reinterpret_cast<const float*>(wb + o.cqkv); g.norm_eps = cfg->eps; g.norm_dim = (int)H;   // norm1
      ZV_TRY(gemm(EPI_QKV_ROPE_LN, g, X16, H, wb + o.wqkv, H, stream));
      ZV_TRY(attention_tc(BIG, Y, S, cfg->heads, (int)(H / cfg->heads), d_full, p->n_full_tiles, stream, f16 != 0));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)H; g.K = (int)H; g.out = X; g.ldo = H; g.out_dtype = ZV_F32;
      g.bias = reinterpret_cast<const float*>(wb + o.bo);
      g.x16_out = X16; g.ln_out = LNS;
      ZV_TRY(gemm(EPI_RESID_LN, g, Y, H, wb + o.wo, H, stream));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)IP; g.K = (int)H; g.out = BIG; g.ldo = IP; g.out_dtype = op;
      g.bias = reinterpret_cast<const float*>(wb + o.bgu);
      g.row_ln = LNS; g.colsum = reinterpret_cast<const float*>(wb + o.cfc1); g.norm_eps = cfg->eps; g.norm_dim = (int)H;   // norm2
      ZV_TRY(gemm(EPI_QGELU, g, X16, H, wb + o.wgu, H, stream));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)H; g.K = (int)IP; g.out = X; g.ldo = H; g.out_dtype = ZV_F32;
      g.bias = reinterpret_cast<const float*>(wb + o.bd);
      if (l + 1 < cfg->depth) { g.x16_out = X16; g.ln_out = LNS; }             // the merger normalises in fp32 itself
      ZV_TRY(gemm(EPI_RESID_LN, g, BIG, IP, wb + o.wd, IP, stream));
    }
  } else {
    ZV_TRY(cast_rows_ss(X, X16, f16, SS, S, (int)H, stream));
    for (int l = 0; l < cfg->depth; ++l) {
      const LayerOff& o = L.layers[l];
      const bool full = (cfg->fullatt_mask_lo >> l) & 1;
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)(3 * H); g.K = (int)H; g.out = BIG; g.ldo = 3 * H; g.out_dtype = op;
      g.bias = reinterpret_cast<const float*>(wb + o.bqkv); g.pos = d_pos; g.rope = d_rope; g.heads = cfg->heads;
      g.row_ss = SS; g.norm_eps = cfg->eps; g.norm_dim = (int)H;               // norm1 (gain folded into Wqkv)
      ZV_TRY(gemm(EPI_QKV_ROPE, g, X16, H, wb + o.wqkv, H, stream));
      if (full)
        ZV_TRY(attention_tc(BIG, Y, S, cfg->heads, (int)(H / cfg->heads), d_full, p->n_full_tiles, stream, f16 != 0));
      else
        ZV_TRY(attention_win_tc(BIG, Y, S, cfg->heads, (int)(H / cfg->heads), d_wblk, p->n_win_blocks, d_wbnd, stream, f16 != 0));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)H; g.K = (int)H; g.out = X; g.ldo = H; g.out_dtype = ZV_F32;
      g.bias = reinterpret_cast<const float*>(wb + o.bo);
      g.x16_out = X16; g.ss_out = SS;
      ZV_TRY(gemm(EPI_RESID, g, Y, H, wb + o.wo, H, stream));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)(2 * IP); g.K = (int)H; g.out = BIG; g.ldo = IP; g.out_dtype = op;
      g.bias = reinterpret_cast<const float*>(wb + o.bgu);
      g.row_ss = SS; g.norm_eps = cfg->eps; g.norm_dim = (int)H;               // norm2 (gain folded into Wgate / Wup)
      ZV_TRY(gemm(EPI_SWIGLU, g, X16, H, wb + o.wgu, H, stream));
      g = GemmArgs{};
      g.op_f16 = f16;
      g.M = (int)S; g.N = (int)H; g.K = (int)IP; g.out = X; g.ldo = H; g.out_dtype = ZV_F32;
      g.bias = reinterpret_cast<const float*>(wb + o.bd);
      if (l + 1 < cfg->depth) { g.x16_out = X16; g.ss_out = SS; }                // the merger normalises in fp32 itself
      ZV_TRY(gemm(EPI_RESID, g, BIG, IP, wb + o.wd, IP, stream));
    }
  }
  if (hidden_out_dev) {
    cudaError_t e = cudaMemcpyAsync(hidden_out_dev, X, (size_t)(S * H * 4), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_visual_forward: hidden copy: %s", cudaGetErrorString(e));
  }
  // merger (HF :133-146; Qwen2-VL: LayerNorm ln_q) + un-reorder (HF :512-513)
  if (qwen2(cfg))
    ZV_TRY(layernorm(X, reinterpret_cast<const float*>(wb + L.ln_q), reinterpret_cast<const float*>(wb + L.ln_qb), Y, f16, S,
                     (int)H, cfg->eps, stream));
  else
    ZV_TRY(rmsnorm(X, reinterpret_cast<const float*>(wb + L.ln_q), Y, f16, S, (int)H, cfg->eps, stream));
  g = GemmArgs{};
  g.op_f16 = f16;
  g.M = (int)T; g.N = (int)(4 * H); g.K = (int)(4 * H); g.out = BIG; g.ldo = 4 * H; g.out_dtype = op;
  g.bias = reinterpret_cast<const float*>(wb + L.b1);
  ZV_TRY(gemm(EPI_GELU, g, Y, 4 * H, wb + L.w1, 4 * H, stream));
  g = GemmArgs{};
  g.op_f16 = f16;
  g.M = (int)T; g.N = (int)O; g.K = (int)(4 * H); g.out = merged_out_dev; g.ldo = O; g.out_dtype = out_dtype;
  g.bias = reinterpret_cast<const float*>(wb + L.b2); g.scatter = d_widx;
  if (dest_rows_dev) {
    // LM hand-off (HF :1301-1307 masked_scatter): the un-reorder and the scatter into inputs_embeds are one index map
    int32_t* comp = reinterpret_cast<int32_t*>(ws + W.comp);
    launch_pdl(compose_rows_kernel, dim3((unsigned)((T + 255) / 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
               dest_rows_dev, d_widx, comp, T, dest_rows_limit);
    count_launch();
    g.scatter = comp;
  }
  g.n_peers = n_peers; g.peer_row_off = peer_row_off;
  for (int i = 0; i < n_peers; ++i) g.peers[i] = peer_out_dev[i];
  ZV_TRY(gemm(EPI_SCATTER, g, BIG, 4 * H, wb + L.w2, 4 * H, stream));
#undef ZV_TRY
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_visual_forward: %s", cudaGetErrorString(e));
  return ZV_OK;
}
}  // namespace

int zv_attention(const void* qkv_dev, void* out_dev, int32_t heads, int32_t head_dim, const int32_t* cu_host,
                 int32_t n_seg, void* work_dev, int64_t work_bytes, int32_t dtype, void* stream) {
  reset_launch_count();
  if (!qkv_dev || !out_dev || !cu_host || n_seg <= 0 || !work_dev) return fail(ZV_EINVAL, "zv_attention: bad argument");
  int rc = check_device("zv_attention");
  if (rc) return rc;
  int32_t longest = 0;
  for (int32_t s = 0; s < n_seg; ++s) longest = std::max(longest, cu_host[s + 1] - cu_host[s]);
  if (longest <= 64) {             // same choice the tower makes: the window kernel, else 128-row q tiles for the full one
    // window layers: row blocks + per-row bounds, uploaded into the work buffer, then the tcgen05 window kernel
    std::vector<int32_t> cu(cu_host, cu_host + n_seg + 1), blocks;
    build_window_blocks(cu, 128, &blocks);
    const int64_t S_ = cu_host[n_seg];
    const int64_t off_bounds = ((int64_t)blocks.size() * 4 + 255) / 256 * 256;
    const int64_t need_w = off_bounds + (S_ + 136) * 8;       // zero padding behind the table (130-row bulk copies)
    if (work_bytes < need_w) return fail(ZV_ENOMEM, "zv_attention: work buffer %lld B < required %lld B", (long long)work_bytes, (long long)need_w);
    std::vector<int32_t> bounds((size_t)(S_ + 136) * 2, 0);
    fill_window_bounds(cu, bounds.data());
    uint8_t* w = static_cast<uint8_t*>(work_dev);
    cudaError_t e1 = cudaMemcpyAsync(w, blocks.data(), blocks.size() * 4, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
    if (e1 == cudaSuccess) e1 = cudaMemcpyAsync(w + off_bounds, bounds.data(), bounds.size() * 4, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
    if (e1 != cudaSuccess) return fail(ZV_ECUDA, "zv_attention: %s", cudaGetErrorString(e1));
    return attention_win_tc(qkv_dev, out_dev, S_, heads, head_dim, reinterpret_cast<const int32_t*>(w), (int)(blocks.size() / 4),
                            reinterpret_cast<const int32_t*>(w + off_bounds), stream, dtype == ZV_F16);
  }
  std::vector<int32_t> tiles;
  for (int32_t s = 0; s < n_seg; ++s)
    for (int32_t q0 = cu_host[s]; q0 < cu_host[s + 1]; q0 += 128) {
      tiles.push_back(q0); tiles.push_back(std::min(128, cu_host[s + 1] - q0));
      tiles.push_back(cu_host[s]); tiles.push_back(cu_host[s + 1]);
    }
  const int64_t S = cu_host[n_seg];
  const int64_t need = ((int64_t)tiles.size() * 4 + 255) / 256 * 256;
  if (work_bytes < need) return fail(ZV_ENOMEM, "zv_attention: work buffer %lld B < required %lld B", (long long)work_bytes, (long long)need);
  cudaError_t e = cudaMemcpyAsync(work_dev, tiles.data(), tiles.size() * 4, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(ZV_ECUDA, "zv_attention: %s", cudaGetErrorString(e));
  return attention_tc(qkv_dev, out_dev, S, heads, head_dim, static_cast<const int32_t*>(work_dev), (int)(tiles.size() / 4), stream,
                      dtype == ZV_F16);
}

}  // extern "C"
