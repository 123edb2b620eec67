// K2: persistent, warp-specialised tcgen05 GEMM for the tower's contractions
//   C[M,N] = A[M,K] (bf16, K-major) x B[N,K]^T (bf16, K-major), fp32 accumulation in TMEM,
// with the epilogues the Qwen2.5-VL vision block needs fused in (HF modeling_qwen2_5_vl.py):
//   EPI_STORE    plain (+bias) store, fp32 or bf16            patch_embed :113, generic
//   EPI_QKV_ROPE bias + 2D rotary on q,k heads -> bf16        attn.qkv :226-229 + apply_rotary_pos_emb_vision :156-167
//   EPI_RESID    X(fp32) += acc + bias                        attn.proj / mlp.down_proj + residual :311-320
//   EPI_SWIGLU   silu(gate+bg) * (up+bu) -> bf16              mlp :88 (gate/up rows interleaved per 128)
//   EPI_GELU     gelu_erf(acc + bias) -> bf16                 merger.mlp.0/1 :138-140
//   EPI_SCATTER  (acc + bias) -> row scatter[row]             merger.mlp.2 + un-reorder :512-513
// and, for the Qwen2-VL tower (HF models/qwen2_vl/modeling_qwen2_vl.py), the LayerNorm-fold variants
//   EPI_QKV_ROPE_LN  r * (acc - mu * c) + b', then the rotary    norm1 + attn.qkv
//   EPI_RESID_LN     EPI_RESID with per-slot (mean, M2) of the new rows   attn.proj / mlp.fc2 + residual
//   EPI_QGELU        quick_gelu(r * (acc - mu * c) + b') -> 16-bit       norm2 + mlp.fc1 + QuickGELU
//
// Structure (one CTA per SM, 384 threads): warp 0 = TMA producer (one elected lane), warp 1 = MMA issuer
// (one elected lane, tcgen05.mma M=128 x N=BN x K=16 from 128B-swizzled smem tiles), warp 2 = TMEM
// allocator, warps 4-11 = epilogue (tcgen05.ld, one accumulator row x half the columns per thread).  Three mbarrier pipelines:
// smem full/empty (TMA <-> MMA), TMEM full/empty (MMA <-> epilogue, two accumulator stages so the epilogue
// of tile i overlaps the MMAs of tile i+1), and a static persistent tile schedule (n fastest, so CTAs that run
// together share the A rows in L2 and the whole B matrix stays L2-resident).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <mutex>

#include "zv_common.h"
#include "zv_gemm.h"
#include "zv_ptx.cuh"

namespace zv {

using namespace ptx;

namespace {

constexpr int BM = 128, BK = 64, UMMA_K = 16;
constexpr int kThreads = 384;          // 4 role warps + 8 epilogue warps
constexpr int kTmemCols = 512;

constexpr int kXposePitch = 36;                                 // floats per staged row (32 + 4: conflict-free 16 B accesses)
constexpr int kXposeBytesPerWarp = 32 * kXposePitch * 4;
// QKV epilogue staging: rotary pairs of the 4 half-0 warps (24 pairs x 32 rows x 8 B), of the 4 half-1 warps (16 pairs),
// then one [32][88] 16-bit output tile per lane quarter
constexpr int kQkvRope0 = 24 * 32 * 8, kQkvRope1 = 16 * 32 * 8, kQkvTilePitch = 88, kQkvTile = 32 * kQkvTilePitch * 2;
constexpr int kQkvStageBytes = 4 * kQkvRope0 + 4 * kQkvRope1 + 4 * kQkvTile;
__host__ __device__ constexpr bool is_resid(int e) { return e == EPI_RESID || e == EPI_RESID_LN; }
__host__ __device__ constexpr bool is_qkv(int e) { return e == EPI_QKV_ROPE || e == EPI_QKV_ROPE_LN; }
template <int BN, int CG, int EPI = 0> struct Cfg {
  static constexpr int kBRows = BN / CG;                       // B rows staged per CTA (half the tile in a CTA pair)
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = kBRows * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // the residual epilogue transposes its tile through shared memory (8 warps x 4.5 KB): one pipeline stage less
  // ... and the QKV epilogue keeps each row's rotary (cos, sin) pairs and a 32 x 80 output tile per lane quarter there
  // ... and the scatter epilogue regroups its 16-bit rows there so that four lanes store 64 contiguous bytes of a row
  static constexpr int kXposeBytes = (is_resid(EPI) || EPI == EPI_SCATTER) ? 8 * kXposeBytesPerWarp : is_qkv(EPI) ? kQkvStageBytes : 0;
  static constexpr int kStages = ((kBRows > 128) ? 4 : 6) - ((is_resid(EPI) || is_qkv(EPI) || EPI == EPI_SCATTER) ? 1 : 0);
  static constexpr int kBarBytes = 256;
  static constexpr int kSmemBytes = kStages * kStageBytes + kBarBytes + kXposeBytes + 1024;   // +1024: manual alignment slack
};

__device__ __forceinline__ float silu(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
__device__ __forceinline__ float quick_gelu(float x) { return __fdividef(x, 1.0f + __expf(-1.702f * x)); }
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
// two fp32 -> packed 16-bit pair, bf16 or fp16 (warp-uniform choice)
__device__ __forceinline__ uint32_t pack2(float a, float b, bool f16) {
  if (f16) { __half2 v = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
}
// 32 consecutive fp32 bias values (warp-uniform address: broadcast loads)
__device__ __forceinline__ void load_bias32(const float* __restrict__ b, float (&v)[32]) {
  const float4* p = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float4 t = __ldg(p + j); v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w; }
}

// folded RMSNorm, consumer side: 1 / rms of accumulator row `row` from the partial sums its producer left (1 when unused)
__device__ __forceinline__ float row_rscale(const GemmArgs& g, int row, bool valid) {
  if (g.row_ss == nullptr || !valid) return 1.f;
  const float2* p = reinterpret_cast<const float2*>(g.row_ss + (int64_t)row * kSsParts);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kSsParts / 2; ++i) { const float2 t = __ldg(p + i); s += t.x; s += t.y; }
  return rsqrtf(s / (float)g.norm_dim + g.norm_eps);
}

// folded LayerNorm, consumer side: mean and 1 / std of accumulator row `row` from its producer's 20 slot statistics
// (64 columns each), merged in slot order with Chan's formula - no E[x^2] - E[x]^2 cancellation (0 and 1 when unused)
__device__ __forceinline__ void row_ln_stats(const GemmArgs& g, int row, bool valid, float& mu, float& rs) {
  mu = 0.f; rs = 1.f;
  if (!valid) return;
  const float4* p = reinterpret_cast<const float4*>(g.row_ln + (int64_t)row * kSsParts);
  float mean = 0.f, m2 = 0.f;
#pragma unroll
  for (int i = 0; i < kSsParts / 2; ++i) {
    const float4 t = __ldg(p + i);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = 2 * i + h;                          // slots merged so far
      const float mb = h ? t.z : t.x, m2b = h ? t.w : t.y;
      if (k == 0) { mean = mb; m2 = m2b; continue; }
      const float d = mb - mean;
      mean = fmaf(d, 1.f / (float)(k + 1), mean);
      m2 += fmaf(d * d, 64.f * (float)k / (float)(k + 1), m2b);
    }
  }
  mu = mean;
  rs = rsqrtf(m2 / (float)g.norm_dim + g.norm_eps);
}

// ---- epilogues.  Eight epilogue warps: lane quarter q = warp & 3 (the TMEM lanes a warp may read), column half
// h = (warp - 4) >> 2.  One thread = one accumulator row, half of the tile's columns.  `taddr` carries the quarter.
template <int BN, int EPI, typename WaitFn>
__device__ __forceinline__ void epilogue_tile(uint32_t taddr, int m_blk, int n_blk, int row_local, int half,
                                              const GemmArgs& g, float* xpose, WaitFn wait_accumulator) {
  const int row = m_blk * BM + row_local;
  const bool valid = row < g.M;
  const bool of16 = g.out_dtype == ZV_F16;
  if constexpr (!is_resid(EPI) && EPI != EPI_QKV_ROPE_LN && EPI != EPI_QGELU) wait_accumulator();
  if constexpr (is_resid(EPI)) {
    // X(fp32) += acc + bias, coalesced: the accumulator chunk (32 rows x 32 columns per warp, one row per thread)
    // is transposed through shared memory so that a warp instruction touches 4 rows x 128 contiguous bytes of X
    // (4 L1 wavefronts) instead of 32 rows x 16 bytes (32 wavefronts).  The residual values of a chunk are fetched
    // before its accumulator is read; the first chunk's even before the MMAs of the tile have finished.
    constexpr int HALF = BN / 2;
    const int lane = row_local & 31;
    const int rr = lane >> 3, cc = (lane & 7) * 4;                      // this lane's row (mod 4) and column in the chunk
    const int row_base = m_blk * BM + (row_local & ~31);
    float* xrow = static_cast<float*>(g.out) + (int64_t)row_base * g.ldo + n_blk * BN + half * HALF + cc;
    float4 xv[8];
    auto load_x = [&](int c) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = 4 * i + rr;
        xv[i] = (row_base + r < g.M) ? *reinterpret_cast<const float4*>(xrow + (int64_t)r * g.ldo + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // folded RMSNorm, producer side: 16-bit copy of the new rows + this thread's share of their sums of squares
    const bool emit = g.x16_out != nullptr;
    uint16_t* x16row = static_cast<uint16_t*>(g.x16_out) + (int64_t)row_base * g.N + n_blk * BN + half * HALF + cc;
    float ssp[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) ssp[i] = 0.f;
    // EPI_RESID_LN: per row, sums of (x - x0) and (x - x0)^2 over this tile half, x0 = the row's first value in it
    constexpr bool LN = EPI == EPI_RESID_LN;
    float x0[8], s1[8], s2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x0[i] = s1[i] = s2[i] = 0.f;
    load_x(0);
    wait_accumulator();
#pragma unroll 1
    for (int c = 0; c < HALF; c += 32) {
      uint32_t r[32];
      __syncwarp();
      tmem_ld_x32(taddr + half * HALF + c, r);
      float v[32];
      load_bias32(g.bias + n_blk * BN + half * HALF + c, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(xpose + lane * kXposePitch + 4 * j) =
            make_float4(v[4 * j] + __uint_as_float(r[4 * j]), v[4 * j + 1] + __uint_as_float(r[4 * j + 1]),
                        v[4 * j + 2] + __uint_as_float(r[4 * j + 2]), v[4 * j + 3] + __uint_as_float(r[4 * j + 3]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rw = 4 * i + rr;
        const float4 a = *reinterpret_cast<const float4*>(xpose + rw * kXposePitch + cc);
        if (row_base + rw < g.M) {
          const float4 nx = make_float4(xv[i].x + a.x, xv[i].y + a.y, xv[i].z + a.z, xv[i].w + a.w);
          *reinterpret_cast<float4*>(xrow + (int64_t)rw * g.ldo + c) = nx;
          if (emit) {
            *reinterpret_cast<uint2*>(x16row + (int64_t)rw * g.N + c) = make_uint2(pack2(nx.x, nx.y, g.op_f16 != 0), pack2(nx.z, nx.w, g.op_f16 != 0));
            if constexpr (!LN) ssp[i] += nx.x * nx.x + nx.y * nx.y + nx.z * nx.z + nx.w * nx.w;
          }
        }
        if constexpr (LN) {
          if (emit) {                                   // whole warp: rows past M compute values nobody stores
            const float4 nx = make_float4(xv[i].x + a.x, xv[i].y + a.y, xv[i].z + a.z, xv[i].w + a.w);
            if (c == 0) x0[i] = __shfl_sync(0xffffffffu, nx.x, lane & ~7);
            const float dx = nx.x - x0[i], dy = nx.y - x0[i], dz = nx.z - x0[i], dw = nx.w - x0[i];
            s1[i] += (dx + dy) + (dz + dw);
            s2[i] += (dx * dx + dy * dy) + (dz * dz + dw * dw);
          }
        }
      }
      if (c + 32 < HALF) load_x(c + 32);
    }
    if (LN && emit) {
      // fixed-order butterfly over the row's 8 lanes, then the half's (mean, M2); a 128-column half stores
      // (mean, M2 / 2) in both of its 64-column slots (merging two equal-mean halves gives back M2 exactly)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float a1 = s1[i], a2 = s2[i];
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
        const float mean_off = a1 / (float)HALF;
        const float m2 = fmaxf(fmaf(-a1, mean_off, a2), 0.f);
        const int rw = 4 * i + rr;
        if ((lane & 7) == 0 && row_base + rw < g.M) {
          float2* o = g.ln_out + (int64_t)(row_base + rw) * kSsParts + (n_blk * BN + half * HALF) / 64;
          if (HALF == 128) { o[0] = o[1] = make_float2(x0[i] + mean_off, 0.5f * m2); }
          else o[0] = make_float2(x0[i] + mean_off, m2);
        }
      }
    } else if (emit) {
      // the 8 lanes that share a row (lane >> 3) each hold 4 of every 32 columns: fixed-order butterfly, then one
      // lane writes the row's partial for this 128-column half (deterministic: no atomics)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float v = ssp[i];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        const int rw = 4 * i + rr;
        if ((lane & 7) == 0 && row_base + rw < g.M)
          g.ss_out[(int64_t)(row_base + rw) * kSsParts + (n_blk * BN + half * HALF) / 64] = v;
      }
    }
  } else if constexpr (EPI == EPI_STORE || EPI == EPI_GELU || EPI == EPI_SCATTER || EPI == EPI_QGELU) {
    constexpr int HALF = BN / 2;
    int64_t orow = row;
    bool keep = valid;
    float mu = 0.f, rs = 1.f;
    if constexpr (EPI == EPI_QGELU) {
      row_ln_stats(g, row, valid, mu, rs);              // folded norm2: the row's statistics while the MMAs run
      wait_accumulator();
    }
    if constexpr (EPI == EPI_SCATTER) { orow = valid ? (int64_t)__ldg(g.scatter + row) : 0; keep = valid && orow >= 0; }
    const int c_begin = half * HALF;
#pragma unroll 1
    for (int c = c_begin; c < c_begin + HALF; c += 32) {
      uint32_t r[32];
      __syncwarp();
      tmem_ld_x32(taddr + c, r);
      const int n0 = n_blk * BN + c;
      float v[32];
      if (g.bias) load_bias32(g.bias + n0, v);
      else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      }
      if constexpr (EPI == EPI_QGELU) {
        float cs[32];
        load_bias32(g.colsum + n0, cs);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = quick_gelu(fmaf(fmaf(-mu, cs[j], __uint_as_float(r[j])), rs, v[j]));
      } else {
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(r[j]);
      }
      if constexpr (EPI == EPI_GELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
      }
      if (keep) {
        if (g.out_dtype == ZV_F32) {
          float4* o = reinterpret_cast<float4*>(static_cast<float*>(g.out) + orow * g.ldo + n0);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        } else {
          uint4 pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            pk[j] = make_uint4(pack2(v[8 * j], v[8 * j + 1], of16), pack2(v[8 * j + 2], v[8 * j + 3], of16),
                               pack2(v[8 * j + 4], v[8 * j + 5], of16), pack2(v[8 * j + 6], v[8 * j + 7], of16));
          if constexpr (EPI != EPI_SCATTER) {
            uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.out) + orow * g.ldo + n0);
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = pk[j];
          } else {
            // this row's 64 bytes -> the warp's staging tile (row pitch 80 B: conflict-free 16-byte accesses)
            uint4* st = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(xpose) + (row_local & 31) * 80);
#pragma unroll
            for (int j = 0; j < 4; ++j) st[j] = pk[j];
          }
        }
      }
      if constexpr (EPI == EPI_SCATTER) {
        if (g.out_dtype != ZV_F32) {
          // Scattered 16-bit rows leave in 64-byte runs: four lanes per row, eight rows per store instruction, instead
          // of 32 lanes x 16 bytes of 32 different rows.  The same runs go straight into every peer's gather buffer
          // (P2P stores over NVLink / NVSwitch) - the fused embedding gather - where small scattered stores cost most.
          __syncwarp();
          const int ln = row_local & 31, piece = ln & 3;
          const int row_base = m_blk * BM + (row_local & ~31);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int rw = 8 * i + (ln >> 2);
            const int64_t dr = row_base + rw < g.M ? (int64_t)__ldg(g.scatter + row_base + rw) : -1;
            if (dr >= 0) {                 // dr < 0: a destination row the caller's index put out of range (dropped)
              const uint4 val = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(xpose) + rw * 80 + piece * 16);
              *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.out) + dr * g.ldo + n0 + piece * 8) = val;
              for (int p = 0; p < g.n_peers; ++p)
                *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.peers[p]) + (g.peer_row_off + dr) * g.ldo + n0 + piece * 8) = val;
            }
          }
          __syncwarp();
        }
      }
    }
  } else if constexpr (EPI == EPI_SWIGLU) {
    static_assert(EPI != EPI_SWIGLU || BN == 256, "SwiGLU tiles hold 128 gate + 128 up columns");
    const float rs = row_rscale(g, row, valid);
#pragma unroll 1
    for (int c = half * 64; c < half * 64 + 64; c += 32) {
      uint32_t a[32], b[32];
      __syncwarp();
      tmem_ld_x32(taddr + c, a);
      tmem_ld_x32(taddr + 128 + c, b);
      float bg[32], bu[32];
      load_bias32(g.bias + (int64_t)n_blk * 256 + c, bg);
      load_bias32(g.bias + (int64_t)n_blk * 256 + 128 + c, bu);
      tmem_ld_wait();
      uint32_t o[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float g0 = fmaf(__uint_as_float(a[2 * j]), rs, bg[2 * j]), g1 = fmaf(__uint_as_float(a[2 * j + 1]), rs, bg[2 * j + 1]);
        const float u0 = fmaf(__uint_as_float(b[2 * j]), rs, bu[2 * j]), u1 = fmaf(__uint_as_float(b[2 * j + 1]), rs, bu[2 * j + 1]);
        o[j] = pack2(silu(g0) * u0, silu(g1) * u1, of16);
      }
      if (valid) {
        uint4* dst = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.out) + (int64_t)row * g.ldo + n_blk * 128 + c);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
      }
    }
  } else if constexpr (is_qkv(EPI)) {
    static_assert(!is_qkv(EPI) || BN == 240, "QKV tiles hold three 80-wide heads");
    // The two warps of a lane quarter split the 40 rotation pairs (d, d+40) of every head 24 : 16 (half 0 owns
    // columns [0,24) + [40,64), half 1 owns [24,40) + [64,80)).  Angle of pair d: pos_h * f_d for d < 20,
    // pos_w * f_(d-20) for d >= 20 (emb = cat(rot, rot), HF :485).  Each thread fetches its row's (cos, sin) pairs ONCE
    // per tile - before the accumulator is ready - and parks them in shared memory; the rotated 16-bit values of a
    // head go through a [32][80] tile per quarter so that the global stores are whole 160-byte head rows.
    const int lane = row_local & 31, q = row_local >> 5;
    uint8_t* stage = reinterpret_cast<uint8_t*>(xpose);
    float2* ropeS = reinterpret_cast<float2*>(stage + (half == 0 ? q * kQkvRope0 : 4 * kQkvRope0 + q * kQkvRope1));
    uint16_t* tileS = reinterpret_cast<uint16_t*>(stage + 4 * kQkvRope0 + 4 * kQkvRope1 + q * kQkvTile);
    const int NP = half == 0 ? 24 : 16, P0 = half == 0 ? 0 : 24;
    {
      int ph = 0, pw = 0;
      if (valid) { ph = __ldg(g.pos + 2 * row); pw = __ldg(g.pos + 2 * row + 1); }
      const float2* rope_h = g.rope + (int64_t)ph * 20;
      const float2* rope_w = g.rope + (int64_t)pw * 20;
      for (int d = 0; d < NP; ++d) {
        const int pair = P0 + d;
        ropeS[d * 32 + lane] = pair < 20 ? __ldg(rope_h + pair) : __ldg(rope_w + (pair - 20));
      }
    }
    float mu = 0.f, rs;
    if constexpr (EPI == EPI_QKV_ROPE_LN) row_ln_stats(g, row, valid, mu, rs);
    else rs = row_rscale(g, row, valid);
    // accumulator of column n with the folded LayerNorm's mean term taken out (EPI_QKV_ROPE: the accumulator itself)
    auto centred = [&](uint32_t acc, int n) {
      if constexpr (EPI == EPI_QKV_ROPE_LN) return fmaf(-mu, __ldg(g.colsum + n), __uint_as_float(acc));
      else return __uint_as_float(acc);
    };
    wait_accumulator();
    const bool rot_heads_possible = n_blk * 3 < 2 * g.heads;
    const int row0 = m_blk * BM + q * 32;                  // first row of this quarter
    const int t64 = half * 32 + lane;                      // thread index inside the quarter's warp pair
#pragma unroll 1
    for (int hh = 0; hh < 3; ++hh) {
      const int n0 = n_blk * 240 + hh * 80;
      const bool rotate = rot_heads_possible && n_blk * 3 + hh < 2 * g.heads;   // q and k heads; v heads pass through
      float lo[24], hi[24];
      if (half == 0) {
        uint32_t l16[16], l8[8], h16[16], h8[8];
        __syncwarp();
        tmem_ld_x16(taddr + hh * 80, l16);
        tmem_ld_x8(taddr + hh * 80 + 16, l8);
        tmem_ld_x16(taddr + hh * 80 + 40, h16);
        tmem_ld_x8(taddr + hh * 80 + 56, h8);
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(g.bias + n0) + j);
          lo[4 * j] = t.x; lo[4 * j + 1] = t.y; lo[4 * j + 2] = t.z; lo[4 * j + 3] = t.w;
          const float4 u = __ldg(reinterpret_cast<const float4*>(g.bias + n0 + 40) + j);
          hi[4 * j] = u.x; hi[4 * j + 1] = u.y; hi[4 * j + 2] = u.z; hi[4 * j + 3] = u.w;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) { lo[j] = fmaf(centred(l16[j], n0 + j), rs, lo[j]); hi[j] = fmaf(centred(h16[j], n0 + 40 + j), rs, hi[j]); }
#pragma unroll
        for (int j = 0; j < 8; ++j) { lo[16 + j] = fmaf(centred(l8[j], n0 + 16 + j), rs, lo[16 + j]); hi[16 + j] = fmaf(centred(h8[j], n0 + 56 + j), rs, hi[16 + j]); }
      } else {
        uint32_t l16[16], h16[16];
        __syncwarp();
        tmem_ld_x16(taddr + hh * 80 + 24, l16);
        tmem_ld_x16(taddr + hh * 80 + 64, h16);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(g.bias + n0 + 24) + j);
          lo[4 * j] = t.x; lo[4 * j + 1] = t.y; lo[4 * j + 2] = t.z; lo[4 * j + 3] = t.w;
          const float4 u = __ldg(reinterpret_cast<const float4*>(g.bias + n0 + 64) + j);
          hi[4 * j] = u.x; hi[4 * j + 1] = u.y; hi[4 * j + 2] = u.z; hi[4 * j + 3] = u.w;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) { lo[j] = fmaf(centred(l16[j], n0 + 24 + j), rs, lo[j]); hi[j] = fmaf(centred(h16[j], n0 + 64 + j), rs, hi[j]); }
      }
      if (rotate) {
#pragma unroll
        for (int d = 0; d < 24; ++d) {
          if (d < NP) {
            const float2 cs = ropeS[d * 32 + lane];
            const float l = lo[d], h = hi[d];
            lo[d] = l * cs.x - h * cs.y;           // x*cos + rotate_half(x)*sin, rotate_half = (-x[40:], x[:40])
            hi[d] = h * cs.x + l * cs.y;
          }
        }
      }
      // this thread's two column runs of the head row -> the quarter's tile, 16 bytes at a time
      uint16_t* trow = tileS + lane * kQkvTilePitch + P0;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        if (8 * j < NP) {
          *reinterpret_cast<uint4*>(trow + 8 * j) = make_uint4(pack2(lo[8 * j], lo[8 * j + 1], of16), pack2(lo[8 * j + 2], lo[8 * j + 3], of16),
                                                               pack2(lo[8 * j + 4], lo[8 * j + 5], of16), pack2(lo[8 * j + 6], lo[8 * j + 7], of16));
          *reinterpret_cast<uint4*>(trow + 40 + 8 * j) = make_uint4(pack2(hi[8 * j], hi[8 * j + 1], of16), pack2(hi[8 * j + 2], hi[8 * j + 3], of16),
                                                                    pack2(hi[8 * j + 4], hi[8 * j + 5], of16), pack2(hi[8 * j + 6], hi[8 * j + 7], of16));
        }
      }
      asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");           // both warps of the quarter have written the tile
      uint16_t* gout = static_cast<uint16_t*>(g.out) + n0;
#pragma unroll
      for (int c = t64; c < 320; c += 64) {
        const int r = c / 10, ch = c - r * 10;
        if (row0 + r < g.M)
          *reinterpret_cast<uint4*>(gout + (int64_t)(row0 + r) * g.ldo + ch * 8) = *reinterpret_cast<const uint4*>(tileS + r * kQkvTilePitch + ch * 8);
      }
      asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");           // tile free for the next head
    }
  }
}

// cta_group::2 helpers (CTA pair = cluster of 2 along M; the even CTA is the MMA leader)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load into this CTA's smem, completing on the LEADER CTA's mbarrier (peer bit of the address cleared)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread are done) on the same barrier in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar, uint32_t cta) {      // arrive on CTA `cta`'s copy of `bar`
  asm volatile(
      "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// CG = 1: one CTA per 128 x BN tile.  CG = 2: a CTA pair (cluster of 2) per 256 x BN tile with tcgen05 cta_group::2:
// each CTA stages its own 128 A rows and HALF of the B rows (BN/2), the leader issues one M=256 MMA that reads both
// CTAs' shared memory and writes both CTAs' TMEM, so per-CTA L2->smem traffic drops by a third (A 16 KB + B 16 KB
// instead of A 16 KB + B 32 KB per k-block) and the smem ring is six stages deep instead of four.
template <int BN, int EPI, int CG>
__global__ void __launch_bounds__(kThreads, 1) gemm_tc(const __grid_constant__ CUtensorMap tma_a,
                                                       const __grid_constant__ CUtensorMap tma_b, const GemmArgs g) {
  using C = Cfg<BN, CG, EPI>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::kStages;
  uint64_t* tfull = bars + 2 * C::kStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0;
  const bool leader = rank == 0;
  const int n_blocks = g.N / BN;
  const int m_blocks = (g.M + BM * CG - 1) / (BM * CG);
  const int num_tiles = m_blocks * n_blocks;
  const int k_blocks = (g.K + BK - 1) / BK;
  const int first_tile = blockIdx.x / CG, tile_step = gridDim.x / CG;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_b);
    for (int s = 0; s < C::kStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull + a, 1); mbar_init(tempty + a, 8 * CG); }
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (CG == 2) tmem_alloc_pair(tmem_slot, kTmemCols);
    else { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch: everything above overlapped the previous kernel's tail.  The producer goes one step
  // further: B is the weight matrix, which no predecessor writes, so the weight tiles of the first ring pass are
  // requested BEFORE the dependency wait (small batches leave SMs idle in the predecessor: the cold weight fetch from
  // HBM then runs under its tail); A (activations) and every other role wait first.
  if (warp != 0) pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      bool first_pass = first_tile < num_tiles;
      if (first_pass) {
        const int n_row = (first_tile % n_blocks) * BN + (int)rank * C::kBRows;
        const int pre = k_blocks < C::kStages ? k_blocks : C::kStages;
        for (int kb = 0; kb < pre; ++kb) {                    // the ring is empty: no wait on `empty`
          uint8_t* sa = smem + kb * C::kStageBytes;
          if constexpr (CG == 2) {
            if (leader) mbar_arrive_expect_tx(full + kb, 2 * C::kStageBytes);
            tma_load_2d_pair(sa + C::kABytes, &tma_b, full + kb, kb * BK, n_row);
          } else {
            mbar_arrive_expect_tx(full + kb, C::kStageBytes);
            tma_load_2d(sa + C::kABytes, &tma_b, full + kb, kb * BK, n_row);
          }
        }
      }
      pdl_wait();                          // the predecessor's outputs (A, and what the epilogue reads) are complete now
      for (int tile = first_tile; tile < num_tiles; tile += tile_step) {
        const int m_row = (tile / n_blocks) * BM * CG + (int)rank * BM;
        const int n_row = (tile % n_blocks) * BN + (int)rank * C::kBRows;
        for (int kb = 0; kb < k_blocks; ++kb) {
          uint8_t* sa = smem + stage * C::kStageBytes;
          const bool b_requested = first_pass && kb < C::kStages;           // first tile, first ring pass: B is already on its way
          if (!b_requested) mbar_wait(empty + stage, phase ^ 1);
          if constexpr (CG == 2) {
            if (!b_requested && leader) mbar_arrive_expect_tx(full + stage, 2 * C::kStageBytes);     // both CTAs' bytes land on the leader
            tma_load_2d_pair(sa, &tma_a, full + stage, kb * BK, m_row);
            if (!b_requested) tma_load_2d_pair(sa + C::kABytes, &tma_b, full + stage, kb * BK, n_row);
          } else {
            if (!b_requested) mbar_arrive_expect_tx(full + stage, C::kStageBytes);
            tma_load_2d(sa, &tma_a, full + stage, kb * BK, m_row);
            if (!b_requested) tma_load_2d(sa + C::kABytes, &tma_b, full + stage, kb * BK, n_row);
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        first_pass = false;
      }
      pdl_trigger();                      // this CTA has requested its last operands: the next kernel may be scheduled
    }
  } else if (warp == 1) {
    if (leader && elect_one()) {
      const uint32_t idesc = umma_idesc_16bit(BM * CG, BN, g.op_f16 != 0);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(tempty + acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * 256;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(full + stage, phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint64_t da = umma_desc_k128(sa), db = umma_desc_k128(sa + C::kABytes);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {                                   // +32 B per K step, in 16 B units
            if constexpr (CG == 2) umma_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            else umma_bf16(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          if constexpr (CG == 2) umma_commit_pair(empty + stage); else umma_commit(empty + stage);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        if constexpr (CG == 2) umma_commit_pair(tfull + acc); else umma_commit(tfull + acc);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3, half = (warp - 4) >> 2;
    float* xpose = reinterpret_cast<float*>(smem + C::kStages * C::kStageBytes + C::kBarBytes) +
                   ((is_resid(EPI) || EPI == EPI_SCATTER) ? (warp - 4) * (kXposeBytesPerWarp / 4) : 0);   // per-warp area; QKV: the CTA's area
    int it = 0;
    for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++it) {
      const int m_blk = (tile / n_blocks) * CG + (int)rank, n_blk = tile % n_blocks;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(q * 32) << 16);
      epilogue_tile<BN, EPI>(taddr, m_blk, n_blk, q * 32 + lane, half, g, xpose, [&] {
        mbar_wait(tfull + acc, acc_phase);
        tc_fence_after();
      });
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) mbar_arrive_cta(tempty + acc, 0); else mbar_arrive(tempty + acc);
      }
    }
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_pair(tmem_base, kTmemCols); else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace
int make_tmap_2d(void* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                 int swizzle_bytes, bool f16);
namespace {

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_tmap(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f16) {
  return make_tmap_2d(tm, base, rows, cols, ld, BK, box_rows, 128, f16);
}

template <int BN, int EPI, int CG>
int launch(const GemmArgs& g, const void* a, int64_t lda, const void* b, int64_t ldb, cudaStream_t stream) {
  using C = Cfg<BN, CG, EPI>;
  if (g.N % BN) return fail(ZV_EINVAL, "gemm: N=%d is not a multiple of the %d-wide tile", g.N, BN);
  CUtensorMap ta, tb;
  int rc = make_tmap(&ta, a, g.M, g.K, lda, BM, g.op_f16 != 0);
  if (rc) return rc;
  rc = make_tmap(&tb, b, g.N, g.K, ldb, C::kBRows, g.op_f16 != 0);
  if (rc) return rc;
  static std::atomic<uint64_t> attr_set{0};
  const int dev = current_device();
  if (device_needs_setup(attr_set, dev)) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc<BN, EPI, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) return fail(ZV_ECUDA, "gemm: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    mark_device(attr_set, dev);
  }
  const int tiles = ((g.M + BM * CG - 1) / (BM * CG)) * (g.N / BN);
  const int slots = num_sms() / CG;
  const int grid = (tiles < slots ? tiles : slots) * CG;
  cudaError_t e;
  {
    static const char* const kNames[] = {"zv:K2 gemm store", "zv:K2 gemm qkv+rope", "zv:K2 gemm residual", "zv:K2 gemm swiglu",
                                         "zv:K2 gemm gelu", "zv:K2 gemm scatter", "zv:K2 gemm qkv+ln+rope",
                                         "zv:K2 gemm residual+ln", "zv:K2 gemm quickgelu"};
    NvtxRange nvtx(kNames[EPI]);
    KernelTimer timer(is_qkv(EPI) ? KC_GEMM_QKV : is_resid(EPI) ? KC_GEMM_RESID : EPI == EPI_QGELU ? KC_GEMM_QGELU : KC_GEMM_STORE + EPI, stream);
    e = launch_pdl(gemm_tc<BN, EPI, CG>, dim3((unsigned)grid), dim3(kThreads), C::kSmemBytes, stream, CG, ta, tb, g);
  }
  count_launch();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ZV_ECUDA, "gemm: launch: %s", cudaGetErrorString(e));
  return ZV_OK;
}

}  // namespace

// 2-D 16-bit tensor (rows, cols), row pitch `ld` elements; box = box_cols x box_rows; swizzle 128 or 32 bytes; OOB = 0.
int make_tmap_2d(void* tm_, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                 int swizzle_bytes, bool f16) {
  CUtensorMap* tm = static_cast<CUtensorMap*>(tm_);
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(ZV_ECUDA, "tma: cuTensorMapEncodeTiled is not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld * 2) % 16)
    return fail(ZV_EINVAL, "tma: operand base/pitch must be 16-byte aligned (base %p, ld %lld)", base, (long long)ld);
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base),
                  dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ZV_ECUDA, "tma: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return ZV_OK;
}

// 2-D uint8 tensor (dim1 rows of dim0 bytes, row pitch stride1 bytes, a multiple of 16), box0 x box1 box, 128-byte swizzle,
// OOB = 0.  K1's tensor-core route: an image seen as super-rows of four rows (zv_k1_tc.cuh).
int make_tmap_u8(void* tm_, const void* base, uint64_t dim0, uint64_t dim1, uint64_t stride1, int box0, int box1) {
  CUtensorMap* tm = static_cast<CUtensorMap*>(tm_);
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(ZV_ECUDA, "tma: cuTensorMapEncodeTiled is not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 15) || stride1 % 16 || dim0 == 0 || dim1 == 0)
    return fail(ZV_EINVAL, "tma: uint8 operand base/pitch must be 16-byte aligned (base %p, pitch %llu)", base, (unsigned long long)stride1);
  cuuint64_t dims[2] = {(cuuint64_t)dim0, (cuuint64_t)dim1};
  cuuint64_t strides[1] = {(cuuint64_t)stride1};
  cuuint32_t box[2] = {(cuuint32_t)box0, (cuuint32_t)box1};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ZV_ECUDA, "tma: cuTensorMapEncodeTiled (uint8) failed with CUresult %d", (int)r);
  return ZV_OK;
}

int gemm(int epi, const GemmArgs& g, const void* a, int64_t lda, const void* b, int64_t ldb, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return fail(ZV_EINVAL, "gemm: empty problem %dx%dx%d", g.M, g.N, g.K);
#ifdef ZV_DEBUG_GEMM_1CTA               // compile-time debug build: single-CTA kernels everywhere
  {
    switch (epi) {
      case EPI_STORE:
        return g.N % 256 == 0 ? launch<256, EPI_STORE, 1>(g, a, lda, b, ldb, stream)
                              : launch<128, EPI_STORE, 1>(g, a, lda, b, ldb, stream);
      case EPI_QKV_ROPE: return launch<240, EPI_QKV_ROPE, 1>(g, a, lda, b, ldb, stream);
      case EPI_RESID: return launch<256, EPI_RESID, 1>(g, a, lda, b, ldb, stream);
      case EPI_SWIGLU: return launch<256, EPI_SWIGLU, 1>(g, a, lda, b, ldb, stream);
      case EPI_GELU: return launch<256, EPI_GELU, 1>(g, a, lda, b, ldb, stream);
      case EPI_SCATTER: return launch<256, EPI_SCATTER, 1>(g, a, lda, b, ldb, stream);
      case EPI_QKV_ROPE_LN: return launch<240, EPI_QKV_ROPE_LN, 1>(g, a, lda, b, ldb, stream);
      case EPI_RESID_LN: return launch<256, EPI_RESID_LN, 1>(g, a, lda, b, ldb, stream);
      case EPI_QGELU: return launch<256, EPI_QGELU, 1>(g, a, lda, b, ldb, stream);
    }
  }
#endif
  switch (epi) {
    case EPI_STORE:
      return g.N % 256 == 0 ? launch<256, EPI_STORE, 2>(g, a, lda, b, ldb, stream)
                            : launch<128, EPI_STORE, 1>(g, a, lda, b, ldb, stream);
    case EPI_QKV_ROPE: return launch<240, EPI_QKV_ROPE, 2>(g, a, lda, b, ldb, stream);
    case EPI_RESID:
    case EPI_RESID_LN: {
      // small batches (a single zoom crop: M = 1296): N = 1280 gives 5 column tiles of 256, i.e. 30 CTA pairs of work for
      // 74 pair slots.  128-wide tiles double the parallelism; taken when they cut the wave count x tile width by >= 20 %.
      const int64_t slots = num_sms() / 2, mp = (g.M + 2 * BM - 1) / (2 * BM);
      const int64_t cost256 = 2 * ((mp * (g.N / 256) + slots - 1) / slots), cost128 = (mp * (g.N / 128) + slots - 1) / slots;
      const bool wide = g.N % 256 == 0 && 5 * cost128 > 4 * cost256;
      if (epi == EPI_RESID_LN)
        return wide ? launch<256, EPI_RESID_LN, 2>(g, a, lda, b, ldb, stream) : launch<128, EPI_RESID_LN, 2>(g, a, lda, b, ldb, stream);
      if (wide) return launch<256, EPI_RESID, 2>(g, a, lda, b, ldb, stream);
      return launch<128, EPI_RESID, 2>(g, a, lda, b, ldb, stream);
    }
    case EPI_SWIGLU: return launch<256, EPI_SWIGLU, 2>(g, a, lda, b, ldb, stream);
    case EPI_GELU: return launch<256, EPI_GELU, 2>(g, a, lda, b, ldb, stream);
    case EPI_SCATTER: return launch<256, EPI_SCATTER, 2>(g, a, lda, b, ldb, stream);
    case EPI_QKV_ROPE_LN: return launch<240, EPI_QKV_ROPE_LN, 2>(g, a, lda, b, ldb, stream);
    case EPI_QGELU: return launch<256, EPI_QGELU, 2>(g, a, lda, b, ldb, stream);
  }
  return fail(ZV_EINVAL, "gemm: unknown epilogue %d", epi);
}

}  // namespace zv

extern "C" int zv_gemm_bf16(const void* a_dev, int64_t lda, const void* b_dev, int64_t ldb, const float* bias_dev,
                            void* c_dev, int64_t ldc, int32_t c_dtype, int64_t m, int64_t n, int64_t k, void* stream) {
  zv::reset_launch_count();
  if (!a_dev || !b_dev || !c_dev) return zv::fail(ZV_EINVAL, "zv_gemm_bf16: null pointer");
  if (n % 128) return zv::fail(ZV_EINVAL, "zv_gemm_bf16: N must be a multiple of 128");
  if (c_dtype != ZV_F32 && c_dtype != ZV_BF16) return zv::fail(ZV_EINVAL, "zv_gemm_bf16: bad c_dtype");
  zv::GemmArgs g{};
  g.M = (int)m; g.N = (int)n; g.K = (int)k;
  g.out = c_dev; g.ldo = ldc; g.out_dtype = c_dtype; g.bias = bias_dev;
  return zv::gemm(zv::EPI_STORE, g, a_dev, lda, b_dev, ldb, stream);
}

// Epilogue-selectable variant, exposed so unit tests can check every fused epilogue in isolation.
extern "C" int zv_gemm_ex(int32_t epilogue, const void* a_dev, int64_t lda, const void* b_dev, int64_t ldb,
                          const float* bias_dev, void* out_dev, int64_t ldo, int32_t out_dtype, int64_t m, int64_t n,
                          int64_t k, const int32_t* pos_dev, const float* rope_dev, const int32_t* scatter_dev,
                          int32_t heads, int32_t op_dtype, void* stream) {
  zv::reset_launch_count();
  if (!a_dev || !b_dev || !out_dev) return zv::fail(ZV_EINVAL, "zv_gemm_ex: null pointer");
  if (epilogue < zv::EPI_STORE || epilogue > zv::EPI_SCATTER) return zv::fail(ZV_EINVAL, "gemm: unknown epilogue %d", epilogue);
  zv::GemmArgs g{};
  g.M = (int)m; g.N = (int)n; g.K = (int)k;
  g.out = out_dev; g.ldo = ldo; g.out_dtype = out_dtype; g.bias = bias_dev;
  g.pos = pos_dev; g.rope = reinterpret_cast<const float2*>(rope_dev); g.scatter = scatter_dev; g.heads = heads;
  g.op_f16 = op_dtype == ZV_F16;
  if (epilogue != zv::EPI_STORE && !bias_dev) return zv::fail(ZV_EINVAL, "zv_gemm_ex: this epilogue needs a bias");
  if (epilogue == zv::EPI_QKV_ROPE && (!pos_dev || !rope_dev)) return zv::fail(ZV_EINVAL, "zv_gemm_ex: rope tables missing");
  if (epilogue == zv::EPI_SCATTER && !scatter_dev) return zv::fail(ZV_EINVAL, "zv_gemm_ex: scatter index missing");
  return zv::gemm(epilogue, g, a_dev, lda, b_dev, ldb, stream);
}
