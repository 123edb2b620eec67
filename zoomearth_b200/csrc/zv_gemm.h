// Internal interface of the tcgen05 GEMM (zv_gemm.cu) and the other tower kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include <utility>

namespace zv {

// Launch with the programmatic-dependent-launch attribute (see zv_ptx.cuh pdl_wait / pdl_trigger); `cluster` > 1 adds a
// cluster dimension.  Kernels launched this way MUST call pdl_wait() before touching predecessor-written global memory.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, int cluster,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
#ifndef ZV_NO_PDL
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
#endif
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = (unsigned)n;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

enum GemmEpilogue { EPI_STORE = 0, EPI_QKV_ROPE = 1, EPI_RESID = 2, EPI_SWIGLU = 3, EPI_GELU = 4, EPI_SCATTER = 5,
                   // LayerNorm folded into the GEMMs around it (Qwen2-VL tower): separate values so that the
                   // instantiations above stay exactly as they are
                   EPI_QKV_ROPE_LN = 6,   // EPI_QKV_ROPE with r * (acc - mu * c_n) + b'_n before the rotary
                   EPI_RESID_LN = 7,      // EPI_RESID emitting per-slot (mean, M2) instead of sums of squares
                   EPI_QGELU = 8 };       // quick_gelu(r * (acc - mu * c_n) + b'_n) -> 16-bit (fc1)

struct GemmArgs {
  int M, N, K;
  int out_dtype;            // ZV_F32 / ZV_BF16 / ZV_F16 element type of `out` (EPI_RESID is always fp32)
  int op_f16;               // operands A, B are fp16 (else bf16)
  void* out;
  int64_t ldo;              // output row pitch in elements
  const float* bias;        // [N] (EPI_SWIGLU: packed like the weight rows); may be null for EPI_STORE
  const int32_t* pos;       // EPI_QKV_ROPE: [M][2] (h, w)
  const float2* rope;       // EPI_QKV_ROPE: [max_pos][20] (cos, sin)
  const int32_t* scatter;   // EPI_SCATTER: [M] output row of accumulator row i
  int heads;                // EPI_QKV_ROPE
  // EPI_SCATTER fused with the embedding gather: besides `out`, row i is also stored at row (peer_row_off +
  // scatter[i]) of every peer buffer (peer-mapped device pointers of the other ranks, written over NVLink)
  void* peers[8];
  int n_peers;
  int64_t peer_row_off;
  // RMSNorm folded into the GEMMs around it (the norm gain is folded into the consumer's weight columns at pack time):
  //   producer (EPI_RESID, N = hidden): besides X += ..., writes the new rows once more as 16-bit operands to `x16_out`
  //     (row pitch N) and, per row, partial sums of squares to `ss_out` [M][kSsParts] (slot = first column / 64 of each tile half);
  //   consumer (EPI_QKV_ROPE, EPI_SWIGLU): `row_ss` [M][kSsParts] of its A rows -> every accumulator row is scaled by
  //     rsqrt(sum / norm_dim + norm_eps) before the bias is added:  (x / rms) W'^T = (x W'^T) / rms.
  void* x16_out;
  float* ss_out;
  const float* row_ss;
  float norm_eps;
  int norm_dim;
  // LayerNorm folded the same way (EPI_*_LN, EPI_QGELU), with LN(x) W^T + b = r (x W'^T) - r mu c + b', r = rsqrt(var + eps):
  //   producer (EPI_RESID_LN): per row and 64-column slot the slot's (mean, M2 = sum of squared deviations) to `ln_out`
  //     [M][kSsParts] - a 128-column tile half writes its (mean, M2 / 2) into both of its slots, which merge back exactly;
  //   consumer: `row_ln` [M][kSsParts] merged in slot order (Chan's formula) into the row's mean and variance, and
  //     `colsum` [N] c_n = sum_k W'[n][k] of the 16-bit weights the MMA multiplies; `bias` is b' = b + W beta.
  float2* ln_out;
  const float2* row_ln;
  const float* colsum;
};
constexpr int kSsParts = 20;   // hidden 1280 = 20 x 64 columns (a 256-wide residual tile fills every other one, a 128-wide tile all)

// C = A[M,K] * B[N,K]^T with the chosen epilogue, enqueued on `stream`.
int gemm(int epi, const GemmArgs& g, const void* a, int64_t lda, const void* b, int64_t ldb, void* stream);

// cuTensorMapEncodeTiled wrapper (tm points at a CUtensorMap): 16-bit 2-D tensor, box_cols x box_rows box.
int make_tmap_2d(void* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                 int swizzle_bytes, bool f16);
// 2-D uint8 tensor map (dim1 rows of dim0 bytes, row pitch stride1 bytes), 128-byte swizzle, OOB = 0 (zv_gemm.cu).
int make_tmap_u8(void* tm, const void* base, uint64_t dim0, uint64_t dim1, uint64_t stride1, int box0, int box1);
// tcgen05 flash attention for long segments (zv_attn_tc.cu): qkv (S, 3*H) 16-bit with rotary applied; tiles
// (q0, q_len, seg_begin, seg_end) with q_len <= 128.
int attention_tc(const void* qkv, void* out, int64_t S, int heads, int head_dim, const int32_t* tiles_dev, int n_tiles,
                 void* stream, bool f16);

// tcgen05 window attention (zv_attn_win_tc.cu): row blocks (row0, n_rows, -, -) of whole windows (<= 128 rows) and the
// per-row window bounds table int32 [S][2]
int attention_win_tc(const void* qkv, void* out, int64_t S, int heads, int head_dim, const int32_t* blocks_dev, int n_blocks,
                     const int32_t* bounds_dev, void* stream, bool f16);

// fp32 (S, H) -> 16-bit copy (S, H) + per-row sum of squares in ss[row][0] (ss[row][1..kSsParts) = 0): the producer side
// of the folded RMSNorm for rows that no residual GEMM has written yet (the patch-embed output)
int cast_rows_ss(const float* x, void* x16, int x16_f16, float* ss, int64_t rows, int hidden, void* stream);
// fp32 (S, H) -> bf16 (S, H): y = w * (x * rsqrt(mean(x^2) + eps))   (HF Qwen2_5_VLRMSNorm :66-71)
int rmsnorm(const float* x, const float* w, void* y, int y_f16, int64_t rows, int hidden, float eps, void* stream);
// fp32 (S, H) -> 16-bit copy (S, H) + per-row, per-64-column-slot (mean, M2) in ln[row][kSsParts]: the producer side of the
// folded LayerNorm for the patch-embed output (two-pass per slot)
int cast_rows_ln(const float* x, void* x16, int x16_f16, float2* ln, int64_t rows, int hidden, void* stream);
// fp32 (S, H) -> 16-bit (S, H): y = (x - mean) * rsqrt(var + eps) * w + b, two-pass fp32 statistics (torch LayerNorm)
int layernorm(const float* x, const float* w, const float* b, void* y, int y_f16, int64_t rows, int hidden, float eps,
              void* stream);
// patches in HF order (f32 or bf16) -> bf16 in window order (groups of `unit` rows move together)
int gather_rows(const void* src, int src_dtype, void* dst, int dst_f16, const int32_t* widx, int64_t n_groups, int unit,
                int cols, void* stream);

}  // namespace zv
