// LM hand-off, device side: the multimodal rotary position index and the placeholder rows of zv_handoff.cpp as kernels
// on the caller's stream, with no host synchronisation, so that the whole hand-off can be captured in one CUDA graph with
// the tower (zv_visual_forward_into).  Bit-identical to zv_rope_index / zv_placeholder_rows for every input those accept;
// where the host function fails, the failure is recorded in a caller-owned device status word instead (int64 [4], see zoomvit.h).
//
//   rope index, images:  handoff_scan   one CTA per sample: compacts the admitted tokens (mask == 1) into a per-token
//                                       class byte, counts the sample's images, finds a video placeholder or a trailing
//                                       vision start
//                        handoff_fill   one CTA per sample: first grid row = images of the samples before it; walks the
//                                       sample's images in order (block-wide search for each placeholder run), writes the
//                                       positions in compacted order, then spreads them to their padded slots in place;
//                                       the last CTA to finish publishes the batch's first error
//   rope index, text:    handoff_text   one CTA per sample (no grid: cumsum of the mask, or an arange)
//   placeholder rows:    rows_count     one CTA per 8192 tokens: placeholders per tile
//                        rows_write     one CTA per tile: row indices in masked_scatter order, -1 in every slot at or
//                                       beyond the count
#include <climits>
#include <cstdint>

#include <cuda_runtime.h>

#include "zv_common.h"
#include "zv_gemm.h"
#include "zv_ptx.cuh"

namespace zv {
namespace {

constexpr int kThreads = 512;          // rope index kernels
constexpr int kRowsThreads = 256;      // placeholder rows kernels
constexpr int kRowsTile = 8192;        // tokens per placeholder-rows CTA
// class byte of a compacted token: bit flags, so that coinciding token ids behave as in the host code
constexpr uint8_t kImg = 1, kVstart = 2, kVid = 4;

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// Exclusive prefix of `flag` over the block in thread order, and the block's total.  Every thread must call it.
__device__ __forceinline__ int block_scan_flag(bool flag, int* warp_tot, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) warp_tot[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {
    int v = lane < nw ? warp_tot[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    if (lane < nw) warp_tot[lane] = v;
  }
  __syncthreads();
  const int before = (warp ? warp_tot[warp - 1] : 0) + __popc(bal & ((1u << lane) - 1u));
  *total = warp_tot[nw - 1];
  __syncthreads();
  return before;
}

__device__ __forceinline__ int64_t block_sum(int64_t v, unsigned long long* acc) {
  if (threadIdx.x == 0) *acc = 0;
  __syncthreads();
  if (v) atomicAdd(acc, (unsigned long long)v);
  __syncthreads();
  const int64_t r = (int64_t)*acc;
  __syncthreads();
  return r;
}

// Device state of one rope-index call (workspace layout in handoff_layout).
struct RopeArgs {
  const int64_t* ids;
  const int64_t* mask;        // may be null
  const int64_t* grid;        // [n_images][3]
  int64_t n_images;
  int64_t B, L;
  int64_t img, vid, vstart;
  int64_t merge;
  int hf5;
  int64_t* pos;               // [3][B][L]
  int64_t* delta;             // [B]
  int64_t* status;            // [4], caller's
  uint8_t* cls;               // [B][L] class bytes of the compacted tokens
  int32_t* n;                 // [B] admitted tokens
  int32_t* nimg;              // [B] images (vision start + image placeholder)
  int32_t* scan;              // [B] error found by handoff_scan (0 or ZV_HANDOFF_*)
  int64_t* payload;           // [B][2] details of a sample's error
  unsigned long long* key;    // (sample << 8) | check of the first error, ~0 when none
  unsigned int* done;         // CTAs finished in handoff_fill
};

__global__ void __launch_bounds__(kThreads) handoff_scan(RopeArgs a) {
  __shared__ int warp_tot[32];
  __shared__ unsigned long long acc;
  const int64_t b = blockIdx.x, L = a.L;
  ptx::pdl_wait();
  if (b == 0 && threadIdx.x == 0) {
    *a.key = ~0ull;
    *a.done = 0;
  }
  const int64_t* ids = a.ids + b * L;
  const int64_t* mask = a.mask ? a.mask + b * L : nullptr;
  uint8_t* cls = a.cls + b * L;
  int n = 0;
  for (int64_t l0 = 0; l0 < L; l0 += blockDim.x) {
    const int64_t l = l0 + threadIdx.x;
    const bool keep = l < L && (!mask || mask[l] == 1);
    int tot;
    const int i = n + block_scan_flag(keep, warp_tot, &tot);
    if (keep) {
      const int64_t v = ids[l];
      cls[i] = (v == a.img ? kImg : 0) | (v == a.vstart ? kVstart : 0) | (v == a.vid ? kVid : 0);
    }
    n += tot;
  }
  __syncthreads();
  // images = vision starts followed by an image placeholder (reference :1034-1037); a vision start followed by a video
  // placeholder fails, and so does a trailing one - the video error first, it can only sit before the last token
  int images = 0;
  bool video = false;
  for (int i = threadIdx.x; i + 1 < n; i += blockDim.x) {
    if (!(cls[i] & kVstart)) continue;
    if (cls[i + 1] & kImg) ++images;
    else if (cls[i + 1] & kVid) video = true;
  }
  images = (int)block_sum(images, &acc);
  video = __syncthreads_or(video);
  if (threadIdx.x == 0) {
    a.n[b] = n;
    a.nimg[b] = images;
    a.scan[b] = video ? ZV_HANDOFF_VIDEO : (n > 0 && (cls[n - 1] & kVstart)) ? ZV_HANDOFF_TRAILING_VSTART : 0;
  }
}

// Positions of sample b in compacted order (pos[d][b][i], i < n), then spread to the padded slots.  Returns the sample's
// error (uniform over the block) with its details in *pa, *pb.
__device__ int fill_sample(const RopeArgs& a, int64_t b, int64_t first_row, int* warp_tot, int* s_ed, int64_t* pa, int64_t* pb) {
  const int64_t B = a.B, L = a.L;
  const int64_t n = a.n[b];
  const int images = a.nimg[b];
  const uint8_t* cls = a.cls + b * L;
  int64_t* p0 = a.pos + b * L;
  int64_t* p1 = a.pos + (B + b) * L;
  int64_t* p2 = a.pos + (2 * B + b) * L;
  int64_t st = 0, lm1 = 0;                       // next text start; last_max + 1 = st_idx (reference :1070)
  for (int k = 0; k < images; ++k) {
    // ed = first image placeholder at or after st
    if (threadIdx.x == 0) *s_ed = INT_MAX;
    __syncthreads();
    int64_t ed = -1;
    for (int64_t i0 = st; i0 < n; i0 += blockDim.x) {
      const int64_t i = i0 + threadIdx.x;
      const bool hit = i < n && (cls[i] & kImg);
      if (hit) atomicMin(s_ed, (int)i);
      if (__syncthreads_or(hit)) {
        ed = *s_ed;
        break;
      }
    }
    __syncthreads();
    if (ed < 0) return ZV_HANDOFF_FEW_PLACEHOLDERS;
    const int64_t r = first_row + k;
    if (r >= a.n_images) {
      *pa = a.n_images;
      return ZV_HANDOFF_GRID_ROWS;
    }
    const int64_t t = a.grid[3 * r], gh = a.grid[3 * r + 1] / a.merge, gw = a.grid[3 * r + 2] / a.merge;
    if (t <= 0 || gh <= 0 || gw <= 0) {
      *pa = r;
      return ZV_HANDOFF_EMPTY_GRID;
    }
    const int64_t base = ed - st + lm1, hw = gh * gw, end = ed + t * hw;
    for (int64_t i = st + threadIdx.x; i < (end < n ? end : n); i += blockDim.x) {
      if (i < ed) {
        p0[i] = p1[i] = p2[i] = lm1 + (i - st);
      } else {
        const int64_t j = i - ed;
        p0[i] = base + j / hw;
        p1[i] = base + (j / gw) % gh;
        p2[i] = base + j % gw;
      }
    }
    lm1 = base + max(t, max(gh, gw));
    st = end;
  }
  if (st > n) {                                  // the placeholder runs overshoot the sample's tokens
    *pa = st;
    *pb = n;
    return ZV_HANDOFF_COUNT;
  }
  for (int64_t i = st + threadIdx.x; i < n; i += blockDim.x) p0[i] = p1[i] = p2[i] = lm1 + (i - st);
  lm1 += n - st;
  if (n == 0) return ZV_HANDOFF_MASKED;
  if (threadIdx.x == 0) a.delta[b] = lm1 - (a.hf5 ? n : L);   // max position + 1 - length
  if (!a.mask || n == L) return 0;
  // spread: token l with compacted index i takes pos[.][i]; pads take 1 (0 under hf5).  Tiles run from the end: a tile's
  // sources [c0, c0 + tot) lie below every slot a later tile wrote, and c0 <= the tile's first slot, so only the tile
  // itself can overlap its sources - they are read before the barrier, written after it
  __syncthreads();
  const int64_t pad = a.hf5 ? 0 : 1;
  const int64_t* mask = a.mask + b * L;
  int64_t above = 0;
  for (int64_t l0 = (L - 1) / blockDim.x * blockDim.x; l0 >= 0; l0 -= blockDim.x) {
    const int64_t l = l0 + threadIdx.x;
    const bool keep = l < L && mask[l] == 1;
    int tot;
    const int before = block_scan_flag(keep, warp_tot, &tot);
    const int64_t i = n - above - tot + before;
    int64_t v0 = pad, v1 = pad, v2 = pad;
    if (keep) { v0 = p0[i]; v1 = p1[i]; v2 = p2[i]; }
    __syncthreads();
    if (l < L) { p0[l] = v0; p1[l] = v1; p2[l] = v2; }
    above += tot;
  }
  return 0;
}

__global__ void __launch_bounds__(kThreads) handoff_fill(RopeArgs a) {
  __shared__ int warp_tot[32];
  __shared__ int s_ed;
  __shared__ unsigned long long acc;
  const int64_t b = blockIdx.x;
  ptx::pdl_wait();
  int64_t part = 0;                              // this sample's first grid row: the images of the samples before it
  for (int64_t s = threadIdx.x; s < b; s += blockDim.x) part += a.nimg[s];
  const int64_t first_row = block_sum(part, &acc);
  int64_t pa = 0, pb = 0;
  int err = a.scan[b];
  if (!err) err = fill_sample(a, b, first_row, warp_tot, &s_ed, &pa, &pb);
  if (threadIdx.x != 0) return;
  if (err) {
    a.payload[2 * b] = pa;
    a.payload[2 * b + 1] = pb;
    __threadfence();
    atomicMin(a.key, ((unsigned long long)b << 8) | (unsigned)err);
  }
  // the last CTA to finish publishes the lowest sample's error: the one the host loop meets first
  __threadfence();
  if (atomicAdd(a.done, 1u) != gridDim.x - 1) return;
  __threadfence();
  const unsigned long long key = atomicAdd(a.key, 0ull);
  int64_t* st = a.status;
  if (key == ~0ull) {
    st[0] = st[1] = st[2] = st[3] = 0;
  } else {
    const int64_t s = (int64_t)(key >> 8);
    st[0] = (int64_t)(key & 255);
    st[1] = s;
    st[2] = *(volatile int64_t*)(a.payload + 2 * s);
    st[3] = *(volatile int64_t*)(a.payload + 2 * s + 1);
  }
}

// Text-only branch (reference :1091-1112): cumsum(mask != 0) - 1 with pads set to 1, or an arange.  Never fails.
__global__ void __launch_bounds__(kThreads) handoff_text(RopeArgs a) {
  __shared__ int warp_tot[32];
  const int64_t b = blockIdx.x, B = a.B, L = a.L;
  ptx::pdl_wait();
  if (b == 0 && threadIdx.x < 4) a.status[threadIdx.x] = 0;
  const int64_t* mask = a.mask ? a.mask + b * L : nullptr;
  int64_t run = 0;
  for (int64_t l0 = 0; l0 < L; l0 += blockDim.x) {
    const int64_t l = l0 + threadIdx.x;
    int64_t v = l;
    if (mask) {
      const bool keep = l < L && mask[l] != 0;
      int tot;
      const int before = block_scan_flag(keep, warp_tot, &tot);
      v = keep ? run + before : 1;
      run += tot;
    }
    if (l < L) a.pos[b * L + l] = a.pos[(B + b) * L + l] = a.pos[(2 * B + b) * L + l] = v;
  }
  if (threadIdx.x == 0) {
    // max over the row: the last cumsum value, or the pads' 1
    const int64_t mx = run == L ? L - 1 : (run - 1 > 1 ? run - 1 : 1);
    a.delta[b] = mask ? mx + 1 - L : 0;
  }
}

__global__ void __launch_bounds__(kRowsThreads) rows_count(const int64_t* ids, int64_t n_tokens, int64_t img, int32_t* tile_cnt) {
  __shared__ unsigned long long acc;
  ptx::pdl_wait();
  const int64_t l0 = (int64_t)blockIdx.x * kRowsTile;
  const int64_t l1 = l0 + kRowsTile < n_tokens ? l0 + kRowsTile : n_tokens;
  int64_t c = 0;
  for (int64_t l = l0 + threadIdx.x; l < l1; l += blockDim.x) c += ids[l] == img;
  c = block_sum(c, &acc);
  if (threadIdx.x == 0) tile_cnt[blockIdx.x] = (int32_t)c;
}

__global__ void __launch_bounds__(kRowsThreads) rows_write(const int64_t* ids, int64_t n_tokens, int64_t img, const int32_t* tile_cnt,
                                                           int64_t* rows, int64_t cap, int64_t* status) {
  __shared__ int warp_tot[32];
  __shared__ unsigned long long acc;
  ptx::pdl_wait();
  const int64_t t = blockIdx.x, n_tiles = gridDim.x;
  int64_t before = 0, all = 0;
  for (int64_t s = threadIdx.x; s < n_tiles; s += blockDim.x) {
    all += tile_cnt[s];
    if (s < t) before += tile_cnt[s];
  }
  before = block_sum(before, &acc);
  all = block_sum(all, &acc);
  const int64_t l0 = t * kRowsTile;
  const int64_t l1 = l0 + kRowsTile < n_tokens ? l0 + kRowsTile : n_tokens;
  for (int64_t s0 = l0; s0 < l1; s0 += blockDim.x) {
    const int64_t l = s0 + threadIdx.x;
    const bool hit = l < l1 && ids[l] == img;
    int tot;
    const int64_t k = before + block_scan_flag(hit, warp_tot, &tot);
    if (hit && k < cap) rows[k] = l;
    before += tot;
  }
  // slots the placeholders do not reach: a negative row is dropped by the scatter (compose_rows_kernel)
  for (int64_t s = all + t * blockDim.x + threadIdx.x; s < cap; s += n_tiles * blockDim.x) rows[s] = -1;
  if (t == 0 && threadIdx.x == 0) {
    status[0] = all == cap ? 0 : ZV_HANDOFF_ROWS_COUNT;
    status[1] = 0;
    status[2] = all;
    status[3] = cap;
  }
}

// Workspace: the placeholder-rows tile counts first (zv_placeholder_rows_dev uses only those), then the rope index's
// state, so that both can run on one workspace for the same batch shape.
inline int64_t rows_tiles_bytes(int64_t n_tokens) { return align_up(4 * ((n_tokens + kRowsTile - 1) / kRowsTile), 256); }
struct HandoffLayout { int64_t cls = 0, n = 0, nimg = 0, scan = 0, payload = 0, key = 0, done = 0, bytes = 0; };
HandoffLayout handoff_layout(int64_t B, int64_t L) {
  HandoffLayout w;
  int64_t off = rows_tiles_bytes(B * L);
  auto take = [&](int64_t bytes) { const int64_t o = off; off = align_up(off + bytes, 256); return o; };
  w.cls = take(B * L);
  w.n = take(4 * B);
  w.nimg = take(4 * B);
  w.scan = take(4 * B);
  w.payload = take(16 * B);
  w.key = take(8);
  w.done = take(4);
  w.bytes = off;
  return w;
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

int launched(const char* who) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ZV_ECUDA, "%s: %s", who, cudaGetErrorString(e));
  return ZV_OK;
}

}  // namespace
}  // namespace zv

using namespace zv;

extern "C" {

int64_t zv_handoff_workspace_bytes(int32_t batch, int32_t seq_len) {
  if (batch <= 0 || seq_len <= 0) return fail(ZV_EINVAL, "zv_handoff_workspace_bytes: batch=%d, seq_len=%d (both must be > 0)", batch, seq_len);
  return handoff_layout(batch, seq_len).bytes;
}

int zv_rope_index_dev(const int64_t* input_ids, const int64_t* attention_mask, int32_t batch, int32_t seq_len,
                      const int64_t* image_grid_thw, int32_t n_images, int64_t image_token_id, int64_t video_token_id,
                      int64_t vision_start_token_id, int32_t merge, int32_t hf5_semantics, int64_t* position_ids,
                      int64_t* deltas, int64_t* status, void* workspace_dev, int64_t workspace_bytes, void* stream) {
  const char* who = "zv_rope_index_dev";
  reset_launch_count();
  if (!input_ids || !position_ids || !deltas || !status || !workspace_dev)
    return fail(ZV_EINVAL, "%s: null argument", who);
  if (batch <= 0 || seq_len <= 0 || merge <= 0)
    return fail(ZV_EINVAL, "%s: batch=%d, seq_len=%d, merge=%d (all must be > 0)", who, batch, seq_len, merge);
  if (image_grid_thw && n_images < 0) return fail(ZV_EINVAL, "%s: n_images=%d", who, n_images);
  const HandoffLayout W = handoff_layout(batch, seq_len);
  if (workspace_bytes < W.bytes)
    return fail(ZV_EINVAL, "%s: workspace %lld B < required %lld B (zv_handoff_workspace_bytes)", who, (long long)workspace_bytes,
                (long long)W.bytes);
  int rc = check_device(who);
  if (rc) return rc;
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  RopeArgs a{};
  a.ids = input_ids; a.mask = attention_mask; a.grid = image_grid_thw; a.n_images = n_images;
  a.B = batch; a.L = seq_len; a.img = image_token_id; a.vid = video_token_id; a.vstart = vision_start_token_id;
  a.merge = merge; a.hf5 = hf5_semantics != 0; a.pos = position_ids; a.delta = deltas; a.status = status;
  a.cls = ws + W.cls;
  a.n = reinterpret_cast<int32_t*>(ws + W.n);
  a.nimg = reinterpret_cast<int32_t*>(ws + W.nimg);
  a.scan = reinterpret_cast<int32_t*>(ws + W.scan);
  a.payload = reinterpret_cast<int64_t*>(ws + W.payload);
  a.key = reinterpret_cast<unsigned long long*>(ws + W.key);
  a.done = reinterpret_cast<unsigned int*>(ws + W.done);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!image_grid_thw) {
    launch_pdl(handoff_text, dim3((unsigned)batch), dim3(kThreads), 0, s, 1, a);
    count_launch();
  } else {
    launch_pdl(handoff_scan, dim3((unsigned)batch), dim3(kThreads), 0, s, 1, a);
    launch_pdl(handoff_fill, dim3((unsigned)batch), dim3(kThreads), 0, s, 1, a);
    count_launch(2);
  }
  return launched(who);
}

int zv_placeholder_rows_dev(const int64_t* input_ids, int64_t n_tokens, int64_t image_token_id, int64_t* rows_out,
                            int64_t rows_cap, int64_t* status, void* workspace_dev, int64_t workspace_bytes, void* stream) {
  const char* who = "zv_placeholder_rows_dev";
  reset_launch_count();
  if (!input_ids || !status || !workspace_dev || (rows_cap > 0 && !rows_out)) return fail(ZV_EINVAL, "%s: null argument", who);
  if (n_tokens <= 0 || rows_cap < 0)
    return fail(ZV_EINVAL, "%s: n_tokens=%lld, rows_cap=%lld", who, (long long)n_tokens, (long long)rows_cap);
  const int64_t n_tiles = (n_tokens + kRowsTile - 1) / kRowsTile, need = rows_tiles_bytes(n_tokens);
  if (workspace_bytes < need)
    return fail(ZV_EINVAL, "%s: workspace %lld B < required %lld B (zv_handoff_workspace_bytes)", who, (long long)workspace_bytes,
                (long long)need);
  int rc = check_device(who);
  if (rc) return rc;
  int32_t* tiles = static_cast<int32_t*>(workspace_dev);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  launch_pdl(rows_count, dim3((unsigned)n_tiles), dim3(kRowsThreads), 0, s, 1, input_ids, n_tokens, image_token_id, tiles);
  launch_pdl(rows_write, dim3((unsigned)n_tiles), dim3(kRowsThreads), 0, s, 1, input_ids, n_tokens, image_token_id,
             (const int32_t*)tiles, rows_out, rows_cap, status);
  count_launch(2);
  return launched(who);
}

}  // extern "C"
