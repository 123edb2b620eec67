// Shared internals of libzoomvit (not part of the C ABI).
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <vector>

#include "zoomvit.h"

struct zv_plan;
namespace zv {

int fail(int code, const char* fmt, ...);   // records the thread-local message, returns code
void count_launch(int64_t n = 1);
void reset_launch_count();

// Per-device one-time setup (cudaFuncSetAttribute is a per-device property): `mask` holds one bit per device ordinal.
// Returns true when the current device has not been marked yet; the caller does its setup and then calls mark_device.
// Two threads may both see "not yet" and both run the (idempotent) setup - harmless.
int current_device();
inline bool device_needs_setup(const std::atomic<uint64_t>& mask, int dev) {
  return (mask.load(std::memory_order_acquire) & (1ull << (dev & 63))) == 0;
}
inline void mark_device(std::atomic<uint64_t>& mask, int dev) { mask.fetch_or(1ull << (dev & 63), std::memory_order_release); }
int num_sms();                              // SM count of the current device (cached per device ordinal)

// NVTX range around one stage of the path (nvtx3 is header-only; a no-op unless a profiler is attached)
class NvtxRange {
 public:
  explicit NvtxRange(const char* name);
  ~NvtxRange();
};

// Kernel classes for the optional event timing (zv_timing_*): one id per kernel template.
enum KernelClass { KC_K1_HPASS = 0, KC_K1_VPASS = 1, KC_GEMM_STORE = 2, KC_GEMM_QKV = 3, KC_GEMM_RESID = 4,
                   KC_GEMM_SWIGLU = 5, KC_GEMM_GELU = 6, KC_GEMM_SCATTER = 7, KC_ATTN_WINDOW = 8, KC_ATTN_FULL = 9,
                   KC_RMSNORM = 10, KC_GATHER = 11, KC_GEMM_QGELU = 12, KC_COUNT = 13 };
// RAII: records an event pair around the launches issued in its scope when timing is enabled.
class KernelTimer {
 public:
  KernelTimer(int cls, void* stream);
  ~KernelTimer();
 private:
  void* stream_;
  int idx_;
};

// ---- host-side math shared by geometry / preprocess / plan
struct AxisCoeffs {
  int32_t in_size = 0, out_size = 0, ksize = 0;
  std::vector<int32_t> bounds;   // [out][2]
  std::vector<int32_t> kk;       // [out][ksize], 22-bit fixed point
  int32_t precision = 22;        // bits of the taps before they were moved to 22 bits (ZV_RESAMPLE_TORCHVISION: p)
};
int32_t resample_ksize(int32_t in_size, int32_t out_size);
int check_resample_kind(int32_t kind, const char* who);   // ZV_OK, or ZV_EINVAL with a message
void resample_coeffs(int32_t kind, int32_t in_size, int32_t out_size, AxisCoeffs* out);
void normalize_lut(const zv_cfg* cfg, float* lut768);      // in the arithmetic of cfg->resample_kind
void plan_device_image(const zv_plan* p, std::vector<uint8_t>* image);
void build_window_blocks(const std::vector<int32_t>& cu, int32_t max_rows, std::vector<int32_t>* blocks);
void fill_window_bounds(const std::vector<int32_t>& cu, int32_t* bounds);

// ---- plan (host tables; device image produced by zv_plan_upload)
struct PlanDeviceLayout {
  int64_t off_pos = 0;                     // int32 [S][2]: (h, w) rotary ids, window order
  int64_t off_rope = 0;                    // float [max_pos][20][2]: (cos, sin) of pos * inv_freq[j]
  int64_t off_widx = 0;                    // int32 [T]: window position i <-> HF merge-group index
  int64_t off_win_tiles = 0, off_full_tiles = 0;  // int4 work items (q0, q_len, seg_begin, seg_end)
  int64_t off_win_blocks = 0;              // int4 (row0, n_rows, 0, 0): row blocks of whole windows, <= 128 rows (window layers)
  int64_t off_win_bounds = 0;              // int32 [S][2]: (first row, end row) of the window of every patch row
  int32_t max_pos = 0;
  int64_t bytes = 0;
};

}  // namespace zv

struct zv_plan {
  zv_cfg cfg;
  int32_t n_images = 0;
  int64_t S = 0, T = 0;
  std::vector<int64_t> grid_thw;
  std::vector<int64_t> window_index, reverse_index;
  std::vector<int32_t> cu_window_raw, cu_window, cu_full;
  std::vector<int32_t> pos_ids;            // [S][2], HF order
  std::vector<int32_t> win_tiles, full_tiles;   // 4 ints per q tile
  std::vector<int32_t> win_blocks;              // 4 ints per row block of the tcgen05 window kernel
  int32_t n_win_tiles = 0, n_full_tiles = 0, n_win_blocks = 0;
  zv::PlanDeviceLayout dev;
};
