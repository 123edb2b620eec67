// K1, video frames: the finished uint8 frames U (oh, ow, 3) of one video -> LUT normalise -> patchify with a temporal patch
// of two DIFFERENT frames -> patch rows at their HF / window-order position.  The video counterpart of k1_patchify_u8, whose
// temporal patch repeats one image.  Included by zv_k1.cu (kPatchElems, window_pos, store_pair).
//
// HF Qwen2VLVideoProcessor._preprocess: frames (T, C, H, W) -> pad T to a multiple of 2 by repeating the last frame ->
// view (grid_t, 2, C, gh/2, 2, 14, gw/2, 2, 14) -> permute (grid_t, gh/2, gw/2, 2, 2, C, 2, 14, 14).  So patch row
// tt gh gw + 4 (my lw + mx) + 2 mh + mw holds, at column c 392 + tp 196 + py 14 + px, pixel (my 28 + mh 14 + py,
// mx 28 + mw 14 + px) of channel c of frame min(2 tt + tp, T - 1).  Window order permutes the merge groups inside each
// frame group (HF get_window_index windows every temporal slice separately): row tt gh gw + 4 window_pos(my, mx).
struct VJob {
  const uint8_t* u;        // frame 0's U; frame f at u + f frame_bytes, row pitch 3 ow
  int64_t frame_bytes;
  int64_t out_row0;        // first patch row of this video
  int32_t lh, lw;          // merge-group grid of one frame group
  int32_t frames;          // T (>= 1)
  int32_t blk0;            // first work unit: units are (frame group, merge group), frame-group major
};

template <typename OutT>
__global__ void __launch_bounds__(256) k1_patchify_video(const VJob* __restrict__ jobs, int n_jobs, int n_groups,
                                                         const float* __restrict__ lut, OutT* __restrict__ out, int row_order,
                                                         int wsz) {
  // persistent like k1_patchify_u8: thread = (row yl of 28, 12-byte segment sg of 7), reading the same 12 bytes of the
  // group's two frames; two staging buffers, one barrier per group
  __shared__ __align__(16) OutT stage[2][4 * kPatchElems];
  __shared__ float s_lut[768];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = lut[i];          // uploaded by a memcpy, not by a kernel
  const int tid = threadIdx.x;
  const bool active = tid < 196;
  const int yl = tid / 7, sg = tid - yl * 7;
  const int roff = (yl / 14) * 2 * kPatchElems + (yl % 14) * 14;
  const int x0 = 4 * sg, x1 = 4 * sg + 2;
  const int e0 = roff + (x0 / 14) * kPatchElems + (x0 % 14), e1 = roff + (x1 / 14) * kPatchElems + (x1 % 14);
  zv::ptx::pdl_wait();                                   // U is the resample kernels' output
  __syncthreads();
  int jn = 0, buf = 0;
  for (int g = blockIdx.x; g < n_groups; g += gridDim.x, buf ^= 1) {
    while (jn + 1 < n_jobs && __ldg(&jobs[jn + 1].blk0) <= g) ++jn;                // groups ascend: the job index only moves forward
    const VJob& j = jobs[jn];
    const int lw = j.lw, per = j.lh * lw;
    const int gl = g - j.blk0, tt = gl / per, gi = gl - tt * per;
    const int my = gi / lw, mx = gi - my * lw;
    OutT* st = stage[buf];
    if (active) {
      const int64_t off = (int64_t)(my * 28 + yl) * (3 * 28 * lw) + mx * 84 + 12 * sg;
#pragma unroll
      for (int tp = 0; tp < 2; ++tp) {
        const int f = min(2 * tt + tp, j.frames - 1);                              // odd T: the last frame again
        const uint32_t* __restrict__ u = reinterpret_cast<const uint32_t*>(j.u + (int64_t)f * j.frame_bytes + off);
        const uint32_t w0 = u[0], w1 = u[1], w2 = u[2];  // R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3
        const int t0 = tp * 196;
        store_pair(st, e0 + t0, s_lut[w0 & 255], s_lut[w0 >> 24]);
        store_pair(st, e1 + t0, s_lut[(w1 >> 16) & 255], s_lut[(w2 >> 8) & 255]);
        store_pair(st, e0 + t0 + 392, s_lut[256 + ((w0 >> 8) & 255)], s_lut[256 + (w1 & 255)]);
        store_pair(st, e1 + t0 + 392, s_lut[256 + (w1 >> 24)], s_lut[256 + ((w2 >> 16) & 255)]);
        store_pair(st, e0 + t0 + 784, s_lut[512 + ((w0 >> 16) & 255)], s_lut[512 + ((w1 >> 8) & 255)]);
        store_pair(st, e1 + t0 + 784, s_lut[512 + (w2 & 255)], s_lut[512 + (w2 >> 24)]);
      }
    }
    __syncthreads();                                     // the group is staged (the other buffer's copy-out is two groups old)
    const int pos = tt * per + (row_order == ZV_ORDER_WINDOW ? window_pos(my, mx, j.lh, lw, wsz) : gi);
    uint4* dst = reinterpret_cast<uint4*>(out + (j.out_row0 + 4 * (int64_t)pos) * kPatchElems);
    const uint4* srcv = reinterpret_cast<const uint4*>(st);
    constexpr int kVec = 4 * kPatchElems * (int)sizeof(OutT) / 16;
    for (int i = tid; i < kVec; i += 256) dst[i] = srcv[i];
  }
}
