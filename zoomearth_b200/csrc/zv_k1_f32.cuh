// K1, ZV_RESAMPLE_TORCHVISION_CUDA: torch's fp32 antialiased bicubic as a CUDA device runs it (what HF's torchvision
// image processor does with device="cuda": uint8 -> fp32, interpolate(bicubic, antialias=True), clamp, round half to
// even, uint8), written as the finished uint8 image U (oh, ow, 3) that k1_patchify_u8 turns into patches.  Included by
// zv_k1.cu (K1Crop, find_slot).
//
// torch's kernel (aten upsample_gen2d_aa_out_frame<float, float, BicubicFilterFunctor>) gives every output its own
// horizontal results: h(y) = src[y][xmin] w0, then h(y) += src[y][xmin + j] w_j in increasing j, one FFMA each, for every
// row y of the output's vertical window, then the same chain down h(ymin .. ymin + ysize) with the y weights.  h(y)
// depends on (y, output column, channel) and not on the output row, so here a CTA owns a tile of output rows x columns,
// computes each h(y) its rows need ONCE into shared memory, and runs every output's vertical chain from there, still in
// increasing y: the same operations in the same order, so the same bits.  Input rows stream through in chunks, so any
// window height works (a downscale of 100x has hundreds of taps per axis).  The weights are torch's, computed on the host
// (zv_host.cpp resample_coeffs_f32) and read as fp32 from the tap slots of the coefficient tables.
constexpr int kF32Cols = 32;                            // output columns per tile
constexpr int kF32Rows = 32;                            // output rows per tile
constexpr int kF32Q = 3 * kF32Cols;                     // (column, channel) lanes of a tile
constexpr int kF32Threads = 384;
constexpr int kF32Groups = kF32Threads / kF32Q;         // row groups: thread = (lane, group)
constexpr int kF32Acc = kF32Rows / kF32Groups;          // vertical chains per thread
constexpr int kF32Chunk = 64;                           // input rows of horizontal results staged at a time

inline int64_t f32_tiles(int32_t oh, int32_t ow) {
  return (int64_t)((oh + kF32Rows - 1) / kF32Rows) * ((ow + kF32Cols - 1) / kF32Cols);
}

// One block = one tile of one crop (blk0: the crops' first tiles).  U = crop.dst, row pitch crop.dst_pitch.
__global__ void __launch_bounds__(kF32Threads, 2) k1_resample_f32(const K1Crop* __restrict__ crops, const int32_t* __restrict__ blk0,
                                                               int n, const int32_t* __restrict__ coef) {
  __shared__ float hbuf[kF32Chunk][kF32Q];
  zv::ptx::pdl_wait();
  const int slot = find_slot(blk0, n, blockIdx.x);
  const K1Crop& c = crops[slot];
  const int tiles_x = (c.ow + kF32Cols - 1) / kF32Cols, tile = blockIdx.x - blk0[slot];
  const int yy0 = (tile / tiles_x) * kF32Rows, xx0 = (tile - (tile / tiles_x) * tiles_x) * kF32Cols;
  const int nrow = min(kF32Rows, c.oh - yy0);
  const int q = threadIdx.x % kF32Q, g = threadIdx.x / kF32Q;
  const int xx = xx0 + q / 3, ch = q % 3;
  const bool col_ok = xx < c.ow;
  const float* __restrict__ wf = reinterpret_cast<const float*>(coef);
  const int32_t* __restrict__ bv = coef + c.off_bv;
  int hx0 = 0, hn = 0;
  const float* __restrict__ wh = wf;
  if (col_ok) {
    hx0 = __ldg(coef + c.off_bh + 2 * xx);
    hn = __ldg(coef + c.off_bh + 2 * xx + 1);
    wh = wf + c.off_kh + (int64_t)xx * c.ksh;
  }
  // the tile's input rows: from the first row's window start to the last row's window end (window starts ascend)
  const int y_lo = __ldg(bv + 2 * yy0), y_hi = __ldg(bv + 2 * (yy0 + nrow - 1)) + __ldg(bv + 2 * (yy0 + nrow - 1) + 1);
  float acc[kF32Acc];
#pragma unroll
  for (int k = 0; k < kF32Acc; ++k) acc[k] = 0.0f;

  for (int r0 = y_lo; r0 < y_hi; r0 += kF32Chunk) {
    const int nr = min(kF32Chunk, y_hi - r0);
    if (col_ok) {
      for (int r = g; r < nr; r += kF32Groups) {
        const int y_img = c.y0 + r0 + r;
        float h = 0.0f;                                 // a row outside the image is zeros (Image.crop)
        if (y_img >= 0 && y_img < c.src_h) {
          const uint8_t* __restrict__ row = c.src + (int64_t)y_img * c.pitch + ch;
          int x_img = c.x0 + hx0;
          h = __fmul_rn(x_img >= 0 && x_img < c.src_w ? (float)__ldg(row + 3 * (int64_t)x_img) : 0.0f, __ldg(wh));
          for (int t = 1; t < hn; ++t) {
            ++x_img;
            const float v = x_img >= 0 && x_img < c.src_w ? (float)__ldg(row + 3 * (int64_t)x_img) : 0.0f;
            h = __fmaf_rn(v, __ldg(wh + t), h);
          }
        }
        hbuf[r][q] = h;
      }
    }
    __syncthreads();
    if (col_ok) {
#pragma unroll
      for (int k = 0; k < kF32Acc; ++k) {
        const int yy = yy0 + g + kF32Groups * k;
        if (yy < yy0 + nrow) {
          const int ymin = __ldg(bv + 2 * yy), y_end = ymin + __ldg(bv + 2 * yy + 1);
          const float* __restrict__ wv = wf + c.off_kv + (int64_t)yy * c.ksv - ymin;
          float a = acc[k];
          for (int y = max(ymin, r0); y < min(y_end, r0 + nr); ++y) {
            const float t = hbuf[y - r0][q], w = __ldg(wv + y);
            a = y == ymin ? __fmul_rn(t, w) : __fmaf_rn(t, w, a);
          }
          acc[k] = a;
        }
      }
    }
    __syncthreads();                                    // the next chunk overwrites hbuf
  }
  if (col_ok) {
#pragma unroll
    for (int k = 0; k < kF32Acc; ++k) {
      const int yy = yy0 + g + kF32Groups * k;
      if (yy < yy0 + nrow)                              // clamp_(0, 255), round_() (half to even), uint8
        c.dst[(int64_t)yy * c.dst_pitch + 3 * xx + ch] = (uint8_t)__float2int_rn(fminf(fmaxf(acc[k], 0.0f), 255.0f));
    }
  }
}
