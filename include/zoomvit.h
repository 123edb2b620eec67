/* zoomvit.h - C ABI of libzoomvit.so: the B200-native drop-in for ZoomEarth's per-zoom-step vision path.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, returns 0 on success or a negative
 * zv_err; the message of the last failure on the calling thread is zv_last_error().  The caller owns every
 * device buffer (inputs, outputs, workspaces); the library never allocates device memory and never
 * synchronises: all device work is enqueued on the stream handle the caller passes (a cudaStream_t).
 * There is NO CPU fallback: device entry points fail with ZV_ENODEV / ZV_EARCH when no sm_100 GPU is current.
 *
 * What each entry point replaces in the reference (earth-insights/ZoomEarth; `HF:` = the transformers
 * package the reference depends on, `HF:models/...` relative to site-packages/transformers):
 *
 *   zv_cut_box            src/eval/infer.py:41-76   cut_image() box arithmetic (= src/demo.py:30-70)
 *   zv_resize_dims        src/eval/infer.py:78-85   resize_image() size arithmetic
 *   zv_resize_dims_ex     resize_image() variants: src/demo.py:86-93 (1024), src/train/SFT.py:76-81 (always resizes),
 *                         src/train/RL/.../open_r1/custom/customized_funcs.py:76-85 (min_scale = 30 / min side)
 *   zv_cut_box_sft        src/train/SFT.py:83-125 cut_image() (else-branch: resize to min side 512 + centre crop)
 *   zv_resize_u8          infer.py:72-75 + 78-85: PIL.Image.crop(box).resize((w, h), Image.BICUBIC) on the device, uint8 out
 *                         (resize_image(cut_image(...)) of infer.py:215,239, demo.py:133,140) - feeds zv_preprocess
 *   zv_smart_resize       HF:models/qwen2_vl/image_processing_pil_qwen2_vl.py:57-83
 *   zv_geometry           infer.py:41-76 + HF smart_resize + grid computation (pil_qwen2_vl.py:186-187)
 *   zv_resample_*         Pillow ImagingResample coefficient tables (reached from infer.py:84,
 *                         HF:image_transforms.py:368); by cfg->resample_kind torch's uint8 antialiased bicubic
 *                         (HF:image_processing_backends.py TorchvisionBackend.resize -> torchvision resize)
 *   zv_normalize_lut      HF:image_transforms.py:89-124 (rescale) + :384-442 (normalize); by cfg->resample_kind
 *                         TorchvisionBackend.rescale_and_normalize (rescale folded into mean and std)
 *   zv_preprocess         infer.py:72-75 (Image.crop) + HF:pil_qwen2_vl.py:143-224 (_preprocess: resize,
 *                         rescale, normalize, patchify) as one fused device pass; by cfg->resample_kind
 *                         HF:models/qwen2_vl/image_processing_qwen2_vl.py (the torchvision backend, on the CPU or,
 *                         kind 2, on a CUDA device) instead
 *   zv_preprocess_video   HF:models/qwen2_vl/video_processing_qwen2_vl.py (Qwen2VLVideoProcessor, torchvision resize on the
 *                         CPU or a CUDA device) as one device pass over all frames of a batch of videos
 *   zv_plan_*             HF:models/qwen2_5_vl/modeling_qwen2_5_vl.py:382-409 (rot_pos_emb ids),
 *                         :411-451 (get_window_index), :470-496 (cu_window_seqlens, cu_seqlens)
 *   zv_weights_*          state-dict import of `visual.*` (HF:modeling_qwen2_5_vl.py:345-380 module tree; Qwen2-VL:
 *                         HF:models/qwen2_vl/modeling_qwen2_vl.py VisionMlp / Qwen2VLVisionBlock / PatchMerger)
 *   zv_visual_forward     HF:modeling_qwen2_5_vl.py:455-518 (Qwen2_5_VisionTransformerPretrainedModel.forward), or with
 *                         tower_kind = ZV_TOWER_QWEN2 Qwen2VisionTransformerPretrainedModel.forward
 *   zv_visual_forward_into  + HF:modeling_qwen2_5_vl.py:1301-1307 (get_placeholder_mask + masked_scatter into
 *                         inputs_embeds; reference copy src/train/RL/.../open_r1/model/modeling_qwen2_vl.py:1191-1207)
 *   zv_rope_index         reference .../open_r1/model/modeling_qwen2_vl.py:967-1114 (get_rope_index; by flag the
 *                         transformers 5.x variant HF:modeling_qwen2_5_vl.py:1024-1135)
 *   zv_placeholder_rows   the row list behind masked_scatter (HF:modeling_qwen2_5_vl.py:1179-1218)
 *   zv_rope_index_dev, zv_placeholder_rows_dev   the same two on the device, stream-ordered and graph-capturable
 */
#ifndef ZOOMVIT_H_
#define ZOOMVIT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZV_API __attribute__((visibility("default")))

typedef enum zv_err {
  ZV_OK = 0,
  ZV_EINVAL = -1,        /* bad argument */
  ZV_EINVAL_ASPECT = -2, /* smart_resize: aspect ratio > 200 (HF raises ValueError) */
  ZV_EINVAL_BOX = -3,    /* crop box right < left or lower < upper (Pillow raises ValueError) */
  ZV_ENOMEM = -4,        /* caller-provided workspace too small */
  ZV_ECUDA = -5,         /* CUDA runtime/driver error, text in zv_last_error() */
  ZV_ENODEV = -6,        /* no CUDA device */
  ZV_EARCH = -7          /* device is not sm_100 */
} zv_err;

enum { ZV_F32 = 0, ZV_BF16 = 1, ZV_F16 = 2 };   /* element types at the boundary */
enum { ZV_ORDER_HF = 0, ZV_ORDER_WINDOW = 1 }; /* patch row order: HF merge-group raster, or tower window order */
/* Vision tower family.  ZV_TOWER_QWEN25: Qwen2.5-VL (RMSNorm, SwiGLU, window attention, HF:modeling_qwen2_5_vl.py).
 * ZV_TOWER_QWEN2: Qwen2-VL (LayerNorm with bias, fc1 -> QuickGELU -> fc2, full attention in every block,
 * HF:models/qwen2_vl/modeling_qwen2_vl.py Qwen2VisionTransformerPretrainedModel); requires fullatt_mask_lo to cover all
 * `depth` blocks and inter = 5120. */
enum { ZV_TOWER_QWEN25 = 0, ZV_TOWER_QWEN2 = 1 };
/* Resample / normalise convention of zv_preprocess and zv_normalize_lut, i.e. which HF image-processor backend the
 * pixels match bit for bit.  ZV_RESAMPLE_PIL: Qwen2VLImageProcessorPil (Pillow bicubic, rescale then normalize).
 * ZV_RESAMPLE_TORCHVISION: Qwen2VLImageProcessor, the transformers 5.x default (torch's uint8 antialiased bicubic:
 * Pillow's windows and weights quantised to int16 at a per-axis precision; normalize with the rescale folded into
 * mean and std, in fp32).  ZV_RESAMPLE_TORCHVISION_CUDA: Qwen2VLImageProcessor called with device="cuda" (torch's fp32
 * antialiased bicubic on a CUDA device: both passes in fp32 with no uint8 rounding between them, then clamp, round half to
 * even and uint8; the same normalisation as ZV_RESAMPLE_TORCHVISION).  It has no integer taps, so zv_resample_coeffs_ex
 * rejects it.  zv_resize_u8 is Pillow-only: it stands for the reference's own resize_image. */
enum { ZV_RESAMPLE_PIL = 0, ZV_RESAMPLE_TORCHVISION = 1, ZV_RESAMPLE_TORCHVISION_CUDA = 2 };

/* Processor + model constants (defaults = Qwen2.5-VL-3B vision config + OPENAI_CLIP statistics). */
typedef struct zv_cfg {
  int32_t patch;        /* 14 */
  int32_t merge;        /* 2  */
  int32_t temporal;     /* 2  */
  int32_t window;       /* 112 */
  int32_t min_size;     /* 512, cut_image() */
  int32_t depth;        /* 32 */
  int32_t hidden;       /* 1280 */
  int32_t heads;        /* 16 */
  int32_t inter;        /* 3420 */
  int32_t out_hidden;   /* 2048 */
  int32_t fullatt_mask_lo; /* bit l set = block l uses full attention (blocks 0..31) */
  int32_t op_dtype;     /* GEMM / attention operand type: ZV_F16 = fp16 (zv_default_cfg), ZV_BF16 or 0 = bf16 (opt-in) */
  int64_t min_pixels;   /* 3136 */
  int64_t max_pixels;   /* per call site */
  double  rescale;      /* 1/255 */
  float   mean[3];
  float   std[3];
  float   eps;          /* 1e-6 */
  float   reserved_f;
  int32_t tower_kind;   /* ZV_TOWER_QWEN25 (zv_default_cfg) or ZV_TOWER_QWEN2 */
  int32_t resample_kind; /* ZV_RESAMPLE_PIL (zv_default_cfg), ZV_RESAMPLE_TORCHVISION or ZV_RESAMPLE_TORCHVISION_CUDA */
} zv_cfg;

ZV_API const char* zv_version(void);
ZV_API const char* zv_last_error(void);
ZV_API void zv_default_cfg(zv_cfg* cfg);

/* ---------------------------------------------------------------- host geometry (pure, no device) */
ZV_API int zv_cut_box(int32_t img_w, int32_t img_h, const double* bbox_xyxy, int32_t min_size, int32_t* box_out4);
ZV_API int zv_resize_dims(int32_t w, int32_t h, int32_t max_size, int32_t* new_wh2, double* inv_scale);
/* mode 0: infer.py / demo.py (resize only when scale < 1); 1: SFT.py (always, may upscale); 2: customized_funcs.py
 * (scale = max(30 / min(w, h), max_size / max(w, h)), resize only when < 1).  new_wh2 = (w, h) after the resize. */
ZV_API int zv_resize_dims_ex(int32_t w, int32_t h, int32_t max_size, int32_t mode, int32_t* new_wh2, double* inv_scale);
/* SFT.py cut_image: box_out4 = the box Image.crop gets.  When both box sides are >= min_size the crop is then resized to
 * resized_wh2 (shorter side = min_size) and centre_box4 (a min_size square inside it) is cut out; otherwise resized_wh2 = 0. */
ZV_API int zv_cut_box_sft(int32_t img_w, int32_t img_h, const double* bbox_xyxy, int32_t min_size, int32_t* box_out4,
                          int32_t* resized_wh2, int32_t* centre_box4);
ZV_API int zv_smart_resize(int32_t height, int32_t width, int32_t factor, int64_t min_pixels, int64_t max_pixels,
                           int32_t* out_hw2);
/* n crops: img_hw[n][2] (h,w), bbox_xyxy[n][4] -> crop_box[n][4] (x0,y0,x1,y1), resized_hw[n][2], grid_thw[n][3].
 * bbox_xyxy == NULL means "whole image"; cfg->min_size < 0 means "boxes are final crop boxes" (no cut_image rule). */
ZV_API int zv_geometry(const zv_cfg* cfg, int32_t n, const int32_t* img_hw, const double* bbox_xyxy,
                       int32_t* crop_box, int32_t* resized_hw, int64_t* grid_thw);

/* Pillow bicubic taps for one axis: ksize, then bounds[out][2] = (first tap, tap count) and kk[out][ksize]
 * (22-bit fixed point). */
ZV_API int32_t zv_resample_ksize(int32_t in_size, int32_t out_size);
ZV_API int zv_resample_coeffs(int32_t in_size, int32_t out_size, int32_t* bounds, int32_t* kk);
/* Same tables for a resample kind (ZV_RESAMPLE_*), as the kernels consume them: 22-bit taps.  ZV_RESAMPLE_TORCHVISION
 * taps are torch's int16 taps at the axis precision p, shifted left by 22 - p; *precision = p (22 for Pillow and for a
 * same-size axis).  Kind ZV_RESAMPLE_PIL equals zv_resample_coeffs. */
ZV_API int zv_resample_coeffs_ex(int32_t kind, int32_t in_size, int32_t out_size, int32_t* bounds, int32_t* kk,
                                 int32_t* precision);
/* lut[3][256] fp32: HF rescale+normalize of every uint8 level, in the arithmetic of cfg->resample_kind. */
ZV_API int zv_normalize_lut(const zv_cfg* cfg, float* lut768);

/* ---------------------------------------------------------------- device: fused crop->resize->normalize->patchify */
/* Bytes of device workspace zv_preprocess needs for these crops (coefficient tables + the uint8
 * intermediate between the two resample passes). */
ZV_API int64_t zv_preprocess_workspace_bytes(int32_t n, const int32_t* crop_box, const int32_t* resized_hw);
/* src_dev[i]: device pointer to image i's (H, W, 3) uint8 pixels, row pitch src_pitch[i] bytes, size src_hw[i].
 * Writes patches for crop i at rows [row_off[i], row_off[i] + gh*gw) of out_dev (row = 1176 elements of
 * out_dtype); row_off == NULL packs crops back to back.  row_order selects HF or window order inside a crop. */
ZV_API int zv_preprocess(const zv_cfg* cfg, int32_t n, const uint8_t* const* src_dev, const int32_t* src_hw,
                         const int64_t* src_pitch, const int32_t* crop_box, const int32_t* resized_hw,
                         const int64_t* row_off, void* out_dev, int32_t out_dtype, int32_t row_order,
                         void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Video frames -> patches (HF:models/qwen2_vl/video_processing_qwen2_vl.py Qwen2VLVideoProcessor._preprocess: resize,
 * fused rescale + normalize, last-frame repeat to an even count, patchify with temporal patches of two frames).
 * frames_per_video[v] = T_v >= 1; frame f (all videos' frames back to back) is frame_dev[f], (H, W, 3) uint8 of size
 * frame_hw[f] = (h, w) with row pitch frame_pitch[f] bytes; video v's frames are resized whole to resized_hw[v] (multiples of
 * 28).  Video v writes ceil(T_v / 2) * gh * gw patch rows (1176 elements of out_dtype), videos back to back; temporal slot
 * tp of frame group t holds frame min(2 t + tp, T_v - 1).  row_order: HF order, or the tower's window order inside every
 * frame group.  cfg->resample_kind must be ZV_RESAMPLE_TORCHVISION (HF's video processor on the CPU) or
 * ZV_RESAMPLE_TORCHVISION_CUDA (on a CUDA device); ZV_RESAMPLE_PIL is ZV_EINVAL, HF has no PIL video backend. */
ZV_API int64_t zv_preprocess_video_workspace_bytes(int32_t n_videos, const int32_t* frames_per_video, const int32_t* frame_hw,
                                                   const int32_t* resized_hw);
ZV_API int zv_preprocess_video(const zv_cfg* cfg, int32_t n_videos, const int32_t* frames_per_video,
                               const uint8_t* const* frame_dev, const int32_t* frame_hw, const int64_t* frame_pitch,
                               const int32_t* resized_hw, void* out_dev, int32_t out_dtype, int32_t row_order,
                               void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Device form of the reference's resize_image(cut_image(...)): crop i = PIL.Image.crop(crop_box[i]) of image i (zero
 * fill outside the image), resized with Pillow-exact bicubic to out_hw[i] = (h, w) and written as a plain (h, w, 3) uint8
 * image at dst_dev[i] with row pitch dst_pitch[i] bytes.  Same-size axes are copied (Pillow skips the pass).  The result is
 * bit-identical to Pillow and can be handed to zv_preprocess as a source image (the reference's two-resample flow:
 * resize_image to <= 512 / 1024 px, then the processor's smart_resize, uint8 rounding in between). */
ZV_API int64_t zv_resize_u8_workspace_bytes(int32_t n, const int32_t* crop_box, const int32_t* out_hw);
ZV_API int zv_resize_u8(int32_t n, const uint8_t* const* src_dev, const int32_t* src_hw, const int64_t* src_pitch,
                        const int32_t* crop_box, const int32_t* out_hw, uint8_t* const* dst_dev, const int64_t* dst_pitch,
                        void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Test hook (CPU, no GPU needed): runs the HOST side of zv_preprocess / zv_resize_u8 - descriptors, tap tables, work
 * lists of the tensor-core route (csrc/zv_k1_tc.cuh) - over HOST pointers and emulates that route's kernels lane by lane
 * on the CPU.  took_tc[i] = 1 for the crops the route accepts (row pitch a multiple of 4 bytes, <= 4 K blocks per chunk);
 * only those are written.  u8_dst_host == NULL: fp32 patches into out_host (zv_preprocess), else uint8 images
 * (zv_resize_u8).  The tables follow cfg->resample_kind (cfg may be NULL in uint8 mode: Pillow's).  Checks everything but
 * the hardware layouts (swizzle, descriptors, TMEM), which the GPU tests cover. */
ZV_API int zv_debug_k1_tc_host(const zv_cfg* cfg, int32_t n, const uint8_t* const* src_host, const int32_t* src_hw,
                               const int64_t* src_pitch, const int32_t* crop_box, const int32_t* resized_hw, float* out_host,
                               int32_t row_order, uint8_t* const* u8_dst_host, const int64_t* u8_pitch, void* workspace_host,
                               int64_t workspace_bytes, int32_t* took_tc);

/* ---------------------------------------------------------------- plan: per-batch integer bookkeeping */
typedef struct zv_plan zv_plan;
ZV_API int zv_plan_create(const zv_cfg* cfg, int32_t n, const int64_t* grid_thw, zv_plan** out);
ZV_API void zv_plan_free(zv_plan* p);
ZV_API int64_t zv_plan_num_patches(const zv_plan* p);              /* S */
ZV_API int64_t zv_plan_num_tokens(const zv_plan* p);               /* T = S/4 */
ZV_API const int64_t* zv_plan_window_index(const zv_plan* p);      /* [T] */
ZV_API const int64_t* zv_plan_reverse_index(const zv_plan* p);     /* [T] argsort(window_index) */
ZV_API const int32_t* zv_plan_cu_window(const zv_plan* p, int32_t* n_out); /* after unique_consecutive */
ZV_API const int32_t* zv_plan_cu_window_raw(const zv_plan* p, int32_t* n_out); /* HF list incl. empty windows */
ZV_API const int32_t* zv_plan_cu_full(const zv_plan* p, int32_t* n_out);
ZV_API const int32_t* zv_plan_pos_ids(const zv_plan* p);           /* [S][2] (h,w), HF row order */
ZV_API int64_t zv_plan_device_bytes(const zv_plan* p);
/* Copies the device-side tables (window-ordered rotary cos/sin, segment work lists, scatter index) into the
 * caller's buffer; must precede zv_visual_forward with the same buffer. */
ZV_API int zv_plan_upload(zv_plan* p, void* plan_dev, int64_t bytes, void* stream);

/* ---------------------------------------------------------------- weights */
typedef struct zv_tensor {
  const char* name;     /* HF state-dict name relative to the tower, e.g. "blocks.0.attn.qkv.weight" */
  const void* data;     /* DEVICE pointer, contiguous */
  int32_t dtype;        /* ZV_F32 or ZV_BF16 */
  int32_t ndim;
  int64_t shape[5];
} zv_tensor;
ZV_API int64_t zv_weights_bytes(const zv_cfg* cfg);
/* Packs an HF state dict (device tensors) into the library's layout inside packed_dev (zv_weights_bytes). */
ZV_API int zv_weights_pack(const zv_cfg* cfg, const zv_tensor* tensors, int32_t n, void* packed_dev,
                           int64_t packed_bytes, void* stream);

/* ---------------------------------------------------------------- tower */
ZV_API int64_t zv_visual_workspace_bytes(const zv_cfg* cfg, const zv_plan* p);
/* patches_dev: (S, 1176) of in_dtype in in_order.  merged_out_dev: (T, out_hidden) of out_dtype, HF order
 * (image-major, merge-group raster).  hidden_out_dev (optional, may be NULL): (S, hidden) fp32 last hidden
 * state in window order. */
ZV_API int zv_visual_forward(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                             const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                             int32_t out_dtype, void* hidden_out_dev, void* workspace_dev,
                             int64_t workspace_bytes, void* stream);
/* Same forward with the embedding gather fused into the last GEMM's epilogue: every output row is also written at
 * row (peer_row_off + row) of each of the n_peers (<= 8) peer buffers - device pointers into the OTHER ranks' gather
 * buffers, mapped into this process (CUDA IPC / symmetric memory), element type out_dtype (16-bit), row = out_hidden
 * elements.  The caller synchronises the ranks afterwards (any barrier); no collective is needed. */
ZV_API int zv_visual_forward_gather(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                                    const void* patches_dev, int32_t in_dtype, int32_t in_order, void* merged_out_dev,
                                    int32_t out_dtype, void* workspace_dev, int64_t workspace_bytes,
                                    void* const* peer_out_dev, int32_t n_peers, int64_t peer_row_off, void* stream);
/* Ragged form of the fused gather (crop-sharded batches whose crops interleave in the global order): embedding k of this
 * rank's batch (HF order) is written to row dest_rows_dev[k] of this rank's own gather buffer gather_local_dev
 * ((gather_rows, out_hidden) of out_dtype) AND to the same row of every peer buffer.  dest_rows_dev: int64 [T] on the device. */
ZV_API int zv_visual_forward_gather_rows(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                                         const void* patches_dev, int32_t in_dtype, int32_t in_order, void* gather_local_dev,
                                         int64_t gather_rows, int32_t out_dtype, const int64_t* dest_rows_dev,
                                         void* workspace_dev, int64_t workspace_bytes, void* const* peer_out_dev,
                                         int32_t n_peers, void* stream);
/* Same forward with the LM hand-off fused into the last GEMM's epilogue: embedding k (HF order) is written to row
 * dest_rows_dev[k] of embeds_dev, the flattened (embeds_rows, out_hidden) inputs_embeds of the language model
 * (element type embeds_dtype) - torch's inputs_embeds.masked_scatter(image_mask, image_embeds) without the
 * (T, out_hidden) round trip.  dest_rows_dev: int64 [T] on the device (zv_placeholder_rows, or nonzero() of the mask). */
ZV_API int zv_visual_forward_into(const zv_cfg* cfg, const void* weights_dev, const zv_plan* p, const void* plan_dev,
                                  const void* patches_dev, int32_t in_dtype, int32_t in_order, void* embeds_dev,
                                  int64_t embeds_rows, int32_t embeds_dtype, const int64_t* dest_rows_dev,
                                  void* workspace_dev, int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- LM hand-off, host side (pure, no device) */
/* Multimodal rotary position index.  input_ids / attention_mask (may be NULL): [batch][seq_len] int64 on the host;
 * image_grid_thw [n_images][3] (NULL = text only); position_ids out [3][batch][seq_len], deltas out [batch].
 * hf5_semantics 0: the reference's copy (padded positions 1, delta against the padded length); 1: transformers 5.x
 * (padded positions 0, delta against the unpadded length). */
ZV_API int zv_rope_index(const int64_t* input_ids, const int64_t* attention_mask, int32_t batch, int32_t seq_len,
                         const int64_t* image_grid_thw, int32_t n_images, int64_t image_token_id,
                         int64_t video_token_id, int64_t vision_start_token_id, int32_t merge, int32_t hf5_semantics,
                         int64_t* position_ids, int64_t* deltas);
/* Flattened rows holding the image placeholder, in order; writes at most rows_cap of them, returns the count. */
ZV_API int64_t zv_placeholder_rows(const int64_t* input_ids, int64_t n_tokens, int64_t image_token_id,
                                   int64_t* rows_out, int64_t rows_cap);

/* ---------------------------------------------------------------- LM hand-off, device side */
/* The two functions above as kernels on `stream`: device pointers in and out, no host synchronisation, no allocation, so
 * that they can be captured in one CUDA graph with zv_visual_forward_into.  Results are bit-identical to the host
 * functions.  A condition on which zv_rope_index fails is recorded in `status` (int64 [4] on the device) instead:
 *   status[0] = ZV_HANDOFF_* check (0 = none), status[1] = sample, status[2..3] = details (below);
 * the error recorded is the one the host function reports: the lowest sample, then the host's check order.  On such an
 * error the positions are unspecified; nothing is written outside the caller's buffers.  Argument errors the host can
 * see (null pointers, batch / seq_len / merge <= 0, a workspace smaller than zv_handoff_workspace_bytes) return ZV_EINVAL
 * before any device work.  One workspace serves both functions for the same (batch, seq_len) on one stream. */
enum {
  ZV_HANDOFF_OK = 0,
  ZV_HANDOFF_VIDEO = 1,             /* a vision start followed by a video placeholder */
  ZV_HANDOFF_TRAILING_VSTART = 2,   /* the sample's last admitted token is a vision start */
  ZV_HANDOFF_FEW_PLACEHOLDERS = 3,  /* fewer image placeholders than images */
  ZV_HANDOFF_GRID_ROWS = 4,         /* image_grid_thw has too few rows; status[2] = n_images */
  ZV_HANDOFF_EMPTY_GRID = 5,        /* status[2] = the image (grid row) with t, h / merge or w / merge <= 0 */
  ZV_HANDOFF_COUNT = 6,             /* status[2] positions for status[3] tokens */
  ZV_HANDOFF_MASKED = 7,            /* every token of the sample is masked */
  ZV_HANDOFF_ROWS_COUNT = 8         /* zv_placeholder_rows_dev: status[2] placeholders for status[3] = rows_cap rows */
};
ZV_API int64_t zv_handoff_workspace_bytes(int32_t batch, int32_t seq_len);
/* input_ids, attention_mask (may be NULL): [batch][seq_len] int64; image_grid_thw: [n_images][3] int64 (NULL = text
 * only); position_ids [3][batch][seq_len], deltas [batch]; all on the device.  2 kernel launches (1 without a grid). */
ZV_API int zv_rope_index_dev(const int64_t* input_ids, const int64_t* attention_mask, int32_t batch, int32_t seq_len,
                             const int64_t* image_grid_thw, int32_t n_images, int64_t image_token_id,
                             int64_t video_token_id, int64_t vision_start_token_id, int32_t merge, int32_t hf5_semantics,
                             int64_t* position_ids, int64_t* deltas, int64_t* status, void* workspace_dev,
                             int64_t workspace_bytes, void* stream);
/* rows_out [rows_cap]: the flattened indices of input_ids == image_token_id in order (masked_scatter order), -1 in every
 * slot at or beyond their count; status[2] = the count, status[0] = ZV_HANDOFF_ROWS_COUNT when it is not rows_cap.
 * The workspace needs zv_handoff_workspace_bytes of any (batch, seq_len) with batch * seq_len >= n_tokens.  2 launches. */
ZV_API int zv_placeholder_rows_dev(const int64_t* input_ids, int64_t n_tokens, int64_t image_token_id, int64_t* rows_out,
                                   int64_t rows_cap, int64_t* status, void* workspace_dev, int64_t workspace_bytes,
                                   void* stream);

/* Number of kernels the last zv_preprocess / zv_visual_forward / hand-off device call on this thread launched. */
ZV_API int64_t zv_last_launch_count(void);

/* Optional per-kernel-class device timing (CUDA events on the launching stream around every launch of that
 * class).  Classes: 0 k1 hpass, 1 k1 vpass, 2 gemm store, 3 gemm qkv+rope, 4 gemm residual, 5 gemm swiglu,
 * 6 gemm gelu, 7 gemm scatter, 8 attention (window layers), 9 attention (full layers), 10 rmsnorm / layernorm +
 * cast_rows_ss / cast_rows_ln, 11 gather, 12 gemm quickgelu (Qwen2-VL fc1), 13 k1 fp32 resample
 * (ZV_RESAMPLE_TORCHVISION_CUDA; its patchify kernel counts as class 1). */
ZV_API void zv_timing_enable(int on);
ZV_API void zv_timing_reset(void);
ZV_API int zv_timing_read(int kernel_class, double* ms_total, int64_t* count);

/* Standalone GEMM entry (the tower's tcgen05 kernel), exposed for unit tests and roofline runs:
 * C[M,N] = A[M,K] (bf16, row-major, lda elements) * B[N,K]^T (bf16) (+ bias[N] fp32), out fp32 or bf16. */
ZV_API int zv_gemm_bf16(const void* a_dev, int64_t lda, const void* b_dev, int64_t ldb, const float* bias_dev,
                        void* c_dev, int64_t ldc, int32_t c_dtype, int64_t m, int64_t n, int64_t k,
                        void* stream);
/* Same kernel with a selectable fused epilogue (0 store, 1 qkv bias+rotary, 2 fp32 residual add, 3 SwiGLU,
 * 4 bias+GELU, 5 bias+row scatter); pos_dev [M][2] int32, rope_dev [max_pos][20][2] fp32, scatter_dev [M] int32. */
ZV_API int zv_gemm_ex(int32_t epilogue, const void* a_dev, int64_t lda, const void* b_dev, int64_t ldb,
                      const float* bias_dev, void* out_dev, int64_t ldo, int32_t out_dtype, int64_t m, int64_t n,
                      int64_t k, const int32_t* pos_dev, const float* rope_dev, const int32_t* scatter_dev,
                      int32_t heads, int32_t op_dtype /* ZV_BF16 or ZV_F16 operands */, void* stream);
/* Standalone varlen attention (rotated q,k already in qkv): qkv (S, 3*hidden) bf16 -> out (S, hidden) bf16. */
ZV_API int zv_attention(const void* qkv_dev, void* out_dev, int32_t heads, int32_t head_dim,
                        const int32_t* cu_seqlens_host, int32_t n_seg, void* work_dev, int64_t work_bytes,
                        int32_t dtype /* ZV_BF16 or ZV_F16 */, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ZOOMVIT_H_ */
