"""FusedVideoProcessor - drop-in for the HF Qwen2-VL video processor, backed by K1's video entry point.

Replaces ``processor.video_processor`` of ``Qwen2VLProcessor`` / ``Qwen2_5_VLProcessor`` (transformers 5.x
``models/qwen2_vl/video_processing_qwen2_vl.py``, ``Qwen2VLVideoProcessor``): same call, same outputs
(``pixel_values_videos (S, 1176) float32``, ``video_grid_thw (N, 3) int64``, ``video_metadata`` when asked), same
attributes the processor reads (``merge_size``, ``temporal_patch_size``, ``get_number_of_video_patches``,
``model_input_names``).  HF resizes every frame with torchvision - torch's uint8 antialiased bicubic on the CPU, its
fp32 one on a CUDA device - then applies the image backend's fused rescale + normalize, repeats the last frame up to an
even count and patchifies two frames per temporal patch.  ``zv_preprocess_video`` does all of it on the GPU for every
frame of a batch, bit-identical to the CPU convention (``backend="torchvision"``) or the CUDA one
(``"torchvision_cuda"``).  HF has no PIL video backend, so there is no "pil" here.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, geometry
from .processor import BACKENDS, BatchFeature, _backend_for_device

_OUT = {torch.float32: _lib.ZV_F32, torch.bfloat16: _lib.ZV_BF16, torch.float16: _lib.ZV_F16}


def sample_indices(total_num_frames, num_frames=None, fps=None, video_fps=None, temporal_patch_size=2, min_frames=4,
                   max_frames=768):
    """``Qwen2VLVideoProcessor.sample_frames``: the frame indices kept (num_frames rounded to the temporal patch, or
    ``fps`` frames per second of a video recorded at ``video_fps``), as an int64 array."""
    import math
    if fps is not None and num_frames is not None:
        raise ValueError("`num_frames` and `fps` are mutually exclusive arguments, please use only one!")
    if num_frames is not None:
        num_frames = round(num_frames / temporal_patch_size) * temporal_patch_size
    elif fps is not None:
        if video_fps is None:
            raise ValueError("Asked to sample `fps` frames per second but no video metadata was provided which is "
                             "required when sampling with `fps`.")
        max_frames = math.floor(min(max_frames, total_num_frames) / temporal_patch_size) * temporal_patch_size
        num_frames = total_num_frames / video_fps * fps
        num_frames = min(max(num_frames, min_frames), max_frames, total_num_frames)
        num_frames = math.floor(num_frames / temporal_patch_size) * temporal_patch_size
    if num_frames is not None and num_frames > total_num_frames:
        raise ValueError(f"Video can't be sampled. The inferred `num_frames={num_frames}` exceeds "
                         f"`total_num_frames={total_num_frames}`. Decrease `num_frames` or `fps` for sampling.")
    if num_frames is None:
        return np.arange(total_num_frames, dtype=np.int64)
    return torch.arange(0, total_num_frames, total_num_frames / num_frames).int().numpy().astype(np.int64)


def _frame_u8(f):
    """One frame (PIL / ndarray / tensor, HWC or CHW) -> (H, W, 3) uint8 tensor."""
    if hasattr(f, "convert") and hasattr(f, "size"):
        f = np.asarray(f.convert("RGB"))
    if isinstance(f, np.ndarray):
        f = torch.from_numpy(np.ascontiguousarray(f))
    if f.ndim == 3 and f.shape[0] == 3 and f.shape[-1] != 3:
        f = f.permute(1, 2, 0)
    return f


def _video_u8(v):
    """A video - (T, H, W, 3) / (T, 3, H, W) array or tensor, or a list of frames - -> (T, H, W, 3) uint8 tensor.
    As HF (``infer_channel_dimension_format``), a 4-D video whose second axis has 3 entries is channels-first."""
    if isinstance(v, (list, tuple)):
        v = torch.stack([_frame_u8(f) for f in v], 0)
    elif isinstance(v, np.ndarray):
        v = torch.from_numpy(np.ascontiguousarray(v))
    if not isinstance(v, torch.Tensor) or v.ndim != 4:
        raise ValueError(f"expected a (T, H, W, 3) or (T, 3, H, W) video, got {type(v).__name__} "
                         f"{tuple(getattr(v, 'shape', ()))}")
    if v.shape[1] == 3:
        v = v.permute(0, 2, 3, 1)
    if v.shape[-1] != 3:
        raise ValueError(f"expected 3 channels, got a video of shape {tuple(v.shape)}")
    if v.dtype != torch.uint8:
        raise NotImplementedError("the fused video path takes uint8 frames")
    return v


def _is_frame(x):
    return (hasattr(x, "convert") and hasattr(x, "size")) or (hasattr(x, "ndim") and x.ndim == 3)


def _batch(videos):
    """HF's ``make_batched_videos`` nesting: one video (4-D, or a list of frames), a list of videos, or a list of lists
    of frames -> list of (T, H, W, 3) uint8 tensors."""
    if hasattr(videos, "ndim") and videos.ndim == 5:
        return [_video_u8(v) for v in videos]
    if hasattr(videos, "ndim") and videos.ndim == 4:
        return [_video_u8(videos)]
    if isinstance(videos, (list, tuple)) and videos:
        if _is_frame(videos[0]):
            return [_video_u8(list(videos))]
        return [_video_u8(v) for v in videos]
    raise ValueError(f"cannot read videos from {type(videos).__name__}")


def upload_video(v, device):
    """(T, H, W, 3) uint8 tensor -> the same on ``device``, rows padded to a multiple of 16 pixels when 3 W is not a
    multiple of 4 (K1's tensor-core route wants a row pitch of 4-byte multiples, as for images).  A CUDA tensor whose
    frames are packed rows is used in place."""
    t, h, w, _ = v.shape
    if v.device.type == "cuda" and v.stride(3) == 1 and v.stride(2) == 3:
        return v
    if w % 4 == 0:
        return v.contiguous().to(device, non_blocking=False)
    buf = torch.empty((t, h, (w + 15) // 16 * 16, 3), dtype=torch.uint8, device=device)
    d = buf[:, :, :w]
    d.copy_(v)
    return d


class FusedVideoProcessor:
    model_input_names = ["pixel_values_videos", "video_grid_thw"]
    valid_kwargs = None

    def __init__(self, min_pixels=None, max_pixels=None, size=None, patch_size=14, temporal_patch_size=2, merge_size=2,
                 image_mean=None, image_std=None, rescale_factor=1 / 255, device=None, output_device="cpu",
                 backend="torchvision", do_sample_frames=False, num_frames=None, fps=None, min_frames=4, max_frames=768,
                 return_metadata=False, **unused):
        """``backend``: "torchvision" (HF's video processor on the CPU) or "torchvision_cuda" (called with
        ``device="cuda"``).  As in HF, a ``device=`` passed to ``preprocess`` picks the convention of that call."""
        if backend not in ("torchvision", "torchvision_cuda"):
            raise ValueError(f"backend must be 'torchvision' or 'torchvision_cuda' (HF has no PIL video backend), "
                             f"got {backend!r}")
        self.backend = backend
        size = dict(size) if size is not None else {"shortest_edge": 128 * 28 * 28, "longest_edge": 768 * 28 * 28}
        if min_pixels is not None:
            size["shortest_edge"] = min_pixels
        if max_pixels is not None:
            size["longest_edge"] = max_pixels
        if not size.get("shortest_edge") or not size.get("longest_edge"):
            raise ValueError("size must contain 'shortest_edge' and 'longest_edge' keys.")
        self.size = size
        self.patch_size, self.temporal_patch_size, self.merge_size = patch_size, temporal_patch_size, merge_size
        self.image_mean = list(image_mean) if image_mean is not None else [0.48145466, 0.4578275, 0.40821073]
        self.image_std = list(image_std) if image_std is not None else [0.26862954, 0.26130258, 0.27577711]
        self.rescale_factor = rescale_factor
        self.do_sample_frames, self.num_frames, self.fps = do_sample_frames, num_frames, fps
        self.min_frames, self.max_frames = min_frames, max_frames
        self.return_metadata = return_metadata
        self.do_resize = self.do_rescale = self.do_normalize = self.do_convert_rgb = True
        self.device = torch.device(device) if device is not None else None
        self.output_device = output_device
        self._ws = None
        self.last_launches = 0

    @property
    def min_pixels(self):
        return self.size["shortest_edge"]

    @property
    def max_pixels(self):
        return self.size["longest_edge"]

    def _device(self):
        if self.device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("FusedVideoProcessor needs a CUDA device (sm_100); there is no CPU fallback")
            self.device = torch.device("cuda", torch.cuda.current_device())
        return self.device

    def get_num_of_video_patches(self, num_frames, height, width, videos_kwargs=None):
        """HF's count (``num_frames // temporal_patch_size`` frame groups, as HF floors it)."""
        kw = videos_kwargs or {}
        rh, rw = geometry.smart_resize(height, width, self.patch_size * self.merge_size,
                                       kw.get("min_pixels") or self.min_pixels, kw.get("max_pixels") or self.max_pixels)
        return (num_frames // self.temporal_patch_size) * (rh // self.patch_size) * (rw // self.patch_size)

    get_number_of_video_patches = get_num_of_video_patches      # the name processing_qwen2_5_vl.py calls

    def sample_frames(self, metadata, num_frames=None, fps=None, **unused):
        total = metadata["total_num_frames"] if isinstance(metadata, dict) else metadata.total_num_frames
        video_fps = metadata.get("fps") if isinstance(metadata, dict) else getattr(metadata, "fps", None)
        if fps is not None and num_frames is not None:
            raise ValueError("`num_frames` and `fps` are mutually exclusive arguments, please use only one!")
        num_frames = num_frames if num_frames is not None else self.num_frames
        fps = fps if fps is not None else self.fps
        return sample_indices(total, num_frames, None if num_frames is not None else fps, video_fps,
                              self.temporal_patch_size, self.min_frames, self.max_frames)

    # ---- device path
    def preprocess_videos(self, videos_dev, out_dtype=torch.float32, window_order=False, min_pixels=None, max_pixels=None,
                          backend=None, out=None):
        """videos_dev: list of (T, H, W, 3) uint8 CUDA tensors (packed pixels, any row pitch).  Returns (patches (S, 1176)
        out_dtype on the GPU - HF order, or the tower's window order inside every frame group -, video_grid_thw (n, 3)
        int64 CPU tensor)."""
        backend = backend or self.backend
        if backend not in ("torchvision", "torchvision_cuda"):
            raise ValueError(f"video backend must be 'torchvision' or 'torchvision_cuda', got {backend!r}")
        cfg = _lib.default_cfg(patch=self.patch_size, merge=self.merge_size, temporal=self.temporal_patch_size,
                               rescale=float(self.rescale_factor), mean=self.image_mean, std=self.image_std,
                               resample_kind=BACKENDS[backend])
        device = videos_dev[0].device
        if device.type != "cuda":
            raise RuntimeError("preprocess_videos takes CUDA tensors; there is no CPU path")
        factor = self.patch_size * self.merge_size
        lo = int(min_pixels if min_pixels is not None else self.min_pixels)
        hi = int(max_pixels if max_pixels is not None else self.max_pixels)
        n = len(videos_dev)
        frames = np.array([v.shape[0] for v in videos_dev], np.int32)
        rhw = np.array([geometry.smart_resize(int(v.shape[1]), int(v.shape[2]), factor, lo, hi) for v in videos_dev], np.int32)
        grid = np.stack([(frames + 1) // 2, rhw[:, 0] // self.patch_size, rhw[:, 1] // self.patch_size], 1).astype(np.int64)
        for v in videos_dev:
            if v.dtype != torch.uint8 or v.ndim != 4 or v.shape[3] != 3 or v.stride(3) != 1 or v.stride(2) != 3 or v.device != device:
                raise ValueError("videos must be (T, H, W, 3) uint8 CUDA tensors with packed pixels, on one device")
        ptrs = [v[k].data_ptr() for v in videos_dev for k in range(v.shape[0])]
        fhw = np.array([[v.shape[1], v.shape[2]] for v in videos_dev for _ in range(v.shape[0])], np.int32)
        pitch = np.array([v.stride(1) for v in videos_dev for _ in range(v.shape[0])], np.int64)
        S = int((grid[:, 0] * grid[:, 1] * grid[:, 2]).sum())
        lib = _lib.lib()
        ws_bytes = _lib.check(lib.zv_preprocess_video_workspace_bytes(n, frames.ctypes.data, fhw.ctypes.data, rhw.ctypes.data))
        if self._ws is None or self._ws.numel() < ws_bytes or self._ws.device != device:
            self._ws = torch.empty(int(ws_bytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        if out is None:
            out = torch.empty((S, 1176), dtype=out_dtype, device=device)
        elif out.shape != (S, 1176) or out.dtype != out_dtype or not out.is_contiguous():
            raise ValueError("preprocess_videos: `out` has the wrong shape/dtype")
        stream = torch.cuda.current_stream(device).cuda_stream
        with torch.cuda.device(device):
            _lib.check(lib.zv_preprocess_video(
                C.byref(cfg), n, frames.ctypes.data, (C.c_void_p * len(ptrs))(*ptrs), fhw.ctypes.data, pitch.ctypes.data,
                rhw.ctypes.data, out.data_ptr(), _OUT[out_dtype], _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF,
                self._ws.data_ptr(), self._ws.numel(), stream))
        self.last_launches = lib.zv_last_launch_count()
        return out, torch.from_numpy(grid)

    # ---- HF surface
    def preprocess(self, videos, return_tensors=None, min_pixels=None, max_pixels=None, size=None, do_resize=None,
                   do_rescale=None, do_normalize=None, device=None, do_sample_frames=None, num_frames=None, fps=None,
                   video_metadata=None, return_metadata=None, **unused):
        for name, flag in (("do_resize", do_resize), ("do_rescale", do_rescale), ("do_normalize", do_normalize)):
            if flag is False:
                raise NotImplementedError(f"{name}=False is not part of the fused path")
        if size is not None:
            min_pixels = size.get("shortest_edge", min_pixels)
            max_pixels = size.get("longest_edge", max_pixels)
        backend = _backend_for_device(self.backend, device)
        vids = _batch(videos)
        if video_metadata is None:
            metas = [{"total_num_frames": int(v.shape[0]), "fps": None, "duration": None,
                      "frames_indices": list(range(int(v.shape[0]))), "height": int(v.shape[1]), "width": int(v.shape[2])}
                     for v in vids]
        else:
            metas = list(video_metadata) if isinstance(video_metadata, (list, tuple)) else [video_metadata]
            if metas and isinstance(metas[0], (list, tuple)):
                metas = [m for ms in metas for m in ms]
            metas = [dict(m) if isinstance(m, dict) else {k: getattr(m, k) for k in ("total_num_frames", "fps", "duration",
                     "frames_indices", "height", "width")} for m in metas]
        sample = self.do_sample_frames if do_sample_frames is None else do_sample_frames
        if sample:
            for k, (v, m) in enumerate(zip(vids, metas)):
                idx = self.sample_frames(m, num_frames=num_frames, fps=fps)
                vids[k] = v[torch.from_numpy(idx).to(v.device)]
                m["frames_indices"] = idx.tolist()
        dev_vids = [upload_video(v, self._device()) for v in vids]
        pv, grid = self.preprocess_videos(dev_vids, torch.float32, False, min_pixels, max_pixels, backend)
        if self.output_device == "cpu":
            pv = pv.cpu()
        data = {"pixel_values_videos": pv, "video_grid_thw": grid}
        if return_tensors in ("np", "numpy"):
            data = {k: v.cpu().numpy() for k, v in data.items()}
        elif return_tensors not in (None, "pt", "torch"):
            raise ValueError(f"unsupported return_tensors={return_tensors!r}")
        if return_metadata if return_metadata is not None else self.return_metadata:
            try:
                from transformers.video_utils import VideoMetadata
                data["video_metadata"] = [VideoMetadata(**m) for m in metas]
            except ImportError:                 # pragma: no cover
                data["video_metadata"] = metas
        return BatchFeature(data=data)

    def __call__(self, videos=None, **kwargs):
        return self.preprocess(videos, **kwargs)
