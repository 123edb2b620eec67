"""Oracle: the HF Qwen2-VL video processor (``Qwen2VLVideoProcessor``, transformers 5.x
``models/qwen2_vl/video_processing_qwen2_vl.py``) in NumPy.  Test infrastructure only.

``_preprocess`` per video: ``smart_resize(h, w, factor=28, min_pixels, max_pixels)`` (the image rule, no frame term), the
torchvision resize of every frame (``oracle.resample_torchvision`` on the CPU, ``oracle.resample_torchvision_cuda`` on a
CUDA device), the fused fp32 rescale + normalize of the torchvision image backend (``processor_torchvision.normalize_lut``),
the last frame repeated up to an even count, and the 10-D transpose to ``(grid_t, gh/2, gw/2, 2, 2, C, 2, 14, 14)``.
``sample_indices`` restates ``Qwen2VLVideoProcessor.sample_frames``.
"""
import math

import numpy as np

from . import geometry, resample_torchvision, resample_torchvision_cuda
from .processor import MERGE, OPENAI_CLIP_MEAN, OPENAI_CLIP_STD, PATCH
from .processor_torchvision import normalize_lut

TEMPORAL = 2
MIN_PIXELS, MAX_PIXELS = 128 * 28 * 28, 768 * 28 * 28


def sample_indices(total_num_frames, num_frames=None, fps=None, video_fps=None, temporal_patch_size=TEMPORAL,
                   min_frames=4, max_frames=768):
    """Frame indices ``sample_frames`` picks (int32, as torch's ``arange(...).int()``)."""
    if fps is not None and num_frames is not None:
        raise ValueError("`num_frames` and `fps` are mutually exclusive arguments, please use only one!")
    if num_frames is not None:
        num_frames = round(num_frames / temporal_patch_size) * temporal_patch_size
    elif fps is not None:
        if video_fps is None:
            raise ValueError("sampling by fps needs the video's fps")
        max_frames = math.floor(min(max_frames, total_num_frames) / temporal_patch_size) * temporal_patch_size
        num_frames = total_num_frames / video_fps * fps
        num_frames = min(max(num_frames, min_frames), max_frames, total_num_frames)
        num_frames = math.floor(num_frames / temporal_patch_size) * temporal_patch_size
    if num_frames is not None and num_frames > total_num_frames:
        raise ValueError(f"Video can't be sampled. The inferred `num_frames={num_frames}` exceeds "
                         f"`total_num_frames={total_num_frames}`.")
    if num_frames is None:
        return np.arange(total_num_frames, dtype=np.int32)
    # torch.arange(0, total, total / num_frames) with a float step: fp32 values start + i * step, truncated
    step = total_num_frames / num_frames
    n = math.ceil(total_num_frames / step)
    return (np.float32(0) + np.arange(n, dtype=np.float64) * step).astype(np.float32).astype(np.int32)


def patchify_video(frames_chw):
    """(T, 3, H, W) fp32 -> (grid_t gh gw, 1176) rows in HF order, the last frame repeated to an even T."""
    T, C, H, W = frames_chw.shape
    if T % TEMPORAL:
        frames_chw = np.concatenate([frames_chw, np.repeat(frames_chw[-1:], TEMPORAL - T % TEMPORAL, 0)], 0)
    gt, gh, gw = frames_chw.shape[0] // TEMPORAL, H // PATCH, W // PATCH
    p = frames_chw.reshape(gt, TEMPORAL, C, gh // MERGE, MERGE, PATCH, gw // MERGE, MERGE, PATCH)
    p = p.transpose(0, 3, 6, 4, 7, 2, 1, 5, 8)
    return np.ascontiguousarray(p.reshape(gt * gh * gw, C * TEMPORAL * PATCH * PATCH)), (gt, gh, gw)


def preprocess(videos_thwc, min_pixels=MIN_PIXELS, max_pixels=MAX_PIXELS, cuda=False, mean=OPENAI_CLIP_MEAN,
               std=OPENAI_CLIP_STD):
    """List of (T, H, W, 3) uint8 arrays -> (pixel_values_videos (S, 1176) f32, video_grid_thw (N, 3) i64).
    ``cuda``: the resize of a processor called with ``device="cuda"`` (torch's fp32 path)."""
    lut = normalize_lut(mean, std)
    resize = resample_torchvision_cuda.resize_u8 if cuda else resample_torchvision.resize_u8
    rows, grids = [], []
    for v in videos_thwc:
        _, h, w, _ = v.shape
        rh, rw = geometry.smart_resize(h, w, PATCH * MERGE, min_pixels, max_pixels)
        frames = np.stack([resize(f, rw, rh) for f in v], 0)                         # (T, rh, rw, 3) uint8
        f32 = np.stack([lut[c][frames[..., c]] for c in range(3)], axis=1)            # (T, 3, rh, rw)
        pv, g = patchify_video(f32)
        rows.append(pv)
        grids.append(g)
    return np.concatenate(rows, 0), np.array(grids, dtype=np.int64)
