"""Oracle: the image branch of the HF Qwen2-VL processor, torchvision backend.  Test infrastructure only.

Follows HF ``models/qwen2_vl/image_processing_qwen2_vl.py`` (``Qwen2VLImageProcessor._preprocess``, the class
``AutoImageProcessor`` returns on transformers 5.x when torchvision is installed) and
``image_processing_backends.py`` ``TorchvisionBackend.rescale_and_normalize``: the rescale is folded into the
statistics, ``mean' = f32(mean) * f32(1 / rescale)``, ``std'`` likewise, then ``(f32(v) - mean') / std'`` in fp32.
The resize is the NumPy restatement in ``oracle.resample_torchvision``; geometry and patch order are those of the
PIL backend (``oracle.processor``).
"""
import numpy as np

from . import geometry, resample_torchvision
from .processor import MERGE, OPENAI_CLIP_MEAN, OPENAI_CLIP_STD, PATCH, patchify


def normalize_lut(mean=OPENAI_CLIP_MEAN, std=OPENAI_CLIP_STD, rescale=1 / 255):
    """(3, 256) f32 table of HF's fused rescale + normalize, every step rounded to f32."""
    inv = np.float32(1.0 / rescale)
    m = np.array(mean, dtype=np.float32) * inv
    s = np.array(std, dtype=np.float32) * inv
    v = np.arange(256, dtype=np.float32)
    return ((v[None, :] - m[:, None]) / s[:, None]).astype(np.float32)


def preprocess_u8(images_hwc, min_pixels=56 * 56, max_pixels=28 * 28 * 1280):
    """List of (H, W, 3) uint8 arrays -> (pixel_values (S,1176) f32, image_grid_thw (N,3) i64, resized u8 list)."""
    lut = normalize_lut()
    rows, grids, resized = [], [], []
    for img in images_hwc:
        h, w, _ = img.shape
        rh, rw = geometry.smart_resize(h, w, PATCH * MERGE, min_pixels, max_pixels)
        r = resample_torchvision.resize_u8(img, rw, rh)
        resized.append(r)
        f = np.stack([lut[c][r[:, :, c]] for c in range(3)], axis=0)
        pv, g = patchify(f)
        rows.append(pv)
        grids.append(g)
    return np.concatenate(rows, 0), np.array(grids, dtype=np.int64), resized
