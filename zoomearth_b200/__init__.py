"""zoomearth_b200 - B200-native drop-in for ZoomEarth's per-zoom-step vision path.

crop -> Pillow-exact bicubic smart_resize -> normalize -> patchify (K1) and the Qwen2.5-VL vision tower
(tcgen05 GEMMs, varlen attention) behind the reference's own surfaces.  Python here is plumbing over the
C ABI in ``include/zoomvit.h``; the CUDA library is mandatory (no fallback path).
"""
from . import _lib, geometry                                    # noqa: F401
from .geometry import cut_box, extract_bbox, resize_dims, smart_resize   # noqa: F401


def __getattr__(name):            # torch-dependent pieces are imported lazily
    if name == "FusedImageProcessor":
        from .processor import FusedImageProcessor
        return FusedImageProcessor
    if name == "FusedVideoProcessor":
        from .video import FusedVideoProcessor
        return FusedVideoProcessor
    if name == "FusedVisual":
        from .visual import FusedVisual
        return FusedVisual
    if name == "ZoomEncoder":
        from .zoom import ZoomEncoder
        return ZoomEncoder
    if name == "ZoomSession":
        from .session import ZoomSession
        return ZoomSession
    if name == "install":
        from .dropin import install
        return install
    if name in ("get_rope_index", "embed_images", "placeholder_rows", "DeviceHandoff"):
        from . import handoff
        return getattr(handoff, name)
    if name == "Plan":
        from .plan import Plan
        return Plan
    raise AttributeError(name)
