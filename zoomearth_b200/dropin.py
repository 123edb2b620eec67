"""install(model, processor): swap the two reference-facing objects for the fused ones, in place.

After this, the reference's own scripts run unchanged on top of the drop-in: ``processor(text=..., images=...)``
(``src/eval/infer.py:102-107``, ``src/demo.py:7-12``) lands on FusedImageProcessor, and the LM forward's
``self.visual(pixel_values, grid_thw=...)`` (HF modeling_qwen2_5_vl.py:1172) lands on FusedVisual.  The module
path is ``model.visual`` on transformers 4.49 (what the reference pins) and ``model.model.visual`` on 5.x.

``image_backend`` picks the HF image-processor backend whose pixels the fused processor reproduces.  On transformers
5.x ``AutoProcessor`` hands Qwen2-VL / Qwen2.5-VL the torchvision backend whenever torchvision is installed, so a 5.x
user who wants the model to keep seeing the same ``pixel_values`` passes ``image_backend="match"``.
"""
import torch

from .processor import FusedImageProcessor
from .visual import FusedVisual


def _find_visual(model):
    for owner in (model, getattr(model, "model", None)):
        if owner is not None and hasattr(owner, "visual"):
            return owner
    raise AttributeError("no `.visual` / `.model.visual` on this model")


def _bicubic(resample):
    try:
        from torchvision.transforms import InterpolationMode
        if resample == InterpolationMode.BICUBIC:
            return True
    except ImportError:                     # pragma: no cover
        pass
    return isinstance(resample, int) and int(resample) == 3      # PILImageResampling.BICUBIC


def _image_backend(old, image_backend):
    """The FusedImageProcessor backend for ``install(..., image_backend=...)`` replacing the image processor ``old``."""
    if image_backend not in ("pil", "torchvision", "match"):
        raise ValueError(f"image_backend must be 'pil', 'torchvision' or 'match', got {image_backend!r}")
    if image_backend == "pil":
        return "pil"
    backend = image_backend
    if image_backend == "match":
        try:
            from transformers.image_processing_backends import PilBackend, TorchvisionBackend
        except ImportError:
            PilBackend = TorchvisionBackend = ()
        if TorchvisionBackend and isinstance(old, TorchvisionBackend):
            backend = "torchvision"
        elif PilBackend and isinstance(old, PilBackend):
            backend = "pil"
        else:
            raise ValueError(f"image_backend='match': cannot tell which backend {type(old).__name__} resamples with "
                             "(known: transformers 5.x TorchvisionBackend / PilBackend); pass 'pil' or 'torchvision'")
    resample = getattr(old, "resample", None)
    if not _bicubic(resample):
        raise NotImplementedError(f"{type(old).__name__} resamples with {resample!r}; the fused processor reproduces "
                                  "bicubic only")
    return backend


def install(model=None, processor=None, device=None, dtype=None, image_backend="pil"):
    """Returns (fused_visual or None, fused_image_processor or None).  ``image_backend``: "pil" (the default) matches
    HF's PIL backend; "torchvision" matches HF's torchvision backend; "match" reads which of the two
    ``processor.image_processor`` is (a transformers 5.x ``TorchvisionBackend`` or ``PilBackend`` instance, anything else
    is a ValueError).  Under "torchvision" / "match" a replaced processor that does not resample bicubic raises
    NotImplementedError."""
    fv = fp = None
    backend = _image_backend(processor.image_processor, image_backend) if processor is not None else None
    if model is not None:
        owner = _find_visual(model)
        hf_visual = owner.visual
        import transformers
        returns_struct = int(transformers.__version__.split(".")[0]) >= 5
        p = next(hf_visual.parameters())
        fv = FusedVisual.from_hf(hf_visual, device=device or (p.device if p.device.type == "cuda" else None),
                                 dtype=dtype or (p.dtype if p.dtype in (torch.float32, torch.bfloat16, torch.float16) else torch.float16),
                                 return_pooling_output=returns_struct)
        owner.visual = fv
    if processor is not None:
        old = processor.image_processor
        fp = FusedImageProcessor(size=dict(getattr(old, "size", None) or {}) or None,
                                 patch_size=getattr(old, "patch_size", 14),
                                 temporal_patch_size=getattr(old, "temporal_patch_size", 2),
                                 merge_size=getattr(old, "merge_size", 2),
                                 image_mean=getattr(old, "image_mean", None), image_std=getattr(old, "image_std", None),
                                 device=device, backend=backend)
        processor.image_processor = fp
    return fv, fp
