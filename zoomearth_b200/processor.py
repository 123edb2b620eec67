"""FusedImageProcessor - drop-in for the HF Qwen2-VL image processor, backed by the fused CUDA kernel K1.

Replaces ``processor.image_processor`` of ``Qwen2_5_VLProcessor`` (reference call sites
``src/eval/infer.py:102-107``, ``src/demo.py:7-12``): same call signature, same outputs
(``pixel_values (S,1176) float32``, ``image_grid_thw (N,3) int64``), same attributes the processor reads
(``merge_size`` HF processing_qwen2_5_vl.py:120, ``get_number_of_image_patches`` :168, ``model_input_names``).
What it replaces inside: HF ``models/qwen2_vl/image_processing_pil_qwen2_vl.py:143-224`` (smart_resize ->
Pillow bicubic -> rescale -> normalize -> patchify); results are bit-identical to that PIL backend.  With
``backend="torchvision"`` they are bit-identical to HF's torchvision backend instead
(``models/qwen2_vl/image_processing_qwen2_vl.py``, what ``AutoImageProcessor`` returns on transformers 5.x when
torchvision is installed): torch's uint8 antialiased bicubic and the fp32 fused rescale + normalize.  The device
kernels are the same; only the coefficient tables and the normalisation LUT differ.

Also the crop-aware entry ``preprocess_crops`` used by the zoom fast path: the source image stays resident on
the GPU as uint8 and every zoom step reads its crop box straight out of it (``Image.crop`` semantics of
``infer.py:72-75`` included, zero fill outside the image).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, geometry

try:                                        # BatchFeature is only a container; keep HF's when it is importable
    from transformers.feature_extraction_utils import BatchFeature
except Exception:                           # pragma: no cover
    class BatchFeature(dict):
        def __init__(self, data=None, tensor_type=None):
            super().__init__(data or {})

        def to(self, *a, **k):
            return BatchFeature({n: (v.to(*a, **k) if hasattr(v, "to") else v) for n, v in self.items()})

        def __getattr__(self, n):
            try:
                return self[n]
            except KeyError as e:
                raise AttributeError(n) from e


def _flatten(images):
    if isinstance(images, (list, tuple)):
        out = []
        for i in images:
            out.extend(_flatten(i))
        return out
    return [images]


def upload_u8(t_host, device, stream=None):
    """Host (H, W, 3) uint8 tensor -> resident CUDA image.  When the packed row pitch (3 W bytes) is not a multiple of 4 -
    three widths out of four - the image is stored with its rows padded to a multiple of 16 pixels and returned as a
    (H, W, 3) view of that buffer: K1's tensor-core route needs a row pitch that is a multiple of 4 bytes (zv_k1_tc.cuh),
    and with a multiple of 16 it needs a single coefficient variant.  Every entry point takes row-pitched views."""
    h, w = int(t_host.shape[0]), int(t_host.shape[1])
    if t_host.device.type != "cpu":
        return t_host
    src = t_host if t_host.is_pinned() else t_host.pin_memory()
    ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.device(device)
    with ctx:
        if w % 4 == 0:
            d = src.to(device, non_blocking=True)
        else:
            buf = torch.empty((h, (w + 15) // 16 * 16, 3), dtype=torch.uint8, device=device)
            d = buf[:, :w]
            d.copy_(src, non_blocking=True)
    d._zv_pinned_src = src                        # the pinned source must outlive the async copy
    return d


def _to_u8_hwc(image):
    """PIL / ndarray / tensor -> contiguous (H, W, 3) uint8 torch tensor on its current device."""
    if hasattr(image, "convert") and hasattr(image, "size"):          # PIL.Image
        image = np.asarray(image.convert("RGB"))
    if isinstance(image, np.ndarray):
        image = torch.from_numpy(np.ascontiguousarray(image))
    if not isinstance(image, torch.Tensor):
        raise TypeError(f"unsupported image type {type(image)}")
    if image.dtype != torch.uint8:
        # HF's PIL backend (image_transforms.py:127-151,196-202) takes any array whose values are whole numbers in
        # [0, 255] and casts it to uint8; arrays of floats in [0, 1] go through a rescale round trip there that the
        # reference never exercises (it feeds PIL images) - not part of the fused path
        f = image.to(torch.float64)
        if not torch.equal(f, f.round()):
            if bool((f >= 0).all()) and bool((f <= 1).all()):
                raise NotImplementedError("float images in [0, 1] are not part of the fused path; pass uint8 pixels")
            raise ValueError("The image to be converted to a PIL image contains values outside the range [0, 1], "
                             f"got [{f.min().item()}, {f.max().item()}] which cannot be converted to uint8.")
        if bool((f < 0).any()) or bool((f > 255).any()):
            raise ValueError("The image to be converted to a PIL image contains values outside the range [0, 255], "
                             f"got [{f.min().item()}, {f.max().item()}] which cannot be converted to uint8.")
        image = image.to(torch.uint8)
    if image.ndim == 2:
        image = image[..., None].expand(-1, -1, 3)
    if image.ndim != 3:
        raise ValueError(f"expected an (H, W, 3) or (3, H, W) image, got shape {tuple(image.shape)}")
    if image.shape[-1] != 3 and image.shape[0] == 3:
        image = image.permute(1, 2, 0)
    if image.shape[-1] != 3:
        raise ValueError(f"expected 3 channels, got shape {tuple(image.shape)}")
    return image.contiguous()


BACKENDS = {"pil": _lib.RESAMPLE_PIL, "torchvision": _lib.RESAMPLE_TORCHVISION}


class FusedImageProcessor:
    model_input_names = ["pixel_values", "image_grid_thw"]
    valid_kwargs = None

    def __init__(self, min_pixels=None, max_pixels=None, size=None, patch_size=14, temporal_patch_size=2,
                 merge_size=2, image_mean=None, image_std=None, rescale_factor=1 / 255, device=None,
                 output_device="cpu", backend="pil", **unused):
        """``backend``: which HF image-processor backend the pixels match bit for bit - "pil" (Qwen2VLImageProcessorPil)
        or "torchvision" (Qwen2VLImageProcessor).  It applies to ``preprocess`` / ``__call__`` and ``preprocess_crops``;
        ``resize_u8`` / ``cut_resize`` are the reference's own Pillow ``resize_image`` under either."""
        if backend not in BACKENDS:
            raise ValueError(f"backend must be one of {sorted(BACKENDS)}, got {backend!r}")
        self.backend = backend
        size = dict(size) if size is not None else {"shortest_edge": 56 * 56, "longest_edge": 28 * 28 * 1280}
        if min_pixels is not None:
            size["shortest_edge"] = min_pixels
        if max_pixels is not None:
            size["longest_edge"] = max_pixels
        if "shortest_edge" not in size or "longest_edge" not in size:
            raise ValueError("size must contain 'shortest_edge' and 'longest_edge' keys.")
        self.size = size
        self.patch_size, self.temporal_patch_size, self.merge_size = patch_size, temporal_patch_size, merge_size
        self.image_mean = list(image_mean) if image_mean is not None else [0.48145466, 0.4578275, 0.40821073]
        self.image_std = list(image_std) if image_std is not None else [0.26862954, 0.26130258, 0.27577711]
        self.rescale_factor = rescale_factor
        self.do_resize = self.do_rescale = self.do_normalize = self.do_convert_rgb = True
        self.device = torch.device(device) if device is not None else None
        self.output_device = output_device
        self._ws = None
        self.last_launches = 0

    # ---- attributes the reference's scripts set / read (qwen_module.py:40-41, grpo_trainer.py:311-315)
    @property
    def min_pixels(self):
        return self.size["shortest_edge"]

    @min_pixels.setter
    def min_pixels(self, v):
        self.size["shortest_edge"] = v

    @property
    def max_pixels(self):
        return self.size["longest_edge"]

    @max_pixels.setter
    def max_pixels(self, v):
        self.size["longest_edge"] = v

    def _cfg(self, min_pixels=None, max_pixels=None):
        return _lib.default_cfg(patch=self.patch_size, merge=self.merge_size, temporal=self.temporal_patch_size,
                                min_pixels=int(min_pixels if min_pixels is not None else self.min_pixels),
                                max_pixels=int(max_pixels if max_pixels is not None else self.max_pixels),
                                rescale=float(self.rescale_factor), mean=self.image_mean, std=self.image_std,
                                resample_kind=BACKENDS[self.backend])

    def _device(self):
        if self.device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("FusedImageProcessor needs a CUDA device (sm_100); there is no CPU fallback")
            self.device = torch.device("cuda", torch.cuda.current_device())
        return self.device

    def _workspace(self, nbytes, device):
        if self._ws is None or self._ws.numel() < nbytes or self._ws.device != device:
            self._ws = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        return self._ws

    def get_number_of_image_patches(self, height, width, images_kwargs=None):
        kw = images_kwargs or {}
        factor = self.patch_size * self.merge_size
        rh, rw = geometry.smart_resize(height, width, factor, kw.get("min_pixels", self.min_pixels),
                                       kw.get("max_pixels", self.max_pixels))
        return (rh // self.patch_size) * (rw // self.patch_size)

    # ---- device path
    def preprocess_crops(self, images_dev, boxes=None, out_dtype=torch.float32, window_order=False,
                         min_pixels=None, max_pixels=None, image_index=None, apply_cut_image=False, out=None):
        """images_dev: list of (H, W, 3) uint8 CUDA tensors.  boxes: (n, 4) crop boxes (x0, y0, x1, y1) in image
        pixels, or None for the whole image; ``image_index[i]`` says which image crop i reads (default i).
        ``apply_cut_image`` first maps each box through the reference's cut_image() rule (min 512 px).
        Returns (patches (S, 1176) out_dtype on the GPU, image_grid_thw (n, 3) int64 CPU tensor, crop boxes)."""
        cfg = self._cfg(min_pixels, max_pixels)
        device = images_dev[0].device
        if device.type != "cuda":
            raise RuntimeError("preprocess_crops takes CUDA tensors; there is no CPU path")
        n = len(images_dev) if boxes is None else len(boxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        img_hw = np.array([[images_dev[i].shape[0], images_dev[i].shape[1]] for i in idx], np.int32)
        if boxes is None:
            crop, rhw, grid = geometry.geometry(cfg, img_hw, None)
        elif apply_cut_image:
            crop, rhw, grid = geometry.geometry(cfg, img_hw, np.asarray(boxes, np.float64))
        else:
            # final crop boxes, PIL.Image.crop semantics: int(round(v)) with Python's round-half-even
            bx = np.rint(np.asarray(boxes, np.float64)).astype(np.int64).reshape(n, 4)
            cfg0 = self._cfg(min_pixels, max_pixels)
            cfg0.min_size = -1                     # boxes are final crop boxes: no cut_image rule
            crop, rhw, grid = geometry.geometry(cfg0, img_hw, bx.astype(np.float64))
        S = int((grid[:, 1] * grid[:, 2]).sum())
        lib = _lib.lib()
        ws_bytes = _lib.check(lib.zv_preprocess_workspace_bytes(n, crop.ctypes.data, rhw.ctypes.data))
        ws = self._workspace(ws_bytes, device)
        if out is None:
            out = torch.empty((S, 1176), dtype=out_dtype, device=device)
        elif out.shape != (S, 1176) or out.dtype != out_dtype or not out.is_contiguous():
            raise ValueError("preprocess_crops: `out` has the wrong shape/dtype")
        ptrs = (C.c_void_p * n)(*[images_dev[i].data_ptr() for i in idx])
        pitch = np.array([images_dev[i].stride(0) for i in idx], np.int64)
        for i in idx:
            t = images_dev[i]
            if t.dtype != torch.uint8 or t.ndim != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
                raise ValueError("images must be (H, W, 3) uint8 CUDA tensors with packed pixels")
        stream = torch.cuda.current_stream(device).cuda_stream
        with torch.cuda.device(device):
            _lib.check(lib.zv_preprocess(
                C.byref(cfg), n, ptrs, img_hw.ctypes.data, pitch.ctypes.data, crop.ctypes.data, rhw.ctypes.data, None,
                out.data_ptr(), {torch.float32: _lib.ZV_F32, torch.bfloat16: _lib.ZV_BF16, torch.float16: _lib.ZV_F16}[out_dtype],
                _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF, ws.data_ptr(), ws.numel(), stream))
        self.last_launches = lib.zv_last_launch_count()
        return out, torch.from_numpy(grid), crop

    # ---- the reference's cut_image / resize_image on the device (uint8 in, uint8 out, Pillow-exact)
    def resize_u8(self, images_dev, boxes, out_wh, image_index=None):
        """``PIL.Image.crop(box).resize((w, h), Image.BICUBIC)`` for n (image, box, size) triples in one call of
        ``zv_resize_u8``.  images_dev: (H, W, 3) uint8 CUDA tensors (row-pitched views are fine); boxes (n, 4) ints
        (x0, y0, x1, y1), may reach outside the image (zero fill, like Image.crop); out_wh (n, 2) (w, h).
        Returns a list of n contiguous (h, w, 3) uint8 CUDA tensors."""
        n = len(boxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        device = images_dev[0].device
        if device.type != "cuda":
            raise RuntimeError("resize_u8 takes CUDA tensors; there is no CPU path")
        crop = np.ascontiguousarray(np.asarray(boxes, np.int64).reshape(n, 4).astype(np.int32))
        if (crop[:, 2] < crop[:, 0]).any():
            raise ValueError("Coordinate 'right' is less than 'left'")
        if (crop[:, 3] < crop[:, 1]).any():
            raise ValueError("Coordinate 'lower' is less than 'upper'")
        out_hw = np.ascontiguousarray(np.asarray(out_wh, np.int64).reshape(n, 2)[:, ::-1].astype(np.int32))
        img_hw = np.array([[images_dev[i].shape[0], images_dev[i].shape[1]] for i in idx], np.int32)
        for i in idx:
            t = images_dev[i]
            if t.dtype != torch.uint8 or t.ndim != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
                raise ValueError("images must be (H, W, 3) uint8 CUDA tensors with packed pixels")
        lib = _lib.lib()
        ws_bytes = _lib.check(lib.zv_resize_u8_workspace_bytes(n, crop.ctypes.data, out_hw.ctypes.data))
        ws = self._workspace(ws_bytes, device)
        outs = [torch.empty((int(h), int(w), 3), dtype=torch.uint8, device=device) for h, w in out_hw]
        src = (C.c_void_p * n)(*[images_dev[i].data_ptr() for i in idx])
        pitch = np.array([images_dev[i].stride(0) for i in idx], np.int64)
        dst = (C.c_void_p * n)(*[o.data_ptr() for o in outs])
        dpitch = np.array([o.stride(0) for o in outs], np.int64)
        stream = torch.cuda.current_stream(device).cuda_stream
        with torch.cuda.device(device):
            _lib.check(lib.zv_resize_u8(n, src, img_hw.ctypes.data, pitch.ctypes.data, crop.ctypes.data, out_hw.ctypes.data,
                                        dst, dpitch.ctypes.data, ws.data_ptr(), ws.numel(), stream))
        self.last_launches = lib.zv_last_launch_count()
        return outs

    def cut_resize(self, images_dev, bboxes=None, image_index=None, variant="infer", max_size=None, min_size=512,
                   apply_cut_image=True):
        """``resize_image(cut_image(image, bbox))`` of the reference on the device, for a batch: what infer.py:215,239 /
        demo.py:133,140 / SFT.py:159-169 / grpo_trainer.py:530,606 hand to the processor.  ``bboxes`` None = the global
        view (``resize_image(image)``).  ``max_size`` 0 = cut_image only.  Returns (list of uint8 CUDA images, list of
        1/scale) - pixels bit-identical to Pillow's.  Crops that need no resampling at all come back as views.
        ``apply_cut_image=False``: ``bboxes`` are final crop boxes (``Image.crop`` semantics) instead of model boxes."""
        n = len(images_dev) if bboxes is None else len(bboxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        if max_size is None:
            max_size = geometry.DEFAULT_MAX_SIZE[variant]
        cur = [images_dev[i] for i in idx]                    # per item: the image its next step reads
        plans, inv = [], [1.0] * n
        for k in range(n):                                    # the whole chain of Pillow calls, sizes known up front
            w, h = int(cur[k].shape[1]), int(cur[k].shape[0])
            if bboxes is None:
                ops = []
            elif apply_cut_image:
                ops = geometry.cut_ops(w, h, bboxes[k], min_size, variant)
            else:                                             # final crop boxes, PIL.Image.crop rounding
                ops = [["crop", [int(v) for v in np.rint(np.asarray(bboxes[k], np.float64))]]]
            for kind, arg in ops:
                w, h = (arg[2] - arg[0], arg[3] - arg[1]) if kind == "crop" else (arg[0], arg[1])
            if max_size:
                nw, nh, inv[k] = geometry.resize_dims_ex(w, h, max_size, variant)
                if (nw, nh) != (w, h) or variant == "sft":
                    ops = ops + [["resize", [nw, nh]]]
            plans.append(ops)
        # a crop followed by a resize is ONE item of a zv_resize_u8 call (infer.py's whole chain); a lone crop is a view,
        # or a same-size zero-filled copy when it leaves the image; at most three rounds (SFT's crop-resize-crop + resize)
        while any(plans):
            todo = []
            for k in range(n):
                ops = plans[k]
                if not ops:
                    continue
                h, w = int(cur[k].shape[0]), int(cur[k].shape[1])
                kind, arg = ops[0]
                if kind == "resize":
                    todo.append((k, [0, 0, w, h], arg))
                    plans[k] = ops[1:]
                elif len(ops) > 1 and ops[1][0] == "resize":
                    todo.append((k, arg, ops[1][1]))
                    plans[k] = ops[2:]
                elif 0 <= arg[0] <= arg[2] <= w and 0 <= arg[1] <= arg[3] <= h:
                    cur[k] = cur[k][arg[1]:arg[3], arg[0]:arg[2]]
                    plans[k] = ops[1:]
                else:
                    todo.append((k, arg, [arg[2] - arg[0], arg[3] - arg[1]]))
                    plans[k] = ops[1:]
            if todo:
                outs = self.resize_u8([cur[k] for k, _, _ in todo], [b for _, b, _ in todo], [s for _, _, s in todo])
                for (k, _, _), o in zip(todo, outs):
                    cur[k] = o
        return cur, inv

    # ---- HF surface
    def preprocess(self, images, videos=None, return_tensors=None, min_pixels=None, max_pixels=None, size=None,
                   do_resize=None, do_rescale=None, do_normalize=None, **unused):
        if videos is not None:
            raise NotImplementedError("FusedImageProcessor covers the image branch only (the reference uses no video)")
        for name, flag in (("do_resize", do_resize), ("do_rescale", do_rescale), ("do_normalize", do_normalize)):
            if flag is False:
                raise NotImplementedError(f"{name}=False is not part of the fused path")
        if size is not None:
            min_pixels = size.get("shortest_edge", min_pixels)
            max_pixels = size.get("longest_edge", max_pixels)
        device = self._device()
        imgs = [_to_u8_hwc(i) for i in _flatten(images)]
        if not imgs:
            raise ValueError("no images given")
        dev_imgs = [upload_u8(t, device) for t in imgs]
        pv, grid, _ = self.preprocess_crops(dev_imgs, None, torch.float32, False, min_pixels, max_pixels)
        if self.output_device == "cpu":
            pv = pv.cpu()
        data = {"pixel_values": pv, "image_grid_thw": grid}
        if return_tensors in ("np", "numpy"):
            data = {k: v.cpu().numpy() for k, v in data.items()}
        elif return_tensors not in (None, "pt", "torch"):
            raise ValueError(f"unsupported return_tensors={return_tensors!r}")
        return BatchFeature(data=data)

    def __call__(self, images, **kwargs):
        return self.preprocess(images, **kwargs)
