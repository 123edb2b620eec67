"""The fused zoom step: crop box -> patches (bf16, window order) -> vision tower -> merged embeddings.

This is the fast path behind the reference's zoom loop (``src/eval/infer.py:236-247``: re-open image ->
``cut_image`` -> ``resize_image`` -> processor -> ``model.visual``): the decoded image is uploaded once and
stays resident on the GPU as uint8; every zoom step is two library calls (``zv_preprocess`` straight out of
the resident pixels, ``zv_visual_forward``) with no host round trip of pixel data.  Crops are independent, so
``encode`` takes any number of (image, box) pairs as one ragged batch.
"""
import numpy as np
import torch

from .processor import FusedImageProcessor
from .visual import FusedVisual


def proc_min_size(proc):
    """cut_image()'s min_size (512 at every call site of the reference)."""
    return getattr(proc, "cut_min_size", 512)


class ZoomEncoder:
    def __init__(self, visual: FusedVisual, processor: FusedImageProcessor = None, max_pixels=128 * 128 * 28 * 28,
                 min_pixels=56 * 56, pre_resize=None):
        """``pre_resize``: None = the fused single-resample step (crop -> smart_resize straight from the source pixels);
        a call-site name - "infer" (512), "demo" (1024), "sft" (1024), "custom" (512) - or a (name, max_size) pair = the
        reference-faithful TWO-resample flow: ``resize_image(cut_image(image, bbox))`` as uint8 on the device
        (``zv_resize_u8``, infer.py:215,239 / demo.py:133,140), then the processor's smart_resize on that image
        (``zv_preprocess``) - bit-identical to what the unmodified scripts feed the tower, with no host trip."""
        self.visual = visual
        self.processor = processor or FusedImageProcessor(min_pixels=min_pixels, max_pixels=max_pixels,
                                                          device=visual.device)
        self.pre_resize = self._norm_pre_resize(pre_resize)
        self.last_launches = 0
        self.last_inv_scales = None

    @staticmethod
    def _norm_pre_resize(pre_resize):
        from . import geometry
        if pre_resize is None:
            return None
        if isinstance(pre_resize, str):
            pre_resize = (pre_resize, geometry.DEFAULT_MAX_SIZE[pre_resize])
        variant, max_size = pre_resize
        if variant not in geometry.RESIZE_MODE:
            raise ValueError(f"pre_resize variant must be one of {sorted(geometry.RESIZE_MODE)}")
        return variant, int(max_size)

    def _patches(self, images_dev, boxes, image_index, apply_cut_image, pre_resize):
        """-> (patches in window order, image_grid_thw, crop boxes in source pixels, K1 launches)."""
        proc = self.processor
        if pre_resize is None:
            pv, grid, crop = proc.preprocess_crops(
                images_dev, boxes, out_dtype=self.visual.operand_dtype, window_order=True, image_index=image_index,
                apply_cut_image=apply_cut_image and boxes is not None)
            self.last_inv_scales = None
            return pv, grid, crop, proc.last_launches
        variant, max_size = pre_resize
        n = len(images_dev) if boxes is None else len(boxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        imgs, inv = proc.cut_resize(images_dev, boxes, image_index, variant, max_size, proc_min_size(proc), apply_cut_image)
        launches = proc.last_launches if any(i is not images_dev[j] for i, j in zip(imgs, idx)) else 0
        pv, grid, _ = proc.preprocess_crops(imgs, None, out_dtype=self.visual.operand_dtype, window_order=True)
        self.last_inv_scales = inv
        from . import geometry
        crop = np.zeros((n, 4), np.int32)
        for k in range(n):
            t = images_dev[idx[k]]
            if boxes is None:
                crop[k] = (0, 0, t.shape[1], t.shape[0])
            elif apply_cut_image:
                ops = geometry.cut_ops(int(t.shape[1]), int(t.shape[0]), boxes[k], proc_min_size(proc), variant)
                crop[k] = ops[0][1] if ops else (0, 0, t.shape[1], t.shape[0])
            else:
                crop[k] = np.rint(np.asarray(boxes[k], np.float64)).astype(np.int32)
        return pv, grid, crop, launches + proc.last_launches

    def upload(self, image):
        """PIL / (H, W, 3) uint8 array or tensor -> resident uint8 CUDA tensor (one H2D copy per image)."""
        from .processor import _to_u8_hwc, upload_u8
        return upload_u8(_to_u8_hwc(image), self.visual.device)     # rows padded when 3 W is not a multiple of 4 (a view comes back)

    @torch.no_grad()
    def encode(self, images_dev, boxes=None, image_index=None, apply_cut_image=True, return_patches=False,
               gather=None, gather_row=0, use_graph=False, pre_resize="default", gather_rows=None):
        """images_dev: resident images; boxes (n, 4) in image pixels (None = global view of every image).
        Returns (embeddings (T, out_hidden), image_grid_thw (n, 3), crop boxes (n, 4)).  ``pre_resize`` overrides the
        encoder's setting for this call (see ``__init__``)."""
        pr = self.pre_resize if isinstance(pre_resize, str) and pre_resize == "default" else self._norm_pre_resize(pre_resize)
        pv, grid, crop, k1 = self._patches(images_dev, boxes, image_index, apply_cut_image, pr)
        emb = self.visual(pv, grid, window_order=True, gather=gather, gather_row=gather_row, use_graph=use_graph,
                          gather_rows=gather_rows)
        self.last_launches = k1 + self.visual.last_launches
        if return_patches:
            return emb, grid, crop, pv
        return emb, grid, crop

    @torch.no_grad()
    def encode_video(self, videos_dev, min_pixels=None, max_pixels=None, backend="torchvision_cuda", use_graph=False,
                     return_patches=False):
        """The device-resident video path: videos_dev, a list of (T, H, W, 3) uint8 CUDA tensors, -> window-ordered
        16-bit patches (``zv_preprocess_video``, every frame in one call) -> the tower.  ``backend`` picks the resampling
        HF's video processor would run: "torchvision_cuda" (frames on a CUDA device, the default here) or "torchvision"
        (the CPU).  ``min_pixels`` / ``max_pixels`` default to the video processor's (128 / 768 x 28^2).
        Returns (embeddings (T, out_hidden) in HF order, video_grid_thw (n, 3))."""
        if not hasattr(self, "video_processor"):
            from .video import FusedVideoProcessor
            self.video_processor = FusedVideoProcessor(device=self.visual.device, backend=backend)
        vp = self.video_processor
        pv, grid = vp.preprocess_videos(videos_dev, out_dtype=self.visual.operand_dtype, window_order=True,
                                        min_pixels=min_pixels, max_pixels=max_pixels, backend=backend)
        emb = self.visual(pv, grid, window_order=True, use_graph=use_graph)
        self.last_launches = vp.last_launches + self.visual.last_launches
        if return_patches:
            return emb, grid, pv
        return emb, grid

    def micro_batches(self, images_dev, boxes, image_index=None, max_patches=400_000, apply_cut_image=True):
        """Splits a ragged crop list into consecutive micro-batches of at most ``max_patches`` patches (a crop larger
        than the budget is a batch of its own), so the tower's workspace stays bounded whatever the batch
        (the reference feeds one question at a time, infer.py:232-247; here hundreds go in one call).
        Returns a list of index lists into ``boxes``."""
        from . import geometry
        n = len(images_dev) if boxes is None else len(boxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        cfg = self.processor._cfg()
        if boxes is None or not apply_cut_image:
            cfg.min_size = -1
        img_hw = np.array([[images_dev[i].shape[0], images_dev[i].shape[1]] for i in idx], np.int32)
        bx = None if boxes is None else np.asarray(boxes, np.float64).reshape(n, 4)
        _, _, grid = geometry.geometry(cfg, img_hw, bx)
        patches = grid[:, 1] * grid[:, 2]
        out, cur, tot = [], [], 0
        for i, s in enumerate(patches):
            if cur and tot + int(s) > max_patches:
                out.append(cur)
                cur, tot = [], 0
            cur.append(i)
            tot += int(s)
        if cur:
            out.append(cur)
        return out

    @torch.no_grad()
    def encode_batched(self, images_dev, boxes=None, image_index=None, max_patches=400_000, apply_cut_image=True,
                       out=None):
        """``encode`` over micro-batches of at most ``max_patches`` patches; embeddings land back to back in one
        tensor, in the order of ``boxes``.  Returns (embeddings, image_grid_thw, crop boxes)."""
        n = len(images_dev) if boxes is None else len(boxes)
        idx = list(range(n)) if image_index is None else list(image_index)
        groups = self.micro_batches(images_dev, boxes, image_index, max_patches, apply_cut_image)
        embs, grids, crops, launches = [], [], [], 0
        for g in groups:
            used = sorted({idx[i] for i in g})
            local = {k: j for j, k in enumerate(used)}
            e, grid, crop = self.encode([images_dev[k] for k in used],
                                        None if boxes is None else [boxes[i] for i in g],
                                        image_index=[local[idx[i]] for i in g], apply_cut_image=apply_cut_image)
            launches += self.last_launches
            embs.append(e); grids.append(grid); crops.append(crop)
        self.last_launches = launches
        if out is None:
            out = torch.cat(embs, 0) if len(embs) > 1 else embs[0]
        else:
            row = 0
            for e in embs:
                out[row:row + e.shape[0]].copy_(e)
                row += e.shape[0]
        return out, torch.cat(grids, 0), np.concatenate(crops, 0)

    @torch.no_grad()
    def encode_host(self, host_images, chunk=8, out_host=None, schedule=None):
        """Global views of HOST images (pinned (H, W, 3) uint8 tensors), pipelined: the pixels of chunk i+1 are
        copied to the GPU on a side stream while chunk i runs through K1 + the tower, and the embeddings of chunk i
        go back to `out_host` (pinned) behind the compute.  Returns (out_host, image_grid_thw).  This is the ingest
        half of the reference loop (`Image.open(...)` -> processor -> `.to(device)`, infer.py:215-223) with the
        copy moved upstream to the raw uint8 pixels."""
        dev = self.visual.device
        compute = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(dev)
            self._d2h_stream = torch.cuda.Stream(dev)
        # a short first chunk keeps the exposed (un-overlapped) first upload small
        # (`schedule`: explicit chunk sizes instead, e.g. a ramp [2, 6, 8, 16, 32]; the last size repeats)
        if schedule:
            groups, i = [], 0
            for k in range(len(host_images)):
                if i >= len(host_images):
                    break
                n = schedule[min(k, len(schedule) - 1)]
                groups.append(host_images[i:i + n])
                i += n
        else:
            first = max(1, chunk // 4) if len(host_images) > chunk else len(host_images)
            groups = [host_images[:first]] + [host_images[i:i + chunk] for i in range(first, len(host_images), chunk)]
        staged = []

        def stage(g):
            with torch.cuda.stream(self._copy_stream):
                t = [h.to(dev, non_blocking=True) for h in g]
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            return t, ev

        staged.append(stage(groups[0]))
        grids, row, launches, keep = [], 0, 0, []
        for i in range(len(groups)):
            imgs, ev = staged[i]
            compute.wait_event(ev)
            for t in imgs:
                t.record_stream(compute)
            emb, grid, _ = self.encode(imgs, None)
            # stage the next chunk only now: the small table uploads of this chunk's kernels must not queue behind a
            # gigabyte of pixels on the host-to-device copy engine
            if i + 1 < len(groups):
                staged.append(stage(groups[i + 1]))
            launches += self.last_launches
            grids.append(grid)
            if out_host is None:
                tokens = sum(self.processor.get_number_of_image_patches(int(h.shape[0]), int(h.shape[1])) for h in host_images)
                out_host = torch.empty((tokens // self.visual.spatial_merge_unit, emb.shape[1]), dtype=emb.dtype).pin_memory()
            done = torch.cuda.Event()
            done.record(compute)
            with torch.cuda.stream(self._d2h_stream):
                self._d2h_stream.wait_event(done)
                out_host[row:row + emb.shape[0]].copy_(emb, non_blocking=True)
                emb.record_stream(self._d2h_stream)
            keep.append(emb)
            row += emb.shape[0]
        self._d2h_stream.synchronize()
        self.last_launches = launches
        return out_host[:row], torch.cat(grids, 0)

    def tokens_per_crop(self, grid_thw):
        g = np.asarray(grid_thw)
        return (g[:, 0] * g[:, 1] * g[:, 2]) // (self.visual.spatial_merge_unit)
