"""LM hand-off (SURVEY 8f-2): what sits between ``model.visual`` and the language model in the reference.

  get_rope_index    reference src/train/RL/src/open-r1-multimodal/src/open_r1/model/modeling_qwen2_vl.py:967-1114
                    (same signature; by ``hf5_semantics`` the transformers 5.x variant, HF modeling_qwen2_5_vl.py:1024-1135)
  embed_images      reference .../modeling_qwen2_vl.py:1191-1207 / HF modeling_qwen2_5_vl.py:1301-1307:
                    ``inputs_embeds.masked_scatter(image_mask, visual(pixel_values, grid_thw))`` - here the tower's last
                    GEMM writes every embedding row straight into its placeholder row of ``inputs_embeds``
                    (``zv_visual_forward_into``), so the (T, 2048) tensor never makes a round trip through HBM.

The position index is host integer work in libzoomvit (``zv_rope_index``); both are thin ctypes calls.
``DeviceHandoff`` does the same two computations as kernels (``zv_rope_index_dev``, ``zv_placeholder_rows_dev``) with no
host synchronisation, so that a zoom step's hand-off and tower can be captured in one CUDA graph.
"""
import ctypes as C
from collections import OrderedDict

import numpy as np
import torch

from . import _lib

IMAGE_TOKEN_ID, VIDEO_TOKEN_ID, VISION_START_TOKEN_ID = 151655, 151656, 151652      # Qwen2.5-VL tokenizer


def get_rope_index(input_ids, image_grid_thw=None, video_grid_thw=None, attention_mask=None, *, spatial_merge_size=2,
                   image_token_id=IMAGE_TOKEN_ID, video_token_id=VIDEO_TOKEN_ID,
                   vision_start_token_id=VISION_START_TOKEN_ID, hf5_semantics=False):
    """-> (position_ids (3, B, L) int64, mrope_position_deltas (B, 1) int64), on ``input_ids``' device."""
    if video_grid_thw is not None:
        raise NotImplementedError("get_rope_index covers images only (the reference's zoom loop feeds no video)")
    dev = input_ids.device
    ids = np.ascontiguousarray(input_ids.detach().cpu().numpy().astype(np.int64))
    if ids.ndim != 2:
        raise ValueError("input_ids must be (batch, seq_len)")
    B, L = ids.shape
    mask = None if attention_mask is None else np.ascontiguousarray(attention_mask.detach().cpu().numpy().astype(np.int64))
    grid = None if image_grid_thw is None else np.ascontiguousarray(
        np.asarray(image_grid_thw.detach().cpu() if isinstance(image_grid_thw, torch.Tensor) else image_grid_thw,
                   dtype=np.int64).reshape(-1, 3))
    pos = np.empty((3, B, L), np.int64)
    delta = np.empty((B, 1), np.int64)
    _lib.check(_lib.lib().zv_rope_index(
        ids.ctypes.data, None if mask is None else mask.ctypes.data, B, L, None if grid is None else grid.ctypes.data,
        0 if grid is None else grid.shape[0], image_token_id, video_token_id, vision_start_token_id, spatial_merge_size,
        1 if hf5_semantics else 0, pos.ctypes.data, delta.ctypes.data))
    return torch.from_numpy(pos).to(dev), torch.from_numpy(delta).to(dev)


def placeholder_rows(input_ids, image_token_id=IMAGE_TOKEN_ID, expected=None):
    """Flattened row indices of the image placeholders (int64 tensor on ``input_ids``' device), in masked_scatter
    order.  ``expected`` = the number of embeddings: a mismatch raises the ValueError HF raises (one host sync)."""
    flat = input_ids.reshape(-1)
    if flat.device.type == "cpu":
        ids = np.ascontiguousarray(flat.numpy().astype(np.int64))
        n = _lib.check(_lib.lib().zv_placeholder_rows(ids.ctypes.data, ids.size, image_token_id, None, 0))
        rows = np.empty(n, np.int64)
        _lib.check(_lib.lib().zv_placeholder_rows(ids.ctypes.data, ids.size, image_token_id, rows.ctypes.data, n))
        rows = torch.from_numpy(rows)
    else:
        rows = torch.nonzero(flat == image_token_id).reshape(-1)
    if expected is not None and rows.numel() != expected:
        raise ValueError(f"Image features and image tokens do not match, tokens: {rows.numel()}, features: {expected}")
    return rows


@torch.no_grad()
def embed_images(visual, inputs_embeds, input_ids, pixel_values, image_grid_thw, image_token_id=IMAGE_TOKEN_ID,
                 window_order=False):
    """In place: ``inputs_embeds`` (B, L, D) gets the tower's embeddings at its image-placeholder rows.  ``visual`` is
    a ``FusedVisual``; ``pixel_values`` as for ``visual.forward`` (HF-order fp32/16-bit patches, or the fused
    preprocess output with ``window_order=True``).  Returns ``inputs_embeds``."""
    plan = visual.plan_for(image_grid_thw)
    rows = placeholder_rows(input_ids, image_token_id, expected=plan.num_tokens).to(visual.device)
    return visual.forward_into(inputs_embeds, rows, pixel_values, image_grid_thw, window_order=window_order)


# zv_rope_index's messages (csrc/zv_handoff.cpp) by the check the device path records (ZV_HANDOFF_* in zoomvit.h)
_ROPE_ERRORS = {
    1: "zv_rope_index: sample {s} holds a video placeholder; only images are supported",
    2: "zv_rope_index: sample {s} ends with a vision-start token",
    3: "zv_rope_index: sample {s} has fewer image placeholders than images",
    4: "zv_rope_index: image_grid_thw has {a} rows, the batch needs more",
    5: "zv_rope_index: image {a} has an empty grid",
    6: "zv_rope_index: sample {s}: {a} positions for {b} tokens (placeholder count does not match image_grid_thw)",
    7: "zv_rope_index: sample {s} is fully masked",
}
_ROWS_COUNT = 8


class DeviceHandoff:
    """``get_rope_index``, ``placeholder_rows`` and ``embed_images`` on the device, for batches of up to ``max_batch`` x
    ``max_seq_len`` tokens.  Every call only enqueues work on the current stream: no host synchronisation and, once warmed
    up, no device allocation beyond the outputs torch's caching allocator hands out, so a zoom step's hand-off can be
    captured in one ``torch.cuda.graph`` together with ``FusedVisual.forward_into``.  Results equal the host functions'.

    Errors the host functions raise at once are recorded on the device instead; ``check()`` - the one synchronising
    method - raises them with the host path's exception and text.  Each of ``rope_index`` and ``placeholder_rows``
    overwrites its own record, so call ``check()`` after the step's calls.  Image grids given on the host are uploaded
    once per distinct content and then reused (a graph captured after one eager call replays without any copy)."""

    def __init__(self, device, max_batch, max_seq_len):
        self.device = torch.device(device)
        self.max_batch, self.max_seq_len = int(max_batch), int(max_seq_len)
        nbytes = _lib.check(_lib.lib().zv_handoff_workspace_bytes(self.max_batch, self.max_seq_len))
        self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._status = torch.zeros(8, dtype=torch.int64, device=self.device)   # [0:4] rope index, [4:8] placeholder rows
        self._rows_status = self._status[4:]
        self._grids = OrderedDict()        # grid bytes -> (pinned host copy, device copy)
        self.last_launches = 0

    def _tokens(self, t, name):
        if not isinstance(t, torch.Tensor) or t.device != self.device or t.dim() != 2:
            raise ValueError(f"{name} must be a (batch, seq_len) tensor on {self.device}")
        if t.shape[0] > self.max_batch or t.shape[1] > self.max_seq_len:
            raise ValueError(f"{name} is {tuple(t.shape)}; this DeviceHandoff holds up to ({self.max_batch}, {self.max_seq_len})")
        return t.to(torch.int64).contiguous()

    def _grid(self, grid):
        if isinstance(grid, torch.Tensor) and grid.device == self.device:
            return grid.to(torch.int64).reshape(-1, 3).contiguous()
        g = np.ascontiguousarray(np.asarray(grid.cpu() if isinstance(grid, torch.Tensor) else grid, dtype=np.int64).reshape(-1, 3))
        key = g.tobytes()
        ent = self._grids.get(key)
        if ent is None:
            host = torch.from_numpy(g).pin_memory()
            ent = (host, host.to(self.device, non_blocking=True))
            self._grids[key] = ent
            if len(self._grids) > 64:
                self._grids.popitem(last=False)
        else:
            self._grids.move_to_end(key)
        return ent[1]

    def rope_index(self, input_ids, image_grid_thw=None, attention_mask=None, *, video_grid_thw=None, spatial_merge_size=2,
                   image_token_id=IMAGE_TOKEN_ID, video_token_id=VIDEO_TOKEN_ID, vision_start_token_id=VISION_START_TOKEN_ID,
                   hf5_semantics=False):
        """-> (position_ids (3, B, L) int64, mrope_position_deltas (B, 1) int64) on the device, as ``get_rope_index``."""
        if video_grid_thw is not None:
            raise NotImplementedError("get_rope_index covers images only (the reference's zoom loop feeds no video)")
        ids = self._tokens(input_ids, "input_ids")
        B, L = ids.shape
        mask = None if attention_mask is None else self._tokens(attention_mask, "attention_mask")
        if mask is not None and mask.shape != ids.shape:
            raise ValueError(f"attention_mask is {tuple(mask.shape)}, input_ids {tuple(ids.shape)}")
        grid = None if image_grid_thw is None else self._grid(image_grid_thw)
        pos = torch.empty((3, B, L), dtype=torch.int64, device=self.device)
        delta = torch.empty((B, 1), dtype=torch.int64, device=self.device)
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            _lib.check(lib.zv_rope_index_dev(
                ids.data_ptr(), None if mask is None else mask.data_ptr(), B, L, None if grid is None else grid.data_ptr(),
                0 if grid is None else grid.shape[0], image_token_id, video_token_id, vision_start_token_id,
                spatial_merge_size, 1 if hf5_semantics else 0, pos.data_ptr(), delta.data_ptr(), self._status.data_ptr(),
                self._ws.data_ptr(), self._ws.numel(), torch.cuda.current_stream(self.device).cuda_stream))
        self.last_launches = lib.zv_last_launch_count()
        return pos, delta

    def placeholder_rows(self, input_ids, n_tokens, image_token_id=IMAGE_TOKEN_ID):
        """(n_tokens,) int64 on the device: the flattened rows of the image placeholders in masked_scatter order, -1 in
        the slots beyond their count.  A count other than ``n_tokens`` is raised by ``check()``."""
        if not isinstance(input_ids, torch.Tensor) or input_ids.device != self.device:
            raise ValueError(f"input_ids must be a tensor on {self.device}")
        if input_ids.numel() > self.max_batch * self.max_seq_len:
            raise ValueError(f"input_ids has {input_ids.numel()} tokens; this DeviceHandoff holds up to "
                             f"{self.max_batch} x {self.max_seq_len}")
        ids = input_ids.to(torch.int64).contiguous()
        rows = torch.empty(int(n_tokens), dtype=torch.int64, device=self.device)
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            _lib.check(lib.zv_placeholder_rows_dev(
                ids.data_ptr(), ids.numel(), image_token_id, rows.data_ptr() if rows.numel() else None, rows.numel(),
                self._rows_status.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
                torch.cuda.current_stream(self.device).cuda_stream))
        self.last_launches = lib.zv_last_launch_count()
        return rows

    @torch.no_grad()
    def embed_images(self, visual, inputs_embeds, input_ids, pixel_values, image_grid_thw, window_order=False,
                     image_token_id=IMAGE_TOKEN_ID):
        """``embed_images`` with the rows found on the device.  ``image_grid_thw`` on the host (the tower's plan is host
        bookkeeping).  On a placeholder count mismatch the embeddings without a placeholder are dropped and the rest of
        ``inputs_embeds`` is untouched; ``check()`` raises HF's ValueError.  Returns ``inputs_embeds``."""
        plan = visual.plan_for(image_grid_thw)
        rows = self.placeholder_rows(input_ids, plan.num_tokens, image_token_id)
        launches = self.last_launches
        visual.forward_into(inputs_embeds, rows, pixel_values, image_grid_thw, window_order=window_order, validate_rows=False)
        self.last_launches = launches + visual.last_launches
        return inputs_embeds

    def check(self):
        """Waits for the work enqueued so far and raises what the host hand-off would have raised for the same inputs:
        ``ZoomVitError`` from the last ``rope_index``, or ``ValueError`` from the last ``placeholder_rows``."""
        code, sample, a, b, rows_code, _, count, cap = self._status.tolist()
        if code:
            raise _lib.ZoomVitError(_lib.ZV_EINVAL, _ROPE_ERRORS[code].format(s=sample, a=a, b=b))
        if rows_code == _ROWS_COUNT:
            raise ValueError(f"Image features and image tokens do not match, tokens: {count}, features: {cap}")
