"""FusedVisual - drop-in for ``model.visual`` (HF ``Qwen2_5_VisionTransformerPretrainedModel``).

Same call as the reference makes through the LM forward (HF modeling_qwen2_5_vl.py:1172,
``self.visual(pixel_values, grid_thw=image_grid_thw)``; reference copy ``qwen2_5vl_monkey_patch.py:93``):
``forward(hidden_states (S,1176), grid_thw (N,3)) -> (T, out_hidden)`` in ``self.dtype``, HF row order.
The whole forward (HF :455-518) runs inside ``zv_visual_forward`` on hand-written sm_100a kernels; this module
only owns the packed weights, a plan cache and a workspace, all as torch tensors (plumbing).
"""
import ctypes as C
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

from . import _lib
from .plan import Plan

_DT = {torch.float32: _lib.ZV_F32, torch.bfloat16: _lib.ZV_BF16, torch.float16: _lib.ZV_F16}


def _vision_cfg_from_hf(config):
    """zv_cfg fields of an HF vision config: ``Qwen2_5_VLVisionConfig`` (tower kind 0) or ``Qwen2VLVisionConfig`` (kind 1,
    whose ``hidden_size`` is the merger's output width and whose blocks are all full attention)."""
    if getattr(config, "model_type", None) == "qwen2_vl":
        if config.hidden_act != "quick_gelu":
            raise NotImplementedError(f"Qwen2-VL tower with hidden_act={config.hidden_act!r}: only quick_gelu is built")
        return dict(depth=config.depth, hidden=config.embed_dim, heads=config.num_heads,
                    inter=int(config.embed_dim * config.mlp_ratio), out_hidden=config.hidden_size, patch=config.patch_size,
                    merge=config.spatial_merge_size, temporal=config.temporal_patch_size,
                    fullatt=list(range(config.depth)), tower_kind=_lib.TOWER_QWEN2)
    return dict(depth=config.depth, hidden=config.hidden_size, heads=config.num_heads,
                inter=config.intermediate_size, out_hidden=config.out_hidden_size, patch=config.patch_size,
                merge=config.spatial_merge_size, temporal=config.temporal_patch_size, window=config.window_size,
                fullatt=list(config.fullatt_block_indexes))


class FusedVisual(nn.Module):
    def __init__(self, state_dict, device=None, dtype=torch.float16, operand_dtype=None,
                 return_pooling_output=False, **cfg_overrides):
        """state_dict: HF names relative to the tower (``visual.`` / ``model.visual.`` prefixes are accepted).
        ``dtype`` is the dtype of the returned embeddings (what callers read as ``visual.dtype``); default float16,
        the dtype the reference's eval loop loads the model in (src/eval/infer.py:149).
        ``operand_dtype`` is the 16-bit type of the GEMM / attention operands: float16 (default: 11-bit mantissa,
        max rel err 1.4e-3 against the fp32 tower at full depth) or bfloat16 (opt-in: 8x the rounding error, 1.15e-2,
        outside the 1e-2 tolerance north_star states - same tensor-core rate).  Accumulation, RMSNorm, rotary, softmax
        and the residual stream are fp32 either way."""
        super().__init__()
        if not torch.cuda.is_available():
            raise RuntimeError("FusedVisual needs a CUDA device (sm_100); there is no CPU fallback")
        self._device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._dtype = dtype
        if dtype not in _DT:
            raise ValueError("FusedVisual returns float32, bfloat16 or float16 embeddings")
        if operand_dtype is None:
            operand_dtype = torch.float16
        if operand_dtype not in (torch.bfloat16, torch.float16):
            raise ValueError("operand_dtype must be torch.bfloat16 or torch.float16")
        self.operand_dtype = operand_dtype
        self.cfg = _lib.default_cfg(op_dtype=_DT[operand_dtype], **cfg_overrides)
        self.spatial_merge_size = self.cfg.merge
        self.patch_size = self.cfg.patch
        self.spatial_merge_unit = self.cfg.merge ** 2
        self.return_pooling_output = return_pooling_output
        self._plans = OrderedDict()
        self._graphs = OrderedDict()      # (grid bytes, input dtype, order) -> captured CUDA graph of the tower
        self._ws = None
        self._rev = {}                    # plan grid bytes -> device reverse index (Qwen2-VL hidden states in HF order)
        self.last_launches = 0
        self._pack(state_dict)

    @classmethod
    def from_hf(cls, hf_visual, **kw):
        """Build from an instantiated HF vision tower (weights are read from its state_dict)."""
        cfg = _vision_cfg_from_hf(hf_visual.config)
        kw.setdefault("dtype", torch.float16)
        return cls(hf_visual.state_dict(), **cfg, **kw)


    def _pack(self, state_dict):
        lib = _lib.lib()
        nbytes = _lib.check(lib.zv_weights_bytes(C.byref(self.cfg)))
        packed = torch.empty(nbytes, dtype=torch.uint8, device=self._device)
        keep, descs = [], []
        for name, t in state_dict.items():
            if not isinstance(t, torch.Tensor) or "inv_freq" in name:
                continue
            if t.dtype not in _DT:
                t = t.float()
            t = t.detach().to(self._device).contiguous()
            keep.append(t)
            d = _lib.ZvTensor()
            d.name = name.encode()
            d.data = t.data_ptr()
            d.dtype = _DT[t.dtype]
            d.ndim = t.ndim
            for i, s in enumerate(t.shape):
                d.shape[i] = s
            descs.append(d)
        arr = (_lib.ZvTensor * len(descs))(*descs)
        stream = torch.cuda.current_stream(self._device).cuda_stream
        with torch.cuda.device(self._device):
            _lib.check(lib.zv_weights_pack(C.byref(self.cfg), arr, len(descs), packed.data_ptr(), nbytes, stream))
            torch.cuda.current_stream(self._device).synchronize()      # sources may be freed after this
        self.register_buffer("packed_weights", packed, persistent=False)

    # ---- attributes callers read
    @property
    def dtype(self):
        return self._dtype

    @property
    def device(self):
        return self._device

    def get_dtype(self):
        return self._dtype

    def get_device(self):
        return self._device

    def plan_for(self, grid_thw):
        g = np.ascontiguousarray(np.asarray(grid_thw.cpu() if isinstance(grid_thw, torch.Tensor) else grid_thw,
                                            dtype=np.int64).reshape(-1, 3))
        key = g.tobytes()
        p = self._plans.get(key)
        if p is None:
            p = Plan(self.cfg, g)
            self._plans[key] = p
            if len(self._plans) > 64:
                self._plans.popitem(last=False)
        else:
            self._plans.move_to_end(key)
        return p

    def _workspace(self, nbytes):
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self._device)
        return self._ws

    # ---- CUDA-graph replay for launch-bound (small) batches
    def graph_buffers(self, grid_thw, in_dtype=None, window_order=True):
        """Static (input, output) tensors of the captured graph for this grid; capturing on first use.  The tower is
        234 kernel launches: for a single zoom crop (1 296 patches) the launches cost more than the kernels, so the
        whole forward is captured once per grid signature and replayed (`forward(..., use_graph=True)`)."""
        plan = self.plan_for(grid_thw)
        in_dtype = in_dtype or self.operand_dtype
        key = (plan.grid_thw.tobytes(), in_dtype, bool(window_order))
        ent = self._graphs.get(key)
        if ent is None:
            x = torch.zeros((plan.num_patches, 1176), dtype=in_dtype, device=self._device)
            self._forward_impl(x, plan, window_order, False, None, 0)          # warm-up: attributes, plan tables, workspace
            torch.cuda.current_stream(self._device).synchronize()
            out = torch.empty((plan.num_tokens, self.cfg.out_hidden), dtype=self._dtype, device=self._device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._forward_impl(x, plan, window_order, False, None, 0, out=out)
            # everything the captured kernels point at must outlive the graph: the workspace, and the plan with its
            # device tables (rotary ids, rope table, window index, attention tiles) - the plan LRU may evict the plan
            # long before the graph is replayed again
            ent = (g, x, out, self._ws, plan, plan._dev)
            self._graphs[key] = ent
            if len(self._graphs) > 16:
                self._graphs.popitem(last=False)
        else:
            self._graphs.move_to_end(key)
        return ent

    @torch.no_grad()
    def forward(self, hidden_states, grid_thw, window_order=False, return_hidden=False, gather=None, gather_row=0,
                use_graph=False, gather_rows=None, **kwargs):
        if use_graph and gather is None and not return_hidden and not self.return_pooling_output:
            x = hidden_states
            if x.dtype not in _DT or (x.dtype != torch.float32 and x.dtype != self.operand_dtype):
                x = x.float()
            g, xin, out = self.graph_buffers(grid_thw, x.dtype, window_order)[:3]
            if x.data_ptr() != xin.data_ptr():
                xin.copy_(x, non_blocking=True)
            g.replay()
            self.last_launches = 1
            # `out` is the graph's static buffer: the next replay for this grid overwrites it, so hand out a copy
            # (0.3 MB for a 512-px crop) unless the caller asked for the buffer itself
            return out if kwargs.get("graph_static_output") else out.clone()
        plan = self.plan_for(grid_thw)
        return self._forward_impl(hidden_states, plan, window_order, return_hidden, gather, gather_row, gather_rows=gather_rows)

    @torch.no_grad()
    def forward_into(self, inputs_embeds, dest_rows, hidden_states, grid_thw, window_order=False, validate_rows=True):
        """Tower forward with the LM hand-off fused into the last GEMM (``zv_visual_forward_into``): embedding k (HF
        order) lands in row ``dest_rows[k]`` of the flattened ``inputs_embeds`` (B, L, out_hidden) - in place, the
        result of ``inputs_embeds.masked_scatter(image_mask, self(hidden_states, grid_thw))`` (HF modeling_qwen2_5_vl.py
        :1301-1307) without materialising the embeddings.  ``dest_rows``: int64 CUDA tensor (see handoff.placeholder_rows)."""
        lib = _lib.lib()
        plan = self.plan_for(grid_thw)
        e = inputs_embeds
        if e.device != self._device or e.dtype not in _DT or not e.is_contiguous() or e.shape[-1] != self.cfg.out_hidden:
            raise ValueError(f"inputs_embeds must be a contiguous (..., {self.cfg.out_hidden}) float32/bfloat16/float16 "
                             f"tensor on {self._device}")
        if dest_rows.dtype != torch.int64 or dest_rows.device != self._device or dest_rows.numel() != plan.num_tokens:
            raise ValueError(f"dest_rows must be {plan.num_tokens} int64 row indices on {self._device}")
        n_rows = e.numel() // e.shape[-1]
        if validate_rows and dest_rows.numel():
            lo, hi = torch.aminmax(dest_rows)                         # one host sync; the kernel also drops bad rows
            if int(lo) < 0 or int(hi) >= n_rows:
                raise IndexError(f"dest_rows spans [{int(lo)}, {int(hi)}] but inputs_embeds has {n_rows} rows")
        x = self._check_input(hidden_states, plan, window_order)
        stream = torch.cuda.current_stream(self._device).cuda_stream
        with torch.cuda.device(self._device):
            tables = plan.device_tables(self._device, stream)
            ws = self._workspace(_lib.check(lib.zv_visual_workspace_bytes(C.byref(self.cfg), plan.handle)))
            _lib.check(lib.zv_visual_forward_into(
                C.byref(self.cfg), self.packed_weights.data_ptr(), plan.handle, tables.data_ptr(), x.data_ptr(),
                _DT[x.dtype], _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF, e.data_ptr(),
                n_rows, _DT[e.dtype], dest_rows.contiguous().data_ptr(), ws.data_ptr(), ws.numel(), stream))
        self.last_launches = lib.zv_last_launch_count()
        return inputs_embeds

    def _check_input(self, hidden_states, plan, window_order):
        x = hidden_states
        if x.device != self._device:
            x = x.to(self._device, non_blocking=True)
        if x.dtype not in _DT or (x.dtype != torch.float32 and x.dtype != self.operand_dtype):
            if window_order:
                raise ValueError(f"window-ordered patches must be {self.operand_dtype} (the fused preprocess output)")
            x = x.float()
        x = x.contiguous()
        if x.shape != (plan.num_patches, 1176):
            raise ValueError(f"pixel_values has shape {tuple(x.shape)}, grid_thw implies ({plan.num_patches}, 1176)")
        return x

    def _hf_order(self, hidden, plan):
        """Window-ordered hidden states (S, hidden) -> HF row order: merge groups of 4 rows gathered by the plan's reverse
        index.  HF's Qwen2-VL tower never reorders, so its ``last_hidden_state`` is in HF order."""
        key = plan.grid_thw.tobytes()
        rev = self._rev.get(key)
        if rev is None:
            rev = torch.from_numpy(plan.reverse_index.copy()).to(self._device)
            self._rev[key] = rev
            if len(self._rev) > 64:
                self._rev.pop(next(iter(self._rev)))
        return hidden.view(-1, self.spatial_merge_unit, hidden.shape[-1]).index_select(0, rev).view(hidden.shape)

    def _forward_impl(self, hidden_states, plan, window_order, return_hidden, gather, gather_row, out=None, gather_rows=None):
        """hidden_states: (S, 1176) patches, float32/bfloat16, HF row order (or the window-ordered bf16 output of
        the fused preprocess when ``window_order=True``).  ``gather`` (a ``sharding.PeerGather``) fuses the multi-GPU
        embedding gather into the last GEMM: this rank's rows land at ``gather_row`` of every rank's gather buffer."""
        lib = _lib.lib()
        x = self._check_input(hidden_states, plan, window_order)
        stream = torch.cuda.current_stream(self._device).cuda_stream
        with torch.cuda.device(self._device):
            tables = plan.device_tables(self._device, stream)
            ws = self._workspace(_lib.check(lib.zv_visual_workspace_bytes(C.byref(self.cfg), plan.handle)))
            if gather is not None:
                if gather.buffer.dtype != self._dtype or self._dtype == torch.float32:
                    raise ValueError("the fused gather needs a 16-bit gather buffer of the tower's output dtype")
                out = gather.buffer[gather_row:gather_row + plan.num_tokens]
            elif out is None:
                out = torch.empty((plan.num_tokens, self.cfg.out_hidden), dtype=self._dtype, device=self._device)
            hidden = (torch.empty((plan.num_patches, self.cfg.hidden), dtype=torch.float32, device=self._device)
                      if (return_hidden or self.return_pooling_output) else None)
            if gather is not None and gather_rows is not None:
                # ragged form: embedding k of this batch lands at row gather_rows[k] of every rank's gather buffer
                if gather_rows.dtype != torch.int64 or gather_rows.device != self._device or gather_rows.numel() != plan.num_tokens:
                    raise ValueError(f"gather_rows must be {plan.num_tokens} int64 row indices on {self._device}")
                peers = (C.c_void_p * max(1, len(gather.peer_ptrs)))(*gather.peer_ptrs)
                _lib.check(lib.zv_visual_forward_gather_rows(
                    C.byref(self.cfg), self.packed_weights.data_ptr(), plan.handle, tables.data_ptr(), x.data_ptr(),
                    _DT[x.dtype], _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF, gather.buffer.data_ptr(),
                    gather.buffer.shape[0], _DT[self._dtype], gather_rows.contiguous().data_ptr(), ws.data_ptr(), ws.numel(),
                    peers, len(gather.peer_ptrs), stream))
                out = gather.buffer
            elif gather is not None:
                peers = (C.c_void_p * len(gather.peer_ptrs))(*gather.peer_ptrs)
                _lib.check(lib.zv_visual_forward_gather(
                    C.byref(self.cfg), self.packed_weights.data_ptr(), plan.handle, tables.data_ptr(), x.data_ptr(),
                    _DT[x.dtype], _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF, out.data_ptr(), _DT[self._dtype],
                    ws.data_ptr(), ws.numel(), peers, len(gather.peer_ptrs), int(gather_row), stream))
            else:
                _lib.check(lib.zv_visual_forward(
                    C.byref(self.cfg), self.packed_weights.data_ptr(), plan.handle, tables.data_ptr(), x.data_ptr(),
                    _DT[x.dtype], _lib.ORDER_WINDOW if window_order else _lib.ORDER_HF, out.data_ptr(), _DT[self._dtype],
                    hidden.data_ptr() if hidden is not None else None, ws.data_ptr(), ws.numel(), stream))
        self.last_launches = lib.zv_last_launch_count()
        if hidden is not None and self.cfg.tower_kind == _lib.TOWER_QWEN2:
            hidden = self._hf_order(hidden, plan)
        if self.return_pooling_output:
            from transformers.modeling_outputs import BaseModelOutputWithPooling
            return BaseModelOutputWithPooling(last_hidden_state=hidden.to(self._dtype), pooler_output=out)
        if return_hidden:
            return out, hidden
        return out
