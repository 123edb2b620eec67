"""Crop-sharded multi-GPU execution (one process per GPU, torch.distributed).

Crops are independent sequences (attention never crosses cu_seqlens, HF modeling_qwen2_5_vl.py:488-502) and
the reference itself only ever runs data-parallel (``src/eval/infer.py:158-171``), so the path shards by crop
with no data-path collective.  The only exchange is the gather of the output embeddings (C1), a ragged
all-gather: counts first, then one ``all_gather`` of max-padded (T_r, out_hidden) blocks, then a permutation
back to the caller's crop order.  Works with NCCL (GPU) and gloo (CPU tests of the host logic).
"""
import numpy as np
import torch
import torch.distributed as dist


def crop_cost(grid_thw, full_layers=4):
    """FLOP estimate per crop (SURVEY 8e) of a 32-block tower: linear + full attention + window attention.
    ``full_layers``: blocks with full attention (4 in Qwen2.5-VL, all 32 in Qwen2-VL); the rest attend in windows.
    Full attention never crosses a frame group of a video (HF cu_seqlens = repeat_interleave(h w, t)): t (h w)^2."""
    g = np.asarray(grid_thw, dtype=np.float64).reshape(-1, 3)
    HW = g[:, 1] * g[:, 2]
    S = g[:, 0] * HW
    T = S / 4
    return 5.125e9 * T + full_layers * 4 * S * HW * 1280 + (32 - full_layers) * 4 * 64 * S * 1280


def partition(costs, world_size):
    """Longest-processing-time-first greedy assignment; deterministic, identical on every rank.
    Returns a list (per rank) of crop indices, each in ascending order."""
    costs = np.asarray(costs, dtype=np.float64)
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    load = [0.0] * world_size
    parts = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (load[k], k))
        parts[r].append(i)
        load[r] += costs[i]
    return [sorted(p) for p in parts]


def gather_embeddings(local_emb, local_tokens, parts, group=None):
    """local_emb: (T_r, D) embeddings of this rank's crops (in the order of parts[rank]); local_tokens: tokens of
    each of those crops.  Returns ((T_total, D) embeddings in global crop order, per-crop token counts)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    dev = local_emb.device
    n_total = sum(len(p) for p in parts)
    counts_local = torch.zeros(n_total, dtype=torch.int64, device=dev)
    if len(parts[rank]):
        counts_local[torch.as_tensor(parts[rank], device=dev)] = torch.as_tensor(local_tokens, dtype=torch.int64, device=dev)
    dist.all_reduce(counts_local, group=group)                       # every crop is owned by exactly one rank
    counts = counts_local.cpu().numpy()
    per_rank = [int(counts[p].sum()) if len(p) else 0 for p in parts]
    tmax = max(per_rank + [1])
    D = local_emb.shape[1]
    padded = torch.zeros((tmax, D), dtype=local_emb.dtype, device=dev)
    padded[: local_emb.shape[0]] = local_emb
    gathered = torch.empty((world, tmax, D), dtype=local_emb.dtype, device=dev)
    dist.all_gather_into_tensor(gathered.view(world * tmax, D), padded, group=group)
    # permutation back to global crop order
    starts = np.concatenate([[0], np.cumsum(counts)])
    out = torch.empty((int(starts[-1]), D), dtype=local_emb.dtype, device=dev)
    for r, p in enumerate(parts):
        off = 0
        for i in p:
            n = int(counts[i])
            out[int(starts[i]): int(starts[i]) + n] = gathered[r, off: off + n]
            off += n
    return out, counts


def sharded_rows(parts, tokens):
    """Row bookkeeping of a crop-sharded batch whose embeddings are gathered in GLOBAL crop order.  tokens: tokens of every
    crop (global order); parts: per rank, the crop indices it owns.  Returns (starts (n + 1,) int64 - first gather row of
    every crop - and, per rank, the int64 array of gather rows of that rank's local embeddings, crops in parts[rank] order)."""
    tokens = np.asarray(tokens, dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(tokens)]).astype(np.int64)
    rows = []
    for p in parts:
        rows.append(np.concatenate([np.arange(starts[i], starts[i + 1], dtype=np.int64) for i in p]) if len(p)
                    else np.zeros(0, np.int64))
    return starts, rows


class PeerGather:
    """Gather buffer in symmetric memory for the fused GEMM -> gather path (C1 without a collective).

    Every rank owns one (rows_total, dim) buffer; all of them are mapped into every process
    (torch.distributed._symmetric_memory: CUDA VMM handles exchanged once at construction).  The tower's last GEMM
    (merger.mlp.2 + un-reorder) then stores each embedding row into its own buffer and, over NVLink, into every
    peer's buffer at the same global row, so after one cross-rank barrier each rank holds all embeddings - the
    transfer overlaps the GEMM tile by tile and no NCCL collective runs on the data path.

    ``double_buffer=True``: two buffers alternate per step and the barrier of step i runs on a side stream; the main
    stream only waits for it at the start of step i + 1 (``begin_step``), i.e. a rank that finishes early starts its next
    step instead of idling until the slowest (power-capped) GPU arrives.  Contract: the buffer ``begin_step`` returns as
    ``ready`` holds the previous step's gather; read it on the current stream before the next ``begin_step``.
    """

    def __init__(self, rows_total, dim, dtype, device, group=None, double_buffer=False):
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self.rows_total, self.dim, self.n_buf = int(rows_total), int(dim), 2 if double_buffer else 1
        self._all = symm_mem.empty((self.n_buf * self.rows_total, dim), dtype=dtype, device=device)
        self.handle = symm_mem.rendezvous(self._all, self.group)
        self._base_ptrs = [int(p) for p in self.handle.buffer_ptrs]
        if len(self._base_ptrs) - 1 > 8:
            raise ValueError("the fused gather supports at most 9 ranks per node")
        self._stride = self.rows_total * dim * self._all.element_size()
        self.cur = 0
        self._side = torch.cuda.Stream(device) if double_buffer else None
        self._pending = None                       # event: the async barrier of the last finished step
        self._select(0)

    def _select(self, b):
        self.cur = b
        self.buffer = self._all[b * self.rows_total:(b + 1) * self.rows_total]
        self.local_ptr = self._base_ptrs[self.rank] + b * self._stride
        self.peer_ptrs = [p + b * self._stride for r, p in enumerate(self._base_ptrs) if r != self.rank]

    def barrier(self):
        """All ranks' stores are visible after this (device-side barrier over the signal pads, on the current stream)."""
        self.handle.barrier(channel=self.cur)

    # ---- pipelined form (double_buffer=True)
    def begin_step(self):
        """Waits (on the current stream) for the previous step's barrier, then switches to the other buffer.  Returns the
        buffer that is now complete on every rank (None before the first step)."""
        ready = None
        if self._pending is not None:
            torch.cuda.current_stream(self._all.device).wait_event(self._pending)
            self._pending = None
            ready = self.buffer
        if self.n_buf == 2:
            self._select(self.cur ^ 1)
        return ready

    def end_step(self):
        """Call after the step's kernels are enqueued: the cross-rank barrier runs on a side stream behind them."""
        if self._side is None:
            self.barrier()
            return
        dev = self._all.device
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self._side):
            self._side.wait_event(ev)
            self.handle.barrier(channel=self.cur)
            done = torch.cuda.Event()
            done.record(self._side)
        self._pending = done

    def finish(self):
        """Waits for the last step's barrier on the current stream; returns that step's buffer."""
        if self._pending is not None:
            torch.cuda.current_stream(self._all.device).wait_event(self._pending)
            self._pending = None
        return self.buffer


def encode_sharded(enc, images_dev, boxes, image_index, gather, max_patches=400_000, apply_cut_image=True):
    """configs[3] / [4]: a ragged crop list sharded over the ranks by LPT partition, every rank encoding its crops in
    bounded micro-batches whose last GEMM scatters each embedding row straight to its GLOBAL row of every rank's gather
    buffer (``zv_visual_forward_gather_rows``) - no padded all-gather, no per-crop copy loop.  Source images are
    replicated.  Returns (gather buffer rows [0, T_total) in global crop order - complete after ``gather.barrier()`` /
    ``end_step()`` -, per-crop token counts, parts)."""
    from . import geometry
    rank, world = gather.rank, gather.world
    n = len(boxes)
    idx = list(range(n)) if image_index is None else [int(i) for i in image_index]
    cfg = enc.processor._cfg()
    if not apply_cut_image:
        cfg.min_size = -1
    img_hw = np.array([[images_dev[i].shape[0], images_dev[i].shape[1]] for i in idx], np.int32)
    _, _, grid = geometry.geometry(cfg, img_hw, np.asarray(boxes, np.float64).reshape(n, 4))
    tokens = (grid[:, 0] * grid[:, 1] * grid[:, 2]) // enc.visual.spatial_merge_unit
    from . import _lib
    full_layers = 32 if enc.visual.cfg.tower_kind == _lib.TOWER_QWEN2 else 4     # Qwen2-VL: every block full attention
    parts = partition(crop_cost(grid, full_layers), world)
    starts, rows = sharded_rows(parts, tokens)
    if starts[-1] > gather.rows_total:
        raise ValueError(f"gather buffer holds {gather.rows_total} rows, the batch needs {int(starts[-1])}")
    mine = parts[rank]
    launches = 0
    if mine:
        lb = [boxes[i] for i in mine]
        li = [idx[i] for i in mine]
        dev = images_dev[0].device
        for g in enc.micro_batches(images_dev, lb, li, max_patches, apply_cut_image):
            used = sorted({li[i] for i in g})
            local = {k: j for j, k in enumerate(used)}
            r = torch.from_numpy(np.concatenate([np.arange(starts[mine[i]], starts[mine[i] + 1], dtype=np.int64) for i in g])).to(dev)
            enc.encode([images_dev[k] for k in used], [lb[i] for i in g], image_index=[local[li[i]] for i in g],
                       apply_cut_image=apply_cut_image, gather=gather, gather_rows=r)
            launches += enc.last_launches
    enc.last_launches = launches
    return gather.buffer[: int(starts[-1])], tokens, parts
