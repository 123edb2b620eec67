"""LM hand-off on the device (DeviceHandoff: zv_rope_index_dev, zv_placeholder_rows_dev).  Integer bookkeeping and data
movement, so the bar is torch.equal against the host path (zv_rope_index / zv_placeholder_rows, themselves pinned to the
reference's get_rope_index and to transformers 5.x in test_handoff.py), on random batches, at the size limits, inside a
CUDA graph with the tower, and with torch's sync debug mode set to raise."""
import types

import numpy as np
import pytest
import torch

from oracle import tower as OT

pytestmark = pytest.mark.gpu
IMG, VID, VSTART, VEND, PAD = 151655, 151656, 151652, 151653, 151643


def _random_batch(seed, left_pad):
    """Copy of test_handoff._random_batch: 1-4 samples of text and 0-3 images, padded."""
    rng = np.random.default_rng(seed)
    rows, grids = [], []
    for _ in range(int(rng.integers(1, 5))):
        ids = []
        for _ in range(int(rng.integers(0, 4))):
            ids += rng.integers(0, 1000, int(rng.integers(0, 9))).tolist()
            gh, gw = 2 * int(rng.integers(1, 12)), 2 * int(rng.integers(1, 12))
            grids.append((1, gh, gw))
            ids += [VSTART] + [IMG] * (gh * gw // 4) + [VEND]
        ids += rng.integers(0, 1000, int(rng.integers(1, 9))).tolist()
        rows.append(ids)
    L = max(len(r) for r in rows)
    ids = np.full((len(rows), L), PAD, np.int64)
    mask = np.zeros((len(rows), L), np.int64)
    for i, r in enumerate(rows):
        sl = slice(L - len(r), L) if left_pad else slice(0, len(r))
        ids[i, sl], mask[i, sl] = r, 1
    return ids, mask, np.asarray(grids, np.int64).reshape(-1, 3)


def _prompt(grid, rng, left_pad=True):
    """test_gpu_handoff's prompt: two samples (two images, then one), padded to one length that depends on grid only."""
    rows, k = [], 0
    for n in (2, 1):
        ids = rng.integers(0, 1000, 3).tolist()
        for _ in range(n):
            t = int(grid[k, 1] * grid[k, 2]) // 4
            ids += [VSTART] + [IMG] * t + [VEND] + rng.integers(0, 1000, 2).tolist()
            k += 1
        rows.append(ids)
    L = max(len(r) for r in rows)
    out = np.full((len(rows), L), PAD, np.int64)
    mask = np.zeros((len(rows), L), np.int64)
    for i, r in enumerate(rows):
        sl = slice(L - len(r), L) if left_pad else slice(0, len(r))
        out[i, sl], mask[i, sl] = r, 1
    return out, mask


def _host(ids, grid, mask, hf5):
    """The host path on the same input: (pos, delta) or the ZoomVitError it raises."""
    from zoomearth_b200 import get_rope_index
    from zoomearth_b200._lib import ZoomVitError
    try:
        return get_rope_index(torch.as_tensor(ids), None if grid is None else torch.as_tensor(grid), None,
                              None if mask is None else torch.as_tensor(mask), hf5_semantics=hf5), None
    except ZoomVitError as e:
        return None, e


def _compare(dh, ids, grid, mask, hf5, cuda):
    """Device rope index == host rope index, or check() raises the host's error with the host's text."""
    from zoomearth_b200._lib import ZoomVitError
    ref, err = _host(ids, grid, mask, hf5)
    pos, delta = dh.rope_index(torch.as_tensor(ids).to(cuda), None if grid is None else torch.as_tensor(grid),
                               None if mask is None else torch.as_tensor(mask).to(cuda), hf5_semantics=hf5)
    if err is not None:
        with pytest.raises(ZoomVitError) as got:
            dh.check()
        assert got.value.code == err.code and got.value.msg == err.msg
        return False
    dh.check()
    assert pos.shape == ref[0].shape and pos.dtype == torch.int64 and delta.shape == ref[1].shape
    assert torch.equal(pos.cpu(), ref[0]) and torch.equal(delta.cpu(), ref[1])
    return True


@pytest.fixture(scope="module")
def dh(cuda):
    from zoomearth_b200 import DeviceHandoff
    return DeviceHandoff(cuda, 1024, 131072)


@pytest.fixture(scope="module")
def visual(cuda):
    from zoomearth_b200 import FusedVisual
    cfg = OT.small_cfg(depth=2, fullatt=(1,))
    return {dt: FusedVisual(OT.make_weights(21, cfg), device=cuda, dtype=dt, operand_dtype=torch.bfloat16,
                            depth=cfg["depth"], fullatt=list(cfg["fullatt"])) for dt in (torch.bfloat16, torch.float32)}


def test_rope_index_equals_host_on_random_batches(dh, cuda):
    """200 seeded batches x both semantics: left / right padding, no mask, masks holding values other than 0 and 1
    (the image branch admits mask == 1 only, the text branch mask != 0), and text-only batches."""
    n_ok = n_err = n_text = 0
    for seed in range(200):
        ids, mask, grid = _random_batch(seed, left_pad=seed % 2 == 0)
        kind = seed % 4
        if kind == 2:
            mask = None
        elif kind == 3:
            rng = np.random.default_rng(1000 + seed)
            odd = rng.choice(np.array([2, -1, 7]), mask.shape)
            pick = rng.random(mask.shape) < (0.9 if seed % 8 == 3 else 0.05)
            mask = np.where(pick & (mask == 0), odd, mask)          # pads marked with other nonzero values
            if seed % 8 == 7:
                mask = np.where(pick & (mask == 1), odd, mask)      # and some real tokens too
        if seed % 10 == 9:                                          # text only: no grid (vision tokens are plain text)
            grid = np.zeros((0, 3), np.int64)
        g = grid if len(grid) else None
        n_text += g is None
        for hf5 in (False, True):
            if _compare(dh, ids, g, mask, hf5, cuda):
                n_ok += 1
            else:
                n_err += 1
    assert n_text >= 20 and n_ok >= 300, (n_ok, n_err, n_text)


def test_rope_index_text_only_batches(dh, cuda):
    rng = np.random.default_rng(7)
    for it in range(12):
        B, L = int(rng.integers(1, 9)), int(rng.integers(1, 700))
        ids = rng.integers(0, 1000, (B, L))
        mask = None if it % 3 == 0 else rng.integers(0, 2 if it % 3 == 1 else 4, (B, L))
        if it == 5:
            mask[0] = 0                                             # a fully masked sample is fine without a grid
        for hf5 in (False, True):
            assert _compare(dh, ids, None, mask, hf5, cuda)
        assert dh.last_launches == 1


def test_rope_index_large_batch_short_rows(dh, cuda):
    rng = np.random.default_rng(11)
    rows, grids = [], []
    for b in range(1024):
        ids = rng.integers(0, 1000, int(rng.integers(1, 6))).tolist()
        for _ in range(int(rng.integers(0, 3))):
            gh, gw = 2 * int(rng.integers(1, 4)), 2 * int(rng.integers(1, 4))
            grids.append((1, gh, gw))
            ids += [VSTART] + [IMG] * (gh * gw // 4) + [VEND] + rng.integers(0, 1000, int(rng.integers(0, 4))).tolist()
        rows.append(ids)
    L = max(len(r) for r in rows)
    ids = np.full((1024, L), PAD, np.int64)
    mask = np.zeros((1024, L), np.int64)
    for i, r in enumerate(rows):
        sl = slice(L - len(r), L) if i % 2 else slice(0, len(r))
        ids[i, sl], mask[i, sl] = r, 1
    grid = np.asarray(grids, np.int64)
    for hf5 in (False, True):
        assert _compare(dh, ids, grid, mask, hf5, cuda)
    assert dh.last_launches == 2
    assert _compare(dh, ids, grid, None, False, cuda)                # no mask: the pads are text


def test_rope_index_long_rows_many_images(dh, cuda):
    """B = 2, L = 131 072: sample 0 holds 150 images between runs of text, sample 1 a few, both left-padded."""
    rng = np.random.default_rng(5)
    L = 131072
    rows, grids = [], []
    for n_img in (150, 3):
        ids = []
        for _ in range(n_img):
            ids += rng.integers(0, 1000, int(rng.integers(0, 300))).tolist()
            gh, gw = 2 * int(rng.integers(1, 20)), 2 * int(rng.integers(1, 20))
            grids.append((1, gh, gw))
            ids += [VSTART] + [IMG] * (gh * gw // 4) + [VEND]
        ids += rng.integers(0, 1000, 500).tolist()
        assert len(ids) < L
        rows.append(ids)
    ids = np.full((2, L), PAD, np.int64)
    mask = np.zeros((2, L), np.int64)
    for i, r in enumerate(rows):
        ids[i, L - len(r):], mask[i, L - len(r):] = r, 1
    grid = np.asarray(grids, np.int64)
    for hf5 in (False, True):
        assert _compare(dh, ids, grid, mask, hf5, cuda)
    full = ids[:, L - len(rows[0]):]                                 # no padding in sample 0, no mask
    assert _compare(dh, full[:1], grid[:150], None, False, cuda)


@pytest.mark.parametrize("seed", range(4))
def test_hf5_semantics_match_installed_transformers(dh, cuda, seed):
    """As test_handoff.test_hf5_semantics_match_installed_transformers (tokens_per_second = 1), for the device path."""
    mod = pytest.importorskip("transformers.models.qwen2_5_vl.modeling_qwen2_5_vl")
    ids, mask, grid = _random_batch(100 + seed, left_pad=True)
    if not len(grid):
        pytest.skip("no image in this batch")
    model_cls = mod.Qwen2_5_VLModel
    me = types.SimpleNamespace(config=types.SimpleNamespace(
        vision_config=types.SimpleNamespace(spatial_merge_size=2, tokens_per_second=1)))
    me.get_vision_position_ids = types.MethodType(model_cls.get_vision_position_ids, me)
    tt = torch.from_numpy((ids == IMG).astype(np.int32))
    ref_pos, ref_delta = model_cls.get_rope_index(me, torch.from_numpy(ids), tt, torch.from_numpy(grid),
                                                  attention_mask=torch.from_numpy(mask))
    p, d = dh.rope_index(torch.from_numpy(ids).to(cuda), torch.from_numpy(grid), torch.from_numpy(mask).to(cuda),
                         hf5_semantics=True)
    dh.check()
    assert torch.equal(p.cpu(), ref_pos) and torch.equal(d.cpu(), ref_delta.to(torch.int64))


def test_rope_index_casts_other_dtypes(dh, cuda):
    ids, mask, grid = _random_batch(3, left_pad=True)
    ref, _ = _host(ids, grid, mask, False)
    p, d = dh.rope_index(torch.from_numpy(ids).to(torch.int32).to(cuda), torch.from_numpy(grid).to(torch.int32).to(cuda),
                         torch.from_numpy(mask).to(torch.bool).to(cuda))
    dh.check()
    assert torch.equal(p.cpu(), ref[0]) and torch.equal(d.cpu(), ref[1])


def test_placeholder_rows_equal_nonzero(dh, cuda):
    rng = np.random.default_rng(3)
    for it in range(10):
        B, L = int(rng.integers(1, 70)), int(rng.integers(1, 3000))
        ids = torch.from_numpy(np.where(rng.random((B, L)) < 0.3, IMG, rng.integers(0, 1000, (B, L)))).to(cuda)
        ref = torch.nonzero(ids.flatten() == IMG).reshape(-1)
        n = ref.numel()
        rows = dh.placeholder_rows(ids, n)
        dh.check()
        assert dh.last_launches == 2 and torch.equal(rows, ref)
        rows = dh.placeholder_rows(ids, n + 37)                          # more slots than placeholders: -1 padding
        assert torch.equal(rows[:n], ref) and bool((rows[n:] == -1).all())
        with pytest.raises(ValueError, match=f"tokens: {n}, features: {n + 37}"):
            dh.check()
        if n > 5:
            rows = dh.placeholder_rows(ids, n - 5)                       # fewer: the first n - 5
            assert torch.equal(rows, ref[:n - 5])
            with pytest.raises(ValueError, match="do not match"):
                dh.check()


@pytest.mark.parametrize("embed_dtype", [torch.bfloat16, torch.float32])
def test_embed_images_equals_masked_scatter(dh, visual, cuda, embed_dtype):
    fv = visual[embed_dtype]
    grid = torch.tensor([[1, 16, 20], [1, 8, 8], [1, 26, 36]])
    ids = torch.from_numpy(_prompt(grid.numpy(), np.random.default_rng(2))[0]).to(cuda)
    S = int((grid[:, 1] * grid[:, 2]).sum())
    pv = torch.randn(S, 1176, generator=torch.Generator().manual_seed(5)).to(cuda)
    emb0 = torch.randn(ids.shape[0], ids.shape[1], 2048, generator=torch.Generator().manual_seed(6)).to(embed_dtype).to(cuda)
    feats = fv(pv, grid)
    image_mask = (ids == IMG).unsqueeze(-1).expand_as(emb0)
    ref = emb0.masked_scatter(image_mask, feats)
    got = dh.embed_images(fv, emb0.clone(), ids, pv, grid)
    dh.check()
    assert torch.equal(got, ref)
    assert dh.last_launches == 2 + fv.last_launches
    # one placeholder fewer than embeddings: check() raises HF's error, and the rows the placeholders reach hold the first
    # embeddings while every other row stays as it was
    short = ids.clone()
    short[0, int((ids[0] == IMG).nonzero()[0])] = PAD
    got = dh.embed_images(fv, emb0.clone(), short, pv, grid)
    T = feats.shape[0]
    with pytest.raises(ValueError, match=f"tokens: {T - 1}, features: {T}"):
        dh.check()
    short_mask = (short == IMG).unsqueeze(-1).expand_as(emb0)
    assert torch.equal(got, emb0.masked_scatter(short_mask, feats[:T - 1]))


def test_embed_images_from_fused_preprocess(dh, cuda):
    from zoomearth_b200 import FusedImageProcessor, FusedVisual
    cfg = OT.small_cfg(depth=2, fullatt=(1,))
    fv = FusedVisual(OT.make_weights(22, cfg), device=cuda, dtype=torch.bfloat16, operand_dtype=torch.bfloat16,
                     depth=cfg["depth"], fullatt=list(cfg["fullatt"]))
    proc = FusedImageProcessor(min_pixels=3136, max_pixels=200704, device=cuda)
    img = torch.from_numpy(np.random.default_rng(9).integers(0, 256, (700, 900, 3), dtype=np.uint8)).to(cuda)
    pv, grid, _ = proc.preprocess_crops([img], [(10, 20, 600, 500)], out_dtype=torch.bfloat16, window_order=True)
    T = int(grid[0, 1] * grid[0, 2]) // 4
    ids = torch.tensor([[1, 2, VSTART] + [IMG] * T + [VEND, 3]], device=cuda)
    emb0 = torch.zeros(1, ids.shape[1], 2048, dtype=torch.bfloat16, device=cuda)
    ref = emb0.clone()
    ref[0, 3:3 + T] = fv(pv, grid, window_order=True)
    got = dh.embed_images(fv, emb0, ids, pv, grid, window_order=True)
    dh.check()
    assert got.data_ptr() == emb0.data_ptr() and torch.equal(got, ref)


def test_errors_match_the_host(dh, cuda):
    from test_handoff_device_host import ERROR_CASES
    for name, ids, mask, grid, status in ERROR_CASES:
        ids = np.asarray(ids, np.int64)
        mask = None if mask is None else np.asarray(mask, np.int64)
        for hf5 in (False, True):
            assert not _compare(dh, ids, np.asarray(grid, np.int64), mask, hf5, cuda), name
            assert tuple(dh._status[:4].tolist()) == status, name
    # a correct call afterwards clears the record
    ids, mask, grid = _random_batch(1, left_pad=True)
    assert _compare(dh, ids, grid if len(grid) else None, mask, False, cuda)


def test_no_host_synchronisation(dh, visual, cuda):
    fv = visual[torch.bfloat16]
    grid = torch.tensor([[1, 16, 20], [1, 8, 8], [1, 26, 36]])
    ids_np, mask_np = _prompt(grid.numpy(), np.random.default_rng(4))
    ids, mask = torch.from_numpy(ids_np).to(cuda), torch.from_numpy(mask_np).to(cuda)
    S = int((grid[:, 1] * grid[:, 2]).sum())
    pv = torch.randn(S, 1176, generator=torch.Generator().manual_seed(5)).to(cuda)
    emb = torch.zeros(ids.shape[0], ids.shape[1], 2048, dtype=torch.bfloat16, device=cuda)
    for _ in range(2):                                               # warm-up: plan, workspaces, grid upload
        dh.rope_index(ids, grid, mask)
        dh.embed_images(fv, emb, ids, pv, grid)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pos, delta = dh.rope_index(ids, grid, mask)
        rows = dh.placeholder_rows(ids, fv.plan_for(grid).num_tokens)
        dh.embed_images(fv, emb, ids, pv, grid)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    dh.check()
    ref, _ = _host(ids_np, grid.numpy(), mask_np, False)
    assert torch.equal(pos.cpu(), ref[0]) and torch.equal(delta.cpu(), ref[1])
    assert torch.equal(rows, torch.nonzero(ids.flatten() == IMG).reshape(-1))


def test_one_cuda_graph_replays_new_inputs(dh, visual, cuda):
    """Rope index, placeholder rows and forward_into captured as one graph; replays after new ids, masks and patches of the
    same shape equal the eager host path."""
    fv = visual[torch.bfloat16]
    grid = torch.tensor([[1, 16, 20], [1, 8, 8], [1, 26, 36]])
    T = fv.plan_for(grid).num_tokens
    S = int((grid[:, 1] * grid[:, 2]).sum())
    ids_np, mask_np = _prompt(grid.numpy(), np.random.default_rng(0))
    ids_s, mask_s = torch.from_numpy(ids_np).to(cuda), torch.from_numpy(mask_np).to(cuda)
    pv_s = torch.zeros(S, 1176, device=cuda)
    emb_s = torch.zeros(ids_s.shape[0], ids_s.shape[1], 2048, dtype=torch.bfloat16, device=cuda)

    def step():
        pos, delta = dh.rope_index(ids_s, grid, mask_s)
        rows = dh.placeholder_rows(ids_s, T)
        fv.forward_into(emb_s, rows, pv_s, grid, validate_rows=False)
        return pos, delta

    side = torch.cuda.Stream(cuda)
    side.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream(cuda).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        pos, delta = step()
    for k, left in enumerate((True, False, True)):
        ids_np, mask_np = _prompt(grid.numpy(), np.random.default_rng(10 + k), left_pad=left)
        if k == 2:
            mask_np = np.where(mask_np == 0, 2, mask_np)           # pads marked 2: still pads in the image branch
        pv = torch.randn(S, 1176, generator=torch.Generator().manual_seed(20 + k)).to(cuda)
        emb0 = torch.randn(emb_s.shape, generator=torch.Generator().manual_seed(30 + k)).to(torch.bfloat16).to(cuda)
        ids_s.copy_(torch.from_numpy(ids_np))
        mask_s.copy_(torch.from_numpy(mask_np))
        pv_s.copy_(pv)
        emb_s.copy_(emb0)
        g.replay()
        dh.check()
        ref, err = _host(ids_np, grid.numpy(), mask_np, False)
        assert err is None
        assert torch.equal(pos.cpu(), ref[0]) and torch.equal(delta.cpu(), ref[1]), k
        ids = torch.from_numpy(ids_np).to(cuda)
        ref_emb = emb0.masked_scatter((ids == IMG).unsqueeze(-1).expand_as(emb0), fv(pv, grid))
        assert torch.equal(emb_s, ref_emb), k
