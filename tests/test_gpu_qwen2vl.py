"""Qwen2-VL tower (tower_kind = 1) on the GPU against the installed HF ``Qwen2VisionTransformerPretrainedModel`` in fp32
(sdpa, TF32 off).  HF initialises LayerNorm gains to 1 and every bias to 0, which would leave both LayerNorm folds
(gain into the weights, bias into the consumer's bias) untested: the towers here get seeded random gains 1 + 0.1 randn
and norm / linear biases 0.1 randn."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _metrics(got, ref):
    got, ref = got.detach().double().cpu().flatten(), ref.detach().double().cpu().flatten()
    cos = (torch.dot(got, ref) / (got.norm() * ref.norm())).item()
    return cos, ((got - ref).abs().max() / ref.abs().max()).item()


def _vision_config(depth, out_width):
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLVisionConfig
    return Qwen2VLVisionConfig(depth=depth, embed_dim=1280, num_heads=16, mlp_ratio=4, hidden_act="quick_gelu",
                               hidden_size=out_width)


@torch.no_grad()
def _randomize(tower, seed):
    g = torch.Generator(device=next(tower.parameters()).device).manual_seed(seed)
    for name, p in tower.named_parameters():
        r = torch.randn(p.shape, generator=g, device=p.device)
        if ("norm" in name or "ln_q" in name) and name.endswith("weight"):
            p.copy_(1 + 0.1 * r)
        elif name.endswith("bias"):
            p.copy_(0.1 * r)
        else:
            p.copy_(0.02 * r)
    return tower


def _hf_tower(depth, out_width, seed, device):
    from transformers.models.qwen2_vl.modeling_qwen2_vl import Qwen2VisionTransformerPretrainedModel
    with torch.device(device):
        m = Qwen2VisionTransformerPretrainedModel._from_config(_vision_config(depth, out_width), attn_implementation="sdpa")
    return _randomize(m.float().eval(), seed)


@torch.no_grad()
def _hf_forward(m, pv, grid):
    """fp32 oracle with TF32 off (the patch embed is a conv3d: cudnn too)."""
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        dev = next(m.parameters()).device
        out = m(pv.to(dev, torch.float32), grid_thw=torch.as_tensor(grid).to(dev))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return out.pooler_output, out.last_hidden_state


def _fused(m, cuda, operand=torch.float16, dtype=torch.float32):
    from zoomearth_b200 import FusedVisual
    return FusedVisual.from_hf(m, device=cuda, dtype=dtype, operand_dtype=operand)


def _pixels(S, seed):
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (S, 1176), generator=g).float()
    return (u8 / 255.0 - 0.45) / 0.27


@pytest.fixture(scope="module")
def small_tower(cuda):
    return _hf_tower(3, 1536, 1, cuda)


@pytest.mark.parametrize("operand", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("grid", [[[1, 2, 2]], [[1, 8, 8]], [[1, 26, 36], [1, 8, 8], [1, 18, 34], [1, 2, 2]], [[1, 36, 36]],
                                  [[1, 2, 200]]])
def test_qwen2vl_small_depth_vs_hf(cuda, small_tower, grid, operand):
    grid = np.array(grid)
    S = int((grid[:, 1] * grid[:, 2]).sum())
    pv = torch.randn(S, 1176, generator=torch.Generator().manual_seed(S))
    ref, ref_hidden = _hf_forward(small_tower, pv, grid)
    fv = _fused(small_tower, cuda, operand)
    assert fv.cfg.tower_kind == 1 and fv.cfg.out_hidden == 1536
    out, hidden = fv(pv.to(cuda), torch.from_numpy(grid), return_hidden=True)
    co, mo = _metrics(out, ref)
    ch, mh = _metrics(hidden, ref_hidden)                   # last_hidden_state in HF order, as HF's class returns it
    assert co >= 0.999 and mo <= 1e-2, f"merged: cos {co} maxrel {mo}"
    assert ch >= 0.999 and mh <= 1e-2, f"hidden: cos {ch} maxrel {mh}"
    if operand == torch.float16:
        assert mo <= 2e-3 and mh <= 2e-3, f"fp16 operands at depth 3: merged {mo}, hidden {mh}"


def test_qwen2vl_return_pooling_output_hf_order(cuda, small_tower):
    grid = np.array([[1, 16, 20], [1, 8, 8]])
    pv = torch.randn(int((grid[:, 1] * grid[:, 2]).sum()), 1176, generator=torch.Generator().manual_seed(3))
    ref, ref_hidden = _hf_forward(small_tower, pv, grid)
    fv = _fused(small_tower, cuda)
    fv.return_pooling_output = True
    o = fv(pv.to(cuda), torch.from_numpy(grid))
    assert _metrics(o.pooler_output, ref)[1] <= 2e-3 and _metrics(o.last_hidden_state, ref_hidden)[1] <= 2e-3


# Full depth (32 blocks, all full attention), fp16 operands.  The offset case adds a common mode to the patch-embed
# weights (W + 1 u^T) so that residual rows carry |mean| / std of about 8: the statistics must not cancel.
FULL_CASES = [
    ("global view 980x980", [[1, 70, 70]], 1536, False, 70),
    ("ragged: 64x92 zoom crop + 4x200 strip", [[1, 26, 36], [1, 8, 8], [1, 64, 92], [1, 4, 200]], 3584, False, 11),
    ("offset guard, global view 980x980", [[1, 70, 70]], 1536, True, 71),
]


@pytest.mark.parametrize("name,grid,width,offset,seed", FULL_CASES, ids=["global980", "ragged", "offset"])
def test_qwen2vl_full_depth_vs_hf(cuda, name, grid, width, offset, seed):
    m = _hf_tower(32, width, 100 + width, cuda)
    if offset:
        with torch.no_grad():
            w = m.patch_embed.proj.weight                    # (1280, 3, 2, 14, 14): every output row gets the same u
            u = 0.24 * torch.randn(w[0].shape, generator=torch.Generator(device=cuda).manual_seed(9), device=cuda)
            w += u
    grid = np.array(grid)
    S = int((grid[:, 1] * grid[:, 2]).sum())
    pv = _pixels(S, seed)
    ref, ref_hidden = _hf_forward(m, pv, grid)
    if offset:
        x0 = m.patch_embed(pv.to(cuda)).double()
        ratio = (x0.mean(1).abs() / x0.std(1)).median().item()
        print(f"offset guard: patch-embed rows |mean|/std median {ratio:.2f}")
        assert ratio >= 7
    fv = _fused(m, cuda)
    out, hidden = fv(pv.to(cuda), torch.from_numpy(grid), return_hidden=True)
    assert out.shape == (S // 4, width)
    cos, maxrel = _metrics(out, ref)
    ch, mh = _metrics(hidden, ref_hidden)
    print(f"PARITY Qwen2-VL full tower fp16 operands vs HF fp32 [{name}, out {width}]: S={S} cosine {cos:.6f}, "
          f"max rel err {maxrel:.3e}; last_hidden_state cosine {ch:.6f}, max rel err {mh:.3e}")
    assert cos >= 0.999 and maxrel <= 1e-2, f"{name}: cos {cos} maxrel {maxrel}"
    assert ch >= 0.999 and mh <= 1e-2, f"{name} hidden: cos {ch} maxrel {mh}"


def test_qwen2vl_install_logits(cuda):
    """install() on a tiny Qwen2VLForConditionalGeneration: the logits of the patched model match the unpatched fp32 one."""
    from transformers import Qwen2VLConfig, Qwen2VLForConditionalGeneration
    from zoomearth_b200 import install
    vis = dict(depth=2, embed_dim=1280, num_heads=16, mlp_ratio=4, hidden_act="quick_gelu", hidden_size=1536)
    text = dict(hidden_size=1536, intermediate_size=512, num_hidden_layers=1, num_attention_heads=12, num_key_value_heads=2,
                vocab_size=152064, max_position_embeddings=4096,
                rope_parameters={"rope_type": "default", "mrope_section": [16, 24, 24], "rope_theta": 1000000.0})
    torch.manual_seed(0)
    with torch.device(cuda):
        model = Qwen2VLForConditionalGeneration(Qwen2VLConfig(vision_config=vis, text_config=text)).float().eval()
    owner = model if hasattr(model, "visual") else model.model
    _randomize(owner.visual, 4)
    grid = torch.tensor([[1, 16, 20], [1, 8, 8]])
    pv = torch.randn(int((grid[:, 1] * grid[:, 2]).sum()), 1176, generator=torch.Generator().manual_seed(2))
    cfg = model.config
    ids = [1, 2, 3]
    for g in grid.tolist():
        ids += [cfg.vision_start_token_id] + [cfg.image_token_id] * (g[1] * g[2] // 4) + [cfg.vision_end_token_id, 7]
    ids = torch.tensor([ids], device=cuda)
    kw = dict(input_ids=ids, attention_mask=torch.ones_like(ids), mm_token_type_ids=(ids == cfg.image_token_id).long(),
              pixel_values=pv.to(cuda), image_grid_thw=grid.to(cuda))
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            ref = model(**kw).logits
            fv, _ = install(model, device=cuda, dtype=torch.float32)
            assert owner.visual is fv and fv.cfg.tower_kind == 1
            got = model(**kw).logits
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    cos, maxrel = _metrics(got, ref)
    print(f"install on Qwen2-VL: logits cosine {cos:.6f}, max rel err {maxrel:.3e}")
    assert cos >= 0.999, f"cos {cos} maxrel {maxrel}"


def _encoder(cuda, m, max_pixels=401408):
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    return ZoomEncoder(_fused(m, cuda), FusedImageProcessor(min_pixels=3136, max_pixels=max_pixels, device=cuda))


def test_qwen2vl_paths(cuda, small_tower):
    """ZoomEncoder (window-ordered K1 patches) vs the HF-order path, CUDA-graph replay vs eager, forward_into vs
    masked_scatter, and the launch accounting of the kind-1 forward."""
    from zoomearth_b200 import _lib
    enc = _encoder(cuda, small_tower)
    fv = enc.visual
    img = np.random.default_rng(3).integers(0, 256, (1500, 2000, 3), dtype=np.uint8)
    dev = enc.upload(img)
    emb, grid, crop, pv = enc.encode([dev], [(100, 200, 1300, 1100), (900.5, 700.2, 1100.9, 800.0)], image_index=[0, 0],
                                     return_patches=True)
    assert enc.visual.last_launches == 2 + 5 * 3 + 3          # patch embed + cast_rows_ln, 5 per block, merger
    plan = fv.plan_for(grid)
    rev = torch.from_numpy(plan.reverse_index.copy()).to(cuda)
    pv_hf = pv.view(-1, 4, 1176).index_select(0, rev).reshape(-1, 1176)
    ref = fv(pv_hf, grid)
    assert fv.last_launches == 1 + 2 + 5 * 3 + 3              # + the HF -> window order gather
    assert _metrics(emb, ref)[1] <= 1e-3
    ref_hf, _ = _hf_forward(small_tower, pv_hf.float(), grid)
    cos, maxrel = _metrics(emb, ref_hf)
    assert cos >= 0.999 and maxrel <= 1e-2
    # CUDA graph
    g1 = fv(pv_hf, grid, use_graph=True)
    assert torch.equal(g1, ref) and torch.equal(fv(pv_hf, grid, use_graph=True), ref)
    # LM hand-off fused into the last GEMM
    T = ref.shape[0]
    L = T + 37
    mask = torch.zeros(2, L, dtype=torch.bool)
    mask[0, 5:5 + T // 2] = True
    mask[1, 3:3 + T - T // 2] = True
    mask = mask.to(cuda)
    e0 = torch.randn(2, L, fv.cfg.out_hidden, generator=torch.Generator().manual_seed(6)).to(cuda)
    want = e0.masked_scatter(mask.unsqueeze(-1).expand_as(e0), ref)
    got = fv.forward_into(e0.clone(), mask.flatten().nonzero().flatten(), pv_hf, grid)
    assert torch.equal(got, want)
    assert fv.last_launches == 1 + 2 + 5 * 3 + 3 + 1          # + compose_rows
    # per-class timing: every block is a full-attention launch, none a window-attention one
    lib = _lib.lib()
    lib.zv_timing_reset()
    lib.zv_timing_enable(1)
    fv(pv_hf, grid)
    torch.cuda.synchronize()
    lib.zv_timing_enable(0)
    counts = {}
    for cls in (8, 9, 12):
        t, n = C.c_double(), C.c_int64()
        _lib.check(lib.zv_timing_read(cls, C.byref(t), C.byref(n)))
        counts[cls] = n.value
    lib.zv_timing_reset()
    assert counts == {8: 0, 9: 3, 12: 3}, counts


def test_qwen2vl_zoom_session(cuda, small_tower):
    from zoomearth_b200 import ZoomSession
    enc = _encoder(cuda, small_tower, 200704)
    sess = ZoomSession(enc)
    img = np.random.default_rng(50).integers(0, 256, (900, 1200, 3), dtype=np.uint8)
    sess.add_image("a", img)
    e1, _ = sess.stage1(["a"])
    out, crop = sess.stage2(["a"], [(100, 100, 700, 600)])
    (embs, grid), = out
    ref, rgrid, _ = enc.encode([sess.add_image("a", None)], [(100, 100, 700, 600)], image_index=[0])
    assert grid[1].tolist() == rgrid[0].tolist()
    cos, maxrel = _metrics(embs[1], ref)
    assert cos >= 0.9995 and maxrel <= 1e-2
    assert e1[0].shape[1] == 1536
