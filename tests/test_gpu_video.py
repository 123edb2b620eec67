"""GPU: video inputs through the fused path.  The drop-in video processor against the live HF ``Qwen2VLVideoProcessor``
(on the CPU, kind 1, and with ``device="cuda"``, kind 2), the window-ordered fp16 patches against the oracle, both
towers at full depth on batches mixing an image and two videos against HF's fp32 towers, CUDA-graph replay and
``return_pooling_output`` on video grids, and ``install()`` under HF's ``get_video_features``."""
import numpy as np
import pytest
import torch

from oracle import processor_video as OV, tower as OT

pytestmark = pytest.mark.gpu

# (frames, h, w, min_pixels, max_pixels): the CPU pin's list - even / odd, 1 and 2 frames, upscale, a 720p clip (tensor-core
# route), downscale past 10x (dp4a / per-tap route), one-axis, same size - plus an odd width (rows padded on upload)
GEOMETRIES = [
    (4, 120, 160, None, None), (5, 90, 200, None, None), (1, 300, 400, None, None), (2, 720, 1280, None, None),
    (3, 1600, 3000, 3136, 56 * 56 * 4), (2, 56, 900, 3136, 56 * 900), (3, 56, 84, 3136, 56 * 84), (3, 101, 333, None, None),
]


def _metrics(got, ref):
    got, ref = got.detach().double().cpu().flatten(), ref.detach().double().cpu().flatten()
    cos = (torch.dot(got, ref) / (got.norm() * ref.norm())).item()
    return cos, ((got - ref).abs().max() / ref.abs().max()).item()


def _video(seed, t, h, w):
    return np.random.default_rng(seed).integers(0, 256, (t, h, w, 3), dtype=np.uint8)


def _hf(mn, mx, **kw):
    from transformers.models.qwen2_vl.video_processing_qwen2_vl import Qwen2VLVideoProcessor
    return Qwen2VLVideoProcessor(min_pixels=mn or OV.MIN_PIXELS, max_pixels=mx or OV.MAX_PIXELS, **kw)


@pytest.mark.parametrize("device", [None, "cuda"], ids=["cpu_kind1", "cuda_kind2"])
@pytest.mark.parametrize("t,h,w,mn,mx", GEOMETRIES)
def test_dropin_bitexact_vs_live(cuda, device, t, h, w, mn, mx):
    from zoomearth_b200 import FusedVideoProcessor
    v = _video(t * 13 + w, t, h, w)
    kw = {} if device is None else {"device": device}
    want = _hf(mn, mx)(videos=[v], return_tensors="pt", **kw)
    vp = FusedVideoProcessor(min_pixels=mn or OV.MIN_PIXELS, max_pixels=mx or OV.MAX_PIXELS, device=cuda)
    got = vp(videos=[v], return_tensors="pt", **kw)
    assert got["video_grid_thw"].tolist() == want["video_grid_thw"].tolist()
    assert torch.equal(got["pixel_values_videos"], want["pixel_values_videos"].cpu())
    if device == "cuda":
        assert vp.last_launches == 2                         # fp32 resample of every frame + the video patchify
    else:
        assert 2 <= vp.last_launches <= 6                    # one integer route's passes for every frame + the patchify


def test_dropin_batch_sampling_and_metadata(cuda):
    """Two videos of different sizes (one channels-first tensor), sampled by fps, through the HF call surface."""
    from zoomearth_b200 import FusedVideoProcessor
    a, b = _video(1, 24, 120, 200), _video(2, 9, 200, 120)
    metas = [{"total_num_frames": 24, "fps": 12.0, "duration": 2.0}, {"total_num_frames": 9, "fps": 3.0, "duration": 3.0}]
    hf = _hf(None, None)
    want = hf(videos=[a, b], do_sample_frames=True, fps=2, video_metadata=metas, return_metadata=True, return_tensors="pt")
    vp = FusedVideoProcessor(device=cuda)
    got = vp(videos=[torch.from_numpy(a), torch.from_numpy(b).permute(0, 3, 1, 2)], do_sample_frames=True, fps=2,
             video_metadata=metas, return_metadata=True, return_tensors="pt")
    assert got["video_grid_thw"].tolist() == want["video_grid_thw"].tolist()
    assert torch.equal(got["pixel_values_videos"], want["pixel_values_videos"])
    assert [m.sampled_fps for m in got["video_metadata"]] == [m.sampled_fps for m in want["video_metadata"]]


@pytest.mark.parametrize("backend", ["torchvision", "torchvision_cuda"])
def test_fp16_window_order_equals_oracle(cuda, backend):
    from zoomearth_b200 import FusedVideoProcessor, Plan, _lib
    from zoomearth_b200.video import upload_video
    vids = [_video(3, 5, 300, 500), _video(4, 2, 720, 1280), _video(5, 1, 90, 90)]
    vp = FusedVideoProcessor(device=cuda)
    pv, grid = vp.preprocess_videos([upload_video(torch.from_numpy(v), cuda) for v in vids], torch.float16, True,
                                    backend=backend)
    ref, rgrid = OV.preprocess(vids, cuda=backend == "torchvision_cuda")
    assert grid.tolist() == rgrid.tolist()
    widx = Plan(_lib.default_cfg(), rgrid).window_index
    want = torch.from_numpy(ref).view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176).to(torch.float16)
    assert torch.equal(pv.cpu(), want)


# ---------------------------------------------------------------------------------------------- towers
MIXED = np.array([[1, 26, 36], [3, 20, 28], [4, 16, 24]])         # one image, two videos (odd and even t)


def _pixels(S, seed):
    u8 = torch.randint(0, 256, (S, 1176), generator=torch.Generator().manual_seed(seed)).float()
    return (u8 / 255.0 - 0.45) / 0.27


@torch.no_grad()
def _hf_forward(m, pv, grid):
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        dev = next(m.parameters()).device
        out = m(pv.to(dev, torch.float32), grid_thw=torch.as_tensor(grid).to(dev))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return out.pooler_output, out.last_hidden_state


def _qwen25(cuda):
    from oracle import hf_live
    return hf_live.hf_tower(None, OT.CFG, seed=21).to(cuda)          # Qwen2.5-VL-3B geometry, 32 blocks, random init


def _qwen2(cuda):
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLVisionConfig
    from transformers.models.qwen2_vl.modeling_qwen2_vl import Qwen2VisionTransformerPretrainedModel
    vc = Qwen2VLVisionConfig(depth=32, embed_dim=1280, num_heads=16, mlp_ratio=4, hidden_act="quick_gelu", hidden_size=1536)
    torch.manual_seed(22)
    with torch.device(cuda):
        m = Qwen2VisionTransformerPretrainedModel._from_config(vc, attn_implementation="sdpa")
    with torch.no_grad():                                  # non-trivial LayerNorm gains and biases (HF inits 1 and 0)
        g = torch.Generator(device=cuda).manual_seed(23)
        for name, p in m.named_parameters():
            r = torch.randn(p.shape, generator=g, device=cuda)
            if ("norm" in name or "ln_q" in name) and name.endswith("weight"):
                p.copy_(1 + 0.1 * r)
            elif name.endswith("bias"):
                p.copy_(0.1 * r)
            else:
                p.copy_(0.02 * r)
    return m.float().eval()


@pytest.mark.parametrize("tower", ["qwen25", "qwen2"])
def test_full_depth_tower_on_image_and_videos_vs_hf(cuda, tower):
    from zoomearth_b200 import FusedVisual
    m = _qwen25(cuda) if tower == "qwen25" else _qwen2(cuda)
    S = int((MIXED[:, 0] * MIXED[:, 1] * MIXED[:, 2]).sum())
    pv = _pixels(S, 31)
    ref, ref_hidden = _hf_forward(m, pv, MIXED)
    fv = FusedVisual.from_hf(m, device=cuda, dtype=torch.float32, operand_dtype=torch.float16)
    out = fv(pv.to(cuda), torch.from_numpy(MIXED))
    cos, maxrel = _metrics(out, ref)
    print(f"{tower} full depth, image + videos t=3, t=4: cosine {cos:.6f}, max rel err {maxrel:.3e}")
    assert cos >= 0.999 and maxrel <= 1e-2, f"cos {cos} maxrel {maxrel}"
    # every frame group's tokens depend on that group only: the video alone gives its rows of the batch
    solo = fv(pv[936:936 + 3 * 560].to(cuda), torch.from_numpy(MIXED[1:2]))
    assert _metrics(solo, out[234:234 + 420])[1] <= 2e-3
    # CUDA-graph replay of the same video grid
    graph = fv(pv.to(cuda), torch.from_numpy(MIXED), use_graph=True)
    assert _metrics(graph, out)[1] <= 1e-3
    # return_pooling_output: last_hidden_state as HF returns it (window order for Qwen2.5-VL, HF order for Qwen2-VL)
    fv.return_pooling_output = True
    o = fv(pv.to(cuda), torch.from_numpy(MIXED))
    assert _metrics(o.pooler_output, ref)[1] <= 1e-2
    if tower == "qwen2":
        ch, mh = _metrics(o.last_hidden_state, ref_hidden)
        assert ch >= 0.999 and mh <= 1e-2, f"hidden: cos {ch} maxrel {mh}"


def test_encode_video_matches_hf_tower_on_oracle_patches(cuda):
    """ZoomEncoder.encode_video: uint8 CUDA frames -> window-order fp16 patches -> tower, against HF's tower on the
    oracle's patches."""
    from oracle import hf_live
    from zoomearth_b200 import FusedVisual, ZoomEncoder
    cfg = OT.small_cfg(depth=4, fullatt=(3,))
    m = hf_live.hf_tower(None, cfg, seed=5).to(cuda)
    fv = FusedVisual.from_hf(m, device=cuda, dtype=torch.float32, operand_dtype=torch.float16)
    enc = ZoomEncoder(fv)
    vids = [_video(6, 5, 240, 320), _video(7, 2, 480, 640)]
    emb, grid = enc.encode_video([torch.from_numpy(v).to(cuda) for v in vids])
    ref_pv, rgrid = OV.preprocess(vids, cuda=True)
    assert grid.tolist() == rgrid.tolist()
    ref, _ = _hf_forward(m, torch.from_numpy(ref_pv), rgrid)
    cos, maxrel = _metrics(emb, ref)
    assert cos >= 0.999 and maxrel <= 1e-2, f"cos {cos} maxrel {maxrel}"
    assert enc.last_launches > 2


def test_install_get_video_features_vs_unreplaced(cuda):
    import transformers
    from transformers import Qwen2_5_VLConfig, Qwen2_5_VLForConditionalGeneration
    from zoomearth_b200 import install
    vis = dict(depth=2, hidden_size=1280, intermediate_size=3420, num_heads=16, out_hidden_size=2048, patch_size=14,
               spatial_merge_size=2, temporal_patch_size=2, window_size=112, fullatt_block_indexes=[1], hidden_act="silu")
    text = dict(hidden_size=2048, intermediate_size=256, num_hidden_layers=1, num_attention_heads=16, num_key_value_heads=2,
                vocab_size=152064, max_position_embeddings=4096,
                rope_parameters={"rope_type": "default", "mrope_section": [16, 24, 24], "rope_theta": 1000000.0})
    try:
        config = Qwen2_5_VLConfig(vision_config=vis, text_config=text)
    except Exception as e:                       # config schema differs across transformers majors
        pytest.skip(f"cannot build a tiny Qwen2_5_VLConfig on transformers {transformers.__version__}: {e}")
    torch.manual_seed(0)
    model = Qwen2_5_VLForConditionalGeneration(config).eval()
    owner = model if hasattr(model, "visual") else model.model
    vgrid = torch.tensor([[3, 16, 20], [2, 8, 8]])
    igrid = torch.tensor([[1, 16, 20]])
    pvv = _pixels(int((vgrid[:, 0] * vgrid[:, 1] * vgrid[:, 2]).sum()), 41)
    pvi = _pixels(320, 42)

    def _split(f):
        f = f.pooler_output if hasattr(f, "pooler_output") else f
        return list(f) if isinstance(f, (list, tuple)) else [f]
    with torch.no_grad():
        ref_v = _split(owner.get_video_features(pvv, vgrid))
        ref_i = _split(owner.get_image_features(pvi, igrid))
    install(model, device=cuda, dtype=torch.float32)
    with torch.no_grad():
        got_v = _split(owner.get_video_features(pvv.to(cuda), vgrid.to(cuda)))
        got_i = _split(owner.get_image_features(pvi.to(cuda), igrid.to(cuda)))
    for got, want in ((got_v, ref_v), (got_i, ref_i)):
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert a.shape == b.shape
            cos, maxrel = _metrics(a, b)
            assert cos >= 0.999 and maxrel <= 1e-2, f"cos {cos} maxrel {maxrel}"
