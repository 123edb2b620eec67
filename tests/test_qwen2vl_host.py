"""Qwen2-VL tower (zv_cfg.tower_kind = 1), host side (no GPU): the HF config mapping, the weight layout size, the argument
checks that run before any device work, and a restatement of the folded-LayerNorm epilogue arithmetic against
torch.nn.functional.layer_norm followed by the linear."""
import ctypes as C

import numpy as np
import pytest
import torch

H, SLOTS = 1280, 20


def _qwen2_cfg(**kw):
    from zoomearth_b200 import _lib
    from zoomearth_b200.visual import _vision_cfg_from_hf
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLVisionConfig
    return _lib.default_cfg(**_vision_cfg_from_hf(Qwen2VLVisionConfig(**kw)))


def test_cfg_from_qwen25_config_unchanged(lib):
    from transformers.models.qwen2_5_vl.configuration_qwen2_5_vl import Qwen2_5_VLVisionConfig
    from zoomearth_b200.visual import _vision_cfg_from_hf
    c = Qwen2_5_VLVisionConfig(hidden_size=1280, out_hidden_size=2048)
    assert _vision_cfg_from_hf(c) == dict(depth=32, hidden=1280, heads=16, inter=3420, out_hidden=2048, patch=14, merge=2,
                                          temporal=2, window=112, fullatt=[7, 15, 23, 31])


@pytest.mark.parametrize("out_width", [1536, 3584, 8192])
def test_cfg_from_qwen2vl_config(lib, out_width):
    from zoomearth_b200 import _lib
    cfg = _qwen2_cfg(embed_dim=1280, num_heads=16, mlp_ratio=4, hidden_act="quick_gelu", hidden_size=out_width)
    dflt = _lib.default_cfg()
    assert (cfg.tower_kind, cfg.depth, cfg.hidden, cfg.heads, cfg.inter, cfg.out_hidden) == (1, 32, 1280, 16, 5120, out_width)
    assert cfg.fullatt_mask_lo & 0xffffffff == 0xffffffff
    for f in ("patch", "merge", "temporal", "window", "min_size", "op_dtype", "min_pixels", "max_pixels", "eps"):
        assert getattr(cfg, f) == getattr(dflt, f), f
    assert dflt.tower_kind == 0


def test_cfg_from_qwen2vl_other_activation_refused(lib):
    with pytest.raises(NotImplementedError, match="quick_gelu"):
        _qwen2_cfg(hidden_act="gelu")


def test_weights_bytes_kind1(lib):
    cfg = _qwen2_cfg(hidden_size=1536)
    L = 32
    al = lambda b: (b + 255) // 256 * 256                                           # noqa: E731
    per_block = 4 * al(H * 4) + al(3 * H * H * 2) + 2 * al(3 * H * 4) + al(H * H * 2) + al(H * 4) \
        + al(5120 * H * 2) + 2 * al(5120 * 4) + al(H * 5120 * 2) + al(H * 4)
    want = al(H * 1176 * 2) + L * per_block + 2 * al(H * 4) + al(16 * H * H * 2) + al(4 * H * 4) + al(1536 * 4 * H * 2) + al(1536 * 4)
    assert lib.zv_weights_bytes(C.byref(cfg)) == want


@pytest.mark.parametrize("change,msg", [(dict(fullatt_mask_lo=0x7fffffff), "window blocks"), (dict(inter=3420), "inter=5120")])
def test_kind1_einval(lib, change, msg):
    from zoomearth_b200 import _lib
    cfg = _qwen2_cfg(hidden_size=1536)
    for k, v in change.items():
        setattr(cfg, k, v)
    assert lib.zv_weights_bytes(C.byref(cfg)) == _lib.ZV_EINVAL
    assert msg in lib.zv_last_error().decode()
    cfg = _lib.default_cfg(tower_kind=2)
    assert lib.zv_weights_bytes(C.byref(cfg)) == _lib.ZV_EINVAL


def _descs(names):
    from zoomearth_b200 import _lib
    arr = (_lib.ZvTensor * len(names))()
    keep = [n.encode() for n in names]
    for d, n in zip(arr, keep):
        d.name, d.data, d.dtype, d.ndim = n, None, _lib.ZV_F32, 1
    return arr, keep


def _tower_names(depth):
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLVisionConfig
    from transformers.models.qwen2_vl.modeling_qwen2_vl import Qwen2VisionTransformerPretrainedModel
    with torch.device("meta"):
        m = Qwen2VisionTransformerPretrainedModel._from_config(Qwen2VLVisionConfig(depth=depth, hidden_size=1536))
    return [k for k in m.state_dict() if "inv_freq" not in k]


@pytest.mark.parametrize("drop,extra", [("blocks.1.norm1.bias", None), ("merger.ln_q.bias", None),
                                        (None, "blocks.2.mlp.gate_proj.weight")])
def test_pack_missing_or_extra_tensor_named(lib, drop, extra):
    """Checked before any device work, so the error is the same with or without a GPU."""
    from zoomearth_b200 import _lib
    cfg = _qwen2_cfg(depth=2, hidden_size=1536)
    names = _tower_names(2)
    assert "blocks.1.norm1.bias" in names and len(names) == 1 + 2 * 12 + 6
    names = [n for n in names if n != drop] + ([extra] if extra else [])
    arr, _keep = _descs(names)
    rc = lib.zv_weights_pack(C.byref(cfg), arr, len(names), C.c_void_p(256), 1 << 40, None)
    assert rc == _lib.ZV_EINVAL
    assert (drop or extra) in lib.zv_last_error().decode()


# ---- the folded LayerNorm, restated: producer slot statistics -> Chan merge in slot order -> r (acc - mu c) + b'
def _slot_stats_two_pass(x):
    """cast_rows_ln: per 64-column slot (mean, M2), two-pass, fp32."""
    s = x.reshape(x.shape[0], SLOTS, 64)
    mean = s.sum(-1, dtype=np.float32) / np.float32(64)
    return mean, ((s - mean[..., None]) ** 2).sum(-1, dtype=np.float32)


def _slot_stats_shifted(x, half=128):
    """EPI_RESID_LN: per tile half, sums of (x - x0) and (x - x0)^2 with x0 the half's first value; a 128-column half
    stores (mean, M2 / 2) in both of its slots."""
    s = x.reshape(x.shape[0], H // half, half)
    d = s - s[..., :1]
    s1, s2 = d.sum(-1, dtype=np.float32), (d * d).sum(-1, dtype=np.float32)
    mo = s1 / np.float32(half)
    mean, m2 = s[..., 0] + mo, np.maximum(s2 - s1 * mo, 0)
    k = half // 64
    return np.repeat(mean, k, 1), np.repeat(m2 / np.float32(k), k, 1)


def _merge(mean_s, m2_s):
    mean, m2 = mean_s[:, 0].copy(), m2_s[:, 0].copy()
    for k in range(1, SLOTS):
        d = mean_s[:, k] - mean
        mean = mean + d * np.float32(1 / (k + 1))
        m2 = m2 + (m2_s[:, k] + d * d * np.float32(64 * k / (k + 1)))
    return mean, m2


@pytest.mark.parametrize("rows", ["offset8", "constant"])
@pytest.mark.parametrize("stats", ["two_pass", "shifted128", "shifted64"])
def test_layernorm_fold_restated(rows, stats):
    g = torch.Generator().manual_seed(5)
    N, eps = 96, 1e-6
    if rows == "offset8":       # |mean| / std = 8: the rows the residual stream carries when the weights have a common mode
        x = torch.randn(16, H, generator=g) * 0.5 + 4.0 * torch.sign(torch.randn(16, 1, generator=g))
    else:                       # constant rows: var = 0, only eps keeps r finite (values exact in fp16)
        x = torch.tensor([2.5, -3.0, 0.0, 1.0]).repeat_interleave(H).view(4, H)
    W = torch.randn(N, H, generator=g) * 0.02
    b = 0.1 * torch.randn(N, generator=g)
    gain = 1 + 0.1 * torch.randn(H, generator=g)
    beta = 0.1 * torch.randn(H, generator=g)
    ref = (torch.nn.functional.layer_norm(x.double(), (H,), gain.double(), beta.double(), eps) @ W.double().t() + b.double())

    Wp = (W * gain).half()                                   # packed weights: gain folded, rounded once
    c = Wp.float().sum(1).numpy()                            # column sums of what the MMA multiplies
    bp = (b + W @ beta).numpy()                              # b' = b + W beta, fp32 from the fp32 weights
    acc = (x.half().float() @ Wp.float().t()).numpy()        # tensor cores: 16-bit operands, fp32 accumulation
    xf = x.numpy().astype(np.float32)
    mean_s, m2_s = {"two_pass": _slot_stats_two_pass, "shifted128": _slot_stats_shifted,
                    "shifted64": lambda v: _slot_stats_shifted(v, 64)}[stats](xf)
    mu, m2 = _merge(mean_s, m2_s)
    np.testing.assert_allclose(mu, xf.astype(np.float64).mean(1), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(m2 / H, xf.astype(np.float64).var(1), rtol=1e-4, atol=1e-9)
    r = 1 / np.sqrt(m2 / np.float32(H) + np.float32(eps))
    out = r[:, None] * (acc - mu[:, None] * c[None, :]) + bp[None, :]
    rel = np.abs(out - ref.numpy()).max() / np.abs(ref.numpy()).max()
    # constant rows: r = 1/sqrt(eps) = 1000 scales the fp32 rounding of acc - mu c up
    assert rel <= (5e-3 if rows == "offset8" else 2e-3), rel


def test_crop_cost_full_layers():
    """Qwen2.5-VL partitions are unchanged by the default; a Qwen2-VL tower (32 full-attention blocks) weighs long crops
    by their quadratic attention term."""
    from zoomearth_b200 import sharding
    grids = np.array([[1, 70, 70], [1, 36, 36], [1, 8, 8]])
    S = (grids[:, 1] * grids[:, 2]).astype(np.float64)
    np.testing.assert_array_equal(sharding.crop_cost(grids), sharding.crop_cost(grids, 4))
    np.testing.assert_allclose(sharding.crop_cost(grids), 5.125e9 * S / 4 + 4 * 4 * S * S * 1280 + 28 * 4 * 64 * S * 1280)
    np.testing.assert_allclose(sharding.crop_cost(grids, 32), 5.125e9 * S / 4 + 32 * 4 * S * S * 1280)
