"""CPU: the torchvision resample / normalise convention (ZV_RESAMPLE_TORCHVISION, FusedImageProcessor(backend=
"torchvision"), install(image_backend=...)).  The NumPy oracle is pinned against the installed torch / torchvision /
transformers run live; the library's tables, LUT and the CPU emulation of K1's tensor-core route are pinned against the
oracle and the live HF torchvision-backend processor."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import geometry as OG, processor as OP, processor_torchvision as PT, resample as OR, resample_torchvision as RT
from zoomearth_b200 import _lib


def _img(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _smooth(seed, h, w):
    """low-frequency content: long runs of near-equal values, where the rounding of a pass decides most outputs"""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    f = [127.5 + 127.5 * np.sin(x / rng.uniform(20, 300) + y / rng.uniform(20, 300) + rng.uniform(0, 6)) for _ in range(3)]
    return np.clip(np.stack(f, -1), 0, 255).astype(np.uint8)


def _tv_resize(img, oh, ow):
    from torchvision.transforms.v2 import functional as tvF
    t = torch.from_numpy(np.ascontiguousarray(img)).permute(2, 0, 1)
    return tvF.resize(t, [oh, ow], interpolation=tvF.InterpolationMode.BICUBIC, antialias=True).permute(1, 2, 0).numpy()


def _hf_tv(images, min_pixels, max_pixels, **kw):
    """the live transformers 5.x torchvision-backend processor (what AutoImageProcessor returns for Qwen2-VL)"""
    from PIL import Image
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    p = Qwen2VLImageProcessor(min_pixels=min_pixels, max_pixels=max_pixels, **kw)
    out = p(images=[Image.fromarray(i) for i in images], return_tensors="pt")
    return out["pixel_values"].numpy(), out["image_grid_thw"].numpy()


def _geometries():
    """(seed, h, w, out_h, out_w, content): downscales up to 35x (5000-wide past 10x), upscales to min_pixels,
    one-axis resizes, same-size axes"""
    rng = np.random.default_rng(2024)
    g = [(1, 900, 1300, 280, 392, "rand"), (2, 300, 5000, 28, 476, "rand"), (3, 200, 5000, 56, 140, "smooth"),
         (4, 120, 5000, 56, 392, "rand"), (5, 400, 5000, 392, 420, "smooth"), (6, 30, 30, 56, 56, "rand"),
         (7, 7, 9, 56, 84, "smooth"), (8, 44, 60, 56, 84, "rand"), (9, 300, 420, 308, 420, "rand"),
         (10, 504, 700, 504, 728, "smooth"), (11, 512, 512, 504, 504, "rand"), (12, 640, 28, 644, 28, "rand"),
         (13, 1500, 1500, 56, 56, "rand"), (14, 100, 100, 3500, 140, "smooth"), (15, 2000, 60, 56, 56, "rand"),
         (16, 256, 4096, 28, 644, "smooth")]
    for k in range(28):
        h, w = int(rng.integers(8, 900)), int(rng.integers(8, 1400))
        s = float(rng.uniform(0.3, 12.0))
        oh = h if k % 7 == 0 else max(1, int(h / s))
        ow = w if k % 7 == 3 else max(1, int(w / rng.uniform(0.3, 12.0)))
        g.append((100 + k, h, w, oh, ow, "smooth" if k % 2 else "rand"))
    return g


GEOMETRIES = _geometries()


def test_oracle_resample_vs_live_torchvision():
    assert len(GEOMETRIES) >= 40
    for seed, h, w, oh, ow, content in GEOMETRIES:
        img = (_smooth if content == "smooth" else _img)(seed, h, w)
        got = RT.resize_u8(img, ow, oh)
        ref = _tv_resize(img, oh, ow)
        assert np.array_equal(got, ref), (h, w, oh, ow, content, int((got != ref).sum()))


def test_oracle_resample_differs_from_pillow():
    """the two conventions really are different pixels (the reason the convention exists)"""
    img = _img(1, 900, 1300)
    assert not np.array_equal(RT.resize_u8(img, 392, 280), OR.resize_u8(img, 392, 280))


def test_oracle_processor_vs_live_hf():
    imgs = [_img(1, 300, 420), _img(2, 60, 44), _smooth(3, 900, 1300), _img(4, 28, 700)]
    pv, grid, _ = PT.preprocess_u8(imgs, 3136, 100352)
    hpv, hgrid = _hf_tv(imgs, 3136, 100352)
    assert hgrid.tolist() == grid.tolist() and np.array_equal(hpv, pv)


@pytest.mark.parametrize("mean,std", [(OP.OPENAI_CLIP_MEAN, OP.OPENAI_CLIP_STD), ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])
def test_lut_all_768_levels_vs_live_hf(lib, mean, std):
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    p = Qwen2VLImageProcessor(image_mean=list(mean), image_std=list(std))
    levels = torch.arange(256, dtype=torch.uint8).view(1, 1, 1, 256).expand(1, 3, 1, 256).contiguous()
    ref = p.rescale_and_normalize(levels, True, p.rescale_factor, True, p.image_mean, p.image_std)[0, :, 0, :].numpy()
    from zoomearth_b200 import geometry as G
    lut = G.normalize_lut(_lib.default_cfg(mean=mean, std=std, resample_kind=_lib.RESAMPLE_TORCHVISION))
    assert lut.view(np.uint32).tolist() == ref.view(np.uint32).tolist()
    assert np.array_equal(PT.normalize_lut(mean, std), ref)
    # the PIL convention keeps its own table, and the two differ
    pil = G.normalize_lut(_lib.default_cfg(mean=mean, std=std))
    assert np.array_equal(pil, OP.normalize_lut(mean, std)) and not np.array_equal(pil, lut)


def test_resample_coeffs_ex_vs_oracle(lib):
    from zoomearth_b200 import geometry as G
    pairs = {(i, o) for _, h, w, oh, ow, _ in GEOMETRIES for i, o in ((h, oh), (w, ow))}
    pairs |= {(5000, 28), (5000, 980), (1, 56), (3, 1), (420, 420)}
    precisions = set()
    for i, o in sorted(pairs):
        ks, b, k, p = G.resample_coeffs_ex(_lib.RESAMPLE_TORCHVISION, i, o)
        rb, rk, rp = RT.coeffs_22bit(i, o)
        assert p == rp and np.array_equal(b, rb), (i, o)
        assert np.array_equal(k[:, :rk.shape[1]], rk) and not k[:, rk.shape[1]:].any(), (i, o)
        assert (k % (1 << (22 - p)) == 0).all()
        precisions.add(p)
        ks0, b0, k0 = G.resample_coeffs(i, o)
        ks1, b1, k1, p1 = G.resample_coeffs_ex(_lib.RESAMPLE_PIL, i, o)
        assert (ks0, p1) == (ks1, 22) and np.array_equal(b0, b1) and np.array_equal(k0, k1), (i, o)
    assert len(precisions) >= 5                       # upscales (14) up to large downscales (21)
    with pytest.raises(_lib.ZoomVitError, match="resample_kind 2"):
        G.resample_coeffs_ex(2, 100, 50)


def test_default_cfg_and_exports(lib):
    assert _lib.default_cfg().resample_kind == _lib.RESAMPLE_PIL == 0
    assert "zv_resample_coeffs_ex" in _lib.EXPORTS and hasattr(lib, "zv_resample_coeffs_ex")
    assert b" 0.3 " in lib.zv_version()
    assert C.sizeof(_lib.ZvCfg) == 112                # the field was renamed, the struct is unchanged
    with pytest.raises(_lib.ZoomVitError, match="resample_kind -1"):
        from zoomearth_b200 import geometry as G
        G.normalize_lut(_lib.default_cfg(resample_kind=-1))


def _aligned(a):
    buf = np.zeros(a.nbytes + 16, np.uint8)
    off = (-buf.ctypes.data) % 16
    v = buf[off:off + a.nbytes].view(np.uint8).reshape(a.shape)
    v[...] = a
    return v


def _emulate(kind, imgs, index, boxes, out_hw):
    """zv_debug_k1_tc_host: the real host code + a lane-by-lane CPU emulation of K1's tensor-core route -> (fp32 patches, took)"""
    lib = _lib.lib()
    n = len(boxes)
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    srcs = (C.c_void_p * n)(*[imgs[k].ctypes.data for k in index])
    src_hw = np.array([[imgs[k].shape[0], imgs[k].shape[1]] for k in index], np.int32)
    pitch = np.array([imgs[k].strides[0] for k in index], np.int64)
    box, hw, took = np.array(boxes, np.int32), np.array(out_hw, np.int32), np.zeros(n, np.int32)
    need = _lib.check(lib.zv_preprocess_workspace_bytes(n, P(box), P(hw)))
    out = np.zeros((sum((h // 14) * (w // 14) for h, w in out_hw), 1176), np.float32)
    ws = np.zeros(need + 512, np.uint8)
    cfg = _lib.default_cfg(resample_kind=kind)
    _lib.check(lib.zv_debug_k1_tc_host(C.byref(cfg), n, srcs, P(src_hw), P(pitch), P(box), P(hw), P(out), _lib.ORDER_HF,
                                       None, None, C.c_void_p((ws.ctypes.data + 255) & ~255), need, P(took)))
    return out, took


def _pil_crop(img, box):
    from PIL import Image
    return np.asarray(Image.fromarray(np.ascontiguousarray(img)).crop(box))


def _hf_pil(images, min_pixels, max_pixels):
    from oracle import hf_live
    pv, grid = hf_live.hf_preprocess(images, min_pixels, max_pixels)
    return pv.numpy(), grid.numpy()


EMU_CASES = [
    # (h, w, box, max_pixels, note)
    (600, 800, (0, 0, 800, 600), 200704, "whole image, 2x downscale"),
    (602, 800, (-20, -30, 480, 470), 12845056, "box that leaves the image (zero fill)"),
    (603, 640, (16, 303, 600, 603), 50176, "height 3 mod 4, box ending on the last row"),
    (1203, 1600, (40, 700, 1500, 1203), 401408, "height 3 mod 4, 2.4x downscale"),
    (64, 64, (8, 8, 40, 40), 12845056, "upscale to min_pixels"),
    (504, 700, (0, 0, 700, 504), 12845056, "vertical identity"),
    (2000, 2000, (0, 0, 2000, 2000), 38416, "10x downscale"),
    (800, 1300, (0, 0, 1300, 800), 43008, "pitch 12 mod 16: four B variants"),
]


@pytest.mark.parametrize("h,w,box,maxp,note", EMU_CASES)
def test_k1_tc_emulation_vs_live_hf_torchvision(lib, h, w, box, maxp, note):
    img = _aligned(_img(h * 5 + w, h, w))
    crop = _pil_crop(img, box)
    ref, grid = _hf_tv([crop], 3136, maxp)
    rh, rw = OG.smart_resize(crop.shape[0], crop.shape[1], 28, 3136, maxp)
    got, took = _emulate(_lib.RESAMPLE_TORCHVISION, [img], [0], [box], [(rh, rw)])
    assert took.tolist() == [1], note
    assert grid.tolist() == [[1, rh // 14, rw // 14]]
    assert got.view(np.uint32).tolist() == ref.view(np.uint32).tolist(), note


def test_k1_tc_emulation_row_pitched_view(lib):
    """a cropped view of a larger image (base not 16-byte aligned, the parent's row pitch), ragged batch of two crops"""
    big = _aligned(_img(4, 1000, 1200))
    view = big[3:803, 5:905]
    boxes = [(0, 0, 900, 800), (7, 9, 507, 409)]
    crops = [_pil_crop(view, b) for b in boxes]
    out_hw = [OG.smart_resize(c.shape[0], c.shape[1], 28, 3136, 200704) for c in crops]
    got, took = _emulate(_lib.RESAMPLE_TORCHVISION, [view], [0, 0], boxes, out_hw)
    assert took.tolist() == [1, 1]
    ref, _ = _hf_tv(crops, 3136, 200704)
    assert np.array_equal(got, ref)


def test_axis_cache_keeps_the_conventions_apart(lib):
    """The per-process table cache is keyed on (kind, in, out): alternating the two conventions on ONE geometry in one
    process gives each its own answer every time."""
    img = _aligned(_smooth(8, 600, 800))
    box, ohw = (0, 0, 800, 600), (420, 560)
    ref_tv, _ = _hf_tv([img], 3136, 235200)
    ref_pil, _ = _hf_pil([img], 3136, 235200)
    assert not np.array_equal(ref_tv, ref_pil)
    for kind in (_lib.RESAMPLE_TORCHVISION, _lib.RESAMPLE_PIL, _lib.RESAMPLE_TORCHVISION, _lib.RESAMPLE_PIL):
        got, took = _emulate(kind, [img], [0], [box], [ohw])
        assert took.tolist() == [1]
        assert np.array_equal(got, ref_tv if kind == _lib.RESAMPLE_TORCHVISION else ref_pil), kind


def test_preprocess_rejects_unknown_kind(lib):
    img = _aligned(_img(1, 64, 64))
    with pytest.raises(_lib.ZoomVitError, match="resample_kind 7"):
        _emulate(7, [img], [0], [(0, 0, 64, 64)], [(56, 56)])


def test_tc_route_declines_a_four_variant_pitch_with_three_k_blocks(lib):
    """the geometry the GPU tests use to reach the dp4a kernels: an upload of a 2812-pixel-wide image (row pitch
    4 mod 16, not padded since 2812 is a multiple of 4) downscaled ~7x across: four B variants x three K blocks do not
    fit the tensor-core route's B buffer, 29 taps stay under the dp4a limit of 45"""
    img = _aligned(_img(2, 300, 2812))
    _, took = _emulate(_lib.RESAMPLE_TORCHVISION, [img], [0], [(0, 0, 2812, 300)], [(56, 392)])
    assert img.strides[0] % 16 == 4 and took.tolist() == [0]


# ---------------------------------------------------------------------------------------------- Python surface
class _StubProcessor:
    def __init__(self, image_processor):
        self.image_processor = image_processor


def test_fused_processor_backend_sets_every_cfg():
    from zoomearth_b200 import FusedImageProcessor
    assert FusedImageProcessor().backend == "pil" and FusedImageProcessor()._cfg().resample_kind == _lib.RESAMPLE_PIL
    fp = FusedImageProcessor(backend="torchvision", min_pixels=3136, max_pixels=50176)
    cfg = fp._cfg(3136, 1003520)
    assert cfg.resample_kind == _lib.RESAMPLE_TORCHVISION and cfg.max_pixels == 1003520
    with pytest.raises(ValueError, match="backend must be one of"):
        FusedImageProcessor(backend="cuda")


def test_install_image_backend_selection():
    from transformers.image_utils import PILImageResampling
    from transformers.models.qwen2_vl.image_processing_pil_qwen2_vl import Qwen2VLImageProcessorPil
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    from zoomearth_b200 import install
    for hf, default_backend in ((Qwen2VLImageProcessor, "torchvision"), (Qwen2VLImageProcessorPil, "pil")):
        for choice, want in (("pil", "pil"), ("torchvision", "torchvision"), ("match", default_backend)):
            proc = _StubProcessor(hf(min_pixels=3136, max_pixels=200704))
            _, fp = install(None, proc, image_backend=choice)
            assert proc.image_processor is fp and fp.backend == want, (hf.__name__, choice)
            assert fp._cfg().resample_kind == (1 if want == "torchvision" else 0)
            assert (fp.min_pixels, fp.max_pixels) == (3136, 200704)
    _, fp = install(None, _StubProcessor(Qwen2VLImageProcessor()))             # the default stays PIL
    assert fp.backend == "pil"

    class Other:                                      # e.g. a transformers 4.x *ImageProcessorFast
        resample = 3
    with pytest.raises(ValueError, match="Other"):
        install(None, _StubProcessor(Other()), image_backend="match")
    _, fp = install(None, _StubProcessor(Other()), image_backend="torchvision")
    assert fp.backend == "torchvision"
    with pytest.raises(ValueError, match="image_backend must be"):
        install(None, _StubProcessor(Qwen2VLImageProcessor()), image_backend="auto")

    for hf in (Qwen2VLImageProcessor, Qwen2VLImageProcessorPil):
        bilinear = hf(resample=PILImageResampling.BILINEAR)
        for choice in ("match", "torchvision"):
            proc = _StubProcessor(bilinear)
            with pytest.raises(NotImplementedError, match="bicubic"):
                install(None, proc, image_backend=choice)
            assert proc.image_processor is bilinear                          # nothing was replaced
        _, fp = install(None, _StubProcessor(bilinear), image_backend="pil")  # today's behaviour: not checked
        assert fp.backend == "pil"
