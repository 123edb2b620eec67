"""GPU (B200): the CUDA-device torchvision convention of K1 (ZV_RESAMPLE_TORCHVISION_CUDA,
FusedImageProcessor(backend="torchvision_cuda")).  The NumPy oracle is pinned against live torch resizing CUDA uint8
tensors; the fused route is bit-identical to the live HF Qwen2VLImageProcessor(device="cuda") and to the oracle, and
the encoder, the pre_resize flow and the window-order output follow the processor's convention."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import geometry as OG, hf_live, processor as OP, processor_torchvision as PT, tower as OT
from oracle import resample_torchvision_cuda as RC
from test_gpu_torchvision_backend import _hf_tv
from test_torchvision_backend import GEOMETRIES, _img, _smooth

pytestmark = pytest.mark.gpu

# beyond GEOMETRIES: downscales of 100x and more (hundreds of taps per axis, windows taller than a shared-memory chunk)
LARGE = [(7, 60, 6000, 28, 56, "rand"), (8, 5000, 400, 28, 112, "smooth")]


def _tv_cuda(img, oh, ow):
    from torchvision.transforms.v2 import functional as tvF
    t = torch.from_numpy(np.ascontiguousarray(img)).permute(2, 0, 1).cuda()
    out = tvF.resize(t, [oh, ow], interpolation=tvF.InterpolationMode.BICUBIC, antialias=True)
    return out.permute(1, 2, 0).cpu().numpy()


def _hf_cuda(images, min_pixels, max_pixels):
    from PIL import Image
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    p = Qwen2VLImageProcessor(min_pixels=min_pixels, max_pixels=max_pixels, device="cuda")
    out = p(images=[Image.fromarray(np.ascontiguousarray(i)) for i in images], return_tensors="pt")
    return out["pixel_values"].cpu(), out["image_grid_thw"].cpu()


def _oracle_pv(u8):
    """normalised patches of an already resized uint8 image, HF order (the torchvision LUT + HF patchify)"""
    lut = PT.normalize_lut()
    pv, _ = OP.patchify(np.stack([lut[c][u8[:, :, c]] for c in range(3)], axis=0))
    return pv


def _pil_crop(img, box):
    from PIL import Image
    return np.asarray(Image.fromarray(np.ascontiguousarray(img)).crop(box))


def _bits_equal(got, ref, note):
    got, ref = np.asarray(got.cpu() if isinstance(got, torch.Tensor) else got), np.asarray(ref.cpu() if isinstance(ref, torch.Tensor) else ref)
    assert got.shape == ref.shape, note
    bad = np.flatnonzero(got.view(np.uint32).ravel() != ref.view(np.uint32).ravel())
    assert bad.size == 0, f"{note}: {bad.size} of {got.size} values differ, first at {bad[:5]}"


def _fused(dev_img, box, oh, ow, kind):
    """zv_preprocess of one crop at an exact output size (multiples of 28) -> fp32 patches (HF order), launches"""
    from zoomearth_b200 import _lib
    lib = _lib.lib()
    box = np.array([box], np.int32)
    hw = np.array([[oh, ow]], np.int32)
    src_hw = np.array([[dev_img.shape[0], dev_img.shape[1]]], np.int32)
    pitch = np.array([dev_img.stride(0)], np.int64)
    need = _lib.check(lib.zv_preprocess_workspace_bytes(1, box.ctypes.data, hw.ctypes.data))
    ws = torch.empty(need, dtype=torch.uint8, device=dev_img.device)
    out = torch.empty(((oh // 14) * (ow // 14), 1176), dtype=torch.float32, device=dev_img.device)
    cfg = _lib.default_cfg(resample_kind=kind)
    ptrs = (C.c_void_p * 1)(dev_img.data_ptr())
    _lib.check(lib.zv_preprocess(C.byref(cfg), 1, ptrs, src_hw.ctypes.data, pitch.ctypes.data, box.ctypes.data,
                                 hw.ctypes.data, None, out.data_ptr(), _lib.ZV_F32, _lib.ORDER_HF, ws.data_ptr(), need,
                                 torch.cuda.current_stream().cuda_stream))
    return out.cpu(), lib.zv_last_launch_count()


def test_oracle_vs_live_torch_cuda(cuda):
    """the oracle == tvF.resize on CUDA uint8 tensors, bit for bit, on the 44 geometries of the CPU convention's pin plus
    two downscales of 100x and more.  Where torch refuses a geometry (its kernel's per-thread weights do not fit shared
    memory) the refusal is recorded and the fused route must still give the oracle's bytes (checked when the output
    sizes are multiples of 28, the only sizes zv_preprocess takes)."""
    refused = []
    for seed, h, w, oh, ow, content in GEOMETRIES + LARGE:
        img = (_smooth if content == "smooth" else _img)(seed, h, w)
        got = RC.resize_u8(img, ow, oh)
        try:
            ref = _tv_cuda(img, oh, ow)
        except RuntimeError as e:
            assert "Too much shared memory" in str(e), str(e)
            refused.append((h, w, oh, ow))
            if oh % 28 == 0 and ow % 28 == 0:
                pv, _ = _fused(torch.from_numpy(img).to(cuda), (0, 0, w, h), oh, ow, 2)
                _bits_equal(pv, _oracle_pv(got), (h, w, oh, ow, "refused by torch"))
            continue
        assert np.array_equal(got, ref), (h, w, oh, ow, content, int((got != ref).sum()))
    print("geometries torch refuses:", refused)
    assert len(refused) < len(GEOMETRIES)


@pytest.mark.parametrize("seed,h,w,oh,ow,content", LARGE)
def test_large_downscale_fused_vs_oracle(cuda, seed, h, w, oh, ow, content):
    """windows of hundreds of taps: the fused route streams them through shared memory in chunks"""
    img = (_smooth if content == "smooth" else _img)(seed, h, w)
    pv, launches = _fused(torch.from_numpy(img).to(cuda), (0, 0, w, h), oh, ow, 2)
    assert launches == 2
    _bits_equal(pv, _oracle_pv(RC.resize_u8(img, ow, oh)), (h, w, oh, ow))


@pytest.mark.parametrize("mean,std", [(OP.OPENAI_CLIP_MEAN, OP.OPENAI_CLIP_STD), ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])
def test_lut_all_768_levels_vs_live_cuda_normalize(cuda, mean, std):
    """kind 2's table is kind 1's, and both equal HF's rescale_and_normalize run on the CUDA device"""
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    from zoomearth_b200 import _lib, geometry as G
    p = Qwen2VLImageProcessor(image_mean=list(mean), image_std=list(std), device="cuda")
    levels = torch.arange(256, dtype=torch.uint8, device=cuda).view(1, 1, 1, 256).expand(1, 3, 1, 256).contiguous()
    ref = p.rescale_and_normalize(levels, True, p.rescale_factor, True, p.image_mean, p.image_std)[0, :, 0, :].cpu().numpy()
    lut = G.normalize_lut(_lib.default_cfg(mean=mean, std=std, resample_kind=_lib.RESAMPLE_TORCHVISION_CUDA))
    assert lut.view(np.uint32).tolist() == ref.view(np.uint32).tolist()


# the CASES list of test_gpu_torchvision_backend.py
CASES = [
    (600, 800, None, 3136, 1003520, "mild downscale"),
    (512, 512, None, 3136, 12845056, "typical zoom crop 512->504"),
    (504, 504, None, 3136, 12845056, "same size: both axes skipped"),
    (30, 30, None, 3136, 12845056, "upscale to min_pixels"),
    (900, 1300, (100, 200, 700, 650), 3136, 200704, "crop + 2.7x downscale"),
    (700, 700, (-20, -30, 480, 470), 3136, 12845056, "box partly outside the image (zero fill)"),
    (1500, 1500, None, 3136, 3136, "27x downscale, 109 taps"),
    (504, 700, None, 3136, 12845056, "vertical identity, horizontal resize only"),
    (640, 28, None, 3136, 12845056, "thin image"),
    (1203, 1600, None, 3136, 1003520, "height not a multiple of 4"),
    (1203, 1600, (40, 700, 1500, 1203), 3136, 12845056, "crop that ends on the image's last row, height = 3 mod 4"),
]


@pytest.mark.parametrize("h,w,box,minp,maxp,note", CASES)
def test_hf_surface_bitexact_vs_live_cuda_processor(cuda, h, w, box, minp, maxp, note):
    """processor(images=[PIL]) == Qwen2VLImageProcessor(device="cuda") bitwise, in two launches; a per-call device on a
    "torchvision" processor gives the same pixels"""
    from PIL import Image
    from zoomearth_b200 import FusedImageProcessor
    img = _img(h * 7 + w, h, w)
    if box is not None:
        img = _pil_crop(img, box)
    ref_pv, ref_grid = _hf_cuda([img], minp, maxp)
    fp = FusedImageProcessor(min_pixels=minp, max_pixels=maxp, device=cuda, backend="torchvision_cuda")
    out = fp(images=[Image.fromarray(img)], return_tensors="pt")
    assert out["image_grid_thw"].tolist() == ref_grid.tolist(), note
    _bits_equal(out["pixel_values"], ref_pv, note)
    assert fp.last_launches == 2, note
    tv = FusedImageProcessor(min_pixels=minp, max_pixels=maxp, device=cuda, backend="torchvision")
    _bits_equal(tv(images=[Image.fromarray(img)], device="cuda")["pixel_values"], ref_pv, note + ", device='cuda' per call")
    # and the other way: a per-call CPU device (or none) on a "torchvision_cuda" processor gives the CPU convention
    ref_cpu, _ = _hf_tv([img], minp, maxp)
    _bits_equal(fp(images=[Image.fromarray(img)], device="cpu")["pixel_values"], ref_cpu, note + ", device='cpu' per call")
    _bits_equal(tv(images=[Image.fromarray(img)])["pixel_values"], ref_cpu, note + ", no device")


def test_every_k1_route_input(cuda):
    """the inputs that reach each integer route (a 2812-wide and a 1220-wide upload, a 701-wide view whose row pitch,
    2103, is not a multiple of 4) all take the fp32 kernel and match the live CUDA processor, in two launches"""
    from zoomearth_b200 import FusedImageProcessor
    from zoomearth_b200.processor import upload_u8
    routes = [("1000 x 1400", _img(1, 1000, 1400), None, 602112), ("2812 wide", _img(2, 600, 2812), None, 43904),
              ("pitch 3660", _img(6, 1220, 1220), None, 50176), ("109 taps", _img(3, 1500, 1500), None, 3136),
              ("pitch 2103", _img(4, 603, 701), (11, 7, 690, 603), 200704)]
    for name, img, box, maxp in routes:
        fp = FusedImageProcessor(min_pixels=3136, max_pixels=maxp, device=cuda, backend="torchvision_cuda")
        h, w, _ = img.shape
        dev = upload_u8(torch.from_numpy(img), cuda) if box is None else torch.from_numpy(img).to(cuda)
        bx = (0, 0, w, h) if box is None else box
        pv, grid, _ = fp.preprocess_crops([dev], [bx], torch.float32)
        assert fp.last_launches == 2, (name, fp.last_launches)
        ref_pv, ref_grid = _hf_cuda([_pil_crop(img, bx)], 3136, maxp)
        assert grid.tolist() == ref_grid.tolist(), name
        _bits_equal(pv, ref_pv, name)


def test_fp16_window_order_ragged_crops_equal_oracle_cast(cuda):
    """a ragged batch of crops on one resident image: fp16 window-order patches == oracle_fp32.to(fp16), permuted"""
    from zoomearth_b200 import FusedImageProcessor
    img = _img(5, 1000, 1400)
    boxes = [(0, 0, 1400, 1000), (100, 50, 900, 800), (300, 300, 812, 812), (-40, 700, 500, 1100)]
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=602112, device=cuda, backend="torchvision_cuda")
    pv, grid, _ = fp.preprocess_crops([torch.from_numpy(img).to(cuda)], boxes, torch.float16, window_order=True,
                                      image_index=[0] * len(boxes))
    refs, grids = [], []
    for b in boxes:
        crop = _pil_crop(img, b)
        rh, rw = OG.smart_resize(crop.shape[0], crop.shape[1], 28, 3136, 602112)
        refs.append(_oracle_pv(RC.resize_u8(crop, rw, rh)))
        grids.append([1, rh // 14, rw // 14])
    rgrid = np.array(grids, np.int64)
    assert grid.tolist() == rgrid.tolist()
    widx, _ = OT.window_index(rgrid)
    ref = torch.from_numpy(np.concatenate(refs, 0)).view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176)
    assert torch.equal(pv.cpu(), ref.to(torch.float16))


def _small_visual(cuda, seed):
    from zoomearth_b200 import FusedVisual
    cfg = OT.small_cfg(depth=2, fullatt=(1,))
    sd = OT.make_weights(seed, cfg)
    return cfg, sd, FusedVisual(sd, device=cuda, dtype=torch.float32, depth=cfg["depth"], fullatt=list(cfg["fullatt"]))


def _close(emb, ref, note):
    got = emb.double().cpu()
    cos = (torch.dot(got.flatten(), ref.double().flatten()) / (got.norm() * ref.double().norm())).item()
    maxrel = ((got - ref.double()).abs().max() / ref.abs().max()).item()
    assert cos >= 0.999 and maxrel <= 1e-2, f"{note}: cos {cos} maxrel {maxrel}"


def test_pre_resize_flow_is_pillow_resize_image_then_live_cuda_processor(cuda):
    from PIL import Image
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    cfg, sd, fv = _small_visual(cuda, 41)
    enc = ZoomEncoder(fv, FusedImageProcessor(min_pixels=3136, max_pixels=12845056, device=cuda,
                                              backend="torchvision_cuda"), pre_resize="infer")
    img = _img(12, 1400, 1900)
    dev = enc.upload(img)
    boxes = [(100, 150, 1500, 1250), (300.5, 200.2, 700.9, 650.0), (-30, -20, 800, 900)]
    for bx in (None, boxes):
        emb, grid, _, pv = enc.encode([dev], bx, image_index=None if bx is None else [0] * len(bx), return_patches=True)
        ims = []
        for b in ([None] if bx is None else bx):
            im = Image.fromarray(img) if b is None else hf_live.pil_cut_image(img, b)[0]
            ims.append(np.asarray(hf_live.pil_resize_image(im, 512)[0]))
        ref_pv, ref_grid = _hf_cuda(ims, 3136, 12845056)
        assert grid.tolist() == ref_grid.tolist()
        widx, _ = OT.window_index(ref_grid.numpy())
        ref_w = ref_pv.view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176).to(fv.operand_dtype)
        assert torch.equal(pv.cpu(), ref_w), "pre_resize patches differ from Pillow resize_image + the live CUDA processor"
        _close(emb, OT.forward(sd, ref_pv, ref_grid.numpy(), cfg), "pre_resize")


def test_zoom_encoder_embeddings_vs_fp32_oracle_tower(cuda):
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    cfg, sd, fv = _small_visual(cuda, 42)
    enc = ZoomEncoder(fv, FusedImageProcessor(min_pixels=3136, max_pixels=401408, device=cuda, backend="torchvision_cuda"))
    img = _img(13, 1300, 1700)
    boxes = [(200, 100, 1300, 900), (100.7, 50.2, 300.9, 260.1), (1500, 1100, 1690, 1290)]
    emb, grid, crop = enc.encode([enc.upload(img)], boxes, image_index=[0] * len(boxes))
    crops = [_pil_crop(img, OG.cut_box(1700, 1300, b)) for b in boxes]
    ref_pv, ref_grid = _hf_cuda(crops, 3136, 401408)
    assert grid.tolist() == ref_grid.tolist()
    _close(emb, OT.forward(sd, ref_pv, ref_grid.numpy(), cfg), "encode")


def test_alternating_kinds_on_one_geometry(cuda):
    """one process alternating kinds 0, 1 and 2 on one geometry gets each kind's own answer every time"""
    from zoomearth_b200 import _lib
    img = _smooth(8, 600, 800)
    dev = torch.from_numpy(img).to(cuda)
    refs = {_lib.RESAMPLE_PIL: hf_live.hf_preprocess([img], 3136, 235200)[0],
            _lib.RESAMPLE_TORCHVISION: torch.from_numpy(PT.preprocess_u8([img], 3136, 235200)[0]),
            _lib.RESAMPLE_TORCHVISION_CUDA: _hf_cuda([img], 3136, 235200)[0]}
    assert not torch.equal(refs[1], refs[2]) and not torch.equal(refs[0], refs[2])
    for kind in (0, 1, 2, 0, 2, 1, 2):
        pv, _ = _fused(dev, (0, 0, 800, 600), 420, 560, kind)
        _bits_equal(pv, refs[kind], f"kind {kind}")
