"""GPU (B200, through the C ABI): the torchvision convention of K1 - FusedImageProcessor(backend="torchvision") - is
bit-identical to the live HF torchvision-backend processor (Qwen2VLImageProcessor, the transformers 5.x default) on the
test_gpu_k1 geometry list and on every K1 route (tcgen05, IMMA / dp4a, per-tap), with the same launches as the PIL
convention; the pre_resize flow and the encoder follow the processor's convention."""
import numpy as np
import pytest
import torch

from oracle import geometry as OG, hf_live, processor_torchvision as PT, tower as OT

pytestmark = pytest.mark.gpu


def _img(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _hf_tv(images, min_pixels, max_pixels):
    from PIL import Image
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    p = Qwen2VLImageProcessor(min_pixels=min_pixels, max_pixels=max_pixels)
    out = p(images=[Image.fromarray(np.ascontiguousarray(i)) for i in images], return_tensors="pt")
    return out["pixel_values"], out["image_grid_thw"]


def _pil_crop(img, box):
    from PIL import Image
    return np.asarray(Image.fromarray(img).crop(box))


def _bits_equal(got, ref, note):
    got, ref = got.cpu().numpy(), ref.cpu().numpy()
    assert got.shape == ref.shape, note
    bad = np.flatnonzero(got.view(np.uint32).ravel() != ref.view(np.uint32).ravel())
    assert bad.size == 0, f"{note}: {bad.size} of {got.size} values differ, first at {bad[:5]}"


# the geometry list of test_gpu_k1.py
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
def test_hf_surface_bitexact_vs_live_torchvision_processor(cuda, h, w, box, minp, maxp, note):
    """processor(images=[PIL]) == HF's torchvision backend bitwise, with the launches of the PIL convention"""
    from PIL import Image
    from zoomearth_b200 import FusedImageProcessor
    img = _img(h * 7 + w, h, w)
    if box is not None:
        img = _pil_crop(img, box)
    fp = FusedImageProcessor(min_pixels=minp, max_pixels=maxp, device=cuda, backend="torchvision")
    out = fp(images=[Image.fromarray(img)], return_tensors="pt")
    ref_pv, ref_grid = _hf_tv([img], minp, maxp)
    assert out["image_grid_thw"].tolist() == ref_grid.tolist(), note
    _bits_equal(out["pixel_values"], ref_pv, note)
    pil = FusedImageProcessor(min_pixels=minp, max_pixels=maxp, device=cuda)
    pil(images=[Image.fromarray(img)])
    assert fp.last_launches == pil.last_launches, note


def test_every_k1_route(cuda):
    """tcgen05 (3 launches: two k1_resample_tc passes + patchify), IMMA / dp4a (an upload 2812 pixels wide: row pitch
    4 mod 16 and a 6.3x horizontal downscale need 4 B variants x 3 K blocks, more than the tensor-core route holds; at
    most 31 taps), per-tap (more than 45 taps; and a plain 701-pixel-wide view, row pitch 2103 not a multiple of 4):
    every one bit-identical to the live processor, with the launch count of the PIL convention"""
    from zoomearth_b200 import FusedImageProcessor
    from zoomearth_b200.processor import upload_u8
    routes = [("tcgen05", _img(1, 1000, 1400), None, 602112, 3), ("IMMA/dp4a", _img(2, 600, 2812), None, 43904, 2),
              ("per-tap, 109 taps", _img(3, 1500, 1500), None, 3136, 2),
              ("per-tap, pitch 2103", _img(4, 603, 701), (11, 7, 690, 603), 200704, 2)]
    for name, img, box, maxp, launches in routes:
        tv = FusedImageProcessor(min_pixels=3136, max_pixels=maxp, device=cuda, backend="torchvision")
        pil = FusedImageProcessor(min_pixels=3136, max_pixels=maxp, device=cuda)
        h, w, _ = img.shape
        dev = upload_u8(torch.from_numpy(img), cuda) if box is None else torch.from_numpy(img).to(cuda)
        bx = (0, 0, w, h) if box is None else box
        pv, grid, _ = tv.preprocess_crops([dev], [bx], torch.float32)
        assert tv.last_launches == launches, (name, tv.last_launches)
        pil.preprocess_crops([dev], [bx], torch.float32)
        assert pil.last_launches == launches, name
        ref_pv, ref_grid = _hf_tv([_pil_crop(img, bx)], 3136, maxp)
        assert grid.tolist() == ref_grid.tolist(), name
        _bits_equal(pv, ref_pv, name)


def test_fp16_window_order_equals_oracle_cast(cuda):
    """fp16 patches in the tower's window order == oracle_fp32.to(fp16), rows permuted; ragged batch on one image"""
    from zoomearth_b200 import FusedImageProcessor
    img = _img(5, 1000, 1400)
    boxes = [(0, 0, 1400, 1000), (100, 50, 900, 800), (300, 300, 812, 812), (-40, 700, 500, 1100)]
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=602112, device=cuda, backend="torchvision")
    pv, grid, _ = fp.preprocess_crops([torch.from_numpy(img).to(cuda)], boxes, torch.float16, window_order=True,
                                      image_index=[0] * len(boxes))
    refs, grids = zip(*[PT.preprocess_u8([_pil_crop(img, b)], 3136, 602112)[:2] for b in boxes])
    rgrid = np.concatenate(grids, 0)
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


def test_pre_resize_flow_is_pillow_resize_image_then_live_torchvision_processor(cuda):
    """ZoomEncoder(pre_resize="infer") with a torchvision-convention processor: Pillow resize_image(cut_image(...)) on the
    device, then the torchvision-convention resample - a transformers 5.x run of the reference loop"""
    from PIL import Image
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    cfg, sd, fv = _small_visual(cuda, 41)
    enc = ZoomEncoder(fv, FusedImageProcessor(min_pixels=3136, max_pixels=12845056, device=cuda, backend="torchvision"),
                      pre_resize="infer")
    img = _img(12, 1400, 1900)
    dev = enc.upload(img)
    boxes = [(100, 150, 1500, 1250), (300.5, 200.2, 700.9, 650.0), (-30, -20, 800, 900)]
    for bx in (None, boxes):
        emb, grid, _, pv = enc.encode([dev], bx, image_index=None if bx is None else [0] * len(bx), return_patches=True)
        ims = []
        for b in ([None] if bx is None else bx):
            im = Image.fromarray(img) if b is None else hf_live.pil_cut_image(img, b)[0]
            ims.append(np.asarray(hf_live.pil_resize_image(im, 512)[0]))
        ref_pv, ref_grid = _hf_tv(ims, 3136, 12845056)
        assert grid.tolist() == ref_grid.tolist()
        widx, _ = OT.window_index(ref_grid.numpy())
        ref_w = ref_pv.view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176).to(fv.operand_dtype)
        assert torch.equal(pv.cpu(), ref_w), "pre_resize patches differ from Pillow resize_image + the live processor"
        _close(emb, OT.forward(sd, ref_pv, ref_grid.numpy(), cfg), "pre_resize")


def test_zoom_encoder_embeddings_vs_fp32_oracle_tower(cuda):
    """ZoomEncoder.encode with the torchvision-convention processor: cut_image crops of a resident image, embeddings
    within the embedding bars of the fp32 oracle tower run on the live processor's pixels"""
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    cfg, sd, fv = _small_visual(cuda, 42)
    enc = ZoomEncoder(fv, FusedImageProcessor(min_pixels=3136, max_pixels=401408, device=cuda, backend="torchvision"))
    img = _img(13, 1300, 1700)
    boxes = [(200, 100, 1300, 900), (100.7, 50.2, 300.9, 260.1), (1500, 1100, 1690, 1290)]
    emb, grid, crop = enc.encode([enc.upload(img)], boxes, image_index=[0] * len(boxes))
    crops = [_pil_crop(img, OG.cut_box(1700, 1300, b)) for b in boxes]
    assert [tuple(int(v) for v in c) for c in crop] == [OG.cut_box(1700, 1300, b) for b in boxes]
    ref_pv, ref_grid = _hf_tv(crops, 3136, 401408)
    assert grid.tolist() == ref_grid.tolist()
    _close(emb, OT.forward(sd, ref_pv, ref_grid.numpy(), cfg), "encode")
