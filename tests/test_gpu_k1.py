"""K1 parity (GPU, through the C ABI): fused crop->resize->normalize->patchify vs the oracle, bit-exact."""
import numpy as np
import pytest
import torch

from oracle import geometry as OG, processor as OP, resample as OR, tower as OT

pytestmark = pytest.mark.gpu


def _img(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _oracle_crop(img, box, min_pixels, max_pixels):
    crop = OR.crop_u8(img, box)
    pv, grid, _ = OP.preprocess_u8([crop], min_pixels, max_pixels)
    return pv, grid


CASES = [
    # (h, w, box or None, min_pixels, max_pixels, note)
    (600, 800, None, 3136, 1003520, "mild downscale"),
    (512, 512, None, 3136, 12845056, "typical zoom crop 512->504"),
    (504, 504, None, 3136, 12845056, "same size: Pillow copies"),
    (30, 30, None, 3136, 12845056, "upscale to min_pixels"),
    (900, 1300, (100, 200, 700, 650), 3136, 200704, "crop + 2.7x downscale"),
    (700, 700, (-20, -30, 480, 470), 3136, 12845056, "box partly outside the image (zero fill)"),
    (1500, 1500, None, 3136, 3136, "22x downscale, 89 taps"),
    (504, 700, None, 3136, 12845056, "vertical identity, horizontal resize only"),
    (640, 28, None, 3136, 12845056, "thin image"),
    (1203, 1600, None, 3136, 1003520, "height not a multiple of 4: the last rows come through the end-aligned tensor map"),
    (1203, 1600, (40, 700, 1500, 1203), 3136, 12845056, "crop that ends on the image's last row, height = 3 mod 4"),
    (1220, 1220, None, 3136, 50176, "row pitch 12 mod 16 at 5.45x: the tensor-core route declines, the dp4a pass takes what IMMA took"),
]


@pytest.mark.parametrize("h,w,box,minp,maxp,note", CASES)
def test_k1_hf_order_fp32_bitexact(cuda, h, w, box, minp, maxp, note):
    from zoomearth_b200 import FusedImageProcessor
    img = _img(h * 7 + w, h, w)
    fp = FusedImageProcessor(min_pixels=minp, max_pixels=maxp, device=cuda)
    dev = torch.from_numpy(img).to(cuda)
    bx = (0, 0, w, h) if box is None else box
    pv, grid, crop = fp.preprocess_crops([dev], [bx], torch.float32, window_order=False)
    ref, rgrid = _oracle_crop(img, bx, minp, maxp)
    assert grid.tolist() == rgrid.tolist(), note
    got = pv.cpu().numpy()
    assert got.shape == ref.shape
    bad = np.flatnonzero(got.view(np.uint32).ravel() != ref.view(np.uint32).ravel())
    assert bad.size == 0, f"{note}: {bad.size} of {got.size} values differ, first at {bad[:5]}, max |d| {np.abs(got - ref).max()}"


def test_k1_bf16_window_order_matches_oracle_cast(cuda):
    """bf16 fast path == oracle_fp32.to(bf16), rows permuted into the tower's window order."""
    from zoomearth_b200 import FusedImageProcessor
    img = _img(5, 1000, 1400)
    boxes = [(0, 0, 1400, 1000), (100, 50, 900, 800), (300, 300, 812, 812)]
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=602112, device=cuda)
    dev = torch.from_numpy(img).to(cuda)
    pv, grid, _ = fp.preprocess_crops([dev], boxes, torch.bfloat16, window_order=True, image_index=[0, 0, 0])
    refs, grids = zip(*[_oracle_crop(img, b, 3136, 602112) for b in boxes])
    ref = torch.from_numpy(np.concatenate(refs, 0))
    rgrid = np.concatenate(grids, 0)
    assert grid.tolist() == rgrid.tolist()
    widx, _ = OT.window_index(rgrid)
    ref_w = ref.view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176).to(torch.bfloat16)
    assert torch.equal(pv.cpu(), ref_w)


def test_k1_fp16_output(cuda):
    from zoomearth_b200 import FusedImageProcessor
    img = _img(6, 600, 600)
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=200704, device=cuda)
    pv, grid, _ = fp.preprocess_crops([torch.from_numpy(img).to(cuda)], None, torch.float16)
    ref, _ = _oracle_crop(img, (0, 0, 600, 600), 3136, 200704)
    assert torch.equal(pv.cpu(), torch.from_numpy(ref).to(torch.float16))


def test_k1_ragged_batch_and_cut_image(cuda):
    """A ragged batch through the reference's cut_image rule (min 512) equals the per-crop oracle."""
    from zoomearth_b200 import FusedImageProcessor
    imgs = [_img(11, 1200, 1600), _img(12, 900, 700)]
    boxes = [(100.7, 50.2, 300.9, 260.1), (200, 100, 1300, 900), (650, 850, 699, 899), (0, 0, 700, 900)]
    index = [0, 0, 1, 1]
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=12845056, device=cuda)
    dev = [torch.from_numpy(i).to(cuda) for i in imgs]
    pv, grid, crop = fp.preprocess_crops(dev, boxes, torch.float32, image_index=index, apply_cut_image=True)
    rows = []
    for b, i, c in zip(boxes, index, crop):
        h, w, _ = imgs[i].shape
        ebox = OG.cut_box(w, h, b, 512)
        assert tuple(int(v) for v in c) == ebox
        rows.append(_oracle_crop(imgs[i], ebox, 3136, 12845056)[0])
    assert np.array_equal(pv.cpu().numpy(), np.concatenate(rows, 0))


def test_k1_hf_surface_matches_live_hf(cuda):
    """The drop-in surface: processor(images=[PIL...]) == the HF PIL-backend processor, bitwise."""
    from PIL import Image
    from oracle import hf_live
    from zoomearth_b200 import FusedImageProcessor
    imgs = [Image.fromarray(_img(21, 700, 1100)), Image.fromarray(_img(22, 512, 354))]
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=401408, device=cuda)
    out = fp(images=[[imgs[0], imgs[1]]], return_tensors="pt")
    ref_pv, ref_grid = hf_live.hf_preprocess(imgs, 3136, 401408)
    assert out["image_grid_thw"].tolist() == ref_grid.tolist()
    assert out["pixel_values"].dtype == torch.float32 and out["pixel_values"].device.type == "cpu"
    assert torch.equal(out["pixel_values"], ref_pv)


def test_k1_full_size_global_view_vs_pillow(cuda):
    """BASELINE config-2 shape (5000x5000 -> 980x980, 23 taps/axis) against live Pillow + the oracle LUT."""
    from PIL import Image
    from zoomearth_b200 import FusedImageProcessor
    img = _img(0, 5000, 5000)
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=1280 * 28 * 28, device=cuda)
    pv, grid, _ = fp.preprocess_crops([torch.from_numpy(img).to(cuda)], None, torch.float32)
    assert grid.tolist() == [[1, 70, 70]]
    assert fp.last_launches == 3, "the bench shape must take the tensor-core route: two k1_resample_tc passes + k1_patchify_u8"
    r = np.asarray(Image.fromarray(img).resize((980, 980), Image.BICUBIC))
    lut = OP.normalize_lut()
    ref, _ = OP.patchify(np.stack([lut[c][r[:, :, c]] for c in range(3)], 0))
    assert np.array_equal(pv.cpu().numpy(), ref)


def test_k1_errors(cuda):
    from zoomearth_b200 import FusedImageProcessor
    fp = FusedImageProcessor(device=cuda)
    dev = torch.zeros((10, 4000, 3), dtype=torch.uint8, device=cuda)
    with pytest.raises(ValueError, match="absolute aspect ratio must be smaller than 200"):
        fp.preprocess_crops([dev], None)
    with pytest.raises(ValueError, match="Coordinate 'right' is less than 'left'"):
        fp.preprocess_crops([dev], [(50, 0, 40, 10)])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_k1_random_sweep_bitexact(cuda, seed):
    """Randomised parity sweep: image sizes with aligned and unaligned row pitches, boxes inside / partly outside the
    image, scales from 4x upscale to 12x downscale (every tap-window class of the dp4a path and the per-tap path),
    ragged batches, fp32 HF order and bf16 window order - all bit-exact against the oracle."""
    from zoomearth_b200 import FusedImageProcessor
    rng = np.random.default_rng(1234 + seed)
    imgs = []
    for _ in range(3):
        h, w = int(rng.integers(120, 1500)), int(rng.integers(120, 1500))
        if rng.random() < 0.5:
            w = (w // 4) * 4 + int(rng.integers(1, 4))          # pitch not a multiple of 4 -> generic kernels
        else:
            w = (w // 4) * 4
        imgs.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    dev = [torch.from_numpy(i).to(cuda) for i in imgs]
    for max_pixels in (3136 * 4, 50176, 401408, 12845056):
        boxes, index = [], []
        for _ in range(6):
            k = int(rng.integers(0, 3))
            h, w, _ = imgs[k].shape
            bw, bh = int(rng.integers(20, w + 40)), int(rng.integers(20, h + 40))
            bw, bh = max(bw, bh // 150 + 1), max(bh, bw // 150 + 1)          # keep the aspect ratio below 200
            x0, y0 = int(rng.integers(-30, max(1, w - bw + 30))), int(rng.integers(-30, max(1, h - bh + 30)))
            boxes.append((x0, y0, x0 + bw, y0 + bh))
            index.append(k)
        fp = FusedImageProcessor(min_pixels=3136, max_pixels=max_pixels, device=cuda)
        pv, grid, crop = fp.preprocess_crops(dev, boxes, torch.float32, image_index=index)
        refs, grids = zip(*[_oracle_crop(imgs[k], b, 3136, max_pixels) for b, k in zip(boxes, index)])
        ref = np.concatenate(refs, 0)
        assert grid.tolist() == np.concatenate(grids, 0).tolist()
        got = pv.cpu().numpy()
        bad = np.flatnonzero(got.view(np.uint32).ravel() != ref.view(np.uint32).ravel())
        assert bad.size == 0, f"max_pixels {max_pixels}: {bad.size} of {got.size} values differ (boxes {boxes})"
        pvw, _, _ = fp.preprocess_crops(dev, boxes, torch.bfloat16, window_order=True, image_index=index)
        widx, _ = OT.window_index(np.concatenate(grids, 0))
        ref_w = torch.from_numpy(ref).view(-1, 4, 1176)[torch.from_numpy(widx)].reshape(-1, 1176).to(torch.bfloat16)
        assert torch.equal(pvw.cpu(), ref_w)


def test_upload_pads_odd_widths_to_a_tensor_core_pitch(cuda):
    """processor.upload_u8: a 701-pixel-wide image (row pitch 2103 bytes, which K1's tensor-core route cannot read) is
    stored with padded rows and handed out as a view; pixels, patches and the device resize stay bit-exact"""
    from zoomearth_b200 import FusedImageProcessor
    from zoomearth_b200.processor import upload_u8
    img = _img(77, 603, 701)
    dev = upload_u8(torch.from_numpy(img), cuda)
    assert dev.shape == (603, 701, 3) and dev.stride(0) % 16 == 0 and dev.stride(1) == 3
    assert torch.equal(dev.cpu(), torch.from_numpy(img))
    fp = FusedImageProcessor(min_pixels=3136, max_pixels=200704, device=cuda)
    boxes = [(0, 0, 701, 603), (11, 7, 690, 603), (-9, -4, 400, 300)]
    pv, grid, _ = fp.preprocess_crops([dev], boxes, torch.float32, image_index=[0, 0, 0])
    assert fp.last_launches == 3, "odd height, a box that leaves the image, a padded pitch: all on the tensor-core route"
    refs, grids = zip(*[_oracle_crop(img, b, 3136, 200704) for b in boxes])
    assert grid.tolist() == np.concatenate(grids, 0).tolist()
    assert np.array_equal(pv.cpu().numpy(), np.concatenate(refs, 0))
    out = fp.resize_u8([dev], [(3, 5, 699, 601)], [(233, 199)])[0]
    assert np.array_equal(out.cpu().numpy(), OR.resize_u8(OR.crop_u8(img, (3, 5, 699, 601)), 233, 199))
