"""CPU: the CUDA-device torchvision convention (ZV_RESAMPLE_TORCHVISION_CUDA, FusedImageProcessor(backend=
"torchvision_cuda"), install(image_backend=...)): host validation, the LUT, the oracle's windows, weights and FFMA
emulation, and backend selection.  The pixels themselves are pinned on the GPU (test_gpu_torchvision_cuda_backend.py)."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from oracle import resample_torchvision_cuda as RC
from test_torchvision_backend import GEOMETRIES, _StubProcessor, _aligned, _emulate, _img
from zoomearth_b200 import _lib


def test_kind2_passes_validation_and_shares_kind1_lut(lib):
    from zoomearth_b200 import geometry as G
    for mean, std in (((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711)), ((0.5,) * 3, (0.5,) * 3)):
        l1 = G.normalize_lut(_lib.default_cfg(mean=mean, std=std, resample_kind=_lib.RESAMPLE_TORCHVISION))
        l2 = G.normalize_lut(_lib.default_cfg(mean=mean, std=std, resample_kind=_lib.RESAMPLE_TORCHVISION_CUDA))
        assert l2.view(np.uint32).tolist() == l1.view(np.uint32).tolist()
    assert _lib.RESAMPLE_TORCHVISION_CUDA == 2 and C.sizeof(_lib.ZvCfg) == 112
    assert b" 0.3 " in lib.zv_version()


def test_kind2_has_no_integer_taps_and_kind3_is_rejected_everywhere(lib):
    from zoomearth_b200 import geometry as G
    with pytest.raises(_lib.ZoomVitError, match="resample_kind 2"):
        G.resample_coeffs_ex(_lib.RESAMPLE_TORCHVISION_CUDA, 100, 50)
    for call in (lambda: G.resample_coeffs_ex(3, 100, 50), lambda: G.normalize_lut(_lib.default_cfg(resample_kind=3)),
                 lambda: _emulate(3, [_aligned(_img(1, 64, 64))], [0], [(0, 0, 64, 64)], [(56, 56)])):
        with pytest.raises(_lib.ZoomVitError, match="resample_kind 3") as e:
            call()
        assert "2 ZV_RESAMPLE_TORCHVISION_CUDA" in str(e.value)


def test_kind2_takes_no_tensor_core_route(lib):
    """the host emulation of the tensor-core route accepts no kind-2 crop: kind 2 runs its own fp32 kernel only"""
    img = _aligned(_img(1, 600, 800))
    _, took = _emulate(_lib.RESAMPLE_TORCHVISION_CUDA, [img], [0], [(0, 0, 800, 600)], [(420, 560)])
    assert took.tolist() == [0]


def _axes():
    pairs = {(i, o) for _, h, w, oh, ow, _ in GEOMETRIES for i, o in ((h, oh), (w, ow)) if i != o}
    return sorted(pairs | {(5000, 980), (6000, 56), (5000, 28), (1220, 224), (2812, 392), (1, 56)})


def test_oracle_windows_weights_and_interp_size(lib):
    """windows and weights follow torch's fp32 formulas; every weight row sums to 1 within fp32; torch's interp_size
    (and so every window) fits Pillow's ksize, the tap slots the library stores the fp32 weights in"""
    f = np.float32
    for i, o in _axes():
        rows, interp = RC.weights(i, o)
        scale = f(i) / f(o)
        support = scale * f(2) if scale >= 1 else f(2)
        assert interp == int(np.ceil(support)) * 2 + 1 <= lib.zv_resample_ksize(i, o), (i, o)
        for xx, (xmin, xsize, w) in enumerate(rows):
            center = float(scale) * (xx + 0.5)                      # exact value of the unrounded centre
            assert xmin == max(int(np.float32(RC.ffma(f(xx + 0.5), scale, -support)) + f(0.5)), 0)
            assert abs(xmin - max(center - float(support) + 0.5, 0)) <= 1 and 1 <= xsize <= interp, (i, o, xx)
            assert xmin + xsize <= i and w.dtype == np.float32 and w.shape == (xsize,)
            assert abs(float(w.astype(np.float64).sum()) - 1.0) <= 1e-5, (i, o, xx)


def _fma_exact(a, b, c):
    """round-to-nearest-even of the exact a b + c to float32, from rationals"""
    x = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    r = np.float32(float(x))
    cands = [r, np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(-np.inf))]
    return min(cands, key=lambda v: (abs(Fraction(float(v)) - x), int(np.float32(v).view(np.uint32)) & 1))


def test_ffma_emulation_is_exact_on_double_rounding_cases():
    """a b + c whose float64 sum rounds onto a float32 midpoint: rounding that sum again gives the wrong neighbour,
    the emulation the right one; and it agrees with exact rational rounding on random operands"""
    f = np.float32
    a, b = f(1 + 2 ** -23), f(0.5 * (1 - 2 ** -23))          # a b = 0.5 - 2^-47: below float64's resolution at 2^23
    for c in (f(2 ** 23 + 1), f(2 ** 23 + 3), f(2 ** 23 + 4097)):
        for sa in (1, -1):
            want = _fma_exact(f(sa) * a, b, c)
            naive = f(np.float64(f(sa) * a) * np.float64(b) + np.float64(c))
            assert want == c and naive != want, (sa, c)
            assert RC.ffma(f(sa) * a, b, c) == want
    rng = np.random.default_rng(0)
    x, y, z = (rng.standard_normal(3000).astype(np.float32) * f(s) for s in (1, 100, 1e4))
    got = RC.ffma(x, y, z)
    assert all(got[k] == _fma_exact(x[k], y[k], z[k]) for k in range(3000))


def test_fused_processor_backend_and_per_call_device():
    import torch
    from zoomearth_b200 import FusedImageProcessor
    from zoomearth_b200.processor import _backend_for_device
    fp = FusedImageProcessor(backend="torchvision_cuda")
    assert fp._cfg().resample_kind == _lib.RESAMPLE_TORCHVISION_CUDA
    for backend in ("torchvision", "torchvision_cuda"):
        assert _backend_for_device(backend, None) == backend
        assert _backend_for_device(backend, "cuda") == _backend_for_device(backend, torch.device("cuda", 1)) == "torchvision_cuda"
        assert _backend_for_device(backend, "cpu") == "torchvision"
    assert _backend_for_device("pil", "cuda") == "pil"
    assert FusedImageProcessor()._cfg(backend=_backend_for_device("pil", "cuda")).resample_kind == _lib.RESAMPLE_PIL
    with pytest.raises(ValueError, match="backend must be one of"):
        FusedImageProcessor(backend="cuda")


def test_preprocess_device_kwarg_picks_the_convention_not_the_processor_device(monkeypatch):
    """the HF ``device=`` of a call picks the torchvision convention; the device the processor itself runs K1 on (here
    a CUDA device) does not"""
    import torch
    from zoomearth_b200 import FusedImageProcessor, processor as P
    seen = []
    monkeypatch.setattr(P, "upload_u8", lambda t, device: t)
    monkeypatch.setattr(FusedImageProcessor, "preprocess_crops",
                        lambda self, *a, backend=None, **k: (seen.append(backend) or torch.zeros(4, 1176), torch.zeros(1, 3), None))
    img = _img(1, 56, 56)
    for backend, device, want in (("torchvision", None, "torchvision"), ("torchvision", "cuda", "torchvision_cuda"),
                                  ("torchvision", "cpu", "torchvision"), ("torchvision_cuda", None, "torchvision_cuda"),
                                  ("torchvision_cuda", "cpu", "torchvision"), ("pil", "cuda", "pil")):
        seen.clear()
        fp = FusedImageProcessor(backend=backend, device="cuda")
        fp(images=[img], **({} if device is None else {"device": device}))
        assert seen == [want], (backend, device, seen)


def test_install_match_reads_the_device_and_checks_bicubic():
    from transformers.image_utils import PILImageResampling
    from transformers.models.qwen2_vl.image_processing_pil_qwen2_vl import Qwen2VLImageProcessorPil
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    from zoomearth_b200 import install
    for hf, want in ((Qwen2VLImageProcessor(device="cuda"), "torchvision_cuda"), (Qwen2VLImageProcessor(), "torchvision"),
                     (Qwen2VLImageProcessor(device="cpu"), "torchvision"), (Qwen2VLImageProcessorPil(), "pil")):
        _, fp = install(None, _StubProcessor(hf), image_backend="match")
        assert fp.backend == want, (type(hf).__name__, getattr(hf, "device", None))
    _, fp = install(None, _StubProcessor(Qwen2VLImageProcessor()), image_backend="torchvision_cuda")
    assert fp.backend == "torchvision_cuda" and fp._cfg().resample_kind == _lib.RESAMPLE_TORCHVISION_CUDA
    bilinear = Qwen2VLImageProcessor(resample=PILImageResampling.BILINEAR, device="cuda")
    for choice in ("torchvision_cuda", "match"):
        proc = _StubProcessor(bilinear)
        with pytest.raises(NotImplementedError, match="bicubic"):
            install(None, proc, image_backend=choice)
        assert proc.image_processor is bilinear
