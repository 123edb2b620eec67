"""CPU: video inputs.  The NumPy video oracle against the live transformers ``Qwen2VLVideoProcessor``, the frame-sampling
restatements against its ``sample_frames``, the plan of mixed image + video grids against both HF towers' own
functions, ``install(video_backend=...)`` against real HF processor instances, and the host side of
``zv_preprocess_video``."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import processor_video as OV

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (frames, h, w, min_pixels, max_pixels): even / odd counts, 1 and 2 frames, upscale, downscale past 10x, one-axis and
# same-size geometries (a 56 x 84 frame at exactly its own pixel budget keeps both axes)
GEOMETRIES = [
    (4, 120, 160, None, None),                  # upscale to the 128 x 28^2 floor
    (5, 90, 200, None, None),                   # odd: the last frame is repeated
    (1, 300, 400, None, None),
    (2, 720, 1280, None, None),                 # a 720p clip at the default budget
    (3, 1600, 3000, 3136, 56 * 56 * 4),         # downscale past 10x on both axes
    (2, 56, 900, 3136, 56 * 900),               # one axis kept, the other resized
    (3, 56, 84, 3136, 56 * 84),                 # same size
]


def _video(seed, t, h, w):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (t, h, w, 3), dtype=np.uint8)
    return base


def _hf_video_processor(**kw):
    """The live processor with an explicit pixel budget: its __init__ writes min_pixels / max_pixels into the class-level
    ``size`` dict, so a bare constructor returns whatever budget the previous instance was built with."""
    from transformers.models.qwen2_vl.video_processing_qwen2_vl import Qwen2VLVideoProcessor
    kw.setdefault("min_pixels", OV.MIN_PIXELS)
    kw.setdefault("max_pixels", OV.MAX_PIXELS)
    return Qwen2VLVideoProcessor(**kw)


def _budget(mn, mx):
    return {} if mn is None else {"size": {"shortest_edge": mn, "longest_edge": mx}}


@pytest.mark.parametrize("t,h,w,mn,mx", GEOMETRIES)
def test_video_oracle_bitexact_vs_live_cpu(t, h, w, mn, mx):
    v = _video(t * 7 + h, t, h, w)
    out = _hf_video_processor()(videos=[v], return_tensors="pt", **_budget(mn, mx))
    pv, grid = OV.preprocess([v], **({} if mn is None else {"min_pixels": mn, "max_pixels": mx}))
    assert out["video_grid_thw"].tolist() == grid.tolist() == [[(t + 1) // 2, grid[0, 1], grid[0, 2]]]
    assert np.array_equal(out["pixel_values_videos"].numpy(), pv)


def test_video_oracle_batch_and_channels_first():
    """Two channels-first videos of different sizes in one call: rows back to back, HF's grids."""
    a, b = _video(1, 3, 100, 140), _video(2, 2, 200, 120)
    out = _hf_video_processor()(videos=[a.transpose(0, 3, 1, 2), b.transpose(0, 3, 1, 2)], return_tensors="pt")
    pv, grid = OV.preprocess([a, b])
    assert out["video_grid_thw"].tolist() == grid.tolist()
    assert np.array_equal(out["pixel_values_videos"].numpy(), pv)


@pytest.mark.parametrize("total,num_frames,fps,video_fps", [(30, 8, None, None), (31, 7, None, None), (7, 3, None, None),
                                                            (100, None, 2, 30.0), (9, None, 1, 1.0),
                                                            (1000, None, 0.5, 29.97), (12, None, 24, 24.0)])
def test_sample_indices_vs_live(total, num_frames, fps, video_fps):
    from transformers.video_utils import VideoMetadata
    from zoomearth_b200.video import FusedVideoProcessor, sample_indices
    want = _hf_video_processor().sample_frames(VideoMetadata(total_num_frames=total, fps=video_fps), num_frames=num_frames,
                                               fps=fps).numpy()
    assert np.array_equal(OV.sample_indices(total, num_frames, fps, video_fps), want)
    assert np.array_equal(sample_indices(total, num_frames, fps, video_fps), want)
    meta = {"total_num_frames": total, "fps": video_fps}
    assert np.array_equal(FusedVideoProcessor().sample_frames(meta, num_frames=num_frames, fps=fps), want)


@pytest.mark.parametrize("kw", [{"num_frames": 4}, {"fps": 2}])
def test_video_oracle_with_sampling_vs_live(kw):
    v = _video(5, 20, 64, 96)
    meta = {"total_num_frames": 20, "fps": 10.0, "duration": 2.0}
    out = _hf_video_processor()(videos=[v], do_sample_frames=True, video_metadata=[meta], return_tensors="pt", **kw)
    idx = OV.sample_indices(20, kw.get("num_frames"), kw.get("fps"), 10.0)
    pv, grid = OV.preprocess([v[idx]])
    assert out["video_grid_thw"].tolist() == grid.tolist()
    assert np.array_equal(out["pixel_values_videos"].numpy(), pv)


# ---------------------------------------------------------------------------------------------- plan
MIXED = [[1, 26, 36], [3, 8, 12], [2, 16, 16], [1, 4, 6], [4, 6, 10]]      # images (t = 1) and videos (odd and even t)


def _hf_qwen25_tower():
    from oracle import hf_live, tower as OT
    return hf_live.hf_tower(None, OT.small_cfg(depth=1, fullatt=()))


def _hf_qwen2_tower():
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLVisionConfig
    from transformers.models.qwen2_vl.modeling_qwen2_vl import Qwen2VisionTransformerPretrainedModel
    vc = Qwen2VLVisionConfig(depth=1, embed_dim=1280, num_heads=16, mlp_ratio=4, hidden_act="quick_gelu", hidden_size=1536)
    vc._attn_implementation = "sdpa"
    return Qwen2VisionTransformerPretrainedModel(vc).eval()


@pytest.mark.parametrize("tower", ["qwen25", "qwen2"])
def test_plan_mixed_image_video_vs_hf(lib, tower):
    """rot_pos_emb, get_window_index (Qwen2.5-VL) and cu_seqlens of HF's forward on a batch mixing images and videos."""
    from zoomearth_b200 import Plan, _lib
    grid = torch.tensor(MIXED)
    m = _hf_qwen25_tower() if tower == "qwen25" else _hf_qwen2_tower()
    cfg = _lib.default_cfg() if tower == "qwen25" else _lib.default_cfg(tower_kind=_lib.TOWER_QWEN2, fullatt=list(range(32)),
                                                                         inter=5120, out_hidden=1536)
    p = Plan(cfg, grid.numpy())
    S = int((grid[:, 0] * grid[:, 1] * grid[:, 2]).sum())
    assert p.num_patches == S and p.num_tokens == S // 4
    # rotary: HF's rot_pos_emb == its frequency table gathered at the plan's (h, w) ids
    with torch.no_grad():
        want = m.rot_pos_emb(grid)
        table = m.rotary_pos_emb(int(grid[:, 1:].max()))
    ids = torch.from_numpy(p.pos_ids.astype(np.int64))
    assert torch.equal(table[ids].flatten(1), want)
    # full attention never crosses a frame (HF forward: repeat_interleave(h w, t).cumsum)
    cu = torch.repeat_interleave(grid[:, 1] * grid[:, 2], grid[:, 0]).cumsum(0)
    assert p.cu_seqlens.tolist() == [0] + cu.tolist()
    if tower == "qwen25":
        w, cu_w = m.get_window_index(grid)
        assert np.array_equal(p.window_index, w.numpy())
        assert p.cu_window_seqlens_raw.tolist() == cu_w
        assert p.cu_window_seqlens.tolist() == torch.unique_consecutive(torch.tensor(cu_w)).tolist()
        assert np.array_equal(np.argsort(p.window_index), p.reverse_index)


def test_crop_cost_video_term():
    """Full attention costs t (h w)^2 for a video (one segment per frame group); images are unchanged."""
    from zoomearth_b200 import sharding
    img = np.array([[1, 26, 36], [1, 70, 70]])
    HW = (img[:, 1] * img[:, 2]).astype(np.float64)
    old = 5.125e9 * HW / 4 + 4 * 4 * HW * HW * 1280 + 28 * 4 * 64 * HW * 1280
    assert np.array_equal(sharding.crop_cost(img), old)
    one, three = sharding.crop_cost([[1, 20, 20]])[0], sharding.crop_cost([[3, 20, 20]])[0]
    assert three == pytest.approx(3 * one)


# ---------------------------------------------------------------------------------------------- host side of the ABI
def _args(frames, hw, rhw):
    f = np.asarray(frames, np.int32)
    fhw = np.asarray([h for h, n in zip(hw, frames) for _ in range(n)], np.int32).reshape(-1, 2)
    return f, fhw, np.asarray(rhw, np.int32).reshape(-1, 2)


def test_preprocess_video_host_checks(lib):
    from zoomearth_b200 import _lib
    f, fhw, rhw = _args([3, 2], [(100, 140), (720, 1280)], [(112, 168), (336, 588)])
    need = lib.zv_preprocess_video_workspace_bytes(2, f.ctypes.data, fhw.ctypes.data, rhw.ctypes.data)
    assert need > 3 * 112 * 168 * 3 + 2 * 336 * 588 * 3
    f0 = np.array([0, 2], np.int32)
    assert lib.zv_preprocess_video_workspace_bytes(2, f0.ctypes.data, fhw.ctypes.data, rhw.ctypes.data) == _lib.ZV_EINVAL
    assert "has 0 frames" in lib.zv_last_error().decode()
    bad = np.array([[112, 170], [336, 588]], np.int32)
    assert lib.zv_preprocess_video_workspace_bytes(2, f.ctypes.data, fhw.ctypes.data, bad.ctypes.data) == _lib.ZV_EINVAL
    ptrs = (C.c_void_p * 5)(*([16] * 5))
    pitch = np.array([420] * 3 + [3840] * 2, np.int64)

    def call(kind):
        cfg = _lib.default_cfg(resample_kind=kind)
        return lib.zv_preprocess_video(C.byref(cfg), 2, f.ctypes.data, ptrs, fhw.ctypes.data, pitch.ctypes.data,
                                       rhw.ctypes.data, 16, _lib.ZV_F32, _lib.ORDER_HF, 16, need, None)
    assert call(_lib.RESAMPLE_PIL) == _lib.ZV_EINVAL                             # HF has no PIL video backend
    assert "no PIL backend" in lib.zv_last_error().decode()
    assert call(3) == _lib.ZV_EINVAL and "resample_kind 3" in lib.zv_last_error().decode()
    if not torch.cuda.is_available():                                            # no fallback: fails loudly
        assert call(_lib.RESAMPLE_TORCHVISION) == _lib.ZV_ENODEV


@pytest.mark.skipif(shutil.which("gcc") is None, reason="gcc not available")
def test_video_workspace_from_c(tmp_path):
    """The two video exports are plain C: a C program sizes a workspace and sees the PIL refusal."""
    from zoomearth_b200 import _lib
    _lib.lib()
    src = tmp_path / "video_abi.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "zoomvit.h"
int main(void) {
  const int32_t frames[1] = {3}, fhw[6] = {100, 140, 100, 140, 100, 140}, rhw[2] = {112, 168};
  int64_t need = zv_preprocess_video_workspace_bytes(1, frames, fhw, rhw);
  zv_cfg cfg;
  zv_default_cfg(&cfg);
  const uint8_t* ptrs[3] = {0, 0, 0};
  const int64_t pitch[3] = {420, 420, 420};
  int rc = zv_preprocess_video(&cfg, 1, frames, ptrs, fhw, pitch, rhw, (void*)16, ZV_F32, ZV_ORDER_HF, (void*)16, need, NULL);
  int ok = need > 3 * 112 * 168 * 3 && rc == ZV_EINVAL && strstr(zv_last_error(), "no PIL backend") != NULL;
  printf("%s %lld\n", ok ? "ok" : "FAILED", (long long)need);
  return ok ? 0 : 1;
}
''')
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = str(tmp_path / "video_abi")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                        "-L", libdir, "-l:libzoomvit.so", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.startswith("ok"), r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------- Python surface
class _StubProcessor:
    def __init__(self, image_processor, video_processor):
        self.image_processor = image_processor
        self.video_processor = video_processor


def test_install_video_backend_selection():
    from transformers.image_utils import PILImageResampling
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    from zoomearth_b200 import FusedVideoProcessor, install
    old = _hf_video_processor(min_pixels=3136, max_pixels=200704)
    proc = _StubProcessor(Qwen2VLImageProcessor(), old)
    install(None, proc)                                                           # default: the video processor stays
    assert proc.video_processor is old
    for choice, device, want in (("torchvision", None, "torchvision"), ("torchvision_cuda", None, "torchvision_cuda"),
                                 ("match", None, "torchvision"), ("match", "cuda", "torchvision_cuda")):
        old = _hf_video_processor(min_pixels=3136, max_pixels=200704, device=device)
        proc = _StubProcessor(Qwen2VLImageProcessor(), old)
        _, fp = install(None, proc, video_backend=choice)
        vp = proc.video_processor
        assert isinstance(vp, FusedVideoProcessor) and vp.backend == want, (choice, device)
        assert (vp.min_pixels, vp.max_pixels, vp.temporal_patch_size, vp.merge_size) == (3136, 200704, 2, 2)
        assert fp.backend == "pil"                                                # image_backend keeps its own default
    vp = FusedVideoProcessor()
    assert (vp.min_pixels, vp.max_pixels) == (128 * 28 * 28, 768 * 28 * 28)
    assert vp.get_number_of_video_patches(9, 720, 1280) == _hf_video_processor().get_num_of_video_patches(9, 720, 1280, {})
    for bad in ("pil", "auto"):
        with pytest.raises(ValueError, match="video_backend must be"):
            install(None, _StubProcessor(Qwen2VLImageProcessor(), _hf_video_processor()), video_backend=bad)
    with pytest.raises(ValueError, match="backend must be"):
        FusedVideoProcessor(backend="pil")

    class Other:
        resample = 3
    with pytest.raises(ValueError, match="Other"):
        install(None, _StubProcessor(Qwen2VLImageProcessor(), Other()), video_backend="match")
    bilinear = _hf_video_processor(resample=PILImageResampling.BILINEAR)
    proc = _StubProcessor(Qwen2VLImageProcessor(), bilinear)
    with pytest.raises(NotImplementedError, match="bicubic"):
        install(None, proc, video_backend="match")
    assert proc.video_processor is bilinear


def test_fused_image_processor_still_refuses_videos():
    from zoomearth_b200 import FusedImageProcessor
    with pytest.raises(NotImplementedError):
        FusedImageProcessor().preprocess(None, videos=[np.zeros((2, 56, 56, 3), np.uint8)])
