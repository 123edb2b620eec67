"""Video clips through the fused path against HF's video processor + HF's vision tower, on one GPU.

    python tools/bench_video.py [--clips 16] [--frames 32] [--hf-clips 2] [--out profiles/r06_bench_video_n1.json]

Seeded workload: ``--clips`` clips of ``--frames`` 720 x 1280 uint8 frames, resident on the GPU, at the video
processor's default pixel budget (128 - 768 x 28^2), through a randomly initialised Qwen2.5-VL-3B tower (32 blocks).
Fused: ``ZoomEncoder.encode_video`` (zv_preprocess_video -> fp16 window-order patches -> zv_visual_forward), fp16 out.
HF: ``Qwen2VLVideoProcessor(device="cuda")`` then ``Qwen2_5_VisionTransformerPretrainedModel`` in bf16 with sdpa, on the
first ``--hf-clips`` clips (it is timed per clip).  Both sides are timed with a device synchronise around warm calls.
The record carries the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                      # pragma: no cover
        return f"unknown ({e})"


def _timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return out, float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=16)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--hf-clips", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video needs a CUDA device; there is no CPU measurement")
    from oracle import hf_live, tower as OT
    from zoomearth_b200 import FusedVisual, ZoomEncoder
    from transformers.models.qwen2_vl.video_processing_qwen2_vl import Qwen2VLVideoProcessor
    dev = torch.device("cuda", 0)
    card = _card()
    g = torch.Generator(device=dev).manual_seed(0)
    clips = [torch.randint(0, 256, (a.frames, 720, 1280, 3), generator=g, device=dev, dtype=torch.uint8) for _ in range(a.clips)]
    hf_tower = hf_live.hf_tower(None, OT.CFG, seed=0).to(dev)
    fv = FusedVisual.from_hf(hf_tower, device=dev, dtype=torch.float16, operand_dtype=torch.float16)
    enc = ZoomEncoder(fv)
    (emb, grid), fused_s, fused_ts = _timed(lambda: enc.encode_video(clips), a.reps)
    tokens = int(emb.shape[0])
    launches = enc.last_launches
    vp = enc.video_processor
    _, k1_s, _ = _timed(lambda: vp.preprocess_videos(clips, torch.float16, True, backend="torchvision_cuda"), a.reps)

    hf_proc = Qwen2VLVideoProcessor(min_pixels=128 * 28 * 28, max_pixels=768 * 28 * 28)
    hf_bf16 = hf_tower.to(torch.bfloat16)
    sub = [c.permute(0, 3, 1, 2) for c in clips[:a.hf_clips]]

    def hf_step():
        o = hf_proc(videos=sub, device="cuda", return_tensors="pt")
        with torch.no_grad():
            return hf_bf16(o["pixel_values_videos"].to(dev, torch.bfloat16), grid_thw=o["video_grid_thw"].to(dev))
    _, hf_s, hf_ts = _timed(hf_step, a.reps)
    _, hf_proc_s, _ = _timed(lambda: hf_proc(videos=sub, device="cuda", return_tensors="pt"), a.reps)
    rec = {
        "card": card, "workload": f"{a.clips} clips x {a.frames} frames of 720x1280 uint8 on the GPU, video defaults "
                                  "128-768 x 28^2, Qwen2.5-VL-3B tower (random init)",
        "grid_thw_first": grid[0].tolist(), "tokens": tokens,
        "fused_s": fused_s, "fused_runs_s": fused_ts, "fused_tokens_per_s": tokens / fused_s, "fused_launches": launches,
        "fused_preprocess_s": k1_s,
        "hf_clips": a.hf_clips, "hf_s": hf_s, "hf_runs_s": hf_ts, "hf_processor_s": hf_proc_s,
        "hf_tokens_per_s": tokens / a.clips * a.hf_clips / hf_s,
        "speedup_per_clip": (hf_s / a.hf_clips) / (fused_s / a.clips),
    }
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
