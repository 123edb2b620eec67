"""K1 under ZV_RESAMPLE_TORCHVISION_CUDA on bench.py's global-view shape, next to the integer route (kind 0) and next
to HF's own path: 64 synthetic 5000 x 5000 uint8 images (4.8 GB, well past the 126 MB L2) -> 980 x 980
(max_pixels 1280 * 28 * 28), fp16 patches in the tower's window order, as ZoomEncoder feeds the tower.

- kind 2 and kind 0: `--iters` zv_preprocess calls per round, alternating which goes first, timed with CUDA events
  around the calls and with the library's per-class event timing (class 13: k1_resample_f32; class 1: patchify).
- HF: the live Qwen2VLImageProcessor(device="cuda") on the same images as CUDA tensors (its resize, normalise and
  patchify; one call per round, it is slow).  Image 0 of the fused kind-2 output is checked bit for bit against it.
- Work from the shapes: the multiply-adds (FFMA / FMUL) k1_resample_f32 issues - each horizontal result once per
  tile, each vertical chain once - and the bytes it must move (source read, U written); its share of the larger of
  the FP32-pipe bound (148 SMs x 128 lanes x the maximum SM clock) and the HBM bound (7.7 TB/s).

    python tools/bench_k1_f32.py [--images 64] [--rounds 4] [--iters 3] [--out profiles/r05_k1_f32_n1.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import resample_torchvision_cuda as RC  # noqa: E402
from zoomearth_b200 import FusedImageProcessor, _lib  # noqa: E402

IMG, OUT, MAX_PIXELS = 5000, 980, 1280 * 28 * 28
TILE = 32                                               # k1_resample_f32: output rows / columns per CTA tile
HBM_BYTES_PER_S = 7.7e12


def f32_work(n_images):
    """(multiply-adds, bytes) of k1_resample_f32 for n_images x IMG^2 -> OUT^2, from the kernel's tiling"""
    rows, _ = RC.weights(IMG, OUT)                      # both axes are IMG -> OUT
    taps = [r[1] for r in rows]
    h = 0
    for t0 in range(0, OUT, TILE):                      # a tile's input rows: first row's window start .. last row's end
        t1 = min(OUT, t0 + TILE) - 1
        span = rows[t1][0] + rows[t1][1] - rows[t0][0]
        h += span * sum(taps) * 3                       # every column of the image, 3 channels, once per row tile
    v = sum(taps) * OUT * 3
    return n_images * (h + v), n_images * (IMG * IMG * 3 + OUT * OUT * 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_k1_f32.py: needs a CUDA device")
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    dev = torch.device("cuda", 0)
    lib = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(1234)
    images = [torch.randint(0, 256, (IMG, IMG, 3), generator=g, dtype=torch.uint8, device=dev) for _ in range(args.images)]
    procs = {b: FusedImageProcessor(min_pixels=3136, max_pixels=MAX_PIXELS, device=dev, backend=b)
             for b in ("torchvision_cuda", "pil")}
    hf = Qwen2VLImageProcessor(min_pixels=3136, max_pixels=MAX_PIXELS, device="cuda")
    chw = [im.permute(2, 0, 1) for im in images]

    def run_hf(imgs):
        return hf(images=imgs, return_tensors="pt")["pixel_values"]

    pv, _, _ = procs["torchvision_cuda"].preprocess_crops(images[:1], None, torch.float32)
    check = bool(torch.equal(pv.view(torch.int32), run_hf(chw[:1]).view(torch.int32)))
    if not check:
        raise SystemExit("bench_k1_f32.py: kind-2 patches differ from the live HF CUDA processor")

    def run(b):
        return procs[b].preprocess_crops(images, None, torch.float16, window_order=True)

    for b in procs:                                     # warm up: module load, table cache, workspace
        for _ in range(2):
            run(b)
    run_hf(chw)
    torch.cuda.synchronize()
    per = {b: {"k1_ms": [], "resample_ms": [], "patchify_or_pass2_ms": [], "launches": None} for b in procs}
    per["hf"] = {"call_ms": []}
    ms, cnt = C.c_double(), C.c_int64()
    for r in range(args.rounds):
        order = ("torchvision_cuda", "pil") if r % 2 == 0 else ("pil", "torchvision_cuda")
        for b in order:
            lib.zv_timing_reset()
            lib.zv_timing_enable(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                run(b)
            e1.record()
            torch.cuda.synchronize()
            lib.zv_timing_enable(0)
            cls = []
            for k in ((13, 1) if b == "torchvision_cuda" else (0, 1)):
                _lib.check(lib.zv_timing_read(k, C.byref(ms), C.byref(cnt)))
                cls.append(ms.value / args.iters)
            per[b]["resample_ms"].append(cls[0])
            per[b]["patchify_or_pass2_ms"].append(cls[1])
            per[b]["k1_ms"].append(e0.elapsed_time(e1) / args.iters)
            per[b]["launches"] = procs[b].last_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_hf(chw)
        e1.record()
        torch.cuda.synchronize()
        per["hf"]["call_ms"].append(e0.elapsed_time(e1))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    clk_mhz = float(smi.split(",")[2].split()[0])
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    fma, nbytes = f32_work(args.images)
    t_f32 = statistics.median(per["torchvision_cuda"]["resample_ms"]) * 1e-3
    t_fma, t_hbm = fma / (sms * 128 * clk_mhz * 1e6), nbytes / HBM_BYTES_PER_S
    res = {"what": f"K1 (zv_preprocess) of {args.images} x {IMG}^2 uint8 -> {OUT}^2, fp16 window-order patches, per call; "
                   "HF: Qwen2VLImageProcessor(device='cuda') on the same CUDA images, fp32 HF-order patches, per call",
           "gpu": smi, "rounds": args.rounds, "iters_per_round": args.iters, "kind2_bitexact_vs_hf_image0": check,
           "summary": {
               "kind2_k1_ms_median": statistics.median(per["torchvision_cuda"]["k1_ms"]),
               "kind2_resample_ms_median": statistics.median(per["torchvision_cuda"]["resample_ms"]),
               "kind2_patchify_ms_median": statistics.median(per["torchvision_cuda"]["patchify_or_pass2_ms"]),
               "kind2_launches_per_call": per["torchvision_cuda"]["launches"],
               "kind0_k1_ms_median": statistics.median(per["pil"]["k1_ms"]),
               "kind0_launches_per_call": per["pil"]["launches"],
               "hf_cuda_call_ms_median": statistics.median(per["hf"]["call_ms"]),
               "resample_multiply_adds": fma, "resample_bytes": nbytes,
               "fp32_bound_ms": t_fma * 1e3, "hbm_bound_ms": t_hbm * 1e3,
               "bound": "fp32 pipe" if t_fma >= t_hbm else "hbm",
               "resample_share_of_bound": max(t_fma, t_hbm) / t_f32},
           "per_round": per}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
