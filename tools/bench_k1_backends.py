"""K1 time of bench.py's global-view shape under both resample conventions, back to back on one GPU: 64 synthetic
5000 x 5000 uint8 images (4.8 GB, well past the 126 MB L2) -> 980 x 980 (max_pixels 1280 * 28 * 28), fp16 patches in
the tower's window order, as ZoomEncoder feeds the tower in bench.py.  The two conventions run the same kernels with
different coefficient tables and LUT, so their times should agree within the run-to-run spread.

Each round times `--iters` zv_preprocess calls of one convention, then of the other (which goes first alternates from
round to round), with the library's per-kernel-class event timing (class 0: pass 1, class 1: pass 2 + patchify) and
CUDA events around the calls.  Before timing, image 0 of each convention is checked against its NumPy oracle.

    python tools/bench_k1_backends.py [--images 64] [--rounds 8] [--iters 5] [--out path.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import processor as OP, processor_torchvision as PT  # noqa: E402
from zoomearth_b200 import FusedImageProcessor, _lib  # noqa: E402

IMG, MAX_PIXELS = 5000, 1280 * 28 * 28


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_k1_backends.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    lib = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(1234)
    images = [torch.randint(0, 256, (IMG, IMG, 3), generator=g, dtype=torch.uint8, device=dev) for _ in range(args.images)]
    procs = {b: FusedImageProcessor(min_pixels=3136, max_pixels=MAX_PIXELS, device=dev, backend=b) for b in ("pil", "torchvision")}
    oracles = {"pil": OP, "torchvision": PT}

    checks = {}
    img0 = images[0].cpu().numpy()
    for b, p in procs.items():
        pv, grid, _ = p.preprocess_crops(images[:1], None, torch.float32)
        ref, rgrid, _ = oracles[b].preprocess_u8([img0], 3136, MAX_PIXELS)
        checks[b] = bool(grid.tolist() == rgrid.tolist() and np.array_equal(pv.cpu().numpy(), ref))
    if not all(checks.values()):
        raise SystemExit(f"bench_k1_backends.py: patches differ from the oracle: {checks}")

    def run(b):
        return procs[b].preprocess_crops(images, None, torch.float16, window_order=True)

    for b in procs:                                    # warm up: module load, table cache, workspace
        for _ in range(3):
            run(b)
    torch.cuda.synchronize()
    per = {b: {"k1_ms": [], "pass1_ms": [], "pass2_ms": [], "launches": None} for b in procs}
    ms, cnt = C.c_double(), C.c_int64()
    for r in range(args.rounds):
        order = ("pil", "torchvision") if r % 2 == 0 else ("torchvision", "pil")
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
            for k in (0, 1):
                _lib.check(lib.zv_timing_read(k, C.byref(ms), C.byref(cnt)))
                cls.append(ms.value / args.iters)
            per[b]["pass1_ms"].append(cls[0])
            per[b]["pass2_ms"].append(cls[1])
            per[b]["k1_ms"].append(e0.elapsed_time(e1) / args.iters)
            per[b]["launches"] = procs[b].last_launches
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    summary = {b: {"k1_ms_median": statistics.median(v["k1_ms"]), "k1_ms_min": min(v["k1_ms"]),
                   "pass1_ms_median": statistics.median(v["pass1_ms"]), "pass2_ms_median": statistics.median(v["pass2_ms"]),
                   "launches_per_call": v["launches"]} for b, v in per.items()}
    res = {"what": f"K1 (zv_preprocess) of {args.images} x {IMG}^2 uint8 -> 980^2, fp16 window-order patches, per call",
           "gpu": smi, "rounds": args.rounds, "iters_per_round": args.iters, "oracle_check_image0": checks,
           "summary": summary,
           "torchvision_over_pil_median": summary["torchvision"]["k1_ms_median"] / summary["pil"]["k1_ms_median"],
           "per_round": per}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
