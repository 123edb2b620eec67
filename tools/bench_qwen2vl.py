"""Qwen2-VL-2B vision tower (tower_kind 1: LayerNorm, QuickGELU MLP, full attention in all 32 blocks, merger out 1536) on
one GPU: 64 global views of 980 x 980 px (grid 1 x 70 x 70) in one batch, and one 504 x 504 px zoom crop (1 x 36 x 36),
eager and as a CUDA-graph replay.  fp16 operands, fp16 embeddings, seeded random weights, HF-order fp16 patches.

Reports tokens/s, the per-kernel-class device times of the library's event timing, and the GEMMs' TFLOP/s against the
fp16 dense rate measured by tools/peak_probe.py (profiles/r02_peak_probe_fp16_vs_bf16.json).

    python tools/bench_qwen2vl.py [--out path.json] [--steps 5]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from zoomearth_b200 import FusedVisual, _lib  # noqa: E402

H, I, O, DEPTH = 1280, 5120, 1536, 32
CLASSES = {"gemm_store": 2, "gemm_qkv": 3, "gemm_resid": 4, "gemm_gelu": 6, "gemm_scatter": 7, "gemm_quickgelu": 12,
           "attn_window": 8, "attn_full": 9, "norm": 10, "gather": 11}
GEMM_CLASSES = ("gemm_store", "gemm_qkv", "gemm_resid", "gemm_gelu", "gemm_scatter", "gemm_quickgelu")


def state_dict(seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, device=dev)                         # noqa: E731
    sd = {"patch_embed.proj.weight": 0.02 * r(H, 3, 2, 14, 14)}
    for i in range(DEPTH):
        p = f"blocks.{i}."
        sd.update({p + "norm1.weight": 1 + 0.1 * r(H), p + "norm1.bias": 0.1 * r(H), p + "norm2.weight": 1 + 0.1 * r(H),
                   p + "norm2.bias": 0.1 * r(H), p + "attn.qkv.weight": 0.02 * r(3 * H, H), p + "attn.qkv.bias": 0.1 * r(3 * H),
                   p + "attn.proj.weight": 0.02 * r(H, H), p + "attn.proj.bias": 0.1 * r(H),
                   p + "mlp.fc1.weight": 0.02 * r(I, H), p + "mlp.fc1.bias": 0.1 * r(I),
                   p + "mlp.fc2.weight": 0.02 * r(H, I), p + "mlp.fc2.bias": 0.1 * r(H)})
    sd.update({"merger.ln_q.weight": 1 + 0.1 * r(H), "merger.ln_q.bias": 0.1 * r(H),
               "merger.mlp.0.weight": 0.02 * r(4 * H, 4 * H), "merger.mlp.0.bias": 0.1 * r(4 * H),
               "merger.mlp.2.weight": 0.02 * r(O, 4 * H), "merger.mlp.2.bias": 0.1 * r(O)})
    return sd


def flops(grid):
    """(GEMM FLOP, attention FLOP) of one forward over `grid` (t, h, w) rows."""
    seg = [t * h * w for t, h, w in grid]
    S = sum(seg)
    T = S // 4
    gemm = 2 * S * 1176 * H + DEPTH * 2 * S * H * (3 * H + H + I + I) + 2 * T * (4 * H) * (4 * H + O)
    attn = DEPTH * sum(4 * s * s * H for s in seg)
    return gemm, attn


def timed(fn, steps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def class_times(fn, steps):
    lib = _lib.lib()
    lib.zv_timing_reset()
    lib.zv_timing_enable(1)
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    lib.zv_timing_enable(0)
    out = {}
    for k, c in CLASSES.items():
        t, n = C.c_double(), C.c_int64()
        _lib.check(lib.zv_timing_read(c, C.byref(t), C.byref(n)))
        out[k] = {"ms_per_step": round(t.value / steps, 4), "launches_per_step": n.value // steps}
    lib.zv_timing_reset()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_qwen2vl needs a CUDA device (sm_100); nothing is measured without one")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    fv = FusedVisual(state_dict(0, dev), device=dev, dtype=torch.float16, operand_dtype=torch.float16,
                     depth=DEPTH, inter=I, out_hidden=O, fullatt=list(range(DEPTH)), tower_kind=_lib.TOWER_QWEN2)
    peak_file = os.path.join(ROOT, "profiles", "r02_peak_probe_fp16_vs_bf16.json")
    peak = max(v["tflops"] for k, v in json.load(open(peak_file)).items() if k.startswith("fp16"))
    rec = {"gpu": smi, "tower": "Qwen2-VL-2B vision (tower_kind 1), fp16 operands, fp16 out",
           "measured_fp16_peak_tflops": round(peak, 1)}
    g = torch.Generator(device=dev).manual_seed(1)
    for name, grid, steps in (("64 x 980^2 global views", [(1, 70, 70)] * 64, args.steps),
                              ("one 504^2 zoom crop", [(1, 36, 36)], 20 * args.steps)):
        gt = torch.tensor(grid)
        S = sum(t * h * w for t, h, w in grid)
        pv = torch.randn(S, 1176, generator=g, device=dev).half()
        ms = timed(lambda: fv(pv, gt), steps)
        cls = class_times(lambda: fv(pv, gt), steps)
        gf, af = flops(grid)
        gemm_ms = sum(cls[k]["ms_per_step"] for k in GEMM_CLASSES)
        attn_ms = cls["attn_full"]["ms_per_step"] + cls["attn_window"]["ms_per_step"]
        r = {"patches": S, "tokens": S // 4, "ms_per_step": round(ms, 3), "tokens_per_s": round(S / 4 / ms * 1e3, 1),
             "launches": fv.last_launches, "gemm_tflop": round(gf / 1e12, 3), "attn_tflop": round(af / 1e12, 3),
             "gemm_tflops": round(gf / gemm_ms / 1e9, 1), "gemm_share_of_measured_peak": round(gf / gemm_ms / 1e9 / peak, 3),
             "attn_tflops": round(af / attn_ms / 1e9, 1), "classes": cls}
        if len(grid) == 1:
            r["graph_ms_per_step"] = round(timed(lambda: fv(pv, gt, use_graph=True), steps), 3)
        rec[name] = r
        print(name, json.dumps({k: v for k, v in r.items() if k != "classes"}), flush=True)
    print(json.dumps(rec, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
