"""The LM hand-off on the host against the device hand-off (DeviceHandoff), on one GPU.

    python tools/bench_handoff.py [--iters 200] [--warmup 20] [--out profiles/r07_bench_handoff_n1.json]

Two seeded workloads:
  zoom   batch 1, a prompt of ~800 tokens holding a 512 x 512 global view and one 512 x 512 crop (324 + 324 image tokens),
         through a randomly initialised Qwen2.5-VL-3B tower (32 blocks, fp16 operands, window-ordered fp16 patches as the
         fused preprocess writes them, fp16 embeddings into a (1, L, 2048) inputs_embeds):
           host    get_rope_index (D2H copy, host loop, H2D copy) + embed_images (nonzero, aminmax: host reads) + tower
           device  DeviceHandoff.rope_index + DeviceHandoff.embed_images, eager tower
           graph   the device hand-off and the tower captured as one CUDA graph, replayed
  grpo   B = 64, L = 2048, two 392 x 392 images per sample (196 tokens each), left-padded: get_rope_index against
         DeviceHandoff.rope_index alone.
Each variant is timed with CUDA events around --iters back-to-back calls after --warmup calls; the record holds the mean
per call.  The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

IMG, VSTART, VEND, PAD = 151655, 151652, 151653, 151643


def _card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                      # pragma: no cover
        return f"unknown ({e})"


def _events(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def _prompt(rng, n_tokens, text):
    """[text] (VSTART IMG*t VEND [text])* for each image of n_tokens placeholders."""
    ids = rng.integers(0, 1000, text[0]).tolist()
    for t, tail in zip(n_tokens, text[1:]):
        ids += [VSTART] + [IMG] * t + [VEND] + rng.integers(0, 1000, tail).tolist()
    return ids


def zoom(a, dev):
    from oracle import tower as OT
    from zoomearth_b200 import DeviceHandoff, FusedVisual, embed_images, get_rope_index
    fv = FusedVisual(OT.make_weights(0), device=dev, dtype=torch.float16, operand_dtype=torch.float16)
    grid = torch.tensor([[1, 36, 36], [1, 36, 36]])                  # 504 x 504 px each: 1296 patches, 324 tokens
    rng = np.random.default_rng(0)
    ids_l = _prompt(rng, [324, 324], [60, 40, 80])
    ids = torch.tensor([ids_l], device=dev)
    mask = torch.ones_like(ids)
    S = int((grid[:, 1] * grid[:, 2]).sum())
    pv = torch.randn(S, 1176, generator=torch.Generator().manual_seed(1)).to(torch.float16).to(dev)
    emb = torch.zeros(1, ids.shape[1], 2048, dtype=torch.float16, device=dev)
    dh = DeviceHandoff(dev, 1, ids.shape[1])

    def host():
        get_rope_index(ids, grid, None, mask)
        embed_images(fv, emb, ids, pv, grid, window_order=True)

    def device():
        dh.rope_index(ids, grid, mask)
        dh.embed_images(fv, emb, ids, pv, grid, window_order=True)

    device()
    torch.cuda.synchronize()
    dh.check()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        device()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        device()
    # the three variants write the same inputs_embeds and positions
    host_pos = get_rope_index(ids, grid, None, mask)
    emb.zero_(); host(); ref = emb.clone()
    emb.zero_(); g.replay(); dh.check()
    assert torch.equal(emb, ref)
    dev_pos = dh.rope_index(ids, grid, mask)
    dh.check()
    assert torch.equal(dev_pos[0], host_pos[0]) and torch.equal(dev_pos[1], host_pos[1])
    res = {"tokens": ids.shape[1], "image_tokens": int((ids == IMG).sum()), "grid_thw": grid.tolist()}
    for name, fn in (("host_handoff_eager_tower_ms", host), ("device_handoff_eager_tower_ms", device),
                     ("device_handoff_graph_ms", g.replay)):
        res[name] = _events(fn, a.iters, a.warmup)
    dh.rope_index(ids, grid, mask)
    launches = dh.last_launches
    rows = dh.placeholder_rows(ids, fv.plan_for(grid).num_tokens)
    res["device_handoff_launches"] = launches + dh.last_launches
    fv.forward_into(emb, rows, pv, grid, window_order=True, validate_rows=False)
    res["tower_launches"] = fv.last_launches
    return res


def grpo(a, dev):
    from zoomearth_b200 import DeviceHandoff, get_rope_index
    B, L = 64, 2048
    rng = np.random.default_rng(1)
    grids, rows = [], []
    for _ in range(B):
        grids += [(1, 28, 28), (1, 28, 28)]
        r = _prompt(rng, [196, 196], [int(rng.integers(20, 200)), int(rng.integers(20, 300)), int(rng.integers(100, 900))])
        rows.append(r)
    ids = np.full((B, L), PAD, np.int64)
    mask = np.zeros((B, L), np.int64)
    for i, r in enumerate(rows):
        ids[i, L - len(r):], mask[i, L - len(r):] = r, 1
    ids, mask, grid = torch.from_numpy(ids).to(dev), torch.from_numpy(mask).to(dev), torch.tensor(grids)
    dh = DeviceHandoff(dev, B, L)
    ref = get_rope_index(ids, grid, None, mask)
    got = dh.rope_index(ids, grid, mask)
    dh.check()
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    res = {"batch": B, "seq_len": L, "images": len(grids), "unmasked_tokens": int(mask.sum())}
    res["host_rope_index_ms"] = _events(lambda: get_rope_index(ids, grid, None, mask), a.iters, a.warmup)
    res["device_rope_index_ms"] = _events(lambda: dh.rope_index(ids, grid, mask), a.iters, a.warmup)
    res["device_rope_index_launches"] = dh.last_launches
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_handoff needs a CUDA device; there is no CPU measurement")
    dev = torch.device("cuda", 0)
    rec = {"card": _card(), "iters": a.iters, "warmup": a.warmup, "zoom": zoom(a, dev), "grpo": grpo(a, dev)}
    line = json.dumps(rec, indent=1)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
