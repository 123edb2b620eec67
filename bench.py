#!/usr/bin/env python
"""bench.py - vision tokens/s through crop -> patchify -> ViT (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 3 --warmup 3            # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus 1 --steps 1      # the reference's CPU path on the host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU, weak scaling by image
    python bench.py --steps 3 --dump-outputs bench_outputs   # + the last timed step's outputs as .npy files

Workload = BASELINE.json configs[1]: "Global view: 64 synthetic 5000x5000 images downscaled to
max_pixels=1280*28*28" -> per image 980x980, grid (1,70,70), 4900 patches, 1225 vision tokens.  One step =
one pass of the hot path over that batch: zv_preprocess (K1, fp16 patches in window order) then
zv_visual_forward (32-block tower + merger), random-init Qwen2.5-VL-3B vision weights, synthetic pixels.

`value`   : tokens/s with the uint8 images already resident in HBM (device-timed, CUDA events, max over ranks).
`e2e`     : same metric through the public Python surface with HOST (pinned) uint8 images: H2D of the pixels and
            D2H of the embeddings inside the timed region.
`roofline`: all tcgen05 GEMM launches of the timed region (event-timed per launch on the launching stream)
            against the measured dense bf16 peak; `roofline_k1` / `roofline_attn` give the other kernel classes.
`cpu_baseline`: the reference's own CPU path (Pillow + HF PIL processor + HF torch tower, fp32) on a bounded
            sample of the same workload, on this box's host cores.

Inputs (weights, pixels) are generated from fixed seeds, so two builds run with the same arguments see the same inputs
and their --dump-outputs directories can be compared file by file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG = 5000
MAX_PIXELS = 1280 * 28 * 28
MIN_PIXELS = 56 * 56
# DRAM traffic of the dominant kernels (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch at this workload) is
# NOT typed in here: tools/ncu_traffic.py turns the ncu CSV of the current tree into profiles/ncu_traffic.json (with the
# commit it was captured at) and this file is read at run time; without it the `traffic` fields are null.
def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


WORKLOAD = ("BASELINE configs[1]: global view, 64 synthetic 5000x5000 uint8 images -> max_pixels=1280*28*28 "
            "(980x980, grid 1x70x70, 1225 tokens/image) -> Qwen2.5-VL-3B vision tower (random init)")
KCLASS = {"k1_hpass": 0, "k1_vpass": 1, "gemm_store": 2, "gemm_qkv": 3, "gemm_resid": 4, "gemm_swiglu": 5,
          "gemm_gelu": 6, "gemm_scatter": 7, "attn_window": 8, "attn_full": 9, "rmsnorm": 10, "gather": 11}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def flops_per_step(n_img, S_img):
    """Algorithmic FLOPs (SURVEY 8d): linear, window attention, full attention.  grid 70x70 per image."""
    S, T = n_img * S_img, n_img * S_img // 4
    f_lin = S * 1262940160 + T * 73400320
    # window attention: 28 layers, sum over windows 4 n^2 1280 ; 70x70 grid -> 35x35 merge groups -> windows of 4x4
    lh = lw = 35
    n_w = []
    for wy in range(0, lh, 4):
        for wx in range(0, lw, 4):
            n_w.append(4 * min(4, lh - wy) * min(4, lw - wx))
    f_win = 28 * n_img * sum(4 * n * n * 1280 for n in n_w)
    f_full = 4 * n_img * 4 * S_img * S_img * 1280
    return f_lin, f_win, f_full


# ------------------------------------------------------------------------------------------- reference arm (CPU)
def reference_step(sample_images, seed0=0):
    """The reference's CPU path on `sample_images` images of the workload: Pillow + HF PIL processor + HF tower."""
    from PIL import Image
    from oracle import hf_live, tower as OT
    torch.set_num_threads(os.cpu_count() or 1)
    model = hf_live.hf_tower(None, OT.CFG, torch.float32, seed=0)
    imgs = [np.random.default_rng(seed0 + i).integers(0, 256, (IMG, IMG, 3), dtype=np.uint8) for i in range(sample_images)]
    t0 = time.perf_counter()
    tokens = 0
    for im in imgs:
        pil = Image.fromarray(im)
        crop, _ = hf_live.pil_cut_image(im, (0, 0, IMG, IMG))          # global view: the full-image box
        pv, grid = hf_live.hf_preprocess([crop], MIN_PIXELS, MAX_PIXELS)
        out = hf_live.hf_tower_forward(model, pv, grid)
        tokens += out.shape[0]
        del pil
    dt = time.perf_counter() - t0
    return tokens, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample of the workload per step (BASELINE.md 3: 4 items), shrunk so that K steps stay within a few minutes
    # (one 5000x5000 image takes ~4 s of the reference's CPU path on 16 cores)
    sample = max(1, min(args.ref_images, 48 // max(1, args.steps)))
    for _ in range(max(0, args.warmup if args.warmup < 2 else 1)):
        reference_step(1)
    times = []
    tokens = 0
    for _ in range(args.steps):
        tokens, dt = reference_step(sample)
        times.append(dt)
    dt = float(np.mean(times))
    v = tokens / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "vision tokens/s crop->patchify->ViT", "value": v, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_step": sample,
                   "sample": f"each step times {sample} of the 64 images on the host cores (bounded sample of the workload)"},
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": cores, "kind": "reference",
                         "sample": f"{sample} of the 64 images per step: PIL crop + HF Qwen2VLImageProcessorPil + HF "
                                   f"Qwen2_5_VisionTransformerPretrainedModel fp32 sdpa, {cores} torch threads"},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def zoom_step_latency(visual, dev, reps=30):
    """The reference's own regime (infer.py:17 BATCH_SIZE = 1): one 512-px zoom crop (324 tokens) and four crops of
    512-1024 px, each as one call of the public fast path with CUDA-graph replay of the tower; wall clock per call."""
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder
    enc = ZoomEncoder(visual, FusedImageProcessor(min_pixels=3136, max_pixels=128 * 128 * 28 * 28, device=dev))
    img = torch.randint(0, 256, (IMG, IMG, 3), dtype=torch.uint8, device=dev)
    out = {}
    for name, boxes in (("one_512px_zoom_step_ms", [(2000, 2000, 2512, 2512)]),
                        ("four_crops_512_to_1024px_ms", [(100, 100, 612, 612), (900, 900, 1700, 1500), (2000, 100, 3024, 1124),
                                                        (3000, 3000, 3700, 3600)])):
        for _ in range(5):
            enc.encode([img], boxes, image_index=[0] * len(boxes), use_graph=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            emb, _, _ = enc.encode([img], boxes, image_index=[0] * len(boxes), use_graph=True)
        torch.cuda.synchronize()
        out[name] = (time.perf_counter() - t0) / reps * 1e3
        out[name.replace("_ms", "_tokens")] = int(emb.shape[0])
    return out


def config3_sharded(enc, visual, dev, rank, world, op_dtype, n_crops):
    """BASELINE configs[3] as a sub-record of the line: `n_crops` mixed-size crops (256-2048 px per side, cut_image rule)
    of 16 replicated source images, STRONG scaling - sharded over the ranks by LPT partition, every rank's merger GEMM
    scattering its embedding rows to their global rows of every rank's gather buffer (ragged fused gather).  One warm-up
    pass, one timed pass (CUDA events, max over ranks).  At N=1 the same crops run through the same micro-batched path."""
    import torch.distributed as dist
    from zoomearth_b200 import FusedImageProcessor, ZoomEncoder, sharding, synthetic
    enc3 = ZoomEncoder(visual, FusedImageProcessor(min_pixels=MIN_PIXELS, max_pixels=16384 * 28 * 28, device=dev))
    g = torch.Generator(device=dev).manual_seed(7)                  # same pool on every rank (images are replicated)
    pool = [torch.randint(0, 256, (IMG, IMG, 3), generator=g, dtype=torch.uint8, device=dev) for _ in range(16)]
    boxes, index = synthetic.mixed_crop_boxes(n_crops, 16)
    pg3, total, check = None, None, None
    if world > 1:
        from zoomearth_b200 import geometry
        cfg = enc3.processor._cfg()
        _, _, grid = geometry.geometry(cfg, np.array([[IMG, IMG]] * n_crops, np.int32), boxes.astype(np.float64))
        total = int(((grid[:, 1] * grid[:, 2]) // 4).sum())
        pg3 = sharding.PeerGather(total, 2048, op_dtype, dev)

    def one_pass():
        if pg3 is None:
            emb, _, _ = enc3.encode_batched(pool, boxes, index)
            return emb
        out, _, _ = sharding.encode_sharded(enc3, pool, boxes, index, pg3)
        pg3.barrier()
        return out

    out = one_pass()
    torch.cuda.synchronize()
    if world > 1:
        # correctness of the ragged fused gather, once: every crop's rows equal what its owner computes on its own
        parts = sharding.partition(sharding.crop_cost(np.asarray(grid)), world)
        mine = parts[rank][:3]
        starts = np.concatenate([[0], np.cumsum((grid[:, 1] * grid[:, 2]) // 4)])
        ok = 1
        for i in mine:
            e, _, _ = enc3.encode([pool[int(index[i])]], [boxes[i]], image_index=[0])
            got = out[int(starts[i]):int(starts[i + 1])].float()
            # not bitwise: a segment's K/V tile split in the full-attention layers depends on its row offset in the batch
            ok &= int(got.shape == e.shape and ((got - e.float()).abs().max() / e.float().abs().max()).item() <= 5e-3)
        t = torch.tensor([ok], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        # ... and every rank holds the same bytes
        h = torch.stack([out.view(torch.int16).to(torch.int64).sum()])
        hs = [torch.zeros_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        check = bool(t.item()) and all(int(x) == int(hs[0]) for x in hs)
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = one_pass()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    tokens = int(out.shape[0])
    del pool
    return {"workload": f"BASELINE configs[3]: {n_crops} mixed-size crops (256-2048 px) of 16 source images, cut_image rule, "
                        f"max_pixels=12845056, sharded by crop (LPT) over {world} GPU(s)", "scaling": "strong",
            "tokens": tokens, "ms": ms, "value": tokens / (ms / 1e3), "unit": "tokens/s",
            "gather": "ragged fused gather (zv_visual_forward_gather_rows): per-row peer stores from the merger GEMM epilogue"
                      if world > 1 else "none (single GPU)", "gather_check": check}


# ------------------------------------------------------------------------------------------- our arm (CUDA)
DUMP_ROWS = 4096            # 4096 x 2048 float32 = 32 MiB of embeddings


def dump_outputs(out_dir, emb, grid, crop):
    """What one step hands its caller, as .npy files: embeddings.npy (a fixed, seeded sample of DUMP_ROWS rows in
    ascending order, all rows when there are fewer; float32 holds the fp16 / bf16 values exactly), image_grid_thw.npy
    and crop_boxes.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    n = emb.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS else np.arange(n)
    sample = emb[torch.from_numpy(rows).to(emb.device)].float().cpu().numpy()
    np.save(os.path.join(out_dir, "embeddings.npy"), sample)
    np.save(os.path.join(out_dir, "image_grid_thw.npy"), np.asarray(grid, np.float64))
    np.save(os.path.join(out_dir, "crop_boxes.npy"), np.asarray(crop, np.float64))


def run_ours(args):
    import torch.distributed as dist
    from zoomearth_b200 import FusedImageProcessor, FusedVisual, ZoomEncoder, _lib
    from zoomearth_b200.synthetic import random_vision_state_dict

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stdout_fd = None
    if world > 1:
        # NCCL prints its version banner to stdout at communicator creation: keep stdout to the one JSON line by
        # pointing fd 1 at stderr until the line is printed
        sys.stdout.flush()
        stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    n_img = args.images
    pk = peaks()

    sd = random_vision_state_dict(0, device=dev)
    op_dtype = torch.float16 if args.operand_dtype == "fp16" else torch.bfloat16
    visual = FusedVisual(sd, device=dev, dtype=op_dtype, operand_dtype=op_dtype)
    del sd
    enc = ZoomEncoder(visual, FusedImageProcessor(min_pixels=MIN_PIXELS, max_pixels=MAX_PIXELS, device=dev))
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    images = [torch.randint(0, 256, (IMG, IMG, 3), generator=g, dtype=torch.uint8, device=dev) for _ in range(n_img)]
    S_img, T_img = 4900, 1225
    tokens_step = n_img * T_img

    pg, gather_kind = None, "none"
    if world > 1:
        gather_kind = "nccl all_gather_into_tensor"
        if not args.nccl_gather:
            try:
                from zoomearth_b200.sharding import PeerGather
                pg = PeerGather(world * tokens_step, 2048, op_dtype, dev, double_buffer=True)
                gather_kind = ("fused: merger GEMM epilogue stores into every rank's buffer over NVLink (symmetric memory); "
                               "two buffers, the barrier of step i is waited on at the start of step i+1")
            except Exception as e:          # symmetric memory unavailable on this box: the NCCL collective still gathers
                pg = None
                if rank == 0:
                    print(f"bench.py: fused peer gather unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
        ok = torch.tensor([1 if pg is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() == 0 and pg is not None:
            pg, gather_kind = None, "nccl all_gather_into_tensor"

    def step():
        """(embeddings of every rank, or None while the fused gather is in flight; grids; crop boxes)"""
        if pg is not None:
            pg.begin_step()                                # waits for the PREVIOUS step's cross-rank barrier, flips buffers
            _, grid, crop = enc.encode(images, None, gather=pg, gather_row=rank * tokens_step)
            pg.end_step()                                  # this step's barrier runs on a side stream behind the kernels
            return None, grid, crop
        emb, grid, crop = enc.encode(images, None)
        if world > 1:
            out = torch.empty((world * emb.shape[0], emb.shape[1]), dtype=emb.dtype, device=dev)
            dist.all_gather_into_tensor(out, emb)          # C1: gather of the output embeddings (equal shards)
            return out, grid, crop
        return emb, grid, crop

    def barrier():
        if pg is not None:
            pg.finish()                                    # the last step's gather is complete on every rank
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    gather_check = None
    if world > 1:
        # correctness of the data path being timed: what step() leaves on every rank must be, bit for bit, NCCL's
        # all_gather_into_tensor of the per-rank embeddings (checked once, outside the timed region)
        got, _, _ = step()
        got = (pg.finish() if pg is not None else got).clone()
        barrier()
        emb, _, _ = enc.encode(images, None)
        want = torch.empty((world * emb.shape[0], emb.shape[1]), dtype=emb.dtype, device=dev)
        dist.all_gather_into_tensor(want, emb)
        same = torch.tensor([1 if torch.equal(got, want) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        gather_check = bool(same.item())
        del got, want, emb
        barrier()
    sampler = ClockSampler(local)
    sampler.start()
    lib.zv_timing_reset()
    lib.zv_timing_enable(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    launches = 0
    for _ in range(args.steps):
        last = step()
        launches += enc.last_launches
    if pg is not None:
        pg.finish()                                        # inside the timed region: every step's gather has landed
    e1.record()
    barrier()
    lib.zv_timing_enable(0)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        emb, grid, crop = last
        dump_outputs(args.dump_outputs, emb if pg is None else pg.finish(), grid, crop)
        del emb
    del last
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    ms_step = ms / args.steps
    value = world * tokens_step / (ms_step / 1e3)

    # per-kernel-class device time inside the timed region
    cls = {}
    for name, cid in KCLASS.items():
        t, n = C.c_double(), C.c_int64()
        _lib.check(lib.zv_timing_read(cid, C.byref(t), C.byref(n)))
        cls[name] = (t.value, n.value)
    lib.zv_timing_reset()
    f_lin, f_win, f_full = flops_per_step(n_img, S_img)
    gemm_ms = sum(cls[k][0] for k in cls if k.startswith("gemm"))
    gemm_n = sum(cls[k][1] for k in cls if k.startswith("gemm"))
    gemm_tf = f_lin * args.steps / (gemm_ms / 1e3) / 1e12 if gemm_ms else 0.0
    k1_ms = cls["k1_hpass"][0] + cls["k1_vpass"][0]
    k1_bytes = n_img * (IMG * IMG * 3 + S_img * 1176 * 2)
    k1_gbs = k1_bytes * args.steps / (k1_ms / 1e3) / 1e9 if k1_ms else 0.0
    attn_ms = cls["attn_window"][0] + cls["attn_full"][0]
    attn_tf = (f_win + f_full) * args.steps / (attn_ms / 1e3) / 1e12 if attn_ms else 0.0
    tower_tf = (f_lin + f_win + f_full) * args.steps / ((ms - k1_ms) / 1e3) / 1e12

    # ---- K1 alone (no GEMMs before it: the SM clock is not dragged down by the power cap), same 64 images, device-timed
    k1_alone = None
    if rank == 0:
        proc = enc.processor
        for _ in range(2):
            proc.preprocess_crops(images, None, out_dtype=op_dtype, window_order=True)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            proc.preprocess_crops(images, None, out_dtype=op_dtype, window_order=True)
        a1.record()
        torch.cuda.synchronize()
        k1a_ms = a0.elapsed_time(a1) / 5
        k1_alone = {"ms_per_step": k1a_ms, "achieved": k1_bytes / (k1a_ms / 1e3) / 1e9, "unit": "GB/s",
                    "frac": k1_bytes / (k1a_ms / 1e3) / 1e9 / pk["hbm"],
                    "note": "zv_preprocess of the same 64 images back to back, nothing else on the GPU (includes the table upload)"}

    # ---- e2e: host (pinned) pixels in, embeddings out to the host, through the public API
    e2e = None
    if not args.no_e2e:
        n_e2e = min(n_img, args.e2e_images)
        e2e_schedule = [int(v) for v in args.e2e_schedule.split(",")] if args.e2e_schedule else None
        host = [im.cpu().pin_memory() for im in images[:n_e2e]]
        out_host = torch.empty((n_e2e * T_img, 2048), dtype=op_dtype).pin_memory()

        def step_e2e():
            # H2D of this step's pixels and D2H of its embeddings, pipelined in chunks behind the compute
            enc.encode_host(host, chunk=args.e2e_chunk, out_host=out_host, schedule=e2e_schedule)

        # the link the e2e figure is bound by: pinned host -> device bandwidth of this box (8 images, 600 MB)
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        tmp_dev = [h.to(dev, non_blocking=True) for h in host[:8]]
        h1.record()
        torch.cuda.synchronize()
        h2d_gbps = sum(h.numel() for h in host[:8]) / (h0.elapsed_time(h1) / 1e3) / 1e9
        del tmp_dev
        for _ in range(2):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        k_e2e = max(1, args.steps)
        for _ in range(k_e2e):
            step_e2e()
        barrier()
        dt = (time.perf_counter() - t0) / k_e2e
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = t.item()
        e2e = {"value": world * n_e2e * T_img / dt, "unit": "tokens/s", "h2d_bytes_per_step": n_e2e * IMG * IMG * 3,
               "d2h_bytes_per_step": n_e2e * T_img * 2048 * 2, "images_per_step": n_e2e, "ms_per_step": dt * 1e3,
               "h2d_gbps_measured": h2d_gbps, "h2d_ms_per_step_at_that_rate": n_e2e * IMG * IMG * 3 / h2d_gbps / 1e6,
               "pipeline": (f"chunks of {e2e_schedule} images (ramp: a short first chunk keeps the exposed upload small, long later "
                            f"chunks keep the tower's batches large)" if e2e_schedule else f"chunks of {args.e2e_chunk} images") +
                           ": H2D on a copy stream, K1+tower, D2H on a third stream"}
        del host

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu:
        tokens, dt = reference_step(args.ref_images)
        cores = torch.get_num_threads()
        cpu_base = {"value": tokens / dt, "unit": "tokens/s", "cores": cores, "kind": "reference",
                    "sample": f"{args.ref_images} of the {n_img} images of one step ({tokens} tokens, {dt:.1f} s): PIL crop + "
                              f"HF Qwen2VLImageProcessorPil + HF vision tower fp32 sdpa on {cores} threads"}

    sharded = None
    if not args.no_sharded:
        sharded = config3_sharded(enc, visual, dev, rank, world, op_dtype, args.sharded_crops)

    latency = None
    if rank == 0 and world == 1 and not args.no_latency:
        latency = zoom_step_latency(visual, dev)

    traffic = ncu_traffic() or {}
    if rank == 0:
        line = {
            "metric": "vision tokens/s crop->patchify->ViT", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.operand_dtype, "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "images_per_step_per_gpu": n_img, "tokens_per_step_per_gpu": tokens_step,
                       "l2": "inputs larger than L2 (4.8 GB of pixels, 5.5 GB of activations per step)",
                       "parallelism": f"dp{world} by image; embedding gather: {gather_kind}" if world > 1 else "single GPU"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": e2e,
            "roofline": {"bound": "tensor", "kernel": "gemm_tc (tcgen05, all epilogues)", "achieved": gemm_tf,
                         "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": gemm_tf / pk["tf_sust"],
                         "frac_of_burst": gemm_tf / pk["tf_burst"], "frac_of_nominal_2250": gemm_tf / 2250.0,
                         "peak_source": pk["src"] + ", sustained",
                         "traffic": traffic.get("gemm_bytes_per_launch") if n_img == 64 else None,
                         "traffic_note": traffic.get("gemm_note", "no ncu capture of this tree under profiles/ncu_traffic.json"),
                         "launches": gemm_n, "ms_total": gemm_ms, "share_of_step": gemm_ms / ms},
            "roofline_k1": {"bound": "hbm", "kernel": "k1_resample_tc x2 (tcgen05 kind::i8 + TMA: horizontal, vertical pass) + k1_patchify_u8", "achieved": k1_gbs, "peak": pk["hbm"],
                            "unit": "GB/s", "frac": k1_gbs / pk["hbm"], "frac_of_nominal_8000": k1_gbs / 8000.0, "ms_total": k1_ms, "share_of_step": k1_ms / ms,
                            "traffic": (traffic.get("k1_bytes_per_image") * n_img) if traffic.get("k1_bytes_per_image") else None,
                            "traffic_note": traffic.get("k1_note", "no ncu capture of this tree under profiles/ncu_traffic.json"),
                            "algorithmic_bytes": k1_bytes, "alone": k1_alone},
            "roofline_attn": {"bound": "tensor", "kernel": "attn_tc_kernel (tcgen05, full layers) + attn_win_tc_kernel (tcgen05, window layers)", "achieved": attn_tf,
                              "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": attn_tf / pk["tf_sust"],
                              "ms_total": attn_ms, "share_of_step": attn_ms / ms,
                              "full_layers_tflops": (f_full * args.steps / (cls["attn_full"][0] / 1e3) / 1e12) if cls["attn_full"][0] else 0.0,
                              "window_layers_gbps": (28 * n_img * S_img * 10240 * args.steps / (cls["attn_window"][0] / 1e3) / 1e9)
                              if cls["attn_window"][0] else 0.0},
            "tower_tflops": tower_tf,
            "kernel_ms": {k: round(v[0] / args.steps, 3) for k, v in cls.items()},
            "cpu_baseline": cpu_base,
            "latency": latency,
            "sharded": sharded,
        }
        if gather_check is not None:
            line["gather_check"] = gather_check
        if stdout_fd is not None:
            sys.stdout.flush()
            C.CDLL(None).fflush(None)           # NCCL's banner may still sit in the C stdio buffer of stdout
            os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images", type=int, default=64, help="images per step per GPU (BASELINE configs[1]: 64)")
    ap.add_argument("--e2e-images", type=int, default=64)
    ap.add_argument("--e2e-chunk", type=int, default=8, help="images per pipelined upload/compute chunk in the e2e leg")
    ap.add_argument("--e2e-schedule", default="2,6,8,16,32", help="chunk sizes of the e2e pipeline (the last repeats); '' = --e2e-chunk")
    ap.add_argument("--ref-images", type=int, default=4, help="images in the CPU reference sample (BASELINE.md 3: 4 items)")
    ap.add_argument("--operand-dtype", default="fp16", choices=["fp16", "bf16"],
                    help="16-bit type of the GEMM / attention operands (fp16 = the shipped default; same tensor-core rate)")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the configs[3] sub-record")
    ap.add_argument("--sharded-crops", type=int, default=1024, help="crops of the configs[3] sub-record (SURVEY: 1024)")
    ap.add_argument("--nccl-gather", action="store_true", help="gather embeddings with NCCL instead of the fused peer stores")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (rank 0; our arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
