"""Oracle: torch's fp32 antialiased bicubic resize as a CUDA device runs it, restated in NumPy.  Test infrastructure only.

This is what HF's torchvision image-processor backend runs when it is called with ``device="cuda"``
(``TorchvisionBackend.resize`` -> ``torchvision.transforms.v2.functional.resize(uint8 CUDA tensor, BICUBIC,
antialias=True)``): the uint8 image is cast to fp32, aten ``upsample_gen2d_aa_out_frame<float, float,
BicubicFilterFunctor>`` resamples both axes with no rounding between them, then ``clamp_(0, 255)``, ``round_()`` (half
to even) and uint8.  When neither size changes the image is returned untouched.

Every step is fp32, in the operations torch's sm_100 SASS performs:

- ``scale = f32(in) / out``; ``support = 2 scale`` if ``scale >= 1`` else 2; ``invscale = 1 / scale`` (correctly
  rounded) if ``scale >= 1`` else 1.
- per output i, with ``ci = f32(i) + 0.5``: ``xmin = max(int(FFMA(ci, scale, -support) + 0.5), 0)``,
  ``xsize = min(int(FFMA(ci, scale, support) + 0.5), in) - xmin``, ``xmin - center = FFMA(-ci, scale, f32(xmin))``
  (the centre ``scale ci`` is never rounded on its own).
- ``w_j = filter(((j + (xmin - center)) + 0.5) invscale)`` with Pillow's cubic, a = -0.5, whose Horner steps are FFMAs;
  the weights are summed in order and each is divided by the sum.
- each pass: ``acc = t_0 w_0``, then ``acc = FFMA(t_j, w_j, acc)`` in increasing j.

FFMA rounds ``a b + c`` once.  ``ffma`` forms the product exactly in float64 (24 + 24 bits), adds in float64 and rounds
to float32; that second rounding can only go wrong when the float64 sum is inexact and lands exactly on a float32
midpoint, and there the exact error of the float64 sum (TwoSum) says which way the true value lies.

Pinned against live torch on a CUDA device in ``tests/test_gpu_torchvision_cuda_backend.py``.
"""
import math

import numpy as np

F32 = np.float32


def ffma(a, b, c):
    """Elementwise fp32 fused multiply-add with one rounding (IEEE fmaf), on float32 arrays or scalars."""
    a, b, c = (np.asarray(v, np.float32).astype(np.float64) for v in (a, b, c))
    p = a * b                                         # exact: 48 significant bits
    s = p + c
    bb = s - c                                        # TwoSum: s + e == p + c exactly
    e = (p - bb) + (c - (s - bb))
    r = s.astype(np.float32)
    r64 = r.astype(np.float64)
    toward = np.where(s > r64, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32)
    other = np.nextafter(r, toward)                   # the float32 neighbour on the other side of s
    tie = (s != r64) & (s == (r64 + other.astype(np.float64)) / 2) & (e != 0)
    pick_hi = e > 0                                   # the true value lies above the midpoint
    fixed = np.where(pick_hi, np.maximum(r, other), np.minimum(r, other))
    return np.where(tie, fixed, r).astype(np.float32)


def _filter(x):
    """Pillow's bicubic (a = -0.5) as torch's SASS evaluates it, on a float32 scalar"""
    x = F32(abs(x))
    if x < 1:
        return ffma(x, x * ffma(x, F32(1.5), F32(-2.5)), F32(1.0))[()]
    if x < 2:
        return F32(ffma(x, ffma(x, x - F32(5), F32(8)), F32(-4))[()] * F32(-0.5))
    return F32(0.0)


def weights(in_size, out_size):
    """Per output index: (xmin, xsize, fp32 weights[xsize]) and interp_size, exactly as torch's kernel computes them."""
    scale = F32(in_size) / F32(out_size)
    support = scale + scale if scale >= 1 else F32(2.0)
    invscale = F32(1.0) / scale if scale >= 1 else F32(1.0)
    interp_size = int(math.ceil(support)) * 2 + 1
    rows = []
    for i in range(out_size):
        ci = F32(i) + F32(0.5)
        xmin = max(int(ffma(ci, scale, -support)[()] + F32(0.5)), 0)
        xsize = min(int(ffma(ci, scale, support)[()] + F32(0.5)), in_size) - xmin
        xmc = ffma(-ci, scale, F32(xmin))[()]
        w = np.array([_filter((F32(j) + xmc + F32(0.5)) * invscale) for j in range(xsize)], np.float32)
        total = F32(0.0)
        for v in w:                                   # sequential, left to right
            total = F32(total + v)
        if total != 0:
            w = (w / total).astype(np.float32)
        rows.append((xmin, xsize, w))
    return rows, interp_size


def _pass_axis1(src, rows):
    """fp32 pass along axis 1 of src[(R, in, C)] -> (R, out, C): t_0 w_0, then FFMA chains in increasing j."""
    out = np.empty((src.shape[0], len(rows), src.shape[2]), np.float32)
    for i, (xmin, xsize, w) in enumerate(rows):
        acc = (src[:, xmin] * w[0]).astype(np.float32)
        for j in range(1, xsize):
            acc = ffma(src[:, xmin + j], w[j], acc)
        out[:, i] = acc
    return out


def resize_u8(src, out_w, out_h):
    """``tvF.resize(uint8 CUDA image, (out_h, out_w), BICUBIC, antialias=True)`` on an (H, W, C) uint8 array."""
    assert src.dtype == np.uint8 and src.ndim == 3
    in_h, in_w, _ = src.shape
    if (in_h, in_w) == (out_h, out_w):
        return src.copy()
    f = src.astype(np.float32)
    f = _pass_axis1(f, weights(in_w, out_w)[0])                                # horizontal, every input row
    f = _pass_axis1(f.transpose(1, 0, 2), weights(in_h, out_h)[0]).transpose(1, 0, 2)
    return np.rint(np.clip(f, 0, 255)).astype(np.uint8)
