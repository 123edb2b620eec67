"""Oracle: torch's uint8 antialiased bicubic resize, restated in NumPy.  Test infrastructure only.

This is what HF's torchvision image-processor backend runs on transformers 5.x
(``image_processing_backends.py`` ``TorchvisionBackend.resize`` ->
``torchvision.transforms.v2.functional.resize(uint8, BICUBIC, antialias=True)``
-> aten ``_upsample_bicubic2d_aa`` on uint8).  The algorithm is Pillow's
(``oracle.resample``): the same windows, the same a = -0.5 bicubic weights,
normalised in fp64.  Only the quantisation differs: each AXIS gets a precision
``p``, the first ``p < 22`` with ``int(0.5 + w_max * 2^(p+1)) >= 2^15``
(``w_max`` = the largest normalised weight over the axis, 22 when none is),
and every tap is rounded to an int16 ``int(+-0.5 + w * 2^p)``.  Each pass
rounds with ``(acc + 2^(p-1)) >> p`` and clips to uint8; the horizontal pass
runs first, an axis whose size does not change is skipped.

Pinned against the installed torch / torchvision in
``tests/test_torchvision_backend.py``.
"""
import math

import numpy as np

from .resample import _bicubic


def precompute_coeffs(in_size, out_size):
    """Per-axis taps: returns (ksize, bounds[out,2] int32 (xmin,count), kk[out,ksize] int32 (int16 values), precision)."""
    scale = in_size / out_size
    support = 2.0 * scale if scale >= 1.0 else 2.0
    ksize = int(math.ceil(support)) * 2 + 1
    invscale = 1.0 / scale if scale >= 1.0 else 1.0
    bounds = np.zeros((out_size, 2), np.int32)
    w = np.zeros((out_size, ksize), np.float64)
    w_max = 0.0
    for xx in range(out_size):
        center = scale * (xx + 0.5)
        xmin = max(int(center - support + 0.5), 0)
        xsize = min(max(min(int(center + support + 0.5), in_size) - xmin, 0), ksize)
        total = 0.0
        for j in range(xsize):
            v = _bicubic((j + xmin - center + 0.5) * invscale)
            w[xx, j] = v
            total += v                                # sequential, left to right
        if total != 0.0:
            for j in range(xsize):
                w[xx, j] /= total
                w_max = max(w_max, w[xx, j])
        bounds[xx] = (xmin, xsize)
    precision = 0
    while precision < 22 and int(0.5 + w_max * (1 << (precision + 1))) < (1 << 15):
        precision += 1
    kk = np.zeros((out_size, ksize), np.int32)
    for xx in range(out_size):
        for j in range(ksize):
            v = w[xx, j] * (1 << precision)
            kk[xx, j] = int(-0.5 + v) if v < 0 else int(0.5 + v)
    return ksize, bounds, kk, precision


def coeffs_22bit(in_size, out_size):
    """The same taps moved to Pillow's 22-bit scale (``kk << (22 - p)``), the form K1 consumes; a same-size axis is one
    exact tap per output, as in ``zv_resample_coeffs``.  Returns (bounds, kk, precision)."""
    if in_size == out_size:
        bounds = np.stack([np.arange(out_size), np.ones(out_size)], 1).astype(np.int32)
        return bounds, np.full((out_size, 1), 1 << 22, np.int32), 22
    _, bounds, kk, p = precompute_coeffs(in_size, out_size)
    return bounds, (kk.astype(np.int64) << (22 - p)).astype(np.int32), p


def _pass_axis1(src, bounds, kk, precision, out_size):
    """Filter along axis 1 of src[(rows, in, C)] u8 -> (rows, out, C) u8."""
    rows, _, ch = src.shape
    out = np.empty((rows, out_size, ch), np.uint8)
    s64 = src.astype(np.int64)
    for xx in range(out_size):
        xmin, n = int(bounds[xx, 0]), int(bounds[xx, 1])
        acc = np.tensordot(s64[:, xmin:xmin + n, :], kk[xx, :n].astype(np.int64), axes=([1], [0]))
        acc = (acc + (1 << (precision - 1))) >> precision
        out[:, xx, :] = np.clip(acc, 0, 255).astype(np.uint8)
    return out


def resize_u8(src, out_w, out_h):
    """``tvF.resize(uint8 image, (out_h, out_w), BICUBIC, antialias=True)`` on an (H, W, C) uint8 array."""
    assert src.dtype == np.uint8 and src.ndim == 3
    in_h, in_w, _ = src.shape
    tmp = src
    if out_w != in_w:
        _, b, k, p = precompute_coeffs(in_w, out_w)
        tmp = _pass_axis1(tmp, b, k, p, out_w)
    if out_h != in_h:
        _, b, k, p = precompute_coeffs(in_h, out_h)
        tmp = _pass_axis1(tmp.transpose(1, 0, 2), b, k, p, out_h).transpose(1, 0, 2)
    return np.ascontiguousarray(tmp)
