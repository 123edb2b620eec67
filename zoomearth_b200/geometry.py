"""Zoom geometry: the host-side mirror of the reference's L3 helpers, evaluated by libzoomvit (C ABI).

Names, argument meaning and error behaviour follow the reference:
  extract_bbox   src/eval/infer.py:20-32   (float parse; demo.py:72-84 is the int-only variant)
  cut_box        src/eval/infer.py:41-76   box that cut_image() crops
  resize_dims    src/eval/infer.py:78-85   size resize_image() produces, and 1/scale
  smart_resize   HF models/qwen2_vl/image_processing_pil_qwen2_vl.py:57-83
"""
import ctypes as C
import math
import re

import numpy as np

from . import _lib

_BBOX_RE = re.compile(r'"bbox_2d"\s*:\s*\[(.*?)\]', re.DOTALL)


def extract_bbox(completion_content, scale, integer_only=False):
    """All ``"bbox_2d": [...]`` lists in the text, each number times ``scale``; unparsable lists are skipped."""
    conv = int if integer_only else float
    bboxes = []
    for m in _BBOX_RE.findall(completion_content):
        try:
            nums = [conv(x.strip()) for x in m.split(",")]
        except ValueError:
            continue
        bboxes.append([n * scale for n in nums])
    return bboxes


def cut_box(img_w, img_h, bbox, min_size=512):
    """The box ``cut_image(image, bbox, min_size)`` crops (infer.py:41-76).  Like the reference's
    ``x1, y1, x2, y2 = map(int, bbox)``: anything but four numbers raises ValueError, a NaN raises ValueError and an
    infinity OverflowError (what ``int()`` raises)."""
    vals = [float(v) for v in bbox]
    if len(vals) != 4:
        raise ValueError(f"{'too many values to unpack (expected 4)' if len(vals) > 4 else f'not enough values to unpack (expected 4, got {len(vals)})'}")
    for v in vals:
        if math.isnan(v):
            raise ValueError("cannot convert float NaN to integer")
        if math.isinf(v):
            raise OverflowError("cannot convert float infinity to integer")
    b = (C.c_double * 4)(*vals)
    out = (C.c_int32 * 4)()
    _lib.check(_lib.lib().zv_cut_box(int(img_w), int(img_h), b, int(min_size), out))
    return tuple(out)


def resize_dims(w, h, max_size=512):
    wh = (C.c_int32 * 2)()
    inv = C.c_double()
    _lib.check(_lib.lib().zv_resize_dims(int(w), int(h), int(max_size), wh, C.byref(inv)))
    return wh[0], wh[1], inv.value


RESIZE_MODE = {"infer": 0, "demo": 0, "sft": 1, "custom": 2}
DEFAULT_MAX_SIZE = {"infer": 512, "demo": 1024, "sft": 1024, "custom": 512}


def resize_dims_ex(w, h, max_size=None, variant="infer"):
    """``resize_image`` at the reference's call sites -> (new_w, new_h, 1/scale).  ``infer`` src/eval/infer.py:78-85 (512),
    ``demo`` src/demo.py:86-93 (1024), ``sft`` src/train/SFT.py:76-81 (1024, always resizes), ``custom``
    open_r1/custom/customized_funcs.py:76-85 (512, scale floored at 30 / min side)."""
    if max_size is None:
        max_size = DEFAULT_MAX_SIZE[variant]
    wh = (C.c_int32 * 2)()
    inv = C.c_double()
    _lib.check(_lib.lib().zv_resize_dims_ex(int(w), int(h), int(max_size), RESIZE_MODE[variant], wh, C.byref(inv)))
    return wh[0], wh[1], inv.value


def cut_ops(img_w, img_h, bbox, min_size=512, variant="infer"):
    """The Pillow operations ``cut_image`` performs at a call site, as ``["crop", box]`` / ``["resize", (w, h)]`` steps:
    ``infer`` / ``demo`` one crop (infer.py:41-76); ``custom`` the same, or nothing at all when ``len(bbox) != 4``
    (customized_funcs.py:38-39); ``sft`` crop, and for boxes with both sides >= min_size a resize to min side = min_size
    plus a centre crop (SFT.py:83-125)."""
    if variant == "custom" and len(bbox) != 4:
        return []
    if variant != "sft":
        return [["crop", list(cut_box(img_w, img_h, bbox, min_size))]]
    cut_box(img_w, img_h, bbox, min_size)                       # same argument checks / errors as the plain rule
    b = (C.c_double * 4)(*[float(v) for v in bbox])
    box, rs, cb = (C.c_int32 * 4)(), (C.c_int32 * 2)(), (C.c_int32 * 4)()
    _lib.check(_lib.lib().zv_cut_box_sft(int(img_w), int(img_h), b, int(min_size), box, rs, cb))
    ops = [["crop", list(box)]]
    if rs[0] > 0:
        ops += [["resize", [rs[0], rs[1]]], ["crop", list(cb)]]
    return ops


def smart_resize(height, width, factor=28, min_pixels=56 * 56, max_pixels=14 * 14 * 4 * 1280):
    out = (C.c_int32 * 2)()
    rc = _lib.lib().zv_smart_resize(int(height), int(width), int(factor), int(min_pixels), int(max_pixels), out)
    if rc == _lib.ZV_EINVAL_ASPECT:
        raise ValueError(_lib.lib().zv_last_error().decode())       # same text HF raises
    _lib.check(rc)
    return out[0], out[1]


def geometry(cfg, img_hw, bboxes=None):
    """Batch form: (n,2) image sizes (h,w) [+ (n,4) boxes] -> crop_box (n,4) i32, resized_hw (n,2) i32, grid_thw (n,3) i64."""
    img_hw = np.ascontiguousarray(img_hw, dtype=np.int32).reshape(-1, 2)
    n = img_hw.shape[0]
    bb = None if bboxes is None else np.ascontiguousarray(bboxes, dtype=np.float64).reshape(n, 4)
    crop = np.empty((n, 4), np.int32)
    rhw = np.empty((n, 2), np.int32)
    grid = np.empty((n, 3), np.int64)
    rc = _lib.lib().zv_geometry(C.byref(cfg), n, img_hw.ctypes.data, None if bb is None else bb.ctypes.data,
                                crop.ctypes.data, rhw.ctypes.data, grid.ctypes.data)
    if rc in (_lib.ZV_EINVAL_ASPECT, _lib.ZV_EINVAL_BOX):
        raise ValueError(_lib.lib().zv_last_error().decode())       # HF / Pillow raise ValueError here
    _lib.check(rc)
    return crop, rhw, grid


def resample_coeffs(in_size, out_size):
    """Pillow bicubic taps for one axis: (ksize, bounds (out,2) i32, kk (out,ksize) i32)."""
    ks = _lib.check(_lib.lib().zv_resample_ksize(int(in_size), int(out_size)))
    bounds = np.empty((out_size, 2), np.int32)
    kk = np.empty((out_size, ks), np.int32)
    _lib.check(_lib.lib().zv_resample_coeffs(int(in_size), int(out_size), bounds.ctypes.data, kk.ctypes.data))
    return ks, bounds, kk


def resample_coeffs_ex(kind, in_size, out_size):
    """The 22-bit taps K1 runs for resample kind ``kind`` (``_lib.RESAMPLE_*``): (ksize, bounds, kk, precision), where
    precision is the axis precision of torchvision's int16 taps (22 for Pillow and same-size axes)."""
    ks = _lib.check(_lib.lib().zv_resample_ksize(int(in_size), int(out_size)))
    bounds = np.empty((out_size, 2), np.int32)
    kk = np.empty((out_size, ks), np.int32)
    p = C.c_int32(0)
    _lib.check(_lib.lib().zv_resample_coeffs_ex(int(kind), int(in_size), int(out_size), bounds.ctypes.data, kk.ctypes.data,
                                                C.byref(p)))
    return ks, bounds, kk, p.value


def normalize_lut(cfg):
    lut = np.empty((3, 256), np.float32)
    _lib.check(_lib.lib().zv_normalize_lut(C.byref(cfg), lut.ctypes.data))
    return lut
