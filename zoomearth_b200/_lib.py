"""ctypes binding of ``libzoomvit.so`` (the C ABI declared in ``include/zoomvit.h``).

There is no fallback: if the shared object is missing this module raises at import of the first symbol,
and every device entry point returns an error when no sm_100 GPU is current.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzoomvit.so")

ZV_F32, ZV_BF16, ZV_F16 = 0, 1, 2
ORDER_HF, ORDER_WINDOW = 0, 1
TOWER_QWEN25, TOWER_QWEN2 = 0, 1
RESAMPLE_PIL, RESAMPLE_TORCHVISION = 0, 1
ZV_EINVAL, ZV_EINVAL_ASPECT, ZV_EINVAL_BOX, ZV_ENOMEM, ZV_ECUDA, ZV_ENODEV, ZV_EARCH = -1, -2, -3, -4, -5, -6, -7


class ZvCfg(C.Structure):
    _fields_ = [
        ("patch", C.c_int32), ("merge", C.c_int32), ("temporal", C.c_int32), ("window", C.c_int32),
        ("min_size", C.c_int32), ("depth", C.c_int32), ("hidden", C.c_int32), ("heads", C.c_int32),
        ("inter", C.c_int32), ("out_hidden", C.c_int32), ("fullatt_mask_lo", C.c_int32), ("op_dtype", C.c_int32),
        ("min_pixels", C.c_int64), ("max_pixels", C.c_int64), ("rescale", C.c_double),
        ("mean", C.c_float * 3), ("std", C.c_float * 3), ("eps", C.c_float), ("reserved_f", C.c_float),
        ("tower_kind", C.c_int32), ("resample_kind", C.c_int32),
    ]


class ZvTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int32), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 5)]


class ZoomVitError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libzoomvit error {code}: {msg}")
        self.code = code
        self.msg = msg


_P = C.POINTER
_PROTOS = {
    "zv_version": (C.c_char_p, []),
    "zv_last_error": (C.c_char_p, []),
    "zv_default_cfg": (None, [_P(ZvCfg)]),
    "zv_cut_box": (C.c_int, [C.c_int32, C.c_int32, _P(C.c_double), C.c_int32, _P(C.c_int32)]),
    "zv_resize_dims": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P(C.c_int32), _P(C.c_double)]),
    "zv_resize_dims_ex": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P(C.c_int32), _P(C.c_double)]),
    "zv_cut_box_sft": (C.c_int, [C.c_int32, C.c_int32, _P(C.c_double), C.c_int32, _P(C.c_int32), _P(C.c_int32), _P(C.c_int32)]),
    "zv_resize_u8_workspace_bytes": (C.c_int64, [C.c_int32, C.c_void_p, C.c_void_p]),
    "zv_resize_u8": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_smart_resize": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P(C.c_int32)]),
    "zv_geometry": (C.c_int, [_P(ZvCfg), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zv_resample_ksize": (C.c_int32, [C.c_int32, C.c_int32]),
    "zv_resample_coeffs": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "zv_resample_coeffs_ex": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, _P(C.c_int32)]),
    "zv_normalize_lut": (C.c_int, [_P(ZvCfg), C.c_void_p]),
    "zv_preprocess_workspace_bytes": (C.c_int64, [C.c_int32, C.c_void_p, C.c_void_p]),
    "zv_preprocess": (C.c_int, [_P(ZvCfg), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_debug_k1_tc_host": (C.c_int, [_P(ZvCfg), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_plan_create": (C.c_int, [_P(ZvCfg), C.c_int32, C.c_void_p, _P(C.c_void_p)]),
    "zv_plan_free": (None, [C.c_void_p]),
    "zv_plan_num_patches": (C.c_int64, [C.c_void_p]),
    "zv_plan_num_tokens": (C.c_int64, [C.c_void_p]),
    "zv_plan_window_index": (_P(C.c_int64), [C.c_void_p]),
    "zv_plan_reverse_index": (_P(C.c_int64), [C.c_void_p]),
    "zv_plan_cu_window": (_P(C.c_int32), [C.c_void_p, _P(C.c_int32)]),
    "zv_plan_cu_window_raw": (_P(C.c_int32), [C.c_void_p, _P(C.c_int32)]),
    "zv_plan_cu_full": (_P(C.c_int32), [C.c_void_p, _P(C.c_int32)]),
    "zv_plan_pos_ids": (_P(C.c_int32), [C.c_void_p]),
    "zv_plan_device_bytes": (C.c_int64, [C.c_void_p]),
    "zv_plan_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_weights_bytes": (C.c_int64, [_P(ZvCfg)]),
    "zv_weights_pack": (C.c_int, [_P(ZvCfg), _P(ZvTensor), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_visual_workspace_bytes": (C.c_int64, [_P(ZvCfg), C.c_void_p]),
    "zv_visual_forward": (C.c_int, [_P(ZvCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_visual_forward_gather": (C.c_int, [_P(ZvCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int64,
                                           C.c_void_p]),
    "zv_visual_forward_gather_rows": (C.c_int, [_P(ZvCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                                C.c_int32, C.c_void_p]),
    "zv_visual_forward_into": (C.c_int, [_P(ZvCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                         C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zv_rope_index": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_int64,
                                C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "zv_placeholder_rows": (C.c_int64, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64]),
    "zv_last_launch_count": (C.c_int64, []),
    "zv_timing_enable": (None, [C.c_int]),
    "zv_timing_reset": (None, []),
    "zv_timing_read": (C.c_int, [C.c_int, _P(C.c_double), _P(C.c_int64)]),
    "zv_gemm_bf16": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                               C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "zv_gemm_ex": (C.c_int, [C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                             C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                             C.c_int32, C.c_void_p]),
    "zv_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                               C.c_int64, C.c_int32, C.c_void_p]),
}
EXPORTS = tuple(_PROTOS)
_lib = None


def lib():
    """The loaded library; raises (loudly) if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: run `python -m zoomearth_b200.build` (nvcc, sm_100a). "
                "zoomearth_b200 has no CPU or PyTorch fallback path.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    """Raise for a negative return code; pass non-negative values (sizes) through."""
    if rc is not None and rc < 0:
        raise ZoomVitError(rc, lib().zv_last_error().decode())
    return rc


def default_cfg(**overrides):
    cfg = ZvCfg()
    lib().zv_default_cfg(C.byref(cfg))
    for k, v in overrides.items():
        if k in ("mean", "std"):
            setattr(cfg, k, (C.c_float * 3)(*v))
        elif k == "fullatt":
            m = 0
            for i in v:
                m |= 1 << i
            cfg.fullatt_mask_lo = m - (1 << 32) if m >= (1 << 31) else m
        else:
            setattr(cfg, k, v)
    return cfg
