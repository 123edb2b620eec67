"""LM hand-off on the device, host side (no GPU needed): the new exports, the argument errors every device entry point
returns before any device work, and the error texts ``DeviceHandoff.check()`` rebuilds from a device status word."""
import ctypes as C
import subprocess

import numpy as np
import pytest
import torch

from zoomearth_b200 import _lib

IMG, VID, VSTART, VEND = 151655, 151656, 151652, 151653
NEW = ("zv_handoff_workspace_bytes", "zv_rope_index_dev", "zv_placeholder_rows_dev")

# host inputs on which zv_rope_index fails -> the status the device path records: (check, sample, detail a, detail b)
ERROR_CASES = [
    ("video", [[VSTART, VID, VEND]], None, [[1, 4, 4]], (1, 0, 0, 0)),
    ("trailing vision start", [[5, VSTART]], None, [[1, 4, 4]], (2, 0, 0, 0)),
    ("fewer placeholders", [[1, VSTART, IMG, VEND, 2, 3], [VSTART, IMG, VSTART, IMG, 7, 8]],
     [[1, 1, 1, 1, 1, 1], [1, 1, 1, 1, 1, 1]], [[1, 2, 2], [1, 4, 4], [1, 2, 2]], (3, 1, 0, 0)),
    ("grid rows", [[VSTART, IMG, VEND, VSTART, IMG, VEND]], None, [[1, 2, 2]], (4, 0, 1, 0)),
    ("empty grid", [[VSTART, IMG, VEND, 4], [VSTART, IMG, VEND, 4]], None, [[1, 2, 2], [1, 1, 4]], (5, 1, 1, 0)),
    ("count", [[5, VSTART, IMG, IMG, IMG, IMG, VEND, 7]], None, [[1, 8, 8]], (6, 0, 18, 8)),
    ("fully masked", [[VSTART, IMG, VEND, 3], [1, 2, 3, 4]], [[1, 1, 1, 1], [0, 0, 0, 0]], [[1, 2, 2]], (7, 1, 0, 0)),
    # the lowest sample wins, whatever its check: sample 1 (count) before sample 2 (video)
    ("lowest sample", [[VSTART, IMG, VEND, 1], [VSTART, IMG, IMG, VEND], [VSTART, VID, VEND, 1]], None,
     [[1, 2, 2], [1, 4, 4]], (6, 1, 5, 4)),
]


def test_new_exports_are_bound_and_exported(lib):
    from zoomearth_b200 import build
    for name in NEW:
        assert name in _lib.EXPORTS and hasattr(lib, name)
    out = subprocess.run(["nm", "-D", "--defined-only", build.LIB], capture_output=True, text=True, check=True).stdout
    syms = {line.split()[-1] for line in out.splitlines() if " T " in line}
    assert set(NEW) <= syms
    assert {s for s in syms if s.startswith("zv_")} == set(_lib.EXPORTS)


def _buf(n=1 << 16):
    b = (C.c_uint8 * n)()
    return C.addressof(b), b


def test_workspace_query(lib):
    assert lib.zv_handoff_workspace_bytes(64, 2048) > 64 * 2048
    assert lib.zv_handoff_workspace_bytes(64, 2048) <= lib.zv_handoff_workspace_bytes(64, 4096)
    for b, l in ((0, 8), (8, 0), (-1, 8)):
        assert lib.zv_handoff_workspace_bytes(b, l) == _lib.ZV_EINVAL
        assert b"zv_handoff_workspace_bytes" in lib.zv_last_error()


def test_rope_index_dev_argument_errors(lib):
    p, keep = _buf()
    ws = lib.zv_handoff_workspace_bytes(2, 16)

    def call(ids=p, batch=2, seq_len=16, merge=2, pos=p, deltas=p, status=p, work=p, work_bytes=ws):
        return lib.zv_rope_index_dev(ids, None, batch, seq_len, p, 1, IMG, VID, VSTART, merge, 0, pos, deltas, status, work,
                                     work_bytes, None)

    for kw, text in [(dict(ids=None), b"null argument"), (dict(pos=None), b"null argument"),
                     (dict(deltas=None), b"null argument"), (dict(status=None), b"null argument"),
                     (dict(work=None), b"null argument"), (dict(batch=0), b"batch=0"), (dict(seq_len=0), b"seq_len=0"),
                     (dict(merge=0), b"merge=0"), (dict(batch=-3), b"batch=-3"),
                     (dict(work_bytes=ws - 1), b"workspace")]:
        assert call(**kw) == _lib.ZV_EINVAL, kw
        err = lib.zv_last_error()
        assert err.startswith(b"zv_rope_index_dev: ") and text in err, (kw, err)
    if not torch.cuda.is_available():
        assert call() == _lib.ZV_ENODEV            # valid arguments reach the device check: there is no CPU path


def test_placeholder_rows_dev_argument_errors(lib):
    p, keep = _buf()
    ws = lib.zv_handoff_workspace_bytes(1, 100000)

    def call(ids=p, n_tokens=100000, rows=p, cap=10, status=p, work=p, work_bytes=ws):
        return lib.zv_placeholder_rows_dev(ids, n_tokens, IMG, rows, cap, status, work, work_bytes, None)

    for kw, text in [(dict(ids=None), b"null argument"), (dict(rows=None), b"null argument"),
                     (dict(status=None), b"null argument"), (dict(work=None), b"null argument"),
                     (dict(n_tokens=0), b"n_tokens=0"), (dict(cap=-1), b"rows_cap=-1"),
                     (dict(work_bytes=0), b"workspace")]:
        assert call(**kw) == _lib.ZV_EINVAL, kw
        err = lib.zv_last_error()
        assert err.startswith(b"zv_placeholder_rows_dev: ") and text in err, (kw, err)
    if not torch.cuda.is_available():
        assert call() == _lib.ZV_ENODEV


@pytest.mark.parametrize("case", ERROR_CASES, ids=[c[0] for c in ERROR_CASES])
def test_check_messages_equal_the_host_messages(lib, case):
    """The text check() builds from a device status is the host function's text for the same input."""
    from zoomearth_b200 import get_rope_index
    from zoomearth_b200.handoff import _ROPE_ERRORS
    _, ids, mask, grid, (code, sample, a, b) = case
    with pytest.raises(_lib.ZoomVitError) as host:
        get_rope_index(torch.tensor(ids), torch.tensor(grid), None, None if mask is None else torch.tensor(mask))
    assert host.value.code == _lib.ZV_EINVAL
    assert host.value.msg == _ROPE_ERRORS[code].format(s=sample, a=a, b=b)


def test_device_handoff_refuses_video_like_the_host():
    from zoomearth_b200.handoff import DeviceHandoff
    dh = DeviceHandoff.__new__(DeviceHandoff)
    with pytest.raises(NotImplementedError):
        dh.rope_index(torch.zeros(1, 4, dtype=torch.int64), np.array([[1, 2, 2]]), video_grid_thw=torch.tensor([[1, 2, 2]]))
