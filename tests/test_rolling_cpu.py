"""CPU checks of the rolling-median background (cvvp_median_rolling_device, cvvp_highlight_device_bg,
cvvp_highlight_rolling_*, TrackObjects' kwargs["cvvp_background_window"]): exported and bound, null contexts rejected,
bad windows refused before any device work, and the kernel compiles for sm_100a without spills."""
import ctypes
import re
import shutil
import subprocess

import numpy as np
import pytest

import cvvidproc_b200 as cvp
from cvvidproc_b200 import _cabi

NEW_SYMBOLS = ["cvvp_median_rolling_device", "cvvp_highlight_device_bg", "cvvp_highlight_rolling_begin",
               "cvvp_highlight_rolling_push", "cvvp_highlight_rolling_close", "cvvp_highlight_rolling_pending",
               "cvvp_highlight_rolling_ready", "cvvp_highlight_rolling_next", "cvvp_highlight_rolling_end"]


def test_new_symbols_are_declared_exported_and_bound():
    lib = _cabi.load()
    raw = ctypes.CDLL(str(_cabi.LIB_PATH))
    declared = set(_cabi.declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared
        assert hasattr(raw, name)
        assert name in _cabi.BOUND_SYMBOLS
        assert getattr(lib, name).argtypes is not None


def test_null_context_calls_are_rejected():
    lib = _cabi.load()
    assert lib.cvvp_median_rolling_device(None, None, 10, 100, 128, 5, 0, 10, None, 128, None) == -1
    assert lib.cvvp_highlight_device_bg(None, None, 1, 16, None, 0, None, 16, None, 0, None, None, 0, None) == -1
    assert lib.cvvp_highlight_rolling_begin(None, 5, 4, None, 0, 0) == -1
    assert lib.cvvp_highlight_rolling_push(None, None, 1, 16) == -1
    assert lib.cvvp_highlight_rolling_close(None) == -1
    assert lib.cvvp_highlight_rolling_ready(None) == -1
    first, n = ctypes.c_longlong(), ctypes.c_longlong()
    assert lib.cvvp_highlight_rolling_next(None, None, 16, 1, ctypes.byref(first), ctypes.byref(n), None, None, None, 0) == -1
    assert lib.cvvp_highlight_rolling_end(None) == -1
    assert lib.cvvp_highlight_rolling_pending(None) == 0
    assert b"null context" in lib.cvvp_last_error(None)


def _pack(kwargs):
    hp = cvp.HighlightObjectsPack(np.zeros((4, 4), np.uint8), np.ones((2, 2), np.uint8), 1, 1, 1, 1, 1, 1)
    ap = cvp.AssignObjectsPack(lambda **kw: 0, kwargs)
    return cvp.VidObjectTrackPack("/nonexistent/video.mp4", hp, ap)


@pytest.mark.parametrize("window", [0, -3, 70000, "x", 2.5, True, None])
def test_track_objects_refuses_a_bad_window_before_any_device_work(window):
    # a missing video makes TrackObjects return {} without raising: the window is checked before that, before any
    # device work
    with pytest.raises(RuntimeError, match="cvvp_background_window"):
        cvp.TrackObjects(_pack({"cvvp_background_window": window}))


@pytest.mark.parametrize("window", [1, 61, 65535, np.int64(16)])
def test_track_objects_accepts_a_good_window(window, capfd):
    assert cvp.TrackObjects(_pack({"cvvp_background_window": window})) == {}
    assert "Video file not detected" in capfd.readouterr().err


def test_rolling_median_kernel_has_no_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not shutil.os.path.exists(nvcc):
        pytest.skip("no nvcc")
    from cvvidproc_b200 import build

    src = build.CSRC / "median_roll.cu"
    proc = subprocess.run([nvcc, "-c", *build.NVCC_FLAGS, "-I", str(build.REPO / "include"), "-o", str(tmp_path / "r.o"),
                           str(src)], capture_output=True, text=True, check=True)
    log = proc.stdout + proc.stderr
    assert "median_roll_kernel" in log
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", log)
    assert spills and all(s == ("0", "0") for s in spills), log
