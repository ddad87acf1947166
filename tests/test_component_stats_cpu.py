"""CPU checks of the component statistics (cvvp_component_stats, cvvp_highlight_set_component_stats, TrackObjects'
kwargs["cvvp_component_stats"]): the header's record compiles as strict C99 with the documented layout and the numpy
dtype matches it; the new symbols are declared, exported and bound and reject a null context; the numpy reference that
the GPU tests hold every record to agrees with cv2.moments and with the polarity references' difference image on
random masks; and TrackObjects refuses a malformed key before any device work."""
import ctypes
import shutil
import subprocess

import cv2
import numpy as np
import pytest

import cvvidproc_b200 as cvp
import polarity_cases as pc
from cvvidproc_b200 import _cabi

NEW_SYMBOLS = ["cvvp_highlight_set_component_stats", "cvvp_highlight_component_stats"]
STATS_FIELDS = ["sum_xx", "sum_xy", "sum_yy", "sum_d", "sum_dx", "sum_dy", "min_d", "max_d"]


def reference_stats(labels, frame, background, polarity, max_comps=None):
    """records (COMPONENT_STATS_DTYPE) of the components of an int32 label image (0 = background, k = component k,
    numbered 1..K), with d the polarity's difference image of frame and background"""
    d = pc.difference_image(background, frame, polarity).astype(np.int64)
    k_max = int(labels.max())
    if max_comps is not None:
        k_max = min(k_max, max_comps)
    out = np.zeros(k_max, _cabi.Context.COMPONENT_STATS_DTYPE)
    for k in range(1, k_max + 1):
        ys, xs = np.nonzero(labels == k)
        xs, ys = xs.astype(np.int64), ys.astype(np.int64)
        dk = d[ys, xs]
        r = out[k - 1]
        c = r["c"]
        c["x0"], c["y0"], c["x1"], c["y1"] = xs.min(), ys.min(), xs.max(), ys.max()
        c["area"] = len(xs)
        c["first_x"], c["first_y"] = xs[0], ys[0]  # np.nonzero is in raster order
        c["sum_x"], c["sum_y"] = xs.sum(), ys.sum()
        out[k - 1]["c"] = c
        out[k - 1]["sum_xx"] = (xs * xs).sum()
        out[k - 1]["sum_xy"] = (xs * ys).sum()
        out[k - 1]["sum_yy"] = (ys * ys).sum()
        out[k - 1]["sum_d"] = dk.sum()
        out[k - 1]["sum_dx"] = (dk * xs).sum()
        out[k - 1]["sum_dy"] = (dk * ys).sum()
        out[k - 1]["min_d"] = dk.min()
        out[k - 1]["max_d"] = dk.max()
    return out


def canonical_labels(mask):
    """8-connected components of a mask numbered in the raster order of their first pixels (the library's numbering)"""
    n, lab = cv2.connectedComponents((mask != 0).astype(np.uint8), connectivity=8, ltype=cv2.CV_32S)
    first = {}
    for idx, v in enumerate(lab.ravel()):
        if v and v not in first:
            first[v] = idx
    order = sorted(first, key=first.get)
    remap = np.zeros(n, np.int32)
    for new, old in enumerate(order, 1):
        remap[old] = new
    return remap[lab]


def test_record_layout_in_c99(tmp_path):
    gcc = shutil.which("gcc") or shutil.which("cc")
    if gcc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "t_stats.c"
    fields = ["c"] + STATS_FIELDS
    src.write_text(
        '#include "cvvp.h"\n#include <stddef.h>\n#include <stdio.h>\n'
        "int main(void) {\n"
        '    printf("%zu", sizeof(cvvp_component_stats));\n'
        + "".join(f'    printf(" %zu", offsetof(cvvp_component_stats, {f}));\n' for f in fields)
        + '    printf("\\n");\n'
        "    return cvvp_highlight_set_component_stats(NULL, 1) == CVVP_ERR_INVALID &&\n"
        "           cvvp_highlight_component_stats(NULL) == CVVP_ERR_INVALID ? 0 : 1;\n"
        "}\n")
    exe = tmp_path / "t_stats"
    lib_dir = _cabi.LIB_PATH.parent
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", str(_cabi.HEADER.parent), str(src),
                    "-L", str(lib_dir), "-lcvvp_cuda", f"-Wl,-rpath,{lib_dir}", "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out == [104, 0, 48, 56, 64, 72, 80, 88, 96, 100]
    dt = _cabi.Context.COMPONENT_STATS_DTYPE
    assert dt.itemsize == out[0]
    assert [dt.fields[f][1] for f in fields] == out[1:]
    assert dt["c"] == _cabi.Context.COMPONENT_DTYPE


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
    for on in (0, 1, 2, -1):
        assert lib.cvvp_highlight_set_component_stats(None, on) == -1
    assert lib.cvvp_highlight_component_stats(None) == -1
    assert b"null context" in lib.cvvp_last_error(None)


@pytest.mark.parametrize("seed", range(12))
@pytest.mark.parametrize("polarity", ["dark", "bright", "both"])
def test_reference_against_cv2_moments_and_the_difference_image(seed, polarity):
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(5, 60)), int(rng.integers(5, 70))
    mask = (rng.random((h, w)) < rng.uniform(0.05, 0.6)).astype(np.uint8) * 255
    frame = rng.integers(0, 256, (h, w), dtype=np.uint8)
    bg = rng.integers(0, 256, (h, w), dtype=np.uint8)
    lab = canonical_labels(mask)
    recs = reference_stats(lab, frame, bg, polarity)
    d = pc.difference_image(bg, frame, polarity).astype(np.float64)
    assert len(recs) == lab.max()
    for k, r in enumerate(recs, 1):
        comp = (lab == k).astype(np.uint8)
        m = cv2.moments(comp, binaryImage=True)
        assert (r["sum_xx"], r["sum_xy"], r["sum_yy"]) == (m["m20"], m["m11"], m["m02"])
        assert (r["c"]["sum_x"], r["c"]["sum_y"], r["c"]["area"]) == (m["m10"], m["m01"], m["m00"])
        # the contrast sums are the moments of d restricted to the component
        md = cv2.moments(d * comp, binaryImage=False)
        assert (r["sum_d"], r["sum_dx"], r["sum_dy"]) == (round(md["m00"]), round(md["m10"]), round(md["m01"]))
        assert (r["min_d"], r["max_d"]) == (d[comp != 0].min(), d[comp != 0].max())
    assert np.array_equal(reference_stats(lab, frame, bg, polarity, max_comps=2), recs[:2])


def test_reference_of_an_all_foreground_frame_with_zero_contrast():
    frame = np.full((9, 13), 77, np.uint8)
    lab = np.ones(frame.shape, np.int32)
    r = reference_stats(lab, frame, frame, "dark")[0]
    assert r["sum_d"] == r["sum_dx"] == r["sum_dy"] == r["min_d"] == r["max_d"] == 0
    xs, ys = np.meshgrid(np.arange(13), np.arange(9))
    assert r["sum_xx"] == (xs * xs).sum() and r["sum_xy"] == (xs * ys).sum() and r["sum_yy"] == (ys * ys).sum()


# ---------------------------------------------------------------------------------------------------------------------
# TrackObjects' kwargs["cvvp_component_stats"]

def _pack(kwargs):
    hp = cvp.HighlightObjectsPack(np.zeros((4, 4), np.uint8), np.ones((2, 2), np.uint8), 1, 1, 1, 1, 1, 1)
    ap = cvp.AssignObjectsPack(lambda **kw: 0, kwargs)
    return cvp.VidObjectTrackPack("/nonexistent/video.mp4", hp, ap)


@pytest.mark.parametrize("kwargs", [
    {"cvvp_component_stats": True},
    {"cvvp_component_stats": True, "cvvp_components": False},
    {"cvvp_component_stats": 1, "cvvp_components": True},
    {"cvvp_component_stats": "yes", "cvvp_components": True},
    {"cvvp_component_stats": None, "cvvp_components": True},
])
def test_track_objects_refuses_a_bad_stats_key_before_any_device_work(kwargs):
    # a missing video makes TrackObjects return {} without raising: the key is checked before that
    with pytest.raises(RuntimeError, match="cvvp_component_stats"):
        cvp.TrackObjects(_pack(kwargs))


@pytest.mark.parametrize("kwargs", [
    {"cvvp_component_stats": True, "cvvp_components": True},
    {"cvvp_component_stats": False},
    {"cvvp_component_stats": True, "cvvp_components": True, "cvvp_polarity": "bright", "cvvp_background_window": 5},
])
def test_track_objects_accepts_a_good_stats_key(kwargs, capfd):
    before = dict(kwargs)
    assert cvp.TrackObjects(_pack(kwargs)) == {}
    assert "Video file not detected" in capfd.readouterr().err
    assert kwargs == before
