"""GPU end-to-end tests of colour frames through the Python surface (TrackObjects' kwargs["cvvp_color"]) on a lossless
colour video whose disks have the background's RGB2GRAY value: in grey they are invisible, in colour they are found,
and the masks equal the host chain (decoded frames -> the colour d of tests/color_cases.py -> the cv2 restatement's
steps) with a static background and a rolling one, on two operators of one device, in small batches, with host-side
frame preparation, and with labels and statistics."""
import dataclasses

import cv2
import numpy as np
import pytest

import color_cases as cc
import cvvidproc_b200 as cvp
import video_util
from oracle import highlight_oracle as ho
from test_track_percentile_gpu import percentile

pytestmark = pytest.mark.gpu

N, H, W = 30, 96, 160
BG = (100, 100, 100)  # channel order as decoded


def _gray(c):
    """OpenCV's 8-bit RGB2GRAY of one pixel (channel 0 first in memory)"""
    return (c[0] * 9798 + c[1] * 19235 + c[2] * 3735 + 16384) >> 15


def _isoluminant():
    """a colour far from BG with BG's grey value"""
    for c1 in range(256):
        c = (190, c1, 40)
        if _gray(c) == _gray(BG):
            return c
    raise AssertionError("no isoluminant colour")


@pytest.fixture(scope="module")
def color_video(tmp_path_factory):
    disk = _isoluminant()
    frames = np.empty((N, H, W, 3), np.uint8)
    frames[:] = BG
    yy, xx = np.mgrid[:H, :W]
    for t in range(N):
        for k, (x0, y0, r) in enumerate(((20, 30, 9), (80, 60, 12), (130, 20, 7))):
            cx = (x0 + 3 * t * (k + 1)) % W
            frames[t][(xx - cx) ** 2 + (yy - y0) ** 2 <= r * r] = disk
    path = video_util.write_lossless(tmp_path_factory.mktemp("v") / "isoluminant.avi", frames)
    decoded = video_util.read_all(path)
    assert decoded.shape == frames.shape
    gray = np.stack([cv2.cvtColor(f, cv2.COLOR_RGB2GRAY) for f in decoded])
    assert np.ptp(gray) == 0  # the disks vanish in grey
    return path, decoded


def _params(bg):
    p = ho.canonical_params(bg[..., 0].copy() if bg.ndim == 3 else bg)
    return dataclasses.replace(p, background=np.ascontiguousarray(bg))


def _masks(path, p, kwargs, **pack):
    seen = {}

    def cb(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs, components=None):
        seen[frames_processed] = (np.array(bw_frame, copy=True), components)
        return next_ID

    hp = cvp.HighlightObjectsPack(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                  p.min_size_hyst, p.min_size_threshold, p.width_border)
    cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(cb, kwargs), **pack))
    assert sorted(seen) == list(range(N))
    return np.stack([seen[t][0] for t in range(N)]), [seen[t][1] for t in range(N)]


def _host(decoded, p, window=None):
    if window is None:
        return cc.masks(decoded, p, "dark")
    out = []
    weff = min(window, N)
    for t in range(N):
        s = min(max(t - window // 2, 0), N - weff)
        out.append(cc.highlight_objects(decoded[t], dataclasses.replace(p, background=percentile(decoded[s:s + weff], 50)),
                                        "dark"))
    return np.stack(out)


def test_grey_misses_the_disks_and_colour_finds_them(color_video, monkeypatch):
    path, decoded = color_video
    grey_bg = np.full((H, W), _gray(BG), np.uint8)
    grey, _ = _masks(path, _params(grey_bg), {}, grayscale=True)
    assert not grey.any()
    p = _params(percentile(decoded, 50))
    want = _host(decoded, p)
    assert all(want[t].any() for t in range(N))
    got, _ = _masks(path, p, {"cvvp_color": True})
    assert np.array_equal(got, want)


@pytest.mark.parametrize("env", [{"CVVP_TRACK_BATCH": "4"}, {"CVVP_DEVICES": "0,0", "CVVP_TRACK_BATCH": "3"},
                                 {"CVVP_HOST_PREP": "1", "CVVP_TRACK_BATCH": "5"}])
def test_static_background_switches(color_video, monkeypatch, env):
    path, decoded = color_video
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    p = _params(percentile(decoded, 50))
    got, _ = _masks(path, p, {"cvvp_color": True, "cvvp_polarity": "both"})
    assert np.array_equal(got, cc.masks(decoded, p, "both"))


@pytest.mark.parametrize("host_prep", [False, True])
def test_rolling_background(color_video, monkeypatch, host_prep):
    path, decoded = color_video
    monkeypatch.setenv("CVVP_TRACK_BATCH", "4")
    if host_prep:
        monkeypatch.setenv("CVVP_HOST_PREP", "1")
    p = _params(np.zeros((H, W, 3), np.uint8))
    got, _ = _masks(path, p, {"cvvp_color": True, "cvvp_background_window": 9})
    want = _host(decoded, p, 9)
    assert want.any()
    assert np.array_equal(got, want)


def test_labels_and_statistics(color_video, monkeypatch):
    path, decoded = color_video
    monkeypatch.setenv("CVVP_TRACK_BATCH", "6")
    p = _params(percentile(decoded, 50))
    kwargs = {"cvvp_color": True, "cvvp_components": True, "cvvp_labels": True, "cvvp_component_stats": True}
    got, comps = _masks(path, p, kwargs)
    want = cc.masks(decoded, p, "dark")
    assert np.array_equal(got, want)
    for t in range(N):
        n_cv, lab_cv = cv2.connectedComponents(want[t], connectivity=8)
        assert comps[t]["count"] == n_cv - 1
        assert np.array_equal(comps[t]["labels"] != 0, want[t] != 0)
        d = cc.color_difference(p.background, decoded[t], "dark").astype(np.int64)
        assert comps[t]["mass"].sum() == d[want[t] != 0].sum()


def test_background_channels_must_match(color_video):
    path, decoded = color_video
    for bg in (percentile(decoded, 50)[..., :2].copy(), percentile(decoded, 50)[..., 0].copy()):
        with pytest.raises(RuntimeError, match="cvvp_color"):
            _masks(path, _params(bg), {"cvvp_color": True})
