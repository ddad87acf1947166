"""GPU end-to-end tests of percentile backgrounds through the Python surface on lossless videos:
GetVideoBackground(bg_algo="cvvp_percentile:P") against numpy over the decoded frames, and TrackObjects with
kwargs["cvvp_background_percentile"] = P against the host chain of test_track_rolling_gpu.py with the window's
percentile in place of its median -- including the case the option exists for, a dark object that sits still for most of
every window, which the median background swallows and a high percentile keeps."""
import dataclasses

import numpy as np
import pytest

import cvvidproc_b200 as cvp
import video_util
from cvvidproc_b200 import synth
from oracle import highlight_oracle as ho
from test_track_rolling_gpu import _count_tracker, _drift, _track, _tracker

pytestmark = pytest.mark.gpu

N = 60


def percentile(stack, p):
    k = min(stack.shape[0] - 1, stack.shape[0] * p // 100)
    return np.partition(stack, k, axis=0)[k]


def host_chain(frames, p, w, pct, kwargs):
    """decoded frames -> each frame's window percentile -> the cv2 restatement of HighlightObjects -> the tracker"""
    n = frames.shape[0]
    weff = min(w, n)
    prev, archive, nid, cache = {}, {}, 0, {}
    for t in range(n):
        s = min(max(t - w // 2, 0), n - weff)
        if s not in cache:
            cache[s] = percentile(frames[s : s + weff], pct)
        bw = ho.highlight_objects(frames[t].copy(), dataclasses.replace(p, background=cache[s]))
        track = _count_tracker if kwargs.get("cvvp_components") else _tracker
        nid = track(bw, t, prev, archive, nid, kwargs)
    return archive


@pytest.fixture(scope="module")
def drift_video(tmp_path_factory):
    frames = _drift(synth.synth_frames(0, N, 160, 96, 7, 8))
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "drift.avi", frames), frames


@pytest.fixture(scope="module")
def colour_video(tmp_path_factory):
    g = synth.synth_frames(0, 40, 96, 64, 11, 6)
    frames = _drift(np.stack([g, np.roll(g, 3, axis=2), 255 - g], axis=-1), 0.8)
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "colour.avi", frames), frames


# a still dark square, present in 7 of every 10 frames: 70 % of any window of 10, 20, ... frames
SQUARE = (slice(30, 50), slice(60, 90))


def _present(t):
    return t % 10 < 7


@pytest.fixture(scope="module")
def settled_video(tmp_path_factory):
    frames = _drift(synth.synth_frames(0, N, 160, 96, 23, 1))
    for t in range(N):
        if _present(t):
            frames[(t,) + SQUARE] = 12
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "settled.avi", frames), frames


# ---- GetVideoBackground ----------------------------------------------------------------------------------------------
def _bg(path, algo, **pack):
    return cvp.GetVideoBackground(cvp.VidBgPack(path, bg_algo=algo, **pack))


@pytest.mark.parametrize("p", [0, 1, 10, 49, 50, 51, 90, 99, 100])
def test_background_grey_colour_crop_and_frame_limit(drift_video, colour_video, p):
    path, frames = drift_video
    assert np.array_equal(_bg(path, f"cvvp_percentile:{p}", vid_is_grayscale=True), percentile(frames, p))
    assert np.array_equal(_bg(path, f"cvvp_percentile:{p}", vid_is_grayscale=True, frame_limit=25),
                          percentile(frames[:25], p))
    cpath, _ = colour_video
    decoded = video_util.read_all(cpath)
    assert np.array_equal(_bg(cpath, f"cvvp_percentile:{p}"), percentile(decoded, p))
    x, y, w, h = 5, 7, 50, 30
    got = _bg(cpath, f"cvvp_percentile:{p}", crop_x=x, crop_y=y, crop_width=w, crop_height=h)
    assert np.array_equal(got, percentile(decoded[:, y : y + h, x : x + w], p))


@pytest.mark.parametrize("p", [0, 25, 50, 90, 100])
def test_background_on_two_devices(drift_video, monkeypatch, p):
    path, frames = drift_video
    monkeypatch.setenv("CVVP_DEVICES", "0,0")
    assert np.array_equal(_bg(path, f"cvvp_percentile:{p}", vid_is_grayscale=True), percentile(frames, p))


def test_percentile_50_is_hist_with_the_same_report(drift_video, capfd):
    path, _ = drift_video
    hist = _bg(path, "hist", vid_is_grayscale=True, print_timing_report=True)
    out_hist = capfd.readouterr().out
    p50 = _bg(path, "cvvp_percentile:50", vid_is_grayscale=True, print_timing_report=True)
    out_p50 = capfd.readouterr().out
    assert np.array_equal(hist, p50)
    strip = lambda s: [line.split(":")[0] for line in s.splitlines()]
    assert out_p50.splitlines()[0] == out_hist.splitlines()[0]  # the info line
    assert strip(out_p50) == strip(out_hist) and "Batch gen" in out_p50


# ---- TrackObjects with a rolling percentile background ---------------------------------------------------------------
@pytest.mark.parametrize("w,batch,pct", [(5, 1, 90), (5, 3, 0), (16, 7, 75), (16, 1, 25), (16, 3, 100), (61, 7, 90)])
def test_rolling_percentile_archive_equals_the_host_chain(drift_video, monkeypatch, w, batch, pct):
    monkeypatch.setenv("CVVP_TRACK_BATCH", str(batch))
    path, frames = drift_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"min_area": 5, "cvvp_background_window": w, "cvvp_background_percentile": pct}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    assert got == host_chain(frames, p, w, pct, {"min_area": 5})


@pytest.mark.parametrize("labels", [False, True])
def test_components_compose(drift_video, monkeypatch, labels):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "5")
    path, frames = drift_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"min_area": 5, "cvvp_background_window": 16, "cvvp_background_percentile": 80, "cvvp_components": True,
              "cvvp_labels": labels}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    assert got == host_chain(frames, p, 16, 80, {"min_area": 5, "cvvp_components": True})


@pytest.mark.parametrize("pct", [10, 50, 90])
def test_window_covering_the_video_equals_the_static_path(drift_video, monkeypatch, pct):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "7")
    path, frames = drift_video
    bg = _bg(path, f"cvvp_percentile:{pct}", vid_is_grayscale=True)
    p = ho.canonical_params(bg)
    static = _track(path, p, {"min_area": 5}, vid_is_grayscale=True)
    for w in (N, 1000):
        kwargs = {"min_area": 5, "cvvp_background_window": w, "cvvp_background_percentile": pct}
        assert _track(path, p, kwargs, vid_is_grayscale=True) == static


def _square_frames(archive):
    """frames with an object whose centroid lies inside the square"""
    ys, xs = SQUARE
    return {o["frame"] for k, o in archive.items() if isinstance(k, int)
            and xs.start <= o["cx"] < xs.stop and ys.start <= o["cy"] < ys.stop}


def test_a_settled_dark_object_needs_a_high_percentile(settled_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "4")
    path, frames = settled_video
    p = ho.canonical_params(percentile(frames, 50))
    w = 20
    present = {t for t in range(N) if _present(t)}
    archives = {}
    for pct in (50, 90):
        kwargs = {"min_area": 20, "cvvp_background_window": w, "cvvp_background_percentile": pct}
        got = _track(path, p, kwargs, vid_is_grayscale=True)
        assert got == host_chain(frames, p, w, pct, {"min_area": 20}), pct
        archives[pct] = got
    # the median window holds the object 14 times in 20: it becomes the background and the masks lose it ...
    assert _square_frames(archives[50]) == set()
    # ... while the 90th percentile (rank 18 of 20) stays above it: every frame that shows the object finds it
    assert _square_frames(archives[90]) == present
