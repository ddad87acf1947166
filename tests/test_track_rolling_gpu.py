"""GPU end-to-end tests of TrackObjects with a rolling median background (kwargs["cvvp_background_window"] = W) on
lossless videos whose brightness drifts, so that a static background and a rolling one give different archives.  The
bar is a host chain: decoded frames -> the oracle's median over each frame's window -> the cv2 restatement of
HighlightObjects with that background -> the same tracker, strictly in frame order."""
import dataclasses

import cv2
import numpy as np
import pytest

import cvvidproc_b200 as cvp
import video_util
from cvvidproc_b200 import synth
from oracle import highlight_oracle as ho

pytestmark = pytest.mark.gpu

N = 60


def _drift(frames, per_frame=0.6):
    t = np.arange(frames.shape[0]).reshape((-1,) + (1,) * (frames.ndim - 1))
    return np.clip(frames.astype(np.int32) + np.round(t * per_frame).astype(np.int32) - 20, 0, 255).astype(np.uint8)


@pytest.fixture(scope="module")
def drift_video(tmp_path_factory):
    frames = _drift(synth.synth_frames(0, N, 160, 96, 7, 8))
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "drift.avi", frames), frames


@pytest.fixture(scope="module")
def drift_colour_video(tmp_path_factory):
    g = synth.synth_frames(0, 40, 96, 64, 11, 6)
    frames = _drift(np.stack([g, np.roll(g, 3, axis=2), 255 - g], axis=-1), 0.8)
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "drift_colour.avi", frames), frames


def _tracker(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs, components=None):
    n, _, stats, cent = cv2.connectedComponentsWithStats(bw_frame, connectivity=8)
    if components is not None:
        assert components["count"] == n - 1
        objects_archive[("count", frames_processed)] = n - 1
    objects_prev.clear()
    for i in range(1, n):
        if stats[i, cv2.CC_STAT_AREA] < kwargs["min_area"]:
            continue
        objects_prev[next_ID] = (frames_processed, int(stats[i, cv2.CC_STAT_AREA]))
        objects_archive[next_ID] = {"frame": frames_processed, "area": int(stats[i, cv2.CC_STAT_AREA]),
                                    "cx": round(float(cent[i][0]), 3), "cy": round(float(cent[i][1]), 3)}
        next_ID += 1
    return next_ID


def _host_chain(frames, p, w, oracle_median, kwargs):
    n = frames.shape[0]
    weff = min(w, n)
    prev, archive, nid, cache = {}, {}, 0, {}
    for t in range(n):
        s = min(max(t - w // 2, 0), n - weff)
        if s not in cache:
            cache[s] = oracle_median(frames[s : s + weff])
        bw = ho.highlight_objects(frames[t].copy(), dataclasses.replace(p, background=cache[s]))
        if kwargs.get("cvvp_components"):
            nid = _count_tracker(bw, t, prev, archive, nid, kwargs)
        else:
            nid = _tracker(bw, t, prev, archive, nid, kwargs)
    return archive


def _count_tracker(bw, t, prev, archive, nid, kwargs):
    n = cv2.connectedComponentsWithStats(bw, connectivity=8)[0]
    archive[("count", t)] = n - 1
    return _tracker(bw, t, prev, archive, nid, kwargs)


def _track(path, p, kwargs, **pack):
    hp = cvp.HighlightObjectsPack(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                  p.min_size_hyst, p.min_size_threshold, p.width_border)
    return cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(_tracker, kwargs), **pack))


@pytest.mark.parametrize("w,batch", [(1, 3), (5, 1), (5, 3), (16, 7), (16, 1), (61, 3), (61, 7)])
def test_rolling_archive_equals_the_host_chain(drift_video, oracle_median, monkeypatch, w, batch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", str(batch))
    path, frames = drift_video
    static_bg = oracle_median(frames)
    p = ho.canonical_params(static_bg)
    kwargs = {"min_area": 5, "cvvp_background_window": w}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    want = _host_chain(frames, p, w, oracle_median, {"min_area": 5})
    assert got == want
    static = _track(path, p, {"min_area": 5}, vid_is_grayscale=True)
    if w == 1:
        assert got == {}  # B_t = f_t: d = 0 everywhere, no pixel passes a non-negative threshold
    elif w < N:
        assert len(want) > 5
        assert got != static  # the drift makes the static archive differ
    else:
        assert got == static  # one window of all N frames: the static median


def test_pack_background_only_sets_the_geometry(drift_video, oracle_median):
    path, frames = drift_video
    p = ho.canonical_params(oracle_median(frames))
    kwargs = {"min_area": 5, "cvvp_background_window": 9}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    assert got == _track(path, dataclasses.replace(p, background=np.zeros_like(p.background)), kwargs, vid_is_grayscale=True)
    with pytest.raises(RuntimeError):  # the reference's validation still holds: the cropped frame's size
        _track(path, dataclasses.replace(p, background=np.zeros((10, 10), np.uint8)), kwargs, vid_is_grayscale=True)


def test_start_frame_and_frame_limit(drift_video, oracle_median, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "4")
    path, frames = drift_video
    p = ho.canonical_params(oracle_median(frames))
    kwargs = {"min_area": 5, "cvvp_background_window": 7}
    got = _track(path, p, kwargs, start_frame=20, frame_limit=25, vid_is_grayscale=True)
    assert got == _host_chain(frames[20:45], p, 7, oracle_median, {"min_area": 5})


def test_cropped_colour_video_with_grayscale(drift_colour_video, oracle_median, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "3")
    path, frames = drift_colour_video
    x, y, cw, ch = 6, 4, 80, 50
    gray = np.stack([cv2.cvtColor(np.ascontiguousarray(f[y : y + ch, x : x + cw]), cv2.COLOR_RGB2GRAY) for f in frames])
    p = ho.canonical_params(oracle_median(gray))
    kwargs = {"min_area": 3, "cvvp_background_window": 11}
    got = _track(path, p, kwargs, grayscale=True, crop_x=x, crop_y=y, crop_width=cw, crop_height=ch)
    want = _host_chain(gray, p, 11, oracle_median, {"min_area": 3})
    assert len(want) > 3
    assert got == want


@pytest.mark.parametrize("labels", [False, True])
def test_components_compose(drift_video, oracle_median, monkeypatch, labels):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "5")
    path, frames = drift_video
    p = ho.canonical_params(oracle_median(frames))
    kwargs = {"min_area": 5, "cvvp_background_window": 16, "cvvp_components": True, "cvvp_labels": labels}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    want = _host_chain(frames, p, 16, oracle_median, {"min_area": 5, "cvvp_components": True})
    assert got == want


def test_window_covering_the_video_equals_the_static_path(drift_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "7")
    path, frames = drift_video
    bg = cvp.GetVideoBackground(cvp.VidBgPack(path, vid_is_grayscale=True))
    p = ho.canonical_params(bg)
    static = _track(path, p, {"min_area": 5}, vid_is_grayscale=True)
    for w in (N, 1000):
        assert _track(path, p, {"min_area": 5, "cvvp_background_window": w}, vid_is_grayscale=True) == static


def test_timing_report_prints_the_same_lines(drift_video, oracle_median, capfd):
    path, frames = drift_video
    p = ho.canonical_params(oracle_median(frames))
    _track(path, p, {"min_area": 5}, vid_is_grayscale=True, print_timing_report=True)
    static_out = capfd.readouterr().out
    _track(path, p, {"min_area": 5, "cvvp_background_window": 5}, vid_is_grayscale=True, print_timing_report=True)
    rolling_out = capfd.readouterr().out
    strip = lambda s: [line.split(":")[0] for line in s.splitlines()]
    assert strip(static_out) == strip(rolling_out) and "Highlight objects timing report" in rolling_out
