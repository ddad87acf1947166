"""GPU end-to-end tests of the object polarity through the Python surface (TrackObjects' kwargs["cvvp_polarity"]) on
lossless videos, against host chains (decoded frames -> the cv2 restatement's steps on the difference image of the
polarity, tests/polarity_cases.py -> the tracker): bright disks on a dark field, which the default polarity does not see; dark and bright disks
together under "both"; a still bright square that a rolling median swallows and a low percentile keeps; components,
two operators on one device and host-side frame preparation."""
import dataclasses

import numpy as np
import pytest

import cvvidproc_b200 as cvp
import polarity_cases as pc
import video_util
from cvvidproc_b200 import synth
from oracle import highlight_oracle as ho
from test_track_percentile_gpu import SQUARE, _present, _square_frames, percentile
from test_track_rolling_gpu import _count_tracker, _drift, _track, _tracker

pytestmark = pytest.mark.gpu

N = 40


@pytest.fixture(scope="module")
def bright_video(tmp_path_factory):
    """the synthetic stream inverted: bright disks on a dark field"""
    frames = (255 - synth.synth_frames(0, N, 160, 96, 7, 8)).astype(np.uint8)
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "bright.avi", frames), frames


@pytest.fixture(scope="module")
def two_sided_video(tmp_path_factory):
    """dark disks on the left half, bright disks on the right"""
    g = synth.synth_frames(0, N, 160, 96, 9, 10)
    bg = percentile(g, 50)
    frames = np.stack([pc.mixed(f, bg) for f in g])
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "two_sided.avi", frames), frames


def _recorder():
    """a tracker callback that keeps every mask and the kwargs it was handed"""
    seen = {"masks": {}, "kwargs": []}

    def cb(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs, components=None):
        seen["masks"][frames_processed] = np.array(bw_frame, copy=True)
        seen["kwargs"].append(dict(kwargs))
        return next_ID

    return cb, seen


def _masks(path, p, kwargs, **pack):
    cb, seen = _recorder()
    hp = cvp.HighlightObjectsPack(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                  p.min_size_hyst, p.min_size_threshold, p.width_border)
    cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(cb, kwargs), vid_is_grayscale=True, **pack))
    assert sorted(seen["masks"]) == list(range(N))
    assert all(k == kwargs for k in seen["kwargs"])  # every cvvp_ key reaches the callback unchanged
    return np.stack([seen["masks"][t] for t in range(N)])


def _host_masks(frames, p, polarity):
    return pc.masks(frames, p, polarity)


def host_chain(frames, p, polarity, kwargs, w=None, pct=50):
    """decoded frames -> the pack's background, or each frame's window percentile (w) -> the masks of the polarity ->
    the tracker (the counting tracker with components)"""
    n = frames.shape[0]
    prev, archive, nid, cache = {}, {}, 0, {}
    track = _count_tracker if kwargs.get("cvvp_components") else _tracker
    for t in range(n):
        q = p
        if w is not None:
            weff = min(w, n)
            s = min(max(t - w // 2, 0), n - weff)
            if s not in cache:
                cache[s] = percentile(frames[s : s + weff], pct)
            q = dataclasses.replace(p, background=cache[s])
        bw = pc.highlight_objects(frames[t].copy(), q, polarity)
        nid = track(bw, t, prev, archive, nid, kwargs)
    return archive


def test_bright_objects_need_the_bright_polarity(bright_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "7")
    path, frames = bright_video
    bg = percentile(frames, 5)  # the dark field under the moving disks
    p = ho.canonical_params(bg)
    disks = frames.astype(np.int32) - bg > 20
    dark = _masks(path, p, {"min_area": 5})
    assert np.array_equal(dark, _host_masks(frames, p, "dark"))
    assert not dark.any()  # nothing of the disks, nor anything else
    bright = _masks(path, p, {"min_area": 5, "cvvp_polarity": "bright"})
    assert np.array_equal(bright, _host_masks(frames, p, "bright"))
    assert (bright.astype(bool) & disks).sum() > 0.9 * disks.sum()
    assert np.array_equal(_masks(path, p, {"min_area": 5, "cvvp_polarity": "dark"}), dark)


def test_dark_and_bright_objects_under_both(two_sided_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "5")
    path, frames = two_sided_video
    p = ho.canonical_params(percentile(frames, 50))
    got = {pol: _masks(path, p, {"min_area": 5, "cvvp_polarity": pol}) for pol in ("dark", "bright", "both")}
    for pol, m in got.items():
        assert np.array_equal(m, _host_masks(frames, p, pol)), pol
    half = frames.shape[2] // 2
    assert got["dark"][:, :, :half].any() and got["bright"][:, :, half:].any()
    assert got["both"][:, :, :half].any() and got["both"][:, :, half:].any()


@pytest.fixture(scope="module")
def settled_bright_video(tmp_path_factory):
    """a still bright square present in 7 of every 10 frames on an inverted, drifting stream"""
    frames = (255 - _drift(synth.synth_frames(0, 60, 160, 96, 23, 1))).astype(np.uint8)
    for t in range(60):
        if _present(t):
            frames[(t,) + SQUARE] = 243
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "settled_bright.avi", frames), frames


def test_a_settled_bright_object_needs_a_low_percentile(settled_bright_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "4")
    path, frames = settled_bright_video
    p = ho.canonical_params(percentile(frames, 50))
    w = 20
    present = {t for t in range(frames.shape[0]) if _present(t)}
    archives = {}
    for pct in (50, 10):
        kwargs = {"min_area": 20, "cvvp_background_window": w, "cvvp_background_percentile": pct,
                  "cvvp_polarity": "bright"}
        got = _track(path, p, kwargs, vid_is_grayscale=True)
        assert got == host_chain(frames, p, "bright", {"min_area": 20}, w, pct), pct
        archives[pct] = got
    # the median window holds the square 14 times in 20: it becomes the background and the masks lose it ...
    assert _square_frames(archives[50]) == set()
    # ... while the 10th percentile (rank 2 of 20) stays below it: every frame that shows the square finds it
    assert _square_frames(archives[10]) == present


@pytest.mark.parametrize("polarity", ["bright", "both"])
def test_components_compose(two_sided_video, monkeypatch, polarity):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "6")
    path, frames = two_sided_video
    p = ho.canonical_params(percentile(frames, 50))
    for labels in (False, True):
        kwargs = {"min_area": 5, "cvvp_components": True, "cvvp_labels": labels, "cvvp_polarity": polarity}
        got = _track(path, p, kwargs, vid_is_grayscale=True)
        assert got == host_chain(frames, p, polarity, {"min_area": 5, "cvvp_components": True}), labels
    kwargs = {"min_area": 5, "cvvp_components": True, "cvvp_background_window": 9, "cvvp_polarity": polarity}
    got = _track(path, p, kwargs, vid_is_grayscale=True)
    assert got == host_chain(frames, p, polarity, {"min_area": 5, "cvvp_components": True}, 9)


def test_two_operators_on_one_device_and_host_preparation(bright_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "3")
    path, frames = bright_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"min_area": 5, "cvvp_polarity": "bright"}
    one = _track(path, p, kwargs, vid_is_grayscale=True)
    assert one == host_chain(frames, p, "bright", {"min_area": 5})
    monkeypatch.setenv("CVVP_DEVICES", "0,0")
    assert _track(path, p, kwargs, vid_is_grayscale=True) == one
    monkeypatch.delenv("CVVP_DEVICES")
    monkeypatch.setenv("CVVP_HOST_PREP", "1")
    assert _track(path, p, kwargs, vid_is_grayscale=True) == one
    rolling = dict(kwargs, cvvp_background_window=11)
    assert _track(path, p, rolling, vid_is_grayscale=True) == host_chain(frames, p, "bright", {"min_area": 5}, 11)
