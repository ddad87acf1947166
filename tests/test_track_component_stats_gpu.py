"""GPU end-to-end tests of TrackObjects' kwargs["cvvp_component_stats"] on lossless videos: the callback's "moments",
"mass", "weighted_centroids" and "contrast" equal host statistics computed from bw_frame, the decoded frames and the
background (the pack's, or each frame's window median), with a static background in the bright polarity, a rolling
window, two operators on one device and small batches."""
import numpy as np
import pytest

import cvvidproc_b200 as cvp
import polarity_cases as pc
import video_util
from cvvidproc_b200 import synth
from oracle import highlight_oracle as ho
from test_component_stats_cpu import canonical_labels, reference_stats
from test_track_percentile_gpu import percentile

pytestmark = pytest.mark.gpu

N = 30


@pytest.fixture(scope="module")
def bright_video(tmp_path_factory):
    frames = (255 - synth.synth_frames(0, N, 160, 96, 7, 8)).astype(np.uint8)
    return video_util.write_lossless(tmp_path_factory.mktemp("v") / "bright.avi", frames), frames


def _run(path, p, kwargs):
    seen = {}

    def cb(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs, components=None):
        seen[frames_processed] = (np.array(bw_frame, copy=True), {k: np.array(v, copy=True) if k != "count" else v
                                                                  for k, v in components.items()})
        return next_ID

    hp = cvp.HighlightObjectsPack(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                  p.min_size_hyst, p.min_size_threshold, p.width_border)
    cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(cb, kwargs), vid_is_grayscale=True))
    assert sorted(seen) == list(range(N))
    return seen


def _backgrounds(frames, p, window):
    if window is None:
        return [p.background] * N
    weff = min(window, N)
    return [percentile(frames[s:s + weff], 50) for s in (min(max(t - window // 2, 0), N - weff) for t in range(N))]


def _check(seen, frames, bgs, polarity):
    total = 0
    for t in range(N):
        bw, comps = seen[t]
        lab = comps["labels"] if "labels" in comps else canonical_labels(bw)
        want = reference_stats(lab, frames[t], bgs[t], polarity, max_comps=comps["moments"].shape[0])
        total += len(want)
        assert comps["count"] == lab.max()
        assert np.array_equal(comps["moments"], np.stack([want["sum_xx"], want["sum_xy"], want["sum_yy"]], 1)), t
        assert np.array_equal(comps["mass"], want["sum_d"]), t
        with np.errstate(invalid="ignore", divide="ignore"):
            wc = np.stack([want["sum_dx"] / want["sum_d"], want["sum_dy"] / want["sum_d"]], 1)
        assert np.array_equal(comps["weighted_centroids"], wc, equal_nan=True), t
        assert np.array_equal(comps["contrast"], np.stack([want["min_d"], want["max_d"]], 1)), t
        assert comps["moments"].dtype == np.int64 and comps["contrast"].dtype == np.int32
    assert total > 0


def test_static_background_bright(bright_video, monkeypatch):
    path, frames = bright_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"cvvp_components": True, "cvvp_component_stats": True, "cvvp_polarity": "bright"}
    seen = _run(path, p, kwargs)
    for t in range(N):
        assert np.array_equal(seen[t][0], pc.highlight_objects(frames[t].copy(), p, "bright"))
    _check(seen, frames, _backgrounds(frames, p, None), "bright")
    # labels take the synchronous path; the statistics are the same
    monkeypatch.setenv("CVVP_TRACK_BATCH", "4")
    seen_l = _run(path, p, dict(kwargs, cvvp_labels=True))
    _check(seen_l, frames, _backgrounds(frames, p, None), "bright")
    for t in range(N):
        for k in ("moments", "mass", "contrast"):
            assert np.array_equal(seen_l[t][1][k], seen[t][1][k])


def test_rolling_window(bright_video, monkeypatch):
    monkeypatch.setenv("CVVP_TRACK_BATCH", "5")
    path, frames = bright_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"cvvp_components": True, "cvvp_component_stats": True, "cvvp_polarity": "bright",
              "cvvp_background_window": 9}
    _check(_run(path, p, kwargs), frames, _backgrounds(frames, p, 9), "bright")


def test_two_operators_on_one_device_small_batches_and_host_preparation(bright_video, monkeypatch):
    path, frames = bright_video
    p = ho.canonical_params(percentile(frames, 50))
    kwargs = {"cvvp_components": True, "cvvp_component_stats": True, "cvvp_polarity": "both"}
    monkeypatch.setenv("CVVP_TRACK_BATCH", "2")
    monkeypatch.setenv("CVVP_DEVICES", "0,0")
    _check(_run(path, p, kwargs), frames, _backgrounds(frames, p, None), "both")
    monkeypatch.delenv("CVVP_DEVICES")
    monkeypatch.setenv("CVVP_HOST_PREP", "1")
    _check(_run(path, p, kwargs), frames, _backgrounds(frames, p, None), "both")
