"""CPU checks of the colour highlight (cvvp_highlight_set_channels / cvvp_highlight_channels, TrackObjects'
kwargs["cvvp_color"]): the symbols are declared, exported and bound and reject a null context; the colour reference of
tests/color_cases.py satisfies its three identities on the cv2 restatement over the random and adversarial cases in
every polarity, and reproduces every stored reference output through identity (2); and TrackObjects refuses a
malformed cvvp_color before any device work."""
import ctypes
import dataclasses
import hashlib

import numpy as np
import pytest

import color_cases as cc
import cvvidproc_b200 as cvp
import polarity_cases as pc
from cvvidproc_b200 import _cabi

NEW_SYMBOLS = ["cvvp_highlight_set_channels", "cvvp_highlight_channels"]
POLS = list(pc.POLARITIES)


def test_new_symbols_are_declared_exported_and_bound():
    lib = _cabi.load()
    raw = ctypes.CDLL(str(_cabi.LIB_PATH))
    declared = set(_cabi.declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared
        assert hasattr(raw, name)
        assert name in _cabi.BOUND_SYMBOLS
        assert getattr(lib, name).argtypes is not None
    assert hasattr(_cabi.Context, "highlight_set_channels") and hasattr(_cabi.Context, "highlight_channels")


def test_null_context_calls_are_rejected():
    lib = _cabi.load()
    for c in (0, 1, 3, 5):
        assert lib.cvvp_highlight_set_channels(None, c) == -1
    assert lib.cvvp_highlight_channels(None) == -1
    assert b"null context" in lib.cvvp_last_error(None)


def test_color_difference_is_the_channel_maximum():
    rng = np.random.default_rng(3)
    f = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    b = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    for polarity in POLS:
        want = np.max(np.stack([pc.model_difference(b[..., k], f[..., k], polarity) for k in range(3)]), axis=0)
        assert np.array_equal(cc.color_difference(b, f, polarity), want)
    with pytest.raises(ValueError):
        cc.color_difference(b, f, "Dark")


GREY = [(f"random_{t}",) + pc.mixed_random_case(t) for t in range(60)] + pc.mixed_adversarial_cases()


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("case", GREY, ids=[c[0] for c in GREY])
def test_identities_one_and_two_on_the_restatement(case, polarity):
    """(1) one channel is the grey job; (2) replication into C channels gives the grey masks"""
    _, frame, p = case
    grey = pc.highlight_objects(frame.copy(), p, polarity)
    for c in cc.CHANNELS:
        f, q = cc.replicated(frame, p, c)
        assert np.array_equal(cc.highlight_objects(f, q, polarity), grey), c


COLOR = [(f"random_{t}_c{c}",) + cc.random_case(t, c) for t in range(0, 60, 3) for c in (2, 3, 4)]
COLOR += [(f"{name}_c{c}", f, q) for c in (2, 3, 4) for name, f, q in cc.adversarial_cases(c)[::2]]


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("case", COLOR, ids=[c[0] for c in COLOR])
def test_identity_three_on_the_restatement(case, polarity):
    """(3) the restatement's own steps on the colour d equal its "dark" path on 255 - d against 255, which equals the
    device's form: d against a zero background"""
    _, frame, p = case
    d = cc.color_difference(p.background, frame, polarity)
    st = {}
    f, q = cc.as_dark(frame, p, polarity)
    via_dark = pc.highlight_objects(f, q, "dark", st)
    assert np.array_equal(st["diff"], d)
    direct = pc.highlight_objects(np.zeros_like(d), dataclasses.replace(p, background=d), "dark")
    assert np.array_equal(via_dark, direct)  # d - 0 saturated is d: the device's zero-background form
    assert np.array_equal(cc.highlight_objects(frame, p, polarity), via_dark)


def test_channels_other_than_the_first_matter():
    """a colour case whose first channel has no object: its masks come from the other channels"""
    changed = 0
    for t in range(0, 60, 3):
        frame, p = cc.random_case(t, 3)
        grey = pc.highlight_objects(frame[..., 0].copy(), dataclasses.replace(p, background=p.background[..., 0]),
                                    "dark")
        changed += not np.array_equal(cc.highlight_objects(frame, p, "dark"), grey)
    assert changed >= 5


def test_every_stored_reference_output_through_identity_two():
    cases = pc.golden_cases()
    assert len(cases) == 83
    for g, frame, p in cases:
        f, q = cc.replicated(frame, p, 3)
        out = cc.highlight_objects(f, q, "dark")
        assert hashlib.sha256(out.tobytes()).hexdigest() == g["output_sha256"], g["name"]


# ---------------------------------------------------------------------------------------------------------------------
# TrackObjects' kwargs["cvvp_color"]

def _pack(kwargs, grayscale=False, vid_is_grayscale=False, bg_shape=(4, 4, 3)):
    hp = cvp.HighlightObjectsPack(np.zeros(bg_shape, np.uint8), np.ones((2, 2), np.uint8), 1, 1, 1, 1, 1, 1)
    ap = cvp.AssignObjectsPack(lambda **kw: 0, kwargs)
    return cvp.VidObjectTrackPack("/nonexistent/video.mp4", hp, ap, grayscale=grayscale, vid_is_grayscale=vid_is_grayscale)


@pytest.mark.parametrize("value", [None, 1, 0, "True", np.bool_(True), [True]])
def test_track_objects_refuses_a_non_bool_color_before_any_device_work(value):
    # a missing video makes TrackObjects return {} without raising: the key is checked before that
    with pytest.raises(RuntimeError, match="cvvp_color"):
        cvp.TrackObjects(_pack({"cvvp_color": value}))


@pytest.mark.parametrize("gray", [(True, False), (False, True), (True, True)])
def test_track_objects_refuses_color_with_a_grayscale_setting(gray):
    with pytest.raises(RuntimeError, match="cvvp_color"):
        cvp.TrackObjects(_pack({"cvvp_color": True}, *gray))


def test_track_objects_accepts_a_good_color_key(capfd):
    for kwargs in ({"cvvp_color": True}, {"cvvp_color": False},
                   {"cvvp_color": True, "cvvp_polarity": "both", "cvvp_background_window": 5}):
        assert cvp.TrackObjects(_pack(dict(kwargs))) == {}
        assert "Video file not detected" in capfd.readouterr().err
    # False is today's behaviour, with a grayscale setting too
    assert cvp.TrackObjects(_pack({"cvvp_color": False}, True, False, (4, 4))) == {}
