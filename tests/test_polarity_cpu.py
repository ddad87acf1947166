"""CPU checks of the object polarity (cvvp_highlight_set_polarity / cvvp_highlight_polarity, TrackObjects'
kwargs["cvvp_polarity"]): the symbols are declared, exported and bound and reject a null context; the host references
of tests/polarity_cases.py equal the oracles they compose at "dark", satisfy the two identities that tie "bright" and
"both" to the reference's "dark" on every case, and reproduce every stored reference output through them; the cv2 and
label-model references agree in the new polarities; and TrackObjects refuses a malformed polarity before any device
work."""
import ctypes
import hashlib

import cv2
import numpy as np
import pytest

import cvvidproc_b200 as cvp
import hl_cases
import polarity_cases as pc
from cvvidproc_b200 import _cabi
from oracle import highlight_model as hm
from oracle import highlight_oracle as ho
from oracle import highlight_ref as href

NEW_SYMBOLS = ["cvvp_highlight_set_polarity", "cvvp_highlight_polarity"]


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
    for polarity in (0, 1, 2, 3):
        assert lib.cvvp_highlight_set_polarity(None, polarity) == -1
    assert lib.cvvp_highlight_polarity(None) == -1
    assert b"null context" in lib.cvvp_last_error(None)


def _ho(frame, p, polarity):
    return pc.highlight_objects(frame.copy(), p, polarity)


def _all_cases():
    cases = [(f"random_{t}",) + hl_cases.random_case(t) for t in range(60)]
    return cases + hl_cases.adversarial_cases()


ALL = _all_cases()


@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_host_references_are_the_oracles_at_dark(case):
    """the polarity references compose the oracles' own steps: at "dark" they are the oracles"""
    _, frame, p = case
    for f in (frame, pc.mixed(frame, p.background)):
        want = ho.highlight_objects(f.copy(), p)
        assert np.array_equal(_ho(f, p, "dark"), want)
        assert np.array_equal(pc.model_highlight_objects(f, p, "dark"), want)


@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_identities_hold_on_the_restatement(case):
    _, frame, p = case
    dark = _ho(frame, p, "dark")
    bright = _ho(frame, p, "bright")
    fi, pi = pc.inverted(frame, p)
    assert np.array_equal(_ho(fi, pi, "bright"), dark)  # (1) read backwards
    assert np.array_equal(_ho(fi, pi, "dark"), bright)  # (1)
    assert np.array_equal(_ho(np.minimum(frame, p.background), p, "both"), dark)  # (2)
    assert np.array_equal(_ho(np.maximum(frame, p.background), p, "both"), bright)  # (2)
    # and on a frame whose difference has both signs
    m = pc.mixed(frame, p.background)
    mi, pmi = pc.inverted(m, p)
    assert np.array_equal(_ho(mi, pmi, "dark"), _ho(m, p, "bright"))
    assert np.array_equal(_ho(mi, pmi, "both"), _ho(m, p, "both"))  # |f - bg| is symmetric under inversion


def test_polarity_changes_only_the_difference_image():
    frame, p = pc.mixed_random_case(3)
    for polarity, want in (("dark", cv2.subtract(p.background, frame)), ("bright", cv2.subtract(frame, p.background)),
                           ("both", cv2.absdiff(frame, p.background))):
        st = {}
        pc.highlight_objects(frame.copy(), p, polarity, st)
        assert np.array_equal(st["diff"], want)
        assert np.array_equal(pc.model_difference(p.background, frame, polarity), want)
    assert np.array_equal(hm.diff_sat(p.background, frame), cv2.subtract(p.background, frame))
    with pytest.raises(ValueError):
        pc.difference_image(p.background, frame, "Bright")


def test_identities_reproduce_every_stored_reference_output():
    """tests/golden/highlight_golden.json holds hashes of the reference's own masks ("dark"): identity (1) and the
    min half of identity (2) turn each stored case into a "bright" and a "both" case with the same stored output"""
    cases = pc.golden_cases()
    assert len(cases) == 83
    for g, frame, p in cases:
        assert hashlib.sha256(frame.tobytes()).hexdigest() == g["input_sha256"], g["name"]
        fi, pi = pc.inverted(frame, p)
        for f, q, polarity in ((fi, pi, "bright"), (np.minimum(frame, p.background), p, "both")):
            out = pc.highlight_objects(f.copy(), q, polarity)
            assert hashlib.sha256(out.tobytes()).hexdigest() == g["output_sha256"], (g["name"], polarity)


def _model(frame, p, polarity):
    return pc.model_highlight_objects(frame, p, polarity)


MIXED = [(f"random_{t}",) + pc.mixed_random_case(t) for t in range(60)] + pc.mixed_adversarial_cases()


@pytest.mark.parametrize("polarity", ["bright", "both"])
@pytest.mark.parametrize("case", MIXED, ids=[c[0] for c in MIXED])
def test_label_model_agrees_with_the_restatement(case, polarity):
    _, frame, p = case
    assert np.array_equal(_model(frame, p, polarity), _ho(frame, p, polarity))


needs_ref = pytest.mark.skipif(not href.available(), reason="oracle/_ref/cvvp_highlight_ref was not built (no /root/reference)")


@needs_ref
@pytest.mark.parametrize("case", MIXED[::3], ids=[c[0] for c in MIXED[::3]])
def test_the_compiled_reference_in_the_new_polarities(case):
    """bright = the compiled HighlightObjectsAlgo on inverted inputs; both = its helper functions (ThresholdImage,
    ThresholdImageWithHysteresis, RemoveSmallObjects, FillHoles) composed on d = |frame - bg| as HighlightObjects
    composes them (:35-77)"""
    _, frame, p = case
    fi, pi = pc.inverted(frame, p)
    assert np.array_equal(href.highlight_objects(fi, pi), _ho(frame, p, "bright"))
    op = href.operator(p)
    d = cv2.absdiff(p.background, frame)
    selem = np.ascontiguousarray(p.struct_element)
    a = cv2.morphologyEx(op.threshold_image(d, p.threshold), cv2.MORPH_OPEN, selem)
    a = op.fill_holes(op.remove_small_objects(a, p.min_size_threshold))
    b = cv2.morphologyEx(op.threshold_image_with_hysteresis(d, p.threshold_lo, p.threshold_hi), cv2.MORPH_OPEN, selem)
    b = op.fill_holes(op.remove_small_objects(b, p.min_size_hyst))
    assert np.array_equal(cv2.bitwise_or(a, b), _ho(frame, p, "both"))


# ---------------------------------------------------------------------------------------------------------------------
# TrackObjects' kwargs["cvvp_polarity"]

def _pack(kwargs):
    hp = cvp.HighlightObjectsPack(np.zeros((4, 4), np.uint8), np.ones((2, 2), np.uint8), 1, 1, 1, 1, 1, 1)
    ap = cvp.AssignObjectsPack(lambda **kw: 0, kwargs)
    return cvp.VidObjectTrackPack("/nonexistent/video.mp4", hp, ap)


@pytest.mark.parametrize("value", [None, 1, True, "Bright", "", b"dark", "DARK", " both", 0, ["dark"]])
def test_track_objects_refuses_a_bad_polarity_before_any_device_work(value):
    # a missing video makes TrackObjects return {} without raising: the polarity is checked before that
    with pytest.raises(RuntimeError, match="cvvp_polarity"):
        cvp.TrackObjects(_pack({"cvvp_polarity": value}))


@pytest.mark.parametrize("value", ["dark", "bright", "both"])
def test_track_objects_accepts_a_good_polarity(value, capfd):
    kwargs = {"cvvp_polarity": value, "cvvp_background_window": 5, "cvvp_background_percentile": 10}
    assert cvp.TrackObjects(_pack(kwargs)) == {}
    assert "Video file not detected" in capfd.readouterr().err
    assert kwargs == {"cvvp_polarity": value, "cvvp_background_window": 5, "cvvp_background_percentile": 10}
    assert cvp.TrackObjects(_pack({"cvvp_polarity": value})) == {}
