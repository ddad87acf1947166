"""CPU tests of the frame-source oracle (oracle/frames_oracle.py): against the reference's own generator compiled
unmodified (oracle/_ref/cvvp_frames_ref, see oracle/frames_ref.py) on lossless videos; the closed form of OpenCV's
8-bit RGB2GRAY against cv2 on ALL 2^24 colour triples; the crop-rectangle rule incl. its quirk; the committed golden
hashes (outputs of the reference where a video can carry the case); and the ctypes view of struct cvvp_frame_format.
No GPU."""
import ctypes
import hashlib
import json
from pathlib import Path

import cv2
import numpy as np
import pytest

import frame_cases
import video_util
from cvvidproc_b200 import _cabi
from oracle import frames_oracle as fo
from oracle import frames_ref as fref

needs_ref = pytest.mark.skipif(not fref.available(), reason="oracle/_ref/cvvp_frames_ref was not built (no /root/reference)")

GOLDEN = json.loads((Path(__file__).parent / "golden" / "frames_golden.json").read_text())


def test_rgb2gray_closed_form_matches_cv2_on_every_triple():
    g, b = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    img = np.empty((256, 256, 3), np.uint8)
    img[..., 1] = g
    img[..., 2] = b
    for r in range(256):
        img[..., 0] = r
        want = cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)
        assert np.array_equal(fo.rgb2gray_fixed_point(img[..., 0], g, b), want), f"first channel {r}"


def test_rgb2gray_ignores_a_fourth_channel():
    img = np.random.default_rng(0).integers(0, 256, (37, 53, 4), dtype=np.uint8)
    want = cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)
    assert np.array_equal(fo.rgb2gray_fixed_point(img[..., 0], img[..., 1], img[..., 2]), want)


def test_crop_rule_follows_the_reference_quirk():
    # cv_vid_bg_helpers.cpp:52-57
    assert fo.get_cropped_frame_dims(0, 0, 0, 0, 640, 480) == (0, 0, 640, 480)
    assert fo.get_cropped_frame_dims(10, 20, 100, 50, 640, 480) == (10, 20, 100, 50)
    assert fo.get_cropped_frame_dims(600, 0, 100, 0, 640, 480) == (600, 0, 40, 480)
    # :56 compares height + y against hor_pixels: 300 + 200 <= 640 is NOT clamped although it leaves the 480 rows
    assert fo.get_cropped_frame_dims(0, 200, 0, 300, 640, 480) == (0, 200, 640, 300)
    # ... and on a portrait frame a legal height is clamped as soon as it exceeds the WIDTH
    assert fo.get_cropped_frame_dims(0, 100, 0, 400, 480, 640) == (0, 100, 480, 540)
    with pytest.raises(AssertionError):
        fo.get_cropped_frame_dims(640, 0, 0, 0, 640, 480)


CASES = frame_cases.cases()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_matches_golden_and_closed_form(case):
    name, frames, crop, mode = case
    res = fo.prepare_frames(frames, crop, mode)
    g = next(e for e in GOLDEN if e["name"] == name)
    assert hashlib.sha256(frames.tobytes()).hexdigest() == g["input_sha256"]
    assert list(res.shape) == g["out_shape"]
    assert hashlib.sha256(res.tobytes()).hexdigest() == g["output_sha256"]
    # the same result from plain slicing + the closed form (what the CUDA kernel computes)
    x, y, w, h = crop
    c = frames[:, y:y + h, x:x + w]
    if mode == fo.RGB2GRAY:
        want = fo.rgb2gray_fixed_point(c[..., 0], c[..., 1], c[..., 2])
    elif mode == fo.CHANNEL0 and c.ndim == 4:
        want = c[..., 0]
    else:
        want = c
    assert np.array_equal(res, want)


VIDEO_CASES = [c for c in CASES if c[1].ndim == 4 and c[1].shape[3] == 3 and c[1].shape[1] % 2 == 0]


@pytest.mark.parametrize("case", VIDEO_CASES, ids=[c[0] for c in VIDEO_CASES])
def test_restatement_matches_the_compiled_reference_generator(case, tmp_path):
    """CvVidFramesGeneratorAlgo::GetTokenSet (cv_vid_frames_generator_algo.h:119-189) on a lossless video of the case's
    frames == oracle.prepare_frames on the decoded frames, and == the golden hash, which is the generator's own output
    (without oracle/_ref the restatement of the decoded frames is held to that hash alone)"""
    name, frames, crop, mode = case
    vid = video_util.write_lossless(tmp_path / "v.avi", frames)
    decoded = video_util.read_all(vid)
    assert np.array_equal(decoded, frames)
    want = fo.prepare_frames(decoded, crop, mode)
    if fref.available():
        toks = fref.tokens(vid, 0, len(frames), crop, mode, frames_in_batch=3)
        assert len(toks) == len(want)
        got = np.stack(toks)
        assert got.dtype == np.uint8 and np.array_equal(got, want)
    g = next(e for e in GOLDEN if e["name"] == name)
    assert g["source"].startswith("reference")
    assert hashlib.sha256(want.tobytes()).hexdigest() == g["output_sha256"]


@needs_ref
def test_reference_generator_frame_range_and_batches(tmp_path):
    """start_frame / last_frame (:97-104, :128-129), a last_frame beyond the stream, batches of any size, and the
    generator's own assertion on a crop rectangle that leaves the frame (:92-93)"""
    frames = np.random.default_rng(3).integers(0, 256, (11, 36, 50, 3), dtype=np.uint8)
    vid = video_util.write_lossless(tmp_path / "v.avi", frames)
    crop = (3, 2, 41, 30)
    for start, last, batch in ((0, 11, 4), (2, 9, 3), (5, 6, 1), (4, 500, 5), (10, 11, 2)):
        for mode in (fo.RGB2GRAY, fo.CHANNEL0, fo.AS_IS):
            toks = fref.tokens(vid, start, last, crop, mode, frames_in_batch=batch)
            want = fo.prepare_frames(frames[start:min(last, len(frames))], crop, mode)
            assert len(toks) == len(want), (start, last, batch, mode)
            assert np.array_equal(np.stack(toks), want), (start, last, batch, mode)
    with pytest.raises(RuntimeError, match="crop_rectangle"):
        fref.tokens(vid, 0, 11, (10, 0, 41, 36), fo.RGB2GRAY)
    with pytest.raises(RuntimeError, match="start_frame"):
        fref.tokens(vid, 11, 12, crop, fo.RGB2GRAY)


def test_frame_format_struct_layout():
    assert ctypes.sizeof(_cabi.FrameFormat) == 32  # eight int32 fields, include/cvvp.h
    f = _cabi.FrameFormat.of((48, 64, 3), _cabi.FRAMES_RGB2GRAY, crop=(1, 2, 30, 20))
    assert (f.src_width, f.src_height, f.src_channels) == (64, 48, 3)
    assert (f.crop_x, f.crop_y, f.crop_width, f.crop_height, f.mode) == (1, 2, 30, 20, 2)
    assert f.out_shape == (20, 30)
    lib = _cabi.load()
    assert lib.cvvp_frame_format_out_bytes(ctypes.byref(f)) == 600
    f.mode = _cabi.FRAMES_AS_IS
    assert f.out_shape == (20, 30, 3)
    assert lib.cvvp_frame_format_out_bytes(ctypes.byref(f)) == 1800
    assert lib.cvvp_frame_format_out_bytes(None) == 0
    assert (frame_cases.AS_IS, frame_cases.CHANNEL0, frame_cases.RGB2GRAY) == (fo.AS_IS, fo.CHANNEL0, fo.RGB2GRAY) == (
        _cabi.FRAMES_AS_IS, _cabi.FRAMES_CHANNEL0, _cabi.FRAMES_RGB2GRAY)


def test_null_context_calls_of_the_new_entry_points_are_rejected():
    lib = _cabi.load()
    assert lib.cvvp_frames_prepare(None, None, 1, 1, None, None, 1) == -1
    assert lib.cvvp_median_push_source(None, None, 1, 1, None) == -1
    assert lib.cvvp_highlight_queue_begin(None, 2, 4, None, 0) == -1
    assert lib.cvvp_highlight_submit(None, None, 1, 1) == -1
    assert lib.cvvp_highlight_queue_pending(None) == 0
