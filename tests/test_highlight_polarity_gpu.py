"""GPU tests of the object polarity through the C ABI (cvvp_highlight_set_polarity): "bright" (d = max(frame - bg, 0))
and "both" (d = |frame - bg|) against the cv2 restatement's steps run on that d (tests/polarity_cases.py) on both builds
of the fused kernel, its 128-bit and byte paths, Otsu and the per-pixel kernels; every stored reference output through
the two identities of tests/polarity_cases.py; full-size frames device against device; components, backgrounds per
frame, the queue and the rolling stream; and the setting's state and argument errors."""
import hashlib

import numpy as np
import pytest
import torch

import hl_cases
import polarity_cases as pc
from cvvidproc_b200 import _cabi, synth
from oracle import frames_oracle as fo
from oracle import highlight_oracle as ho
from test_components_gpu import _check_frame
from test_highlight_bg_gpu import _backgrounds, _device_bg
from test_highlight_rolling_stream_gpu import (SMALL, assert_same_results, device_reference, fine_params, host_backgrounds,
                                               make_frames, run_stream)

pytestmark = pytest.mark.gpu

FUSED, PIXEL = 0, 1
ERR_INVALID, ERR_STATE = -1, -4


@pytest.fixture(scope="module")
def ctx():
    # a context of its own: the polarity is a setting of the context
    c = _cabi.Context(0)
    yield c
    c.close()


def _begin(ctx, p):
    ctx.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                        p.min_size_hyst, p.min_size_threshold, p.width_border)


def _gpu(ctx, frames, p, polarity, path=FUSED):
    ctx.highlight_set_polarity(pc.POLARITIES[polarity])
    _begin(ctx, p)
    try:
        ctx.highlight_set_path(path)
        return ctx.highlight_frames(frames)
    finally:
        ctx.highlight_end()
        ctx.highlight_set_polarity(0)


def _want(frame, p, polarity):
    return pc.highlight_objects(frame.copy(), p, polarity)


def _check(ctx, frame, p, polarity, path=FUSED, what=""):
    got = _gpu(ctx, frame[None], p, polarity, path)[0]
    want = _want(frame, p, polarity)
    assert np.array_equal(got, want), f"{what} {polarity}: {(got != want).sum()} pixels differ"


POLS = ["bright", "both"]
MIXED_ADV = pc.mixed_adversarial_cases()


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("t", range(60))
def test_random_cases_match_oracle(ctx, t, polarity):
    frame, p = pc.mixed_random_case(t)
    _check(ctx, frame, p, polarity)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("case", MIXED_ADV, ids=[c[0] for c in MIXED_ADV])
def test_adversarial_cases_match_oracle(ctx, case, polarity):
    name, frame, p = case
    _check(ctx, frame, p, polarity, what=name)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("variant", ["large", "small"])
def test_both_builds_of_the_fused_kernel(ctx, monkeypatch, variant, polarity):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    for t in range(0, 60, 4):
        frame, p = pc.mixed_random_case(t)
        _check(ctx, frame, p, polarity, what=f"{variant} random_{t}")
    for name, frame, p in MIXED_ADV[::2]:
        _check(ctx, frame, p, polarity, what=f"{variant} {name}")


@pytest.mark.parametrize("polarity", POLS)
def test_per_pixel_path(ctx, polarity):
    for t in range(0, 60, 5):
        frame, p = pc.mixed_random_case(t)
        _check(ctx, frame, p, polarity, PIXEL, what=f"random_{t}")
    for name, frame, p in MIXED_ADV[::2]:
        _check(ctx, frame, p, polarity, PIXEL, what=name)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("path", [FUSED, PIXEL])
@pytest.mark.parametrize("hw", [(40, 32), (33, 64), (21, 128), (17, 640), (9, 1056), (30, 75), (19, 33), (25, 150)])
def test_aligned_and_unaligned_widths_with_otsu(ctx, hw, path, polarity):
    """W % 32 == 0 takes the fused kernel's 128-bit path, other widths its byte path; threshold -1 is Otsu on d"""
    h, w = hw
    for seed in range(2):
        frame, bg = hl_cases.blob_frame(h, w, 400 + seed, sigma=2.0, amp=70)
        frame = pc.mixed(frame, bg)
        for p in (ho.canonical_params(bg), ho.HighlightParams(bg, np.ones((1, 1), np.uint8), 12, 6, 20, 0, 3, 5),
                  ho.HighlightParams(bg, np.ones((3, 2), np.uint8), -1, 9, 14, 10, 30, 5),
                  ho.HighlightParams(bg, np.ones((1, 1), np.uint8), -1, 20, 8, 0, 0, 5)):
            _check(ctx, frame, p, polarity, path, what=f"{h}x{w} seed {seed} th {p.threshold}")


@pytest.mark.parametrize("path", [FUSED, PIXEL])
def test_every_stored_reference_output_through_the_identities(ctx, path):
    """the reference's own masks (dark) are reproduced by bright on inverted inputs (1), by both on min(f, bg) and --
    as bright of the same inputs -- by both on max(f, bg) (2), and by an explicit dark"""
    cases = pc.golden_cases()
    assert len(cases) == 83
    for g, frame, p in cases:
        fi, pi = pc.inverted(frame, p)
        for polarity, f, q in (("dark", frame, p), ("bright", fi, pi), ("both", np.minimum(frame, p.background), p)):
            got = _gpu(ctx, f[None], q, polarity, path)[0]
            assert hashlib.sha256(got.tobytes()).hexdigest() == g["output_sha256"], (g["name"], polarity)
        bright = _gpu(ctx, frame[None], p, "bright", path)[0]
        assert np.array_equal(_gpu(ctx, np.maximum(frame, p.background)[None], p, "both", path)[0], bright), g["name"]


@pytest.mark.parametrize("cfg,n", [("C3", 6), ("C4", 40)])
def test_full_size_frames(ctx, cfg, n):
    """1080p C3 and 512x256 C4 frames: bright on inverted frames equals dark on the originals, and the fused and per-pixel
    paths agree in both"""
    q = synth.CONFIG_PARAMS[cfg]
    w, h = q["width"], q["height"]
    bg = np.sort(synth.synth_frames(0, 31, w, h, q["seed"], q["ndisks"]), axis=0)[15]
    p = ho.canonical_params(bg)
    frames = synth.synth_frames(200, n, w, h, q["seed"], q["ndisks"])
    dark = _gpu(ctx, frames, p, "dark")
    fi, pi = pc.inverted(frames, p)
    assert np.array_equal(_gpu(ctx, fi, pi, "bright"), dark)
    assert dark[::max(1, n // 4)].any()  # the frames have objects
    mixed = np.stack([pc.mixed(f, bg) for f in frames])
    fused = _gpu(ctx, mixed, p, "both", FUSED)
    assert np.array_equal(fused, _gpu(ctx, mixed, p, "both", PIXEL))
    assert np.array_equal(fused[1], _want(mixed[1], p, "both"))


def test_components_in_bright(ctx):
    ctx.highlight_set_polarity(1)
    try:
        for t in range(0, 60, 6):
            frame, p = pc.mixed_random_case(t)
            _begin(ctx, p)
            try:
                masks, comps, ncomps, labels = ctx.highlight_frames_cc(frame[None], max_comps=512, labels=True)
            finally:
                ctx.highlight_end()
            want = _want(frame, p, "bright")
            assert np.array_equal(masks[0], want)
            _check_frame(masks[0], comps[0], int(ncomps[0]), labels[0])
    finally:
        ctx.highlight_set_polarity(0)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("path", [FUSED, PIXEL])
def test_a_background_per_frame(ctx, path, polarity):
    rng = np.random.default_rng(17)
    ctx.highlight_set_polarity(pc.POLARITIES[polarity])
    try:
        for t in range(0, 60, 7):
            frame, p = pc.mixed_random_case(t)
            frames, bgs = _backgrounds(frame, p.background, rng)
            got = _device_bg(ctx, frames, bgs, p, path)
            assert np.array_equal(got, pc.masks(frames, p, polarity, bgs)), t
    finally:
        ctx.highlight_set_polarity(0)


@pytest.mark.parametrize("polarity", POLS)
def test_queue_with_decoded_colour_frames_and_a_crop(ctx, polarity):
    """the queue's copying (submit / next) and zero-copy (slot_acquire / commit / next_view) forms on decoded
    3-channel frames with a crop, prepared on the device"""
    rng = np.random.default_rng(23)
    h, w, n, batch = 70, 120, 13, 4
    crop = (9, 4, 100, 60)
    frames = np.empty((n, h, w, 3), np.uint8)
    for i in range(n):
        f, bg = hl_cases.blob_frame(h, w, 950 + i, bgv=128, sigma=2.0, amp=70)
        frames[i] = np.stack([pc.mixed(f, bg), np.roll(f, 3, axis=1), rng.integers(0, 256, (h, w), dtype=np.uint8)],
                             axis=-1)
    prepared = fo.prepare_frames(frames, crop, fo.CHANNEL0)
    p = ho.canonical_params(np.full(prepared.shape[1:], 128, np.uint8))
    want = pc.masks(prepared, p, polarity)
    assert want.any()
    fb = h * w * 3
    ctx.highlight_set_polarity(pc.POLARITIES[polarity])
    _begin(ctx, p)
    try:
        ctx.highlight_queue_begin(2, batch, _cabi.FrameFormat.of((h, w, 3), fo.CHANNEL0, crop))
        got, i, k = [], 0, 0
        while i < n or ctx.highlight_queue_pending():
            while i < n and ctx.highlight_queue_pending() < 2:
                m = min(batch, n - i)
                if k % 2:
                    ctx.highlight_submit(frames[i:i + m])
                else:
                    slot = ctx.highlight_slot_acquire()
                    slot[:m, :fb] = frames[i:i + m].reshape(m, fb)
                    ctx.highlight_slot_commit(m)
                i += m
                k += 1
            if len(got) % 2:
                got.append(ctx.highlight_next().copy())
            else:
                got.append(np.array(ctx.highlight_next_view()))
                ctx.highlight_view_release()
        ctx.highlight_queue_end()
    finally:
        ctx.highlight_end()
        ctx.highlight_set_polarity(0)
    assert np.array_equal(np.concatenate(got), want)


@pytest.mark.parametrize("polarity", POLS)
def test_rolling_stream(polarity):
    """the rolling-median stream against the host chain (window order statistic by np.partition, then the restatement
    with the new d) and against its device building blocks"""
    h, w = SMALL
    window, mb = 7, 3
    n = 3 * (window + mb) + 4
    frames = make_frames(n, h, w, seed=90)
    if polarity == "bright":
        frames = (255 - frames).astype(np.uint8)  # the disks become bright
    p = fine_params(h, w)
    with _cabi.Context(0) as c:
        c.highlight_set_polarity(pc.POLARITIES[polarity])
        _begin(c, p)
        want = device_reference(c, frames, window)
        got = run_stream(c, frames, h, w, window, mb, "poll", seed=5)
        c.highlight_end()
    assert_same_results(got, want, what=polarity)
    bgs = host_backgrounds(frames, window)
    assert np.array_equal(want["masks"], pc.masks(frames, p, polarity, bgs))
    assert not np.array_equal(want["masks"], pc.masks(frames, p, "dark", bgs))


def test_state_and_argument_errors():
    frame, p = pc.mixed_random_case(1)
    with _cabi.Context(0) as c:
        lib = c._lib
        assert c.highlight_polarity() == 0  # the default
        for bad in (3, -1, 255):
            assert lib.cvvp_highlight_set_polarity(c.handle, bad) == ERR_INVALID
        assert c.highlight_polarity() == 0
        c.highlight_set_polarity(1)
        assert c.highlight_polarity() == 1
        _begin(c, p)  # this job takes "bright"
        assert lib.cvvp_highlight_set_polarity(c.handle, 2) == ERR_STATE
        assert lib.cvvp_highlight_set_polarity(c.handle, 0) == ERR_STATE
        assert c.highlight_polarity() == 1
        assert np.array_equal(c.highlight_frames(frame[None])[0], _want(frame, p, "bright"))
        c.highlight_end()
        c.highlight_set_polarity(2)  # a job begun after a change uses the new value
        _begin(c, p)
        assert np.array_equal(c.highlight_frames(frame[None])[0], _want(frame, p, "both"))
        _begin(c, p)  # beginning again while open re-takes the (unchanged) setting
        assert np.array_equal(c.highlight_frames(frame[None])[0], _want(frame, p, "both"))
        c.highlight_end()
        c.highlight_set_polarity(0)
        _begin(c, p)
        assert np.array_equal(c.highlight_frames(frame[None])[0], _want(frame, p, "dark"))
        c.highlight_end()
    with _cabi.Context(0) as other:  # a fresh context: every other context is left alone
        assert other.highlight_polarity() == 0
