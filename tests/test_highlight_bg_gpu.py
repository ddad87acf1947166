"""GPU parity of the highlight stage with a background per frame (cvvp_highlight_device_bg) against the cv2 restatement
of highlight_objects_algo.cpp run with each frame's own background, on both builds of the fused kernel and the
per-pixel kernels; bg_stride = 0 is cvvp_highlight_device byte for byte, and the components are those of
cvvp_highlight_device_cc run with the same background."""
import dataclasses

import numpy as np
import pytest
import torch

import hl_cases
from oracle import highlight_oracle as ho

pytestmark = pytest.mark.gpu

FUSED, PIXEL = 0, 1


def _begin(ctx, p):
    ctx.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                        p.min_size_hyst, p.min_size_threshold, p.width_border)


def _backgrounds(frame, bg, rng):
    """three frames, each with a background of its own: the case's, a shifted copy, a noisy copy"""
    frames = np.stack([frame, frame, np.roll(frame, 1, axis=1)])
    bgs = np.stack([bg, np.clip(bg.astype(int) + 9, 0, 255).astype(np.uint8),
                    np.clip(bg.astype(int) + rng.integers(-6, 7, bg.shape), 0, 255).astype(np.uint8)])
    return frames, bgs


def _device_bg(ctx, frames, bgs, p, path=FUSED, bg_stride=None, comps=0, pad=16):
    """masks (and components) of cvvp_highlight_device_bg; frame / background / mask pitches padded to 16 bytes"""
    n, h, w = frames.shape
    npix = h * w
    pitch = (npix + pad - 1) // pad * pad
    def dev(a):
        host = np.zeros((a.shape[0], pitch), np.uint8)
        host[:, :npix] = a.reshape(a.shape[0], npix)
        return torch.from_numpy(host).cuda()
    d_f, d_b = dev(frames), dev(bgs)
    d_o = torch.zeros((n, pitch), dtype=torch.uint8, device="cuda")
    d_c = torch.zeros((n, max(comps, 1) * 48), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    _begin(ctx, p)
    try:
        ctx.highlight_set_path(path)
        ctx.highlight_device_bg(d_f.data_ptr(), n, pitch, d_b.data_ptr(), pitch if bg_stride is None else bg_stride,
                                d_o.data_ptr(), pitch, d_c.data_ptr() if comps else 0, comps, d_n.data_ptr() if comps else 0)
        ctx.synchronize()
    finally:
        ctx.highlight_end()
    masks = d_o.cpu().numpy()[:, :npix].reshape(n, h, w)
    if not comps:
        return masks
    c = np.frombuffer(d_c.cpu().numpy().tobytes(), ctx.COMPONENT_DTYPE).reshape(n, comps)
    return masks, c, d_n.cpu().numpy()


def _oracle(frames, bgs, p):
    return np.stack([ho.highlight_objects(f.copy(), dataclasses.replace(p, background=b)) for f, b in zip(frames, bgs)])


ADV = hl_cases.adversarial_cases()
VARIANTS = ["large", "small"]


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("case", ADV, ids=[c[0] for c in ADV])
def test_adversarial_cases_with_a_background_per_frame(gpu_ctx, monkeypatch, variant, case):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    _, frame, p = case
    frames, bgs = _backgrounds(frame, p.background, np.random.default_rng(1))
    got = _device_bg(gpu_ctx, frames, bgs, p)
    want = _oracle(frames, bgs, p)
    assert np.array_equal(got, want), f"{(got != want).sum()} pixels differ"


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("t", range(0, 60, 3))
def test_random_cases_with_a_background_per_frame(gpu_ctx, monkeypatch, variant, t):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    frame, p = hl_cases.random_case(t)
    frames, bgs = _backgrounds(frame, p.background, np.random.default_rng(t))
    assert np.array_equal(_device_bg(gpu_ctx, frames, bgs, p), _oracle(frames, bgs, p))


@pytest.mark.parametrize("t", range(0, 60, 5))
def test_pixel_path_with_a_background_per_frame(gpu_ctx, t):
    frame, p = hl_cases.random_case(t)
    frames, bgs = _backgrounds(frame, p.background, np.random.default_rng(t))
    assert np.array_equal(_device_bg(gpu_ctx, frames, bgs, p, PIXEL), _oracle(frames, bgs, p))


@pytest.mark.parametrize("case", ADV[::3], ids=[c[0] for c in ADV[::3]])
def test_pixel_path_adversarial_cases(gpu_ctx, case):
    _, frame, p = case
    frames, bgs = _backgrounds(frame, p.background, np.random.default_rng(2))
    assert np.array_equal(_device_bg(gpu_ctx, frames, bgs, p, PIXEL), _oracle(frames, bgs, p))


@pytest.mark.parametrize("hw", [(40, 64), (33, 96), (21, 128)])
def test_word_aligned_widths_take_the_wide_loads(gpu_ctx, hw):
    """W % 32 == 0 and 16-byte pitches: the fused kernel's 128-bit loads read every frame's own background"""
    h, w = hw
    rng = np.random.default_rng(h)
    frame, bg = hl_cases.blob_frame(h, w, 400 + h, sigma=2.0, amp=70)
    for p in (ho.canonical_params(bg), ho.HighlightParams(bg, np.ones((3, 2), np.uint8), -1, 9, 14, 10, 30, 5)):
        frames, bgs = _backgrounds(frame, bg, rng)
        assert np.array_equal(_device_bg(gpu_ctx, frames, bgs, p), _oracle(frames, bgs, p))
        # a pitch that is not a multiple of 16 takes the byte path: same masks
        assert np.array_equal(_device_bg(gpu_ctx, frames, bgs, p, pad=1), _oracle(frames, bgs, p))


@pytest.mark.parametrize("path", [FUSED, PIXEL])
def test_zero_stride_is_the_shared_background(gpu_ctx, path):
    from cvvidproc_b200 import synth

    bgf = synth.synth_frames(0, 1, 160, 96, 7, 8)[0]
    frames = synth.synth_frames(10, 12, 160, 96, 7, 8)
    for p in (ho.canonical_params(bgf), ho.HighlightParams(bgf, np.ones((3, 3), np.uint8), -1, 5, 12, 4, 8, 5)):
        got = _device_bg(gpu_ctx, frames, bgf[None], p, path, bg_stride=0)
        d = torch.from_numpy(frames.reshape(12, -1)).cuda()
        o = torch.zeros_like(d)
        torch.cuda.synchronize()
        _begin(gpu_ctx, p)
        try:
            gpu_ctx.highlight_set_path(path)
            gpu_ctx.highlight_device(d.data_ptr(), 12, 160 * 96, o.data_ptr(), 160 * 96)
            gpu_ctx.synchronize()
        finally:
            gpu_ctx.highlight_end()
        assert np.array_equal(got, o.cpu().numpy().reshape(12, 96, 160))


def test_components_equal_those_of_the_cc_entry_point(gpu_ctx):
    rng = np.random.default_rng(4)
    for t in (1, 8, 22):
        frame, p = hl_cases.random_case(t)
        frames, bgs = _backgrounds(frame, p.background, rng)
        masks, comps, ncomps = _device_bg(gpu_ctx, frames, bgs, p, comps=64)
        for i in range(3):
            _begin(gpu_ctx, dataclasses.replace(p, background=bgs[i]))
            try:
                m, c, n = gpu_ctx.highlight_frames_cc(frames[i : i + 1], max_comps=64)
            finally:
                gpu_ctx.highlight_end()
            assert np.array_equal(masks[i], m[0])
            assert ncomps[i] == n[0]
            k = min(int(n[0]), 64)
            assert np.array_equal(comps[i, :k], c[0, :k])
