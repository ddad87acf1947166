"""GPU parity of the rolling temporal median (cvvp_median_rolling_device, csrc/median_roll.cu) against the CPU oracle of
HistogramMedianAlgo taken over every frame's window: s(t) = min(max(t - W/2, 0), N - W), all N frames when N <= W,
upper median sorted[Weff/2]."""
import numpy as np
import pytest
import torch

from cvvidproc_b200 import _cabi

pytestmark = pytest.mark.gpu


def window_start(t, w, n):
    weff = min(w, n)
    return min(max(t - w // 2, 0), n - weff), weff


def rolling_oracle(frames, w, median):
    """B_t for every t: the oracle's median of each distinct window (windows repeat at the clamped ends)"""
    n = frames.shape[0]
    cache = {}
    out = []
    for t in range(n):
        s, weff = window_start(t, w, n)
        if s not in cache:
            cache[s] = median(frames[s : s + weff])
        out.append(cache[s])
    return np.stack(out)


def gpu_rolling(ctx, frames, w, t0=0, t1=None, pad=0):
    """frames (N, ...) uint8 -> backgrounds of frames [t0, t1) from the device; pad: extra bytes per frame row"""
    n = frames.shape[0]
    t1 = n if t1 is None else t1
    nelem = int(np.prod(frames.shape[1:]))
    stride = nelem + pad
    host = np.zeros((n, stride), np.uint8)
    host[:, :nelem] = frames.reshape(n, nelem)
    d = torch.from_numpy(host).cuda()
    out = torch.full((max(t1 - t0, 1), stride), 77, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.median_rolling_device(d.data_ptr(), n, nelem, stride, w, t0, t1, out.data_ptr(), stride)
    ctx.synchronize()
    got = out.cpu().numpy()[: t1 - t0]
    assert np.all(got[:, nelem:] == 77), "wrote beyond nelem"
    return got[:, :nelem].reshape((t1 - t0,) + frames.shape[1:])


WINDOWS = [1, 2, 3, 4, 7, 100, 101, 255, 256, 1000]


def _counts(w):
    return sorted({c for c in (1, w - 1, w, w + 1, 3 * w + 5) if c >= 1})


@pytest.mark.parametrize("w", WINDOWS)
def test_uniform_noise_every_window_and_length(gpu_ctx, oracle_median, w):
    rng = np.random.default_rng(w)
    for n in _counts(w):
        frames = rng.integers(0, 256, (n, 5, 37), dtype=np.uint8)  # 185 elements: two tiles, the second partial
        want = rolling_oracle(frames, w, oracle_median)
        got = gpu_rolling(gpu_ctx, frames, w)
        assert np.array_equal(got, want), f"W={w} N={n}: {(got != want).sum()} bytes differ"


@pytest.mark.parametrize("w", [2, 4, 100, 256, 1000])
def test_two_value_splits_at_even_windows(gpu_ctx, oracle_median, w):
    """half the window at one value, half at the other: the upper median is the larger one, and a one-frame move flips it"""
    n = 3 * w + 5
    rng = np.random.default_rng(100 + w)
    lo, hi = 40, 41
    frames = np.where(rng.integers(0, 2, (n, 3, 50)) == 0, lo, hi).astype(np.uint8)
    frames[:, 0, :] = np.where((np.arange(n) // 1) % 2 == 0, lo, hi)[:, None]  # exact 50/50 in every even window
    got = gpu_rolling(gpu_ctx, frames, w)
    assert np.array_equal(got, rolling_oracle(frames, w, oracle_median))
    if w % 2 == 0:
        assert np.all(got[:, 0, :] == hi)


@pytest.mark.parametrize("w", [1, 3, 7, 101, 255, 1000])
def test_constant_stacks_and_scene_cuts(gpu_ctx, oracle_median, w):
    n = 3 * w + 5
    rng = np.random.default_rng(200 + w)
    const = np.full((n, 4, 33), 123, np.uint8)
    assert np.array_equal(gpu_rolling(gpu_ctx, const, w), const)
    # a scene cut of 200 levels half-way, with sensor noise: the median walks up to 255 levels in one move
    cut = np.where(np.arange(n)[:, None, None] < n // 2, 20, 220) + rng.integers(-3, 4, (n, 4, 33))
    cut = np.clip(cut, 0, 255).astype(np.uint8)
    assert np.array_equal(gpu_rolling(gpu_ctx, cut, w), rolling_oracle(cut, w, oracle_median))
    # and from 255 down to 0
    edge = np.where(np.arange(n)[:, None, None] < n // 3, 255, 0).repeat(4, 1).repeat(33, 2).astype(np.uint8)
    assert np.array_equal(gpu_rolling(gpu_ctx, edge, w), rolling_oracle(edge, w, oracle_median))


def test_more_than_255_equal_values_in_a_window(gpu_ctx, oracle_median):
    """counts above 255 must not wrap (16-bit counts): 700 equal values and 300 others in a window of 1000"""
    w, n = 1000, 2400
    rng = np.random.default_rng(5)
    frames = np.full((n, 2, 64), 90, np.uint8)
    mask = rng.random((n, 2, 64)) < 0.3
    frames[mask] = rng.integers(0, 256, mask.sum(), dtype=np.uint8)
    frames[:, 1, :] = np.where(rng.random((n, 64)) < 0.7, 0, 255)  # 700 zeros vs 300 x 255
    assert np.array_equal(gpu_rolling(gpu_ctx, frames, w), rolling_oracle(frames, w, oracle_median))


def test_frames_of_641x479_and_padded_strides(gpu_ctx, oracle_median):
    """nelem not a multiple of 128, and a frame pitch larger than a frame"""
    rng = np.random.default_rng(9)
    n, w = 24, 7
    frames = (rng.integers(0, 30, (n, 479, 641)) + np.linspace(0, 200, n)[:, None, None]).astype(np.uint8)
    want = rolling_oracle(frames, w, oracle_median)
    assert np.array_equal(gpu_rolling(gpu_ctx, frames, w), want)
    assert np.array_equal(gpu_rolling(gpu_ctx, frames, w, pad=128 - (479 * 641) % 128), want)


@pytest.mark.parametrize("w", [2, 5, 16])
def test_colour_stacks_work_element_by_element(gpu_ctx, oracle_median, w):
    rng = np.random.default_rng(w)
    frames = rng.integers(0, 256, (3 * w + 5, 20, 30, 3), dtype=np.uint8)
    assert np.array_equal(gpu_rolling(gpu_ctx, frames, w), rolling_oracle(frames, w, oracle_median))


@pytest.mark.parametrize("w", [1, 4, 7, 101])
def test_sub_ranges_give_the_bytes_of_the_full_range(gpu_ctx, w):
    rng = np.random.default_rng(300 + w)
    n = 3 * w + 5
    frames = rng.integers(0, 256, (n, 6, 40), dtype=np.uint8)
    full = gpu_rolling(gpu_ctx, frames, w)
    cuts = [(0, n), (0, 1), (n - 1, n), (w // 2, w // 2 + 3)] + [tuple(sorted(rng.integers(0, n + 1, 2))) for _ in range(8)]
    for t0, t1 in cuts:
        if t0 == t1:
            continue
        assert np.array_equal(gpu_rolling(gpu_ctx, frames, w, t0, t1), full[t0:t1]), (t0, t1)


@pytest.mark.parametrize("w,n", [(5, 5), (7, 3), (256, 200), (1000, 1000)])
def test_window_covering_the_stack_equals_the_static_median(gpu_ctx, w, n):
    rng = np.random.default_rng(n)
    frames = rng.integers(0, 256, (n, 8, 48), dtype=np.uint8)
    nelem = 8 * 48
    d = torch.from_numpy(frames.reshape(n, nelem)).cuda()
    out = torch.empty(nelem, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    gpu_ctx.median_device(d.data_ptr(), n, nelem, nelem, out.data_ptr())
    gpu_ctx.synchronize()
    static = out.cpu().numpy().reshape(8, 48)
    got = gpu_rolling(gpu_ctx, frames, w)
    assert all(np.array_equal(g, static) for g in got)


def test_sample_of_windows_against_the_compiled_reference(gpu_ctx, ref_median):
    if ref_median is None:
        pytest.skip("oracle/_ref is not built here; the oracle tests above hold the windows to the CPU restatement")
    rng = np.random.default_rng(11)
    for w in (4, 101, 256):
        frames = rng.integers(0, 256, (3 * w + 5, 4, 40), dtype=np.uint8)
        got = gpu_rolling(gpu_ctx, frames, w)
        for t in rng.integers(0, frames.shape[0], 6):
            s, weff = window_start(int(t), w, frames.shape[0])
            assert np.array_equal(got[t], ref_median(frames[s : s + weff]))


def test_bad_arguments_are_rejected(gpu_ctx):
    d = torch.zeros((10, 128), dtype=torch.uint8, device="cuda")
    out = torch.zeros((10, 128), dtype=torch.uint8, device="cuda")
    p, o = d.data_ptr(), out.data_ptr()
    for args in ((p, 10, 128, 128, 0, 0, 10, o, 128), (p, 10, 128, 128, 65536, 0, 10, o, 128),
                 (p, 10, 128, 128, 3, -1, 5, o, 128), (p, 10, 128, 128, 3, 0, 11, o, 128), (p, 10, 128, 128, 3, 6, 5, o, 128),
                 (p, 10, 128, 100, 3, 0, 10, o, 128), (p, 10, 128, 128, 3, 0, 10, o, 100), (p, 0, 128, 128, 3, 0, 0, o, 128)):
        with pytest.raises(_cabi.CvvpError) as ei:
            gpu_ctx.median_rolling_device(*args)
        assert ei.value.code == -1, args
    gpu_ctx.median_rolling_device(p, 10, 128, 128, 65535, 3, 3, o, 128)  # empty range: nothing to do
