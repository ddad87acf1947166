"""GPU tests of the rolling median kernel (cvvp_median_rolling_device, csrc/median_roll.cu) beyond
test_median_rolling_gpu.py: windows of up to 65535 frames, where the 16-bit bin counts packed two to a word reach their
limit, and the launch's chunk layouts (nchunks = min(ceil(12 * SMs / tiles), T / Weff)) crossed with sub-ranges whose ends
fall on the boundaries where the windows stop being clamped.  The bar is the order statistic
k = min(Weff - 1, Weff * p // 100) of each frame's window s(t) = min(max(t - W // 2, 0), N - Weff), computed on the host."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROLL_E = 128  # elements per CTA of median_roll_kernel


def window_starts(n, window):
    weff = min(window, n)
    return [min(max(t - window // 2, 0), n - weff) for t in range(n)], weff


def rank(weff, percent):
    return min(weff - 1, weff * percent // 100)


def oracle_partition(frames, window, percent=50):
    """np.partition over every distinct window"""
    starts, weff = window_starts(frames.shape[0], window)
    k = rank(weff, percent)
    cache = {}
    for s in starts:
        if s not in cache:
            cache[s] = np.partition(frames[s : s + weff], k, axis=0)[k]
    return np.stack([cache[s] for s in starts])


def oracle_histogram(frames, window, percent=50):
    """the same order statistics from exact int64 per-element histograms, updated from one distinct window to the next:
    for windows of tens of thousands of frames np.partition over every distinct window is too slow"""
    n = frames.shape[0]
    flat = frames.reshape(n, -1)
    ne = flat.shape[1]
    e = np.arange(ne)
    starts, weff = window_starts(n, window)
    k = rank(weff, percent)
    hist = np.bincount((flat[:weff].astype(np.int64) + 256 * e).ravel(), minlength=ne * 256).reshape(ne, 256)
    cur, cache = 0, {}
    for s in starts:
        while cur < s:
            hist[e, flat[cur]] -= 1
            hist[e, flat[cur + weff]] += 1
            cur += 1
        if s not in cache:
            cache[s] = (np.cumsum(hist, axis=1) > k).argmax(axis=1).astype(np.uint8)
    return np.stack([cache[s] for s in starts]).reshape(frames.shape)


def run(ctx, d_frames, n, nelem, window, t0, t1, pad=61, extra_rows=2):
    """backgrounds of [t0, t1) from frames already on the device (stride nelem + pad); checks that nothing beyond nelem in
    a row, and no row beyond t1 - t0, was written"""
    stride = nelem + pad
    rows = t1 - t0
    out = torch.full((rows + extra_rows, stride), 0x77, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.median_rolling_device(d_frames.data_ptr(), n, nelem, stride, window, t0, t1, out.data_ptr(), stride)
    ctx.synchronize()
    got = out.cpu().numpy()
    assert np.all(got[:rows, nelem:] == 0x77), "wrote beyond nelem"
    assert np.all(got[rows:] == 0x77), "wrote beyond t1"
    return got[:rows, :nelem]


def upload(frames, pad=61):
    n = frames.shape[0]
    nelem = int(np.prod(frames.shape[1:]))
    host = np.full((n, nelem + pad), 0xC3, np.uint8)
    host[:, :nelem] = frames.reshape(n, nelem)
    return torch.from_numpy(host).cuda(), nelem


# ---------------------------------------------------------------------------------------------------------------------
# windows above 1000: the packed 16-bit counts at their limit

def long_window_columns(window, seed):
    """N = W + 37 frames of 200 elements (two tiles, the second partial)"""
    rng = np.random.default_rng(seed)
    n = window + 37
    f = rng.integers(0, 256, (n, 200), dtype=np.uint8)
    f[:, 0] = 100  # every value in an even bin (low half of its word): the count reaches W, moves enter and leave 100
    f[:, 1] = 101  # the same in an odd bin (high half)
    f[:, 2] = 100
    f[0, 2] = 7  # W - 1 -> W across the first move
    f[:, 3] = 101
    f[0, 3] = 250  # the same in the high half
    f[:, 4] = 100
    f[-1, 4] = 3  # W -> W - 1 across the last move
    f[:, 5] = np.where(np.arange(n) % 2 == 0, 100, 101)  # both halves of one word near W / 2
    f[:, 6] = 0
    f[:, 7] = 255
    f[:, 8] = 255
    f[: n // 2, 8] = 254
    f[:, 9] = 0
    f[0, 9] = 1
    f[:, 10:30] = rng.integers(0, 2, (n, 20))  # bins 0 / 1
    f[:, 30:50] = rng.integers(254, 256, (n, 20))  # bins 254 / 255
    f[:, 50:70] = np.where(rng.random((n, 20)) < 0.5, 0, 255)
    # near-even splits that a single move tips: exactly half of the first window at 0, the rest at 255
    f[:, 70:80] = np.where(np.arange(n)[:, None] < window // 2, 0, 255)
    f[:, 80:100] = np.clip(128 + np.cumsum(rng.integers(-1, 2, (n, 20)), axis=0) // 64, 0, 255)  # slow walk
    return f


@pytest.mark.parametrize("percent", [0, 50, 100])
@pytest.mark.parametrize("window", [1023, 1024, 4095, 65534, 65535])
def test_windows_up_to_65535(gpu_ctx, window, percent):
    frames = long_window_columns(window, seed=window + percent)
    n = frames.shape[0]
    want = oracle_histogram(frames, window, percent)
    if window <= 4095:
        assert np.array_equal(want, oracle_partition(frames, window, percent))
    d, nelem = upload(frames)
    gpu_ctx.median_set_percentile(percent)
    try:
        got = run(gpu_ctx, d, n, nelem, window, 0, n)
        bounds = sorted({window // 2, window // 2 + 1, n - window + window // 2, n - window + window // 2 + 1, n - 1})
        for t0 in bounds:
            assert np.array_equal(run(gpu_ctx, d, n, nelem, window, t0, n), got[t0:]), t0
    finally:
        gpu_ctx.median_set_percentile(50)
    bad = np.nonzero((got != want).any(axis=0))[0]
    assert bad.size == 0, f"W={window} p={percent}: columns {bad[:10].tolist()} differ"
    # the constant columns hold their value whatever the percentile
    assert np.all(got[:, 0] == 100) and np.all(got[:, 1] == 101) and np.all(got[:, 6] == 0) and np.all(got[:, 7] == 255)


# ---------------------------------------------------------------------------------------------------------------------
# chunk layouts crossed with sub-ranges on the clamp boundaries

def launch_layout(sm_count, nelem, t, weff):
    """(outputs per chunk, chunks) of median_roll_launch for t outputs"""
    tiles = -(-nelem // ROLL_E)
    nchunks = min(-(-12 * sm_count // tiles), max(t // weff, 1), 65535)
    chunk = -(-t // max(nchunks, 1))
    return chunk, -(-t // chunk)


def layouts(sm):
    target = 12 * sm
    # (name, window, tiles, frames, check on the full range's (chunk, nchunks))
    return [
        ("one output per chunk", 1, 1, 40, lambda c, k: c == 1),
        ("two outputs per chunk", 2, 1, 40, lambda c, k: c == 2),
        ("about Weff outputs", 7, 2, 60, lambda c, k: 7 <= c <= 9),
        ("far more than Weff", 4, -(-target // 2), 100, lambda c, k: c == 50 and k == 2),
        ("around 12 SMs / 3 tiles", 5, target // 3 - 1, 61, lambda c, k: c >= 15 and k >= 3),
        ("single chunk", 4, target, 60, lambda c, k: k == 1),
    ]


@pytest.mark.parametrize("case", range(6))
def test_chunk_layouts_and_clamp_boundaries(gpu_ctx, case):
    sm = gpu_ctx.sm_count
    name, window, tiles, n, check = layouts(sm)[case]
    nelem = tiles * ROLL_E - 29  # the last tile is partial
    rng = np.random.default_rng(case)
    frames = rng.integers(0, 256, (n, nelem), dtype=np.uint8)
    frames[:, : nelem // 2] //= 16  # half the elements in 16 levels: ties in every window
    weff = min(window, n)
    assert check(*launch_layout(sm, nelem, n, weff)), (name, launch_layout(sm, nelem, n, weff))
    want = oracle_partition(frames, window)
    d, _ = upload(frames)
    full = run(gpu_ctx, d, n, nelem, window, 0, n)
    assert np.array_equal(full, want), name
    half = window // 2
    points = sorted({min(max(v, 0), n) for v in (0, half - 1, half, half + 1, n - weff + half - 1, n - weff + half,
                                                 n - weff + half + 1, n)})
    for i, t0 in enumerate(points):
        for t1 in points[i + 1 :]:
            got = run(gpu_ctx, d, n, nelem, window, t0, t1)
            assert np.array_equal(got, full[t0:t1]), (name, t0, t1, launch_layout(sm, nelem, t1 - t0, weff))
