"""GPU parity of the percentile backgrounds (cvvp_median_set_percentile) in every median form against numpy: the result
is np.partition(stack, k, axis=0)[k] with k = min(N - 1, N p // 100) -- on chip, through the counting path and its
fallbacks, the streaming job (resident and folded), sharded worlds and the rolling median -- and p = 50 set explicitly
gives exactly what a fresh context and the stored reference hashes give."""
import hashlib
import importlib.util
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from cvvidproc_b200 import _cabi, sharded

pytestmark = pytest.mark.gpu

PS = [0, 1, 25, 49, 50, 51, 75, 99, 100]


def rank(n, p):
    return min(n - 1, n * p // 100)


def oracle(stack, p):
    """stack (N, ...) -> the percentile image"""
    k = rank(stack.shape[0], p)
    return np.partition(stack, k, axis=0)[k]


def mixed_stack(n, nelem, seed, p):
    """constant, two-level 50/50, rank-boundary splits for p, sensor noise, uniform noise and a scene cut"""
    rng = np.random.default_rng(seed)
    s = np.empty((n, nelem), np.uint8)
    q = nelem // 8
    s[:, :q] = 77                                                        # constant
    s[:, q:2 * q] = np.where(np.arange(n)[:, None] < n // 2, 30, 220)    # two levels, 50/50
    k = rank(n, p)
    s[:, 2 * q:3 * q] = np.where(np.arange(n)[:, None] < k, 16, 32)      # k low values: sorted[k] is the high one
    s[:, 3 * q:4 * q] = np.where(np.arange(n)[:, None] <= k, 0x51, 0x5E)  # k + 1 low values: sorted[k] is the low one
    s[:, 4 * q:6 * q] = np.clip(128 + rng.normal(0, 2, (n, 2 * q)), 0, 255).astype(np.uint8)  # sensor noise
    s[:, 6 * q:7 * q] = rng.integers(0, 256, (n, q), dtype=np.uint8)     # uniform noise: forces the fallbacks
    cut = np.where(np.arange(n)[:, None] < n // 3, 40, 200)              # scene cut
    s[:, 7 * q:] = np.clip(cut + rng.integers(-3, 4, (n, nelem - 7 * q)), 0, 255).astype(np.uint8)
    perm = rng.permutation(n)  # frame order is irrelevant to an order statistic: mix it
    return s[perm]


def device_select(ctx, stack, stride=None):
    n, nelem = stack.shape
    stride = stride or (nelem + 15) // 16 * 16
    t = torch.zeros((n, stride), dtype=torch.uint8, device="cuda")
    t[:, :nelem] = torch.from_numpy(np.ascontiguousarray(stack)).cuda()
    out = torch.full((stride + 4,), 77, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.median_device(t.data_ptr(), n, nelem, stride, out.data_ptr())
    ctx.synchronize()
    got = out.cpu().numpy()
    assert (got[nelem:] == 77).all(), "wrote beyond nelem"
    return got[:nelem]


@pytest.fixture
def pctx():
    ctx = _cabi.Context(0)
    yield ctx
    ctx.close()


# ---- device-resident form: on-chip select and the counting path ------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 100, 101, 255, 256, 1000, 1280])
def test_on_chip_select(pctx, n):
    nelem = 777  # ragged: the last tile is partial
    for p in PS:
        stack = mixed_stack(n, nelem, n * 131 + p, p)
        pctx.median_set_percentile(p)
        assert np.array_equal(device_select(pctx, stack), oracle(stack, p)), p


@pytest.mark.parametrize("n", [1281, 2048, 3000])
@pytest.mark.parametrize("window", ["1", "0"])
def test_counting_path(pctx, monkeypatch, n, window):
    monkeypatch.setenv("CVVP_MEDIAN_WINDOW", window)
    for p in PS:
        stack = mixed_stack(n, 1000, n + p, p)
        pctx.median_set_percentile(p)
        assert np.array_equal(device_select(pctx, stack), oracle(stack, p)), p


@pytest.mark.parametrize("n", [1, 33, 200, 1000])
@pytest.mark.parametrize("window", ["1", "0"])
def test_counting_path_forced_at_small_stacks(pctx, monkeypatch, n, window):
    monkeypatch.setenv("CVVP_MEDIAN_TWO_PASS", "1")
    monkeypatch.setenv("CVVP_MEDIAN_WINDOW", window)
    for p in PS:
        stack = mixed_stack(n, 640, n * 7 + p, p)
        pctx.median_set_percentile(p)
        assert np.array_equal(device_select(pctx, stack), oracle(stack, p)), p


def test_narrower_tile_variants(pctx, monkeypatch):
    # 2048 frames on chip need 64-byte tiles; CVVP_MEDIAN_LOG2S walks the 32- and 16-byte ones too
    monkeypatch.setenv("CVVP_MEDIAN_TWO_PASS", "0")
    for log2s, n in (("1", 2000), ("2", 700), ("3", 300)):
        monkeypatch.setenv("CVVP_MEDIAN_LOG2S", log2s)
        for p in (0, 10, 50, 90, 100):
            stack = mixed_stack(n, 400, n + p, p)
            pctx.median_set_percentile(p)
            assert np.array_equal(device_select(pctx, stack), oracle(stack, p)), (log2s, p)


# ---- streaming job from host memory ----------------------------------------------------------------------------------
@pytest.mark.parametrize("n,cap", [(300, None), (300, 16), (2000, 700), (40, 1)])
def test_streaming_job_resident_and_folded(pctx, monkeypatch, n, cap):
    if cap:
        monkeypatch.setenv("CVVP_MEDIAN_RESIDENT_MAX", str(cap))
    for p in PS:
        stack = mixed_stack(n, 9 * 131, n + p, p).reshape(n, 9, 131)
        pctx.median_set_percentile(p)
        assert np.array_equal(pctx.median(stack, chunk=97), oracle(stack, p)), p


def test_colour_push_source(pctx, monkeypatch):
    rng = np.random.default_rng(3)
    n = 120
    frames = rng.integers(0, 256, (n, 20, 24, 3), dtype=np.uint8)
    frames[: n // 4, :5] = 0  # a dark object over a quarter of the frames
    fmt = _cabi.FrameFormat.of(frames.shape[1:], _cabi.FRAMES_AS_IS, crop=(2, 3, 17, 11))
    crop = frames[:, 3:14, 2:19]
    for cap in (None, "32"):
        if cap:
            monkeypatch.setenv("CVVP_MEDIAN_RESIDENT_MAX", cap)
        for p in (0, 30, 50, 90, 100):
            pctx.median_set_percentile(p)
            pctx.median_begin(int(np.prod(crop.shape[1:])), n)
            for i in range(0, n, 25):
                pctx.median_push_source(frames[i:i + 25], fmt)
            got = pctx.median_finish(nelem=int(np.prod(crop.shape[1:]))).reshape(crop.shape[1:])
            assert np.array_equal(got, oracle(crop, p)), (cap, p)


# ---- sharded worlds (ranks = contexts of this process on one device) -------------------------------------------------
def _sharded(parts, nelem, p, form):
    world = len(parts)
    ctxs = [_cabi.Context(0) for _ in range(world)]
    jobs = []
    try:
        for c in ctxs:
            c.median_set_percentile(p)
        stride = (nelem + 127) // 128 * 128
        most = max(1, max(fr.shape[0] for fr in parts))
        stacks = []
        for r, fr in enumerate(parts):
            jobs.append(sharded.ShardedMedian(ctxs[r], nelem, r, world, max_rank_frames=most))
            t = torch.zeros((max(fr.shape[0], 1), stride), dtype=torch.uint8, device="cuda:0")
            if fr.shape[0]:
                t[: fr.shape[0], :nelem] = torch.from_numpy(np.ascontiguousarray(fr)).cuda()
            stacks.append(t)
        torch.cuda.synchronize()
        sharded.ShardedMedian.connect_local(jobs)

        def walk(phases):
            for ph in phases:
                for r, job in enumerate(jobs):
                    job.phase(ph, stacks[r].data_ptr(), parts[r].shape[0], stride)
                for c in ctxs:
                    c.synchronize()

        if form == "two_round":
            walk(range(4))
        else:
            walk((4, 5))
            left = {job.ctx.median_shard_unresolved() for job in jobs}
            assert len(left) == 1
            if left.pop():
                walk(range(4) if form == "window_then_full" else range(10, 14))
        return [job.ctx.copy_to_host(job.result_ptr(), nelem) for job in jobs]
    finally:
        for job in jobs:
            job.close()
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("form", ["window", "window_then_full", "two_round"])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_shard_worlds(world, form):
    n, nelem = 1500, 1000
    for p in (0, 1, 49, 50, 51, 99, 100):
        stack = mixed_stack(n, nelem, world * 100 + p, p)
        # ragged chunks, an empty one where the world allows
        cuts = np.sort(np.random.default_rng(p).choice(np.arange(1, n), world - 1, replace=False)) if world > 1 else []
        bounds = [0, *cuts, n]
        parts = [stack[bounds[r]:bounds[r + 1]] for r in range(world)]
        if world >= 3:
            parts = [parts[0], stack[:0], np.concatenate(parts[1:])] + [stack[:0]] * (world - 3)
        want = oracle(stack, p)
        for got in _sharded(parts, nelem, p, form):
            assert np.array_equal(got, want), (p, form)


# ---- rolling median --------------------------------------------------------------------------------------------------
def rolling_oracle(frames, w, p):
    n = frames.shape[0]
    weff = min(w, n)
    out = []
    for t in range(n):
        s = min(max(t - w // 2, 0), n - weff)
        out.append(oracle(frames[s:s + weff], p))
    return np.stack(out)


def gpu_rolling(ctx, frames, w, t0=0, t1=None):
    n = frames.shape[0]
    t1 = n if t1 is None else t1
    nelem = int(np.prod(frames.shape[1:]))
    d = torch.from_numpy(np.ascontiguousarray(frames.reshape(n, nelem))).cuda()
    out = torch.full((max(t1 - t0, 1), nelem), 77, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.median_rolling_device(d.data_ptr(), n, nelem, nelem, w, t0, t1, out.data_ptr(), nelem)
    ctx.synchronize()
    return out.cpu().numpy()[: t1 - t0].reshape((t1 - t0,) + frames.shape[1:])


@pytest.mark.parametrize("w", [1, 2, 5, 25, 101])
def test_rolling_windows(pctx, w):
    for n in sorted({c for c in (1, w - 1, w, w + 1, 3 * w + 5) if c >= 1}):
        for p in PS:
            frames = mixed_stack(n, 200, w * 1000 + n + p, p).reshape(n, 8, 25)
            pctx.median_set_percentile(p)
            want = rolling_oracle(frames, w, p)
            assert np.array_equal(gpu_rolling(pctx, frames, w), want), (n, p)
            if n >= 3:
                t0, t1 = n // 3, n - n // 4
                assert np.array_equal(gpu_rolling(pctx, frames, w, t0, t1), want[t0:t1]), (n, p, t0, t1)


# ---- the setting itself ----------------------------------------------------------------------------------------------
def test_set_get_and_state_rules(pctx):
    assert pctx.median_percentile() == 50
    for p in (0, 100, 37):
        pctx.median_set_percentile(p)
        assert pctx.median_percentile() == p
    for bad in (-1, 101, 1000):
        with pytest.raises(_cabi.CvvpError) as ei:
            pctx.median_set_percentile(bad)
        assert ei.value.code == -1
        assert pctx.median_percentile() == 37
    frames = mixed_stack(64, 300, 1, 90)

    def refused():
        with pytest.raises(_cabi.CvvpError) as ei:
            pctx.median_set_percentile(90)
        assert ei.value.code == -4
        assert pctx.median_percentile() == 37

    # a streaming job keeps the percentile it began with
    pctx.median_begin(300, 64)
    pctx.median_push(frames[:32])
    refused()
    pctx.median_push(frames[32:])
    assert np.array_equal(pctx.median_finish(nelem=300), oracle(frames, 37))
    pctx.median_set_percentile(90)  # the job is over
    pctx.median_begin(300, 64)
    refused_at = pctx.median_percentile()
    pctx.median_abort()
    assert refused_at == 90
    pctx.median_set_percentile(37)
    # a sharded job
    pctx.median_shard_begin(300, 0, 1)
    refused()
    pctx.median_shard_end()
    # a rolling stream
    pctx.highlight_begin(np.zeros((8, 8), np.uint8), np.ones((3, 3), np.uint8), 10, 5, 15, 1, 1)
    pctx.highlight_rolling_begin(5, 4)
    refused()
    pctx.highlight_rolling_end()
    pctx.highlight_end()
    # the device-resident forms read the setting at the call
    pctx.median_set_percentile(0)
    lo = device_select(pctx, frames)
    pctx.median_set_percentile(100)
    hi = device_select(pctx, frames)
    assert np.array_equal(lo, frames.min(axis=0)) and np.array_equal(hi, frames.max(axis=0))


# ---- p = 50 is the upper median, byte for byte -----------------------------------------------------------------------
def _golden_cases():
    gdir = Path(__file__).parent / "golden"
    spec = importlib.util.spec_from_file_location("make_golden", gdir / "make_golden.py")
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return [(case, mg.case_input(case)) for case in json.loads((gdir / "median_golden.json").read_text())
            if not case.get("bin_bytes")]


def test_explicit_50_equals_a_fresh_context_and_the_golden_hashes(pctx, monkeypatch):
    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    fresh = _cabi.Context(0)
    try:
        pctx.median_set_percentile(0)
        pctx.median_set_percentile(50)
        for case, frames in _golden_cases():
            n = frames.shape[0]
            want = case["output_sha256"]
            flat = frames.reshape(n, -1)
            assert sha(fresh.median(frames)) == want, case["name"]
            assert sha(pctx.median(frames)) == want, case["name"]
            assert sha(device_select(pctx, flat)) == want, case["name"]
            assert sha(gpu_rolling(pctx, frames, n, 0, 1)[0]) == want, case["name"]  # one window = the whole stack
            assert sha(_sharded([flat[: n // 2], flat[n // 2:]], flat.shape[1], 50, "window")[0]) == want, case["name"]
            with monkeypatch.context() as m:
                m.setenv("CVVP_MEDIAN_RESIDENT_MAX", "7")
                assert sha(pctx.median(frames)) == want, case["name"]  # folded into value histograms
            with monkeypatch.context() as m:
                m.setenv("CVVP_MEDIAN_TWO_PASS", "1")
                assert sha(device_select(pctx, flat)) == want, case["name"]
    finally:
        fresh.close()
