"""GPU tests of the rolling-background highlight stream (cvvp_highlight_rolling_*, csrc/highlight_rolling.cu) through its
C ABI, against two references:

  (A) a host chain: the order statistic k = min(Weff - 1, Weff * p // 100) of every frame's window
      s(t) = min(max(t - W // 2, 0), N - Weff) by np.partition, then the cv2 restatement of HighlightObjects with that
      background (oracle/highlight_oracle.py); masks are compared byte for byte;
  (B) the device building blocks the stream is made of: cvvp_median_rolling_device over a contiguous copy of the
      prepared frames, then cvvp_highlight_device_bg with bg_stride = the ring's pitch, in the same context.  This is the
      stream's arithmetic without the ring, the chunks and the result slots, so the stream must equal it byte for byte
      (masks, components, counts, labels).

The stream is driven through ctypes (ctx._lib) so that tests can pass what the Python binding does not: frame strides
larger than a frame, `next` with too little room, calls on a closed stream.  Every run also checks the ordering contract
against a model of the stream: which chunks exist after each push (the readiness rule
ready = 0 if received < W else received - ceil(W/2) + 1, chunks of at most max_batch frames), pending(), and what `next`
returns when nothing is pending."""
from __future__ import annotations

import ctypes as C
import dataclasses
from collections import deque

import cv2
import numpy as np
import pytest
import torch

from cvvidproc_b200 import _cabi, synth
from oracle import highlight_oracle as ho

pytestmark = pytest.mark.gpu

COMP = _cabi.Context.COMPONENT_DTYPE
OK, ERR_INVALID, ERR_STATE = 0, -1, -4


def pitch_of(npix):
    return (npix + 127) // 128 * 128


def fine_params(h, w):
    """thresholds of the reference with a 2x2 opening and small minimum sizes: masks follow small background changes"""
    return ho.HighlightParams(background=np.zeros((h, w), np.uint8), struct_element=np.ones((2, 2), np.uint8),
                              threshold=14, threshold_lo=7, threshold_hi=16, min_size_hyst=4, min_size_threshold=4,
                              width_border=0)


def canonical(h, w):
    return ho.canonical_params(np.zeros((h, w), np.uint8))


def highlight_begin(ctx, p):
    ctx.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                        p.min_size_hyst, p.min_size_threshold, p.width_border)


# ---------------------------------------------------------------------------------------------------------------------
# data that tells windows apart

def make_frames(n, h, w, seed, ndisks=2):
    """per-pixel random-walk brightness (with a block-coherent part, so that it survives the opening) and moving dark
    disks in the top quarter; below it 3x3 blocks of noise, new in every frame, from two clusters (40 and 200, +-15)
    of equal weight.  A block's order statistic jumps between the clusters whenever its count in the low cluster is
    near the rank, so a window shifted by one frame or a rank one off changes the masks of most frames"""
    rng = np.random.default_rng(seed)
    base = synth.synth_frames(0, n, w, h, seed, ndisks).astype(np.int32) - 20
    bh, bw = -(-h // 6), -(-w // 6)
    blocks = np.cumsum(rng.integers(-5, 6, (n, bh, bw), dtype=np.int8), axis=0, dtype=np.int16)
    walk = np.repeat(np.repeat(blocks, 6, axis=1), 6, axis=2)[:, :h, :w]
    walk = walk + np.cumsum(rng.integers(-2, 3, (n, h, w), dtype=np.int8), axis=0, dtype=np.int16)
    f = base + np.clip(walk, -60, 60)
    r0 = h // 4
    shape = (n, -(-(h - r0) // 3), -(-w // 3))
    noise = np.where(rng.random(shape) < 0.5, 40, 200) + rng.integers(-15, 16, shape)
    f[:, r0:] = np.repeat(np.repeat(noise, 3, axis=1), 3, axis=2)[:, : h - r0, :w]
    # a still border: the corners stay out of every mask, else FillHoles (seeded at a corner) turns a mask all white
    for edge in (np.s_[:, :2], np.s_[:, -2:], np.s_[:, :, :2], np.s_[:, :, -2:]):
        f[edge] = 128
    return np.clip(f, 0, 255).astype(np.uint8)


def window_starts(n, window, half=None, shift=0):
    weff = min(window, n)
    half = window // 2 if half is None else half
    return [min(max(min(max(t - half, 0), n - weff) + shift, 0), n - weff) for t in range(n)], weff


def host_backgrounds(frames, window, percent=50, shift=0, half=None, rank_delta=0, shortened=False):
    """(A)'s backgrounds; the keyword arguments make the wrong rules of the data guard"""
    n = frames.shape[0]
    out, cache = [], {}
    starts, weff = window_starts(n, window, half, shift)
    for t in range(n):
        if shortened:
            lo, hi = max(t - window // 2, 0), min(t - window // 2 + window, n)
        else:
            lo, hi = starts[t], starts[t] + weff
        if (lo, hi) not in cache:
            m = hi - lo
            k = min(m - 1, m * percent // 100) + rank_delta
            cache[(lo, hi)] = np.partition(frames[lo:hi], k, axis=0)[k]
        out.append(cache[(lo, hi)])
    return np.stack(out)


def host_masks(frames, bgs, p, only=None):
    idx = range(frames.shape[0]) if only is None else only
    return {t: ho.highlight_objects(frames[t].copy(), dataclasses.replace(p, background=bgs[t])) for t in idx}


def host_chain(frames, window, p, percent=50, only=None):
    masks = host_masks(frames, host_backgrounds(frames, window, percent), p, only)
    return masks if only is not None else np.stack([masks[t] for t in range(frames.shape[0])])


def assert_data_tells_windows_apart(frames, window, p, right_masks):
    """every wrong rule changes the masks of most frames whose background it changes"""
    n = frames.shape[0]
    right = host_backgrounds(frames, window)
    weff = min(window, n)
    k = min(weff - 1, weff // 2)
    rules = {"start+1": dict(shift=1), "start-1": dict(shift=-1), "shortened ends": dict(shortened=True)}
    if k + 1 <= weff - 1:
        rules["rank+1"] = dict(rank_delta=1)
    if k - 1 >= 0:
        rules["rank-1"] = dict(rank_delta=-1)
    if window % 2 == 0:
        rules["(W - 1) // 2 for W // 2"] = dict(half=(window - 1) // 2)
    for name, kw in rules.items():
        wrong = host_backgrounds(frames, window, **kw)
        hit = [t for t in range(n) if not np.array_equal(wrong[t], right[t])]
        if not hit:
            continue
        masks = host_masks(frames, wrong, p, hit)
        changed = sum(not np.array_equal(masks[t], right_masks[t]) for t in hit)
        assert changed * 2 > len(hit), f"W={window} N={n}: rule '{name}' changes {changed} of {len(hit)} masks it affects"


# ---------------------------------------------------------------------------------------------------------------------
# reference (B): the device building blocks

def device_reference(ctx, frames, window, max_comps=0, labels=False):
    n, h, w = frames.shape
    npix = h * w
    pitch = pitch_of(npix)
    host = np.zeros((n, pitch), np.uint8)
    host[:, :npix] = frames.reshape(n, npix)
    d = torch.from_numpy(host).cuda()
    bgs = torch.empty((n, pitch), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, pitch), dtype=torch.uint8, device="cuda")
    comps = torch.zeros(n * max(max_comps, 1) * COMP.itemsize, dtype=torch.uint8, device="cuda")
    ncomps = torch.zeros(n, dtype=torch.int32, device="cuda")
    lab = torch.zeros((n, npix), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.median_rolling_device(d.data_ptr(), n, npix, pitch, window, 0, n, bgs.data_ptr(), pitch)
    ctx.highlight_device_bg(d.data_ptr(), n, pitch, bgs.data_ptr(), pitch, out.data_ptr(), pitch,
                            comps.data_ptr() if max_comps else 0, max_comps, ncomps.data_ptr() if max_comps else 0,
                            lab.data_ptr() if labels else 0, npix)
    ctx.synchronize()
    res = {"masks": out.cpu().numpy()[:, :npix].reshape(n, h, w)}
    if max_comps:
        res["comps"] = comps.cpu().numpy().view(COMP).reshape(n, max_comps)
        res["ncomps"] = ncomps.cpu().numpy()
    if labels:
        res["labels"] = lab.cpu().numpy().reshape(n, h, w)
    return res


def assert_same_results(got, want, max_comps=0, what=""):
    bad = [t for t in range(want["masks"].shape[0]) if not np.array_equal(got["masks"][t], want["masks"][t])]
    assert not bad, f"{what}: masks of frames {bad[:10]} differ"
    if max_comps:
        assert np.array_equal(got["ncomps"], want["ncomps"]), what
        for t in range(want["masks"].shape[0]):
            k = min(int(want["ncomps"][t]), max_comps)
            assert np.array_equal(got["comps"][t, :k], want["comps"][t, :k]), f"{what}: components of frame {t}"
    if "labels" in want:
        assert np.array_equal(got["labels"], want["labels"]), what


# ---------------------------------------------------------------------------------------------------------------------
# the stream, through ctypes, checked against a model of its ordering contract

def ready_count(received, window, closed):
    if closed:
        return received
    return 0 if received < window else received - (window + 1) // 2 + 1


class Stream:
    """one cvvp_highlight_rolling_* stream and the model of what it has launched: push, close and next assert that the
    chunks, pending() and the results' frame indices follow the readiness rule"""

    def __init__(self, ctx, h, w, window, max_batch, fmt=None, max_comps=0, labels=False):
        self.ctx, self.lib = ctx, ctx._lib
        self.h, self.w, self.window, self.max_batch = h, w, window, max_batch
        self.max_comps, self.labels = max_comps, labels
        self.rc = self.lib.cvvp_highlight_rolling_begin(ctx.handle, window, max_batch, C.byref(fmt) if fmt else None,
                                                        max_comps, 1 if labels else 0)
        self.received = self.launched = self.returned = 0
        self.closed = False
        self.chunks = deque()  # (first, n) launched and not yet returned, by the model

    def err(self):
        return (self.lib.cvvp_last_error(self.ctx.handle) or b"").decode()

    def _model_launch(self):
        upto = ready_count(self.received, self.window, self.closed)
        while self.launched < upto:
            k = min(upto - self.launched, self.max_batch)
            self.chunks.append((self.launched, k))
            self.launched += k

    def push_raw(self, buf, n, stride):
        return self.lib.cvvp_highlight_rolling_push(self.ctx.handle, buf.ctypes.data, n, stride)

    def push(self, frames, stride=None):
        """frames (n, ...) uint8; stride > frame bytes: pushed from a buffer whose rows are that long"""
        n = frames.shape[0]
        fb = int(np.prod(frames.shape[1:]))
        stride = fb if stride is None else stride
        buf = np.full((n, stride), 0xEE, np.uint8)
        buf[:, :fb] = frames.reshape(n, fb)
        rc = self.push_raw(buf, n, stride)
        assert rc == OK, self.err()
        self.received += n
        self._model_launch()
        assert self.pending() == len(self.chunks)

    def close(self):
        rc = self.lib.cvvp_highlight_rolling_close(self.ctx.handle)
        assert rc == OK, self.err()
        self.closed = True
        self._model_launch()
        assert self.pending() == len(self.chunks)

    def pending(self):
        return self.lib.cvvp_highlight_rolling_pending(self.ctx.handle)

    def ready(self):
        rc = self.lib.cvvp_highlight_rolling_ready(self.ctx.handle)
        assert rc in (0, 1), self.err()
        return rc == 1

    def next_raw(self, max_n=None):
        h, w = self.h, self.w
        max_n = self.max_batch if max_n is None else max_n
        rows = max(max_n, 1)
        masks = np.full((rows, h, w), 0xA5, np.uint8)
        comps = np.zeros((rows, max(self.max_comps, 1)), COMP)
        ncomps = np.full(rows, -7, np.int32)
        lab = np.full((rows, h, w), -9, np.int32)
        first, n = C.c_longlong(-1), C.c_longlong(-1)
        rc = self.lib.cvvp_highlight_rolling_next(self.ctx.handle, masks.ctypes.data, h * w, max_n, C.byref(first),
                                                  C.byref(n), comps.ctypes.data if self.max_comps else None,
                                                  ncomps.ctypes.data if self.max_comps else None,
                                                  lab.ctypes.data if self.labels else None, h * w)
        k = int(n.value)
        return rc, int(first.value), k, {"masks": masks[:k], "comps": comps[:k], "ncomps": ncomps[:k], "labels": lab[:k]}

    def next(self, res):
        """one `next`, checked against the model; its results go into res (arrays over all frames)"""
        rc, first, k, got = self.next_raw()
        assert rc == OK, self.err()
        if not self.chunks:
            assert (first, k) == (self.launched, 0)
            return 0
        assert (first, k) == self.chunks.popleft()
        assert 1 <= k <= self.max_batch and first == self.returned
        self.returned += k
        assert self.pending() == len(self.chunks)
        for key, v in got.items():
            if key in res:
                res[key][first : first + k] = v
        return k

    def drain(self, res):
        while self.chunks:
            self.next(res)
        assert self.pending() == 0
        self.next(res)  # nothing pending: n = 0, first = frames launched so far

    def end(self):
        assert self.lib.cvvp_highlight_rolling_end(self.ctx.handle) == OK


def push_sizes(n, max_batch, seed):
    """a seeded sequence of push sizes in [1, max_batch] with runs of 1 and runs of max_batch"""
    rng = np.random.default_rng(seed)
    sizes, total = [], 0
    while total < n:
        mode = rng.integers(0, 3)
        for _ in range(int(rng.integers(1, 4))):
            s = 1 if mode == 0 else max_batch if mode == 1 else int(rng.integers(1, max_batch + 1))
            s = min(s, n - total)
            if s == 0:
                break
            sizes.append(s)
            total += s
    return sizes


def run_stream(ctx, pushed, h, w, window, max_batch, schedule="push", seed=0, fmt=None, max_comps=0, labels=False,
               stride=None, sizes=None):
    """pushed: the frames as the stream takes them (prepared, or decoded with fmt).  schedule: "close" drains only
    after close, "push" drains after every push (and checks the readiness rule), "poll" is a seeded interleaving that
    polls ready()"""
    n = pushed.shape[0]
    res = {"masks": np.full((n, h, w), 0x5A, np.uint8)}
    if max_comps:
        res["comps"] = np.zeros((n, max_comps), COMP)
        res["ncomps"] = np.full(n, -1, np.int32)
    if labels:
        res["labels"] = np.full((n, h, w), -1, np.int32)
    s = Stream(ctx, h, w, window, max_batch, fmt, max_comps, labels)
    assert s.rc == OK, s.err()
    rng = np.random.default_rng(seed)
    try:
        s.next(res)  # nothing pushed yet
        done = 0
        for size in sizes or push_sizes(n, max_batch, seed):
            s.push(pushed[done : done + size], stride)
            done += size
            if schedule == "push":
                s.drain(res)
                assert s.returned == ready_count(done, window, False)
            elif schedule == "poll":
                while s.chunks and rng.random() < 0.7:
                    if s.ready() or rng.random() < 0.3:
                        s.next(res)
        assert done == n
        s.close()
        s.drain(res)
        assert s.returned == n
    finally:
        s.end()
    return res


# ---------------------------------------------------------------------------------------------------------------------
# 1-3. ragged pushes, ring wrap, readiness, when `next` is called

MATRIX_WINDOWS = [1, 2, 3, 4, 7, 16, 33, 100]
SMALL = (29, 37)  # 1073 pixels: the ring's pitch is padded to 1152


def batches_for(window):
    return sorted({b for b in (1, 3, window - 1, window, window + 1, 64) if b >= 1})


@pytest.mark.parametrize("window", MATRIX_WINDOWS)
def test_ragged_pushes_and_ring_wrap(gpu_ctx, window):
    h, w = SMALL
    p = fine_params(h, w)
    batches = batches_for(window)
    n_long = 2 * (window + max(batches)) + 3  # more than two ring lengths for every max_batch
    counts = sorted({c for c in (1, window - 1, window, window + 1, 3 * window + 5, n_long) if c >= 1})
    video = make_frames(n_long, h, w, seed=window)
    highlight_begin(gpu_ctx, p)
    try:
        for n in counts:
            frames = video[:n]
            want = device_reference(gpu_ctx, frames, window)
            host = host_chain(frames, window, p)
            assert np.array_equal(want["masks"], host), f"(B) != (A) at W={window} N={n}"
            if n in (3 * window + 5, n_long):
                assert_data_tells_windows_apart(frames, window, p, host)
            for i, mb in enumerate(batches):
                schedule = ("push", "close", "poll")[(i + n) % 3]
                got = run_stream(gpu_ctx, frames, h, w, window, mb, schedule, seed=1000 * window + 10 * n + mb)
                assert_same_results(got, want, what=f"W={window} max_batch={mb} N={n} {schedule}")
    finally:
        gpu_ctx.highlight_end()


@pytest.mark.parametrize("window,max_batch", [(1, 3), (4, 4), (7, 3), (16, 5), (33, 64)])
def test_readiness_and_every_schedule_agree(gpu_ctx, window, max_batch):
    """drain after close (many slots allocated), after every push (slots reused), and a seeded interleaving that polls
    ready(): identical results, equal to (B)"""
    h, w = SMALL
    p = fine_params(h, w)
    n = 3 * (window + max_batch) + 2
    frames = make_frames(n, h, w, seed=50 + window)
    highlight_begin(gpu_ctx, p)
    try:
        want = device_reference(gpu_ctx, frames, window)
        runs = [run_stream(gpu_ctx, frames, h, w, window, max_batch, sched, seed=7) for sched in ("close", "push", "poll")]
        for got, sched in zip(runs, ("close", "push", "poll")):
            assert_same_results(got, want, what=sched)
        # single-frame pushes: the readiness rule frame by frame
        one = run_stream(gpu_ctx, frames, h, w, window, max_batch, "push", sizes=[1] * n)
        assert_same_results(one, want, what="pushes of one frame")
    finally:
        gpu_ctx.highlight_end()


# ---------------------------------------------------------------------------------------------------------------------
# 4. geometries and highlight paths

@pytest.mark.parametrize("h,w", [(29, 37), (96, 160), (479, 641), (1080, 1920)])
def test_geometries(gpu_ctx, h, w):
    window, mb, n = 5, 4, 17
    frames = make_frames(n, h, w, seed=h, ndisks=6 if w > 200 else 2)
    p = canonical(h, w)
    highlight_begin(gpu_ctx, p)
    try:
        want = device_reference(gpu_ctx, frames, window)
        got = run_stream(gpu_ctx, frames, h, w, window, mb, "poll", seed=h)
    finally:
        gpu_ctx.highlight_end()
    assert_same_results(got, want, what=f"{w}x{h}")
    sample = range(n) if h * w < 200_000 else sorted(np.random.default_rng(h).choice(n, 4, replace=False))
    host = host_chain(frames, window, p, only=sample)
    for t in sample:
        assert np.array_equal(want["masks"][t], host[t]), f"(B) != (A) at {w}x{h} frame {t}"
    assert any(want["masks"][t].any() for t in sample)


@pytest.mark.parametrize("variant", ["large", "small"])
def test_fused_variants_and_the_per_pixel_path(gpu_ctx, monkeypatch, variant):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    h, w = 479, 641
    window, mb, n = 5, 4, 15
    frames = make_frames(n, h, w, seed=3, ndisks=6)
    p = canonical(h, w)
    highlight_begin(gpu_ctx, p)
    try:
        want = device_reference(gpu_ctx, frames, window)
        fused = run_stream(gpu_ctx, frames, h, w, window, mb, "push")
        gpu_ctx.highlight_set_path(1)
        pixel = run_stream(gpu_ctx, frames, h, w, window, mb, "close")
    finally:
        gpu_ctx.highlight_end()
    assert_same_results(fused, want, what=f"fused {variant}")
    assert_same_results(pixel, want, what="per-pixel path")
    host = host_chain(frames, window, p, only=[0, 7, 14])
    for t in host:
        assert np.array_equal(want["masks"][t], host[t])


# ---------------------------------------------------------------------------------------------------------------------
# 5. percentiles

@pytest.mark.parametrize("percent", [0, 1, 50, 90, 100])
def test_percentiles(percent):
    h, w = SMALL
    window, mb = 7, 3
    n = 3 * (window + mb) + 4
    frames = make_frames(n, h, w, seed=80)
    p = fine_params(h, w)
    with _cabi.Context(0) as ctx:
        ctx.median_set_percentile(percent)
        highlight_begin(ctx, p)
        want = device_reference(ctx, frames, window)
        got = run_stream(ctx, frames, h, w, window, mb, "poll", seed=percent)
        ctx.highlight_end()
    assert_same_results(got, want, what=f"p={percent}")
    assert np.array_equal(want["masks"], host_chain(frames, window, p, percent))
    if percent == 50:
        with _cabi.Context(0) as fresh:
            highlight_begin(fresh, p)
            default = run_stream(fresh, frames, h, w, window, mb, "push")
            fresh.highlight_end()
        assert_same_results(default, got, what="explicit p = 50 vs a fresh context")


def test_a_new_stream_takes_the_percentile_set_between_streams():
    h, w = SMALL
    window, mb, n = 5, 4, 23
    frames = make_frames(n, h, w, seed=81)
    p = fine_params(h, w)
    with _cabi.Context(0) as ctx:
        ctx.median_set_percentile(10)
        highlight_begin(ctx, p)
        lo = run_stream(ctx, frames, h, w, window, mb, "push")
        ctx.median_set_percentile(90)
        hi = run_stream(ctx, frames, h, w, window, mb, "push")
        ctx.highlight_end()
    assert np.array_equal(lo["masks"], host_chain(frames, window, p, 10))
    assert np.array_equal(hi["masks"], host_chain(frames, window, p, 90))
    assert not np.array_equal(lo["masks"], hi["masks"])


# ---------------------------------------------------------------------------------------------------------------------
# 6. frame formats

def _formats(h, w):
    """(name, fmt, decoded frame shape, host preparation of a decoded frame)"""
    def gray(f, x, y):
        return cv2.cvtColor(np.ascontiguousarray(f[y : y + h, x : x + w]), cv2.COLOR_RGB2GRAY)

    return [
        ("as-is full width", _cabi.FrameFormat.of((h + 7, w), _cabi.FRAMES_AS_IS, (0, 3, w, h)), (h + 7, w),
         lambda f: f[3 : 3 + h]),
        ("rgb2gray crop", _cabi.FrameFormat.of((h + 6, w + 10, 3), _cabi.FRAMES_RGB2GRAY, (4, 2, w, h)), (h + 6, w + 10, 3),
         lambda f: gray(f, 4, 2)),
        ("channel0 crop", _cabi.FrameFormat.of((h + 5, w + 9, 3), _cabi.FRAMES_CHANNEL0, (9, 5, w, h)), (h + 5, w + 9, 3),
         lambda f: f[5 : 5 + h, 9 : 9 + w, 0]),
    ]


@pytest.mark.parametrize("which", range(3))
@pytest.mark.parametrize("padded", [False, True])
def test_frame_formats_equal_host_prepared_frames(gpu_ctx, which, padded):
    h, w = 96, 160
    window, mb = 5, 4
    n = 3 * (window + mb) + 3
    name, fmt, shape, prep = _formats(h, w)[which]
    rng = np.random.default_rng(which)
    gray = make_frames(n, shape[0], shape[1], seed=90 + which)
    decoded = gray if len(shape) == 2 else np.stack([gray, np.roll(gray, 5, axis=2), 255 - gray], axis=-1)
    decoded = np.ascontiguousarray(decoded)
    prepared = np.stack([np.ascontiguousarray(prep(f)) for f in decoded])
    in_bytes = int(np.prod(shape))
    p = fine_params(h, w)
    highlight_begin(gpu_ctx, p)
    try:
        sizes = push_sizes(n, mb, which)
        want = run_stream(gpu_ctx, prepared, h, w, window, mb, "push", sizes=sizes,
                          stride=h * w + 37 if padded else None)
        got = run_stream(gpu_ctx, decoded, h, w, window, mb, "poll", seed=int(rng.integers(1 << 30)), fmt=fmt,
                         sizes=sizes, stride=in_bytes + 64 if padded else None)
        ref = device_reference(gpu_ctx, prepared, window)
    finally:
        gpu_ctx.highlight_end()
    assert_same_results(want, ref, what="prepared frames")
    assert_same_results(got, want, what=name)


# ---------------------------------------------------------------------------------------------------------------------
# 7. components and labels

def _check_frame(mask, comps, ncomp, labels):
    n_cv, lab_cv, stats_cv, cent_cv = cv2.connectedComponentsWithStats(mask, connectivity=8, ltype=cv2.CV_32S)
    assert ncomp == n_cv - 1
    assert np.array_equal(labels != 0, mask != 0)
    # identical partition: the (gpu label, cv label) pairs form a bijection
    pairs = np.unique(np.stack([labels.ravel(), lab_cv.ravel()], axis=1), axis=0)
    assert not np.any((pairs[:, 0] == 0) != (pairs[:, 1] == 0))
    pairs = pairs[pairs[:, 0] != 0]
    assert len(pairs) == n_cv - 1
    assert len(np.unique(pairs[:, 0])) == n_cv - 1 and len(np.unique(pairs[:, 1])) == n_cv - 1
    to_cv = dict(map(tuple, pairs))
    prev_first = -1
    for k in range(min(ncomp, comps.shape[0])):
        c = comps[k]
        ys, xs = np.nonzero(labels == k + 1)
        assert c["area"] == len(xs) == stats_cv[to_cv[k + 1], cv2.CC_STAT_AREA]
        assert (c["x0"], c["y0"], c["x1"], c["y1"]) == (xs.min(), ys.min(), xs.max(), ys.max())
        assert c["sum_x"] == xs.sum() and c["sum_y"] == ys.sum()
        cx, cy = cent_cv[to_cv[k + 1]]
        assert abs(c["sum_x"] / c["area"] - cx) < 1e-9 and abs(c["sum_y"] / c["area"] - cy) < 1e-9
        # canonical numbering: components in the raster order of their first pixels
        first = ys[0] * mask.shape[1] + xs[ys == ys[0]].min()
        assert (c["first_y"], c["first_x"]) == divmod(first, mask.shape[1])
        assert first > prev_first
        prev_first = first


def _speckled(n, h, w, seed):
    """frames of make_frames, and some frames with a grid of 6x6 dark squares: far more than 64 components"""
    frames = make_frames(n, h, w, seed)
    for t in range(3, n, 7):
        for y in range(2, h - 8, 10):
            for x in range(2, w - 8, 10):
                frames[t, y : y + 6, x : x + 6] //= 4
    return frames


@pytest.mark.parametrize("max_comps", [1, 64])
@pytest.mark.parametrize("labels", [False, True])
def test_components_and_labels(gpu_ctx, max_comps, labels):
    h, w = 96, 160
    window, mb = 5, 4
    n = 3 * (window + mb) + 1
    frames = _speckled(n, h, w, seed=max_comps)
    p = fine_params(h, w)
    highlight_begin(gpu_ctx, p)
    try:
        want = device_reference(gpu_ctx, frames, window, max_comps, labels)
        got = run_stream(gpu_ctx, frames, h, w, window, mb, "poll", seed=max_comps, max_comps=max_comps, labels=labels)
    finally:
        gpu_ctx.highlight_end()
    assert want["ncomps"].max() > max(max_comps, 64)
    assert_same_results(got, want, max_comps, what=f"max_comps={max_comps} labels={labels}")
    assert np.array_equal(want["masks"], host_chain(frames, window, p))
    if labels:
        for t in (0, 3, n // 2, n - 1):
            _check_frame(got["masks"][t], got["comps"][t], int(got["ncomps"][t]), got["labels"][t])


# ---------------------------------------------------------------------------------------------------------------------
# 8. pooled buffers come back dirty

def _dirty_stream(ctx, h, w, window, mb):
    """a stream big enough for its ring, backgrounds and result slots to be parked in the pool when it ends, leaving 255
    and 0 frames in the ring, 255 backgrounds and 255 masks behind"""
    n = 3 * (window + mb)
    frames = np.full((n, h, w), 255, np.uint8)
    frames[::3] = 0
    s = Stream(ctx, h, w, window, mb)
    assert s.rc == OK
    res = {"masks": np.zeros((n, h, w), np.uint8)}
    for i in range(0, n, mb):
        s.push(frames[i : i + mb])
    s.close()
    s.drain(res)
    s.end()
    assert res["masks"][0].all()


@pytest.mark.parametrize("window,max_batch,dirty_window,dirty_batch", [(8, 16, 8, 16), (12, 12, 8, 16)])
def test_pooled_buffers_come_back_dirty(gpu_ctx, window, max_batch, dirty_window, dirty_batch):
    """320x240: ring (W + max_batch) x 76800 bytes and, at max_batch 16, backgrounds and result slots of 1.2 MB are all
    parked.  The first case takes them all back from the pool; the second only the ring (same W + max_batch)"""
    h, w = 240, 320
    n = 3 * (window + max_batch) + 5
    frames = make_frames(n, h, w, seed=window, ndisks=5)
    p = fine_params(h, w)
    highlight_begin(gpu_ctx, p)
    try:
        gpu_ctx._lib.cvvp_pool_trim()
        clean = run_stream(gpu_ctx, frames, h, w, window, max_batch, "close")
        gpu_ctx._lib.cvvp_pool_trim()
        _dirty_stream(gpu_ctx, h, w, dirty_window, dirty_batch)
        dirty = run_stream(gpu_ctx, frames, h, w, window, max_batch, "close")
        want = device_reference(gpu_ctx, frames, window)
    finally:
        gpu_ctx.highlight_end()
        gpu_ctx._lib.cvvp_pool_trim()
    assert_same_results(clean, want, what="after a trim")
    assert_same_results(dirty, clean, what="pooled buffers")


# ---------------------------------------------------------------------------------------------------------------------
# 9. state and error rules

def test_state_and_error_rules(gpu_ctx):
    h, w = SMALL
    window, mb = 5, 4
    n = 3 * (window + mb)
    frames = make_frames(n, h, w, seed=99)
    p = fine_params(h, w)
    lib, hd = gpu_ctx._lib, gpu_ctx.handle

    # no highlight parameters
    with _cabi.Context(0) as bare:
        assert Stream(bare, h, w, window, mb).rc == ERR_STATE
    highlight_begin(gpu_ctx, p)
    try:
        want = device_reference(gpu_ctx, frames, window)
        for args in ((0, mb, 0, 0), (65536, mb, 0, 0), (window, 0, 0, 0), (window, (1 << 20) + 1, 0, 0), (window, mb, 0, 1)):
            assert lib.cvvp_highlight_rolling_begin(hd, args[0], args[1], None, args[2], args[3]) == ERR_INVALID, args
        bad_crop = _cabi.FrameFormat.of((h + 4, w), _cabi.FRAMES_AS_IS, (0, 0, w, h + 1))
        colour = _cabi.FrameFormat.of((h, w, 3), _cabi.FRAMES_AS_IS)
        for fmt in (bad_crop, colour):
            assert lib.cvvp_highlight_rolling_begin(hd, window, mb, C.byref(fmt), 0, 0) == ERR_INVALID

        s = Stream(gpu_ctx, h, w, window, mb)
        assert s.rc == OK
        assert lib.cvvp_highlight_rolling_begin(hd, window, mb, None, 0, 0) == ERR_STATE  # begun twice
        res = {"masks": np.zeros((n, h, w), np.uint8)}
        buf = np.ascontiguousarray(frames[:mb + 1].reshape(mb + 1, h * w))
        assert s.push_raw(buf, 0, h * w) == ERR_INVALID
        assert s.push_raw(buf, mb + 1, h * w) == ERR_INVALID
        assert s.push_raw(buf, 1, h * w - 1) == ERR_INVALID
        assert s.pending() == 0
        # the refused calls uploaded nothing: the stream goes on as if they had not been made
        s.push(frames[:3])
        s.push(frames[3:7])
        assert s.chunks and s.chunks[0][1] >= 2
        rc = s.next_raw(max_n=s.chunks[0][1] - 1)[0]  # too little room: the chunk stays pending
        assert rc == ERR_INVALID and s.pending() == len(s.chunks)
        s.next(res)
        for i in range(7, n, mb):
            s.push(frames[i : i + mb])
        s.close()
        assert s.push_raw(buf, 1, h * w) == ERR_STATE
        assert lib.cvvp_highlight_rolling_close(hd) == ERR_STATE
        s.drain(res)
        assert np.array_equal(res["masks"], want["masks"])
        s.end()

        # end with chunks pending, then a new stream
        s = Stream(gpu_ctx, h, w, window, mb)
        for i in range(0, n, mb):
            s.push(frames[i : i + mb])
        assert s.pending() > 1
        s.end()
        assert lib.cvvp_highlight_rolling_pending(hd) == 0
        again = run_stream(gpu_ctx, frames, h, w, window, mb, "close")
        assert_same_results(again, want, what="after an end with chunks pending")

        # highlight_end while a stream is open releases it
        s = Stream(gpu_ctx, h, w, window, mb)
        s.push(frames[:mb])
        s.push(frames[mb : 2 * mb])
    finally:
        gpu_ctx.highlight_end()
    assert lib.cvvp_highlight_rolling_pending(hd) == 0
    assert s.push_raw(buf, 1, h * w) == ERR_STATE
    assert lib.cvvp_highlight_rolling_begin(hd, window, mb, None, 0, 0) == ERR_STATE
    highlight_begin(gpu_ctx, p)
    try:
        again = run_stream(gpu_ctx, frames, h, w, window, mb, "push")
    finally:
        gpu_ctx.highlight_end()
    assert_same_results(again, want, what="after highlight_end with a stream open")

    # closing a context with a stream open
    with _cabi.Context(0) as other:
        highlight_begin(other, p)
        s = Stream(other, h, w, window, mb)
        s.push(frames[:mb])
        s.push(frames[mb : 2 * mb])
    with _cabi.Context(0) as other:
        highlight_begin(other, p)
        again = run_stream(other, frames, h, w, window, mb, "poll")
        other.highlight_end()
    assert_same_results(again, want, what="after a context closed with a stream open")


# ---------------------------------------------------------------------------------------------------------------------
# 10. long windows

def host_backgrounds_long(frames, window, percent=50):
    """(A)'s backgrounds by exact (int64) per-element histograms updated window to window: np.partition over 4095
    frames for every distinct window would take minutes"""
    n = frames.shape[0]
    flat = frames.reshape(n, -1).astype(np.int64)
    e = np.arange(flat.shape[1])
    weff = min(window, n)
    k = min(weff - 1, weff * percent // 100)
    starts, _ = window_starts(n, window)
    hist = np.zeros((flat.shape[1], 256), np.int64)
    np.add.at(hist, (np.broadcast_to(e, (weff, e.size)), flat[:weff]), 1)
    cur, out, cache = 0, [], {}
    for t in range(n):
        s = starts[t]
        while cur < s:
            hist[e, flat[cur]] -= 1
            hist[e, flat[cur + weff]] += 1
            cur += 1
        if s not in cache:
            cache[s] = (np.cumsum(hist, axis=1) > k).argmax(axis=1).astype(np.uint8).reshape(frames.shape[1:])
        out.append(cache[s])
    return np.stack(out)


def test_long_window_through_the_stream(gpu_ctx):
    h, w = 8, 16
    window, mb = 4095, 1024
    n = 3 * window + 17
    frames = make_frames(n, h, w, seed=4095, ndisks=1)
    p = ho.HighlightParams(background=np.zeros((h, w), np.uint8), struct_element=np.ones((1, 1), np.uint8), threshold=14,
                           threshold_lo=7, threshold_hi=16, min_size_hyst=0, min_size_threshold=0, width_border=0)
    bgs = host_backgrounds_long(frames, window)
    for s in (0, 1000, n - window):  # the incremental histograms against np.partition
        assert np.array_equal(np.partition(frames[s : s + window], window // 2, axis=0)[window // 2],
                              bgs[min(s + window // 2, n - 1) if s else 0])
    host = host_masks(frames, bgs, p)
    highlight_begin(gpu_ctx, p)
    try:
        got = run_stream(gpu_ctx, frames, h, w, window, mb, "poll", seed=5)
    finally:
        gpu_ctx.highlight_end()
    bad = [t for t in range(n) if not np.array_equal(got["masks"][t], host[t])]
    assert not bad, f"masks of {len(bad)} frames differ, first {bad[:5]}"
    assert sum(host[t].any() for t in range(n)) > n // 4
