"""GPU tests of the component statistics through the C ABI (cvvp_highlight_set_component_stats): every record equals
the numpy reference of tests/test_component_stats_cpu.py computed from the returned label image (or the mask's
canonical labelling), the frames and the backgrounds, exactly; with statistics off, masks, counts and the plain record
are byte-identical to the same job with them on.  Covers the hl_cases in all three polarities, both fused builds, the
128-bit and byte paths with Otsu, per-frame backgrounds, an all-foreground frame, more components than records, more
frames than are in flight, the queue (copying and zero-copy, decoded colour frames with a crop), the rolling stream,
the in-place rejection and the setting's state errors."""
import numpy as np
import pytest
import torch

import hl_cases
import polarity_cases as pc
from cvvidproc_b200 import _cabi
from oracle import frames_oracle as fo
from oracle import highlight_oracle as ho
from test_component_stats_cpu import canonical_labels, reference_stats
from test_highlight_rolling_stream_gpu import SMALL, fine_params, host_backgrounds, make_frames

pytestmark = pytest.mark.gpu

POLS = ["dark", "bright", "both"]
ERR_INVALID, ERR_STATE = -1, -4


@pytest.fixture(scope="module")
def ctx():
    c = _cabi.Context(0)  # a context of its own: the statistics and the polarity are settings of the context
    yield c
    c.close()


def _begin(ctx, p, polarity="dark", stats=True):
    ctx.highlight_set_polarity(pc.POLARITIES[polarity])
    ctx.highlight_set_component_stats(stats)
    ctx.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                        p.min_size_hyst, p.min_size_threshold, p.width_border)


def _end(ctx):
    ctx.highlight_end()
    ctx.highlight_set_polarity(0)
    ctx.highlight_set_component_stats(False)


def _frames_cc(ctx, frames, p, polarity, stats=True, max_comps=512, labels=True):
    _begin(ctx, p, polarity, stats)
    try:
        assert ctx.highlight_component_dtype() == (ctx.COMPONENT_STATS_DTYPE if stats else ctx.COMPONENT_DTYPE)
        return ctx.highlight_frames_cc(frames, max_comps=max_comps, labels=labels)
    finally:
        _end(ctx)


def check_records(recs, ncomp, labels, frame, bg, polarity, what=""):
    want = reference_stats(labels, frame, bg, polarity, max_comps=recs.shape[0])
    assert int(labels.max()) == ncomp, what
    k = len(want)
    assert recs[:k].tobytes() == want.tobytes(), f"{what}: {np.nonzero(recs[:k] != want)[0][:8]}"


def _check_case(ctx, frame, p, polarity, what=""):
    masks, recs, ncomps, labels = _frames_cc(ctx, frame[None], p, polarity)
    assert np.array_equal(masks[0], pc.highlight_objects(frame.copy(), p, polarity)), what
    check_records(recs[0], int(ncomps[0]), labels[0], frame, p.background, polarity, what)
    # off: the same masks, counts and plain records (the records past the count are not written)
    m0, c0, n0, l0 = _frames_cc(ctx, frame[None], p, polarity, stats=False)
    assert m0.tobytes() == masks.tobytes() and n0.tobytes() == ncomps.tobytes() and l0.tobytes() == labels.tobytes()
    k = min(int(ncomps[0]), recs.shape[1])
    assert c0[0, :k].tobytes() == np.ascontiguousarray(recs[0, :k]["c"]).tobytes(), what


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("t", range(0, 60, 3))
def test_random_cases(ctx, t, polarity):
    frame, p = pc.mixed_random_case(t) if polarity != "dark" else hl_cases.random_case(t)
    _check_case(ctx, frame, p, polarity, f"random_{t}")


ADV = hl_cases.adversarial_cases()


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("case", ADV, ids=[c[0] for c in ADV])
def test_adversarial_cases(ctx, case, polarity):
    name, frame, p = case
    if polarity != "dark":
        frame = pc.mixed(frame, p.background)
    _check_case(ctx, frame, p, polarity, name)


@pytest.mark.parametrize("variant", ["large", "small"])
def test_both_builds_of_the_fused_kernel(ctx, monkeypatch, variant):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    for t in range(0, 60, 6):
        frame, p = pc.mixed_random_case(t)
        for polarity in POLS:
            _check_case(ctx, frame, p, polarity, f"{variant} random_{t}")


@pytest.mark.parametrize("hw", [(40, 32), (21, 128), (17, 640), (9, 1056), (30, 75), (19, 33), (25, 150)])
def test_aligned_and_unaligned_widths_with_otsu(ctx, hw):
    """W % 32 == 0 takes the 128-bit path (word-wise contrast sums), other widths the byte path; threshold -1 is Otsu"""
    h, w = hw
    frame, bg = hl_cases.blob_frame(h, w, 400, sigma=2.0, amp=70)
    frame = pc.mixed(frame, bg)
    for p in (ho.canonical_params(bg), ho.HighlightParams(bg, np.ones((1, 1), np.uint8), 12, 6, 20, 0, 3, 5),
              ho.HighlightParams(bg, np.ones((3, 2), np.uint8), -1, 9, 14, 10, 30, 5)):
        for polarity in POLS:
            _check_case(ctx, frame, p, polarity, f"{h}x{w} th {p.threshold} {polarity}")


def _device_bg(ctx, frames, bgs, bg_stride, p, polarity, max_comps=256, stats=True, in_place=None):
    """cvvp_highlight_device_bg with components; in_place: "frames" / "bg" makes d_out alias that buffer"""
    n, h, w = frames.shape
    npix = h * w
    pitch = (npix + 15) // 16 * 16
    def dev(a):
        host = np.zeros((a.shape[0], pitch), np.uint8)
        host[:, :npix] = a.reshape(a.shape[0], npix)
        return torch.from_numpy(host).cuda()
    d_f, d_b = dev(frames), dev(bgs)
    d_o = torch.zeros((n, pitch), dtype=torch.uint8, device="cuda")
    rec = 104 if stats else 48
    d_c = torch.zeros((n, max_comps * rec), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(n, dtype=torch.int32, device="cuda")
    d_l = torch.zeros((n, npix), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    out = {"frames": d_f, "bg": d_b}.get(in_place, d_o)
    _begin(ctx, p, polarity, stats)
    try:
        rc = ctx._lib.cvvp_highlight_device_bg(ctx.handle, d_f.data_ptr(), n, pitch, d_b.data_ptr(), bg_stride,
                                               out.data_ptr(), pitch, d_c.data_ptr(), max_comps, d_n.data_ptr(),
                                               d_l.data_ptr(), npix, None)
        ctx.synchronize()
    finally:
        _end(ctx)
    if in_place:
        return rc
    assert rc == 0
    dt = _cabi.Context.COMPONENT_STATS_DTYPE if stats else _cabi.Context.COMPONENT_DTYPE
    return (d_o.cpu().numpy()[:, :npix].reshape(n, h, w), d_c.cpu().numpy().view(dt).reshape(n, max_comps),
            d_n.cpu().numpy(), d_l.cpu().numpy().reshape(n, h, w))


@pytest.mark.parametrize("polarity", POLS)
def test_a_background_per_frame_and_an_all_foreground_frame(ctx, polarity):
    rng = np.random.default_rng(5)
    frame, p = pc.mixed_random_case(11)
    h, w = frame.shape
    bg = p.background
    frames = np.stack([frame, np.roll(frame, 2, axis=0), frame, frame])
    bgs = np.stack([bg, np.clip(bg.astype(int) + 9, 0, 255).astype(np.uint8),
                    np.clip(bg.astype(int) + rng.integers(-6, 7, bg.shape), 0, 255).astype(np.uint8),
                    np.full_like(bg, 255 if polarity == "dark" else 0)])  # the last: every pixel passes, d = 0 possible
    p4 = ho.HighlightParams(bg, p.struct_element, 3, 2, 4, p.min_size_hyst, p.min_size_threshold, p.width_border)
    for q in (p, p4):
        masks, recs, ncomps, labels = _device_bg(ctx, frames, bgs, (h * w + 15) // 16 * 16, q, polarity)
        for i in range(len(frames)):
            assert np.array_equal(masks[i], pc.masks(frames[i:i + 1], q, polarity, bgs[i:i + 1])[0])
            check_records(recs[i], int(ncomps[i]), labels[i], frames[i], bgs[i], polarity, f"frame {i}")
        m0, c0, n0, l0 = _device_bg(ctx, frames, bgs, (h * w + 15) // 16 * 16, q, polarity, stats=False)
        assert m0.tobytes() == masks.tobytes() and n0.tobytes() == ncomps.tobytes()
        for i in range(len(frames)):
            k = min(int(ncomps[i]), recs.shape[1])
            assert c0[i, :k].tobytes() == np.ascontiguousarray(recs[i, :k]["c"]).tobytes()
    # an all-foreground 1080p frame (the FillHoles all-255 quirk): 1080 runs of 1920 pixels
    big = np.random.default_rng(1).integers(0, 256, (1, 1080, 1920), dtype=np.uint8)
    bg0 = np.full((1080, 1920), 128, np.uint8)
    pq = ho.HighlightParams(bg0, np.ones((1, 1), np.uint8), -2, -2, -2, 0, 0, 0)  # negative: every pixel passes
    masks, recs, ncomps, labels = _device_bg(ctx, big, bg0[None], 0, pq, polarity, max_comps=4)
    assert (masks == 255).all() and int(ncomps[0]) == 1
    check_records(recs[0], 1, labels[0], big[0], bg0, polarity, "all foreground")


def test_more_components_than_records(ctx):
    h, w = 64, 96
    frame = np.full((h, w), 200, np.uint8)
    frame[2::4, 3::5] = 20  # isolated dots: many components
    p = ho.HighlightParams(np.full((h, w), 200, np.uint8), np.ones((1, 1), np.uint8), 50, 40, 60, 0, 0, 0)
    masks, recs, ncomps, labels = _frames_cc(ctx, frame[None], p, "dark", max_comps=17)
    assert int(ncomps[0]) > 17 and recs.shape == (1, 17)
    want = reference_stats(labels[0], frame, p.background, "dark", max_comps=17)
    assert recs[0].tobytes() == want.tobytes()


def test_more_frames_than_in_flight_with_and_without_labels(ctx):
    frame, p = pc.mixed_random_case(21)
    _begin(ctx, p, "both")
    n = ctx.highlight_frames_in_flight() * 2 + 3
    _end(ctx)
    frames = np.stack([np.roll(frame, i, axis=1) for i in range(n)])
    masks, recs, ncomps, labels = _frames_cc(ctx, frames, p, "both", max_comps=64)
    m2, r2, n2 = _frames_cc(ctx, frames, p, "both", max_comps=64, labels=False)
    assert m2.tobytes() == masks.tobytes() and r2.tobytes() == recs.tobytes() and n2.tobytes() == ncomps.tobytes()
    for i in range(n):
        assert np.array_equal(canonical_labels(masks[i]), labels[i])
        check_records(recs[i], int(ncomps[i]), labels[i], frames[i], p.background, "both", f"frame {i}")


@pytest.mark.parametrize("polarity", POLS)
def test_queue_with_decoded_colour_frames_and_a_crop(ctx, polarity):
    rng = np.random.default_rng(23)
    h, w, n, batch, mc = 70, 120, 13, 4, 32
    crop = (9, 4, 100, 60)
    frames = np.empty((n, h, w, 3), np.uint8)
    for i in range(n):
        f, bg = hl_cases.blob_frame(h, w, 950 + i, bgv=128, sigma=2.0, amp=70)
        frames[i] = np.stack([pc.mixed(f, bg), np.roll(f, 3, axis=1), rng.integers(0, 256, (h, w), dtype=np.uint8)],
                             axis=-1)
    prepared = fo.prepare_frames(frames, crop, fo.CHANNEL0)
    p = ho.canonical_params(np.full(prepared.shape[1:], 128, np.uint8))
    fb = h * w * 3
    _begin(ctx, p, polarity)
    try:
        ctx.highlight_queue_begin(2, batch, _cabi.FrameFormat.of((h, w, 3), fo.CHANNEL0, crop), mc)
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
                got.append(tuple(a.copy() for a in ctx.highlight_next()))
            else:
                got.append(tuple(np.array(a) for a in ctx.highlight_next_view()))
                ctx.highlight_view_release()
        ctx.highlight_queue_end()
    finally:
        _end(ctx)
    masks = np.concatenate([g[0] for g in got])
    recs = np.concatenate([g[1] for g in got])
    ncomps = np.concatenate([g[2] for g in got])
    assert recs.dtype == _cabi.Context.COMPONENT_STATS_DTYPE
    assert np.array_equal(masks, pc.masks(prepared, p, polarity))
    assert ncomps.sum() > 0
    for t in range(n):
        check_records(recs[t], int(ncomps[t]), canonical_labels(masks[t]), prepared[t], p.background, polarity, str(t))


@pytest.mark.parametrize("polarity", ["dark", "bright"])
def test_rolling_stream(polarity):
    """cvvp_highlight_rolling_next with statistics: every frame against its own window median"""
    h, w = SMALL
    window, mb, mc = 7, 3, 40
    n = 3 * (window + mb) + 4
    frames = make_frames(n, h, w, seed=90)
    if polarity == "bright":
        frames = (255 - frames).astype(np.uint8)
    p = fine_params(h, w)
    got = {}
    with _cabi.Context(0) as c:
        _begin(c, p, polarity)
        c.highlight_rolling_begin(window, mb, None, mc, labels=True)
        def drain():
            while c.highlight_rolling_pending():
                first, masks, recs, ncomps, labels = c.highlight_rolling_next()
                for i in range(masks.shape[0]):
                    got[first + i] = (masks[i].copy(), recs[i].copy(), int(ncomps[i]), labels[i].copy())
        for i in range(0, n, mb):
            c.highlight_rolling_push(frames[i:i + mb])
            if c.highlight_rolling_ready():
                first, masks, recs, ncomps, labels = c.highlight_rolling_next()
                for j in range(masks.shape[0]):
                    got[first + j] = (masks[j].copy(), recs[j].copy(), int(ncomps[j]), labels[j].copy())
        c.highlight_rolling_close()
        drain()
        c.highlight_rolling_end()
        c.highlight_end()
    assert sorted(got) == list(range(n))
    bgs = host_backgrounds(frames, window)
    want = pc.masks(frames, p, polarity, bgs)
    assert sum(g[2] for g in got.values()) > 0
    for t in range(n):
        mask, recs, ncomp, labels = got[t]
        assert recs.dtype == _cabi.Context.COMPONENT_STATS_DTYPE
        assert np.array_equal(mask, want[t]), t
        check_records(recs, ncomp, labels, frames[t], bgs[t], polarity, str(t))


def test_in_place_output_is_rejected_and_state_errors(ctx):
    frame, p = pc.mixed_random_case(3)
    frames, bgs = frame[None], p.background[None]
    for where in ("frames", "bg"):
        assert _device_bg(ctx, frames, bgs, 0, p, "dark", in_place=where) == ERR_INVALID
        assert b"overlaps" in ctx._lib.cvvp_last_error(ctx.handle)
    # without statistics the same in-place call is accepted, as before
    assert _device_bg(ctx, frames, bgs, 0, p, "dark", stats=False, in_place="frames") == 0
    with _cabi.Context(0) as c:
        lib = c._lib
        assert c.highlight_component_stats() is False  # the default
        for bad in (2, -1, 255):
            assert lib.cvvp_highlight_set_component_stats(c.handle, bad) == ERR_INVALID
        c.highlight_set_component_stats(True)
        c.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo,
                          p.threshold_hi, p.min_size_hyst, p.min_size_threshold, p.width_border)
        assert lib.cvvp_highlight_set_component_stats(c.handle, 0) == ERR_STATE
        assert lib.cvvp_highlight_set_component_stats(c.handle, 1) == ERR_STATE
        assert c.highlight_component_stats() is True
        assert c.highlight_frames_cc(frame[None], max_comps=8)[1].dtype == c.COMPONENT_STATS_DTYPE
        c.highlight_end()
        c.highlight_set_component_stats(False)
        c.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo,
                          p.threshold_hi, p.min_size_hyst, p.min_size_threshold, p.width_border)
        assert c.highlight_frames_cc(frame[None], max_comps=8)[1].dtype == c.COMPONENT_DTYPE
        c.highlight_end()
