"""GPU tests of colour highlight jobs through the C ABI (cvvp_highlight_set_channels): masks, component counts, plain
records and statistics against the cv2 restatement through identity (3) of tests/color_cases.py, for 1 to 4 channels in
every polarity; both builds of the fused kernel, the colour kernel's 128-bit and byte paths, Otsu and the per-pixel
path; a background per frame; more frames than are in flight and than one scratch chunk; the host, components and
device forms; the queue (copying and zero-copy, decoded colour frames with a crop, and prepared colour frames); the
rolling stream against a host rolling percentile per colour element; byte equality of one channel with a job that never
set it; and the setting's state and argument errors."""
import dataclasses

import cv2
import numpy as np
import pytest
import torch

import color_cases as cc
import hl_cases
import polarity_cases as pc
from cvvidproc_b200 import _cabi, synth
from oracle import frames_oracle as fo
from oracle import highlight_oracle as ho
from test_components_gpu import _check_frame
from test_highlight_rolling_stream_gpu import fine_params, host_backgrounds, make_frames

pytestmark = pytest.mark.gpu

FUSED, PIXEL = 0, 1
ERR_INVALID, ERR_STATE = -1, -4
POLS = list(pc.POLARITIES)


@pytest.fixture(scope="module")
def ctx():
    # a context of its own: the channel count and the polarity are settings of the context
    c = _cabi.Context(0)
    yield c
    c.close()


def _begin(ctx, p):
    ctx.highlight_begin(p.background, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                        p.min_size_hyst, p.min_size_threshold, p.width_border)


class _job:
    """a highlight job of p's channels in `polarity`; the context's settings are restored afterwards"""

    def __init__(self, ctx, p, polarity, path=FUSED):
        self.ctx, self.p, self.polarity, self.path = ctx, p, polarity, path

    def __enter__(self):
        c = self.p.background.shape[2] if self.p.background.ndim == 3 else 1
        self.ctx.highlight_set_polarity(pc.POLARITIES[self.polarity])
        self.ctx.highlight_set_channels(c)
        _begin(self.ctx, self.p)
        self.ctx.highlight_set_path(self.path)
        return self.ctx

    def __exit__(self, *exc):
        self.ctx.highlight_end()
        self.ctx.highlight_set_polarity(0)
        self.ctx.highlight_set_channels(1)


def _host(ctx, frames, p, polarity, path=FUSED):
    with _job(ctx, p, polarity, path):
        return ctx.highlight_frames(frames)


def _check(ctx, frame, p, polarity, path=FUSED, what=""):
    got = _host(ctx, frame[None], p, polarity, path)[0]
    want = cc.highlight_objects(frame, p, polarity)
    assert np.array_equal(got, want), f"{what} {polarity}: {(got != want).sum()} pixels differ"


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("c", [2, 3, 4])
def test_random_and_adversarial_cases(ctx, c, polarity):
    for t in range(0, 60, 2):
        frame, p = cc.random_case(t, c)
        _check(ctx, frame, p, polarity, what=f"random_{t}")
    for name, frame, p in cc.adversarial_cases(c):
        _check(ctx, frame, p, polarity, what=name)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("variant", ["large", "small"])
def test_both_builds_of_the_fused_kernel(ctx, monkeypatch, variant, polarity):
    monkeypatch.setenv("CVVP_HL_VARIANT", variant)
    for c in (2, 3, 4):
        for t in range(1, 60, 7):
            frame, p = cc.random_case(t, c)
            _check(ctx, frame, p, polarity, what=f"{variant} c{c} random_{t}")


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("path", [FUSED, PIXEL])
@pytest.mark.parametrize("c", [2, 3, 4])
@pytest.mark.parametrize("hw", [(40, 32), (21, 128), (17, 640), (9, 1056), (30, 75), (19, 33), (25, 150), (13, 7)])
def test_aligned_and_unaligned_widths_with_otsu(ctx, hw, c, path, polarity):
    """frames of 16 pixels or more take the colour kernel's 128-bit path, frame tails its byte path (widths with
    3w a multiple of 16 and not); threshold -1 is Otsu on the colour d"""
    h, w = hw
    for seed in range(2):
        frame, p0 = cc.blob_case(h, w, c, 400 + seed)
        bg = p0.background
        for p in (p0, ho.HighlightParams(bg, np.ones((1, 1), np.uint8), 12, 6, 20, 0, 3, 5),
                  ho.HighlightParams(bg, np.ones((3, 2), np.uint8), -1, 9, 14, 10, 30, 5),
                  ho.HighlightParams(bg, np.ones((1, 1), np.uint8), -1, 20, 8, 0, 0, 5)):
            _check(ctx, frame, p, polarity, path, what=f"{h}x{w}x{c} seed {seed} th {p.threshold}")


@pytest.mark.parametrize("path", [FUSED, PIXEL])
def test_every_stored_reference_output_through_the_identities(ctx, path):
    """identity (2): the reference's masks from frames replicated into 2, 3 and 4 channels; identity (3): a colour job
    equals the grey dark job on 255 - D against 255"""
    import hashlib

    cases = pc.golden_cases()
    assert len(cases) == 83
    for i, (g, frame, p) in enumerate(cases):
        for c in (2, 3, 4):
            f, q = cc.replicated(frame, p, c)
            got = _host(ctx, f[None], q, "dark", path)[0]
            assert hashlib.sha256(got.tobytes()).hexdigest() == g["output_sha256"], (g["name"], c)
        f, q = cc.colorize(frame, p, 3, 3000 + i)
        polarity = POLS[i % 3]
        fd, qd = cc.as_dark(f, q, polarity)
        assert np.array_equal(_host(ctx, f[None], q, polarity, path)[0], _host(ctx, fd[None], qd, "dark", path)[0])


def test_one_channel_is_the_grey_job_byte_for_byte(ctx):
    """set_channels(1) and a context that never set it give the same bytes, for (H, W) and (H, W, 1) backgrounds"""
    frames = np.stack([pc.mixed_random_case(t)[0] for t in (4, 4, 4)])
    _, p = pc.mixed_random_case(4)
    with _cabi.Context(0) as fresh:
        _begin(fresh, p)
        want = fresh.highlight_frames(frames)
        fresh.highlight_end()
    assert want.any()
    ctx.highlight_set_channels(1)
    assert ctx.highlight_channels() == 1
    for q in (p, dataclasses.replace(p, background=p.background[..., None].copy())):
        _begin(ctx, q)
        assert np.array_equal(ctx.highlight_frames(frames), want)
        ctx.highlight_end()


def _device_pitch(nbytes, pad):
    return (nbytes + pad - 1) // pad * pad


def _device_bg(ctx, frames, bgs, p, polarity, path=FUSED, comps=0, stats=False, pad=16, form="bg"):
    """masks (and components) of cvvp_highlight_device_bg / _device / _device_cc on colour frames at a pitch padded
    to `pad` bytes; bgs None: the job's own background"""
    n, h, w, c = frames.shape
    fb, npix = h * w * c, h * w
    fp, mp = _device_pitch(fb, pad), _device_pitch(npix, 16)

    def dev(a):
        host = np.zeros((a.shape[0], fp), np.uint8)
        host[:, :fb] = a.reshape(a.shape[0], fb)
        return torch.from_numpy(host).cuda()

    d_f = dev(frames)
    d_b = dev(bgs) if bgs is not None else None
    d_o = torch.zeros((n, mp), dtype=torch.uint8, device="cuda")
    rec = 104 if stats else 48
    d_c = torch.zeros((n, max(comps, 1) * rec), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.highlight_set_component_stats(stats)
    try:
        with _job(ctx, p, polarity, path):
            if form == "bg":
                ctx.highlight_device_bg(d_f.data_ptr(), n, fp, d_b.data_ptr(), fp if bgs.shape[0] > 1 else 0,
                                        d_o.data_ptr(), mp, d_c.data_ptr() if comps else 0, comps,
                                        d_n.data_ptr() if comps else 0)
            elif form == "device":
                ctx.highlight_device(d_f.data_ptr(), n, fp, d_o.data_ptr(), mp)
            else:
                ctx._check(ctx._lib.cvvp_highlight_device_cc(ctx.handle, d_f.data_ptr(), n, fp, d_o.data_ptr(), mp,
                                                             d_c.data_ptr(), comps, d_n.data_ptr(), None, 0, None))
            ctx.synchronize()
    finally:
        ctx.highlight_set_component_stats(False)
    masks = d_o.cpu().numpy()[:, :npix].reshape(n, h, w)
    if not comps:
        return masks
    dt = ctx.COMPONENT_STATS_DTYPE if stats else ctx.COMPONENT_DTYPE
    return masks, np.frombuffer(d_c.cpu().numpy().tobytes(), dt).reshape(n, comps), d_n.cpu().numpy()


def _colour_stack(c, n, seed):
    """n colour frames against one background: a random case's frame shifted by i columns, coloured alike"""
    frame, p = pc.mixed_random_case(seed % 60)
    stack = [cc.colorize(np.roll(frame, i, axis=1), p, c, seed) for i in range(n)]
    return np.stack([f for f, _ in stack]), stack[0][1]


def _check_plain(mask, comps, ncomp):
    """count and areas of the plain records against cv2.connectedComponentsWithStats"""
    n_cv, _, stats_cv, _ = cv2.connectedComponentsWithStats(mask, connectivity=8, ltype=cv2.CV_32S)
    assert ncomp == n_cv - 1
    k = min(ncomp, comps.shape[0])
    assert sorted(comps["area"][:k]) == sorted(stats_cv[1:, cv2.CC_STAT_AREA])[:k] or k < ncomp


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("path", [FUSED, PIXEL])
@pytest.mark.parametrize("c", [2, 3, 4])
def test_a_background_per_frame(ctx, c, path, polarity):
    """bg_stride > 0, at 16-byte and odd pitches (the colour kernel's byte path for every frame but the first)"""
    for t in range(0, 60, 12):
        frame, p = pc.mixed_random_case(t)
        frames = np.stack([cc.colorize(frame, p, c, 50 + k)[0] for k in range(4)])
        bgs = np.stack([cc.colorize(frame, p, c, 70 + k)[1].background for k in range(4)])
        q = dataclasses.replace(p, background=bgs[0])
        want = cc.masks(frames, q, polarity, bgs)
        for pad in (16, 1):
            got = _device_bg(ctx, frames, bgs, q, polarity, path, pad=pad)
            assert np.array_equal(got, want), (t, pad)


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("c", [2, 3, 4])
def test_components_and_statistics(ctx, c, polarity):
    """plain records and statistics of the device and host forms; the statistics' d is the colour d"""
    for t in range(0, 60, 10):
        frame, p = cc.random_case(t, c)
        want = cc.highlight_objects(frame, p, polarity)
        d = cc.color_difference(p.background, frame, polarity).astype(np.int64)
        for stats in (False, True):
            masks, comps, ncomps = _device_bg(ctx, frame[None], p.background[None], p, polarity, comps=512, stats=stats)
            assert np.array_equal(masks[0], want), t
            plain = comps["c"] if stats else comps
            _check_plain(masks[0], plain[0], int(ncomps[0]))
            if stats:
                ys, xs = np.nonzero(want)
                assert comps["sum_d"][0, :int(ncomps[0])].sum() == d[ys, xs].sum()
        ctx.highlight_set_component_stats(True)
        try:
            with _job(ctx, p, polarity):
                hm, hc, hn, lab = ctx.highlight_frames_cc(frame[None], max_comps=512, labels=True)
        finally:
            ctx.highlight_set_component_stats(False)
        assert np.array_equal(hm[0], want)
        _check_frame(hm[0], hc["c"][0], int(hn[0]), lab[0])


@pytest.mark.parametrize("c", [3, 4])
def test_device_and_device_cc_forms_with_many_frames(ctx, monkeypatch, c):
    """more frames than the fused kernel keeps in flight, and than one scratch chunk (CVVP_HL_SLOTS shrinks both)"""
    monkeypatch.setenv("CVVP_HL_SLOTS", "5")
    n = 23
    frames, p = _colour_stack(c, n, 700)
    want = cc.masks(frames, p, "both")
    assert np.array_equal(_device_bg(ctx, frames, None, p, "both", form="device"), want)
    masks, comps, ncomps = _device_bg(ctx, frames, None, p, "both", comps=256, form="device_cc")
    assert np.array_equal(masks, want)
    for i in range(n):
        _check_plain(masks[i], comps[i], int(ncomps[i]))
    assert np.array_equal(_host(ctx, frames, p, "both"), want)
    assert np.array_equal(_host(ctx, frames, p, "both", PIXEL), want)


@pytest.mark.parametrize("cfg,n", [("C3", 6), ("C4", 40)])
def test_full_size_frames(ctx, cfg, n):
    """1080p and 512x256 frames in three channels: replicated grey frames give the grey masks, and a colour job's fused
    and per-pixel paths agree and match the host reference on one frame"""
    q = synth.CONFIG_PARAMS[cfg]
    w, h = q["width"], q["height"]
    bg = np.sort(synth.synth_frames(0, 31, w, h, q["seed"], q["ndisks"]), axis=0)[15]
    p = ho.canonical_params(bg)
    frames = synth.synth_frames(200, n, w, h, q["seed"], q["ndisks"])
    with _cabi.Context(0) as grey:
        _begin(grey, p)
        want = grey.highlight_frames(frames)
        grey.highlight_end()
    rf, rp = cc.replicated(frames, p, 3)
    assert np.array_equal(_host(ctx, rf, rp, "dark"), want)
    f3 = np.stack([frames, np.roll(frames, 11, axis=2), 255 - frames], axis=-1)
    p3 = dataclasses.replace(p, background=np.stack([bg, np.roll(bg, 11, axis=1), 255 - bg], axis=-1))
    fused = _host(ctx, f3, p3, "both")
    assert np.array_equal(fused, _host(ctx, f3, p3, "both", PIXEL))
    assert np.array_equal(fused[1], cc.highlight_objects(f3[1], p3, "both"))


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("c", [3, 4])
def test_queue_with_decoded_colour_frames_and_a_crop(ctx, c, polarity):
    """the queue's copying (submit / next) and zero-copy (slot_acquire / commit / next_view) forms on decoded frames of
    c channels with a crop: one kernel crops them and writes d"""
    h, w, n, batch = 70, 120, 13, 4
    crop = (9, 4, 100, 60)
    frames = np.empty((n, h, w, c), np.uint8)
    bgfull = None
    for i in range(n):
        f, bg = hl_cases.blob_frame(h, w, 950 + i, bgv=128, sigma=2.0, amp=70)
        fc, pc_ = cc.colorize(pc.mixed(f, bg), ho.canonical_params(bg), c, 60 + i)
        frames[i] = fc
        bgfull = pc_.background
    prepared = fo.prepare_frames(frames, crop, fo.AS_IS)
    x, y, cw, ch = crop
    p = dataclasses.replace(ho.canonical_params(bgfull[y:y + ch, x:x + cw, 0].copy()),
                            background=np.ascontiguousarray(bgfull[y:y + ch, x:x + cw]))
    want = cc.masks(prepared, p, polarity)
    assert want.any()
    fb = h * w * c
    with _job(ctx, p, polarity):
        for fmt_mode in (fo.AS_IS, fo.CHANNEL0):  # a colour job takes AS_IS frames of its channel count only
            if fmt_mode != fo.AS_IS:
                rc = ctx._lib.cvvp_highlight_queue_begin(ctx.handle, 2, batch,
                                                         _cabi.C.byref(_cabi.FrameFormat.of((h, w, c), fmt_mode, crop)), 0)
                assert rc == ERR_INVALID
        ctx.highlight_queue_begin(2, batch, _cabi.FrameFormat.of((h, w, c), fo.AS_IS, crop))
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
    assert np.array_equal(np.concatenate(got), want)


@pytest.mark.parametrize("c", [2, 3])
def test_queue_with_prepared_colour_frames_and_components(ctx, c):
    n, batch = 11, 3
    frames, p = _colour_stack(c, n, 800)
    want = cc.masks(frames, p, "dark")
    fb = frames[0].size
    with _job(ctx, p, "dark"):
        ctx.highlight_queue_begin(2, batch, None, 256)
        got, i, k = [], 0, 0
        while i < n or ctx.highlight_queue_pending():
            while i < n and ctx.highlight_queue_pending() < 2:
                m = min(batch, n - i)
                if k % 2:
                    ctx.highlight_submit(frames[i:i + m])
                else:
                    slot = ctx.highlight_slot_acquire()
                    assert slot.shape[1] >= fb
                    slot[:m, :fb] = frames[i:i + m].reshape(m, fb)
                    ctx.highlight_slot_commit(m)
                i += m
                k += 1
            masks, comps, ncomps = ctx.highlight_next()
            for j in range(masks.shape[0]):
                _check_plain(masks[j], comps[j], int(ncomps[j]))
            got.append(masks.copy())
        ctx.highlight_queue_end()
    assert np.array_equal(np.concatenate(got), want)


def _run_rolling(ctx, pushed, h, w, window, mb, fmt=None):
    ctx.highlight_rolling_begin(window, mb, fmt)
    n = pushed.shape[0]
    out = np.full((n, h, w), 0x5A, np.uint8)

    def drain():
        while True:
            first, masks = ctx.highlight_rolling_next()
            if masks.shape[0] == 0:
                return
            out[first:first + masks.shape[0]] = masks

    for i in range(0, n, mb):
        ctx.highlight_rolling_push(pushed[i:i + mb])
        drain()
    ctx.highlight_rolling_close()
    drain()
    ctx.highlight_rolling_end()
    return out


@pytest.mark.parametrize("polarity", POLS)
@pytest.mark.parametrize("c", [2, 3, 4])
def test_rolling_stream(c, polarity):
    """colour frames in the ring: every colour element's rolling upper median (a host percentile of the window), then
    the colour d; prepared frames, and decoded frames with a crop"""
    h, w = 29, 37
    window, mb = 7, 3
    n = 2 * (window + mb) + 4
    chans = [make_frames(n, h, w, seed=90 + k) for k in range(c)]
    if polarity == "bright":
        chans[0] = (255 - chans[0]).astype(np.uint8)
    frames = np.ascontiguousarray(np.stack(chans, axis=-1))
    bgs = host_backgrounds(frames.reshape(n, h, w * c), window).reshape(n, h, w, c)
    p0 = fine_params(h, w)
    p = dataclasses.replace(p0, background=np.zeros((h, w, c), np.uint8))
    want = cc.masks(frames, p, polarity, bgs)
    assert want.any()
    with _cabi.Context(0) as ctx:
        ctx.highlight_set_polarity(pc.POLARITIES[polarity])
        ctx.highlight_set_channels(c)
        _begin(ctx, p)
        assert np.array_equal(_run_rolling(ctx, frames, h, w, window, mb), want)
        # decoded frames two rows and three columns larger, cropped on the device
        big = np.zeros((n, h + 2, w + 3, c), np.uint8)
        big[:, 1:1 + h, 2:2 + w] = frames
        fmt = _cabi.FrameFormat.of((h + 2, w + 3, c), fo.AS_IS, (2, 1, w, h))
        assert np.array_equal(_run_rolling(ctx, big, h, w, window, mb, fmt), want)
        assert ctx._lib.cvvp_highlight_rolling_begin(
            ctx.handle, window, mb, _cabi.C.byref(_cabi.FrameFormat.of((h + 2, w + 3, c + 1 if c < 4 else 3), fo.AS_IS,
                                                                       (2, 1, w, h))), 0, 0) == ERR_INVALID
        ctx.highlight_end()


def test_state_and_argument_errors():
    frame, p = cc.random_case(5, 3)
    with _cabi.Context(0) as c:
        lib = c._lib
        assert c.highlight_channels() == 1  # the default
        for bad in (0, 5, -1, 255):
            assert lib.cvvp_highlight_set_channels(c.handle, bad) == ERR_INVALID
        assert c.highlight_channels() == 1
        with pytest.raises(TypeError):
            _begin(c, p)  # a colour background on a one-channel context
        c.highlight_set_channels(3)
        assert c.highlight_channels() == 3
        _begin(c, p)
        for bad in (1, 2, 3):
            assert lib.cvvp_highlight_set_channels(c.handle, bad) == ERR_STATE
        assert c.highlight_channels() == 3
        assert np.array_equal(c.highlight_frames(frame[None])[0], cc.highlight_objects(frame, p, "dark"))
        with pytest.raises(TypeError):
            c.highlight_frames(frame[None, ..., 0].copy())  # grey frames on a colour job
        # strides shorter than a colour frame, and an output overlapping the frames or the backgrounds
        h, w = frame.shape[:2]
        fb = h * w * 3
        d_f = torch.zeros(2 * fb, dtype=torch.uint8, device="cuda")
        d_o = torch.zeros(2 * fb, dtype=torch.uint8, device="cuda")
        fp, op = d_f.data_ptr(), d_o.data_ptr()
        assert lib.cvvp_highlight_device(c.handle, fp, 2, h * w, op, h * w, None) == ERR_INVALID
        assert lib.cvvp_highlight_device_bg(c.handle, fp, 1, fb, fp, h * w, op, h * w, None, 0, None, None, 0,
                                            None) == ERR_INVALID
        assert lib.cvvp_highlight_device(c.handle, fp, 2, fb, fp + fb, h * w, None) == ERR_INVALID
        assert lib.cvvp_highlight_device_bg(c.handle, fp, 1, fb, op, 0, op + 8, h * w, None, 0, None, None, 0,
                                            None) == ERR_INVALID
        assert lib.cvvp_highlight_device(c.handle, fp, 2, fb, op, h * w, None) == 0
        c.synchronize()
        c.highlight_end()
        c.highlight_set_channels(1)
        _, pg = pc.mixed_random_case(5)
        _begin(c, pg)  # a job begun after a change uses the new value
        assert np.array_equal(c.highlight_frames(frame[None, ..., 0].copy())[0],
                              pc.highlight_objects(frame[..., 0].copy(), pg, "dark"))
        c.highlight_end()
    with _cabi.Context(0) as other:  # a fresh context: every other context is left alone
        assert other.highlight_channels() == 1
