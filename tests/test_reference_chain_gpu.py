"""GPU parity against the reference's OWN compiled sources, with no restatement in between: the three modules of
oracle/_ref (built from /root/reference where it is mounted, shipped with the snapshot) --
    libcvvp_median_ref.so   HistogramMedianAlgo<T>        histogram_median_algo.h
    cvvp_highlight_ref      HighlightObjectsAlgo          highlight_objects_algo.{h,cpp}   (cv:: -> cv2 shim)
    cvvp_frames_ref         CvVidFramesGeneratorAlgo      cv_vid_frames_generator_algo.h   (cv:: -> cv2 shim)
-- chained the way the reference chains them (generator tokens -> median; generator tokens + background -> highlight
-> callback), held against the C ABI and against the drop-in Python surface."""
import hashlib

import cv2
import numpy as np
import pytest

import cvvidproc_b200 as cvp
import hl_cases
import video_util
from cvvidproc_b200 import _cabi, synth
from oracle import frames_oracle as fo
from oracle import frames_ref as fref
from oracle import highlight_oracle as ho
from oracle import highlight_ref as href

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not (href.available() and fref.available()), reason="oracle/_ref was not built")

ADV = hl_cases.adversarial_cases()


def _gpu_masks(ctx, frames, p):
    ctx.highlight_begin(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi, p.min_size_hyst,
                        p.min_size_threshold, p.width_border)
    try:
        return ctx.highlight_frames(frames)
    finally:
        ctx.highlight_end()


def _is_reference_output(name, frame, p, got):
    """the compiled reference where it was built, else the stored hash of its output; None: neither is there"""
    if href.available():
        return np.array_equal(got, href.highlight_objects(frame, p))
    sha = hl_cases.reference_sha256(name)
    return None if sha is None else hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == sha


@pytest.mark.parametrize("case", ADV, ids=[c[0] for c in ADV])
def test_highlight_adversarial_cases_against_the_compiled_reference(gpu_ctx, case):
    name, frame, p = case
    got = _gpu_masks(gpu_ctx, frame[None], p)[0]
    same = _is_reference_output(name, frame, p, got)
    if same is None:
        pytest.skip(f"oracle/_ref was not built and no output of the reference is stored for {name}")
    assert same


@pytest.mark.parametrize("t0", range(0, 120, 20))
def test_highlight_random_cases_against_the_compiled_reference(gpu_ctx, t0):
    checked = 0
    for t in range(t0, t0 + 20):
        frame, p = hl_cases.random_case(t)
        got = _gpu_masks(gpu_ctx, frame[None], p)[0]
        same = _is_reference_output(f"random_{t}", frame, p, got)
        assert same is not False, f"random case {t}"
        checked += same is not None
    if not checked:
        pytest.skip(f"oracle/_ref was not built and no output of the reference is stored for random cases {t0}..{t0 + 19}")


@needs_ref
@pytest.mark.parametrize("cfg,count", [("C3", 12), ("C4", 200)])
def test_highlight_of_the_benchmark_streams_against_the_compiled_reference(gpu_ctx, cfg, count):
    """frames of the C3 (1080p) and C4 (512x256) streams at full size, canonical parameters, one batch on the device;
    every mask against HighlightObjectsAlgo::Insert -> TryGetResult"""
    p_ = synth.CONFIG_PARAMS[cfg]
    w, h = p_["width"], p_["height"]
    stack = synth.synth_frames(0, 15, w, h, p_["seed"], p_["ndisks"])
    p = ho.canonical_params(np.sort(stack, axis=0)[7])
    idx = [97 * k + 1000 for k in range(count)]
    frames = np.stack([synth.synth_frame(f, w, h, p_["seed"], p_["ndisks"]) for f in idx])
    got = _gpu_masks(gpu_ctx, frames, p)
    op = href.operator(p)
    some = 0
    for k in range(count):
        want = op.insert(frames[k])
        some += int(want.any())
        assert np.array_equal(got[k], want), f"{cfg} frame {idx[k]}: {(got[k] != want).sum()} pixels differ"
    assert some > count // 2


@pytest.fixture(scope="module")
def colour_stream(tmp_path_factory):
    """a colour video with dark moving disks (the C1 stream with a tint per channel), FFV1: decodes bit-exactly"""
    g = synth.synth_frames(0, 48, 176, 100, 11, 6).astype(np.int16)
    frames = np.clip(np.stack([g + 5, g - 3, g + 1], axis=-1), 0, 255).astype(np.uint8)
    path = video_util.write_lossless(tmp_path_factory.mktemp("v") / "colour.avi", frames)
    assert np.array_equal(video_util.read_all(path), frames)
    return path, frames


@needs_ref
@pytest.mark.parametrize("mode", ["grayscale", "vid_is_grayscale"])
def test_the_whole_path_against_the_reference_chain(colour_stream, ref_median, mode):
    """GetVideoBackground and TrackObjects of the drop-in module on a cropped colour video against the chain of
    the reference's own classes: CvVidFramesGeneratorAlgo tokens -> HistogramMedianAlgo -> HighlightObjectsAlgo"""
    if ref_median is None:
        pytest.skip("oracle/_ref/libcvvp_median_ref.so was not built")
    path, frames = colour_stream
    crop = (8, 6, 150, 90)
    kw = dict(crop_x=crop[0], crop_y=crop[1], crop_width=crop[2], crop_height=crop[3], **{mode: True})
    fmode = fo.RGB2GRAY if mode == "grayscale" else fo.CHANNEL0
    # background: the reference's generator feeds the reference's median class
    tokens = np.stack(fref.tokens(path, 0, len(frames), crop, fmode, frames_in_batch=5))
    assert tokens.shape == (len(frames), crop[3], crop[2])
    want_bg = ref_median(tokens)
    bg = cvp.GetVideoBackground(cvp.VidBgPack(path, **kw))
    assert bg.dtype == np.uint8 and np.array_equal(bg, want_bg)
    # a window of the stream for the median (start_frame is not a VidBgPack field: frame_limit only)
    bg20 = cvp.GetVideoBackground(cvp.VidBgPack(path, frame_limit=20, **kw))
    assert np.array_equal(bg20, ref_median(np.stack(fref.tokens(path, 0, 20, crop, fmode))))
    # highlight: every mask the callback receives, in order, against the reference's operator on the generator's tokens
    p = ho.canonical_params(want_bg)
    hp = cvp.HighlightObjectsPack(bg, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi, p.min_size_hyst,
                                  p.min_size_threshold, p.width_border)
    seen = []

    def collect(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs):
        seen.append((frames_processed, bw_frame.copy()))
        objects_archive[frames_processed] = int(cv2.countNonZero(bw_frame))
        return next_ID + 1

    for start, limit in ((0, 10_000), (7, 25)):
        seen.clear()
        archive = cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(collect, {}), start_frame=start,
                                                          frame_limit=limit, **kw))
        last = min(start + limit, len(frames))
        toks = fref.tokens(path, start, last, crop, fmode, frames_in_batch=3)
        assert [k for k, _ in seen] == list(range(last - start)) == sorted(archive)
        op = href.operator(p)
        white = 0
        for (k, mask), tok in zip(seen, toks):
            want = op.insert(tok)
            white += int(want.any())
            assert np.array_equal(mask, want), f"frame {start + k}"
            assert archive[k] == int(cv2.countNonZero(want))
        assert white > (last - start) // 2


@needs_ref
def test_median_c_abi_against_the_reference_class_on_generator_tokens(gpu_ctx, colour_stream, ref_median):
    """the C ABI's frame source + median (cvvp_median_push_source) against generator tokens -> reference median"""
    if ref_median is None:
        pytest.skip("oracle/_ref/libcvvp_median_ref.so was not built")
    path, frames = colour_stream
    decoded = video_util.read_all(path)
    for crop, mode in (((0, 0, 176, 100), fo.AS_IS), ((3, 1, 171, 97), fo.RGB2GRAY), ((16, 8, 64, 64), fo.CHANNEL0)):
        want = ref_median(np.stack(fref.tokens(path, 0, len(frames), crop, mode)))
        fmt = _cabi.FrameFormat.of(decoded.shape[1:], mode, crop)  # the mode numbers are the C ABI's (include/cvvp.h)
        nelem = int(np.prod(want.shape))
        gpu_ctx.median_begin(nelem, len(decoded))
        for i in range(0, len(decoded), 11):
            gpu_ctx.median_push_source(decoded[i:i + 11], fmt)
        got = gpu_ctx.median_finish(nelem=nelem).reshape(want.shape)
        assert np.array_equal(got, want), (crop, mode)


@needs_ref
def test_get_video_background_equals_the_reference_entry_point(colour_stream, tmp_path, capfd):
    """The drop-in claim at the public entry point: the reference's own GetVideoBackground -- cv_vid_bg_helpers.cpp with
    the whole AsyncTokens pipeline behind it, compiled unmodified (oracle/_ref/cvvp_background_ref; run in a child
    process with a time limit, see oracle/background_ref.py) -- and this module's GetVideoBackground get the same
    VidBgPack fields and must return the same image and print the same video-information line"""
    from oracle import background_ref as bgref

    if not bgref.available():
        pytest.skip("oracle/_ref/cvvp_background_ref was not built")
    path, frames = colour_stream
    rng = np.random.default_rng(21)
    portrait = np.clip(rng.integers(0, 256, (60, 40, 3), dtype=np.int16)[None] + rng.integers(-30, 31, (33, 60, 40, 3)), 0,
                       255).astype(np.uint8)
    ppath = video_util.write_lossless(tmp_path / "portrait.avi", portrait)
    packs = [
        (path, dict()),
        (path, dict(grayscale=True)),
        (path, dict(vid_is_grayscale=True, max_threads=3)),
        (path, dict(grayscale=True, crop_x=8, crop_y=6, crop_width=150, crop_height=90, max_threads=5)),
        (path, dict(frame_limit=17, crop_x=100, crop_width=500)),            # width clamped to the frame
        (path, dict(frame_limit=10_000, vid_is_grayscale=True, crop_y=50)),   # limit beyond the stream
        (ppath, dict(vid_is_grayscale=True, crop_y=30, crop_width=20, crop_height=25)),   # the :56 quirk: 30 rows come back
        (ppath, dict(grayscale=True, max_threads=2, frame_limit=32)),
        ("/no/such/video.avi", dict()),                                       # a missing video: an empty result
        (path, dict(bg_algo="mean")),                                         # an unknown algorithm name (:20-31, :262-266)
    ]
    reference = bgref.run_isolated(packs)
    for (vid, kw), (want, ref_out, _) in zip(packs, reference):
        capfd.readouterr()
        got = cvp.GetVideoBackground(cvp.VidBgPack(vid, **kw))
        our_out = capfd.readouterr().out
        if want is None:
            assert got is None, (vid, kw)
            continue
        assert got.dtype == np.uint8 and got.shape == want.shape, kw
        assert np.array_equal(got, want), kw
        info = [ln for ln in ref_out.splitlines() if ln.startswith("Frames:")]
        assert info and info[0] in our_out.splitlines(), (info, our_out)
