"""Cost of colour highlight jobs (cvvp_highlight_set_channels) on one GPU.

    python tools/probe_color.py OUT_PREFIX [--track-frames N]

Writes OUT_PREFIX.txt and OUT_PREFIX.json:
  * the colour-difference kernel (color_diff_kernel, torch.profiler kernel time inside cvvp_highlight_device) per frame
    and its HBM rate (frame + d plane bytes; the background is read from L2), against a device-to-device copy of the
    same frames timed with CUDA events in the same run, at 1080p x 3 and 512x256 x 3; inputs larger than L2;
  * the queue's crop + difference kernel against the RGB2GRAY preparation (frames_prepare_kernel) on the same decoded
    frames;
  * device time of cvvp_highlight_device on the colour frames against the grey frames (CUDA events);
  * TrackObjects ms per frame on a lossless 1080p colour video: cvvp_color against grayscale=True.
The card's name and power limit are read in the same run.
"""
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tests"))

from cvvidproc_b200 import _cabi, synth  # noqa: E402
from oracle import highlight_oracle as ho  # noqa: E402

GEOMS = {"1080p": (1920, 1080, "C3"), "512x256": (512, 256, "C4")}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def events_ms(fn, reps, stream=None):
    """ms per call of fn, CUDA events on `stream` (the stream fn's work goes to; None: torch's current stream)"""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    s.record(stream)
    for _ in range(reps):
        fn()
    e.record(stream)
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def kernel_us(fn, names, reps=5):
    """summed device time of kernels whose name contains one of `names`, per call"""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = {n: 0.0 for n in names}
    for ev in prof.key_averages():
        for n in names:
            if n in ev.key:
                tot[n] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return {n: v / reps for n, v in tot.items()}


def colour_of(grey):
    return np.ascontiguousarray(np.stack([grey, np.roll(grey, 9, axis=-1), 255 - grey], axis=-1))


def replicated(grey):
    return np.ascontiguousarray(np.repeat(grey[..., None], 3, axis=-1))


def probe_geometry(name, res):
    w, h, cfg = GEOMS[name]
    q = synth.CONFIG_PARAMS[cfg]
    npix = w * h
    # 3.2 GB (1080p) and 1.6 GB (512x256) of colour frames: larger than L2, and several launches' worth of frames
    n = 512 if name == "1080p" else 4096
    base = synth.synth_frames(100, 32, w, h, q["seed"], q["ndisks"])
    bg = np.sort(synth.synth_frames(0, 31, w, h, q["seed"], q["ndisks"]), axis=0)[15]
    grey = np.concatenate([base] * (n // 32 + 1))[:n]
    p = ho.canonical_params(bg)
    d_grey = torch.from_numpy(grey.reshape(n, npix)).cuda()
    # the grey frames replicated into three channels: a colour job then makes the grey job's masks (identity (2) of
    # tests/color_cases.py), so the two differ by the colour pass alone
    d_col = torch.from_numpy(replicated(grey).reshape(n, 3 * npix)).cuda()
    d_out = torch.empty((n, npix), dtype=torch.uint8, device="cuda")
    d_copy = torch.empty_like(d_col)
    out = {"frames": n}
    with _cabi.Context(0) as g, _cabi.Context(0) as c:
        g.highlight_begin(bg, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                          p.min_size_hyst, p.min_size_threshold)
        c.highlight_set_channels(3)
        c.highlight_begin(replicated(bg), np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo,
                          p.threshold_hi, p.min_size_hyst, p.min_size_threshold)
        # each call runs on its context's compute stream; the events go there too
        run_g = lambda: g.highlight_device(d_grey.data_ptr(), n, npix, d_out.data_ptr(), npix)  # noqa: E731
        run_c = lambda: c.highlight_device(d_col.data_ptr(), n, 3 * npix, d_out.data_ptr(), npix)  # noqa: E731
        sg, sc = torch.cuda.ExternalStream(g.stream), torch.cuda.ExternalStream(c.stream)
        ms_g, ms_c = events_ms(run_g, 5, sg), events_ms(run_c, 5, sc)
        ms_g2, ms_c2 = events_ms(run_g, 5, sg), events_ms(run_c, 5, sc)
        ms_copy = events_ms(lambda: d_copy.copy_(d_col), 10)
        k = kernel_us(run_c, ["color_diff_kernel", "highlight_fused"])
        g.highlight_end()
        c.highlight_end()
    per = k["color_diff_kernel"] / n
    moved = 3 * npix + npix  # frame in, d plane out (the background comes from L2 after the first frame)
    out.update(
        color_diff_us_per_frame=per,
        color_diff_GBps=moved / (per * 1e-6) / 1e9,
        copy_us_per_frame=ms_copy * 1e3 / n,
        copy_GBps=2 * 3 * npix / (ms_copy * 1e-3 / n) / 1e9,
        fused_us_per_frame_colour=k["highlight_fused"] / n,
        highlight_grey_us_per_frame=[ms_g * 1e3 / n, ms_g2 * 1e3 / n],
        highlight_colour_us_per_frame=[ms_c * 1e3 / n, ms_c2 * 1e3 / n],
    )
    res[name] = out


def probe_prepare(res):
    """the queue on decoded 1080p frames: RGB2GRAY preparation (grey job) against crop + colour difference (colour
    job), kernel time per frame from the profiler"""
    w, h, cfg = GEOMS["1080p"]
    q = synth.CONFIG_PARAMS[cfg]
    batch, nb = 32, 4
    grey = synth.synth_frames(100, batch, w, h, q["seed"], q["ndisks"])
    dec = colour_of(grey)
    bg = np.sort(synth.synth_frames(0, 31, w, h, q["seed"], q["ndisks"]), axis=0)[15]
    crop = (0, 0, w, h - 8)  # a crop, so that the preparation kernels run (full frames are copied as they are)
    x, y, cw, chh = crop
    p = ho.canonical_params(bg[y:y + chh, x:x + cw].copy())
    out = {}
    for what, channels, mode, name in (("rgb2gray_prepare", 1, 2, "frames_prepare_kernel"),
                                       ("crop_color_diff", 3, 0, "color_diff_kernel")):
        with _cabi.Context(0) as c:
            c.highlight_set_channels(channels)
            b = p.background if channels == 1 else colour_of(bg)[y:y + chh, x:x + cw].copy()
            c.highlight_begin(b, np.ascontiguousarray(p.struct_element), p.threshold, p.threshold_lo, p.threshold_hi,
                              p.min_size_hyst, p.min_size_threshold)
            c.highlight_queue_begin(2, batch, _cabi.FrameFormat.of((h, w, 3), mode, crop))

            def run():
                for _ in range(nb):
                    c.highlight_submit(dec)
                    c.highlight_next()

            k = kernel_us(run, [name], reps=2)
            out[what + "_us_per_frame"] = k[name] / (nb * batch)
            c.highlight_queue_end()
            c.highlight_end()
    res["queue_1080p"] = out


def probe_track(res, nframes):
    import cv2

    import cvvidproc_b200 as cvp
    import video_util

    w, h, cfg = GEOMS["1080p"]
    q = synth.CONFIG_PARAMS[cfg]
    grey = synth.synth_frames(0, nframes, w, h, q["seed"], q["ndisks"])
    frames = colour_of(grey)
    out = {"frames": nframes}
    with tempfile.TemporaryDirectory() as d:
        path = video_util.write_lossless(Path(d) / "colour1080.avi", frames)
        dec = video_util.read_all(path)
        bg_c = np.median(dec[:31], axis=0).astype(np.uint8)
        bg_g = cv2.cvtColor(bg_c, cv2.COLOR_RGB2GRAY)
        for label, kwargs, pack, bg in (("grayscale", {}, {"grayscale": True}, bg_g),
                                        ("colour", {"cvvp_color": True}, {}, bg_c)) * 2:
            p = ho.canonical_params(bg_g)
            hp = cvp.HighlightObjectsPack(bg, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                          p.min_size_hyst, p.min_size_threshold, p.width_border)
            t0 = time.perf_counter()
            cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(lambda **kw: kw["next_ID"], kwargs),
                                                    **pack))
            out.setdefault(label + "_ms_per_frame", []).append((time.perf_counter() - t0) * 1e3 / nframes)
    res["track_1080p"] = out


def main():
    prefix = Path(sys.argv[1])
    nframes = int(sys.argv[sys.argv.index("--track-frames") + 1]) if "--track-frames" in sys.argv else 300
    res = {"card": card()}
    for name in GEOMS:
        probe_geometry(name, res)
    probe_prepare(res)
    probe_track(res, nframes)
    prefix.parent.mkdir(parents=True, exist_ok=True)
    Path(str(prefix) + ".json").write_text(json.dumps(res, indent=1))
    lines = [f"card, power limit: {res['card']}"]
    for name in GEOMS:
        r = res[name]
        lines.append(f"{name} x 3, {r['frames']} frames: colour difference {r['color_diff_us_per_frame']:.2f} us/frame "
                     f"({r['color_diff_GBps']:.0f} GB/s frame + d); device copy of the colour frames "
                     f"{r['copy_us_per_frame']:.2f} us/frame ({r['copy_GBps']:.0f} GB/s read + write); highlight grey "
                     f"{r['highlight_grey_us_per_frame'][0]:.2f} / {r['highlight_grey_us_per_frame'][1]:.2f} us/frame, "
                     f"colour (the same frames in three channels) {r['highlight_colour_us_per_frame'][0]:.2f} / "
                     f"{r['highlight_colour_us_per_frame'][1]:.2f} us/frame (fused kernel in it "
                     f"{r['fused_us_per_frame_colour']:.2f})")
    qq = res["queue_1080p"]
    lines.append(f"queue 1080p decoded frames: RGB2GRAY preparation {qq['rgb2gray_prepare_us_per_frame']:.2f} us/frame, "
                 f"crop + colour difference {qq['crop_color_diff_us_per_frame']:.2f} us/frame")
    t = res["track_1080p"]
    lines.append(f"TrackObjects 1080p lossless colour video, {t['frames']} frames: grayscale=True "
                 f"{' / '.join(f'{v:.2f}' for v in t['grayscale_ms_per_frame'])} ms/frame, cvvp_color "
                 f"{' / '.join(f'{v:.2f}' for v in t['colour_ms_per_frame'])} ms/frame")
    Path(str(prefix) + ".txt").write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
