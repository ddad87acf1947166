"""Timing of the rolling-median background (csrc/median_roll.cu, cvvp_highlight_device_bg, TrackObjects with
kwargs["cvvp_background_window"]) on one GPU.  Writes <out>/r3_rolling_probe.{json,txt} with the GPU's name and power
limit read in the same run.

  1. rolling median, kernel-resident: CUDA events around cvvp_median_rolling_device over a device-resident stack, at
     1920x1080 and 512x256 for W in {25, 101, 255}; rate against the kernel's own bytes (every chunk reads W rows to
     build its window, then two rows per output whose window moves, and writes one row per output), as a share of the
     HBM rate measured here (a device-to-device copy of 4 GiB)
  2. rolling median + per-frame-background highlight against today's static highlight, Mpx-frames/s
  3. TrackObjects per frame on a lossless 1080p video: static, rolling (W = 101), and the decoder alone

    python tools/probe_rolling.py [--out profiles] [--video-frames 1000]
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch

from cvvidproc_b200 import _cabi, synth
from oracle import highlight_oracle as ho

SIZES = [("1080p", 1920, 1080, 600), ("512x256", 512, 256, 4000)]
WINDOWS = [25, 101, 255]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def hbm_rate():
    a = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    del a, b
    return 2 * (4 << 30) / (ms * 1e-3)


def roll_bytes(nelem, n, w, sm_count):
    """bytes the kernel moves for outputs [0, n): mirrors the chunking of median_roll_launch"""
    weff = min(w, n)
    tiles = (nelem + 127) // 128
    nchunks = max(1, min(-(-12 * sm_count // tiles), max(1, n // weff), 65535))
    chunk = -(-n // nchunks)
    nchunks = -(-n // chunk)
    moves = max(0, min(n - 1, n - weff + w // 2) - (w // 2 + 1) + 1)
    return nelem * (nchunks * weff + 2 * moves + n)


def timed(fn, stream, reps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_rates(ctx, peak):
    rows = []
    stream = torch.cuda.ExternalStream(ctx.stream)
    for name, w_, h_, n in SIZES:
        npix = w_ * h_
        p = synth.CONFIG_PARAMS["C3" if name == "1080p" else "C4"]
        frames = torch.empty((n, npix), dtype=torch.uint8, device="cuda")
        ctx.synth_frames_device(frames.data_ptr(), npix, w_, h_, 0, n, p["seed"], p["ndisks"])
        bgs = torch.empty_like(frames)
        masks = torch.empty_like(frames)
        ctx.synchronize()
        static_bg = torch.empty(npix, dtype=torch.uint8, device="cuda")
        ctx.median_device(frames.data_ptr(), min(n, 255), npix, npix, static_bg.data_ptr())
        ctx.synchronize()
        hp = ho.canonical_params(static_bg.cpu().numpy().reshape(h_, w_))
        ctx.highlight_begin(hp.background, hp.struct_element, hp.threshold, hp.threshold_lo, hp.threshold_hi,
                            hp.min_size_hyst, hp.min_size_threshold, hp.width_border)
        with torch.cuda.stream(stream):
            static_ms = timed(lambda: ctx.highlight_device(frames.data_ptr(), n, npix, masks.data_ptr(), npix), stream, 3)
            for w in WINDOWS:
                med_ms = timed(lambda: ctx.median_rolling_device(frames.data_ptr(), n, npix, npix, w, 0, n, bgs.data_ptr(),
                                                                 npix), stream, 3)
                hl_ms = timed(lambda: ctx.highlight_device_bg(frames.data_ptr(), n, npix, bgs.data_ptr(), npix,
                                                              masks.data_ptr(), npix), stream, 3)
                nbytes = roll_bytes(npix, n, w, ctx.sm_count)
                rate = nbytes / (med_ms * 1e-3)
                rows.append({"size": name, "frames": n, "window": w, "median_ms": round(med_ms, 3),
                             "median_us_per_frame": round(med_ms / n * 1e3, 3), "median_bytes": nbytes,
                             "median_GBps": round(rate / 1e9, 1), "median_share_of_hbm": round(rate / peak, 3),
                             "median_plus_bg_highlight_Mpx_frames_per_s": round(n * npix / 1e6 / ((med_ms + hl_ms) * 1e-3)),
                             "bg_highlight_us_per_frame": round(hl_ms / n * 1e3, 3),
                             "static_highlight_us_per_frame": round(static_ms / n * 1e3, 3),
                             "static_highlight_Mpx_frames_per_s": round(n * npix / 1e6 / (static_ms * 1e-3))})
                print(json.dumps(rows[-1]), flush=True)
        ctx.highlight_end()
        del frames, bgs, masks
        torch.cuda.empty_cache()
    return rows


def track_times(nframes):
    import cv2

    import cvvidproc_b200 as cvp

    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tests"))
    import video_util

    p = synth.CONFIG_PARAMS["C3"]
    with tempfile.TemporaryDirectory() as td:
        frames = synth.synth_frames(0, nframes, 1920, 1080, p["seed"], p["ndisks"])
        path = video_util.write_lossless(Path(td) / "c3.avi", frames)
        bg = frames[: min(nframes, 255)].copy()
        bg = np.median(bg, axis=0).astype(np.uint8)
        del frames
        hp = ho.canonical_params(bg)
        pack = cvp.HighlightObjectsPack(hp.background, hp.struct_element, hp.threshold, hp.threshold_lo, hp.threshold_hi,
                                        hp.min_size_hyst, hp.min_size_threshold, hp.width_border)

        def cb(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs):
            return next_ID

        out = {"video": f"FFV1 1920x1080 x {nframes}"}
        t = time.perf_counter()
        cap = cv2.VideoCapture(path)
        while cap.read()[0]:
            pass
        out["decode_ms_per_frame"] = round((time.perf_counter() - t) * 1e3 / nframes, 3)
        for label, kw in (("static", {}), ("rolling_w101", {"cvvp_background_window": 101})):
            cvp.TrackObjects(cvp.VidObjectTrackPack(path, pack, cvp.AssignObjectsPack(cb, dict(kw)), vid_is_grayscale=True,
                                                    frame_limit=32))  # warm: pools, module load
            t = time.perf_counter()
            cvp.TrackObjects(cvp.VidObjectTrackPack(path, pack, cvp.AssignObjectsPack(cb, dict(kw)), vid_is_grayscale=True))
            out[f"track_{label}_ms_per_frame"] = round((time.perf_counter() - t) * 1e3 / nframes, 3)
            print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--video-frames", type=int, default=1000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_rolling: no GPU (nothing here is measured without one)")
    ident = gpu_identity()
    print(json.dumps(ident), flush=True)
    peak = hbm_rate()
    print(f"measured HBM rate (4 GiB device copy): {peak / 1e12:.2f} TB/s", flush=True)
    ctx = _cabi.Context(0)
    kernels = kernel_rates(ctx, peak)
    ctx.close()
    track = track_times(args.video_frames)
    res = dict(ident, measured_hbm_TBps=round(peak / 1e12, 3), kernels=kernels, track=track)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "r3_rolling_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    lines = [f"{ident['gpu']}, power limit {ident['power_limit']}, max SM clock {ident['max_sm_clock']}; "
             f"measured HBM rate {peak / 1e12:.2f} TB/s (4 GiB device copy)", "",
             "size     frames  W    median us/frame  GB/s   share  bg-highlight us/frame  static us/frame  "
             "median+bg-hl Mpx-f/s  static Mpx-f/s"]
    for r in kernels:
        lines.append(f"{r['size']:8s} {r['frames']:6d} {r['window']:4d} {r['median_us_per_frame']:14.3f} {r['median_GBps']:7.1f} "
                     f"{r['median_share_of_hbm']:6.3f} {r['bg_highlight_us_per_frame']:20.3f} "
                     f"{r['static_highlight_us_per_frame']:16.3f} {r['median_plus_bg_highlight_Mpx_frames_per_s']:21d} "
                     f"{r['static_highlight_Mpx_frames_per_s']:15d}")
    lines += ["", "TrackObjects, " + track["video"] + ": " + ", ".join(f"{k} {v}" for k, v in track.items() if k != "video")]
    (out / "r3_rolling_probe.txt").write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
