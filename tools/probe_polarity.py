"""Timing of the object polarities (cvvp_highlight_set_polarity) on one GPU.  Writes <out>/r5_polarity_probe.{json,txt}
with the GPU's name and power limit read in the same run.  CUDA events around cvvp_highlight_device (the fused kernel,
one launch per call) on synthetic video frames generated on the device (cvvp_synth_frames_device), background = the
median of the first 31 frames; every input is larger than L2 (126 MB), so each pass streams its frames from HBM:

  C3 scene, 1920x1080 x 1024 frames (2.1 GB)
  C4 scene,  512x256  x 8192 frames (1.1 GB)

The polarities are timed in alternation: `--reps` rounds of one sample per row after a warm-up pass per row, a sample
being `--calls` passes back to back (one job); the json keeps every sample, the text the median per row.  The scenes have dark objects, so "bright" finds little in them and its later
phases have less to do; the row "bright, inverted" runs it on 255 - frames against 255 - background, which gives the
same masks as "dark" (identity (1) of tests/polarity_cases.py) and so the same work after the difference image.

    python tools/probe_polarity.py [--out profiles] [--reps 7] [--calls 20]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

from cvvidproc_b200 import _cabi, synth
from oracle import highlight_oracle as ho

POLARITIES = {"dark": 0, "bright": 1, "both": 2}
ROWS = [("dark", "dark", False), ("bright", "bright", False), ("both", "both", False), ("bright, inverted", "bright", True)]
SCENES = [("C3", 1920, 1080, 1024), ("C4", 512, 256, 8192)]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def scene(ctx, cfg, w, h, n):
    npix = w * h
    frames = torch.empty((n, npix), dtype=torch.uint8, device="cuda")
    q = synth.CONFIG_PARAMS[cfg]
    ctx.synth_frames_device(frames.data_ptr(), npix, w, h, 0, n, q["seed"], q["ndisks"])
    ctx.synchronize()
    bg = torch.sort(frames[:31], dim=0).values[15].cpu().numpy().reshape(h, w)
    return frames, ho.canonical_params(bg), ho.canonical_params(255 - bg)


def one_pass(ctx, frames, out, p, polarity, stream, calls=1):
    """`calls` calls over every frame, timed with CUDA events on `stream`; the job is begun outside the timed window.
    Returns the milliseconds of one call and the white fraction of the masks."""
    n, npix = frames.shape
    ctx.highlight_set_polarity(POLARITIES[polarity])
    ctx.highlight_begin(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi, p.min_size_hyst,
                        p.min_size_threshold, p.width_border)
    try:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(calls):
            ctx.highlight_device(frames.data_ptr(), n, npix, out.data_ptr(), npix, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        white = float(out[:: max(1, n // 16)].float().mean().item() / 255.0)
    finally:
        ctx.highlight_end()
        ctx.highlight_set_polarity(0)
    return e0.elapsed_time(e1) / calls, white


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_polarity needs a GPU")
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    ident = gpu_identity()
    ctx = _cabi.Context(0)
    stream = torch.cuda.Stream()
    res = {"identity": ident, "reps": args.reps, "calls": args.calls, "scenes": []}
    lines = [f"# {ident['gpu']}, power limit {ident['power_limit']}, max SM clock {ident['max_sm_clock']}",
             "# fused kernel (cvvp_highlight_device), one launch over all frames per call; inputs larger than L2",
             f"# {args.reps} samples per row, rows alternated; a sample = {args.calls} calls back to back",
             "# scene  geometry    frames  row               median us/frame  min us/frame  max us/frame  white fraction"]
    for cfg, w, h, n in SCENES:
        frames, p, p_inv = scene(ctx, cfg, w, h, n)
        inv = 255 - frames
        out = torch.empty_like(frames)
        args_of = {row: (inv if flip else frames, p_inv if flip else p, pol) for row, pol, flip in ROWS}
        for row in args_of:  # warm-up: module load, scratch, the polarity's branch
            f, q, pol = args_of[row]
            one_pass(ctx, f, out, q, pol, stream)
        passes = {row: [] for row in args_of}
        white = {}
        for _ in range(args.reps):
            for row in args_of:
                f, q, pol = args_of[row]
                ms, white[row] = one_pass(ctx, f, out, q, pol, stream, args.calls)
                passes[row].append(1000.0 * ms / n)
        res["scenes"].append({"scene": cfg, "width": w, "height": h, "frames": n, "us_per_frame": passes,
                              "white_fraction": white})
        for pol, v in passes.items():
            lines.append(f"  {cfg}     {w}x{h:<5d}  {n:6d}  {pol:16s}  {statistics.median(v):15.2f}  {min(v):12.2f}  "
                         f"{max(v):12.2f}  {white[pol]:14.4f}")
        del frames, inv, out
        torch.cuda.empty_cache()
    ctx.close()
    (out_dir / "r5_polarity_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    (out_dir / "r5_polarity_probe.txt").write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
