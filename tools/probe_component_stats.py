"""Timing of the component statistics (cvvp_highlight_set_component_stats) on one GPU.  Writes
<out>/r6_component_stats_probe.{json,txt} with the GPU's name and power limit read in the same run.  CUDA events around
cvvp_highlight_device_cc (the fused kernel with its components phase, one launch per call) on synthetic video frames
generated on the device (cvvp_synth_frames_device), background = the median of the first 31 frames; every input is
larger than L2 (126 MB), so each pass streams its frames from HBM:

  C3 scene, 1920x1080 x 1024 frames (2.1 GB)
  C4 scene,  512x256  x 8192 frames (1.1 GB)
  all-foreground, the C3 frames with negative thresholds: every mask is one component of 1080 runs of 1920 pixels

Statistics off and on are timed in alternation: `--reps` rounds of one sample per row after a warm-up pass per row, a
sample being `--calls` calls back to back (one job); the json keeps every sample, the text the median per row.

    python tools/probe_component_stats.py [--out profiles] [--reps 7] [--calls 20]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch

from cvvidproc_b200 import _cabi, synth
from oracle import highlight_oracle as ho

SCENES = [("C3", "C3", 1920, 1080, 1024), ("C4", "C4", 512, 256, 8192), ("all-fg", "C3", 1920, 1080, 1024)]
MAX_COMPS = 256


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def scene(ctx, name, cfg, w, h, n):
    npix = w * h
    frames = torch.empty((n, npix), dtype=torch.uint8, device="cuda")
    q = synth.CONFIG_PARAMS[cfg]
    ctx.synth_frames_device(frames.data_ptr(), npix, w, h, 0, n, q["seed"], q["ndisks"])
    ctx.synchronize()
    bg = torch.sort(frames[:31], dim=0).values[15].cpu().numpy().reshape(h, w)
    if name == "all-fg":  # negative thresholds pass every pixel
        return frames, ho.HighlightParams(bg, np.ones((1, 1), np.uint8), -2, -2, -2, 0, 0, 0)
    return frames, ho.canonical_params(bg)


def one_pass(ctx, frames, out, comps, ncomps, p, stats, stream, calls=1):
    """`calls` calls over every frame, timed with CUDA events on `stream`; the job is begun outside the timed window.
    Returns the milliseconds of one call and the mean component count."""
    n, npix = frames.shape
    ctx.highlight_set_component_stats(stats)
    ctx.highlight_begin(p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi, p.min_size_hyst,
                        p.min_size_threshold, p.width_border)
    try:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(calls):
            rc = ctx._lib.cvvp_highlight_device_cc(ctx.handle, frames.data_ptr(), n, npix, out.data_ptr(), npix,
                                                   comps.data_ptr(), MAX_COMPS, ncomps.data_ptr(), None, 0,
                                                   stream.cuda_stream)
            ctx._check(rc)
        e1.record(stream)
        torch.cuda.synchronize()
        mean_comps = float(ncomps.float().mean().item())
    finally:
        ctx.highlight_end()
        ctx.highlight_set_component_stats(False)
    return e0.elapsed_time(e1) / calls, mean_comps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_component_stats needs a GPU")
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    ident = gpu_identity()
    ctx = _cabi.Context(0)
    stream = torch.cuda.Stream()
    res = {"identity": ident, "reps": args.reps, "calls": args.calls, "max_comps": MAX_COMPS, "scenes": []}
    lines = [f"# {ident['gpu']}, power limit {ident['power_limit']}, max SM clock {ident['max_sm_clock']}",
             f"# fused kernel with components (cvvp_highlight_device_cc, max_comps {MAX_COMPS}), one launch over all "
             "frames per call; inputs larger than L2",
             f"# {args.reps} samples per row, rows alternated; a sample = {args.calls} calls back to back",
             "# scene   geometry    frames  stats  median us/frame  min us/frame  max us/frame  components/frame"]
    for name, cfg, w, h, n in SCENES:
        frames, p = scene(ctx, name, cfg, w, h, n)
        out = torch.empty_like(frames)
        comps = torch.zeros((n, MAX_COMPS * 104), dtype=torch.uint8, device="cuda")
        ncomps = torch.zeros(n, dtype=torch.int32, device="cuda")
        rows = {"off": False, "on": True}
        for stats in rows.values():  # warm-up
            one_pass(ctx, frames, out, comps, ncomps, p, stats, stream)
        passes = {row: [] for row in rows}
        ncomp = {}
        for _ in range(args.reps):
            for row, stats in rows.items():
                ms, ncomp[row] = one_pass(ctx, frames, out, comps, ncomps, p, stats, stream, args.calls)
                passes[row].append(1000.0 * ms / n)
        res["scenes"].append({"scene": name, "width": w, "height": h, "frames": n, "us_per_frame": passes,
                              "components_per_frame": ncomp})
        for row, v in passes.items():
            lines.append(f"  {name:7s} {w}x{h:<5d}  {n:6d}  {row:5s}  {statistics.median(v):15.2f}  {min(v):12.2f}  "
                         f"{max(v):12.2f}  {ncomp[row]:16.1f}")
        del frames, out, comps
        torch.cuda.empty_cache()
    ctx.close()
    (out_dir / "r6_component_stats_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    (out_dir / "r6_component_stats_probe.txt").write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
