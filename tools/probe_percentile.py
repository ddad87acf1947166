"""Timing of the percentile backgrounds (cvvp_median_set_percentile) on one GPU.  Writes <out>/r4_percentile_probe.{json,txt}
with the GPU's name and power limit read in the same run.  CUDA events around device-resident calls on synthetic video
frames (cvvp_synth_frames_device; the scenes of synth.CONFIG_PARAMS C2, C5 and C3), each input larger than L2.

  1. on-chip select, 1920x1080 x 1000 frames (cvvp_median_device, median_pipe_kernel MODE 0), p in {0, 10, 50, 90, 100}
  2. counting path, 3840x2160 x 5000 frames (cvvp_median_device -> window pass + fallback tiles), same p; the elements
     the window pass left unresolved come from a one-rank sharded job over the same stack (phases 4, 5), which runs the
     same kernels
  3. rolling median, 1920x1080 x 600 frames, W = 101 (cvvp_median_rolling_device), p in {50, 90}

    python tools/probe_percentile.py [--out profiles] [--reps 5]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

from cvvidproc_b200 import _cabi, synth

PS = [0, 10, 50, 90, 100]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, stream, reps):
    fn()  # warm: module load, shape
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def make_stack(ctx, w, h, n, cfg):
    npix = w * h
    frames = torch.empty((n, npix), dtype=torch.uint8, device="cuda")
    p = synth.CONFIG_PARAMS[cfg]
    ctx.synth_frames_device(frames.data_ptr(), npix, w, h, 0, n, p["seed"], p["ndisks"])
    ctx.synchronize()
    return frames


def unresolved(nelem, frames, n, p):
    """elements the window pass leaves undecided at percentile p: a one-rank sharded job, phases 4 and 5"""
    c = _cabi.Context(0)
    try:
        c.median_set_percentile(p)
        c.median_shard_begin(nelem, 0, 1, n)
        c.median_shard_phase(4, frames.data_ptr(), n, nelem)
        c.median_shard_phase(5)
        left = c.median_shard_unresolved()
        c.median_shard_end()
        return left
    finally:
        c.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_percentile: no GPU (nothing here is measured without one)")
    ident = gpu_identity()
    print(json.dumps(ident), flush=True)
    ctx = _cabi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream)
    res = dict(ident, on_chip=[], counting=[], rolling=[])

    def dev_median(frames, n, nelem, out):
        return lambda: ctx.median_device(frames.data_ptr(), n, nelem, nelem, out.data_ptr())

    with torch.cuda.stream(stream):
        # 1. on-chip select
        w, h, n = 1920, 1080, 1000
        frames = make_stack(ctx, w, h, n, "C2")
        out = torch.empty(w * h, dtype=torch.uint8, device="cuda")
        for p in PS:
            ctx.median_set_percentile(p)
            ms = timed(dev_median(frames, n, w * h, out), stream, args.reps)
            res["on_chip"].append({"size": "1920x1080", "frames": n, "p": p, "ms": round(ms, 3),
                                   "GBps": round(n * w * h / (ms * 1e-3) / 1e9, 1)})
            print(json.dumps(res["on_chip"][-1]), flush=True)
        del frames
        torch.cuda.empty_cache()
        # 2. counting path
        w, h, n = 3840, 2160, 5000
        frames = make_stack(ctx, w, h, n, "C5")
        out = torch.empty(w * h, dtype=torch.uint8, device="cuda")
        for p in PS:
            ctx.median_set_percentile(p)
            ms = timed(dev_median(frames, n, w * h, out), stream, args.reps)
            left = unresolved(w * h, frames, n, p)
            res["counting"].append({"size": "3840x2160", "frames": n, "p": p, "ms": round(ms, 3),
                                    "GBps_one_read": round(n * w * h / (ms * 1e-3) / 1e9, 1), "unresolved_elements": left})
            print(json.dumps(res["counting"][-1]), flush=True)
        del frames
        torch.cuda.empty_cache()
        # 3. rolling median
        w, h, n, win = 1920, 1080, 600, 101
        frames = make_stack(ctx, w, h, n, "C3")
        bgs = torch.empty_like(frames)
        for p in (50, 90):
            ctx.median_set_percentile(p)
            ms = timed(lambda: ctx.median_rolling_device(frames.data_ptr(), n, w * h, w * h, win, 0, n, bgs.data_ptr(),
                                                         w * h), stream, args.reps)
            res["rolling"].append({"size": "1920x1080", "frames": n, "window": win, "p": p, "ms": round(ms, 3),
                                   "us_per_frame": round(ms / n * 1e3, 3)})
            print(json.dumps(res["rolling"][-1]), flush=True)
    ctx.close()
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / "r4_percentile_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    lines = [f"{ident['gpu']}, power limit {ident['power_limit']}, max SM clock {ident['max_sm_clock']}; CUDA events, "
             f"mean of {args.reps} calls after one warm-up", "",
             "on-chip select (median_device, MODE 0), 1920x1080 x 1000:"]
    lines += [f"  p={r['p']:3d}  {r['ms']:8.3f} ms  {r['GBps']:7.1f} GB/s" for r in res["on_chip"]]
    lines += ["", "counting path (median_device: window pass + fallback tiles), 3840x2160 x 5000:"]
    lines += [f"  p={r['p']:3d}  {r['ms']:8.3f} ms  {r['GBps_one_read']:7.1f} GB/s (one read of the stack)  "
              f"unresolved after the window pass: {r['unresolved_elements']}" for r in res["counting"]]
    lines += ["", "rolling median (median_rolling_device), 1920x1080 x 600, W = 101:"]
    lines += [f"  p={r['p']:3d}  {r['ms']:8.3f} ms  {r['us_per_frame']:7.3f} us/frame" for r in res["rolling"]]
    (out_dir / "r4_percentile_probe.txt").write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
