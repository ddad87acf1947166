#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json): temporal-median background + per-frame highlight.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C1..C5]      # this repo's CUDA path
    python bench.py --impl reference [...]                                       # the reference's CPU path
    python bench.py --dump-outputs DIR [...]      # also write the outputs of the last timed step to DIR (OutputDump)

The line's headline (`metric`, `value`, `e2e`, `roofline`, `cpu_baseline`) is the workload `--config` names; the default
is C2 = BASELINE.json configs[1], the configuration the metric is quoted on:

    C1  640x480 x 100 frames       median       (the reference's own CPU-runnable case; launch-latency bound)
    C2  1920x1080 x 1000 frames    median       N > 1: weak scaling, every GPU holds its own 1000-frame chunk
    C3  1080p x 10 000 frames      highlight    N > 1: frames split over the GPUs
    C4  512x256 x 200 000 frames   highlight    N > 1: frames split over the GPUs
    C5  3840x2160 x 5000 frames    median       N > 1: frames split over the GPUs (strong scaling)

One "step" = one pass of the hot path over the whole workload.  `value` is megapixel-frames/s with the input already
resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` is the same metric through the C ABI's
host-buffer calls with the frames in pinned host memory, H2D and D2H inside the timed region.  Every input is far
larger than the 126 MB L2, so no flush is needed between timed iterations.

The default (C2) line also carries the other halves of BASELINE's metric as objects of their own, each with `value`,
`e2e`, `roofline` and a parity spot check: `highlight` (C3 geometry, 1024 frames per GPU and step), `c5_median`,
`c4_highlight` and, at one GPU, `frame_source` (the stage in front of both operators) and `track_e2e` (the drop-in
`TrackObjects` on a lossless 1080p video with the host tracker in the loop, the reference-shaped cv2 pipeline timed
beside it).

N > 1 (one process per GPU under torchrun): the median shards over FRAME chunks (BASELINE north_star); the merge is
the count exchange of csrc/median_shard.cu -- one pass of window counting whose 20-byte records are stored into the
owner rank's memory over NVLink by the counting kernel, and the two-round nibble exchange behind it for elements the
one pass cannot decide (none on a video background).  `--median-sharding rows` instead splits the single C2 stack into
row bands (no data-path collective; strong scaling).  The highlight stage shards by frame with no collective.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

# seeds / disk counts: SURVEY.md 8d (the same table as cvvidproc_b200/synth.py; repeated here because the reference arm
# must not import the package)
CONFIGS = {
    "C1": dict(kind="median", width=640, height=480, nframes=100, seed=1, ndisks=4, scaling="strong",
               name="C1: 640x480 uint8 x 100 frames, temporal median (BASELINE.json configs[0])"),
    "C2": dict(kind="median", width=1920, height=1080, nframes=1000, seed=2, ndisks=30, scaling="weak",
               name="C2: 1920x1080 uint8 x 1000 frames, temporal median (BASELINE.json configs[1])"),
    "C3": dict(kind="highlight", width=1920, height=1080, nframes=10000, seed=3, ndisks=30, scaling="strong",
               name="C3: 1920x1080 uint8 x 10000 frames, per-frame highlight (BASELINE.json configs[2]), background = "
                    "device median of the stream's first 255 frames, canonical parameters"),
    "C4": dict(kind="highlight", width=512, height=256, nframes=200000, seed=4, ndisks=6, scaling="strong",
               name="C4: 512x256 uint8 x 200000 frames, per-frame highlight sharded by frame (BASELINE.json configs[3]), "
                    "background = device median of the stream's first 255 frames, canonical parameters"),
    "C5": dict(kind="median", width=3840, height=2160, nframes=5000, seed=5, ndisks=60, scaling="strong",
               name="C5: 3840x2160 uint8 x 5000 frames, temporal median, frames split over the GPUs (BASELINE.json configs[4])"),
}
HL_STEP = dict(kind="highlight", width=1920, height=1080, seed=3, ndisks=30, frames_per_gpu=1024,
               name="C3 geometry: 1920x1080 uint8 frames, per-frame highlight, 1024 frames per GPU and step, background = "
                    "device median of the stream's first 255 frames, canonical parameters")
CANONICAL_HIGHLIGHT = dict(struct_element=((0, 0, 1, 0), (1, 1, 1, 1), (1, 1, 1, 1), (1, 1, 1, 1)), threshold=14,
                           threshold_lo=7, threshold_hi=16, min_size_hyst=20, min_size_threshold=20, width_border=5)
UNIT = "Mpx-frames/s"
FALLBACK_HBM_GBS = 6650.0
PINNED_CAP_BYTES = 2_200_000_000  # pinned host memory a rank's e2e leg may hold
L2_BYTES = 126 << 20


def metric_name(cfg):
    if cfg["kind"] == "median":
        return f"megapixel-frames/sec (temporal-median background, {cfg['width']}x{cfg['height']} x {cfg['nframes']}-frame stack)"
    return f"megapixel-frames/sec (per-frame highlight, {cfg['width']}x{cfg['height']} x {cfg['nframes']} frames)"


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def load_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def load_traffic(name: str):
    """dram bytes per launch of a kernel from its committed `ncu --set full` capture under profiles/ (bench.py cannot
    read DRAM counters itself); returns (bytes, where it came from)."""
    p = REPO / "profiles" / name
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), f"profiles/{name} (ncu --set full capture, not measured in this run)"
        except Exception:
            pass
    return None, None


def roofline(algo_bytes, kernel_ms, kernel, traffic_file=None, note=None):
    peak, peak_src = load_peaks()
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, tsrc = load_traffic(traffic_file) if traffic_file else (None, None)
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
           "peak_source": peak_src, "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": algo_bytes}
    if tsrc:
        out["traffic_source"] = tsrc
    if note:
        out["note"] = note
    return out


class ClockSampler:
    """Polls NVML for SM clock and throttle reasons while a timed region is active."""

    def __init__(self, device_index: int):
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.active = False
        self._stop = False
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = None
            try:
                import torch

                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            except Exception:
                pass
            self.h = None
            if uuid:
                for cand in (uuid, "GPU-" + uuid):
                    try:
                        self.h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        try:
                            self.h = pynvml.nvmlDeviceGetHandleByUUID(cand)
                            break
                        except Exception:
                            continue
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    _REASONS = {
        "hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
        "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2,
        "display_clock_setting": 0x100,
    }

    def _loop(self):
        nv = self.nv
        while not self._stop:
            if self.active:
                try:
                    mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    try:
                        mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.samples.append(mhz)
                    for name, bit in self._REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        if self.nv is None:
            return
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop = True
        if self._thread:
            self._thread.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


class OutputDump:
    """--dump-outputs DIR: the arrays the timed path returned in its last step, written after the timed steps as
    DIR/<name>.npy in float32 (the uint8 results are exact in it; the tracker's records stay float64), so that two builds
    can be compared output for output: the inputs are seeded and identical from run to run.  The run declares up front
    the arrays it will write, and each one may take an equal share of what TOTAL_BYTES has left.  An array larger than
    its share keeps a fixed, seeded sample of its entries along the first axis (frames of a stack of masks, rows of an
    image), whose positions go to DIR/<name>_index.npy (float64).

    Rank 0 alone writes.  A median is the whole image at any world size; a highlight stack is rank 0's share of the
    frames, so its sample is the same only between runs on the same number of GPUs."""

    TOTAL_BYTES = 64 << 20

    def __init__(self, path, names):
        self.dir = Path(path) if path else None
        self.pending = list(names)
        self.written = 0
        if self.dir is not None:
            self.dir.mkdir(parents=True, exist_ok=True)

    def add(self, name: str, arr) -> None:
        """arr: a numpy array or a torch tensor on any device, indexed along its first axis before any copy to the host."""
        if self.dir is None:
            return
        self.pending.remove(name)  # a name the run did not declare is an error: it would take a share nobody left it
        share = (self.TOTAL_BYTES - self.written) // (len(self.pending) + 1)
        n = arr.shape[0]
        entry_bytes = int(np.prod(arr.shape[1:])) * (8 if arr.dtype == np.float64 else 4)
        index = None
        if n * entry_bytes > share:
            k = share // (entry_bytes + 8)
            if k < 1:
                raise RuntimeError(f"--dump-outputs: one entry of {name} is larger than its share of {share} bytes")
            index = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
            if hasattr(arr, "cpu"):
                import torch

                arr = arr[torch.as_tensor(index, device=arr.device)]
            else:
                arr = arr[index]
        host = arr.cpu().numpy() if hasattr(arr, "cpu") else np.asarray(arr)
        host = host.astype(np.float64 if host.dtype == np.float64 else np.float32)
        np.save(self.dir / f"{name}.npy", host)
        self.written += host.nbytes
        if index is not None:
            np.save(self.dir / f"{name}_index.npy", index.astype(np.float64))
            self.written += index.size * 8


def bind_near_gpu(device_index: int) -> int:
    """Pin this process to the CPUs NVML reports as local to the GPU, so that the pinned host buffers it allocates
    afterwards come from that NUMA node.  Returns the number of CPUs in the set (0: left unchanged)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def shard_plan(height: int, rank: int, world: int):
    """Row-band partition (the reference's own spatial sharding, cv_vid_frames_generator_algo.h:159-164, with horizontal
    bands instead of vertical strips so that every band is contiguous in memory)."""
    base = height // world
    row0 = base * rank
    nrows = base if rank < world - 1 else height - row0
    return row0, nrows


def frame_chunk(nframes: int, rank: int, world: int):
    base, extra = divmod(nframes, world)
    return rank * base + min(rank, extra), base + (1 if rank < extra else 0)


# ------------------------------------------------------------------------------------------------
# CPU legs (test infrastructure under oracle/: the reference's class, its C port, the host frame generator)
# ------------------------------------------------------------------------------------------------
_SIG = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]


def cpu_median_fn():
    """oracle/_ref (the reference's own class, kind='reference') when it was built, else the C port."""
    ref = REPO / "oracle" / "_ref" / "libcvvp_median_ref.so"
    port = REPO / "oracle" / "_build" / "libcvvp_oracle.so"
    if ref.exists():
        lib, name, kind = ctypes.CDLL(str(ref)), "cvvp_ref_median", "reference"
    elif port.exists():
        lib, name, kind = ctypes.CDLL(str(port)), "cvvp_oracle_median", "port"
    else:
        raise RuntimeError("neither oracle/_ref nor oracle/_build is built; run __graft_entry__.build()")
    fn = getattr(lib, name)
    fn.argtypes = _SIG
    fn.restype = ctypes.c_int

    def run(frames: np.ndarray, nthreads: int) -> np.ndarray:
        n = frames.shape[0]
        nelem = int(np.prod(frames.shape[1:]))
        out = np.empty(nelem, np.uint8)
        rc = fn(frames.ctypes.data, n, nelem, frames.strides[0], 0, nthreads, out.ctypes.data)
        if rc != 0:
            raise RuntimeError(f"{name} failed: {rc}")
        return out

    return run, kind


def host_synth(cfg, first, n, rows, nthreads):
    """rows [0, rows) of frames first .. first+n-1 of the config's stream, generated on the host cores by
    oracle/synth_oracle.c (bit-identical to cvvidproc_b200/synth.py and csrc/synth.cu)."""
    lib = ctypes.CDLL(str(REPO / "oracle" / "_build" / "libcvvp_oracle.so"))
    fn = lib.cvvp_oracle_synth_frames
    fn.argtypes = [ctypes.c_void_p, ctypes.c_size_t] + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 2 + [ctypes.c_uint32, ctypes.c_int,
                                                                                                        ctypes.c_int]
    fn.restype = ctypes.c_int
    out = np.empty((n, rows, cfg["width"]), np.uint8)
    rc = fn(out.ctypes.data, rows * cfg["width"], cfg["width"], cfg["height"], 0, rows, first, n, cfg["seed"], cfg["ndisks"], nthreads)
    if rc != 0:
        raise RuntimeError(f"cvvp_oracle_synth_frames failed: {rc}")
    return out


def cpu_highlight_rate(frames: np.ndarray, bg: np.ndarray, threads: int, seconds: float = 12.0):
    """cv2 restatement of highlight_objects_algo.cpp (oracle/highlight_oracle.py), one frame per task, cv2 internal
    threading off, `threads` Python threads (cv2 releases the GIL) -- the reference's frame-level data parallelism
    (cv_vid_objecttrack_helpers.cpp:72-84).  Returns (Mpx-frames/s, frames done, last mask)."""
    import concurrent.futures as cf

    import cv2

    from oracle import highlight_oracle as ho

    cv2.setNumThreads(1)
    p = ho.canonical_params(bg)
    n = frames.shape[0]
    done = 0
    last = None
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(max_workers=threads) as ex:
        while time.perf_counter() - t0 < seconds:
            res = list(ex.map(lambda i: ho.highlight_objects(frames[i % n].copy(), p), range(done, done + 2 * threads)))
            done += len(res)
            last = res[-1]
    dt = time.perf_counter() - t0
    return frames.shape[1] * frames.shape[2] * done / 1e6 / dt, done, last


def job_config(cfg, world, args):
    """The `config` object of a line: identical in both arms (the driver compares them)."""
    c = {"workload": cfg["name"], "width": cfg["width"], "height": cfg["height"], "nframes": cfg["nframes"], "seed": cfg["seed"],
         "ndisks": cfg["ndisks"], "n_gpus": world}
    if cfg["kind"] == "median":
        if world > 1 and cfg["scaling"] == "weak" and args.median_sharding == "frames":
            c["nframes"] = cfg["nframes"] * world
            c["frames_per_gpu"] = cfg["nframes"]
            c["sharding"] = (f"frame chunks x{world}: every GPU holds its own {cfg['nframes']}-frame chunk, the job is the median "
                             f"of the {cfg['nframes'] * world}-frame stack")
        elif world > 1 and args.median_sharding == "rows" and cfg["scaling"] == "weak":
            c["sharding"] = f"row bands x{world}, no data-path collective"
        elif world > 1:
            c["sharding"] = f"frame chunks x{world}: the {cfg['nframes']} frames are split over the GPUs"
        else:
            c["sharding"] = "single GPU"
    else:
        c["sharding"] = "single GPU" if world == 1 else f"by frame x{world}, no collective"
    per_gpu = cfg["width"] * cfg["height"] * (cfg["nframes"] if (cfg["kind"] == "median" and cfg["scaling"] == "weak") else
                                               -(-cfg["nframes"] // world))
    c["l2"] = ("the input of every GPU exceeds the 126 MB L2 many times over; no flush needed" if per_gpu > 4 * L2_BYTES else
               "the input fits the 126 MB L2: a 256 MB buffer is written between timed iterations (outside the timed events)")
    return c


def run_reference_arm(args, rank: int, world: int):
    """The reference's own CPU implementation of the path on the host cores: HistogramMedianAlgo (oracle/_ref, compiled
    from /root/reference) for a median config, the cv2 restatement of HighlightObjects for a highlight config.  Loads
    nothing of this repo's CUDA side (no package import)."""
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    conf = job_config(cfg, world, args)
    W, H = cfg["width"], cfg["height"]
    if cfg["kind"] == "median":
        nframes = conf["nframes"]
        run, kind = cpu_median_fn()
        # the whole frame when its stack fits a few GB of host memory, else the largest band of rows that does
        rows = int(min(H, max(8, 4_200_000_000 // (W * nframes))))
        frames = host_synth(cfg, 0, nframes, rows, cores)
        # keep the whole run within a few minutes: shrink the band if one step is slow
        t0 = time.perf_counter()
        run(frames, cores)
        t1 = time.perf_counter() - t0
        budget = 150.0 / max(1, args.steps + args.warmup)
        if t1 > budget:
            rows = max(8, int(rows * budget / t1))
            frames = np.ascontiguousarray(frames[:, :rows])
        for _ in range(max(0, args.warmup - 1)):
            run(frames, cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            run(frames, cores)
        dt = (time.perf_counter() - t0) / args.steps
        mpxf = rows * W * nframes / 1e6
        sample = (f"{'the whole frame' if rows == H else f'rows [0,{rows})'} of all {nframes} frames ({mpxf:.1f} Mpx-frames per "
                  f"step), frames resident in host memory, {cores} worker threads each owning a strip "
                  f"(cv_vid_bg_helpers.cpp:105-117)")
    else:
        from oracle import highlight_oracle as ho  # noqa: F401

        kind = "port"
        st = host_synth(cfg, 0, 33, H, cores)
        bg = np.sort(st, axis=0)[16]
        nfr = 16 if W * H > 500_000 else 256
        frames = host_synth(cfg, 1000, nfr, H, cores)
        seconds = max(2.0, min(10.0, 120.0 / max(1, args.steps + args.warmup)))
        cpu_highlight_rate(frames, bg, cores, seconds=1.0)
        rates = []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r, done, _ = cpu_highlight_rate(frames, bg, cores, seconds=seconds)
            rates.append(r)
        dt = (time.perf_counter() - t0) / args.steps
        mpxf = float(np.mean(rates)) * dt
        sample = (f"{nfr} frames of the stream cycled for {seconds:.0f} s per step, cv2 restatement of highlight_objects_algo.cpp, "
                  f"{cores} threads x cv2.setNumThreads(1), background = median of 33 frames")
    value = mpxf / dt
    line = {
        "impl": "reference", "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak" if (cfg["scaling"] == "weak" and args.median_sharding == "frames") else "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": conf,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------
class Env:
    """What every GPU leg needs: the context, torch, the process group, the stream."""

    def __init__(self, args, rank, local_rank, world):
        import torch

        from cvvidproc_b200 import _cabi

        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback")
        self.torch, self.cabi, self.args = torch, _cabi, args
        self.rank, self.local_rank, self.world = rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        if world > 1:
            bind_near_gpu(local_rank)
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.ctx = _cabi.Context(local_rank)
        self.lib = _cabi.load()
        self.dump = OutputDump(args.dump_outputs if rank == 0 else None, dump_names(args, world))
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def all_true(self, flag: bool) -> bool:
        t = self.torch.tensor([1 if flag else 0], dtype=self.torch.int32, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t[0]))

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)

    def close(self):
        self.ctx.close()
        if self.dist is not None:
            self.dist.destroy_process_group()


def pinned_prefix(E: Env, stack, n_rank, nelem):
    """Frames [0, n0) of the rank's resident stack copied into pinned host memory (outside every timed region); n0 is
    all of them when they fit PINNED_CAP_BYTES.  The e2e legs push this buffer ceil(n / n0) times when the chunk is
    larger (the bytes that cross the link are the workload's; a rank does not hold 41 GB of pinned memory)."""
    n0 = int(max(1, min(n_rank, PINNED_CAP_BYTES // nelem)))
    pinned = E.cabi.PinnedBuffer(n0 * nelem)
    host = pinned.array.reshape(n0, nelem)
    chunk = max(1, (64 << 20) // nelem)
    for i in range(0, n0, chunk):
        m = min(chunk, n0 - i)
        host[i : i + m] = stack[i : i + m, :nelem].cpu().numpy()
    return pinned, host, n0


def push_all(E: Env, host, n0, n_rank, nelem, per_call=125):
    for base in range(0, n_rank, n0):
        m = min(n0, n_rank - base)
        for i in range(0, m, per_call):
            E.ctx.median_push_raw(host[i].ctypes.data, min(per_call, m - i), nelem)


def median_single(E: Env, cfg, steps, warmup, sampler, e2e_steps, with_cpu, dump_name, row_band=None):
    """Median of a stack resident on ONE device (all frames; optionally a band of rows of every frame)."""
    torch, ctx = E.torch, E.ctx
    W, H, N = cfg["width"], cfg["height"], cfg["nframes"]
    row0, nrows = row_band if row_band else (0, H)
    nelem = nrows * W
    stride = (nelem + 127) // 128 * 128
    stack = torch.empty((N, stride), dtype=torch.uint8, device=E.dev)
    out = torch.empty(stride, dtype=torch.uint8, device=E.dev)
    ctx.synth_frames_device(stack.data_ptr(), stride, W, H, 0, N, cfg["seed"], cfg["ndisks"], row0=row0, nrows=nrows)
    ctx.synchronize()
    gathered = out_pad = None
    if row_band and E.world > 1:
        band_max = (H - (H // E.world) * (E.world - 1)) * W
        out_pad = torch.zeros(band_max, dtype=torch.uint8, device=E.dev)
        gathered = torch.empty(E.world * band_max, dtype=torch.uint8, device=E.dev)
    # an input that fits the L2 is flushed out of it between timed iterations (the flush is outside the kernel events)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=E.dev) if N * stride <= 4 * L2_BYTES else None
    with torch.cuda.stream(E.stream):
        for _ in range(warmup):
            ctx.median_device(stack.data_ptr(), N, nelem, stride, out.data_ptr())
        E.barrier()
        l0 = ctx.launch_count
        ev0, ev1 = E.event(), E.event()
        kern = []
        sampler.active = True
        ev0.record(E.stream)
        for _ in range(steps):
            if flush is not None:
                flush.zero_()
            a, b = E.event(), E.event()
            a.record(E.stream)
            ctx.median_device(stack.data_ptr(), N, nelem, stride, out.data_ptr())
            b.record(E.stream)
            kern.append((a, b))
            if gathered is not None:
                out_pad[:nelem].copy_(out[:nelem], non_blocking=True)
                E.dist.all_gather_into_tensor(gathered, out_pad)
        ev1.record(E.stream)
        E.barrier()
        sampler.active = False
        launches = ctx.launch_count - l0
    if gathered is None:
        E.dump.add(dump_name, out[:nelem].view(nrows, W))
    elif E.dump.dir is not None:  # the bands of all ranks, as the all-gather of the last step left them
        bands = gathered.view(E.world, band_max)
        E.dump.add(dump_name, torch.cat([bands[r, : shard_plan(H, r, E.world)[1] * W] for r in range(E.world)]).view(H, W))
    total_ms, kern_ms = E.max_over_ranks([ev0.elapsed_time(ev1), float(np.mean([a.elapsed_time(b) for a, b in kern]))])
    ms = kern_ms if flush is not None else total_ms / steps  # with a flush in the loop only the kernel events count
    job_mpxf = W * H * N / 1e6
    res = {"ms_per_step": ms, "value": job_mpxf / (ms * 1e-3), "gpu_launches": int(launches), "kernel_ms": kern_ms}
    res["roofline"] = roofline(float(N) * nelem + nelem, kern_ms,
                               "median_pipe_kernel<MODE 0> (on-chip bit-sliced select)" if N <= 1024 else
                               "median_pipe_kernel<MODE 3> x ceil(N/1024) launches + shard_window_final_kernel (one pass of window "
                               "counting; the gated two-pass fallback returns at once)",
                               "median_ncu_summary.json" if (N, W, H, E.world) == (1000, 1920, 1080, 1) else None)
    # ---- end to end through the host-buffer C ABI: pinned host frames -> result in host memory
    pinned, host, n0 = pinned_prefix(E, stack, N, nelem)
    host_out = np.empty(nelem, np.uint8)

    def e2e_step():
        ctx.median_begin(nelem, N)
        push_all(E, host, n0, N, nelem)
        ctx.median_finish(host_out)

    e2e_step()
    E.barrier()
    sampler.active = True
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    E.barrier()
    (e2e_s,) = E.max_over_ranks([(time.perf_counter() - t0) / e2e_steps])
    sampler.active = False
    res["e2e"] = {"value": job_mpxf / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(N * nelem) * (E.world if row_band else 1),
                  "d2h_bytes_per_step": int(nelem) * (E.world if row_band else 1), "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                  "api": "cvvp_median_begin / cvvp_median_push (pinned host frames) / cvvp_median_finish"}
    if n0 < N:
        res["e2e"]["host_buffer"] = f"frames [0,{n0}) of the stack, pushed {-(-N // n0)} times ({PINNED_CAP_BYTES / 1e9:.1f} GB of pinned memory)"
    same = n0 < N or bool(np.array_equal(host_out, out[:nelem].cpu().numpy()))
    # ---- CPU baseline: the reference class on the WHOLE workload (bounded: a prefix of the frames when it is huge)
    res["cpu_baseline"] = None
    if with_cpu:
        try:
            run, kind = cpu_median_fn()
            cores = os.cpu_count() or 1
            if n0 == N:
                sample_frames = host.reshape(N, nrows, W)
                want = run(sample_frames, cores)  # warm-up + parity of EVERY pixel against the device result
                same = same and bool(np.array_equal(want, host_out))
                reps = 3
                t0 = time.perf_counter()
                for _ in range(reps):
                    run(sample_frames, cores)
                dt = (time.perf_counter() - t0) / reps
                res["cpu_baseline"] = {"value": nrows * W * N / 1e6 / dt, "unit": UNIT, "cores": cores, "kind": kind,
                                       "sample": f"the whole frame of all {N} frames, {reps} repetitions, frames resident in host "
                                                 f"memory, {cores} worker threads each owning a strip"}
            else:
                rows = max(8, int(nrows * n0 / N) // 8 * 8)
                band = torch.empty((N, rows * W), dtype=torch.uint8, device=E.dev)
                ctx.synth_frames_device(band.data_ptr(), rows * W, W, H, 0, N, cfg["seed"], cfg["ndisks"], row0=row0, nrows=rows)
                ctx.synchronize()
                sample_frames = band.cpu().numpy().reshape(N, rows, W)
                del band
                want = run(sample_frames, cores)
                same = same and bool(np.array_equal(want, out[: rows * W].cpu().numpy()))
                t0 = time.perf_counter()
                run(sample_frames, cores)
                dt = time.perf_counter() - t0
                res["cpu_baseline"] = {"value": rows * W * N / 1e6 / dt, "unit": UNIT, "cores": cores, "kind": kind,
                                       "sample": f"rows [0,{rows}) of all {N} frames (every pixel of the band checked against the "
                                                 f"device result), {cores} worker threads"}
        except Exception as exc:  # the baseline must never take the GPU number down with it
            res["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "unavailable",
                                   "sample": f"failed: {exc}"}
    res["parity_spot_check"] = same
    pinned.close()
    del stack
    return res


def median_sharded(E: Env, cfg, n_rank, first_frame, total_frames, steps, warmup, sampler, e2e_steps, dump_name):
    """Frame-sharded median: this rank holds frames [first_frame, first_frame + n_rank) of the stream; the job is the
    median of all `total_frames`.  One step = ShardedMedian.run: window counting (phase 4), barrier, owner kernel
    (phase 5), barrier, the undecided-element count fetched from the device, and the two-round exchange only if it is not
    zero.  The barrier is a one-element NCCL all-reduce on the context's stream."""
    from cvvidproc_b200 import sharded

    torch, ctx, dist = E.torch, E.ctx, E.dist
    W, H = cfg["width"], cfg["height"]
    nelem = W * H
    stack = torch.empty((max(n_rank, 1), nelem), dtype=torch.uint8, device=E.dev)
    if n_rank:
        ctx.synth_frames_device(stack.data_ptr(), nelem, W, H, first_frame, n_rank, cfg["seed"], cfg["ndisks"])
    ctx.synchronize()
    most = int(E.max_over_ranks([n_rank])[0])
    job = sharded.ShardedMedian(ctx, nelem, E.rank, E.world, max_rank_frames=most)
    job.connect_processes()
    for _ in range(warmup):
        job.run(stack.data_ptr(), n_rank, nelem)
    E.barrier()
    l0 = ctx.launch_count
    ev0, ev1 = E.event(), E.event()
    phase_evs, undecided = [], 0
    sampler.active = True
    ev0.record(E.stream)
    for _ in range(steps):
        evs = []
        for p in (4, 5):
            a, b = E.event(), E.event()
            a.record(E.stream)
            job.phase(p, stack.data_ptr(), n_rank, nelem)
            b.record(E.stream)
            job.barrier()
            evs.append((a, b))
        left = ctx.median_shard_unresolved()
        undecided = max(undecided, left)
        if left:
            job.run_two_round(stack.data_ptr(), n_rank, nelem)
        phase_evs.append(evs)
    ev1.record(E.stream)
    E.barrier()
    sampler.active = False
    launches = ctx.launch_count - l0
    pm = [float(np.mean([evs[i][0].elapsed_time(evs[i][1]) for evs in phase_evs])) for i in range(2)]
    total_ms, p4, p5 = E.max_over_ranks([ev0.elapsed_time(ev1)] + pm)
    ms = total_ms / steps
    job_mpxf = W * H * total_frames / 1e6
    res = {"ms_per_step": ms, "value": job_mpxf / (ms * 1e-3), "gpu_launches": int(launches), "kernel_ms": p4,
           "undecided_elements": int(undecided)}
    res["roofline"] = roofline(float(most) * nelem + 20.0 * nelem * -(-most // 1024), p4,
                               "median_pipe_kernel<MODE 3> (window counting, one pass over the rank's frames)",
                               note="algorithmic bytes = every input byte once + one 20-byte record per element and launch")
    res["roofline"]["phase_ms"] = {"window_count": p4, "window_final": p5,
                                   "barriers_and_host_check": max(0.0, ms - p4 - p5)}
    res["barrier"] = job.barrier_kind
    result_dev = ctx.copy_to_host(job.result_ptr(), nelem)
    E.dump.add(dump_name, result_dev.reshape(H, W))
    # ---- end to end through the host-buffer C ABI: cvvp_median_push of this rank's pinned frames, the exchange on the
    # pushed stack (cvvp_median_stack_device), the full result image back in host memory
    pinned, host, n0 = pinned_prefix(E, stack, max(n_rank, 1), nelem)
    host_out = None

    def e2e_step():
        nonlocal host_out
        ctx.median_begin(nelem, max(n_rank, 1))
        if n_rank:
            push_all(E, host, n0, n_rank, nelem)
        d_ptr, d_stride, d_n = ctx.median_stack_device()
        job.run(d_ptr, d_n, d_stride)
        host_out = ctx.copy_to_host(job.result_ptr(), nelem)
        ctx.median_abort()

    e2e_step()
    E.barrier()
    sampler.active = True
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    E.barrier()
    (e2e_s,) = E.max_over_ranks([(time.perf_counter() - t0) / e2e_steps])
    sampler.active = False
    res["e2e"] = {"value": job_mpxf / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(total_frames) * nelem,
                  "d2h_bytes_per_step": int(nelem) * E.world, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                  "api": "cvvp_median_begin / cvvp_median_push (pinned host frames) / cvvp_median_stack_device / "
                         "cvvp_median_shard_phase / cvvp_ctx_copy_to_host"}
    if n0 < n_rank:
        res["e2e"]["host_buffer"] = f"frames [0,{n0}) of the rank's chunk, pushed {-(-n_rank // n0)} times"
    # ---- parity spot check (outside the timed regions): every rank holds the same image, and on sampled elements it
    # is the order statistic of ALL ranks' frames (gathered through NCCL for the sample only)
    same = n0 < n_rank or bool(np.array_equal(host_out, result_dev))
    cols = torch.arange(0, nelem, max(1, nelem // 4096), device=E.dev)
    mine = stack[:n_rank][:, cols].contiguous()
    if dist is not None:
        cnt = torch.tensor([n_rank], dtype=torch.int64, device=E.dev)
        cnts = [torch.zeros_like(cnt) for _ in range(E.world)]
        dist.all_gather(cnts, cnt)
        sizes = [int(c[0]) for c in cnts]
        allc = [torch.empty((sz, cols.numel()), dtype=torch.uint8, device=E.dev) for sz in sizes]
        if len(set(sizes)) == 1:
            dist.all_gather(allc, mine)
        else:
            _gather_ragged(dist, allc, mine, E)
        allv = torch.cat(allc, 0)
    else:
        allv = mine
    want = torch.sort(allv, dim=0).values[total_frames // 2].cpu().numpy()
    same = same and bool(np.array_equal(want, result_dev[cols.cpu().numpy()]))
    res["parity_spot_check"] = E.all_true(same)
    res["cpu_baseline"] = None
    pinned.close()
    job.close()
    del stack
    return res


def _gather_ragged(dist, outs, mine, E):
    """all_gather of per-rank samples with different frame counts (broadcast one rank at a time)"""
    for r in range(E.world):
        if r == E.rank:
            outs[r].copy_(mine)
        dist.broadcast(outs[r], src=r)


def highlight_bench(E: Env, cfg, frames_rank, first_frame, total_frames, steps, sampler, with_cpu, dump_name, traffic_file=None,
                    frames_per_launch=None):
    """Highlight of this rank's frames [first_frame, first_frame + frames_rank) of the config's stream, resident in HBM
    (`value`, CUDA events, max over ranks) and from pinned host memory through cvvp_highlight_frames (`e2e`).  Frames
    are independent (highlight_objects_algo.h:82-85): sharded by frame, no collective."""
    torch, ctx = E.torch, E.ctx
    W, H = cfg["width"], cfg["height"]
    npix = W * H
    bgstack = torch.empty((255, npix), dtype=torch.uint8, device=E.dev)
    bg = torch.empty(npix, dtype=torch.uint8, device=E.dev)
    ctx.synth_frames_device(bgstack.data_ptr(), npix, W, H, 0, 255, cfg["seed"], cfg["ndisks"])
    ctx.median_device(bgstack.data_ptr(), 255, npix, npix, bg.data_ptr())
    ctx.synchronize()
    del bgstack
    bg_h = bg.cpu().numpy().reshape(H, W)
    cp = CANONICAL_HIGHLIGHT
    nfr = frames_rank
    frames = torch.empty((nfr, npix), dtype=torch.uint8, device=E.dev)
    masks = torch.empty((nfr, npix), dtype=torch.uint8, device=E.dev)
    ctx.synth_frames_device(frames.data_ptr(), npix, W, H, first_frame, nfr, cfg["seed"], cfg["ndisks"])
    ctx.highlight_begin(bg_h, np.array(cp["struct_element"], np.uint8), cp["threshold"], cp["threshold_lo"], cp["threshold_hi"],
                        cp["min_size_hyst"], cp["min_size_threshold"], cp["width_border"])
    per = frames_per_launch or nfr

    def step():
        for i in range(0, nfr, per):
            m = min(per, nfr - i)
            ctx.highlight_device(frames[i:].data_ptr(), m, npix, masks[i:].data_ptr(), npix)

    with torch.cuda.stream(E.stream):
        for _ in range(3):
            step()
        E.barrier()
        l0 = ctx.launch_count
        e0, e1 = E.event(), E.event()
        sampler.active = True
        e0.record(E.stream)
        for _ in range(steps):
            step()
        e1.record(E.stream)
        E.barrier()
        sampler.active = False
        launches = ctx.launch_count - l0
    E.dump.add(dump_name, masks.view(nfr, H, W))
    (ms,) = E.max_over_ranks([e0.elapsed_time(e1) / steps])
    # end to end from pinned host memory through cvvp_highlight_frames (bounded pinned buffers: a prefix of the frames,
    # processed ceil(n / n0) times per step when the rank's share is larger)
    n0 = int(max(1, min(nfr, PINNED_CAP_BYTES // npix)))  # one pinned buffer in, one out
    pin_in = E.cabi.PinnedBuffer(n0 * npix)
    pin_out = E.cabi.PinnedBuffer(n0 * npix)
    pin_in.array[:] = frames[:n0].cpu().numpy().reshape(-1)

    def e2e_step():
        for base in range(0, nfr, n0):
            m = min(n0, nfr - base)
            rc = E.lib.cvvp_highlight_frames(ctx.handle, pin_in.array.ctypes.data, m, npix, pin_out.array.ctypes.data, npix)
            if rc != 0:
                raise RuntimeError(E.lib.cvvp_last_error(ctx.handle).decode())

    e2e_steps = max(1, min(steps, 3 if nfr * npix > 4_000_000_000 else steps))
    e2e_step()
    E.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    E.barrier()
    (e2e_s,) = E.max_over_ranks([(time.perf_counter() - t0) / e2e_steps])
    total_mpx = total_frames * npix / 1e6
    last = min(n0, nfr - (nfr - 1) // n0 * n0)
    same = bool(np.array_equal(pin_out.array.reshape(n0, npix)[:last], masks[:last].cpu().numpy()))
    out = {
        "metric": f"megapixel-frames/sec (per-frame highlight, {W}x{H})", "unit": UNIT,
        "value": total_mpx / (ms * 1e-3), "ms_per_step": ms, "frames_per_step": int(total_frames), "steps": steps,
        "gpu_launches": int(launches), "sharding": "single GPU" if E.world == 1 else f"by frame x{E.world}, no collective",
        "e2e": {"value": total_mpx / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(total_frames) * npix,
                "d2h_bytes_per_step": int(total_frames) * npix, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                "api": "cvvp_highlight_frames (pinned host frames in, pinned host masks out)"},
        "roofline": roofline(2.0 * nfr * npix, ms, "highlight_fused_kernel", traffic_file,
                             "algorithmic bytes = frame in + mask out (2 B/px); one fused kernel launch per "
                             f"{per} frames"),
        "config": {"workload": cfg["name"], "frames_per_gpu": int(nfr)},
    }
    if n0 < nfr:
        out["e2e"]["host_buffer"] = f"frames [0,{n0}) of the rank's share, processed {-(-nfr // n0)} times per step"
    if with_cpu:
        try:
            k = min(16, nfr)
            host_frames = frames[:k].cpu().numpy().reshape(k, H, W)
            cores = os.cpu_count() or 1
            rate, done, lastm = cpu_highlight_rate(host_frames, bg_h, cores, seconds=10.0)
            same = same and bool(np.array_equal(lastm.reshape(-1), masks[(done - 1) % k].cpu().numpy()))
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": f"{done} frames in ~10 s, cv2 restatement of highlight_objects_algo.cpp, "
                                             f"{cores} threads x cv2.setNumThreads(1)"}
        except Exception as exc:
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "unavailable",
                                   "sample": f"failed: {exc}"}
    out["parity_spot_check"] = E.all_true(same)
    ctx.highlight_end()
    pin_in.close()
    pin_out.close()
    del frames, masks
    return out


def frame_source_bench(E: Env, steps):
    """The stage in front of both operators (SURVEY 8f rank 1): decoded 1080p 3-channel frames resident in HBM ->
    grey frames (crop = whole frame, COLOR_RGB2GRAY; cv_vid_frames_generator_algo.h:141-156) by csrc/frames.cu."""
    torch, ctx = E.torch, E.ctx
    W, H, n = 1920, 1080, 96  # 597 MB of decoded frames: larger than the 126 MB L2
    gen = torch.Generator(device=E.dev)
    gen.manual_seed(11)
    src = torch.randint(0, 256, (n, H * W * 3), dtype=torch.uint8, device=E.dev, generator=gen)
    dst = torch.empty((n, H * W), dtype=torch.uint8, device=E.dev)
    fmt = E.cabi.FrameFormat.of((H, W, 3), E.cabi.FRAMES_RGB2GRAY)
    with torch.cuda.stream(E.stream):
        for _ in range(3):
            ctx.frames_prepare_device(src.data_ptr(), n, H * W * 3, fmt, dst.data_ptr(), H * W)
        torch.cuda.synchronize()
        l0 = ctx.launch_count
        e0, e1 = E.event(), E.event()
        e0.record(E.stream)
        for _ in range(steps):
            ctx.frames_prepare_device(src.data_ptr(), n, H * W * 3, fmt, dst.data_ptr(), H * W)
        e1.record(E.stream)
        torch.cuda.synchronize()
        launches = ctx.launch_count - l0
    E.dump.add("frame_source_gray", dst.view(n, H, W))
    ms = e0.elapsed_time(e1) / steps
    out = {
        "metric": "megapixel-frames/sec (frame source: 1080p decoded 3-channel -> grey)", "unit": UNIT,
        "value": n * W * H / 1e6 / (ms * 1e-3), "ms_per_step": ms, "frames_per_step": n, "steps": steps, "gpu_launches": int(launches),
        "roofline": roofline(4.0 * n * W * H, ms, "frames_prepare_kernel", "frames_ncu_summary.json",
                             "algorithmic bytes = 3 B/px decoded frame in + 1 B/px prepared frame out"),
    }
    if not E.args.no_cpu_baseline:
        import concurrent.futures as cf

        import cv2

        cv2.setNumThreads(1)
        host = src[:16].cpu().numpy().reshape(16, H, W, 3)
        cores = os.cpu_count() or 1
        done, last = 0, None
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(max_workers=cores) as ex:
            while time.perf_counter() - t0 < 3.0:
                res = list(ex.map(lambda i: cv2.cvtColor(host[i % 16], cv2.COLOR_RGB2GRAY), range(done, done + 4 * cores)))
                done += len(res)
                last = res[-1]
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": done * W * H / 1e6 / dt, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": f"{done} frames in ~3 s, cv2.cvtColor(COLOR_RGB2GRAY), {cores} threads x cv2.setNumThreads(1)"}
        out["parity_spot_check"] = bool(np.array_equal(last.reshape(-1), dst[(done - 1) % 16].cpu().numpy()))
    return out


def cpu_track_pipeline(path, bg, tracker, nframes, cores):
    """The reference-shaped CPU pipeline on a video file (cv_vid_objecttrack_helpers.cpp:71-133): one decode thread, the cv2
    restatement of HighlightObjects on the reference's own worker count, the tracker in frame order on the calling
    thread.  Timed with cv2's internal threading off and on; the faster one is reported."""
    import concurrent.futures as cf
    import queue as queue_mod

    import cv2

    from oracle import highlight_oracle as ho

    p = ho.canonical_params(bg)
    workers = max(1, cores - 2)  # the reference's own batch_size (cv_vid_objecttrack_helpers.cpp:182)

    def run(cv_threads):
        cv2.setNumThreads(cv_threads)
        arch = {}
        q = queue_mod.Queue(maxsize=2 * workers)
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(max_workers=workers) as ex:
            def produce():
                cap = cv2.VideoCapture(path)
                while True:
                    ok, fr = cap.read()
                    if not ok:
                        break
                    q.put(ex.submit(ho.highlight_objects, cv2.extractChannel(fr, 0), p))
                q.put(None)

            th = threading.Thread(target=produce)
            th.start()
            k, nid = 0, 0
            while True:
                fut = q.get()
                if fut is None:
                    break
                nid = tracker(fut.result(), k, {}, arch, nid, {})
                k += 1
            th.join()
        return time.perf_counter() - t0, arch

    runs = {t: run(t) for t in (1, cores)}
    best = min(runs, key=lambda t: runs[t][0])
    cv2.setNumThreads(cores)
    t_cpu, arch = runs[best]
    return {"value": None, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_frame": t_cpu / nframes * 1e3,
            "sample": f"all {nframes} frames: one decode thread, cv2 restatement of HighlightObjects on {workers} worker threads, "
                      f"stand-in tracker in frame order on the calling thread; the faster of cv2.setNumThreads(1) / ({cores}): "
                      f"{best} ({runs[1][0] / nframes * 1e3:.2f} / {runs[cores][0] / nframes * 1e3:.2f} ms per frame)"}, arch


class StdoutToStderr:
    """The drop-in entry points print the reference's video-info line to stdout (cv_vid_bg_helpers.cpp:212-223); the
    bench's stdout carries exactly one JSON line, so fd 1 points at stderr while they run."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)


def track_e2e_bench(E: Env, nframes):
    """BASELINE configs[2] as the USER sees it: the drop-in TrackObjects on a lossless 1080p video (cv2 FFV1, decode
    INSIDE the timed region), with a no-op tracker callback and with the stand-in tracker of SURVEY 8c
    (cv2.connectedComponentsWithStats on every mask), the reference-shaped cv2 pipeline timed beside it: one decode
    thread, highlight on all other host threads (cv_vid_objecttrack_helpers.cpp:71-133), the callback in order."""
    import concurrent.futures as cf
    import tempfile

    import cv2

    import cvvidproc_b200 as cvp

    cfg = CONFIGS["C3"]
    W, H = cfg["width"], cfg["height"]
    torch, ctx = E.torch, E.ctx
    cores = os.cpu_count() or 1
    out = {"metric": "megapixel-frames/sec (TrackObjects on a lossless 1080p video, decode and tracker included)", "unit": UNIT,
           "frames": int(nframes), "config": {"workload": f"{W}x{H} x {nframes} frames of the C3 stream written as FFV1/AVI"}}
    with tempfile.TemporaryDirectory() as d:
        path = str(Path(d) / "c3.avi")
        vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (W, H), isColor=True)
        if not vw.isOpened():
            return {"value": None, "error": "no FFV1 writer in this cv2 build"}
        chunk = 50
        for f0 in range(0, nframes, chunk):
            m = min(chunk, nframes - f0)
            t = torch.empty((m, W * H), dtype=torch.uint8, device=E.dev)
            ctx.synth_frames_device(t.data_ptr(), W * H, W, H, f0, m, cfg["seed"], cfg["ndisks"])
            ctx.synchronize()
            for fr in t.cpu().numpy().reshape(m, H, W):
                vw.write(cv2.cvtColor(fr, cv2.COLOR_GRAY2BGR))
        vw.release()
        # decode alone, into rotating buffers (a pipeline cannot decode every frame into one cache-resident array)
        cv2.setNumThreads(cores)  # the CPU legs of earlier sections switch cv2's own threading off; a user's tracker has it on
        t0 = time.perf_counter()
        cap = cv2.VideoCapture(path)
        k = 0
        bufs = np.empty((32, H, W, 3), np.uint8)
        while cap.read(bufs[k % 32])[0]:
            k += 1
        t_dec = time.perf_counter() - t0
        del bufs
        out["decode_alone_ms_per_frame"] = t_dec / max(k, 1) * 1e3
        bg = cvp.GetVideoBackground(cvp.VidBgPack(path, vid_is_grayscale=True, frame_limit=255))
        cp = CANONICAL_HIGHLIGHT
        hp = cvp.HighlightObjectsPack(bg, np.array(cp["struct_element"], np.uint8), cp["threshold"], cp["threshold_lo"],
                                      cp["threshold_hi"], cp["min_size_hyst"], cp["min_size_threshold"], cp["width_border"])

        def noop(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs):
            return next_ID

        def ccl(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs):
            n, _, stats, cent = cv2.connectedComponentsWithStats(bw_frame, connectivity=8)
            objects_archive[frames_processed] = [(int(stats[i, cv2.CC_STAT_AREA]), round(float(cent[i][0]), 2),
                                                  round(float(cent[i][1]), 2)) for i in range(1, n)]
            return next_ID + n - 1

        def run(fn):
            t0 = time.perf_counter()
            arch = cvp.TrackObjects(cvp.VidObjectTrackPack(path, hp, cvp.AssignObjectsPack(fn, {}), vid_is_grayscale=True))
            return time.perf_counter() - t0, arch

        run(noop)  # warm-up: scratch allocation, module load
        t_noop, _ = run(noop)
        t_ccl, arch_gpu = run(ccl)
        E.dump.add("track_e2e_objects", np.array([(f, *obj) for f in sorted(arch_gpu) for obj in arch_gpu[f]], np.float64).reshape(-1, 4))
        mpx = nframes * W * H / 1e6
        out["value"] = mpx / t_ccl
        out["ms_per_frame"] = {"noop_callback": t_noop / nframes * 1e3, "ccl_tracker": t_ccl / nframes * 1e3}
        out["no_op_callback"] = {"value": mpx / t_noop, "unit": UNIT}
        out["vs_decode_alone"] = (t_ccl / nframes * 1e3) / out["decode_alone_ms_per_frame"]
        # the reference-shaped CPU pipeline: decode thread -> highlight workers -> ordered callback
        if not E.args.no_cpu_baseline:
            cpu, arch_cpu = cpu_track_pipeline(path, bg, ccl, nframes, cores)
            cpu["value"] = mpx / (cpu["ms_per_frame"] * 1e-3 * nframes)
            out["cpu_baseline"] = cpu
            out["parity_spot_check"] = arch_cpu == arch_gpu
    return out


# ------------------------------------------------------------------------------------------------
# the GPU arm
# ------------------------------------------------------------------------------------------------
def dump_names(args, world):
    """The arrays run_gpu_arm hands to OutputDump, in its order and under its conditions."""
    names = ["background" if CONFIGS[args.config]["kind"] == "median" else "masks"]
    if args.config == "C2" and not args.no_highlight:
        names += ["highlight_masks"] + (["frame_source_gray"] if world == 1 else [])
        if not args.no_extra_configs:
            names += ["c5_median_background", "c4_highlight_masks"]
            names += ["track_e2e_objects"] if world == 1 and not args.no_track else []
    return names


def run_gpu_arm(args, rank, local_rank, world):
    E = Env(args, rank, local_rank, world)
    cfg = CONFIGS[args.config]
    conf = job_config(cfg, world, args)
    sampler = ClockSampler(local_rank)
    sampler.start()
    steps, warmup = args.steps, args.warmup
    with_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    extras = {}

    def median_of(c, st, wu, e2e_steps, cpu, dump_name):
        if world == 1:
            return median_single(E, c, st, wu, sampler, e2e_steps, cpu, dump_name)
        if c["scaling"] == "weak" and args.median_sharding == "rows":
            return median_single(E, c, st, wu, sampler, e2e_steps, False, dump_name, row_band=shard_plan(c["height"], rank, world))
        if c["scaling"] == "weak":
            return median_sharded(E, c, c["nframes"], c["nframes"] * rank, c["nframes"] * world, st, wu, sampler, e2e_steps,
                                  dump_name)
        first, cnt = frame_chunk(c["nframes"], rank, world)
        return median_sharded(E, c, cnt, first, c["nframes"], st, wu, sampler, e2e_steps, dump_name)

    def highlight_of(c, st, cpu, dump_name, traffic=None):
        first, cnt = frame_chunk(c["nframes"], rank, world)
        per = 1024 if c["width"] * c["height"] > 500_000 else 16384
        return highlight_bench(E, c, cnt, 1000 + first, c["nframes"], st, sampler, cpu, dump_name, traffic, frames_per_launch=per)

    if cfg["kind"] == "median":
        main = median_of(cfg, steps, warmup, steps, with_cpu, "background")
    else:
        main = highlight_of(cfg, steps, with_cpu, "masks")
        main["steps_timed"] = main.pop("steps")
    clocks = sampler.summary()
    sampler.stop()

    if args.config == "C2" and not args.no_highlight:
        s2 = ClockSampler(local_rank)
        s2.start()
        sampler = s2
        try:
            hl_cfg = dict(HL_STEP, nframes=HL_STEP["frames_per_gpu"] * world)
            h = highlight_bench(E, hl_cfg, HL_STEP["frames_per_gpu"], 1000 + rank * HL_STEP["frames_per_gpu"], hl_cfg["nframes"],
                                max(3, min(steps, 10)), sampler, with_cpu, "highlight_masks",
                                "highlight_ncu_summary.json" if world == 1 else None)
            h["scaling"] = "weak"
            h["clocks"] = s2.summary()
            extras["highlight"] = h
            if world == 1:
                extras["frame_source"] = frame_source_bench(E, max(3, min(steps, 10)))
            if not args.no_extra_configs:
                c5 = median_of(CONFIGS["C5"], 3, 3, 2, with_cpu, "c5_median_background")
                c5["metric"], c5["unit"], c5["scaling"] = metric_name(CONFIGS["C5"]), UNIT, "strong"
                c5["config"] = job_config(CONFIGS["C5"], world, args)
                extras["c5_median"] = c5
                c4 = highlight_of(CONFIGS["C4"], 3, False, "c4_highlight_masks")
                c4["scaling"] = "strong"
                extras["c4_highlight"] = c4
                if world == 1 and not args.no_track:
                    try:
                        with StdoutToStderr():
                            extras["track_e2e"] = track_e2e_bench(E, args.track_frames)
                    except Exception as exc:
                        extras["track_e2e"] = {"value": None, "error": f"{type(exc).__name__}: {exc}"}
        finally:
            s2.stop()

    if rank == 0:
        scaling = "weak" if world == 1 or (cfg["scaling"] == "weak" and args.median_sharding == "frames") else "strong"
        line = {
            "metric": metric_name(cfg), "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": conf, "clocks": clocks, "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
            "roofline": main["roofline"], "cpu_baseline": main.get("cpu_baseline"), "parity_spot_check": main["parity_spot_check"],
        }
        for k in ("undecided_elements", "barrier", "steps_timed", "frames_per_step"):
            if k in main:
                line[k] = main[k]
        line.update(extras)
        print(json.dumps(line), flush=True)
    E.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline workload; the extra objects of the C2 line time their own fixed "
                         "counts (3 to 10 steps)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["cuda", "reference"], default="cuda")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="C2", help="the workload of the line's headline (default: C2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-highlight", action="store_true", help="C2 only: skip every extra object of the line")
    ap.add_argument("--no-extra-configs", action="store_true", help="C2 only: skip the c5_median / c4_highlight / track_e2e objects")
    ap.add_argument("--no-track", action="store_true", help="skip the track_e2e object")
    ap.add_argument("--track-frames", type=int, default=1000, help="frames of the lossless video of the track_e2e object")
    ap.add_argument("--median-sharding", choices=["frames", "rows"], default="frames",
                    help="N > 1, C2: frame chunks with the NVLink count exchange (default, weak scaling) or row bands of "
                         "the single stack with no data-path collective (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32, at most 64 MB in "
                         "all, shared among the arrays the run writes; larger results as a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path")
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun (one process per GPU); running the single-GPU job", file=sys.stderr)
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    else:
        run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
