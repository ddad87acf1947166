"""bench.py --dump-outputs and --steps: what the timed path computed is written for comparison between builds, and the
number of timed steps is the one asked for."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parent.parent
_spec = importlib.util.spec_from_file_location("bench_mod", REPO / "bench.py")
bench = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(bench)


def test_dump_writes_float32_and_samples_what_exceeds_its_share(tmp_path, monkeypatch):
    monkeypatch.setattr(bench.OutputDump, "TOTAL_BYTES", 8000)
    d = bench.OutputDump(tmp_path / "out", ["small", "stack"])
    img = np.arange(20 * 30, dtype=np.uint8).reshape(20, 30) % 251
    d.add("small", img)  # 2400 bytes: within its share of 4000
    stack = np.random.default_rng(1).integers(0, 256, (50, 10, 40), dtype=np.uint8)
    d.add("stack", stack)  # the 5600 bytes left hold 3 frames of 1600 bytes and their positions
    small = np.load(tmp_path / "out" / "small.npy")
    assert small.dtype == np.float32 and np.array_equal(small, img)
    assert not (tmp_path / "out" / "small_index.npy").exists()
    got = np.load(tmp_path / "out" / "stack.npy")
    idx = np.load(tmp_path / "out" / "stack_index.npy")
    assert got.shape == (3, 10, 40) and idx.dtype == np.float64
    assert np.array_equal(got, stack[idx.astype(int)])
    assert d.written <= bench.OutputDump.TOTAL_BYTES
    # the sample is fixed: a second dump picks the same entries
    bench.OutputDump(tmp_path / "again", ["stack"]).add("stack", stack)
    assert len(np.load(tmp_path / "again" / "stack_index.npy")) == 4  # alone, the stack has all 8000 bytes
    d3 = bench.OutputDump(tmp_path / "third", ["small", "stack"])
    d3.add("small", img)
    d3.add("stack", stack)
    assert np.array_equal(np.load(tmp_path / "third" / "stack_index.npy"), idx)


def test_dump_refuses_undeclared_arrays_and_entries_larger_than_a_share(tmp_path, monkeypatch):
    monkeypatch.setattr(bench.OutputDump, "TOTAL_BYTES", 1000)
    d = bench.OutputDump(tmp_path, ["a", "b"])
    with pytest.raises(ValueError):
        d.add("c", np.zeros(4, np.uint8))
    with pytest.raises(RuntimeError):
        d.add("a", np.zeros((2, 200), np.uint8))


@pytest.mark.parametrize("config", ["C2", "C3", "C4"])
def test_declared_arrays_fit_the_limit(config):
    """every array the run declares gets a share that holds at least one frame or row of it"""
    args = bench.argparse.Namespace(config=config, no_highlight=False, no_extra_configs=False, no_track=False)
    names = bench.dump_names(args, 1)
    assert bench.OutputDump.TOTAL_BYTES // len(names) > 1920 * 1080 * 4 + 8


def _run_bench(*args):
    out = subprocess.run([sys.executable, str(REPO / "bench.py"), "--no-cpu-baseline", *args],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dumps_the_median_of_its_last_step_and_times_the_steps_asked_for(tmp_path, oracle_median):
    from cvvidproc_b200 import synth

    p = synth.CONFIG_PARAMS["C1"]
    lines = {k: _run_bench("--config", "C1", "--steps", str(k), "--warmup", "3", "--dump-outputs", str(tmp_path / str(k)))
             for k in (2, 5)}
    assert [lines[k]["steps"] for k in (2, 5)] == [2, 5]
    # C1 is one launch per median: the launches counted over the timed steps are the steps
    assert lines[5]["gpu_launches"] * 2 == lines[2]["gpu_launches"] * 5
    frames = synth.synth_frames(0, p["nframes"], p["width"], p["height"], p["seed"], p["ndisks"])
    want = oracle_median(frames)
    for k in (2, 5):
        got = np.load(tmp_path / str(k) / "background.npy")
        assert got.dtype == np.float32 and np.array_equal(got, want.astype(np.float32))


@pytest.mark.gpu
def test_bench_highlight_headline_times_the_steps_asked_for_and_dumps_its_masks(tmp_path, oracle_median):
    """C4 (a highlight headline) once capped --steps at 5; its dumped masks are the cv2 restatement's on those frames"""
    from cvvidproc_b200 import synth
    from oracle import highlight_oracle as ho

    lines = {k: _run_bench("--config", "C4", "--steps", str(k), "--warmup", "3", "--dump-outputs", str(tmp_path / str(k)))
             for k in (2, 7)}
    assert [lines[k]["steps_timed"] for k in (2, 7)] == [2, 7]
    assert lines[7]["gpu_launches"] * 2 == lines[2]["gpu_launches"] * 7
    p = synth.CONFIG_PARAMS["C4"]
    w, h = p["width"], p["height"]
    masks = np.load(tmp_path / "7" / "masks.npy")
    idx = np.load(tmp_path / "7" / "masks_index.npy").astype(int)
    assert masks.dtype == np.float32 and masks.shape == (len(idx), h, w) and len(idx) > 100
    assert np.array_equal(np.load(tmp_path / "2" / "masks.npy"), masks)
    # the background is the device median of the stream's first 255 frames; the masks cover frames 1000 onwards
    hp = ho.canonical_params(oracle_median(synth.synth_frames(0, 255, w, h, p["seed"], p["ndisks"])))
    for i in idx[:: max(1, len(idx) // 8)]:
        frame = synth.synth_frame(1000 + int(i), w, h, p["seed"], p["ndisks"])
        assert np.array_equal(masks[list(idx).index(i)], ho.highlight_objects(frame, hp).astype(np.float32)), int(i)
