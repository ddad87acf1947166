"""CPU tests of the highlight oracles: the cv2 restatement of highlight_objects_algo.cpp (oracle/highlight_oracle.py)
against the reference's own source compiled unmodified (oracle/_ref/cvvp_highlight_ref, see oracle/highlight_ref.py),
function by function; against the independent label-based model (oracle/highlight_model.py), stage by stage, on random
and adversarial images (SURVEY.md 9.7); and against the committed golden hashes, which are the reference's outputs."""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

import hl_cases
from oracle import highlight_model as hm
from oracle import highlight_oracle as ho
from oracle import highlight_ref as href

needs_ref = pytest.mark.skipif(not href.available(), reason="oracle/_ref/cvvp_highlight_ref was not built (no /root/reference)")

STAGES = ["diff", "a_thresh", "a_open", "a_rso", "a_fill", "b_hyst", "b_open", "b_rso", "b_fill"]


def _run_both(frame, p):
    so, sm = {}, {}
    a = ho.highlight_objects(frame.copy(), p, so)
    b = hm.highlight_objects(frame, p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                             p.min_size_hyst, p.min_size_threshold, sm)
    return a, b, so, sm


@pytest.mark.parametrize("t", range(120))
def test_model_matches_cv2_random(t):
    frame, p = hl_cases.random_case(t)
    a, b, so, sm = _run_both(frame, p)
    for k in STAGES:
        assert np.array_equal(so[k], sm[k]), f"stage {k}"
    assert np.array_equal(a, b)


ADV = hl_cases.adversarial_cases()


@pytest.mark.parametrize("case", ADV, ids=[c[0] for c in ADV])
def test_model_matches_cv2_adversarial(case):
    _, frame, p = case
    a, b, so, sm = _run_both(frame, p)
    for k in STAGES:
        assert np.array_equal(so[k], sm[k]), f"stage {k}"
    assert np.array_equal(a, b)


def _against_reference(name, frame, p, out):
    """out == the reference's output: the compiled reference where it was built, else its stored hash"""
    if href.available():
        got = href.highlight_objects(frame, p)
        assert got.dtype == np.uint8 and got.shape == frame.shape
        assert np.array_equal(got, out)
        return
    sha = hl_cases.reference_sha256(name)
    if sha is None:
        pytest.skip(f"oracle/_ref/cvvp_highlight_ref was not built and no output of the reference is stored for {name}")
    assert hashlib.sha256(out.tobytes()).hexdigest() == sha


@pytest.mark.parametrize("t", range(120))
def test_restatement_matches_the_compiled_reference_random(t):
    """HighlightObjectsAlgo::Insert -> TryGetResult of the reference's own source == oracle.highlight_objects"""
    frame, p = hl_cases.random_case(t)
    _against_reference(f"random_{t}", frame, p, ho.highlight_objects(frame.copy(), p))


@pytest.mark.parametrize("case", ADV, ids=[c[0] for c in ADV])
def test_restatement_matches_the_compiled_reference_adversarial(case):
    name, frame, p = case
    _against_reference(name, frame, p, ho.highlight_objects(frame.copy(), p))


@needs_ref
@pytest.mark.parametrize("t", range(0, 120, 3))
def test_every_restated_function_matches_the_reference_function(t):
    """ThresholdImage (fixed and Otsu), ThresholdImageWithHysteresis, RemoveSmallObjects, FillHoles one by one, each fed
    with the intermediate image the pipeline would hand it (highlight_objects_algo.cpp:81-221)"""
    frame, p = hl_cases.random_case(t)
    op = href.operator(p)
    st = {}
    ho.highlight_objects(frame.copy(), p, st)
    diff = st["diff"]
    for th in (p.threshold, -1, 0, 255):
        assert np.array_equal(op.threshold_image(diff, th), ho.threshold_image(diff, th)), f"ThresholdImage({th})"
    for lo, hi in ((p.threshold_lo, p.threshold_hi), (p.threshold_hi, p.threshold_lo), (0, 0)):
        assert np.array_equal(op.threshold_image_with_hysteresis(diff, lo, hi),
                              ho.threshold_image_with_hysteresis(diff, lo, hi)), f"hysteresis({lo},{hi})"
    for name, ms in (("a_open", p.min_size_threshold), ("b_open", p.min_size_hyst), ("a_open", 0), ("b_open", 10 ** 6)):
        want = st[name].copy()
        ho.remove_small_objects(want, ms)
        assert np.array_equal(op.remove_small_objects(st[name], ms), want), f"RemoveSmallObjects({name},{ms})"
    for name in ("a_rso", "b_rso", "a_thresh"):
        want = st[name].copy()
        ho.fill_holes(want)
        assert np.array_equal(op.fill_holes(st[name]), want), f"FillHoles({name})"


@needs_ref
def test_reference_operator_interface():
    """the four-method shape (highlight_objects_algo.h:57-91): null and empty tokens leave no result, one operator
    serves many tokens, the caller's frame is not written"""
    frame, p = hl_cases.random_case(5)
    op = href.operator(p)
    assert op.insert(None) is None and not op.has_results()
    assert op.insert(np.zeros((0, frame.shape[1]), np.uint8)) is None
    keep = frame.copy()
    a = op.insert(frame)
    assert not op.has_results()  # TryGetResult moved it out
    b = op.insert(frame)
    op.notify_no_more_tokens()
    assert np.array_equal(a, b) and np.array_equal(frame, keep)
    assert set(np.unique(a)) <= {0, 255}


@needs_ref
def test_reference_at_full_hd_and_on_the_small_geometry():
    """frames of the C3 (1080p) and C4 (512x256) streams, canonical parameters: restatement == compiled reference"""
    from cvvidproc_b200 import synth

    for cfg, idx in (("C3", (1000, 1097, 4321)), ("C4", (3, 97, 194, 5000, 150000))):
        p_ = synth.CONFIG_PARAMS[cfg]
        w, h = p_["width"], p_["height"]
        stack = synth.synth_frames(0, 15, w, h, p_["seed"], p_["ndisks"])
        p = ho.canonical_params(np.sort(stack, axis=0)[7])
        op = href.operator(p)
        for f in idx:
            fr = synth.synth_frame(f, w, h, p_["seed"], p_["ndisks"])
            want = ho.highlight_objects(fr.copy(), p)
            assert want.any()
            assert np.array_equal(op.insert(fr), want), f"{cfg} frame {f}"


def test_quirks_are_reproduced():
    """the three places where the code differs from the prose (SURVEY.md section 10, Q1 Q2 Q4)"""
    by = {c[0]: c for c in ADV}
    # Q1: saturating bg - frame: a frame brighter than the background highlights nothing
    _, f, p = by["brighter_everywhere"]
    assert not ho.highlight_objects(f.copy(), p).any()
    # Q4: an object covering pixel (0,0) turns the whole frame white
    _, f, p = by["covers_origin"]
    assert (ho.highlight_objects(f.copy(), p) == 255).all()
    _, f, p = by["covers_bottom_right"]
    assert (ho.highlight_objects(f.copy(), p) == 255).all()


def test_synthetic_stream_case():
    frame, p = hl_cases.synthetic_case()
    a, b, so, sm = _run_both(frame, p)
    assert np.array_equal(a, b)
    assert 0 < (a == 255).mean() < 0.5


def test_golden_hashes():
    golden = json.loads((Path(__file__).parent / "golden" / "highlight_golden.json").read_text())
    by = {c[0]: c for c in ADV}
    for g in golden:
        if g["kind"] == "adversarial":
            _, frame, p = by[g["name"]]
        elif g["kind"] == "random":
            frame, p = hl_cases.random_case(g["t"])
        else:
            frame, p = hl_cases.synthetic_case(g["cfg"], g["frame_index"], g["scale"])
        assert hashlib.sha256(frame.tobytes()).hexdigest() == g["input_sha256"], g["name"]
        out = ho.highlight_objects(frame.copy(), p)
        assert hashlib.sha256(out.tobytes()).hexdigest() == g["output_sha256"], g["name"]
        if href.available():  # the hashes were taken from the reference's own output (make_highlight_golden.py)
            ref_out = href.highlight_objects(frame, p)
            assert hashlib.sha256(ref_out.tobytes()).hexdigest() == g["output_sha256"], g["name"]


def test_workload_parameters_match_the_oracle():
    """cvvidproc_b200.synth.CANONICAL_HIGHLIGHT (what bench.py's GPU arm uses) == oracle.canonical_params"""
    from cvvidproc_b200 import synth

    p = ho.canonical_params(np.zeros((4, 4), np.uint8))
    c = synth.CANONICAL_HIGHLIGHT
    assert np.array_equal(synth.canonical_struct_element(), p.struct_element)
    for k in ("threshold", "threshold_lo", "threshold_hi", "min_size_hyst", "min_size_threshold", "width_border"):
        assert c[k] == getattr(p, k)


def test_bench_workload_tables_match_the_package():
    """bench.py repeats the workload tables (its reference arm must not import the package): they are the package's"""
    import importlib.util
    from pathlib import Path

    from cvvidproc_b200 import synth

    spec = importlib.util.spec_from_file_location("bench_mod", Path(__file__).resolve().parent.parent / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for name, p in synth.CONFIG_PARAMS.items():
        assert {k: bench.CONFIGS[name][k] for k in p} == p, name
    assert bench.CANONICAL_HIGHLIGHT == synth.CANONICAL_HIGHLIGHT


def test_bench_gpu_arm_does_not_touch_the_oracle():
    """only the cpu_baseline / reference legs of bench.py may use oracle/ (it is the checker, never the product)"""
    import ast
    from pathlib import Path

    tree = ast.parse((Path(__file__).resolve().parent.parent / "bench.py").read_text())
    allowed = {"cpu_median_fn", "cpu_highlight_rate", "run_reference_arm", "host_synth", "cpu_track_pipeline"}
    for fn in [n for n in tree.body if isinstance(n, ast.FunctionDef)]:
        uses = [n for n in ast.walk(fn) if (isinstance(n, (ast.Import, ast.ImportFrom)) and "oracle" in ast.dump(n))
                or (isinstance(n, ast.Constant) and isinstance(n.value, str) and n.value == "oracle")]
        assert not uses or fn.name in allowed, fn.name


def test_label_model_matches_cv2_restatement_at_full_hd():
    """the independent label model against the cv2 restatement on full 1080p frames of the C3 stream (the geometry the
    benchmark runs): the second opinion on the oracle at the size that matters"""
    from cvvidproc_b200 import synth

    p_ = synth.CONFIG_PARAMS["C3"]
    w, h = p_["width"], p_["height"]
    stack = synth.synth_frames(0, 15, w, h, p_["seed"], p_["ndisks"])
    bg = np.sort(stack, axis=0)[7]
    p = ho.canonical_params(bg)
    frames = [synth.synth_frame(f, w, h, p_["seed"], p_["ndisks"]) for f in (1000, 1097, 1194, 4321, 9999)]
    for i, fr in enumerate(frames):
        want = ho.highlight_objects(fr.copy(), p)
        got = hm.highlight_objects(fr, p.background, p.struct_element, p.threshold, p.threshold_lo, p.threshold_hi,
                                   p.min_size_hyst, p.min_size_threshold)
        assert np.array_equal(got, want), f"frame {i}: {(got != want).sum()} pixels differ"
