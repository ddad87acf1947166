"""Shared input builders for the highlight tests (CPU oracle tests and GPU parity tests use the same cases)."""
import cv2
import numpy as np

from oracle import highlight_oracle as ho


def blob_frame(h, w, seed, bgv=160, amp=60, sigma=2.0, noise=5):
    r = np.random.default_rng(seed)
    n = r.random((h, w)).astype(np.float32)
    n = cv2.GaussianBlur(n, (0, 0), sigma)
    n = (n - n.min()) / max(float(n.max() - n.min()), 1e-6)
    bg = np.full((h, w), bgv, np.uint8)
    frame = np.clip(bgv - (n * amp).astype(np.int32) + r.integers(-noise, noise + 1, (h, w)), 0, 255).astype(np.uint8)
    return frame, bg


def random_case(t):
    rng = np.random.default_rng(1000 + t)
    h = int(rng.integers(8, 70))
    w = int(rng.integers(8, 90))
    frame, bg = blob_frame(h, w, t, bgv=int(rng.integers(100, 220)), sigma=float(rng.uniform(0.8, 3.0)))
    if t % 3:
        se = ho.canonical_struct_element()
    else:
        se = rng.integers(0, 2, (int(rng.integers(1, 6)), int(rng.integers(1, 6)))).astype(np.uint8)
        if se.sum() == 0:
            se[0, 0] = 1
    p = ho.HighlightParams(bg, se, int(rng.integers(5, 40)), int(rng.integers(3, 30)), int(rng.integers(3, 45)),
                           int(rng.choice([0, 1, 5, 20, 40, 100])), int(rng.choice([0, 1, 5, 20, 40, 100])), 5)
    return frame, p


def _params(bg, se=None, th=14, lo=7, hi=16, ms_h=20, ms_t=20):
    return ho.HighlightParams(bg, ho.canonical_struct_element() if se is None else se, th, lo, hi, ms_h, ms_t, 5)


def _with_rects(h, w, rects, bgv=200, depth=60):
    """frame = background minus `depth` inside the given (y0, y1, x0, x1, depth?) rectangles"""
    bg = np.full((h, w), bgv, np.uint8)
    f = bg.astype(np.int32).copy()
    for r in rects:
        y0, y1, x0, x1 = r[:4]
        dep = r[4] if len(r) > 4 else depth
        f[y0:y1, x0:x1] -= dep
    return np.clip(f, 0, 255).astype(np.uint8), bg


def adversarial_cases():
    """SURVEY.md 9.7.  Returns a list of (name, frame, params)."""
    out = []
    h, w = 40, 56
    one = np.ones((1, 1), np.uint8)
    # object covering pixel (0,0) / the bottom-right pixel (FillHoles seed quirk -> all-white frames)
    f, bg = _with_rects(h, w, [(0, 12, 0, 14)])
    out.append(("covers_origin", f, _params(bg)))
    f, bg = _with_rects(h, w, [(h - 12, h, w - 14, w)])
    out.append(("covers_bottom_right", f, _params(bg)))
    # full-height and full-width objects
    f, bg = _with_rects(h, w, [(0, h, 20, 30)])
    out.append(("full_height", f, _params(bg)))
    f, bg = _with_rects(h, w, [(15, 25, 0, w)])
    out.append(("full_width", f, _params(bg)))
    # all-zero diff, frame brighter than the background everywhere, all-255 mask
    bg = np.full((h, w), 100, np.uint8)
    out.append(("zero_diff", bg.copy(), _params(bg)))
    out.append(("brighter_everywhere", np.full((h, w), 180, np.uint8), _params(bg)))
    out.append(("all_set", np.zeros((h, w), np.uint8), _params(np.full((h, w), 255, np.uint8))))
    # single pixel / two pixel components and a 1-pixel hole, with the 1x1 structuring element so they survive opening
    for ms in (0, 1, 2, 5):
        f, bg = _with_rects(h, w, [(5, 6, 5, 6), (5, 6, 9, 11), (10, 12, 10, 11), (20, 27, 20, 27), (23, 24, 23, 24, -60)])
        out.append((f"tiny_components_ms{ms}", f, _params(bg, se=one, ms_h=ms, ms_t=ms)))
    # nested ring > gap > blob, for both remove-small and hysteresis, several min sizes
    for ms in (5, 20, 40, 100, 1000):
        f, bg = _with_rects(h, w, [(4, 36, 6, 50), (9, 31, 11, 45, -60), (14, 26, 18, 38), (18, 22, 24, 32, -60),
                                   (19, 21, 27, 29)])
        out.append((f"nested_rings_ms{ms}", f, _params(bg, se=one, ms_h=ms, ms_t=ms)))
    # hi blob nested inside a hi ring (RETR_EXTERNAL drops it), lo region spanning both
    f, bg = _with_rects(h, w, [(4, 36, 6, 50, 10), (8, 32, 10, 46, 10), (12, 28, 16, 40, -10), (17, 23, 24, 32, 12)])
    out.append(("hyst_nested_hi", f, _params(bg, se=one, lo=7, hi=16, ms_h=0, ms_t=0)))
    # diagonal-only connections (S8 vs S4)
    bg = np.full((h, w), 200, np.uint8)
    f = bg.copy()
    for i in range(12):
        f[5 + i, 5 + i] = 100
        f[5 + i, 30 - i] = 100
    f[25:30, 25:30] = 100
    f[30:35, 30:35] = 100
    out.append(("diagonals", f, _params(bg, se=one, ms_h=0, ms_t=0)))
    out.append(("diagonals_ms3", f, _params(bg, se=one, ms_h=3, ms_t=3)))
    # components touching every image edge
    f, bg = _with_rects(h, w, [(0, 6, 10, 20), (h - 6, h, 30, 40), (10, 20, 0, 6), (22, 30, w - 6, w)])
    out.append(("touching_edges", f, _params(bg)))
    # lo > hi
    f, bgb = blob_frame(48, 64, 5)
    out.append(("lo_gt_hi", f, _params(bgb, lo=30, hi=12)))
    out.append(("lo_gt_hi_1x1", f, _params(bgb, se=one, lo=35, hi=10, ms_h=0, ms_t=0)))
    # thresholds at and beyond the value range, and Otsu
    for th in (-5, -1, 0, 254, 255, 300):
        out.append((f"threshold_{th}", f, _params(bgb, th=th)))
    # structuring elements
    ses = {
        "ellipse5": cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (5, 5)),
        "one": one,
        "asym": np.array([[1, 0, 0], [1, 1, 0]], np.uint8),
        "row": np.ones((1, 4), np.uint8),
        "col": np.ones((5, 1), np.uint8),
        "allzero": np.zeros((3, 3), np.uint8),
        "values": np.array([[0, 7, 0], [200, 1, 2], [0, 9, 0]], np.uint8),  # any non-zero value counts as set
    }
    for name, se in ses.items():
        out.append((f"selem_{name}", f, _params(bgb, se=se)))
    # non-multiple-of-16 geometry
    f2, bg2 = blob_frame(479 // 4, 641 // 4, 9)
    out.append(("ragged_geometry", f2, _params(bg2)))
    f3, bg3 = blob_frame(3, 5, 10)
    out.append(("tiny_image", f3, _params(bg3, se=one, ms_h=0, ms_t=0)))
    f4, bg4 = blob_frame(1, 40, 11)
    out.append(("one_row", f4, _params(bg4, se=one, ms_h=0, ms_t=0)))
    f5, bg5 = blob_frame(40, 1, 12)
    out.append(("one_col", f5, _params(bg5, se=one, ms_h=0, ms_t=0)))
    return out


def synthetic_case(cfg="C3", frame_index=7, scale=4):
    """A reduced-size frame of the BASELINE synthetic stream with the median of its first frames as background."""
    from cvvidproc_b200 import synth

    p = synth.CONFIG_PARAMS[cfg]
    w, h = p["width"] // scale, p["height"] // scale
    stack = synth.synth_frames(0, 31, w, h, p["seed"], p["ndisks"])
    bg = np.sort(stack, axis=0)[31 // 2]
    frame = synth.synth_frame(frame_index, w, h, p["seed"], p["ndisks"])
    return frame, ho.canonical_params(bg)


def reference_sha256(name):
    """SHA-256 of the reference's own HighlightObjectsAlgo output on the case `name` (an adversarial case's name or
    random_<t>), as tests/golden/make_highlight_golden.py stored it; None for a case it did not store."""
    import json
    from pathlib import Path

    global _REF_SHA
    if _REF_SHA is None:
        golden = json.loads((Path(__file__).parent / "golden" / "highlight_golden.json").read_text())
        _REF_SHA = {g["name"]: g["output_sha256"] for g in golden}
    return _REF_SHA.get(name)


_REF_SHA = None
