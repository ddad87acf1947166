"""Host references and input builders for the object-polarity tests (cvvp_highlight_set_polarity, TrackObjects'
kwargs["cvvp_polarity"]).

The reference only computes the "dark" difference d = saturate_u8(bg - frame) (highlight_objects_algo.cpp:27-29).  The
restatements of oracle/ compute exactly that; the functions below run their later steps -- which depend only on d -- on
the difference image of any polarity:

  highlight_objects        the cv2 restatement's steps (oracle/highlight_oracle.py, :35-77) on d
  model_highlight_objects  the label model's steps (oracle/highlight_model.py) on d

At "dark" both are held to the oracle functions they compose (tests/test_polarity_cpu.py).  Two identities tie the
other polarities to "dark", and so to the stored reference outputs:

  (1) bright(f, bg) == dark(255 - f, 255 - bg)
  (2) both(min(f, bg), bg) == dark(f, bg)   and   both(max(f, bg), bg) == bright(f, bg)
"""
import dataclasses

import cv2
import numpy as np

import hl_cases
from oracle import highlight_model as hm
from oracle import highlight_oracle as ho

POLARITIES = {"dark": 0, "bright": 1, "both": 2}  # CVVP_POLARITY_*


def difference_image(background, frame, polarity):
    """:27-30 in a polarity: cv::subtract(bg, frame) (the reference), cv::subtract(frame, bg), or cv::absdiff (the line
    the reference left commented out at :30)"""
    if polarity == "dark":
        return cv2.subtract(background, frame)
    if polarity == "bright":
        return cv2.subtract(frame, background)
    if polarity == "both":
        return cv2.absdiff(background, frame)
    raise ValueError(f"unknown polarity {polarity!r}")


def highlight_objects(frame, p, polarity="dark", stages=None):
    """HighlightObjects :17-78 as oracle/highlight_oracle.py restates it, on the difference image of `polarity`"""
    assert frame.dtype == np.uint8 and frame.ndim == 2
    im_diff = difference_image(p.background, frame, polarity)
    selem = np.ascontiguousarray(p.struct_element)
    a = cv2.morphologyEx(ho.threshold_image(im_diff, p.threshold), cv2.MORPH_OPEN, selem)  # :35, :39
    ho.remove_small_objects(a, p.min_size_threshold)  # :43
    ho.fill_holes(a)  # :47
    b = cv2.morphologyEx(ho.threshold_image_with_hysteresis(im_diff, p.threshold_lo, p.threshold_hi), cv2.MORPH_OPEN,
                         selem)  # :54, :61
    ho.remove_small_objects(b, p.min_size_hyst)  # :65
    ho.fill_holes(b)  # :73
    if stages is not None:
        stages.update(diff=im_diff)
    return cv2.bitwise_or(a, b)  # :77


def model_difference(background, frame, polarity):
    """the label model's d (hm.diff_sat at "dark") in int arithmetic"""
    s = background.astype(np.int16) - frame.astype(np.int16)
    if polarity == "dark":
        return np.clip(s, 0, 255).astype(np.uint8)
    if polarity == "bright":
        return np.clip(-s, 0, 255).astype(np.uint8)
    if polarity == "both":
        return np.abs(s).astype(np.uint8)
    raise ValueError(f"unknown polarity {polarity!r}")


def model_highlight_objects(frame, p, polarity="dark"):
    """oracle/highlight_model.py's highlight_objects on the difference image of `polarity`"""
    d = model_difference(p.background, frame, polarity)
    selem = np.asarray(p.struct_element) != 0
    a = hm.fill_holes(hm.remove_small_objects(hm.morph_open(hm.threshold_mask(d, p.threshold), selem),
                                              p.min_size_threshold))
    b = hm.fill_holes(hm.remove_small_objects(hm.morph_open(hm.hysteresis(d, p.threshold_lo, p.threshold_hi), selem),
                                              p.min_size_hyst))
    return ((a | b).astype(np.uint8)) * 255


def masks(frames, p, polarity, backgrounds=None):
    """highlight_objects of every frame; frame t against backgrounds[t] when given"""
    if backgrounds is None:
        return np.stack([highlight_objects(f.copy(), p, polarity) for f in frames])
    return np.stack([highlight_objects(f.copy(), dataclasses.replace(p, background=b), polarity)
                     for f, b in zip(frames, backgrounds)])


def inverted(frame, p):
    """identity (1)'s input: 255 - frame against 255 - background"""
    return (255 - frame).astype(np.uint8), dataclasses.replace(p, background=(255 - p.background).astype(np.uint8))


def mixed(frame, bg):
    """a frame whose difference has both signs: the right half of (frame - bg) mirrored about the background, so dark
    objects on the left become bright objects on the right"""
    f = frame.astype(np.int32)
    b = bg.astype(np.int32)
    half = frame.shape[1] // 2
    f[:, half:] = 2 * b[:, half:] - f[:, half:]
    return np.clip(f, 0, 255).astype(np.uint8)


def mixed_random_case(t):
    frame, p = hl_cases.random_case(t)
    return mixed(frame, p.background), p


def mixed_adversarial_cases():
    return [(name, mixed(frame, p.background), p) for name, frame, p in hl_cases.adversarial_cases()]


def golden_cases():
    """(entry, frame, params) of every stored reference output (tests/golden/highlight_golden.json)"""
    import json
    from pathlib import Path

    golden = json.loads((Path(__file__).parent / "golden" / "highlight_golden.json").read_text())
    by = {c[0]: c for c in hl_cases.adversarial_cases()}
    out = []
    for g in golden:
        if g["kind"] == "adversarial":
            _, frame, p = by[g["name"]]
        elif g["kind"] == "random":
            frame, p = hl_cases.random_case(g["t"])
        else:
            frame, p = hl_cases.synthetic_case(g["cfg"], g["frame_index"], g["scale"])
        out.append((g, frame, p))
    return out
