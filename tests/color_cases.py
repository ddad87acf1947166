"""Host reference and input builders for the colour highlight tests (cvvp_highlight_set_channels, TrackObjects'
kwargs["cvvp_color"]).

A job of C channels takes frames and backgrounds of C interleaved channels, and its difference image is

    d(x, y) = max over c of d_c,   d_c = the polarity's difference of channel c (tests/polarity_cases.py)

Everything after d is the grey stage.  Three identities tie the colour mode to the reference's stored outputs:

  (1) C = 1 is the grey job
  (2) a grey frame and background replicated into C channels give the grey masks
  (3) colour(f, bg, polarity) == dark(255 - D, 255), D the colour d above: the grey "dark" path's d of that pair is D
"""
import dataclasses

import numpy as np

import hl_cases
import polarity_cases as pc

CHANNELS = (1, 2, 3, 4)


def color_difference(background, frame, polarity):
    """d = the largest per-channel difference of `polarity` over the last axis (int arithmetic)"""
    assert background.dtype == np.uint8 and frame.dtype == np.uint8 and background.shape == frame.shape[-background.ndim:]
    s = background.astype(np.int16) - frame.astype(np.int16)
    if polarity == "dark":
        d = np.clip(s, 0, 255)
    elif polarity == "bright":
        d = np.clip(-s, 0, 255)
    elif polarity == "both":
        d = np.abs(s)
    else:
        raise ValueError(f"unknown polarity {polarity!r}")
    return d.max(axis=-1).astype(np.uint8)


def as_dark(frame, p, polarity):
    """identity (3)'s input: the grey frame 255 - D against a background of 255, with p's other parameters"""
    d = color_difference(p.background, frame, polarity)
    return (255 - d).astype(np.uint8), dataclasses.replace(p, background=np.full(d.shape, 255, np.uint8))


def highlight_objects(frame, p, polarity="dark"):
    """the colour job's masks of one (H, W, C) frame against p.background (H, W, C), through identity (3)"""
    f, q = as_dark(frame, p, polarity)
    return pc.highlight_objects(f, q, "dark")


def masks(frames, p, polarity, backgrounds=None):
    if backgrounds is None:
        return np.stack([highlight_objects(f, p, polarity) for f in frames])
    return np.stack([highlight_objects(f, dataclasses.replace(p, background=b), polarity)
                     for f, b in zip(frames, backgrounds)])


def replicated(frame, p, c):
    """identity (2)'s input: frame and background repeated into c channels"""
    rep = lambda a: np.ascontiguousarray(np.repeat(a[..., None], c, axis=-1))
    return rep(frame), dataclasses.replace(p, background=rep(p.background))


def colorize(frame, p, c, seed):
    """a colour case of c channels built on a grey one: channel 0 is the grey frame against the grey background; the
    other channels carry objects of their own (the frame rolled sideways, with noise) against backgrounds offset by
    a few grey levels, so that the largest channel changes from pixel to pixel"""
    rng = np.random.default_rng(seed)
    f = [frame]
    b = [p.background]
    for k in range(1, c):
        off = int(rng.integers(-6, 7))
        bk = np.clip(p.background.astype(np.int16) + off, 0, 255)
        fk = np.roll(frame, 7 * k, axis=1).astype(np.int16) + off + rng.integers(-3, 4, frame.shape)
        b.append(bk.astype(np.uint8))
        f.append(np.clip(fk, 0, 255).astype(np.uint8))
    return (np.ascontiguousarray(np.stack(f, axis=-1)),
            dataclasses.replace(p, background=np.ascontiguousarray(np.stack(b, axis=-1))))


def random_case(t, c):
    frame, p = pc.mixed_random_case(t)
    return colorize(frame, p, c, 1000 + t)


def adversarial_cases(c):
    return [(name,) + colorize(frame, p, c, 2000 + i) for i, (name, frame, p) in enumerate(pc.mixed_adversarial_cases())]


def blob_case(h, w, c, seed):
    frame, bg = hl_cases.blob_frame(h, w, seed, sigma=2.0, amp=70)
    from oracle import highlight_oracle as ho

    return colorize(pc.mixed(frame, bg), ho.canonical_params(bg), c, seed)
