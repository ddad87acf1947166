"""CPU checks of the percentile backgrounds (cvvp_median_set_percentile, GetVideoBackground's "cvvp_percentile:P",
TrackObjects' kwargs["cvvp_background_percentile"]): the symbols are bound and reject a null context, the one rank rule
k(N, p) = min(N - 1, floor(N p / 100)) of csrc/median_common.cuh selects np.sort(...)[k] and is N // 2 at p = 50,
malformed algorithm names stay unknown, and bad percentiles are refused before any device work."""
import ctypes
import shutil
import subprocess

import numpy as np
import pytest

import cvvidproc_b200 as cvp
import video_util
from cvvidproc_b200 import _cabi

NEW_SYMBOLS = ["cvvp_median_set_percentile", "cvvp_median_percentile"]


def test_new_symbols_are_declared_exported_and_bound():
    lib = _cabi.load()
    raw = ctypes.CDLL(str(_cabi.LIB_PATH))
    declared = set(_cabi.declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared
        assert hasattr(raw, name)
        assert name in _cabi.BOUND_SYMBOLS
        assert getattr(lib, name).argtypes is not None


def test_null_context_calls_are_rejected():
    lib = _cabi.load()
    assert lib.cvvp_median_set_percentile(None, 50) == -1
    assert lib.cvvp_median_percentile(None) == -1
    assert b"null context" in lib.cvvp_last_error(None)


# A host program that asks csrc/median_common.cuh itself: line 1 = 1 if percentile_rank(N, 50) == N / 2 for every
# N <= 70000, then one rank per (N, p) read from stdin.
_RANK_PROGRAM = r"""
#include <cstdio>
#include "median_common.cuh"
int main()
{
    bool ok = true;
    for (unsigned long long n = 1; n <= 70000; ++n)
        ok = ok && cvvp::percentile_rank(n, 50) == n / 2;
    std::printf("%d\n", ok ? 1 : 0);
    unsigned long long n;
    unsigned p;
    while (std::scanf("%llu %u", &n, &p) == 2)
        std::printf("%llu\n", (unsigned long long)cvvp::percentile_rank(n, p));
    return 0;
}
"""


@pytest.fixture(scope="module")
def rank_program(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not shutil.os.path.exists(nvcc):
        pytest.skip("no nvcc")
    from cvvidproc_b200 import build

    d = tmp_path_factory.mktemp("rank")
    (d / "rank.cu").write_text(_RANK_PROGRAM)
    subprocess.run([nvcc, "-std=c++17", "-I", str(build.CSRC), "-o", str(d / "rank"), str(d / "rank.cu")], check=True,
                   capture_output=True, text=True)
    return d / "rank"


def _ranks(program, pairs):
    text = "".join(f"{n} {p}\n" for n, p in pairs)
    out = subprocess.run([str(program)], input=text, capture_output=True, text=True, check=True).stdout.split()
    return int(out[0]), [int(v) for v in out[1:]]


def test_rank_rule_is_the_upper_median_at_50(rank_program):
    half_ok, ranks = _ranks(rank_program, [(0, 50), (1, 0), (1, 100), (2, 100), (100, 100), (101, 99), (3, 1)])
    assert half_ok == 1  # every N up to 70 000
    assert ranks == [0, 0, 0, 1, 99, 99, 0]


def test_rank_rule_selects_the_numpy_order_statistic(rank_program):
    rng = np.random.default_rng(5)
    ns = [1, 2, 3, 31, 32, 33, 100, 101, 255, 256, 1000, 1281, 3000, 65535, 70000]
    pairs = [(n, p) for n in ns for p in range(101)]
    _, ranks = _ranks(rank_program, pairs)
    for (n, p), k in zip(pairs, ranks):
        assert k == min(n - 1, n * p // 100)
    # the rule the kernels apply -- the first value whose cumulative count exceeds k -- gives np.sort(...)[k]
    for n in (1, 2, 33, 101, 1000):
        stack = rng.integers(0, 256, (n, 64), dtype=np.uint8)
        stack[:, :8] = 7  # constant elements
        stack[:, 8:16] = np.where(np.arange(n)[:, None] < n // 2, 10, 200)  # a two-level split
        srt = np.sort(stack, axis=0)
        cum = np.cumsum(np.stack([(stack == v).sum(axis=0) for v in range(256)]), axis=0)
        for p in (0, 1, 25, 49, 50, 51, 75, 99, 100):
            k = ranks[pairs.index((n, p))]
            first = np.argmax(cum > k, axis=0)
            assert np.array_equal(first, srt[k]), (n, p)
            assert np.array_equal(np.partition(stack, k, axis=0)[k], srt[k])


@pytest.fixture(scope="module")
def still_video(tmp_path_factory):
    # every frame the same: every percentile of it is that frame, with or without a GPU
    frame = np.random.default_rng(1).integers(0, 256, (24, 32), dtype=np.uint8)
    return video_util.write_lossless(tmp_path_factory.mktemp("vid") / "still.avi", np.stack([frame] * 5))


@pytest.mark.parametrize("name", ["cvvp_percentile", "cvvp_percentile:", "cvvp_percentile:101", "cvvp_percentile:-1",
                                  "cvvp_percentile:050", "cvvp_percentile:00", "cvvp_percentile:5.5", "cvvp_percentile:1000",
                                  "cvvp_percentile: 5", "cvvp_percentile:5 ", "CVVP_PERCENTILE:5", "percentile:5",
                                  "cvvp_percentile:+5", "hist:50"])
def test_malformed_percentile_names_are_unknown_algorithms(still_video, capfd, name):
    assert cvp.GetVideoBackground(cvp.VidBgPack(still_video, bg_algo=name)) is None
    err = capfd.readouterr().err
    assert f"Unknown background algorithm detected: {name}\n" in err
    assert f"tried to get vid background with unknown algorithm: {name}\n" in err


def _outcome(path, algo, capfd):
    try:
        res = ("ok", cvp.GetVideoBackground(cvp.VidBgPack(path, bg_algo=algo)).tobytes())
    except Exception as e:  # noqa: BLE001 -- the outcome of both names is compared, whatever it is
        res = (type(e).__name__, str(e))
    cap = capfd.readouterr()
    return res, cap.out


@pytest.mark.parametrize("p", [0, 1, 9, 10, 50, 99, 100])
def test_well_formed_percentile_names_run_the_hist_path(still_video, capfd, p):
    # without a GPU both fail the same way at the first device call; with one both return the frame
    want, out_hist = _outcome(still_video, "hist", capfd)
    got, out_p = _outcome(still_video, f"cvvp_percentile:{p}", capfd)
    assert got == want
    assert out_p == out_hist and "Frames: 5; Res: 32x24" in out_p
    assert "unknown algorithm" not in capfd.readouterr().err


def _pack(kwargs):
    hp = cvp.HighlightObjectsPack(np.zeros((4, 4), np.uint8), np.ones((2, 2), np.uint8), 1, 1, 1, 1, 1, 1)
    ap = cvp.AssignObjectsPack(lambda **kw: 0, kwargs)
    return cvp.VidObjectTrackPack("/nonexistent/video.mp4", hp, ap)


@pytest.mark.parametrize("p", [-1, 101, 1000, "50", 2.5, True, False, None, np.float32(5)])
def test_track_objects_refuses_a_bad_percentile_before_any_device_work(p):
    # a missing video makes TrackObjects return {} without raising: the percentile is checked before that
    with pytest.raises(RuntimeError, match="cvvp_background_percentile"):
        cvp.TrackObjects(_pack({"cvvp_background_window": 5, "cvvp_background_percentile": p}))


@pytest.mark.parametrize("p", [0, 50, 90])
def test_track_objects_refuses_a_percentile_without_a_window(p):
    with pytest.raises(RuntimeError, match="cvvp_background_percentile"):
        cvp.TrackObjects(_pack({"cvvp_background_percentile": p}))


@pytest.mark.parametrize("p", [0, 1, 50, 99, 100, np.int64(90)])
def test_track_objects_accepts_a_good_percentile(p, capfd):
    kwargs = {"cvvp_background_window": 5, "cvvp_background_percentile": p}
    assert cvp.TrackObjects(_pack(kwargs)) == {}
    assert "Video file not detected" in capfd.readouterr().err
    assert kwargs == {"cvvp_background_window": 5, "cvvp_background_percentile": p}
