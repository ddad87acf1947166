"""ctypes view of libcvvp_cuda.so (include/cvvp.h).

This is what tests/ and bench.py call: every GPU test goes through the C ABI exactly as the
reference-side binding in INTEGRATION.md would.  There is no CPU fallback here: if the library is
missing or no B200 is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libcvvp_cuda.so"
HEADER = PKG_DIR.parent / "include" / "cvvp.h"

_lib = None
BOUND_SYMBOLS: list[str] = []


class CvvpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"cvvp error {code}: {message}")
        self.code = code


def declared_symbols() -> list[str]:
    """Every function name include/cvvp.h declares (used by the symbol-export test)."""
    text = HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cvvp_[a-z0-9_]+)\s*\(", text)))


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the CUDA path)"
        )
    lib = C.CDLL(str(LIB_PATH))
    vp, i32, i64, sz, u32 = C.c_void_p, C.c_int, C.c_longlong, C.c_size_t, C.c_uint32
    sigs = {
        "cvvp_abi_version": (i32, []),
        "cvvp_ctx_create": (i32, [i32, C.POINTER(vp)]),
        "cvvp_ctx_destroy": (None, [vp]),
        "cvvp_last_error": (C.c_char_p, [vp]),
        "cvvp_ctx_synchronize": (i32, [vp]),
        "cvvp_ctx_stream": (vp, [vp]),
        "cvvp_ctx_device": (i32, [vp]),
        "cvvp_ctx_sm_count": (i32, [vp]),
        "cvvp_ctx_launch_count": (i64, [vp]),
        "cvvp_pool_trim": (sz, []),
        "cvvp_host_alloc": (i32, [sz, C.POINTER(vp)]),
        "cvvp_host_free": (i32, [vp]),
        "cvvp_ctx_copy_to_host": (i32, [vp, vp, vp, sz]),
        "cvvp_median_begin": (i32, [vp, sz, i64]),
        "cvvp_median_push": (i32, [vp, vp, i64, sz]),
        "cvvp_median_count": (i64, [vp]),
        "cvvp_median_stack_device": (i32, [vp, C.POINTER(vp), C.POINTER(sz), C.POINTER(i64)]),
        "cvvp_median_finish": (i32, [vp, vp]),
        "cvvp_median_abort": (i32, [vp]),
        "cvvp_median_device": (i32, [vp, vp, i64, sz, sz, vp, vp]),
        "cvvp_median_last_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
        "cvvp_median_rolling_device": (i32, [vp, vp, i64, sz, sz, i32, i64, i64, vp, sz, vp]),
        "cvvp_median_set_percentile": (i32, [vp, i32]),
        "cvvp_median_percentile": (i32, [vp]),
        "cvvp_highlight_begin": (i32, [vp, vp, i32, i32, vp, i32, i32, i32, i32, i32, i32, i32, i32]),
        "cvvp_highlight_frames": (i32, [vp, vp, i64, sz, vp, sz]),
        "cvvp_highlight_device": (i32, [vp, vp, i64, sz, vp, sz, vp]),
        "cvvp_highlight_end": (i32, [vp]),
        "cvvp_highlight_set_polarity": (i32, [vp, i32]),
        "cvvp_highlight_polarity": (i32, [vp]),
        "cvvp_highlight_set_channels": (i32, [vp, i32]),
        "cvvp_highlight_channels": (i32, [vp]),
        "cvvp_highlight_set_component_stats": (i32, [vp, i32]),
        "cvvp_highlight_component_stats": (i32, [vp]),
        "cvvp_highlight_device_cc": (i32, [vp, vp, i64, sz, vp, sz, vp, i32, vp, vp, sz, vp]),
        "cvvp_highlight_frames_cc": (i32, [vp, vp, i64, sz, vp, sz, vp, i32, vp, vp, sz]),
        "cvvp_highlight_device_bg": (i32, [vp, vp, i64, sz, vp, sz, vp, sz, vp, i32, vp, vp, sz, vp]),
        "cvvp_highlight_rolling_begin": (i32, [vp, i32, i64, vp, i32, i32]),
        "cvvp_highlight_rolling_push": (i32, [vp, vp, i64, sz]),
        "cvvp_highlight_rolling_close": (i32, [vp]),
        "cvvp_highlight_rolling_pending": (i32, [vp]),
        "cvvp_highlight_rolling_ready": (i32, [vp]),
        "cvvp_highlight_rolling_next": (i32, [vp, vp, sz, i64, C.POINTER(i64), C.POINTER(i64), vp, vp, vp, sz]),
        "cvvp_highlight_rolling_end": (i32, [vp]),
        "cvvp_highlight_set_path": (i32, [vp, i32]),
        "cvvp_highlight_frames_in_flight": (i32, [vp, C.POINTER(i32)]),
        "cvvp_synth_frames_device": (i32, [vp, vp, sz, i32, i32, i32, i32, i64, i64, u32, i32, vp]),
        "cvvp_median_shard_begin": (i32, [vp, sz, i32, i32]),
        "cvvp_median_shard_begin_frames": (i32, [vp, sz, i32, i32, i64]),
        "cvvp_median_shard_unresolved": (i32, [vp, vp, C.POINTER(i64)]),
        "cvvp_median_shard_barrier": (i32, [vp, vp]),
        "cvvp_median_shard_export": (i32, [vp, vp]),
        "cvvp_median_shard_import": (i32, [vp, i32, vp]),
        "cvvp_median_shard_attach": (i32, [vp, i32, vp]),
        "cvvp_median_shard_phase": (i32, [vp, i32, vp, i64, sz, vp]),
        "cvvp_median_shard_result": (i32, [vp, C.POINTER(vp)]),
        "cvvp_median_shard_end": (i32, [vp]),
        "cvvp_frame_format_out_bytes": (sz, [vp]),
        "cvvp_frames_prepare_device": (i32, [vp, vp, i64, sz, vp, vp, sz, vp]),
        "cvvp_frames_prepare": (i32, [vp, vp, i64, sz, vp, vp, sz]),
        "cvvp_median_push_source": (i32, [vp, vp, i64, sz, vp]),
        "cvvp_highlight_queue_begin": (i32, [vp, i32, i64, vp, i32]),
        "cvvp_highlight_queue_pending": (i32, [vp]),
        "cvvp_highlight_submit": (i32, [vp, vp, i64, sz]),
        "cvvp_highlight_queue_ready": (i32, [vp]),
        "cvvp_highlight_next": (i32, [vp, vp, sz, C.POINTER(i64), vp, vp]),
        "cvvp_highlight_queue_end": (i32, [vp]),
        "cvvp_highlight_slot_acquire": (i32, [vp, C.POINTER(vp), C.POINTER(sz), C.POINTER(i64)]),
        "cvvp_highlight_slot_commit": (i32, [vp, i64]),
        "cvvp_highlight_next_view": (i32, [vp, C.POINTER(vp), C.POINTER(sz), C.POINTER(i64), C.POINTER(vp), C.POINTER(vp)]),
        "cvvp_highlight_view_release": (i32, [vp]),
    }
    global BOUND_SYMBOLS
    BOUND_SYMBOLS = sorted(sigs)
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


FRAMES_AS_IS, FRAMES_CHANNEL0, FRAMES_RGB2GRAY = 0, 1, 2


class FrameFormat(C.Structure):
    """struct cvvp_frame_format (include/cvvp.h): geometry of the decoded frames, the resolved crop rectangle and
    the channel reduction of CvVidFramesGeneratorAlgo::GetTokenSet."""

    _fields_ = [("src_width", C.c_int32), ("src_height", C.c_int32), ("src_channels", C.c_int32),
                ("crop_x", C.c_int32), ("crop_y", C.c_int32), ("crop_width", C.c_int32), ("crop_height", C.c_int32),
                ("mode", C.c_int32)]

    @classmethod
    def of(cls, frame_shape, mode: int, crop=None) -> "FrameFormat":
        """frame_shape: (H, W) or (H, W, C) of one decoded frame; crop: (x, y, w, h) or None for the whole frame"""
        h, w = int(frame_shape[0]), int(frame_shape[1])
        c = int(frame_shape[2]) if len(frame_shape) == 3 else 1
        x, y, cw, ch = crop if crop is not None else (0, 0, w, h)
        return cls(w, h, c, x, y, cw, ch, mode)

    @property
    def out_shape(self):
        if self.mode == FRAMES_AS_IS and self.src_channels > 1:
            return (self.crop_height, self.crop_width, self.src_channels)
        return (self.crop_height, self.crop_width)


class PinnedBuffer:
    """Page-locked host memory from cvvp_host_alloc, exposed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        lib = load()
        p = C.c_void_p()
        rc = lib.cvvp_host_alloc(nbytes, C.byref(p))
        if rc != 0:
            raise CvvpError(rc, (lib.cvvp_last_error(None) or b"").decode())
        self._ptr = p
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes,))

    def close(self):
        if self._ptr is not None:
            self.array = None
            load().cvvp_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One cvvp_ctx (one CUDA device)."""

    def __init__(self, device: int = -1):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.cvvp_ctx_create(device, C.byref(h))
        if rc != 0:
            raise CvvpError(rc, (self._lib.cvvp_last_error(None) or b"").decode())
        self._h = h

    # -- plumbing -------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise CvvpError(rc, (self._lib.cvvp_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.cvvp_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return int(self._lib.cvvp_ctx_stream(self._h) or 0)

    @property
    def device(self) -> int:
        return self._lib.cvvp_ctx_device(self._h)

    @property
    def sm_count(self) -> int:
        return self._lib.cvvp_ctx_sm_count(self._h)

    @property
    def launch_count(self) -> int:
        return int(self._lib.cvvp_ctx_launch_count(self._h))

    def synchronize(self):
        self._check(self._lib.cvvp_ctx_synchronize(self._h))

    def copy_to_host(self, device_ptr: int, nbytes: int) -> np.ndarray:
        out = np.empty(nbytes, np.uint8)
        self._check(self._lib.cvvp_ctx_copy_to_host(self._h, out.ctypes.data, device_ptr, nbytes))
        return out

    # -- median ---------------------------------------------------------------------------
    def median_begin(self, nelem: int, nframes_hint: int = -1):
        self._check(self._lib.cvvp_median_begin(self._h, nelem, nframes_hint))

    def median_push(self, frames: np.ndarray):
        """frames: uint8 array (n, ...) whose trailing dims are one frame; frame bytes must be contiguous."""
        if frames.dtype != np.uint8 or frames.ndim < 2:
            raise TypeError("frames must be a uint8 array of shape (n, ...)")
        n = frames.shape[0]
        if n == 0:
            return
        nelem = int(np.prod(frames.shape[1:]))
        one = frames[0]
        if not one.flags.c_contiguous:
            frames = np.ascontiguousarray(frames)
        stride = frames.strides[0] if n > 1 else nelem
        if stride < nelem:
            frames = np.ascontiguousarray(frames)
            stride = nelem
        self._check(self._lib.cvvp_median_push(self._h, frames.ctypes.data, n, stride))
        self._keepalive = frames

    def median_push_source(self, frames: np.ndarray, fmt: FrameFormat):
        """frames: DECODED uint8 frames (n, H, W[, C]); cropped / channel-reduced on the device into the stack"""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("frames must be uint8")
        n = frames.shape[0]
        stride = int(np.prod(frames.shape[1:]))
        self._check(self._lib.cvvp_median_push_source(self._h, frames.ctypes.data, n, stride, C.byref(fmt)))
        self._keepalive = frames

    def frames_prepare(self, frames: np.ndarray, fmt: FrameFormat) -> np.ndarray:
        """DECODED uint8 frames (n, H, W[, C]) -> prepared frames (n, crop_h, crop_w[, C]) (host in, host out)"""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("frames must be uint8")
        n = frames.shape[0]
        stride = int(np.prod(frames.shape[1:]))
        out = np.empty((n,) + tuple(fmt.out_shape), np.uint8)
        ob = int(np.prod(fmt.out_shape))
        self._check(self._lib.cvvp_frames_prepare(self._h, frames.ctypes.data, n, stride, C.byref(fmt), out.ctypes.data, ob))
        return out

    def frames_prepare_device(self, d_src: int, n: int, src_stride: int, fmt: FrameFormat, d_dst: int, dst_stride: int,
                              stream: int = 0):
        self._check(self._lib.cvvp_frames_prepare_device(self._h, d_src, n, src_stride, C.byref(fmt), d_dst, dst_stride,
                                                         stream or None))

    def median_push_raw(self, ptr: int, n: int, stride: int):
        self._check(self._lib.cvvp_median_push(self._h, ptr, n, stride))

    def median_stack_device(self):
        """(device pointer, frame stride, frames) of the running job's stack; pushes so far are ordered before later work
        on the compute stream"""
        p, st, n = C.c_void_p(), C.c_size_t(), C.c_longlong()
        self._check(self._lib.cvvp_median_stack_device(self._h, C.byref(p), C.byref(st), C.byref(n)))
        return int(p.value or 0), int(st.value), int(n.value)

    def median_count(self) -> int:
        return int(self._lib.cvvp_median_count(self._h))

    def median_finish(self, out: np.ndarray | None = None, nelem: int | None = None) -> np.ndarray:
        if out is None:
            out = np.empty(nelem, np.uint8)
        if out.dtype != np.uint8 or not out.flags.c_contiguous:
            raise TypeError("out must be a contiguous uint8 array")
        self._check(self._lib.cvvp_median_finish(self._h, out.ctypes.data))
        self._keepalive = None
        return out

    def median_abort(self):
        self._check(self._lib.cvvp_median_abort(self._h))

    def median(self, frames: np.ndarray, chunk: int = 64) -> np.ndarray:
        """Whole job through the streaming host interface: begin, push in chunks, finish."""
        n = frames.shape[0]
        nelem = int(np.prod(frames.shape[1:]))
        self.median_begin(nelem, n)
        try:
            for i in range(0, n, chunk):
                self.median_push(frames[i : i + chunk])
        except Exception:
            self.median_abort()
            raise
        return self.median_finish(nelem=nelem).reshape(frames.shape[1:])

    def median_device(self, d_frames: int, nframes: int, nelem: int, frame_stride: int, d_out: int, stream: int = 0):
        self._check(self._lib.cvvp_median_device(self._h, d_frames, nframes, nelem, frame_stride, d_out, stream or None))

    def median_rolling_device(self, d_frames: int, nframes: int, nelem: int, frame_stride: int, window: int, t0: int,
                              t1: int, d_out: int, out_stride: int, stream: int = 0):
        """backgrounds of frames [t0, t1): the context's percentile (the upper median at the default) of each frame's
        centred window of `window` frames"""
        self._check(self._lib.cvvp_median_rolling_device(self._h, d_frames, nframes, nelem, frame_stride, window, t0, t1,
                                                         d_out, out_stride, stream or None))

    def median_set_percentile(self, percent: int):
        """every background of this context becomes sorted[min(N - 1, N * percent // 100)]; jobs take it when they begin"""
        self._check(self._lib.cvvp_median_set_percentile(self._h, percent))

    def median_percentile(self) -> int:
        return int(self._lib.cvvp_median_percentile(self._h))

    def median_last_kernel_ms(self) -> float:
        v = C.c_float()
        self._check(self._lib.cvvp_median_last_kernel_ms(self._h, C.byref(v)))
        return float(v.value)

    # -- frame-sharded median (one context per rank) ----------------------------------------
    IPC_HANDLE_BYTES = 64

    def median_shard_begin(self, nelem: int, rank: int, world: int, max_rank_frames: int | None = None):
        if max_rank_frames is None:
            self._check(self._lib.cvvp_median_shard_begin(self._h, nelem, rank, world))
        else:
            self._check(self._lib.cvvp_median_shard_begin_frames(self._h, nelem, rank, world, max_rank_frames))

    def median_shard_barrier(self, stream: int = 0):
        """the library's own cross-rank barrier on the stream (ranks = processes with one GPU each)"""
        self._check(self._lib.cvvp_median_shard_barrier(self._h, stream or None))

    def median_shard_unresolved(self, stream: int = 0) -> int:
        """elements the one-pass form (phases 4, 5) left undecided; waits for the stream"""
        v = C.c_longlong()
        self._check(self._lib.cvvp_median_shard_unresolved(self._h, stream or None, C.byref(v)))
        return int(v.value)

    def median_shard_export(self) -> bytes:
        buf = C.create_string_buffer(self.IPC_HANDLE_BYTES)
        self._check(self._lib.cvvp_median_shard_export(self._h, buf))
        return bytes(buf.raw)

    def median_shard_import(self, peer: int, handle: bytes):
        if len(handle) != self.IPC_HANDLE_BYTES:
            raise ValueError("an exported handle is 64 bytes")
        self._check(self._lib.cvvp_median_shard_import(self._h, peer, C.create_string_buffer(handle, len(handle))))

    def median_shard_attach(self, peer: int, peer_ctx: "Context"):
        self._check(self._lib.cvvp_median_shard_attach(self._h, peer, peer_ctx.handle))

    def median_shard_phase(self, phase: int, d_frames: int = 0, nframes: int = 0, frame_stride: int = 0, stream: int = 0):
        self._check(self._lib.cvvp_median_shard_phase(self._h, phase, d_frames or None, nframes, frame_stride, stream or None))

    def median_shard_result(self) -> int:
        p = C.c_void_p()
        self._check(self._lib.cvvp_median_shard_result(self._h, C.byref(p)))
        return int(p.value or 0)

    def median_shard_end(self):
        self._check(self._lib.cvvp_median_shard_end(self._h))

    # -- highlight ------------------------------------------------------------------------
    def highlight_begin(self, background: np.ndarray, struct_element: np.ndarray, threshold: int, threshold_lo: int,
                        threshold_hi: int, min_size_hyst: int, min_size_threshold: int, width_border: int = 0):
        bg = np.ascontiguousarray(background)
        se = np.ascontiguousarray(struct_element)
        channels = self.highlight_channels()
        if bg.dtype != np.uint8 or not (bg.ndim == 2 or (bg.ndim == 3 and bg.shape[2] == channels)) or \
                (bg.ndim == 2 and channels != 1):
            raise TypeError("background must be a uint8 array (H, W), or (H, W, C) with C the context's channels "
                            f"({channels})")
        if se.dtype != np.uint8 or se.ndim != 2:
            raise TypeError("struct_element must be a 2-D uint8 array (cv::morphologyEx asserts CV_8U)")
        h, w = bg.shape[:2]
        kh, kw = se.shape
        self._check(self._lib.cvvp_highlight_begin(self._h, bg.ctypes.data, w, h, se.ctypes.data, kw, kh, threshold,
                                                   threshold_lo, threshold_hi, min_size_hyst, min_size_threshold,
                                                   width_border))
        self._hl_shape = (h, w)
        # what one frame of the job is: (H, W), or (H, W, C) for a colour job (cvvp_highlight_set_channels)
        self._hl_frame = (h, w) if channels == 1 else (h, w, channels)
        # the job's component records (cvvp_highlight_set_component_stats)
        self._hl_dtype = self.COMPONENT_STATS_DTYPE if self.highlight_component_stats() else self.COMPONENT_DTYPE

    POLARITY_DARK, POLARITY_BRIGHT, POLARITY_BOTH = 0, 1, 2  # CVVP_POLARITY_*

    def highlight_set_polarity(self, polarity: int):
        """objects darker than the background (0, the default: d = max(bg - frame, 0)), brighter (1: max(frame - bg, 0))
        or both (2: |frame - bg|); a highlight job takes it when it begins, and none may be open"""
        self._check(self._lib.cvvp_highlight_set_polarity(self._h, polarity))

    def highlight_polarity(self) -> int:
        return int(self._lib.cvvp_highlight_polarity(self._h))

    def highlight_set_channels(self, channels: int):
        """channels (1..4) of the frames and backgrounds of the highlight jobs that begin after this; d is the largest
        per-channel difference of the polarity; none may be open"""
        self._check(self._lib.cvvp_highlight_set_channels(self._h, channels))

    def highlight_channels(self) -> int:
        return int(self._lib.cvvp_highlight_channels(self._h))

    def highlight_set_component_stats(self, on: bool):
        """shape and contrast statistics in every component record (COMPONENT_STATS_DTYPE) of the highlight jobs that
        begin after this; none may be open"""
        self._check(self._lib.cvvp_highlight_set_component_stats(self._h, int(on)))

    def highlight_component_stats(self) -> bool:
        rc = self._lib.cvvp_highlight_component_stats(self._h)
        if rc < 0:
            self._check(rc)
        return rc == 1

    def highlight_component_dtype(self) -> np.dtype:
        """the records of the open job's component outputs: COMPONENT_DTYPE, or COMPONENT_STATS_DTYPE with statistics"""
        return self._hl_dtype

    def highlight_frames(self, frames: np.ndarray) -> np.ndarray:
        """frames: uint8 (n, H, W) (a colour job: (n, H, W, C)) -> masks uint8 (n, H, W) of 0/255"""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8 or frames.shape[1:] != self._hl_frame:
            raise TypeError(f"frames must be uint8 of shape (n, {', '.join(map(str, self._hl_frame))}) matching the "
                            "background")
        n = frames.shape[0]
        npix = frames.shape[1] * frames.shape[2]
        out = np.empty(frames.shape[:3], np.uint8)
        self._check(self._lib.cvvp_highlight_frames(self._h, frames.ctypes.data, n, int(np.prod(self._hl_frame)),
                                                    out.ctypes.data, npix))
        return out

    # numpy view of struct cvvp_component (include/cvvp.h)
    COMPONENT_DTYPE = np.dtype([("x0", "<i4"), ("y0", "<i4"), ("x1", "<i4"), ("y1", "<i4"), ("area", "<i4"),
                                ("first_x", "<i4"), ("first_y", "<i4"), ("reserved", "<i4"), ("sum_x", "<i8"),
                                ("sum_y", "<i8")])
    # numpy view of struct cvvp_component_stats: the plain record, then the shape and contrast statistics
    COMPONENT_STATS_DTYPE = np.dtype([("c", COMPONENT_DTYPE), ("sum_xx", "<i8"), ("sum_xy", "<i8"), ("sum_yy", "<i8"),
                                      ("sum_d", "<i8"), ("sum_dx", "<i8"), ("sum_dy", "<i8"), ("min_d", "<i4"),
                                      ("max_d", "<i4")])

    def highlight_frames_cc(self, frames: np.ndarray, max_comps: int = 256, labels: bool = False):
        """frames uint8 (n, H, W) -> (masks, comps, ncomps[, labels]): the masks plus the 8-connected components of
        every mask (structured array (n, max_comps) of the job's component dtype, raster-first order) and, if asked, the int32
        label images (0 = background, k = component k of that frame)."""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8 or frames.shape[1:] != self._hl_frame:
            raise TypeError(f"frames must be uint8 of shape (n, {', '.join(map(str, self._hl_frame))}) matching the "
                            "background")
        n = frames.shape[0]
        npix = frames.shape[1] * frames.shape[2]
        out = np.empty(frames.shape[:3], np.uint8)
        comps = np.zeros((n, max_comps), self._hl_dtype)
        ncomps = np.zeros(n, np.int32)
        lab = np.empty(frames.shape[:3], np.int32) if labels else None
        self._check(self._lib.cvvp_highlight_frames_cc(self._h, frames.ctypes.data, n, int(np.prod(self._hl_frame)),
                                                       out.ctypes.data, npix,
                                                       comps.ctypes.data, max_comps, ncomps.ctypes.data,
                                                       lab.ctypes.data if labels else None, npix))
        return (out, comps, ncomps, lab) if labels else (out, comps, ncomps)

    # asynchronous ordered queue (cvvp_highlight_queue_*): the reference's bounded token queues on streams and events
    def highlight_queue_begin(self, depth: int, max_batch: int, fmt: FrameFormat | None = None, max_comps: int = 0):
        self._check(self._lib.cvvp_highlight_queue_begin(self._h, depth, max_batch, C.byref(fmt) if fmt is not None else None,
                                                         max_comps))
        self._hq = (max_batch, max_comps)

    def highlight_queue_pending(self) -> int:
        return int(self._lib.cvvp_highlight_queue_pending(self._h))

    def highlight_submit(self, frames: np.ndarray):
        """frames: uint8 (n, ...) -- prepared (n, H, W) frames, or decoded frames when the queue has a format"""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("frames must be uint8")
        n = frames.shape[0]
        stride = int(np.prod(frames.shape[1:]))
        self._check(self._lib.cvvp_highlight_submit(self._h, frames.ctypes.data, n, stride))

    def highlight_queue_ready(self) -> bool:
        rc = self._lib.cvvp_highlight_queue_ready(self._h)
        if rc < 0:
            self._check(rc)
        return rc == 1

    def highlight_next(self):
        """-> masks (n, H, W) of the oldest pending batch [, comps (n, max_comps), ncomps (n,)]"""
        max_batch, max_comps = self._hq
        h, w = self._hl_shape
        out = np.empty((max_batch, h, w), np.uint8)
        comps = np.zeros((max_batch, max_comps), self._hl_dtype) if max_comps else None
        ncomps = np.zeros(max_batch, np.int32) if max_comps else None
        n = C.c_longlong(0)
        self._check(self._lib.cvvp_highlight_next(self._h, out.ctypes.data, h * w, C.byref(n),
                                                  comps.ctypes.data if max_comps else None,
                                                  ncomps.ctypes.data if max_comps else None))
        k = int(n.value)
        return (out[:k], comps[:k], ncomps[:k]) if max_comps else out[:k]

    # zero-copy forms: the decoder writes into the slot's pinned input, the consumer reads the slot's pinned results
    def highlight_slot_acquire(self) -> np.ndarray:
        """-> uint8 view (max_batch, frame_pitch) of the next free slot's pinned input (frame i = row i)"""
        p, pitch, mx = C.c_void_p(), C.c_size_t(), C.c_longlong()
        self._check(self._lib.cvvp_highlight_slot_acquire(self._h, C.byref(p), C.byref(pitch), C.byref(mx)))
        buf = (C.c_uint8 * (int(mx.value) * int(pitch.value))).from_address(p.value)
        return np.frombuffer(buf, np.uint8).reshape(int(mx.value), int(pitch.value))

    def highlight_slot_commit(self, n: int):
        self._check(self._lib.cvvp_highlight_slot_commit(self._h, n))

    def highlight_next_view(self):
        """-> masks (n, H, W) view of the oldest batch's pinned results [, comps (n, max_comps), ncomps (n,)]; valid until
        highlight_view_release()"""
        max_batch, max_comps = self._hq
        h, w = self._hl_shape
        pm, pitch, n, pc, pn = C.c_void_p(), C.c_size_t(), C.c_longlong(), C.c_void_p(), C.c_void_p()
        self._check(self._lib.cvvp_highlight_next_view(self._h, C.byref(pm), C.byref(pitch), C.byref(n), C.byref(pc), C.byref(pn)))
        k, pt = int(n.value), int(pitch.value)
        buf = (C.c_uint8 * (k * pt)).from_address(pm.value)
        masks = np.frombuffer(buf, np.uint8).reshape(k, pt)[:, : h * w].reshape(k, h, w)
        if not max_comps:
            return masks
        cbuf = (C.c_uint8 * (k * max_comps * self._hl_dtype.itemsize)).from_address(pc.value)
        nbuf = (C.c_int32 * k).from_address(pn.value)
        return masks, np.frombuffer(cbuf, self._hl_dtype).reshape(k, max_comps), np.frombuffer(nbuf, np.int32)

    def highlight_view_release(self):
        self._check(self._lib.cvvp_highlight_view_release(self._h))

    def highlight_queue_end(self):
        self._check(self._lib.cvvp_highlight_queue_end(self._h))

    def highlight_device(self, d_frames: int, n: int, frame_stride: int, d_out: int, out_stride: int, stream: int = 0):
        self._check(self._lib.cvvp_highlight_device(self._h, d_frames, n, frame_stride, d_out, out_stride, stream or None))

    def highlight_device_bg(self, d_frames: int, n: int, frame_stride: int, d_backgrounds: int, bg_stride: int, d_out: int,
                            out_stride: int, d_comps: int = 0, max_comps: int = 0, d_ncomps: int = 0, d_labels: int = 0,
                            labels_stride: int = 0, stream: int = 0):
        """frame f against its own background at d_backgrounds + f * bg_stride (0: one background for all)"""
        self._check(self._lib.cvvp_highlight_device_bg(self._h, d_frames, n, frame_stride, d_backgrounds, bg_stride, d_out,
                                                       out_stride, d_comps or None, max_comps, d_ncomps or None,
                                                       d_labels or None, labels_stride, stream or None))

    # rolling-median background stream (cvvp_highlight_rolling_*): masks come back later than their frames go in
    def highlight_rolling_begin(self, window: int, max_batch: int, fmt: FrameFormat | None = None, max_comps: int = 0,
                                labels: bool = False):
        self._check(self._lib.cvvp_highlight_rolling_begin(self._h, window, max_batch,
                                                           C.byref(fmt) if fmt is not None else None, max_comps,
                                                           1 if labels else 0))
        self._hr = (max_batch, max_comps, bool(labels))

    def highlight_rolling_push(self, frames: np.ndarray):
        """frames: uint8 (n, ...) -- prepared (n, H, W) frames, or decoded frames when the stream has a format"""
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("frames must be uint8")
        self._check(self._lib.cvvp_highlight_rolling_push(self._h, frames.ctypes.data, frames.shape[0],
                                                          int(np.prod(frames.shape[1:]))))

    def highlight_rolling_close(self):
        self._check(self._lib.cvvp_highlight_rolling_close(self._h))

    def highlight_rolling_pending(self) -> int:
        return int(self._lib.cvvp_highlight_rolling_pending(self._h))

    def highlight_rolling_ready(self) -> bool:
        rc = self._lib.cvvp_highlight_rolling_ready(self._h)
        if rc < 0:
            self._check(rc)
        return rc == 1

    def highlight_rolling_next(self):
        """-> (first frame index, masks (n, H, W)[, comps (n, max_comps), ncomps (n,)[, labels (n, H, W)]]); n = 0 when
        nothing is pending"""
        max_batch, max_comps, labels = self._hr
        h, w = self._hl_shape
        out = np.empty((max_batch, h, w), np.uint8)
        comps = np.zeros((max_batch, max_comps), self._hl_dtype) if max_comps else None
        ncomps = np.zeros(max_batch, np.int32) if max_comps else None
        lab = np.zeros((max_batch, h, w), np.int32) if labels else None
        first, n = C.c_longlong(0), C.c_longlong(0)
        self._check(self._lib.cvvp_highlight_rolling_next(self._h, out.ctypes.data, h * w, max_batch, C.byref(first),
                                                          C.byref(n), comps.ctypes.data if max_comps else None,
                                                          ncomps.ctypes.data if max_comps else None,
                                                          lab.ctypes.data if labels else None, h * w))
        k = int(n.value)
        res = (int(first.value), out[:k])
        if max_comps:
            res += (comps[:k], ncomps[:k])
        if labels:
            res += (lab[:k],)
        return res

    def highlight_rolling_end(self):
        self._check(self._lib.cvvp_highlight_rolling_end(self._h))

    def highlight_set_path(self, path: int):
        """0 = fused kernel (default), 1 = per-pixel kernels (on-device cross-check)"""
        self._check(self._lib.cvvp_highlight_set_path(self._h, path))

    def highlight_frames_in_flight(self) -> int:
        v = C.c_int()
        self._check(self._lib.cvvp_highlight_frames_in_flight(self._h, C.byref(v)))
        return int(v.value)

    def highlight_end(self):
        self._check(self._lib.cvvp_highlight_end(self._h))

    # -- synthetic frames -----------------------------------------------------------------
    def synth_frames_device(self, d_frames: int, frame_stride: int, width: int, height: int, first_frame: int,
                            nframes: int, seed: int, ndisks: int, row0: int = 0, nrows: int | None = None,
                            stream: int = 0):
        if nrows is None:
            nrows = height - row0
        self._check(
            self._lib.cvvp_synth_frames_device(self._h, d_frames, frame_stride, width, height, row0, nrows, first_frame,
                                               nframes, seed, ndisks, stream or None)
        )
