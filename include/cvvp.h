/*
 * cvvp.h -- C ABI of libcvvp_cuda.so, the B200 (sm_100a) implementation of CvVidProc's
 * data-parallel hot path: the per-pixel temporal-median background model and the per-frame
 * highlight stage.
 *
 * Boundary rules
 *   - plain pointers and sizes only; no C++ types, no exceptions cross this boundary;
 *   - every function returns 0 on success or a negative cvvp_status; the text of the last
 *     failure of a context is available from cvvp_last_error(ctx) (ctx == NULL: the last
 *     failure of a call that had no context, thread-local);
 *   - the caller owns every host buffer; the library owns device memory, streams, events and
 *     pinned staging inside the opaque context; a context is bound to ONE CUDA device (one
 *     process per GPU, as torch.distributed launches them) and is not thread-safe;
 *   - there is no CPU fallback: every entry point fails with CVVP_ERR_CUDA if no sm_100 device
 *     is usable.
 *
 * Each entry point cites the reference interface (file:line under /root/reference) it replaces.
 */
#ifndef CVVP_H
#define CVVP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVVP_ABI_VERSION 3

#if defined(__GNUC__)
#define CVVP_API __attribute__((visibility("default")))
#else
#define CVVP_API
#endif

typedef enum cvvp_status {
    CVVP_OK = 0,
    CVVP_ERR_INVALID = -1, /* bad argument / call order                                   */
    CVVP_ERR_CUDA = -2,    /* CUDA runtime/driver failure (text in cvvp_last_error)       */
    CVVP_ERR_NOMEM = -3,   /* host or device allocation failed                            */
    CVVP_ERR_STATE = -4,   /* object is in the wrong state for this call                  */
    CVVP_ERR_UNSUPPORTED = -5
} cvvp_status;

typedef struct cvvp_ctx cvvp_ctx;

/* ---------------------------------------------------------------------------------------------
 * context
 * ------------------------------------------------------------------------------------------- */
CVVP_API int cvvp_abi_version(void);
/* device: CUDA ordinal, or -1 for the current device. */
CVVP_API int cvvp_ctx_create(int device, cvvp_ctx **out_ctx);
CVVP_API void cvvp_ctx_destroy(cvvp_ctx *ctx);
CVVP_API const char *cvvp_last_error(const cvvp_ctx *ctx);
/* block until all work queued on the context's streams is complete */
CVVP_API int cvvp_ctx_synchronize(cvvp_ctx *ctx);
/* the context's compute stream as a cudaStream_t (void* to keep CUDA types out of the ABI) */
CVVP_API void *cvvp_ctx_stream(cvvp_ctx *ctx);
CVVP_API int cvvp_ctx_device(const cvvp_ctx *ctx);
CVVP_API int cvvp_ctx_sm_count(const cvvp_ctx *ctx);

/* pinned (page-locked) host memory for callers that want zero-staging H2D/D2H.
 * Replaces nothing in the reference (its tokens are pageable cv::Mat); it is the "frames are
 * batched into pinned buffers" part of BASELINE.json:north_star. */
CVVP_API int cvvp_host_alloc(size_t bytes, void **out_ptr);
CVVP_API int cvvp_host_free(void *ptr);
/* The library parks the large buffers of a finished job -- the highlight queue's pinned slots and device buffers, the
 * fused highlight kernel's scratch -- for the next job of the same geometry in this process (page-locking a few
 * hundred MB costs more than highlighting a short clip): at most 3 GB of pinned and 24 GB of device memory.
 * cvvp_pool_trim releases everything that is parked and returns the bytes released.  Thread-safe. */
CVVP_API size_t cvvp_pool_trim(void);
/* synchronous device -> host copy on the context's compute stream (after everything queued there): lets callers
 * of the device-resident entry points fetch a result without a CUDA binding of their own */
CVVP_API int cvvp_ctx_copy_to_host(cvvp_ctx *ctx, void *host_dst, const void *device_src, size_t bytes);

/* ---------------------------------------------------------------------------------------------
 * temporal median -- replaces HistogramMedianAlgo<T>
 *   Sources/ProcessorAlgos/histogram_median_algo.h
 *     Insert :66-87 / ConsumeVector :116-141        -> cvvp_median_push
 *     NotifyNoMoreTokens :101-108 / MedianFromHistograms :144-193 / TryGetResult :90-98
 *                                                   -> cvvp_median_finish
 *   bin-width choice (cv_vid_bg_helpers.cpp:232-253) has no equivalent: the device path is an
 *   exact rank selection, i.e. the result the reference computes whenever its counters do not
 *   saturate, which GetVideoBackground's choice guarantees (SURVEY.md 8a a5).
 *
 * An "element" is one byte of a frame (rows*cols*channels of them, cv_util.cpp:251-254); the
 * median is taken per element over all pushed frames and is sorted[k(N, p)], the upper median
 * sorted[N/2] (histogram_median_algo.h:160-166) at the default (see cvvp_median_set_percentile).
 * ------------------------------------------------------------------------------------------- */

/* Percentile backgrounds.  Every background of a context -- the streaming job, the device-resident form, the
 * frame-sharded job and the rolling median -- is the per-element order statistic sorted[k(N, p)] of its N values
 * (N = Weff for a rolling window), with
 *     k(N, p) = min(N - 1, floor(N * p / 100))      (integer arithmetic, p an integer percent in [0, 100])
 * p = 50 (the default) gives N / 2, the reference's upper median; p = 0 the minimum, p = 100 the maximum.  A higher
 * percentile keeps dark objects that cover a pixel in a fraction c < p / 100 of the frames out of the background.
 * The percentile is a setting of the context: jobs take it when they begin (cvvp_median_begin -- and so push,
 * push_source and finish --, cvvp_median_shard_begin*, cvvp_highlight_rolling_begin); the device-resident forms
 * (cvvp_median_device, cvvp_median_rolling_device) read it at the call.  CVVP_ERR_INVALID for p outside [0, 100];
 * CVVP_ERR_STATE while a median, sharded or rolling job is open on the context.  Every rank of a sharded job must
 * use the same percentile: the host operators of this library set it on all their contexts, but ranks in other
 * processes are not checked for agreement. */
CVVP_API int cvvp_median_set_percentile(cvvp_ctx *ctx, int percent);
/* the context's percentile (50 unless set), or CVVP_ERR_INVALID for a NULL context */
CVVP_API int cvvp_median_percentile(const cvvp_ctx *ctx);

/* Start a median job on frames of `nelem` bytes.  nframes_hint > 0 sizes the device stack for exactly that many
 * frames (rounded up to 16; it grows by half if more are pushed, and the old and new stacks coexist while it does).
 * While they fit, the job keeps every pushed frame resident in device memory (frames x round_up(nelem, 128) bytes) and
 * selects the median on chip.  When the stack cannot be allocated or grown any further, the resident frames are folded
 * into per-element value histograms (256 x round_up(nelem, 128) x 4 bytes, 32-bit counts) and the stack is reused for
 * the frames that follow: from there on the job's memory is independent of the frame count, like the reference's
 * histograms (histogram_median_algo.h:123-126), and the result is the same sorted[k(N, p)] of ALL frames.
 * CVVP_ERR_NOMEM only when neither a stack of 16 frames nor the histograms fit. */
CVVP_API int cvvp_median_begin(cvvp_ctx *ctx, size_t nelem, long long nframes_hint);
/* Append n frames from HOST memory; frame i starts at frames + i*frame_stride and holds nelem
 * contiguous bytes.  The copy is asynchronous when `frames` is pinned (cvvp_host_alloc or
 * cudaHostRegister'ed); the buffer must then stay valid until cvvp_median_finish or
 * cvvp_ctx_synchronize returns.  Pageable memory is staged through the context's pinned ring
 * and may be reused as soon as the call returns. */
CVVP_API int cvvp_median_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride);
/* Number of frames pushed so far. */
CVVP_API long long cvvp_median_count(const cvvp_ctx *ctx);
/* The running job's device stack (frame f at *d_frames + f * *frame_stride), for callers that run a device-resident
 * form on the pushed frames -- a rank of a frame-sharded job uploads its chunk with cvvp_median_push and hands this
 * pointer to cvvp_median_shard_phase.  Orders every push made so far before work queued on the compute stream
 * afterwards; the pointer is valid until the next push (the stack may move when it grows) or the end of the job. */
CVVP_API int cvvp_median_stack_device(cvvp_ctx *ctx, const uint8_t **d_frames, size_t *frame_stride, long long *nframes);
/* Run the select over everything pushed and copy the nelem result bytes to HOST memory `out`
 * (synchronous: the result is valid on return).  Ends the job. */
CVVP_API int cvvp_median_finish(cvvp_ctx *ctx, uint8_t *out);
/* Drop a job without computing. */
CVVP_API int cvvp_median_abort(cvvp_ctx *ctx);

/* Device-resident form: d_frames is a DEVICE pointer to nframes frames, frame f at
 * d_frames + f*frame_stride (frame_stride % 16 == 0 and d_frames 16-byte aligned, the TMA
 * tensor-map constraints), d_out a DEVICE pointer to nelem bytes (4-byte aligned).  Runs on
 * `stream` (a cudaStream_t, NULL = the context's compute stream) and does not synchronize: frames
 * written on ANOTHER stream must be complete (or ordered by an event) before the call.
 * Up to 1280 frames (1024 when frame_stride exceeds 2.5 MiB) the select happens on chip in one pass
 * over the frames; longer stacks (up to 16 x 65535 = 1048560 frames; more fails with
 * CVVP_ERR_UNSUPPORTED) are counted in chunks of at most 1024 frames: one pass of window counting around per-chunk pilot medians, and -- only if that leaves an
 * element undecided, checked on the device -- two passes of nibble counting, 16-bit counts per
 * 65535 frames summed in 32 bits: the reference's analogue of widening its histogram bins with the
 * frame count (cv_vid_bg_helpers.cpp:232-253). */
CVVP_API int cvvp_median_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem,
                       size_t frame_stride, uint8_t *d_out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * rolling temporal median -- a background that follows the video.  The reference has one static background per
 *   TrackObjects call (Sources/cv_vid_objecttrack_helpers.cpp:167-175, the pack's background); here frame t of a
 *   stream of N frames gets sorted[k(Weff, p)] (Weff = min(W, N)), the upper median sorted[Weff/2]
 *   (histogram_median_algo.h:160-166) at the default, of a window of W frames centred on it and shifted, not
 *   shortened, at both ends:
 *     N <= W : every window is all N frames
 *     N >  W : window of frame t = frames s(t) .. s(t) + W - 1, s(t) = min(max(t - W/2, 0), N - W)
 * Device-resident form, layout as cvvp_median_device (frame f at d_frames + f*frame_stride, nelem bytes each, any
 * nelem: colour stacks work element by element): writes the backgrounds of frames t in [t0, t1) to
 * d_out + (t - t0)*out_stride.  Exact for every window (16-bit counts per element and value, 1 <= window <= 65535).
 * Runs on `stream` (NULL = the context's compute stream) and does not synchronize.  CVVP_ERR_INVALID for window < 1 or
 * > 65535, nframes < 1, t0 / t1 outside 0 <= t0 <= t1 <= nframes, a stride shorter than nelem or a NULL pointer.
 * ------------------------------------------------------------------------------------------- */
CVVP_API int cvvp_median_rolling_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem,
                                        size_t frame_stride, int window, long long t0, long long t1, uint8_t *d_out,
                                        size_t out_stride, void *stream);

/* ---------------------------------------------------------------------------------------------
 * frame-sharded temporal median across GPUs (one process -- or at least one context -- per GPU).
 *   The reference splits the frame range of a video over its generator threads
 *   (Sources/cv_vid_bg_helpers.cpp:84-120) and merges them in ONE order-independent histogram
 *   (histogram_median_algo.h:116-141); here every rank keeps a chunk of the frames in its own HBM
 *   and the merge is a two-round exchange of 16-bin nibble counts written directly into the
 *   owner rank's memory over NVLink (csrc/median_shard.cu).  The result is the same sorted[k(N, p)]
 *   of ALL ranks' frames, the upper median sorted[N/2] (:160-166) at the default, delivered to every rank.
 *
 *   call order on every rank:
 *     cvvp_median_shard_begin
 *     cvvp_median_shard_export -> (the host exchanges the 64-byte handles, e.g. torch.distributed
 *                                  all_gather) -> cvvp_median_shard_import for every other rank
 *                                  (or cvvp_median_shard_attach for a context of the same process)
 *     per job: phase 0, BARRIER, phase 1, BARRIER, phase 2, BARRIER, phase 3, BARRIER
 *     cvvp_median_shard_result ; cvvp_median_shard_end
 *   BARRIER = a cross-rank barrier ordered on the stream (e.g. a one-element NCCL all-reduce):
 *   phase p+1 of any rank must not start before phase p of every rank has completed.  No kernel
 *   of this library waits for another rank.
 *
 *   One-pass form (reads every frame once instead of twice; try it first):
 *     per job: phase 4, BARRIER, phase 5, BARRIER, cvvp_median_shard_unresolved
 *   Phase 4 counts each rank's frames in an 8-value window around a pilot median the kernel picks
 *   on chip from 256 of its own frames (per launch of <= 1024 frames), phase 5 lets the owner name
 *   the median of ALL frames wherever it lies inside every window.  The result is exact where it
 *   is given; cvvp_median_shard_unresolved returns how many elements could NOT be decided (the
 *   same number on every rank; 0 for an ordinary video).  When it is not 0 run
 *     phase 10, BARRIER, phase 11, BARRIER, phase 12, BARRIER, phase 13, BARRIER
 *   = phases 0..3 restricted to the 128-element tiles that hold an undecided element (phase 5
 *   flagged them on every rank), or phases 0..3 themselves, which rewrite the whole image.
 * ------------------------------------------------------------------------------------------- */
#define CVVP_IPC_HANDLE_BYTES 64
/* rank in [0, world), world <= 16; allocates this rank's exchange buffers (64 B per element and
 * rank for the counts + 5 B per element) */
CVVP_API int cvvp_median_shard_begin(cvvp_ctx *ctx, size_t nelem, int rank, int world);
/* same, for ranks that hold up to max_rank_frames frames each: room for one window record per 1024 frames
 * (phase 4) and one 16-bit count vector per 65535 frames (phases 0 / 2).  cvvp_median_shard_begin is this call with
 * max_rank_frames = 1024 for the window records and 65535 for the counts. */
CVVP_API int cvvp_median_shard_begin_frames(cvvp_ctx *ctx, size_t nelem, int rank, int world, long long max_rank_frames);
/* CVVP_IPC_HANDLE_BYTES bytes that let another PROCESS on the same box map this rank's buffers */
CVVP_API int cvvp_median_shard_export(cvvp_ctx *ctx, void *handle_out);
CVVP_API int cvvp_median_shard_import(cvvp_ctx *ctx, int peer_rank, const void *handle);
/* same-process peer (several contexts in one process, on one or several devices) */
CVVP_API int cvvp_median_shard_attach(cvvp_ctx *ctx, int peer_rank, cvvp_ctx *peer_ctx);
/* phases 0, 2, 4, 10 and 12 read this rank's frames (device pointer, same layout rules as cvvp_median_device;
 * nframes may be 0, may differ between ranks, at most what the job was begun for); phases 1, 3, 5, 11 and 13 ignore
 * the frame arguments.
 * Runs on `stream` (NULL = the context's compute stream) and does not synchronize. */
CVVP_API int cvvp_median_shard_phase(cvvp_ctx *ctx, int phase, const uint8_t *d_frames, long long nframes,
                                     size_t frame_stride, void *stream);
/* A BARRIER of the library's own, for ranks that are processes with ONE GPU EACH (what torchrun launches): a one-warp
 * kernel on `stream` that signals every peer through its mapped exchange buffer and waits for every peer's signal
 * (a few microseconds; a one-element NCCL all-reduce costs 15-25).  Every rank must call it the same number of
 * times.  Not for ranks that share a device (CVVP_ERR_UNSUPPORTED for attached ranks; processes that share a GPU must
 * not call it: the waiting kernel would keep the peer's kernel from running) -- those use a host-side barrier.  A
 * wait of more than 2 s traps (the stream reports a CUDA error) instead of hanging. */
CVVP_API int cvvp_median_shard_barrier(cvvp_ctx *ctx, void *stream);
/* after the barrier that follows phase 5: waits for `stream` (NULL = the context's compute stream) and returns the
 * number of elements the one-pass form left undecided, summed over all owners (identical on every rank) */
CVVP_API int cvvp_median_shard_unresolved(cvvp_ctx *ctx, void *stream, long long *out_elements);
/* device pointer to the nelem result bytes (complete on every rank after the barrier that follows phase 3 / 5) */
CVVP_API int cvvp_median_shard_result(cvvp_ctx *ctx, const uint8_t **d_result);
CVVP_API int cvvp_median_shard_end(cvvp_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * per-frame highlight -- replaces HighlightObjectsAlgo
 *   Sources/ProcessorAlgos/highlight_objects_algo.h
 *     TokenProcessorPack<HighlightObjectsAlgo> :21-32   -> cvvp_highlight_begin (parameters, moved in once)
 *     Insert :60-69 / TryGetResult :72-79               -> cvvp_highlight_frames (batch of tokens in, masks out,
 *                                                          same order; the reference mutates each token in place)
 *   Sources/ProcessorAlgos/highlight_objects_algo.cpp
 *     HighlightObjects :17-78 and its helpers :81-221   -> the device kernels (csrc/highlight.cu)
 *
 * Frames and the background are 8-bit single channel, width*height contiguous bytes (findContours requires
 * 8UC1).  Output masks are 0 / 255.  The structuring element is kh x kw bytes, any non-zero entry is set
 * (cv::morphologyEx asserts CV_8U), anchor (kw/2, kh/2).  threshold == -1 selects Otsu (:89-95).
 * width_border is accepted and ignored, like the reference (:68-71).
 * ------------------------------------------------------------------------------------------- */
CVVP_API int cvvp_highlight_begin(cvvp_ctx *ctx, const uint8_t *background, int width, int height,
                                  const uint8_t *struct_element, int kw, int kh, int threshold, int threshold_lo,
                                  int threshold_hi, int min_size_hyst, int min_size_threshold, int width_border);
/* n frames from HOST memory (frame i at frames + i*frame_stride) -> n masks in HOST memory (mask i at
 * masks_out + i*out_stride); synchronous; H2D, kernels and D2H of consecutive chunks overlap internally.
 * masks_out may alias frames (in-place, like the reference's tokens) when the strides are equal. */
CVVP_API int cvvp_highlight_frames(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride,
                                   uint8_t *masks_out, size_t out_stride);
/* device-resident form; runs on `stream` (NULL = the context's compute stream), does not synchronize */
CVVP_API int cvvp_highlight_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride,
                                   uint8_t *d_out, size_t out_stride, void *stream);
CVVP_API int cvvp_highlight_end(cvvp_ctx *ctx);

/* Object polarity: which sign of (frame - background) counts as an object.  Every mask starts from the difference
 * image d of a frame and its background; the reference computes d = saturate_u8(background - frame) (:27-29), which
 * finds objects DARKER than the background.  The polarity chooses d:
 *     CVVP_POLARITY_DARK   (0, the default)  d = max(bg - frame, 0)   the reference (:27-29)
 *     CVVP_POLARITY_BRIGHT (1)               d = max(frame - bg, 0)   objects brighter than the background
 *     CVVP_POLARITY_BOTH   (2)               d = |frame - bg|         cv::absdiff, commented out at :30
 * Everything after d (thresholds, Otsu, opening, hysteresis, small-object removal, hole filling, components) is
 * unchanged.  The polarity is a setting of the context (no counterpart in the reference): a highlight job takes it in
 * cvvp_highlight_begin, and every call of that job (frames / device forms, the queue, the rolling stream) uses it.
 * CVVP_ERR_INVALID for a value outside {0, 1, 2} or a NULL context; CVVP_ERR_STATE while a highlight job is open on
 * the context (between cvvp_highlight_begin and cvvp_highlight_end). */
#define CVVP_POLARITY_DARK 0   /* max(bg - frame, 0): the reference (default) */
#define CVVP_POLARITY_BRIGHT 1 /* max(frame - bg, 0) */
#define CVVP_POLARITY_BOTH 2   /* |frame - bg| (cv::absdiff) */
CVVP_API int cvvp_highlight_set_polarity(cvvp_ctx *ctx, int polarity);
/* the context's polarity (CVVP_POLARITY_DARK unless set), or CVVP_ERR_INVALID for a NULL context */
CVVP_API int cvvp_highlight_polarity(const cvvp_ctx *ctx);

/* Colour frames (no counterpart in the reference, whose highlight stage takes 8UC1 frames only).  A job of C channels
 * (1..4) takes frames and backgrounds of width*height*C interleaved bytes, and its difference image is the largest
 * per-channel difference of the polarity:
 *     d(x, y) = max over c of d_c,   d_c = the polarity's d of channel c of the background and of the frame
 * so the thresholds stay grey levels of one channel.  Everything after d is unchanged, and C = 1 is the grey job.
 * The channel count is a setting of the context, like the polarity: a highlight job takes it in cvvp_highlight_begin.
 * With C > 1:
 *   - the background of cvvp_highlight_begin is width*height*C bytes;
 *   - frames of cvvp_highlight_frames*, cvvp_highlight_device*, of the queue and of the rolling stream without a frame
 *     format are width*height*C bytes each, and every frame stride (and cvvp_highlight_device_bg's backgrounds and
 *     bg_stride) is at least that;
 *   - a frame format of the queue or of the rolling stream must be CVVP_FRAMES_AS_IS with src_channels == C
 *     (CVVP_ERR_INVALID otherwise);
 *   - the slots of cvvp_highlight_slot_acquire hold width*height*C bytes per frame (without a frame format);
 *   - the device forms return CVVP_ERR_INVALID when d_out overlaps the frames or the backgrounds (d is computed
 *     ahead of the masks, in chunks);
 *   - masks, components, labels and records are unchanged: one byte (0 / 255) per pixel, and the statistics' d is
 *     the d above.
 * set: CVVP_ERR_INVALID outside 1..4 or for a NULL context, CVVP_ERR_STATE while a highlight job is open on the
 * context.  get: the context's channel count (1 unless set), or CVVP_ERR_INVALID for a NULL context. */
CVVP_API int cvvp_highlight_set_channels(cvvp_ctx *ctx, int channels);
CVVP_API int cvvp_highlight_channels(const cvvp_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * components of the highlight masks (opt-in) -- the connected-component labelling that feeds the
 * object tracker.  In the reference this happens on the host inside the user's tracker callback,
 * which receives only bw_frame (Sources/ProcessorAlgos/assign_objects_algo.h:124-130) and
 * typically calls cv2.connectedComponentsWithStats(bw_frame, connectivity=8) (cf. the note at
 * highlight_objects_algo.cpp:152-153).  Here the fused kernel labels the final mask once more and
 * returns, per frame, its 8-connected components numbered 1.. in the raster order of their first
 * pixels (the canonical labelling: the same label SETS as OpenCV's, whose numbering depends on
 * its scan), with the statistics a tracker needs.
 * ------------------------------------------------------------------------------------------- */
typedef struct cvvp_component {
    int32_t x0, y0, x1, y1;   /* bounding box, inclusive */
    int32_t area;             /* pixels */
    int32_t first_x, first_y; /* raster-first pixel */
    int32_t reserved;
    int64_t sum_x, sum_y;     /* coordinate sums: centroid = (sum_x / area, sum_y / area) */
} cvvp_component;
/* Like cvvp_highlight_device, plus: d_comps[f * max_comps + k] = component k + 1 of frame f (the first
 * min(ncomps, max_comps) of them), d_ncomps[f] = number of components of frame f (may exceed max_comps),
 * d_labels (may be NULL) = int32 label image of frame f at d_labels + f * labels_stride elements
 * (0 = background).  All DEVICE pointers.  n <= 2^20 frames per call. */
CVVP_API int cvvp_highlight_device_cc(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride,
                                      uint8_t *d_out, size_t out_stride, cvvp_component *d_comps, int max_comps,
                                      int *d_ncomps, int32_t *d_labels, size_t labels_stride, void *stream);
/* Like cvvp_highlight_device_cc, but frame f is compared with its OWN background at d_backgrounds + f * bg_stride
 * (DEVICE pointer; bg_stride = 0: the one image at d_backgrounds for every frame; else bg_stride >= width*height).
 * The background given to cvvp_highlight_begin only sets the geometry here.  d_comps / d_ncomps / d_labels NULL =
 * no components (then max_comps is ignored); with components, fused path only, like cvvp_highlight_device_cc. */
CVVP_API int cvvp_highlight_device_bg(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride,
                                      const uint8_t *d_backgrounds, size_t bg_stride, uint8_t *d_out, size_t out_stride,
                                      cvvp_component *d_comps, int max_comps, int *d_ncomps, int32_t *d_labels,
                                      size_t labels_stride, void *stream);
/* HOST-buffer form (synchronous): masks, components, counts and (optionally, NULL = off) label images */
CVVP_API int cvvp_highlight_frames_cc(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride,
                                      uint8_t *masks_out, size_t out_stride, cvvp_component *comps_out, int max_comps,
                                      int *ncomps_out, int32_t *labels_out, size_t labels_stride);
/* Shape and contrast statistics of the components (opt-in; no counterpart in the reference).  Over the pixels (x, y)
 * of a component, with d the job's difference image (the polarity's d of the frame and its own background, the d
 * the thresholds saw):
 *     sum_xx, sum_xy, sum_yy   sum of x*x, x*y, y*y: the raw moments m20, m11, m02 of cv::moments(component mask,
 *                              binaryImage=true); central moments and the ellipse follow from them and c's sums
 *     sum_d                    contrast mass: sum of d (0 is possible: hole filling and the FillHoles all-255 quirk
 *                              put pixels with d = 0 into masks)
 *     sum_dx, sum_dy           sum of d*x, d*y: contrast-weighted centroid (sum_dx / sum_d, sum_dy / sum_d)
 *     min_d, max_d             smallest and largest d
 * All values are exact integers.  The setting belongs to the context, like the polarity: a highlight job takes it in
 * cvvp_highlight_begin.  While a job has it on, EVERY cvvp_component * output of that job (cvvp_highlight_device_cc,
 * _device_bg, _frames_cc, cvvp_highlight_next, cvvp_highlight_next_view, cvvp_highlight_rolling_next) points to an
 * array of cvvp_component_stats, and max_comps counts those records; pass (cvvp_component *)stats (c is the first
 * member).  The statistics read the frames and backgrounds after the masks are written, so with statistics on the
 * device forms return CVVP_ERR_INVALID when d_out overlaps the frames or the backgrounds (no in-place output).
 * set: 0 = off (default) or 1 = on; CVVP_ERR_INVALID for another value or a NULL context, CVVP_ERR_STATE while a
 * highlight job is open on the context.  get: the context's setting, or CVVP_ERR_INVALID for a NULL context. */
typedef struct cvvp_component_stats {
    cvvp_component c;               /* exactly what the plain form returns */
    int64_t sum_xx, sum_xy, sum_yy; /* second-order raw moments (cv::moments m20, m11, m02) */
    int64_t sum_d, sum_dx, sum_dy;  /* contrast mass and contrast-weighted coordinate sums */
    int32_t min_d, max_d;
} cvvp_component_stats; /* 104 bytes */
CVVP_API int cvvp_highlight_set_component_stats(cvvp_ctx *ctx, int on);
CVVP_API int cvvp_highlight_component_stats(const cvvp_ctx *ctx);
/* Device implementation used by the calls above (after cvvp_highlight_begin; both give identical masks):
 *   0 = fused (default): one persistent-CTA kernel launch per batch, run-based labelling (csrc/highlight_fused.cu)
 *   1 = per-pixel kernels (csrc/highlight.cu), ~35 launches per batch; kept as an on-device cross-check.
 * Has no counterpart in the reference; it exists so that tests can hold the two device paths to each other at sizes
 * where the CPU oracle is slow. */
CVVP_API int cvvp_highlight_set_path(cvvp_ctx *ctx, int path);
/* Frames the fused kernel keeps in flight on this device (= resident CTAs; one scratch slot each). */
CVVP_API int cvvp_highlight_frames_in_flight(cvvp_ctx *ctx, int *out_frames);

/* ---------------------------------------------------------------------------------------------
 * frame source on the device -- replaces the per-frame host work of CvVidFramesGeneratorAlgo::GetTokenSet
 *   Sources/ProcessorTokenHandlers/cv_vid_frames_generator_algo.h
 *     frame = frame(crop_rectangle) :141; cv::extractChannel(frame, 0) :149-151 (vid_is_grayscale);
 *     cv::cvtColor(COLOR_RGB2GRAY) :152-154 (convert_to_grayscale); the frame as is :155-156
 * Decoded frames are src_height x src_width x src_channels interleaved bytes (what cv::VideoCapture hands
 * out).  The crop rectangle is the RESOLVED one (GetCroppedFrameDims, Sources/cv_vid_bg_helpers.cpp:39-60, is
 * host logic and stays with the caller).  Output frames are crop_height x crop_width x (1 | src_channels)
 * contiguous bytes.  RGB2GRAY is OpenCV's 8-bit fixed point, y = (c0*9798 + c1*19235 + c2*3735 + 16384) >> 15
 * with c0 the FIRST channel in memory (the reference converts whatever order the decoder produced), a fourth
 * channel is ignored.
 * ------------------------------------------------------------------------------------------- */
#define CVVP_FRAMES_AS_IS 0    /* crop only; output keeps src_channels */
#define CVVP_FRAMES_CHANNEL0 1 /* crop + cv::extractChannel(frame, 0) */
#define CVVP_FRAMES_RGB2GRAY 2 /* crop + cv::cvtColor(frame, COLOR_RGB2GRAY); src_channels 3 or 4 */
typedef struct cvvp_frame_format {
    int32_t src_width, src_height, src_channels;
    int32_t crop_x, crop_y, crop_width, crop_height;
    int32_t mode;
} cvvp_frame_format;
/* bytes of one prepared frame (0 if fmt is NULL) */
CVVP_API size_t cvvp_frame_format_out_bytes(const cvvp_frame_format *fmt);
/* device-resident form: n decoded frames at d_src + i*src_stride -> prepared frames at d_dst + i*dst_stride;
 * runs on `stream` (NULL = the context's compute stream), does not synchronize */
CVVP_API int cvvp_frames_prepare_device(cvvp_ctx *ctx, const uint8_t *d_src, long long n, size_t src_stride,
                                        const cvvp_frame_format *fmt, uint8_t *d_dst, size_t dst_stride, void *stream);
/* HOST-buffer form (synchronous): only the crop's rows of every frame cross the link */
CVVP_API int cvvp_frames_prepare(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride,
                                 const cvvp_frame_format *fmt, uint8_t *out, size_t out_stride);
/* cvvp_median_push for DECODED frames: the crop's rows are uploaded and one kernel crops / reduces them straight
 * into the device frame stack (the job's nelem must equal cvvp_frame_format_out_bytes(fmt)).  `frames` may be
 * reused when the call returns. */
CVVP_API int cvvp_median_push_source(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride,
                                     const cvvp_frame_format *fmt);

/* ---------------------------------------------------------------------------------------------
 * highlight, asynchronous ordered form -- replaces the token queues around HighlightObjectsAlgo
 *   Sources/AsyncTokens/token_queue.h:209-214 (bounded by token_storage_limit),
 *   Sources/AsyncTokens/token_processing_unit.h:293-307 (Insert / TryGetResult from a worker thread),
 *   Sources/ProcessorTokenHandlers/mat_set_intermediary.h:50-68,84-114 (results handed on in frame order)
 * rebuilt on CUDA streams and events: a ring of `depth` batch slots, each with pinned input / output staging;
 * submit copies the caller's frames into the slot (the caller's buffer is free on return, like a moved token),
 * queues H2D -> [frame preparation] -> highlight kernel -> D2H on three streams and returns; batches complete
 * and are returned strictly in submission order.  The host is free to decode the next batch and run the tracker
 * on the previous one meanwhile.
 *   cvvp_highlight_begin ... cvvp_highlight_queue_begin, { submit | next }*, cvvp_highlight_queue_end
 * ------------------------------------------------------------------------------------------- */
/* depth >= 1 batches in flight, each of at most max_batch frames.  fmt != NULL: submitted frames are DECODED
 * frames prepared on the device (the prepared geometry must be the background's, one channel); NULL: frames are
 * already width*height bytes.  max_comps > 0 additionally returns the components of every mask (see below). */
CVVP_API int cvvp_highlight_queue_begin(cvvp_ctx *ctx, int depth, long long max_batch, const cvvp_frame_format *fmt,
                                        int max_comps);
/* batches submitted and not yet returned by cvvp_highlight_next */
CVVP_API int cvvp_highlight_queue_pending(const cvvp_ctx *ctx);
/* 1 <= n <= max_batch frames.  CVVP_ERR_STATE when `depth` batches are pending (back-pressure: call
 * cvvp_highlight_next first). */
CVVP_API int cvvp_highlight_submit(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride);
/* 1 if the oldest pending batch is complete, 0 if not (or nothing is pending); never blocks */
CVVP_API int cvvp_highlight_queue_ready(cvvp_ctx *ctx);
/* Wait for the oldest pending batch; copy its *n_out masks to masks_out (mask i at masks_out + i*out_stride) and,
 * when the queue was begun with max_comps > 0 and the pointers are not NULL, its components
 * (comps_out[i*max_comps + k]) and counts (ncomps_out[i]).  The buffers must have room for max_batch frames (the
 * batch's size is only known on return).  CVVP_ERR_STATE when nothing is pending. */
CVVP_API int cvvp_highlight_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long *n_out,
                                 cvvp_component *comps_out, int *ncomps_out);
/* Zero-copy forms of submit / next -- the "frames are batched into pinned buffers" of BASELINE.json:north_star.  The
 * reference's generator fills a token that then moves through the queues without being copied
 * (Sources/AsyncTokens/token_batch_generator.h:52-67, token_queue.h:60-97); here the token's storage IS the slot:
 *   cvvp_highlight_slot_acquire  hands out the pinned input of the next free slot: the caller (a video decoder) writes
 *                                up to *max_frames whole frames into it, frame i at *h_frames + i * *frame_pitch
 *                                (decoded frames when the queue has a frame format, prepared frames otherwise).
 *                                Several slots may be out at once (a decoder working ahead); CVVP_ERR_STATE when
 *                                `depth` batches are pending or being filled;
 *   cvvp_highlight_slot_commit   queues the n frames written to the OLDEST acquired slot (slots are committed in the
 *                                order they were acquired).  n = 0 hands it back unused -- the end of the stream: slots
 *                                acquired after it can then only be handed back as well;
 *   cvvp_highlight_next_view     waits for the oldest pending batch and lends out its pinned results: mask i at
 *                                *h_masks + i * *mask_pitch, components at (*comps)[i * max_comps + k], counts
 *                                (*ncomps)[i] (NULL when the queue was begun with max_comps = 0);
 *   cvvp_highlight_view_release  gives the batch's slot back to the ring.
 * The pointers are valid until the matching commit / release.  submit / next (copying forms) may be mixed in. */
CVVP_API int cvvp_highlight_slot_acquire(cvvp_ctx *ctx, uint8_t **h_frames, size_t *frame_pitch, long long *max_frames);
CVVP_API int cvvp_highlight_slot_commit(cvvp_ctx *ctx, long long n);
CVVP_API int cvvp_highlight_next_view(cvvp_ctx *ctx, const uint8_t **h_masks, size_t *mask_pitch, long long *n_out,
                                      const cvvp_component **comps, const int **ncomps);
CVVP_API int cvvp_highlight_view_release(cvvp_ctx *ctx);
/* drains and frees the ring (pending results are dropped) */
CVVP_API int cvvp_highlight_queue_end(cvvp_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * highlight against a rolling median background, ordered stream -- TrackObjects with a background that follows the
 *   video (see cvvp_median_rolling_device for the windows).  The mask of frame t is HighlightObjects(f_t) (highlight_
 *   objects_algo.cpp:17-78) with B_t, the rolling percentile of its window, in place of the pack's background.  Masks come
 *   back LATER than their frames go in: frame t needs W - 1 frames ahead at the start of the stream and
 *   ceil(W/2) - 1 afterwards; the last ones are computed when the stream is closed (the frame count is only known
 *   then), with windows clamped to the frames pushed.  The device keeps a ring of (W + max_batch) prepared frames of
 *   round_up(width*height, 128) bytes.
 *   cvvp_highlight_begin ... cvvp_highlight_rolling_begin, { push | next }*, close, next*, cvvp_highlight_rolling_end
 * ------------------------------------------------------------------------------------------- */
/* 1 <= window <= 65535, 1 <= max_batch <= 2^20 frames per push.  fmt != NULL: pushed frames are DECODED frames
 * prepared on the device (prepared geometry = the background's, one channel); NULL: frames of width*height bytes.
 * max_comps > 0 also returns the components of every mask; labels != 0 (needs max_comps > 0) also the label images.
 * CVVP_ERR_NOMEM naming the window when the ring does not fit. */
CVVP_API int cvvp_highlight_rolling_begin(cvvp_ctx *ctx, int window, long long max_batch, const cvvp_frame_format *fmt,
                                          int max_comps, int labels);
/* n frames from HOST memory (may be reused on return); queues the backgrounds, masks and downloads of every frame whose
 * window is now complete, in chunks of at most max_batch frames */
CVVP_API int cvvp_highlight_rolling_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride);
/* end of the stream: queues the remaining frames; no push after it */
CVVP_API int cvvp_highlight_rolling_close(cvvp_ctx *ctx);
/* result chunks queued and not yet returned by cvvp_highlight_rolling_next */
CVVP_API int cvvp_highlight_rolling_pending(const cvvp_ctx *ctx);
/* 1 if the oldest pending chunk is complete, 0 if not (or nothing is pending); never blocks */
CVVP_API int cvvp_highlight_rolling_ready(cvvp_ctx *ctx);
/* Waits for the oldest pending chunk and copies its *n_out (<= max_n, at most max_batch) masks of frames
 * *first_index, *first_index + 1, ... to masks_out (mask i at masks_out + i*out_stride) and, when begun with them and
 * the pointers are not NULL, components (comps_out[i*max_comps + k]), counts and label images (labels_out +
 * i*labels_stride elements).  *n_out = 0 when nothing is pending. */
CVVP_API int cvvp_highlight_rolling_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long max_n,
                                         long long *first_index, long long *n_out, cvvp_component *comps_out,
                                         int *ncomps_out, int32_t *labels_out, size_t labels_stride);
/* drains and frees the stream (pending results are dropped) */
CVVP_API int cvvp_highlight_rolling_end(cvvp_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * synthetic input (SURVEY.md 8d): deterministic integer-hash frames generated directly in
 * device memory, bit-identical to cvvidproc_b200/synth.py on the host.
 * frames first_frame .. first_frame+nframes-1 of the stream (seed, K disks) are written to
 * d_frames + i*frame_stride, rows [row0, row0+nrows) of each (a row band for row-sharded jobs).
 * ------------------------------------------------------------------------------------------- */
CVVP_API int cvvp_synth_frames_device(cvvp_ctx *ctx, uint8_t *d_frames, size_t frame_stride, int width,
                             int height, int row0, int nrows, long long first_frame,
                             long long nframes, uint32_t seed, int ndisks, void *stream);

/* ---------------------------------------------------------------------------------------------
 * timing of the last median kernel (CUDA events on the launching stream), for the
 * print_timing_report equivalent (Sources/AsyncTokens/async_token_process.h:273-414).
 * ------------------------------------------------------------------------------------------- */
CVVP_API int cvvp_median_last_kernel_ms(cvvp_ctx *ctx, float *out_ms);
/* how many kernels of this library the context has launched so far */
CVVP_API long long cvvp_ctx_launch_count(const cvvp_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* CVVP_H */
