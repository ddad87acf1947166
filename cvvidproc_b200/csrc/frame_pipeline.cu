// Host side of the frame path between the decoder and the two operators: upload of decoded frames with the device
// frame preparation (frames.cu), and the asynchronous, ordered highlight queue.
//
// What it replaces in the reference:
//   * the generator's per-frame crop / channel reduction
//     (Sources/ProcessorTokenHandlers/cv_vid_frames_generator_algo.h:140-156) -- now a kernel after the upload;
//   * the bounded token queues and worker hand-off around HighlightObjectsAlgo
//     (Sources/AsyncTokens/token_queue.h:209-214, token_processing_unit.h:293-307) and the in-order hand-over of
//     MatSetIntermediary (ProcessorTokenHandlers/mat_set_intermediary.h:50-68) -- now a ring of batch slots whose
//     H2D, kernels and D2H are ordered by CUDA events on three streams; batches complete in submission order.
#include "context.hpp"
#include "pool.hpp"

#include <cstring>
#include <new>
#include <vector>

namespace cvvp
{
namespace
{
constexpr size_t kRawChunkBytes = size_t(64) << 20; // decoded bytes per upload chunk

// the rows of a decoded frame that the crop needs: [crop_y, crop_y + crop_height), a contiguous band
struct Band {
    size_t offset; // of the band inside a decoded frame
    size_t bytes;
    size_t pitch; // device pitch between bands (16-byte aligned so that every band allows 128-bit loads)
};

Band crop_band(const cvvp_frame_format &f)
{
    Band b;
    const size_t row = size_t(f.src_width) * size_t(f.src_channels);
    b.offset = size_t(f.crop_y) * row;
    b.bytes = size_t(f.crop_height) * row;
    b.pitch = round_up(b.bytes, 16);
    return b;
}

template <typename T>
void free_dev(T *&p)
{
    if (p)
        cudaFree(p);
    p = nullptr;
}
template <typename T>
void free_host(T *&p)
{
    if (p)
        cudaFreeHost(p);
    p = nullptr;
}
} // namespace

void raw_stage_release(cvvp_ctx *ctx)
{
    RawStage &r = ctx->raw;
    for (int i = 0; i < 2; ++i) {
        free_dev(r.d[i]);
        if (r.up[i])
            cudaEventDestroy(r.up[i]);
        if (r.consumed[i])
            cudaEventDestroy(r.consumed[i]);
        r.up[i] = r.consumed[i] = nullptr;
        r.used[i] = false;
    }
    free_dev(r.d_out);
    r.cap = r.out_cap = 0;
}

int raw_stage_ensure(cvvp_ctx *ctx, size_t bytes_per_half)
{
    RawStage &r = ctx->raw;
    for (int i = 0; i < 2; ++i) {
        if (!r.up[i])
            CVVP_CUDA_OK(ctx, cudaEventCreateWithFlags(&r.up[i], cudaEventDisableTiming));
        if (!r.consumed[i])
            CVVP_CUDA_OK(ctx, cudaEventCreateWithFlags(&r.consumed[i], cudaEventDisableTiming));
    }
    if (r.cap >= bytes_per_half)
        return CVVP_OK;
    // the halves may still be read by queued kernels
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy));
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
    for (int i = 0; i < 2; ++i) {
        free_dev(r.d[i]);
        r.used[i] = false;
    }
    r.cap = 0;
    for (int i = 0; i < 2; ++i) {
        if (cudaMalloc(&r.d[i], bytes_per_half) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM, "frames: cudaMalloc of %zu bytes for the decoded-frame staging failed", bytes_per_half);
        }
    }
    r.cap = bytes_per_half;
    return CVVP_OK;
}

// Decoded HOST frames -> prepared frames in DEVICE memory at d_dst (+ i*dst_stride), asynchronously: the crop bands
// go up on the copy stream in chunks, each followed by one preparation kernel on the compute stream.  On return the
// work is queued; it is complete when the compute stream reaches this point.
int frames_upload_prepare(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format &f,
                          uint8_t *d_dst, size_t dst_stride)
{
    const Band band = crop_band(f);
    if (f.mode == CVVP_FRAMES_AS_IS && f.crop_x == 0 && f.crop_width == f.src_width) {
        // full-width rows kept as they are (the default of VidBgPack on a colour video): the band IS the prepared frame,
        // the copy engine puts it in place and no kernel runs
        int rc = raw_stage_ensure(ctx, 16);
        if (rc != CVVP_OK)
            return rc;
        RawStage &r = ctx->raw;
        CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(d_dst, dst_stride, frames + band.offset, frame_stride, band.bytes, size_t(n),
                                            cudaMemcpyHostToDevice, ctx->copy));
        CVVP_CUDA_OK(ctx, cudaEventRecord(r.up[0], ctx->copy));
        CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->compute, r.up[0], 0));
        return CVVP_OK;
    }
    long long per = (long long)(kRawChunkBytes / band.pitch);
    if (per < 1)
        per = 1;
    if (per > n)
        per = n;
    int rc = raw_stage_ensure(ctx, size_t(per) * band.pitch);
    if (rc != CVVP_OK)
        return rc;
    RawStage &r = ctx->raw;
    for (long long done = 0; done < n; done += per) {
        const long long nb = n - done < per ? n - done : per;
        const int b = r.next;
        r.next ^= 1;
        if (r.used[b])
            CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy, r.consumed[b], 0));
        CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(r.d[b], band.pitch, frames + size_t(done) * frame_stride + band.offset, frame_stride,
                                            band.bytes, size_t(nb), cudaMemcpyHostToDevice, ctx->copy));
        CVVP_CUDA_OK(ctx, cudaEventRecord(r.up[b], ctx->copy));
        CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->compute, r.up[b], 0));
        rc = frames_prepare_launch(ctx, r.d[b], nb, band.pitch, size_t(nb) * band.pitch, f, f.crop_y,
                                   d_dst + size_t(done) * dst_stride, dst_stride, ctx->compute);
        if (rc != CVVP_OK)
            return rc;
        CVVP_CUDA_OK(ctx, cudaEventRecord(r.consumed[b], ctx->compute));
        r.used[b] = true;
    }
    return CVVP_OK;
}

int frames_prepare_host(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format &f,
                        uint8_t *out, size_t out_stride)
{
    const size_t ob = frames_out_bytes(f);
    const size_t opitch = round_up(ob, 16);
    const Band band = crop_band(f);
    long long per = (long long)(kRawChunkBytes / band.pitch);
    if (per < 1)
        per = 1;
    if (per > n)
        per = n;
    RawStage &r = ctx->raw;
    if (r.out_cap < size_t(per) * opitch) {
        CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
        free_dev(r.d_out);
        r.out_cap = 0;
        if (cudaMalloc(&r.d_out, size_t(per) * opitch) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM, "frames: cudaMalloc of the result staging failed");
        }
        r.out_cap = size_t(per) * opitch;
    }
    for (long long done = 0; done < n; done += per) {
        const long long nb = n - done < per ? n - done : per;
        int rc = frames_upload_prepare(ctx, frames + size_t(done) * frame_stride, nb, frame_stride, f, r.d_out, opitch);
        if (rc != CVVP_OK)
            return rc;
        CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(out + size_t(done) * out_stride, out_stride, r.d_out, opitch, ob, size_t(nb),
                                            cudaMemcpyDeviceToHost, ctx->compute));
        CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
    }
    return CVVP_OK;
}

/* ------------------------------------------------------------------------------------------------------------------- */
/* shared by the highlight queue and the rolling stream (highlight_rolling.cu)                                         */
/* ------------------------------------------------------------------------------------------------------------------- */
bool hl_results_alloc(HlResults &r, long long max_batch, size_t npix, size_t pitch, int max_comps, size_t rec_bytes,
                      bool labels)
{
    const size_t nb = size_t(max_batch);
    r.npix = npix;
    r.pitch = pitch;
    r.max_comps = max_comps;
    r.rec_bytes = rec_bytes;
    r.labels = labels;
    r.mask_bytes = nb * pitch;
    // the masks come from the process-wide pool: a job on the next video of the same geometry reuses them
    void *p = nullptr;
    bool ok = pool_host_alloc(&p, r.mask_bytes) == cudaSuccess;
    if (ok) {
        r.h_out = static_cast<uint8_t *>(p);
        ok = pool_dev_alloc(&p, r.mask_bytes) == cudaSuccess;
    }
    if (ok)
        r.d_out = static_cast<uint8_t *>(p);
    if (max_comps > 0) {
        ok = ok && cudaMallocHost(&r.h_comps, nb * size_t(max_comps) * rec_bytes) == cudaSuccess;
        ok = ok && cudaMallocHost(&r.h_ncomps, nb * sizeof(int)) == cudaSuccess;
        ok = ok && cudaMalloc(&r.d_comps, nb * size_t(max_comps) * rec_bytes) == cudaSuccess;
        ok = ok && cudaMalloc(&r.d_ncomps, nb * sizeof(int)) == cudaSuccess;
    }
    if (labels) {
        ok = ok && cudaMallocHost(&r.h_labels, nb * npix * sizeof(int32_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&r.d_labels, nb * npix * sizeof(int32_t)) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&r.down, cudaEventDisableTiming) == cudaSuccess;
    if (!ok)
        cudaGetLastError();
    return ok;
}

void hl_results_free(HlResults &r)
{
    pool_host_free(r.h_out, r.mask_bytes);
    pool_dev_free(r.d_out, r.mask_bytes);
    free_host(r.h_comps);
    free_host(r.h_ncomps);
    free_host(r.h_labels);
    free_dev(r.d_comps);
    free_dev(r.d_ncomps);
    free_dev(r.d_labels);
    if (r.down)
        cudaEventDestroy(r.down);
    r = HlResults();
}

CcOut hl_results_cc(const HlResults &r, long long first)
{
    CcOut cc;
    if (r.max_comps > 0) {
        cc.comps = reinterpret_cast<cvvp_component *>(reinterpret_cast<uint8_t *>(r.d_comps) +
                                                      size_t(first) * size_t(r.max_comps) * r.rec_bytes);
        cc.max_comps = r.max_comps;
        cc.ncomps = r.d_ncomps + first;
        cc.labels = r.labels ? r.d_labels + size_t(first) * r.npix : nullptr;
        cc.labels_stride = r.npix;
    }
    return cc;
}

int hl_results_download(cvvp_ctx *ctx, HlResults &r)
{
    const size_t n = size_t(r.n);
    CVVP_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copy, ctx->compute));
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_copy, 0));
    CVVP_CUDA_OK(ctx, cudaMemcpyAsync(r.h_out, r.d_out, n * r.pitch, cudaMemcpyDeviceToHost, ctx->copy_out));
    if (r.max_comps > 0) {
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(r.h_comps, r.d_comps, n * size_t(r.max_comps) * r.rec_bytes,
                                          cudaMemcpyDeviceToHost, ctx->copy_out));
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(r.h_ncomps, r.d_ncomps, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    if (r.labels)
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(r.h_labels, r.d_labels, n * r.npix * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                          ctx->copy_out));
    CVVP_CUDA_OK(ctx, cudaEventRecord(r.down, ctx->copy_out));
    return CVVP_OK;
}

int hl_results_ready(cvvp_ctx *ctx, const HlResults &r, const char *who)
{
    const cudaError_t e = cudaEventQuery(r.down);
    if (e == cudaSuccess)
        return 1;
    if (e != cudaErrorNotReady)
        return fail(ctx, CVVP_ERR_CUDA, "%s: %s", who, cudaGetErrorString(e));
    return 0;
}

int hl_results_wait(cvvp_ctx *ctx, const HlResults &r, const char *who)
{
    const cudaError_t e = cudaEventSynchronize(r.down);
    if (e != cudaSuccess)
        return fail(ctx, CVVP_ERR_CUDA, "%s: batch failed: %s", who, cudaGetErrorString(e));
    return CVVP_OK;
}

void hl_results_copy(const HlResults &r, uint8_t *masks, size_t mask_stride, cvvp_component *comps, int *ncomps,
                     int32_t *labels, size_t labels_stride)
{
    const size_t n = size_t(r.n);
    for (size_t i = 0; i < n; ++i)
        std::memcpy(masks + i * mask_stride, r.h_out + i * r.pitch, r.npix);
    if (r.max_comps > 0 && comps)
        std::memcpy(comps, r.h_comps, n * size_t(r.max_comps) * r.rec_bytes);
    if (r.max_comps > 0 && ncomps)
        std::memcpy(ncomps, r.h_ncomps, n * sizeof(int));
    if (r.labels && labels)
        for (size_t i = 0; i < n; ++i)
            std::memcpy(labels + i * labels_stride, r.h_labels + i * r.npix, r.npix * sizeof(int32_t));
}

void sync_streams(cvvp_ctx *ctx)
{
    cudaStreamSynchronize(ctx->copy);
    cudaStreamSynchronize(ctx->compute);
    cudaStreamSynchronize(ctx->copy_out);
}

int drain_after_failure(cvvp_ctx *ctx, bool &failed, int rc)
{
    failed = true;
    const std::string why = ctx->err;
    sync_streams(ctx);
    cudaGetLastError();
    ctx->err = why;
    return rc;
}

int highlight_stream_check(cvvp_ctx *ctx, const char *who, bool begun, int args_rc, const cvvp_frame_format *fmt, int *W, int *H)
{
    if (!highlight_geometry(ctx, W, H))
        return fail(ctx, CVVP_ERR_STATE, "%s: no parameters set (call cvvp_highlight_begin first)", who);
    if (begun)
        return fail(ctx, CVVP_ERR_STATE, "%s: already begun", who);
    if (args_rc != CVVP_OK)
        return args_rc;
    if (!fmt)
        return CVVP_OK;
    const int rc = frames_check_format(ctx, fmt);
    if (rc != CVVP_OK)
        return rc;
    const int C = highlight_job_channels(ctx);
    if (C > 1) { // a colour job takes the cropped frames as they are: its kernel computes d from all their channels
        if (fmt->mode != CVVP_FRAMES_AS_IS || fmt->src_channels != C || fmt->crop_width != *W || fmt->crop_height != *H)
            return fail(ctx, CVVP_ERR_INVALID,
                        "%s: frames of a %d-channel highlight job must be CVVP_FRAMES_AS_IS with src_channels %d, cropped "
                        "to %dx%d like the background", who, C, C, *W, *H);
        return CVVP_OK;
    }
    if (fmt->crop_width != *W || fmt->crop_height != *H || frames_out_bytes(*fmt) != size_t(*W) * size_t(*H))
        return fail(ctx, CVVP_ERR_INVALID,
                    "%s: prepared frames must be single-channel %dx%d like the background (cv::findContours requires 8UC1)",
                    who, *W, *H);
    return CVVP_OK;
}

/* ------------------------------------------------------------------------------------------------------------------- */
/* asynchronous ordered highlight queue                                                                                */
/* ------------------------------------------------------------------------------------------------------------------- */
// A slot's pinned input holds WHOLE frames as the caller has them (decoded frames when the queue has a frame format,
// prepared frames otherwise), one every host_pitch bytes, so that a decoder can write straight into it
// (cvvp_highlight_slot_acquire); only the crop band of every frame crosses the link.
struct HqSlot {
    size_t b_h_in{0}, b_raw{0}, b_in{0}; // bytes of the pooled buffers below (pool.hpp)
    uint8_t *h_in{nullptr};              // pinned
    uint8_t *d_raw{nullptr}, *d_in{nullptr};
    cudaEvent_t up{nullptr};
    HlResults res;
};

struct HighlightQueue {
    int depth{0};
    long long max_batch{0};
    bool has_fmt{false};
    cvvp_frame_format fmt{};
    bool color{false};        // a colour job: the uploaded frames go through highlight_color_d into d_in
    size_t npix{0}, pitch{0}; // prepared frame bytes / device pitch
    size_t in_bytes{0}, in_pitch{0}, in_offset{0}; // what one frame uploads (crop band or the frame) and where it starts
    size_t host_pitch{0};                          // bytes between the caller's frames in a slot's pinned input
    std::vector<HqSlot> slots;
    int head{0}, count{0};
    int acquired{0};      // slots after the pending ones that are in the caller's hands (slot_acquire .. slot_commit)
    bool gap{false};      // an acquired slot was handed back unused while later ones were still out: those cannot be queued
    bool lent{false};     // the oldest pending slot's results are in the caller's hands (next_view .. view_release)
    bool failed{false};   // a submit died half-way: work of unknown extent is queued on the slot (ADVICE r1)
};

void highlight_queue_release(cvvp_ctx *ctx)
{
    HighlightQueue *q = ctx->hq;
    if (!q)
        return;
    sync_streams(ctx);
    for (HqSlot &s : q->slots) {
        pool_host_free(s.h_in, s.b_h_in);
        pool_dev_free(s.d_raw, s.b_raw);
        pool_dev_free(s.d_in, s.b_in);
        if (s.up)
            cudaEventDestroy(s.up);
        hl_results_free(s.res);
    }
    cudaGetLastError();
    delete q;
    ctx->hq = nullptr;
}

int highlight_queue_begin(cvvp_ctx *ctx, int depth, long long max_batch, const cvvp_frame_format *fmt, int max_comps)
{
    const int args = depth < 1 || depth > 64 || max_batch < 1 || max_batch > (1ll << 20) || max_comps < 0
                         ? fail(ctx, CVVP_ERR_INVALID,
                                "highlight queue: depth must be in [1, 64], max_batch in [1, 2^20], max_comps >= 0")
                         : CVVP_OK;
    int W = 0, H = 0;
    const int rc = highlight_stream_check(ctx, "highlight queue", ctx->hq != nullptr, args, fmt, &W, &H);
    if (rc != CVVP_OK)
        return rc;
    HighlightQueue *q = new (std::nothrow) HighlightQueue();
    if (!q)
        return fail(ctx, CVVP_ERR_NOMEM, "out of host memory");
    ctx->hq = q;
    q->depth = depth;
    q->max_batch = max_batch;
    q->has_fmt = fmt != nullptr;
    if (fmt)
        q->fmt = *fmt;
    q->npix = size_t(W) * size_t(H);
    q->pitch = round_up(q->npix, 128);
    q->color = highlight_job_channels(ctx) > 1;
    if (fmt) {
        const Band band = crop_band(*fmt);
        q->in_bytes = band.bytes;
        q->in_pitch = band.pitch;
        q->in_offset = band.offset;
        q->host_pitch = round_up(size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels), 64);
    } else {
        q->in_bytes = q->npix * size_t(highlight_job_channels(ctx));
        q->in_pitch = round_up(q->in_bytes, 128);
        q->in_offset = 0;
        q->host_pitch = q->in_pitch;
    }
    q->slots.resize(size_t(depth));
    const size_t nb = size_t(max_batch);
    bool ok = true;
    for (HqSlot &s : q->slots) {
        // the big buffers come from the process-wide pool: a job on the next video of the same geometry reuses them
        auto dev = [&](uint8_t *&p, size_t &b, size_t bytes) {
            void *v = nullptr;
            if (pool_dev_alloc(&v, bytes) != cudaSuccess)
                return false;
            p = static_cast<uint8_t *>(v);
            b = bytes;
            return true;
        };
        void *h = nullptr;
        ok = ok && pool_host_alloc(&h, nb * q->host_pitch) == cudaSuccess;
        if (ok) {
            s.h_in = static_cast<uint8_t *>(h);
            s.b_h_in = nb * q->host_pitch;
        }
        if (fmt || q->color)
            ok = ok && dev(s.d_raw, s.b_raw, nb * q->in_pitch);
        ok = ok && dev(s.d_in, s.b_in, nb * q->pitch);
        ok = ok && cudaEventCreateWithFlags(&s.up, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && hl_results_alloc(s.res, max_batch, q->npix, q->pitch, max_comps, highlight_record_bytes(ctx), false);
        if (!ok)
            break;
    }
    if (!ok) {
        cudaGetLastError();
        highlight_queue_release(ctx);
        return fail(ctx, CVVP_ERR_NOMEM, "highlight queue: allocation of %d slots of %lld frames failed", depth, max_batch);
    }
    return CVVP_OK;
}

int highlight_queue_pending(const cvvp_ctx *ctx)
{
    return ctx->hq ? ctx->hq->count : 0;
}

// queues H2D (crop bands only) -> [frame preparation] -> highlight kernel -> D2H for the n frames in the slot's pinned input
static int launch_slot(cvvp_ctx *ctx, HighlightQueue *q, HqSlot &s, long long n)
{
    s.res.n = n;
    uint8_t *up_to = q->has_fmt || q->color ? s.d_raw : s.d_in;
    CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(up_to, q->in_pitch, s.h_in + q->in_offset, q->host_pitch, q->in_bytes, size_t(n),
                                        cudaMemcpyHostToDevice, ctx->copy));
    CVVP_CUDA_OK(ctx, cudaEventRecord(s.up, ctx->copy));
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->compute, s.up, 0));
    int rc;
    if (q->color) {
        // one kernel makes the d planes straight from the uploaded frames (the crop of the decoded rows with a format)
        const size_t row_stride = q->has_fmt ? size_t(q->fmt.src_width) * size_t(q->fmt.src_channels) : 0;
        rc = highlight_color_d(ctx, s.d_raw, n, q->in_pitch, row_stride, q->has_fmt ? q->fmt.crop_x : 0, nullptr, 0, s.d_in,
                               q->pitch, ctx->compute);
        if (rc == CVVP_OK)
            rc = highlight_device_planes(ctx, s.d_in, n, q->pitch, s.res.d_out, q->pitch, hl_results_cc(s.res, 0),
                                         ctx->compute);
        if (rc != CVVP_OK)
            return rc;
        return hl_results_download(ctx, s.res);
    }
    if (q->has_fmt) {
        rc = frames_prepare_launch(ctx, s.d_raw, n, q->in_pitch, size_t(n) * q->in_pitch, q->fmt, q->fmt.crop_y, s.d_in, q->pitch,
                                   ctx->compute);
        if (rc != CVVP_OK)
            return rc;
    }
    rc = highlight_device_bg(ctx, s.d_in, n, q->pitch, nullptr, 0, s.res.d_out, q->pitch, hl_results_cc(s.res, 0),
                             ctx->compute);
    if (rc != CVVP_OK)
        return rc;
    return hl_results_download(ctx, s.res);
}

static int check_can_fill(cvvp_ctx *ctx, HighlightQueue *q)
{
    if (!q)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: not begun");
    if (q->failed)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: an earlier submit failed; end the queue and begin a new one");
    if (q->count + q->acquired >= q->depth)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: %d batches pending or being filled; call cvvp_highlight_next first",
                    q->depth);
    return CVVP_OK;
}

// A launch that failed half-way leaves copies / kernels of unknown extent queued on the slot while the slot is not
// counted as pending: the next submit would overwrite pinned memory an earlier H2D may still be reading.  Further
// submits are refused; cvvp_highlight_queue_end (or cvvp_highlight_end) clears the state.
static int queue_slot(cvvp_ctx *ctx, HighlightQueue *q, HqSlot &s, long long n)
{
    const int rc = launch_slot(ctx, q, s, n);
    if (rc != CVVP_OK)
        return drain_after_failure(ctx, q->failed, rc);
    q->count++;
    return CVVP_OK;
}

int highlight_queue_submit(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    HighlightQueue *q = ctx->hq;
    int rc = check_can_fill(ctx, q);
    if (rc != CVVP_OK)
        return rc;
    if (q->acquired)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: slots are acquired; commit them before submitting");
    if (!frames || n < 1 || n > q->max_batch || frame_stride < q->in_offset + q->in_bytes)
        return fail(ctx, CVVP_ERR_INVALID, "highlight queue: bad submit arguments (1 <= n <= %lld frames of at least %zu bytes)",
                    q->max_batch, q->in_offset + q->in_bytes);
    HqSlot &s = q->slots[size_t((q->head + q->count) % q->depth)];
    // a slot is handed out again only after cvvp_highlight_next waited for its `down` event: nothing of it is in flight
    for (long long i = 0; i < n; ++i)
        std::memcpy(s.h_in + size_t(i) * q->host_pitch + q->in_offset, frames + size_t(i) * frame_stride + q->in_offset, q->in_bytes);
    return queue_slot(ctx, q, s, n);
}

int highlight_slot_acquire(cvvp_ctx *ctx, uint8_t **h_frames, size_t *frame_pitch, long long *max_frames)
{
    HighlightQueue *q = ctx->hq;
    int rc = check_can_fill(ctx, q);
    if (rc != CVVP_OK)
        return rc;
    HqSlot &s = q->slots[size_t((q->head + q->count + q->acquired) % q->depth)];
    q->acquired++;
    *h_frames = s.h_in;
    *frame_pitch = q->host_pitch;
    if (max_frames)
        *max_frames = q->max_batch;
    return CVVP_OK;
}

int highlight_slot_commit(cvvp_ctx *ctx, long long n)
{
    HighlightQueue *q = ctx->hq;
    if (!q || !q->acquired)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: no slot is acquired");
    if (n < 0 || n > q->max_batch)
        return fail(ctx, CVVP_ERR_INVALID, "highlight queue: a slot takes 0 .. %lld frames", q->max_batch);
    if (n > 0 && q->gap)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: a slot acquired earlier was handed back unused; batches are queued in "
                                         "the order their slots were acquired");
    q->acquired--; // the oldest acquired slot
    if (n == 0) {  // handed back unused (end of the stream)
        q->gap = q->acquired > 0;
        return CVVP_OK;
    }
    return queue_slot(ctx, q, q->slots[size_t((q->head + q->count) % q->depth)], n);
}

int highlight_queue_ready(cvvp_ctx *ctx)
{
    HighlightQueue *q = ctx->hq;
    if (!q || q->count == 0)
        return 0;
    if (q->lent)
        return 1;
    return hl_results_ready(ctx, q->slots[size_t(q->head)].res, "highlight queue");
}

int highlight_queue_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long *n_out, cvvp_component *comps_out,
                         int *ncomps_out)
{
    HighlightQueue *q = ctx->hq;
    if (!q)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: not begun");
    if (!masks_out || !n_out || out_stride < q->npix)
        return fail(ctx, CVVP_ERR_INVALID, "highlight queue: bad arguments to next");
    if (q->count == 0)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: nothing pending");
    if (q->lent)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: the oldest batch is lent out; release the view first");
    const HlResults &r = q->slots[size_t(q->head)].res;
    const int rc = hl_results_wait(ctx, r, "highlight queue");
    q->head = (q->head + 1) % q->depth;
    q->count--;
    if (rc != CVVP_OK)
        return rc;
    hl_results_copy(r, masks_out, out_stride, comps_out, ncomps_out, nullptr, 0);
    *n_out = r.n;
    return CVVP_OK;
}

int highlight_queue_next_view(cvvp_ctx *ctx, const uint8_t **h_masks, size_t *mask_pitch, long long *n_out,
                              const cvvp_component **comps, const int **ncomps)
{
    HighlightQueue *q = ctx->hq;
    if (!q)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: not begun");
    if (!h_masks || !mask_pitch || !n_out)
        return fail(ctx, CVVP_ERR_INVALID, "highlight queue: bad arguments to next_view");
    if (q->count == 0)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: nothing pending");
    if (q->lent)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: the oldest batch is already lent out");
    const HlResults &r = q->slots[size_t(q->head)].res;
    const int rc = hl_results_wait(ctx, r, "highlight queue");
    if (rc != CVVP_OK) {
        q->head = (q->head + 1) % q->depth;
        q->count--;
        return rc;
    }
    q->lent = true;
    *h_masks = r.h_out;
    *mask_pitch = q->pitch;
    *n_out = r.n;
    if (comps)
        *comps = r.h_comps; // null without components
    if (ncomps)
        *ncomps = r.h_ncomps;
    return CVVP_OK;
}

int highlight_queue_view_release(cvvp_ctx *ctx)
{
    HighlightQueue *q = ctx->hq;
    if (!q || !q->lent)
        return fail(ctx, CVVP_ERR_STATE, "highlight queue: no view is lent out");
    q->lent = false;
    q->head = (q->head + 1) % q->depth;
    q->count--;
    return CVVP_OK;
}
} // namespace cvvp
