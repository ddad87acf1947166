// Highlight against a rolling temporal-median background, as an ordered stream whose masks come back LATER than their
// frames go in: the mask of frame t needs the window s(t) .. s(t) + W - 1 of median_roll.cu, i.e. W - 1 frames ahead
// at the start of the stream and ceil(W / 2) - 1 frames ahead afterwards; the last ones only once the stream is closed
// (the frame count of a video is only known when the decoder stops).
//
//   push  : the batch goes up (decoded frames through the frame preparation of frames.cu) into a device ring of
//           W + max_batch prepared frames; every frame whose window is now complete gets its background
//           (median_roll_launch, straight from the ring) and its mask (highlight_device_bg), in chunks of at most
//           max_batch frames; each chunk's masks (and components) go down into a pinned result slot
//   close : the same for the rest of the frames, with the windows clamped to the frames actually pushed
//   next  : the oldest result chunk, in frame order
// Ring size: after every push all frames whose window is complete are launched, and the first frame whose window is not
// complete needs nothing older than frame received - W + 1; the next push adds at most max_batch frames: W - 1 +
// max_batch frames are live at any time.  Every kernel and the uploads into the ring are ordered on the compute
// stream, so a push never overwrites a slot that an earlier launch still reads.
#include "context.hpp"
#include "pool.hpp"

#include <cstring>
#include <deque>
#include <memory>
#include <new>
#include <vector>

namespace cvvp
{
namespace
{
size_t round_up(size_t v, size_t a)
{
    return (v + a - 1) / a * a;
}

struct RollSlot {
    long long first{0}, n{0}; // frames [first, first + n)
    size_t b_h_out{0}, b_d_out{0};
    uint8_t *h_out{nullptr}, *d_out{nullptr}; // h_out: pinned (pool), d_out: device (pool)
    cvvp_component *h_comps{nullptr}, *d_comps{nullptr};
    int *h_ncomps{nullptr}, *d_ncomps{nullptr};
    int32_t *h_labels{nullptr}, *d_labels{nullptr};
    cudaEvent_t down{nullptr};
};
} // namespace

struct RollingStream {
    int window{0};
    int percent{50}; // the context's percentile when the stream began
    long long max_batch{0};
    bool has_fmt{false};
    cvvp_frame_format fmt{};
    int max_comps{0};
    bool labels{false};
    size_t npix{0}, pitch{0}, in_bytes{0}; // prepared frame bytes / device pitch / bytes of one pushed frame
    long long ring{0};                     // frames the ring holds
    uint8_t *d_ring{nullptr}, *d_bgs{nullptr};
    size_t b_ring{0}, b_bgs{0};
    long long received{0}, launched{0};
    bool closed{false}, failed{false};
    std::vector<std::unique_ptr<RollSlot>> slots; // every slot ever allocated
    std::vector<RollSlot *> idle;
    std::deque<RollSlot *> pending;
};

static void free_slot(RollSlot &s)
{
    pool_host_free(s.h_out, s.b_h_out);
    pool_dev_free(s.d_out, s.b_d_out);
    if (s.h_comps) cudaFreeHost(s.h_comps);
    if (s.h_ncomps) cudaFreeHost(s.h_ncomps);
    if (s.h_labels) cudaFreeHost(s.h_labels);
    if (s.d_comps) cudaFree(s.d_comps);
    if (s.d_ncomps) cudaFree(s.d_ncomps);
    if (s.d_labels) cudaFree(s.d_labels);
    if (s.down) cudaEventDestroy(s.down);
    s = RollSlot();
}

void highlight_rolling_release(cvvp_ctx *ctx)
{
    RollingStream *r = ctx->hr;
    if (!r)
        return;
    cudaStreamSynchronize(ctx->copy);
    cudaStreamSynchronize(ctx->compute);
    cudaStreamSynchronize(ctx->copy_out);
    for (auto &s : r->slots)
        free_slot(*s);
    pool_dev_free(r->d_ring, r->b_ring);
    pool_dev_free(r->d_bgs, r->b_bgs);
    cudaGetLastError();
    delete r;
    ctx->hr = nullptr;
}

int highlight_rolling_begin(cvvp_ctx *ctx, int window, long long max_batch, const cvvp_frame_format *fmt, int max_comps,
                            int labels)
{
    int W = 0, H = 0;
    if (!highlight_geometry(ctx, &W, &H))
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: no parameters set (call cvvp_highlight_begin first)");
    if (ctx->hr)
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: already begun");
    if (window < 1 || window > 65535)
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: window %d outside [1, 65535]", window);
    if (max_batch < 1 || max_batch > (1ll << 20) || max_comps < 0 || (labels && max_comps < 1))
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: max_batch must be in [1, 2^20], max_comps >= 0 (>= 1 with labels)");
    if (fmt) {
        int rc = frames_check_format(ctx, fmt);
        if (rc != CVVP_OK)
            return rc;
        if (fmt->crop_width != W || fmt->crop_height != H || frames_out_bytes(*fmt) != size_t(W) * size_t(H))
            return fail(ctx, CVVP_ERR_INVALID,
                        "rolling highlight: prepared frames must be single-channel %dx%d like the background (cv::findContours "
                        "requires 8UC1)", W, H);
    }
    RollingStream *r = new (std::nothrow) RollingStream();
    if (!r)
        return fail(ctx, CVVP_ERR_NOMEM, "out of host memory");
    ctx->hr = r;
    r->window = window;
    r->percent = ctx->percent;
    r->max_batch = max_batch;
    r->has_fmt = fmt != nullptr;
    if (fmt)
        r->fmt = *fmt;
    r->max_comps = max_comps;
    r->labels = labels != 0;
    r->npix = size_t(W) * size_t(H);
    r->pitch = round_up(r->npix, 128);
    r->in_bytes = fmt ? size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels) : r->npix;
    r->ring = (long long)window + max_batch;
    void *p = nullptr;
    if (pool_dev_alloc(&p, size_t(r->ring) * r->pitch) != cudaSuccess) {
        cudaGetLastError();
        const size_t bytes = size_t(r->ring) * r->pitch;
        highlight_rolling_release(ctx);
        return fail(ctx, CVVP_ERR_NOMEM,
                    "rolling highlight: the ring of %lld frames (window %d + batch %lld, %zu bytes) does not fit on the device; "
                    "use a smaller window", (long long)window + max_batch, window, max_batch, bytes);
    }
    r->d_ring = static_cast<uint8_t *>(p);
    r->b_ring = size_t(r->ring) * r->pitch;
    if (pool_dev_alloc(&p, size_t(max_batch) * r->pitch) != cudaSuccess) {
        cudaGetLastError();
        highlight_rolling_release(ctx);
        return fail(ctx, CVVP_ERR_NOMEM, "rolling highlight: allocation of %lld backgrounds failed", max_batch);
    }
    r->d_bgs = static_cast<uint8_t *>(p);
    r->b_bgs = size_t(max_batch) * r->pitch;
    return CVVP_OK;
}

static int get_slot(cvvp_ctx *ctx, RollingStream *r, RollSlot **out)
{
    if (!r->idle.empty()) {
        *out = r->idle.back();
        r->idle.pop_back();
        return CVVP_OK;
    }
    auto s = std::make_unique<RollSlot>();
    const size_t nb = size_t(r->max_batch);
    void *p = nullptr;
    bool ok = pool_host_alloc(&p, nb * r->pitch) == cudaSuccess;
    if (ok) {
        s->h_out = static_cast<uint8_t *>(p);
        s->b_h_out = nb * r->pitch;
        ok = pool_dev_alloc(&p, nb * r->pitch) == cudaSuccess;
    }
    if (ok) {
        s->d_out = static_cast<uint8_t *>(p);
        s->b_d_out = nb * r->pitch;
    }
    if (ok && r->max_comps > 0) {
        ok = ok && cudaMallocHost(&s->h_comps, nb * size_t(r->max_comps) * sizeof(cvvp_component)) == cudaSuccess;
        ok = ok && cudaMallocHost(&s->h_ncomps, nb * sizeof(int)) == cudaSuccess;
        ok = ok && cudaMalloc(&s->d_comps, nb * size_t(r->max_comps) * sizeof(cvvp_component)) == cudaSuccess;
        ok = ok && cudaMalloc(&s->d_ncomps, nb * sizeof(int)) == cudaSuccess;
    }
    if (ok && r->labels) {
        ok = ok && cudaMallocHost(&s->h_labels, nb * r->npix * sizeof(int32_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&s->d_labels, nb * r->npix * sizeof(int32_t)) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&s->down, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        free_slot(*s);
        return fail(ctx, CVVP_ERR_NOMEM, "rolling highlight: allocation of a result slot of %lld frames failed", r->max_batch);
    }
    *out = s.get();
    r->slots.push_back(std::move(s));
    return CVVP_OK;
}

// frames whose window is complete: all of them once the stream is closed, else those with s(t) + W <= received
static long long ready_count(const RollingStream *r)
{
    if (r->closed)
        return r->received;
    if (r->received < r->window)
        return 0;
    return r->received - (r->window + 1) / 2 + 1;
}

// backgrounds, masks and the D2H of every ready frame that has not been launched yet
static int launch_ready(cvvp_ctx *ctx, RollingStream *r)
{
    const long long upto = ready_count(r);
    while (r->launched < upto) {
        const long long t0 = r->launched;
        const long long n = upto - t0 < r->max_batch ? upto - t0 : r->max_batch;
        RollSlot *s = nullptr;
        int rc = get_slot(ctx, r, &s);
        if (rc != CVVP_OK)
            return rc;
        s->first = t0;
        s->n = n;
        r->pending.push_back(s);
        rc = median_roll_launch(ctx, r->d_ring, r->ring, r->pitch, r->received, r->npix, r->window, r->percent, t0, t0 + n,
                                r->d_bgs, r->pitch, ctx->compute);
        if (rc != CVVP_OK)
            return rc;
        // the frames themselves, in at most two contiguous runs of ring slots
        for (long long done = 0; done < n;) {
            const long long slot = (t0 + done) % r->ring;
            const long long k = n - done < r->ring - slot ? n - done : r->ring - slot;
            rc = highlight_device_bg(ctx, r->d_ring + size_t(slot) * r->pitch, k, r->pitch, r->d_bgs + size_t(done) * r->pitch,
                                     r->pitch, s->d_out + size_t(done) * r->pitch, r->pitch,
                                     s->d_comps ? s->d_comps + size_t(done) * size_t(r->max_comps) : nullptr, r->max_comps,
                                     s->d_ncomps ? s->d_ncomps + done : nullptr,
                                     s->d_labels ? s->d_labels + size_t(done) * r->npix : nullptr, r->npix, ctx->compute);
            if (rc != CVVP_OK)
                return rc;
            done += k;
        }
        CVVP_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copy, ctx->compute));
        CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_copy, 0));
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(s->h_out, s->d_out, size_t(n) * r->pitch, cudaMemcpyDeviceToHost, ctx->copy_out));
        if (s->d_comps) {
            CVVP_CUDA_OK(ctx, cudaMemcpyAsync(s->h_comps, s->d_comps, size_t(n) * size_t(r->max_comps) * sizeof(cvvp_component),
                                              cudaMemcpyDeviceToHost, ctx->copy_out));
            CVVP_CUDA_OK(ctx, cudaMemcpyAsync(s->h_ncomps, s->d_ncomps, size_t(n) * sizeof(int), cudaMemcpyDeviceToHost, ctx->copy_out));
        }
        if (s->d_labels)
            CVVP_CUDA_OK(ctx, cudaMemcpyAsync(s->h_labels, s->d_labels, size_t(n) * r->npix * sizeof(int32_t),
                                              cudaMemcpyDeviceToHost, ctx->copy_out));
        CVVP_CUDA_OK(ctx, cudaEventRecord(s->down, ctx->copy_out));
        r->launched = t0 + n;
    }
    return CVVP_OK;
}

// work of unknown extent may be queued after a failure half-way: drain, and refuse further pushes
static int stream_failed(cvvp_ctx *ctx, RollingStream *r, int rc)
{
    const std::string why = ctx->err;
    cudaStreamSynchronize(ctx->copy);
    cudaStreamSynchronize(ctx->compute);
    cudaStreamSynchronize(ctx->copy_out);
    cudaGetLastError();
    r->failed = true;
    ctx->err = why;
    return rc;
}

static int check_open(cvvp_ctx *ctx, RollingStream *r)
{
    if (!r)
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: not begun");
    if (r->failed)
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: an earlier call failed; end the stream and begin a new one");
    if (r->closed)
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: the stream is closed");
    return CVVP_OK;
}

int highlight_rolling_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    RollingStream *r = ctx->hr;
    int rc = check_open(ctx, r);
    if (rc != CVVP_OK)
        return rc;
    if (!frames || n < 1 || n > r->max_batch || frame_stride < r->in_bytes)
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: bad push arguments (1 <= n <= %lld frames of at least %zu bytes)",
                    r->max_batch, r->in_bytes);
    // the uploads of decoded full-width frames go into the ring on the copy stream: after everything queued so far
    CVVP_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copy, ctx->compute));
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy, ctx->ev_copy, 0));
    for (long long done = 0; done < n;) {
        const long long slot = (r->received + done) % r->ring;
        const long long k = n - done < r->ring - slot ? n - done : r->ring - slot;
        uint8_t *dst = r->d_ring + size_t(slot) * r->pitch;
        if (r->has_fmt) {
            rc = frames_upload_prepare(ctx, frames + size_t(done) * frame_stride, k, frame_stride, r->fmt, dst, r->pitch);
            if (rc != CVVP_OK)
                return stream_failed(ctx, r, rc);
        } else {
            const cudaError_t e = cudaMemcpy2DAsync(dst, r->pitch, frames + size_t(done) * frame_stride, frame_stride, r->npix,
                                                    size_t(k), cudaMemcpyHostToDevice, ctx->compute);
            if (e != cudaSuccess)
                return stream_failed(ctx, r, fail(ctx, CVVP_ERR_CUDA, "rolling highlight: H2D failed: %s", cudaGetErrorString(e)));
        }
        done += k;
    }
    r->received += n;
    rc = launch_ready(ctx, r);
    return rc == CVVP_OK ? rc : stream_failed(ctx, r, rc);
}

int highlight_rolling_close(cvvp_ctx *ctx)
{
    RollingStream *r = ctx->hr;
    int rc = check_open(ctx, r);
    if (rc != CVVP_OK)
        return rc;
    r->closed = true;
    rc = launch_ready(ctx, r);
    return rc == CVVP_OK ? rc : stream_failed(ctx, r, rc);
}

int highlight_rolling_pending(const cvvp_ctx *ctx)
{
    return ctx->hr ? int(ctx->hr->pending.size()) : 0;
}

int highlight_rolling_ready(cvvp_ctx *ctx)
{
    RollingStream *r = ctx->hr;
    if (!r || r->pending.empty())
        return 0;
    const cudaError_t e = cudaEventQuery(r->pending.front()->down);
    if (e == cudaSuccess)
        return 1;
    if (e != cudaErrorNotReady)
        return fail(ctx, CVVP_ERR_CUDA, "rolling highlight: %s", cudaGetErrorString(e));
    return 0;
}

int highlight_rolling_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long max_n, long long *first_index,
                           long long *n_out, cvvp_component *comps_out, int *ncomps_out, int32_t *labels_out,
                           size_t labels_stride)
{
    RollingStream *r = ctx->hr;
    if (!r)
        return fail(ctx, CVVP_ERR_STATE, "rolling highlight: not begun");
    if (!masks_out || !first_index || !n_out || out_stride < r->npix || (labels_out && labels_stride < r->npix))
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: bad arguments to next");
    if (r->pending.empty()) {
        *first_index = r->launched;
        *n_out = 0;
        return CVVP_OK;
    }
    RollSlot *s = r->pending.front();
    if (max_n < s->n)
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: the next batch holds %lld frames, the buffers %lld", s->n, max_n);
    const cudaError_t e = cudaEventSynchronize(s->down);
    r->pending.pop_front();
    r->idle.push_back(s);
    if (e != cudaSuccess)
        return fail(ctx, CVVP_ERR_CUDA, "rolling highlight: batch failed: %s", cudaGetErrorString(e));
    for (long long i = 0; i < s->n; ++i)
        std::memcpy(masks_out + size_t(i) * out_stride, s->h_out + size_t(i) * r->pitch, r->npix);
    if (r->max_comps > 0 && comps_out)
        std::memcpy(comps_out, s->h_comps, size_t(s->n) * size_t(r->max_comps) * sizeof(cvvp_component));
    if (r->max_comps > 0 && ncomps_out)
        std::memcpy(ncomps_out, s->h_ncomps, size_t(s->n) * sizeof(int));
    if (r->labels && labels_out)
        for (long long i = 0; i < s->n; ++i)
            std::memcpy(labels_out + size_t(i) * labels_stride, s->h_labels + size_t(i) * r->npix, r->npix * sizeof(int32_t));
    *first_index = s->first;
    *n_out = s->n;
    return CVVP_OK;
}
} // namespace cvvp
