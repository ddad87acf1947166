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

#include <deque>
#include <memory>
#include <new>
#include <vector>

namespace cvvp
{
namespace
{
struct RollSlot {
    long long first{0}; // frames [first, first + res.n)
    HlResults res;
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
    size_t npix{0}, pitch{0}, in_bytes{0}; // mask bytes / mask pitch / bytes of one pushed frame
    size_t nelem{0}, fpitch{0};            // bytes of a prepared frame (npix * the job's channels) / its pitch in the ring
    long long ring{0};                     // frames the ring holds
    uint8_t *d_ring{nullptr}, *d_bgs{nullptr};
    size_t b_ring{0}, b_bgs{0};
    long long received{0}, launched{0};
    bool closed{false}, failed{false};
    std::vector<std::unique_ptr<RollSlot>> slots; // every slot ever allocated
    std::vector<RollSlot *> idle;
    std::deque<RollSlot *> pending;
};

void highlight_rolling_release(cvvp_ctx *ctx)
{
    RollingStream *r = ctx->hr;
    if (!r)
        return;
    sync_streams(ctx);
    for (auto &s : r->slots)
        hl_results_free(s->res);
    pool_dev_free(r->d_ring, r->b_ring);
    pool_dev_free(r->d_bgs, r->b_bgs);
    cudaGetLastError();
    delete r;
    ctx->hr = nullptr;
}

int highlight_rolling_begin(cvvp_ctx *ctx, int window, long long max_batch, const cvvp_frame_format *fmt, int max_comps,
                            int labels)
{
    int args = CVVP_OK;
    if (window < 1 || window > 65535)
        args = fail(ctx, CVVP_ERR_INVALID, "rolling highlight: window %d outside [1, 65535]", window);
    else if (max_batch < 1 || max_batch > (1ll << 20) || max_comps < 0 || (labels && max_comps < 1))
        args = fail(ctx, CVVP_ERR_INVALID, "rolling highlight: max_batch must be in [1, 2^20], max_comps >= 0 (>= 1 with labels)");
    int W = 0, H = 0;
    const int rc = highlight_stream_check(ctx, "rolling highlight", ctx->hr != nullptr, args, fmt, &W, &H);
    if (rc != CVVP_OK)
        return rc;
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
    // a colour job's ring holds colour frames, and its backgrounds are colour too (the median is element-wise)
    r->nelem = r->npix * size_t(highlight_job_channels(ctx));
    r->fpitch = round_up(r->nelem, 128);
    r->in_bytes = fmt ? size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels) : r->nelem;
    r->ring = (long long)window + max_batch;
    void *p = nullptr;
    if (pool_dev_alloc(&p, size_t(r->ring) * r->fpitch) != cudaSuccess) {
        cudaGetLastError();
        const size_t bytes = size_t(r->ring) * r->fpitch;
        highlight_rolling_release(ctx);
        return fail(ctx, CVVP_ERR_NOMEM,
                    "rolling highlight: the ring of %lld frames (window %d + batch %lld, %zu bytes) does not fit on the device; "
                    "use a smaller window", (long long)window + max_batch, window, max_batch, bytes);
    }
    r->d_ring = static_cast<uint8_t *>(p);
    r->b_ring = size_t(r->ring) * r->fpitch;
    if (pool_dev_alloc(&p, size_t(max_batch) * r->fpitch) != cudaSuccess) {
        cudaGetLastError();
        highlight_rolling_release(ctx);
        return fail(ctx, CVVP_ERR_NOMEM, "rolling highlight: allocation of %lld backgrounds failed", max_batch);
    }
    r->d_bgs = static_cast<uint8_t *>(p);
    r->b_bgs = size_t(max_batch) * r->fpitch;
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
    if (!hl_results_alloc(s->res, r->max_batch, r->npix, r->pitch, r->max_comps, highlight_record_bytes(ctx), r->labels)) {
        hl_results_free(s->res);
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
        s->res.n = n;
        r->pending.push_back(s);
        rc = median_roll_launch(ctx, r->d_ring, r->ring, r->fpitch, r->received, r->nelem, r->window, r->percent, t0, t0 + n,
                                r->d_bgs, r->fpitch, ctx->compute);
        if (rc != CVVP_OK)
            return rc;
        // the frames themselves, in at most two contiguous runs of ring slots
        for (long long done = 0; done < n;) {
            const long long slot = (t0 + done) % r->ring;
            const long long k = n - done < r->ring - slot ? n - done : r->ring - slot;
            rc = highlight_device_bg(ctx, r->d_ring + size_t(slot) * r->fpitch, k, r->fpitch,
                                     r->d_bgs + size_t(done) * r->fpitch, r->fpitch, s->res.d_out + size_t(done) * r->pitch,
                                     r->pitch, hl_results_cc(s->res, done), ctx->compute);
            if (rc != CVVP_OK)
                return rc;
            done += k;
        }
        if ((rc = hl_results_download(ctx, s->res)) != CVVP_OK)
            return rc;
        r->launched = t0 + n;
    }
    return CVVP_OK;
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
        uint8_t *dst = r->d_ring + size_t(slot) * r->fpitch;
        if (r->has_fmt) {
            rc = frames_upload_prepare(ctx, frames + size_t(done) * frame_stride, k, frame_stride, r->fmt, dst, r->fpitch);
            if (rc != CVVP_OK)
                return drain_after_failure(ctx, r->failed, rc);
        } else {
            const cudaError_t e = cudaMemcpy2DAsync(dst, r->fpitch, frames + size_t(done) * frame_stride, frame_stride, r->nelem,
                                                    size_t(k), cudaMemcpyHostToDevice, ctx->compute);
            if (e != cudaSuccess)
                return drain_after_failure(ctx, r->failed,
                                           fail(ctx, CVVP_ERR_CUDA, "rolling highlight: H2D failed: %s", cudaGetErrorString(e)));
        }
        done += k;
    }
    r->received += n;
    rc = launch_ready(ctx, r);
    return rc == CVVP_OK ? rc : drain_after_failure(ctx, r->failed, rc);
}

int highlight_rolling_close(cvvp_ctx *ctx)
{
    RollingStream *r = ctx->hr;
    int rc = check_open(ctx, r);
    if (rc != CVVP_OK)
        return rc;
    r->closed = true;
    rc = launch_ready(ctx, r);
    return rc == CVVP_OK ? rc : drain_after_failure(ctx, r->failed, rc);
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
    return hl_results_ready(ctx, r->pending.front()->res, "rolling highlight");
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
    if (max_n < s->res.n)
        return fail(ctx, CVVP_ERR_INVALID, "rolling highlight: the next batch holds %lld frames, the buffers %lld", s->res.n,
                    max_n);
    const int rc = hl_results_wait(ctx, s->res, "rolling highlight");
    r->pending.pop_front();
    r->idle.push_back(s);
    if (rc != CVVP_OK)
        return rc;
    hl_results_copy(s->res, masks_out, out_stride, comps_out, ncomps_out, labels_out, labels_stride);
    *first_index = s->first;
    *n_out = s->res.n;
    return CVVP_OK;
}
} // namespace cvvp
