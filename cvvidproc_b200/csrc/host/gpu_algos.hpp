// C++ host layer over the C ABI (include/cvvp.h): the two hot-path operators with the reference's own plugin shape.
//
// The reference's operator interface is TokenProcessorAlgo<Algo, TokenT, ResultT>
// (/root/reference/Sources/AsyncTokens/token_processor_algo.h:52-61):
//     Insert(unique_ptr<TokenT>), TryGetResult() -> unique_ptr<ResultT> (null = none), NotifyNoMoreTokens(), HasResults()
// with the parameter pack moved in by value (:37).  GpuMedianAlgo / GpuHighlightAlgo keep exactly that shape; the only
// change is that a token is a BATCH of frames (FrameBatch) instead of one cv::Mat, because a GPU wants many frames
// per submission.  No OpenCV types: OpenCV C++ is not part of this build (decode is done by the caller).
//
// Error convention (Sources/Utility/exception_assert.cpp:22-33): validation failures throw std::runtime_error with a
// "cvvidproc(<ver>) <file>:<line>: assert failed in function '<f>()'" text; C-ABI failures are converted the same way.
#pragma once
#include <cstdint>
#include <cstring>
#include <algorithm>
#include <deque>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "cvvp.h"

#define CVVP_HOST_VERSION "b200-0.1"

namespace cvvp_host
{
[[noreturn]] inline void assert_fail(const char *expr, const char *func, const char *file, int line, const char *msg)
{
    std::ostringstream os;
    os << "cvvidproc(" << CVVP_HOST_VERSION << ") " << file << ':' << line << ": assert failed in function '" << func
       << "()'\n" << expr;
    if (msg && *msg)
        os << "\nassert msg: " << msg;
    throw std::runtime_error(os.str());
}
#define CVVP_ASSERT(expr) \
    do { if (!(expr)) ::cvvp_host::assert_fail(#expr, __func__, __FILE__, __LINE__, ""); } while (0)
#define CVVP_ASSERT_MSG(expr, msg) \
    do { if (!(expr)) ::cvvp_host::assert_fail(#expr, __func__, __FILE__, __LINE__, msg); } while (0)

// owning 8-bit image / image batch: n frames of rows x cols x channels bytes, contiguous
struct FrameBatch {
    int n{0}, rows{0}, cols{0}, channels{1};
    std::vector<std::uint8_t> data;
    std::size_t frame_bytes() const { return std::size_t(rows) * cols * channels; }
    bool empty() const { return n == 0 || data.empty(); }
    // highlight results with the opt-in components: max_comps records and one count per frame, optional label images
    int max_comps{0};
    std::size_t rec_bytes{sizeof(cvvp_component)}; // sizeof(cvvp_component_stats) when the job computes statistics
    std::vector<std::uint8_t> comps;               // [frame][max_comps] records of rec_bytes each
    std::vector<int> ncomps;
    std::vector<std::int32_t> labels;
    int component_count(int i) const { return ncomps.empty() ? 0 : ncomps[std::size_t(i)]; }
    cvvp_component *component_records() { return reinterpret_cast<cvvp_component *>(comps.data()); }
    const std::int32_t *label_image(int i) const { return labels.empty() ? nullptr : labels.data() + std::size_t(i) * frame_bytes(); }
};

// How decoded frames become tokens (CvVidFramesGeneratorAlgo::GetTokenSet,
// Sources/ProcessorTokenHandlers/cv_vid_frames_generator_algo.h:141-156): crop, then channel 0 / RGB2GRAY / as is.
// With a SourceFormat the operators take DECODED frames and the device does that work (csrc/frames.cu).
struct SourceFormat {
    bool enabled{false};
    cvvp_frame_format fmt{};
    int out_rows() const { return fmt.crop_height; }
    int out_cols() const { return fmt.crop_width; }
    int out_channels() const { return fmt.mode == CVVP_FRAMES_AS_IS ? fmt.src_channels : 1; }
    std::size_t src_bytes() const { return std::size_t(fmt.src_width) * fmt.src_height * fmt.src_channels; }
};

class Context
{
public:
    explicit Context(int device = -1)
    {
        if (cvvp_ctx_create(device, &m_ctx) != CVVP_OK)
            throw std::runtime_error(std::string("cvvidproc(" CVVP_HOST_VERSION "): ") + cvvp_last_error(nullptr));
    }
    ~Context() { cvvp_ctx_destroy(m_ctx); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    cvvp_ctx *get() const { return m_ctx; }
    void check(int rc) const
    {
        if (rc != CVVP_OK)
            throw std::runtime_error(std::string("cvvidproc(" CVVP_HOST_VERSION "): ") + cvvp_last_error(m_ctx));
    }

private:
    cvvp_ctx *m_ctx{nullptr};
};

// ---------------------------------------------------------------------------------------------------------------------
// temporal median: replaces HistogramMedianAlgo<T> (Sources/ProcessorAlgos/histogram_median_algo.h:41-222)
// ---------------------------------------------------------------------------------------------------------------------
struct GpuMedianPack {
    int device{-1};
    long long frames_hint{-1}; // frames_to_analyze of GetVideoBackground (cv_vid_bg_helpers.cpp:226-229)
    SourceFormat source{};     // enabled: InsertDecoded takes decoded frames
    int percent{50};           // the result is sorted[k(N, percent)] per element (cvvp_median_set_percentile)
};

class GpuMedianAlgo
{
public:
    using token_type = FrameBatch;
    using result_type = FrameBatch;
    explicit GpuMedianAlgo(GpuMedianPack pack) : m_pack{pack}, m_ctx{pack.device}
    {
        m_ctx.check(cvvp_median_set_percentile(m_ctx.get(), m_pack.percent));
    }

    // histogram_median_algo.h:66-87 -- null / empty tokens are skipped without counting
    void Insert(std::unique_ptr<FrameBatch> batch)
    {
        if (!batch || batch->empty())
            return;
        if (!m_started) {
            m_rows = batch->rows;
            m_cols = batch->cols;
            m_channels = batch->channels;
            m_ctx.check(cvvp_median_begin(m_ctx.get(), batch->frame_bytes(), m_pack.frames_hint));
            m_started = true;
        }
        CVVP_ASSERT_MSG(batch->rows == m_rows && batch->cols == m_cols && batch->channels == m_channels,
                        "all frames must have the geometry of the first one");
        m_ctx.check(cvvp_median_push(m_ctx.get(), batch->data.data(), batch->n, batch->frame_bytes()));
    }
    // raw form for callers that already hold the bytes (no extra copy)
    void InsertRaw(const std::uint8_t *frames, long long n, int rows, int cols, int channels, std::size_t stride)
    {
        if (!frames || n <= 0)
            return;
        if (!m_started) {
            m_rows = rows;
            m_cols = cols;
            m_channels = channels;
            m_ctx.check(cvvp_median_begin(m_ctx.get(), std::size_t(rows) * cols * channels, m_pack.frames_hint));
            m_started = true;
        }
        CVVP_ASSERT_MSG(rows == m_rows && cols == m_cols && channels == m_channels,
                        "all frames must have the geometry of the first one");
        m_ctx.check(cvvp_median_push(m_ctx.get(), frames, n, stride));
    }
    // decoded frames (rows x cols x channels of the decoder): cropped and channel-reduced on the device
    void InsertDecoded(const std::uint8_t *frames, long long n, std::size_t stride)
    {
        CVVP_ASSERT_MSG(m_pack.source.enabled, "InsertDecoded needs a SourceFormat in the pack");
        if (!frames || n <= 0)
            return;
        const SourceFormat &sf = m_pack.source;
        if (!m_started) {
            m_rows = sf.out_rows();
            m_cols = sf.out_cols();
            m_channels = sf.out_channels();
            m_ctx.check(cvvp_median_begin(m_ctx.get(), cvvp_frame_format_out_bytes(&sf.fmt), m_pack.frames_hint));
            m_started = true;
        }
        m_ctx.check(cvvp_median_push_source(m_ctx.get(), frames, n, stride, &sf.fmt));
    }
    // :101-108 -- end of stream: publish the result once, reset
    void NotifyNoMoreTokens()
    {
        if (!m_started)
            return;
        auto out = std::make_unique<FrameBatch>();
        out->n = 1;
        out->rows = m_rows;
        out->cols = m_cols;
        out->channels = m_channels;
        out->data.resize(out->frame_bytes());
        m_started = false;
        m_ctx.check(cvvp_median_finish(m_ctx.get(), out->data.data()));
        m_result = std::move(out);
    }
    std::unique_ptr<FrameBatch> TryGetResult() { return std::move(m_result); } // :90-98
    bool HasResults() const { return static_cast<bool>(m_result); }            // :110-113
    long long FramesInserted() const { return cvvp_median_count(m_ctx.get()); }

private:
    GpuMedianPack m_pack;
    Context m_ctx;
    bool m_started{false};
    int m_rows{0}, m_cols{0}, m_channels{1};
    std::unique_ptr<FrameBatch> m_result{};
};

// The same operator over SEVERAL devices of one process: tokens go to the devices in turn (the reference's analogue: the
// frame range of the video split over its generator threads, Sources/cv_vid_bg_helpers.cpp:84-120 -- the histogram is
// order-independent, so it does not matter which worker sees which frame), and the end of the stream runs the
// frame-sharded job of csrc/median_shard.cu with one rank per device: one pass of window counting with the count
// records written into the owner device's memory over NVLink, the two-round nibble exchange behind it when an element
// stayed undecided.  The barrier between phases is a synchronize of every context (all ranks live in this process).
class GpuShardedMedianAlgo
{
public:
    using token_type = FrameBatch;
    using result_type = FrameBatch;
    // percent: every device's context selects sorted[k(N, percent)] -- the ranks of one job must agree on it
    GpuShardedMedianAlgo(const std::vector<int> &devices, long long frames_hint, SourceFormat source, int percent = 50)
        : m_source{source}
    {
        CVVP_ASSERT_MSG(!devices.empty() && devices.size() <= 16, "1..16 devices");
        CVVP_ASSERT_MSG(source.enabled, "the multi-device median takes decoded frames");
        for (int d : devices) {
            m_ctx.push_back(std::make_unique<Context>(d));
            m_ctx.back()->check(cvvp_median_set_percentile(m_ctx.back()->get(), percent));
        }
        m_hint = frames_hint > 0 ? (frames_hint + (long long)devices.size() - 1) / (long long)devices.size() : -1;
    }
    // `turn` tokens in a row go to one device, then the next device takes over
    void InsertDecoded(const std::uint8_t *frames, long long n, std::size_t stride)
    {
        if (!frames || n <= 0)
            return;
        if (!m_started) {
            m_rows = m_source.out_rows();
            m_cols = m_source.out_cols();
            m_channels = m_source.out_channels();
            for (auto &c : m_ctx)
                c->check(cvvp_median_begin(c->get(), cvvp_frame_format_out_bytes(&m_source.fmt), m_hint));
            m_started = true;
        }
        Context &c = *m_ctx[std::size_t((m_inserted / kTurn) % (long long)m_ctx.size())];
        c.check(cvvp_median_push_source(c.get(), frames, n, stride, &m_source.fmt));
        m_inserted += n;
    }
    void NotifyNoMoreTokens()
    {
        if (!m_started)
            return;
        m_started = false;
        const int world = int(m_ctx.size());
        const std::size_t nelem = cvvp_frame_format_out_bytes(&m_source.fmt);
        std::vector<const std::uint8_t *> d_frames(m_ctx.size());
        std::vector<std::size_t> strides(m_ctx.size());
        std::vector<long long> counts(m_ctx.size());
        long long most = 1;
        for (int r = 0; r < world; ++r) {
            Context &c = *m_ctx[std::size_t(r)];
            c.check(cvvp_median_stack_device(c.get(), &d_frames[std::size_t(r)], &strides[std::size_t(r)], &counts[std::size_t(r)]));
            most = std::max(most, counts[std::size_t(r)]);
        }
        for (int r = 0; r < world; ++r)
            m_ctx[std::size_t(r)]->check(cvvp_median_shard_begin_frames(m_ctx[std::size_t(r)]->get(), nelem, r, world, most));
        for (int r = 0; r < world; ++r)
            for (int p = 0; p < world; ++p)
                if (p != r)
                    m_ctx[std::size_t(r)]->check(cvvp_median_shard_attach(m_ctx[std::size_t(r)]->get(), p, m_ctx[std::size_t(p)]->get()));
        auto walk = [&](int first, int last) {
            for (int phase = first; phase <= last; ++phase) {
                for (int r = 0; r < world; ++r)
                    m_ctx[std::size_t(r)]->check(cvvp_median_shard_phase(m_ctx[std::size_t(r)]->get(), phase, d_frames[std::size_t(r)],
                                                                         counts[std::size_t(r)], strides[std::size_t(r)], nullptr));
                for (auto &c : m_ctx) // the cross-rank barrier: every rank of this process has finished the phase
                    c->check(cvvp_ctx_synchronize(c->get()));
            }
        };
        walk(4, 5);
        long long undecided = 0;
        m_ctx[0]->check(cvvp_median_shard_unresolved(m_ctx[0]->get(), nullptr, &undecided));
        if (undecided != 0)
            walk(10, 13); // the two-round exchange over the tiles that hold an undecided element
        auto out = std::make_unique<FrameBatch>();
        out->n = 1;
        out->rows = m_rows;
        out->cols = m_cols;
        out->channels = m_channels;
        out->data.resize(out->frame_bytes());
        const std::uint8_t *d_res = nullptr;
        m_ctx[0]->check(cvvp_median_shard_result(m_ctx[0]->get(), &d_res));
        m_ctx[0]->check(cvvp_ctx_copy_to_host(m_ctx[0]->get(), out->data.data(), d_res, nelem));
        for (auto &c : m_ctx) {
            c->check(cvvp_median_shard_end(c->get()));
            c->check(cvvp_median_abort(c->get()));
        }
        m_result = std::move(out);
    }
    std::unique_ptr<FrameBatch> TryGetResult() { return std::move(m_result); }
    bool HasResults() const { return static_cast<bool>(m_result); }
    long long FramesInserted() const { return m_inserted; }
    static constexpr long long kTurn = 32;

private:
    SourceFormat m_source;
    std::vector<std::unique_ptr<Context>> m_ctx;
    long long m_hint{-1};
    bool m_started{false};
    long long m_inserted{0};
    int m_rows{0}, m_cols{0}, m_channels{1};
    std::unique_ptr<FrameBatch> m_result{};
};

// ---------------------------------------------------------------------------------------------------------------------
// highlight: replaces HighlightObjectsAlgo (Sources/ProcessorAlgos/highlight_objects_algo.h:21-107)
// ---------------------------------------------------------------------------------------------------------------------
struct GpuHighlightPack { // TokenProcessorPack<HighlightObjectsAlgo> :21-32
    int device{-1};
    FrameBatch background{};     // 1 frame of `channels` channels
    FrameBatch struct_element{}; // 1 "frame" of kh x kw bytes
    int threshold{}, threshold_lo{}, threshold_hi{}, min_size_hyst{}, min_size_threshold{}, width_border{};
    // opt-in extras (no counterpart in the reference's pack): 8-connected components of every mask for the tracker
    bool components{false};
    bool labels{false};
    bool component_stats{false}; // the records are cvvp_component_stats (cvvp_highlight_set_component_stats)
    int max_components{1024};
    // queue_depth > 0: tokens are processed asynchronously, at most queue_depth batches in flight (the reference's
    // token_storage_limit, Sources/AsyncTokens/token_queue.h:209-214) of at most max_batch frames each; results come
    // back in Insert order (mat_set_intermediary.h:50-68).  queue_depth == 0: Insert is synchronous.
    int queue_depth{0};
    long long max_batch{0};
    SourceFormat source{}; // enabled (queue mode only): tokens are DECODED frames, prepared on the device
    int polarity{CVVP_POLARITY_DARK}; // which difference image the masks start from (cvvp_highlight_set_polarity)
    int channels{1}; // channels of the frames and the background (cvvp_highlight_set_channels)
};

// What the two highlight operators below share: the job's parameters, the check of a token's geometry, and the
// batch their results are read into.
inline void begin_highlight(const Context &ctx, const GpuHighlightPack &p)
{
    CVVP_ASSERT(!p.background.empty());
    CVVP_ASSERT(!p.struct_element.empty());
    CVVP_ASSERT_MSG(p.background.channels == p.channels, "the background's channels must be the highlight stage's");
    ctx.check(cvvp_highlight_set_polarity(ctx.get(), p.polarity));
    ctx.check(cvvp_highlight_set_channels(ctx.get(), p.channels));
    ctx.check(cvvp_highlight_set_component_stats(ctx.get(), p.component_stats ? 1 : 0));
    ctx.check(cvvp_highlight_begin(ctx.get(), p.background.data.data(), p.background.cols, p.background.rows,
                                   p.struct_element.data.data(), p.struct_element.cols, p.struct_element.rows, p.threshold,
                                   p.threshold_lo, p.threshold_hi, p.min_size_hyst, p.min_size_threshold, p.width_border));
}

// tokens are decoded frames of the pack's source format, or prepared frames of the background's geometry
inline void check_token_geometry(const GpuHighlightPack &p, const FrameBatch &b)
{
    if (p.source.enabled)
        CVVP_ASSERT_MSG(b.rows == p.source.fmt.src_height && b.cols == p.source.fmt.src_width &&
                            b.channels == p.source.fmt.src_channels,
                        "decoded frame geometry must match the source format");
    else
        CVVP_ASSERT_MSG(b.channels == p.channels && b.rows == p.background.rows && b.cols == p.background.cols,
                        "frame geometry must match the background");
}

// room for max_batch frames of masks, with components and label images when the pack asks for them; the caller reads
// n frames into it and calls trim_result_batch
inline std::size_t record_bytes(const GpuHighlightPack &p)
{
    return p.component_stats ? sizeof(cvvp_component_stats) : sizeof(cvvp_component);
}

inline std::unique_ptr<FrameBatch> result_batch(const GpuHighlightPack &p)
{
    auto out = std::make_unique<FrameBatch>();
    out->rows = p.background.rows;
    out->cols = p.background.cols;
    out->channels = 1;
    out->data.resize(std::size_t(p.max_batch) * out->frame_bytes());
    if (p.components) {
        out->max_comps = p.max_components;
        out->rec_bytes = record_bytes(p);
        out->comps.resize(std::size_t(p.max_batch) * p.max_components * out->rec_bytes);
        out->ncomps.resize(std::size_t(p.max_batch));
        if (p.labels)
            out->labels.resize(std::size_t(p.max_batch) * out->frame_bytes());
    }
    return out;
}

inline void trim_result_batch(FrameBatch &out, long long n)
{
    out.n = int(n);
    out.data.resize(std::size_t(n) * out.frame_bytes());
    if (!out.labels.empty())
        out.labels.resize(std::size_t(n) * out.frame_bytes());
}

class GpuHighlightAlgo
{
public:
    using token_type = FrameBatch;
    using result_type = FrameBatch;
    explicit GpuHighlightAlgo(GpuHighlightPack pack) : m_pack{std::move(pack)}, m_ctx{m_pack.device}
    {
        begin_highlight(m_ctx, m_pack);
        if (m_pack.labels) // label images only travel through the synchronous entry point
            m_pack.queue_depth = 0;
        CVVP_ASSERT_MSG(m_pack.queue_depth > 0 || !m_pack.source.enabled, "decoded-frame tokens need the queue");
        if (m_pack.queue_depth > 0) {
            CVVP_ASSERT(m_pack.max_batch > 0);
            m_ctx.check(cvvp_highlight_queue_begin(m_ctx.get(), m_pack.queue_depth, m_pack.max_batch,
                                                   m_pack.source.enabled ? &m_pack.source.fmt : nullptr,
                                                   m_pack.components ? m_pack.max_components : 0));
        }
    }
    // highlight_objects_algo.h:60-69 -- the token is processed in place and becomes the result
    void Insert(std::unique_ptr<FrameBatch> batch)
    {
        if (!batch || batch->empty())
            return;
        check_token_geometry(m_pack, *batch);
        if (m_pack.queue_depth > 0) {
            // back-pressure: a full ring first gives up its oldest batch (the reference's TryInsert fails until a
            // result was taken, token_processing_unit.h:117-135)
            if (cvvp_highlight_queue_pending(m_ctx.get()) == m_pack.queue_depth)
                m_ready.push_back(take_next());
            m_ctx.check(cvvp_highlight_submit(m_ctx.get(), batch->data.data(), batch->n, batch->frame_bytes()));
            return; // the token's bytes were copied into the slot: it is dropped here like a consumed token
        }
        if (m_pack.components) {
            batch->max_comps = m_pack.max_components;
            batch->rec_bytes = record_bytes(m_pack);
            batch->comps.assign(std::size_t(batch->n) * m_pack.max_components * batch->rec_bytes, 0);
            batch->ncomps.assign(std::size_t(batch->n), 0);
            // a colour token's masks land in place at its frame stride; its labels are one int32 per pixel
            const std::size_t npix = std::size_t(batch->rows) * batch->cols;
            if (m_pack.labels)
                batch->labels.resize(std::size_t(batch->n) * npix);
            m_ctx.check(cvvp_highlight_frames_cc(m_ctx.get(), batch->data.data(), batch->n, batch->frame_bytes(),
                                                 batch->data.data(), batch->frame_bytes(), batch->component_records(),
                                                 m_pack.max_components, batch->ncomps.data(),
                                                 m_pack.labels ? batch->labels.data() : nullptr, npix));
        } else {
            m_ctx.check(cvvp_highlight_frames(m_ctx.get(), batch->data.data(), batch->n, batch->frame_bytes(),
                                              batch->data.data(), batch->frame_bytes()));
        }
        m_ready.push_back(std::move(batch));
    }
    int max_components() const { return m_pack.max_components; }
    // :72-79 -- null = none.  Queue mode: never blocks before NotifyNoMoreTokens (a batch still on the device is "no
    // result yet", exactly what a busy worker reports); after it, waits for what is pending, in order.
    std::unique_ptr<FrameBatch> TryGetResult()
    {
        if (!m_ready.empty()) {
            std::unique_ptr<FrameBatch> r = std::move(m_ready.front());
            m_ready.pop_front();
            return r;
        }
        if (m_pack.queue_depth > 0 && cvvp_highlight_queue_pending(m_ctx.get()) > 0) {
            const int ready = cvvp_highlight_queue_ready(m_ctx.get());
            if (ready < 0)
                m_ctx.check(ready);
            if (ready == 1 || m_no_more)
                return take_next();
        }
        return nullptr;
    }
    void NotifyNoMoreTokens() { m_no_more = true; } // :82-85 (tokens are independent; nothing is held back)

    // ---- zero-copy token path (queue mode): the token's storage is the queue slot's pinned memory ----
    // Where the reference's generator fills a fresh cv::Mat that then MOVES through the queues
    // (Sources/AsyncTokens/token_batch_generator.h:52-67), the decoder here writes its frames straight into the
    // slot AcquireSlot hands out, and the consumer reads the masks from the view NextView lends.
    struct Slot {
        std::uint8_t *frames{nullptr}; // frame i at frames + i * pitch (decoded frames with a SourceFormat, else prepared)
        std::size_t pitch{0};
        long long max_frames{0};
    };
    struct MaskView {
        const std::uint8_t *masks{nullptr}; // mask i at masks + i * pitch
        std::size_t pitch{0};
        long long n{0};
        const cvvp_component *comps{nullptr}; // [i * max_comps + k] records of record_bytes, null without components
        const int *ncomps{nullptr};
    };
    int Pending() const { return cvvp_highlight_queue_pending(m_ctx.get()); }
    int Depth() const { return m_pack.queue_depth; }
    bool Ready() const
    {
        const int r = cvvp_highlight_queue_ready(m_ctx.get());
        if (r < 0)
            m_ctx.check(r);
        return r == 1;
    }
    Slot AcquireSlot()
    {
        Slot s;
        m_ctx.check(cvvp_highlight_slot_acquire(m_ctx.get(), &s.frames, &s.pitch, &s.max_frames));
        return s;
    }
    void CommitSlot(long long n) { m_ctx.check(cvvp_highlight_slot_commit(m_ctx.get(), n)); }
    MaskView NextView() // blocks until the oldest pending batch is complete
    {
        MaskView v;
        m_ctx.check(cvvp_highlight_next_view(m_ctx.get(), &v.masks, &v.pitch, &v.n, &v.comps, &v.ncomps));
        return v;
    }
    void ReleaseView() { m_ctx.check(cvvp_highlight_view_release(m_ctx.get())); }
    int rows() const { return m_pack.background.rows; }
    int cols() const { return m_pack.background.cols; }

    bool HasResults() const { return !m_ready.empty() || (m_pack.queue_depth > 0 && cvvp_highlight_queue_pending(m_ctx.get()) > 0); } // :88-91

private:
    std::unique_ptr<FrameBatch> take_next()
    {
        auto out = result_batch(m_pack); // (queue mode has no label images)
        long long n = 0;
        m_ctx.check(cvvp_highlight_next(m_ctx.get(), out->data.data(), out->frame_bytes(), &n,
                                        m_pack.components ? out->component_records() : nullptr,
                                        m_pack.components ? out->ncomps.data() : nullptr));
        trim_result_batch(*out, n);
        return out;
    }

    GpuHighlightPack m_pack;
    Context m_ctx;
    std::deque<std::unique_ptr<FrameBatch>> m_ready{};
    bool m_no_more{false};
};

// ---------------------------------------------------------------------------------------------------------------------
// highlight against a rolling temporal-median background (no counterpart in the reference, whose background is static):
// frame t is compared with the percentile `percent` (the upper median at 50) of a window of `window` frames centred on
// it (cvvp_highlight_rolling_*).  The reference's four-method shape, but TryGetResult legitimately lags Insert: a
// frame's mask needs frames up to ceil(window / 2) - 1 ahead of it (window - 1 at the start), and the last ones only
// come after NotifyNoMoreTokens.
// The pack's background only sets the geometry.  Result batches are in frame order.
// ---------------------------------------------------------------------------------------------------------------------
class GpuRollingHighlightAlgo
{
public:
    using token_type = FrameBatch;
    using result_type = FrameBatch;
    // pack.max_batch: frames per Insert (at most); pack.source: tokens are DECODED frames, prepared on the device
    GpuRollingHighlightAlgo(GpuHighlightPack pack, int window, int percent = 50) : m_pack{std::move(pack)}, m_ctx{m_pack.device}
    {
        CVVP_ASSERT(m_pack.max_batch > 0);
        begin_highlight(m_ctx, m_pack);
        m_ctx.check(cvvp_median_set_percentile(m_ctx.get(), percent));
        m_ctx.check(cvvp_highlight_rolling_begin(m_ctx.get(), window, m_pack.max_batch,
                                                 m_pack.source.enabled ? &m_pack.source.fmt : nullptr,
                                                 m_pack.components ? m_pack.max_components : 0,
                                                 m_pack.components && m_pack.labels ? 1 : 0));
    }
    void Insert(std::unique_ptr<FrameBatch> batch)
    {
        if (!batch || batch->empty())
            return;
        check_token_geometry(m_pack, *batch);
        for (int done = 0; done < batch->n;) {
            const int k = int(std::min<long long>(batch->n - done, m_pack.max_batch));
            m_ctx.check(cvvp_highlight_rolling_push(m_ctx.get(), batch->data.data() + std::size_t(done) * batch->frame_bytes(), k,
                                                    batch->frame_bytes()));
            done += k;
        }
    }
    // null = none yet.  Before NotifyNoMoreTokens only a batch that is complete on the device is returned; after it,
    // waits for what is pending, in order.
    std::unique_ptr<FrameBatch> TryGetResult()
    {
        if (cvvp_highlight_rolling_pending(m_ctx.get()) == 0)
            return nullptr;
        const int ready = cvvp_highlight_rolling_ready(m_ctx.get());
        if (ready < 0)
            m_ctx.check(ready);
        if (ready == 0 && !m_no_more)
            return nullptr;
        auto out = result_batch(m_pack);
        long long first = 0, n = 0;
        m_ctx.check(cvvp_highlight_rolling_next(m_ctx.get(), out->data.data(), out->frame_bytes(), m_pack.max_batch, &first, &n,
                                                m_pack.components ? out->component_records() : nullptr,
                                                m_pack.components ? out->ncomps.data() : nullptr,
                                                out->labels.empty() ? nullptr : out->labels.data(), out->frame_bytes()));
        CVVP_ASSERT_MSG(first == m_returned, "rolling highlight results out of order");
        m_returned += n;
        trim_result_batch(*out, n);
        return out;
    }
    // end of the stream: the last frames' windows clamp to the frames inserted
    void NotifyNoMoreTokens()
    {
        if (m_no_more)
            return;
        m_no_more = true;
        m_ctx.check(cvvp_highlight_rolling_close(m_ctx.get()));
    }
    bool HasResults() const { return cvvp_highlight_rolling_pending(m_ctx.get()) > 0; }
    int max_components() const { return m_pack.max_components; }

private:
    GpuHighlightPack m_pack;
    Context m_ctx;
    bool m_no_more{false};
    long long m_returned{0};
};
} // namespace cvvp_host
