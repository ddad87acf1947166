// pybind11 module `_core`: the reference's Python surface (Sources/py_bindings.cpp:26-131) on top of the C++ host
// operators (gpu_algos.hpp) and the C ABI.  Same class names, argument names, order and defaults; same observable
// behaviour of the two entry points:
//
//   GetVideoBackground(pack) -> ndarray | None     Sources/cv_vid_bg_helpers.cpp:197-264
//   TrackObjects(pack)       -> dict               Sources/cv_vid_objecttrack_helpers.cpp:153-210
//
// OpenCV C++ is not part of this build, so the numpy<->cv::Mat caster (Sources/Utility/ndarray_converter.*) is replaced
// by py::array_t<uint8_t>, and video decode goes through the Python `cv2` module (the only decoder in the image),
// reproducing CvVidFramesGeneratorAlgo::GetTokenSet (ProcessorTokenHandlers/cv_vid_frames_generator_algo.h:120-185):
// crop, then channel 0 (vid_is_grayscale) or RGB2GRAY (grayscale) or the frame as is.  That per-frame work runs on the
// DEVICE (csrc/frames.cu): the decoded frame is handed over untouched together with a SourceFormat.  CVVP_HOST_PREP=1
// keeps it on the host through cv2 instead (cross-check; tests hold the two to each other).
//
// TrackObjects is a pipeline like the reference's (decode thread || highlight process || assign process,
// cv_vid_objecttrack_helpers.cpp:71-133): a C++ decode thread (the reference's generator thread, :71-93) takes the GIL
// only around VideoCapture.read -- which drops it again while it decodes -- and writes every frame straight into the
// pinned input slot of the device queue; the calling thread submits the filled slots (at most token_storage_limit in
// flight per device), and runs the tracker callback on the masks that have come back, strictly in frame order, reading
// them from the queue's pinned output.  CVVP_DEVICES=0,1,... spreads the batches over several GPUs round-robin; the
// masks are still handed over in frame order (the MatSetIntermediary role, mat_set_intermediary.h:50-68,84-114).
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdlib>
#include <deque>
#include <functional>
#include <iostream>
#include <limits>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>

#include "gpu_algos.hpp"

namespace py = pybind11;
using namespace cvvp_host;

namespace
{
using u8array = py::array_t<std::uint8_t, py::array::c_style | py::array::forcecast>;

// ---- packs (plain data, only __init__ is exposed, like the reference) -------------------------------------------------
struct VidBgPack { // cv_vid_bg_helpers.h:30-60
    std::string vid_path;
    std::string bg_algo;
    int max_threads;
    long long frame_limit;
    bool grayscale;
    bool vid_is_grayscale;
    int crop_x, crop_y, crop_width, crop_height;
    int token_storage_limit;
    bool print_timing_report;
};

struct HighlightObjectsPack { // highlight_objects_algo.h:21-32
    py::array background;
    py::array struct_element;
    int threshold, threshold_lo, threshold_hi, min_size_hyst, min_size_threshold, width_border;
};

struct AssignObjectsPack { // assign_objects_algo.h:28-44
    py::function function;
    py::dict kwargs;
};

struct VidObjectTrackPack { // cv_vid_objecttrack_helpers.h:23-60
    std::string vid_path;
    HighlightObjectsPack highlight_objects_pack;
    AssignObjectsPack assign_objects_pack;
    int max_threads;
    long long start_frame;
    long long frame_limit;
    bool grayscale;
    bool vid_is_grayscale;
    int crop_x, crop_y, crop_width, crop_height;
    int token_storage_limit;
    bool print_timing_report;
};

struct Rect {
    int x, y, width, height;
};

// cv_vid_bg_helpers.cpp:39-60 -- including its quirk: the height clamp compares against hor_pixels (:56)
Rect GetCroppedFrameDims(int x, int y, int width, int height, int hor_pixels, int vert_pixels)
{
    CVVP_ASSERT(x >= 0);
    CVVP_ASSERT(y >= 0);
    CVVP_ASSERT(width >= 0);
    CVVP_ASSERT(height >= 0);
    CVVP_ASSERT_MSG(hor_pixels > 0, "frame must have horizontal size");
    CVVP_ASSERT_MSG(vert_pixels > 0, "frame must have verical size");
    CVVP_ASSERT_MSG(x < hor_pixels, "start of crop window can't be outside frame");
    CVVP_ASSERT_MSG(y < vert_pixels, "start of crop window can't be outside frame");
    if (width == 0 || width + x > hor_pixels)
        width = hor_pixels - x;
    if (height == 0 || height + y > hor_pixels)
        height = vert_pixels - y;
    return Rect{x, y, width, height};
}

// One decoded, cropped, channel-reduced frame as a contiguous uint8 array (H, W) or (H, W, C).
// Mirrors CvVidFramesGeneratorAlgo::GetTokenSet (:137-156).  Returns an empty object at end of stream.
class FrameSource
{
public:
    FrameSource(const std::string &path, bool grayscale, bool vid_is_grayscale)
        : m_cv2{py::module_::import("cv2")}, m_np{py::module_::import("numpy")}, m_gray{grayscale}, m_is_gray{vid_is_grayscale}
    {
        m_vid = m_cv2.attr("VideoCapture")(path);
    }
    bool opened() const { return m_vid.attr("isOpened")().cast<bool>(); }
    double get(const char *prop) const { return m_vid.attr("get")(m_cv2.attr(prop)).cast<double>(); }
    void set(const char *prop, double v) { m_vid.attr("set")(m_cv2.attr(prop), v); }
    void set_crop(Rect r) { m_crop = r; }
    void configure()
    {
        // :103-105 interpret frames as RGB for consistency unless the video is declared grayscale
        if (!m_is_gray)
            set("CAP_PROP_CONVERT_RGB", 1.0);
    }
    // the decoded frame as the decoder produced it (contiguous uint8), or None at end of stream
    py::object next_decoded()
    {
        py::tuple res = m_vid.attr("read")().cast<py::tuple>();
        if (!res[0].cast<bool>() || res[1].is_none())
            return py::none();
        return m_np.attr("ascontiguousarray")(res[1], py::arg("dtype") = m_np.attr("uint8"));
    }
    // Decode the next frame INTO dst (rows x cols x channels contiguous bytes: a queue slot, a pinned buffer); false at
    // end of stream.  VideoCapture.read(image) reuses a matching array, so the decoder's copy-out is the only write.
    bool read_into(std::uint8_t *dst, int rows, int cols, int channels)
    {
        std::vector<py::ssize_t> shape{rows, cols};
        if (channels > 1)
            shape.push_back(channels);
        py::array_t<std::uint8_t> view(shape, dst, m_np); // a base object: the array is a view, not a copy
        py::tuple res = m_vid.attr("read")(view).cast<py::tuple>();
        if (!res[0].cast<bool>() || res[1].is_none())
            return false;
        py::array out = res[1].cast<py::array>();
        if (out.data() != static_cast<const void *>(dst)) { // the decoder allocated its own array (geometry changed?)
            py::array c = m_np.attr("ascontiguousarray")(out, py::arg("dtype") = m_np.attr("uint8")).cast<py::array>();
            CVVP_ASSERT_MSG(std::size_t(c.nbytes()) == std::size_t(rows) * cols * channels,
                            "all frames must have the geometry of the first one");
            std::memcpy(dst, c.data(), std::size_t(c.nbytes()));
        }
        return true;
    }
    // what the device has to do with a decoded frame of `channels` channels (:141-156)
    SourceFormat format_for(int rows, int cols, int channels) const
    {
        // cv::cvtColor(COLOR_RGB2GRAY) throws on anything but 3 or 4 channels (:152-154)
        CVVP_ASSERT_MSG(!(m_gray && !m_is_gray && channels < 3),
                        "grayscale conversion needs a 3- or 4-channel frame (cv::cvtColor COLOR_RGB2GRAY)");
        SourceFormat sf;
        sf.enabled = true;
        sf.fmt.src_width = cols;
        sf.fmt.src_height = rows;
        sf.fmt.src_channels = channels;
        sf.fmt.crop_x = m_crop.x;
        sf.fmt.crop_y = m_crop.y;
        sf.fmt.crop_width = m_crop.width;
        sf.fmt.crop_height = m_crop.height;
        if (m_is_gray)
            sf.fmt.mode = CVVP_FRAMES_CHANNEL0; // :149-151
        else if (m_gray && channels >= 3)
            sf.fmt.mode = CVVP_FRAMES_RGB2GRAY; // :152-154
        else
            sf.fmt.mode = CVVP_FRAMES_AS_IS; // :155-156
        return sf;
    }
    py::object next()
    {
        py::tuple res = m_vid.attr("read")().cast<py::tuple>();
        if (!res[0].cast<bool>() || res[1].is_none())
            return py::none();
        py::object frame = res[1];
        // :141 crop
        frame = frame[py::make_tuple(py::slice(m_crop.y, m_crop.y + m_crop.height, 1),
                                     py::slice(m_crop.x, m_crop.x + m_crop.width, 1))];
        const int ndim = frame.attr("ndim").cast<int>();
        if (m_is_gray) {
            if (ndim == 3)
                frame = m_cv2.attr("extractChannel")(frame, 0); // :149-151
        } else if (m_gray) {
            frame = m_cv2.attr("cvtColor")(frame, m_cv2.attr("COLOR_RGB2GRAY")); // :152-154 (throws on < 3 channels)
        }
        return m_np.attr("ascontiguousarray")(frame, py::arg("dtype") = m_np.attr("uint8"));
    }

private:
    py::module_ m_cv2, m_np;
    py::object m_vid;
    bool m_gray, m_is_gray;
    Rect m_crop{0, 0, 0, 0};
};

bool host_prep()
{
    const char *e = std::getenv("CVVP_HOST_PREP");
    return e && *e && *e != '0';
}

void array_geometry(const py::array &a, int &rows, int &cols, int &channels)
{
    CVVP_ASSERT_MSG(a.ndim() == 2 || a.ndim() == 3, "frames must be 2-D or 3-D uint8 arrays");
    rows = int(a.shape(0));
    cols = int(a.shape(1));
    channels = a.ndim() == 3 ? int(a.shape(2)) : 1;
}

// print_timing_report: the reference's report lines (AsyncTokenProcess::GetTimingInfoAndResetTimer,
// Sources/AsyncTokens/async_token_process.h:273-414; whole milliseconds like its default TimingReportUnitT).  The
// roles map as: batch generator = the decode loop, unit [1] = the device operator's Insert, consumer = result hand-off.
struct IntervalTimer {
    std::chrono::steady_clock::duration total{};
    long long count{0};
    std::chrono::steady_clock::time_point t0{};
    void start() { t0 = std::chrono::steady_clock::now(); }
    void stop()
    {
        total += std::chrono::steady_clock::now() - t0;
        ++count;
    }
    long long ms() const { return std::chrono::duration_cast<std::chrono::milliseconds>(total).count(); }
    long long avg_ms() const { return count ? std::chrono::duration_cast<std::chrono::milliseconds>(total / count).count() : 0; }
};

std::string timing_report(const IntervalTimer &batches, const IntervalTimer &gen, const IntervalTimer &consume,
                          const IntervalTimer &unit)
{
    if (!batches.count)
        return "";
    std::ostringstream ss;
    ss << "Batch loading: " << batches.ms() << " ms (" << batches.count << " batches; " << batches.avg_ms()
       << " ms avg) on time between each generated batch\n";
    ss << "Batch gen: " << gen.ms() << " ms (" << gen.count << " batches; " << gen.avg_ms() << " ms avg) on generating batches\n";
    ss << "Result consume: " << consume.ms() << " ms (" << consume.count << " tokens; " << consume.avg_ms()
       << " ms avg) on handling results\n";
    if (unit.count)
        ss << "Unit [1]: " << unit.ms() << " ms (" << unit.count << " tokens; " << unit.avg_ms()
           << " ms avg) on ingesting tokens in workers\n";
    return ss.str();
}

// CVVP_DEVICES=0,1,...: the CUDA devices the two entry points spread their work over (default: the current device)
std::vector<int> device_list()
{
    std::vector<int> out;
    if (const char *e = std::getenv("CVVP_DEVICES")) {
        std::stringstream ss{std::string(e)};
        std::string tok;
        while (std::getline(ss, tok, ','))
            if (!tok.empty())
                out.push_back(std::atoi(tok.c_str()));
    }
    if (out.empty())
        out.push_back(-1);
    return out;
}

// page-locked host buffer (cvvp_host_alloc): a decoded frame written here goes to the device without staging
struct PinnedBuffer {
    std::uint8_t *p{nullptr};
    explicit PinnedBuffer(std::size_t bytes)
    {
        void *q = nullptr;
        if (cvvp_host_alloc(bytes, &q) != CVVP_OK)
            throw std::runtime_error(std::string("cvvidproc(" CVVP_HOST_VERSION "): ") + cvvp_last_error(nullptr));
        p = static_cast<std::uint8_t *>(q);
    }
    ~PinnedBuffer() { cvvp_host_free(p); }
    PinnedBuffer(const PinnedBuffer &) = delete;
    PinnedBuffer &operator=(const PinnedBuffer &) = delete;
};

// The decode thread (the reference's generator thread, cv_vid_objecttrack_helpers.cpp:71-93): it is handed storage for
// a batch of frames and fills it with VideoCapture.read, taking the GIL frame by frame (cv2 drops it while decoding,
// so the tracker callback on the calling thread and the decoder run side by side).
class DecodeWorker
{
public:
    struct Job {
        std::uint8_t *dst;
        std::size_t pitch;
        long long max_frames, prefilled;
    };
    struct Done {
        long long n{0};
        bool eof{false};
        std::string error;
    };
    DecodeWorker(FrameSource &vid, int rows, int cols, int channels, long long frames_left)
        : m_vid{vid}, m_rows{rows}, m_cols{cols}, m_channels{channels}, m_left{frames_left}
    {
        m_thread = std::thread([this] { run(); });
    }
    ~DecodeWorker() // callers hold the GIL or not: the worker never blocks on it while stopping
    {
        {
            std::lock_guard<std::mutex> lk(m_mu);
            m_stop = true;
        }
        m_cv.notify_all();
        if (m_thread.joinable()) {
            py::gil_scoped_release nogil; // a read in flight needs the GIL to finish
            m_thread.join();
        }
    }
    void push(const Job &j)
    {
        {
            std::lock_guard<std::mutex> lk(m_mu);
            m_jobs.push_back(j);
        }
        m_cv.notify_all();
    }
    // a finished batch, if any; waits up to `wait_us` for one (call without the GIL when waiting)
    bool pop(Done &d, long long wait_us)
    {
        std::unique_lock<std::mutex> lk(m_mu);
        if (m_done.empty() && wait_us > 0)
            m_cv_done.wait_for(lk, std::chrono::microseconds(wait_us), [this] { return !m_done.empty(); });
        if (m_done.empty())
            return false;
        d = std::move(m_done.front());
        m_done.pop_front();
        return true;
    }

    // where the decode thread's time went (developer aid, CVVP_TRACK_DEBUG): inside VideoCapture.read, waiting for the
    // GIL, waiting for a slot to fill
    std::chrono::steady_clock::duration t_read{}, t_gil_wait{}, t_job_wait{};
    // is the decode thread waiting for the GIL right now?  The calling thread hands it over between tracker callbacks:
    // CPython switches a thread that holds the GIL out only after its switch interval (5 ms), which would leave the
    // decoder idle after every frame while a batch of callbacks runs.
    bool wants_gil() const { return m_wants_gil.load(std::memory_order_acquire); }
    // waits up to `wait_us` for a finished batch without taking it (call without the GIL)
    void wait_done(long long wait_us)
    {
        std::unique_lock<std::mutex> lk(m_mu);
        if (m_done.empty())
            m_cv_done.wait_for(lk, std::chrono::microseconds(wait_us), [this] { return !m_done.empty(); });
    }

private:
    void run()
    {
        for (;;) {
            Job j;
            {
                const auto tj = std::chrono::steady_clock::now();
                std::unique_lock<std::mutex> lk(m_mu);
                m_cv.wait(lk, [this] { return m_stop || !m_jobs.empty(); });
                if (m_stop)
                    return;
                j = m_jobs.front();
                m_jobs.pop_front();
                t_job_wait += std::chrono::steady_clock::now() - tj;
            }
            Done d;
            d.n = j.prefilled;
            while (d.n < j.max_frames && m_left > 0 && !d.eof) {
                {
                    std::lock_guard<std::mutex> lk(m_mu);
                    if (m_stop)
                        return;
                }
                const auto tw = std::chrono::steady_clock::now();
                m_wants_gil.store(true, std::memory_order_release);
                py::gil_scoped_acquire gil;
                m_wants_gil.store(false, std::memory_order_release);
                const auto tr = std::chrono::steady_clock::now();
                t_gil_wait += tr - tw;
                struct Stop {
                    std::chrono::steady_clock::duration &acc;
                    std::chrono::steady_clock::time_point t0;
                    ~Stop() { acc += std::chrono::steady_clock::now() - t0; }
                } stop{t_read, tr};
                try {
                    if (m_vid.read_into(j.dst + std::size_t(d.n) * j.pitch, m_rows, m_cols, m_channels)) {
                        ++d.n;
                        --m_left;
                    } else {
                        d.eof = true;
                    }
                } catch (py::error_already_set &e) {
                    d.error = e.what();
                    d.eof = true;
                } catch (const std::exception &e) {
                    d.error = e.what();
                    d.eof = true;
                }
            }
            if (m_left <= 0)
                d.eof = true;
            {
                std::lock_guard<std::mutex> lk(m_mu);
                m_done.push_back(std::move(d));
            }
            m_cv_done.notify_all();
        }
    }
    FrameSource &m_vid;
    int m_rows, m_cols, m_channels;
    long long m_left;
    std::thread m_thread;
    std::mutex m_mu;
    std::condition_variable m_cv, m_cv_done;
    std::deque<Job> m_jobs;
    std::deque<Done> m_done;
    bool m_stop{false};
    std::atomic<bool> m_wants_gil{false};
};

// ---------------------------------------------------------------------------------------------------------------------
// GetVideoBackground  (cv_vid_bg_helpers.cpp:197-264)
// ---------------------------------------------------------------------------------------------------------------------
// The background algorithm names GetVideoBackground accepts (GetBGAlgo, cv_vid_bg_helpers.cpp:27-37): the reference's
// "hist" (the upper median), and "cvvp_percentile:P" -- P an integer percent written without leading zeros, 0..100 --,
// the same histogram path selecting sorted[k(N, P)] (cvvp_median_set_percentile).  false: an unknown algorithm.
bool background_percent(const std::string &algo, int *percent)
{
    if (algo == "hist") {
        *percent = 50;
        return true;
    }
    static const std::string prefix = "cvvp_percentile:";
    if (algo.compare(0, prefix.size(), prefix) != 0)
        return false;
    const std::string digits = algo.substr(prefix.size());
    if (digits.empty() || digits.size() > 3 || (digits.size() > 1 && digits[0] == '0'))
        return false;
    int v = 0;
    for (char c : digits) {
        if (c < '0' || c > '9')
            return false;
        v = v * 10 + (c - '0');
    }
    if (v > 100)
        return false;
    *percent = v;
    return true;
}

py::object GetVideoBackground(const VidBgPack &pack)
{
    FrameSource vid{pack.vid_path, pack.grayscale, pack.vid_is_grayscale};
    if (!vid.opened()) {
        std::cerr << "Video file not detected: " << pack.vid_path << '\n';
        return py::none(); // the reference returns an empty Mat, which its caster turns into None
    }
    const long long total_frames = static_cast<long long>(vid.get("CAP_PROP_FRAME_COUNT"));
    const double fw = vid.get("CAP_PROP_FRAME_WIDTH"), fh = vid.get("CAP_PROP_FRAME_HEIGHT");
    std::cout << "Frames: " << total_frames << "; Res: " << fw << 'x' << fh; // :212-223
    if (pack.crop_x || pack.crop_y || pack.crop_width || pack.crop_height) {
        const Rect r = GetCroppedFrameDims(pack.crop_x, pack.crop_y, pack.crop_width, pack.crop_height, int(fw), int(fh));
        std::cout << "(" << r.width << 'x' << r.height << " cropped)";
    }
    std::cout << "; FPS: " << vid.get("CAP_PROP_FPS") << '\n';
    std::cout.flush();

    long long frames_to_analyze = pack.frame_limit; // :226-229
    if (frames_to_analyze <= 0 || frames_to_analyze > total_frames)
        frames_to_analyze = total_frames;

    int percent = 50;
    if (!background_percent(pack.bg_algo, &percent)) { // GetBGAlgo :27-37 + the switch default :255-260
        std::cerr << "Unknown background algorithm detected: " << pack.bg_algo << '\n';
        std::cerr << "tried to get vid background with unknown algorithm: " << pack.bg_algo << '\n';
        return py::none();
    }
    if (frames_to_analyze > static_cast<long long>(std::numeric_limits<std::uint32_t>::max())) { // :249-260 falls through
        std::cerr << "warning, video appears to have over 2^32 frames! (" << total_frames << ") is way too many!\n";
        std::cerr << "tried to get vid background with unknown algorithm: " << pack.bg_algo << '\n';
        return py::none();
    }

    const Rect crop = GetCroppedFrameDims(pack.crop_x, pack.crop_y, pack.crop_width, pack.crop_height, int(fw), int(fh));
    CVVP_ASSERT(crop.x + crop.width <= int(fw) && crop.y + crop.height <= int(fh)); // generator ctor :90-92
    vid.set_crop(crop);
    vid.configure();

    // The reference releases the GIL for this whole call (py_bindings.cpp:63-66).  Here the decoder is Python's cv2, which
    // needs the GIL to be CALLED but drops it while it decodes; everything else that takes time -- the uploads, the
    // device frame preparation, the select at the end -- runs with the GIL released, so other Python threads make
    // progress throughout.
    const bool on_device = !host_prep();
    const std::vector<int> devices = device_list();
    std::unique_ptr<GpuMedianAlgo> algo_p; // built once the first decoded frame tells the channel count
    std::unique_ptr<GpuShardedMedianAlgo> sharded_p; // CVVP_DEVICES names several devices
    std::unique_ptr<PinnedBuffer> pinned;  // the decoder writes every frame here: no fresh array, no staging copy
    long long consumed = 0;
    int rows = 0, cols = 0, channels = 1;
    IntervalTimer t_batch, t_gen, t_unit, t_consume;
    while (consumed < frames_to_analyze) { // generator :128-135
        t_batch.start();
        t_gen.start();
        const std::uint8_t *data = nullptr;
        py::object keep; // keeps the decoded array alive until it has been pushed
        if (on_device && pinned) {
            if (!vid.read_into(pinned->p, rows, cols, channels)) {
                t_gen.stop();
                break;
            }
            data = pinned->p;
        } else {
            keep = on_device ? vid.next_decoded() : vid.next();
            if (keep.is_none()) {
                t_gen.stop();
                break;
            }
            py::array a = keep.cast<py::array>();
            array_geometry(a, rows, cols, channels);
            data = static_cast<const std::uint8_t *>(a.data());
        }
        t_gen.stop();
        if (!algo_p && !sharded_p) {
            if (on_device && devices.size() > 1) {
                sharded_p = std::make_unique<GpuShardedMedianAlgo>(devices, frames_to_analyze, vid.format_for(rows, cols, channels),
                                                                   percent);
            } else {
                GpuMedianPack mp{devices[0], frames_to_analyze, {}, percent};
                if (on_device)
                    mp.source = vid.format_for(rows, cols, channels);
                algo_p = std::make_unique<GpuMedianAlgo>(mp);
            }
        }
        t_unit.start();
        if (on_device) {
            CVVP_ASSERT(rows == int(fh) && cols == int(fw));
            const std::size_t bytes = std::size_t(rows) * cols * channels;
            {
                py::gil_scoped_release nogil;
                if (sharded_p)
                    sharded_p->InsertDecoded(data, 1, bytes);
                else
                    algo_p->InsertDecoded(data, 1, bytes);
            }
            if (!pinned)
                pinned = std::make_unique<PinnedBuffer>(bytes);
        } else {
            py::gil_scoped_release nogil;
            algo_p->InsertRaw(data, 1, rows, cols, channels, std::size_t(rows) * cols * channels);
        }
        t_unit.stop();
        t_batch.stop();
        ++consumed;
    }
    t_consume.start();
    std::unique_ptr<FrameBatch> res;
    {
        py::gil_scoped_release nogil;
        if (sharded_p) {
            sharded_p->NotifyNoMoreTokens();
            res = sharded_p->TryGetResult();
        } else if (algo_p) {
            algo_p->NotifyNoMoreTokens();
            res = algo_p->TryGetResult();
        }
    }
    t_consume.stop();
    if (pack.print_timing_report) // cv_vid_bg_helpers.cpp:154-155: printed inside VidBackgroundWithAlgo, result or not
        std::cout << timing_report(t_batch, t_gen, t_consume, t_unit);
    if (!res || res->empty())
        return py::none();
    // shape (H, W) for one channel, (H, W, C) otherwise (ndarray_converter.cpp:141-142)
    std::vector<py::ssize_t> shape{res->rows, res->cols};
    if (res->channels > 1)
        shape.push_back(res->channels);
    py::array_t<std::uint8_t> out(shape);
    std::memcpy(out.mutable_data(), res->data.data(), res->data.size());
    return std::move(out);
}

// ---------------------------------------------------------------------------------------------------------------------
// TrackObjects  (cv_vid_objecttrack_helpers.cpp:153-210, :30-150; assign_objects_algo.h:94-161)
// ---------------------------------------------------------------------------------------------------------------------
// with_channels: an (h, w, C) array is accepted too (a colour background)
FrameBatch to_u8_image(const py::array &src, const char *what, bool with_channels = false)
{
    CVVP_ASSERT_MSG(src.size() > 0, what);
    CVVP_ASSERT_MSG(src.ndim() == 2 || (with_channels && src.ndim() == 3), "expected a 2-D array");
    CVVP_ASSERT_MSG(src.dtype().is(py::dtype::of<std::uint8_t>()), "expected a uint8 array (OpenCV asserts CV_8U here)");
    u8array a = u8array::ensure(src);
    FrameBatch b;
    b.n = 1;
    b.rows = int(a.shape(0));
    b.cols = int(a.shape(1));
    b.channels = a.ndim() == 3 ? int(a.shape(2)) : 1;
    b.data.assign(a.data(), a.data() + a.size());
    return b;
}

// kwargs["cvvp_background_window"]: 0 when absent, else an int in [1, 65535] (RuntimeError otherwise)
int background_window(const py::dict &kwargs)
{
    if (!kwargs.contains("cvvp_background_window"))
        return 0;
    py::object w = kwargs["cvvp_background_window"];
    bool ok = PyIndex_Check(w.ptr()) && !PyBool_Check(w.ptr());
    long long v = 0;
    if (ok) {
        int overflow = 0;
        py::int_ iw = py::reinterpret_steal<py::int_>(PyNumber_Index(w.ptr()));
        v = PyLong_AsLongLongAndOverflow(iw.ptr(), &overflow);
        ok = overflow == 0 && v >= 1 && v <= 65535;
    }
    CVVP_ASSERT_MSG(ok, "kwargs['cvvp_background_window'] must be an int in [1, 65535]");
    return int(v);
}

// kwargs["cvvp_background_percentile"]: 50 when absent, else an int (not a bool) in [0, 100] -- and only together with a
// window: the static path computes no background (RuntimeError otherwise)
int background_percentile(const py::dict &kwargs)
{
    if (!kwargs.contains("cvvp_background_percentile"))
        return 50;
    CVVP_ASSERT_MSG(kwargs.contains("cvvp_background_window"),
                    "kwargs['cvvp_background_percentile'] needs kwargs['cvvp_background_window']: only the rolling "
                    "background has a percentile");
    py::object p = kwargs["cvvp_background_percentile"];
    bool ok = PyIndex_Check(p.ptr()) && !PyBool_Check(p.ptr());
    long long v = 0;
    if (ok) {
        int overflow = 0;
        py::int_ ip = py::reinterpret_steal<py::int_>(PyNumber_Index(p.ptr()));
        v = PyLong_AsLongLongAndOverflow(ip.ptr(), &overflow);
        ok = overflow == 0 && v >= 0 && v <= 100;
    }
    CVVP_ASSERT_MSG(ok, "kwargs['cvvp_background_percentile'] must be an int in [0, 100]");
    return int(v);
}

// kwargs["cvvp_polarity"]: CVVP_POLARITY_DARK when absent, else exactly the str "dark", "bright" or "both"
// (RuntimeError otherwise)
int object_polarity(const py::dict &kwargs)
{
    if (!kwargs.contains("cvvp_polarity"))
        return CVVP_POLARITY_DARK;
    py::object v = kwargs["cvvp_polarity"];
    int polarity = -1;
    if (PyUnicode_Check(v.ptr())) {
        const std::string name = v.cast<std::string>();
        polarity = name == "dark" ? CVVP_POLARITY_DARK
                 : name == "bright" ? CVVP_POLARITY_BRIGHT
                 : name == "both" ? CVVP_POLARITY_BOTH : -1;
    }
    CVVP_ASSERT_MSG(polarity >= 0, "kwargs['cvvp_polarity'] must be \"dark\", \"bright\" or \"both\"");
    return polarity;
}

// kwargs["cvvp_component_stats"]: false when absent, else exactly a bool; True needs kwargs["cvvp_components"] = True
bool component_stats(const py::dict &kwargs)
{
    if (!kwargs.contains("cvvp_component_stats"))
        return false;
    py::object v = kwargs["cvvp_component_stats"];
    CVVP_ASSERT_MSG(py::isinstance<py::bool_>(v), "kwargs['cvvp_component_stats'] must be True or False");
    const bool on = v.cast<bool>();
    CVVP_ASSERT_MSG(!on || (kwargs.contains("cvvp_components") && kwargs["cvvp_components"].cast<bool>()),
                    "kwargs['cvvp_component_stats'] needs kwargs['cvvp_components'] = True");
    return on;
}

// kwargs["cvvp_color"]: false when absent, else exactly a bool; True keeps every channel of the decoded frames, so it
// cannot go with grayscale or vid_is_grayscale (RuntimeError otherwise)
bool color_frames(const py::dict &kwargs, bool grayscale, bool vid_is_grayscale)
{
    if (!kwargs.contains("cvvp_color"))
        return false;
    py::object v = kwargs["cvvp_color"];
    CVVP_ASSERT_MSG(py::isinstance<py::bool_>(v), "kwargs['cvvp_color'] must be True or False");
    const bool on = v.cast<bool>();
    CVVP_ASSERT_MSG(!on || (!grayscale && !vid_is_grayscale),
                    "kwargs['cvvp_color'] = True uses the decoded frames' channels: it cannot go with grayscale or "
                    "vid_is_grayscale");
    return on;
}

py::dict TrackObjects(const VidObjectTrackPack &pack)
{
    // Opt-in extra of this implementation (the reference has no counterpart): kwargs["cvvp_background_window"] = W
    // compares frame t with the rolling upper median of a window of W frames centred on it (shifted, not shortened,
    // at both ends of the processed frames; cvvp_median_rolling_device) instead of the pack's background, which is
    // then only validated (non-empty, the cropped frame's size) and not used for the masks.  Checked before any
    // device work.  The masks reach the callback in frame order as always, but later than their frames are decoded
    // (up to W - 1 frames).  With several devices in CVVP_DEVICES this mode runs on the first one.
    // kwargs["cvvp_background_percentile"] = P (with a window) makes that background the window's percentile P instead
    // of its upper median (P = 50).
    const int roll_window = background_window(pack.assign_objects_pack.kwargs);
    const int roll_percent = background_percentile(pack.assign_objects_pack.kwargs);
    // kwargs["cvvp_polarity"] = "bright" finds objects brighter than the background (d = max(frame - bg, 0)), "both"
    // objects on either side (d = |frame - bg|); "dark", the default, is the reference's d = max(bg - frame, 0).
    const int polarity = object_polarity(pack.assign_objects_pack.kwargs);
    // kwargs["cvvp_component_stats"] = True (with cvvp_components) adds shape and contrast statistics to `components`
    const bool want_stats = component_stats(pack.assign_objects_pack.kwargs);
    // kwargs["cvvp_color"] = True highlights the frames as decoded, with all their channels, against an (h, w, C)
    // background: d is the largest per-channel difference (cvvp_highlight_set_channels), so objects that differ from
    // the background in colour but not in grey level are found.
    const bool color = color_frames(pack.assign_objects_pack.kwargs, pack.grayscale, pack.vid_is_grayscale);
    const bool rolling = roll_window > 0;
    FrameSource vid{pack.vid_path, pack.grayscale, pack.vid_is_grayscale};
    if (!vid.opened()) {
        std::cerr << "Video file not detected: " << pack.vid_path << '\n';
        return py::dict{};
    }
    const int fw = int(vid.get("CAP_PROP_FRAME_WIDTH")), fh = int(vid.get("CAP_PROP_FRAME_HEIGHT"));
    // validation :167-175 (raises RuntimeError like EXCEPTION_ASSERT)
    const py::array &bg = pack.highlight_objects_pack.background;
    CVVP_ASSERT_MSG(bg.size() > 0, "background must not be empty");
    const Rect crop = GetCroppedFrameDims(pack.crop_x, pack.crop_y, pack.crop_width, pack.crop_height, fw, fh);
    CVVP_ASSERT(bg.ndim() >= 2 && crop.width == int(bg.shape(1)));
    CVVP_ASSERT(bg.ndim() >= 2 && crop.height == int(bg.shape(0)));
    CVVP_ASSERT_MSG(pack.highlight_objects_pack.struct_element.size() > 0, "struct element must not be empty");

    long long num_frames = static_cast<long long>(vid.get("CAP_PROP_FRAME_COUNT")); // :54-66
    const long long total = num_frames;
    if (pack.frame_limit > 0 && num_frames > pack.frame_limit)
        num_frames = pack.frame_limit;
    // generator constructor checks (cv_vid_frames_generator_algo.h:94-101)
    CVVP_ASSERT(pack.start_frame >= 0);
    CVVP_ASSERT(pack.start_frame < total);
    CVVP_ASSERT(pack.start_frame + num_frames > 0);
    CVVP_ASSERT(num_frames > 0);
    CVVP_ASSERT(crop.x + crop.width <= fw && crop.y + crop.height <= fh);
    vid.set("CAP_PROP_POS_FRAMES", double(pack.start_frame));
    vid.set_crop(crop);
    vid.configure();

    GpuHighlightPack hp;
    hp.background = to_u8_image(bg, "background must not be empty", color);
    hp.struct_element = to_u8_image(pack.highlight_objects_pack.struct_element, "struct element must not be empty");
    hp.threshold = pack.highlight_objects_pack.threshold;
    hp.threshold_lo = pack.highlight_objects_pack.threshold_lo;
    hp.threshold_hi = pack.highlight_objects_pack.threshold_hi;
    hp.min_size_hyst = pack.highlight_objects_pack.min_size_hyst;
    hp.min_size_threshold = pack.highlight_objects_pack.min_size_threshold;
    hp.width_border = pack.highlight_objects_pack.width_border;
    hp.polarity = polarity;
    // Opt-in extra of this implementation (the reference has no counterpart): kwargs["cvvp_components"] = True makes
    // the device label the 8-connected components of every mask and hands the callback one more keyword argument,
    // `components` = {"count", "stats" (count x 5: x, y, w, h, area -- cv2.connectedComponentsWithStats columns),
    // "centroids" (count x 2), "first" (count x 2: raster-first pixel x, y)[, "labels" (int32 H x W) with
    // kwargs["cvvp_labels"] = True]}; components are numbered in the raster order of their first pixels.
    // kwargs["cvvp_component_stats"] = True adds "moments" (count x 3 int64: m20, m11, m02), "mass" (count int64: sum of
    // d), "weighted_centroids" (count x 2: sum(d x) / mass, sum(d y) / mass; NaN where the mass is 0) and "contrast"
    // (count x 2 int32: min d, max d), d being the difference image the thresholds saw (cvvp_component_stats).
    const py::dict &user_kwargs = pack.assign_objects_pack.kwargs;
    const bool want_comps = user_kwargs.contains("cvvp_components") && user_kwargs["cvvp_components"].cast<bool>();
    const bool want_labels = want_comps && user_kwargs.contains("cvvp_labels") && user_kwargs["cvvp_labels"].cast<bool>();
    hp.components = want_comps;
    hp.component_stats = want_stats;
    hp.labels = want_labels;
    if (want_comps && user_kwargs.contains("cvvp_max_components"))
        hp.max_components = std::max(1, user_kwargs["cvvp_max_components"].cast<int>());
    // label images only travel through the synchronous entry point; everything else is queued
    const bool on_device = !host_prep() && !want_labels;
    // rolling mode takes the synchronous loop below (the rolling stream handles labels itself): frames are prepared on
    // the device unless CVVP_HOST_PREP=1
    const bool pipelined = on_device && !rolling;
    const bool device_prep = rolling ? !host_prep() : on_device;
    std::unique_ptr<GpuHighlightAlgo> highlighter; // built once the first decoded frame tells the channel count
    std::unique_ptr<GpuRollingHighlightAlgo> roller; // rolling mode's operator

    // frames per device batch: the reference's batch_size is a thread count; here it is sized for the GPU, and at most
    // token_storage_limit batches are in flight like the reference's queues (token_queue.h:209-214)
    const long long npix = static_cast<long long>(crop.width) * crop.height;
    long long batch_frames = (32ll << 20) / npix + 1;
    if (batch_frames > 256)
        batch_frames = 256;
    if (const char *e = std::getenv("CVVP_TRACK_BATCH")) // developer switch: frames per batch (tests use small batches)
        batch_frames = std::max(1, std::atoi(e));
    const int depth = std::min(std::max(pack.token_storage_limit, 1), 3);

    // AssignObjectsAlgo state (assign_objects_algo.h:172-178)
    py::dict objects_active, objects_archive;
    long long num_processed = 0;
    int next_id = 0;
    bool any = false;
    IntervalTimer h_batch, h_gen, h_unit, h_consume, a_batch, a_gen, a_unit, a_consume;

    // the assign stage: strictly in frame order, one call per frame (assign_objects_algo.h:111-133).  The callback gets a
    // numpy array that OWNS its bytes (it may keep it), copied from wherever the masks lie (a batch, a pinned view).
    const int mrows = crop.height, mcols = crop.width;
    const std::size_t mbytes = std::size_t(mrows) * mcols;
    std::function<void()> between_frames; // pipelined path: keeps the decoder and the device fed while a batch is delivered
    const std::size_t rec_bytes = record_bytes(hp);
    auto deliver_raw = [&](const std::uint8_t *masks, std::size_t pitch, long long n, const cvvp_component *comps_all,
                           const int *ncomps_all, int max_comps, const std::int32_t *labels_all) {
        a_batch.start();
        a_gen.start(); // the intermediary hands the ordered masks over (mat_set_intermediary.h:84-114)
        a_gen.stop();
        for (long long i = 0; i < n; ++i) {
            if (between_frames)
                between_frames();
            py::array_t<std::uint8_t> bw({mrows, mcols});
            std::memcpy(bw.mutable_data(), masks + std::size_t(i) * pitch, mbytes);
            using namespace pybind11::literals;
            a_unit.start();
            if (want_comps) {
                const int total = ncomps_all ? ncomps_all[i] : 0;
                const int cnt = std::min(total, max_comps);
                const std::uint8_t *recs = reinterpret_cast<const std::uint8_t *>(comps_all) +
                                           std::size_t(i) * max_comps * rec_bytes;
                auto rec = [&](int k) -> const cvvp_component & {
                    return *reinterpret_cast<const cvvp_component *>(recs + std::size_t(k) * rec_bytes);
                };
                py::array_t<std::int32_t> stats({cnt, 5});
                py::array_t<double> cents({cnt, 2});
                py::array_t<std::int32_t> first({cnt, 2});
                auto st = stats.mutable_unchecked<2>();
                auto ce = cents.mutable_unchecked<2>();
                auto fi = first.mutable_unchecked<2>();
                for (int k = 0; k < cnt; ++k) {
                    const cvvp_component &c = rec(k);
                    st(k, 0) = c.x0;
                    st(k, 1) = c.y0;
                    st(k, 2) = c.x1 - c.x0 + 1;
                    st(k, 3) = c.y1 - c.y0 + 1;
                    st(k, 4) = c.area;
                    ce(k, 0) = double(c.sum_x) / double(c.area);
                    ce(k, 1) = double(c.sum_y) / double(c.area);
                    fi(k, 0) = c.first_x;
                    fi(k, 1) = c.first_y;
                }
                py::dict comps;
                comps["count"] = total;
                comps["stats"] = stats;
                comps["centroids"] = cents;
                comps["first"] = first;
                if (hp.component_stats) {
                    py::array_t<std::int64_t> moments({cnt, 3});
                    py::array_t<std::int64_t> mass(cnt);
                    py::array_t<double> wcents({cnt, 2});
                    py::array_t<std::int32_t> contrast({cnt, 2});
                    auto mo = moments.mutable_unchecked<2>();
                    auto ma = mass.mutable_unchecked<1>();
                    auto wc = wcents.mutable_unchecked<2>();
                    auto co = contrast.mutable_unchecked<2>();
                    for (int k = 0; k < cnt; ++k) {
                        const cvvp_component_stats &c = reinterpret_cast<const cvvp_component_stats &>(rec(k));
                        mo(k, 0) = c.sum_xx;
                        mo(k, 1) = c.sum_xy;
                        mo(k, 2) = c.sum_yy;
                        ma(k) = c.sum_d;
                        // a component whose pixels all have d = 0 (hole filling, the all-255 quirk) has no weighted centroid
                        wc(k, 0) = c.sum_d ? double(c.sum_dx) / double(c.sum_d) : std::nan("");
                        wc(k, 1) = c.sum_d ? double(c.sum_dy) / double(c.sum_d) : std::nan("");
                        co(k, 0) = c.min_d;
                        co(k, 1) = c.max_d;
                    }
                    comps["moments"] = moments;
                    comps["mass"] = mass;
                    comps["weighted_centroids"] = wcents;
                    comps["contrast"] = contrast;
                }
                if (want_labels && labels_all) {
                    py::array_t<std::int32_t> lab({mrows, mcols});
                    std::memcpy(lab.mutable_data(), labels_all + std::size_t(i) * mbytes, mbytes * sizeof(std::int32_t));
                    comps["labels"] = lab;
                }
                next_id = pack.assign_objects_pack.function("bw_frame"_a = bw, "frames_processed"_a = num_processed,
                                                            "objects_prev"_a = objects_active,
                                                            "objects_archive"_a = objects_archive, "next_ID"_a = next_id,
                                                            "kwargs"_a = pack.assign_objects_pack.kwargs,
                                                            "components"_a = comps)
                              .cast<int>();
            } else {
                next_id = pack.assign_objects_pack.function("bw_frame"_a = bw, "frames_processed"_a = num_processed,
                                                            "objects_prev"_a = objects_active,
                                                            "objects_archive"_a = objects_archive, "next_ID"_a = next_id,
                                                            "kwargs"_a = pack.assign_objects_pack.kwargs)
                              .cast<int>();
            }
            a_unit.stop();
            ++num_processed;
            any = true;
        }
        a_batch.stop();
    };
    auto deliver = [&](const FrameBatch &masks) {
        deliver_raw(masks.data.data(), masks.frame_bytes(), masks.n,
                    masks.comps.empty() ? nullptr : reinterpret_cast<const cvvp_component *>(masks.comps.data()),
                    masks.ncomps.empty() ? nullptr : masks.ncomps.data(), masks.max_comps,
                    masks.labels.empty() ? nullptr : masks.labels.data());
    };

    // colour: the first decoded frame tells the channel count, which the background must have; checked before the
    // operators are built
    auto take_channels = [&](int ch) {
        if (!color)
            return;
        CVVP_ASSERT_MSG(hp.background.channels == ch && bg.ndim() == 3,
                        "kwargs['cvvp_color']: the background must be (h, w, C) with the channel count of the decoded "
                        "frames");
        hp.channels = ch;
    };
    const std::vector<int> devices = device_list();
    if (rolling)
        hp.device = devices.front();
    if (pipelined) {
        // ---- pipelined path: decode thread -> pinned queue slots -> device(s) -> ordered callbacks ----
        // the first frame is decoded here: it tells the channel count the device format needs
        h_gen.start();
        py::object f0 = vid.next_decoded();
        h_gen.stop();
        if (!f0.is_none()) {
            py::array a0 = f0.cast<py::array>();
            int r, c, ch;
            array_geometry(a0, r, c, ch);
            CVVP_ASSERT(r == fh && c == fw);
            hp.queue_depth = depth;
            hp.max_batch = batch_frames;
            hp.source = vid.format_for(r, c, ch);
            take_channels(ch);
            CVVP_ASSERT_MSG(hp.source.out_channels() == hp.channels,
                            "TrackObjects needs single-channel frames: set grayscale or "
                            "vid_is_grayscale (cv::findContours requires 8UC1)");
            std::vector<std::unique_ptr<GpuHighlightAlgo>> lanes; // one operator (context + queue) per device
            for (int d : devices) {
                GpuHighlightPack lp = hp;
                lp.device = d;
                lanes.push_back(std::make_unique<GpuHighlightAlgo>(std::move(lp)));
            }
            const long long D = (long long)lanes.size();
            const int max_comps = lanes[0]->max_components();
            const std::size_t frame_bytes = std::size_t(r) * c * ch;
            DecodeWorker worker{vid, r, c, ch, num_frames - 1};
            // batches in frame order: batch k lives on lane k % D.  handed >= committed >= delivered.
            long long handed = 0, popped = 0, committed = 0, delivered = 0; // popped: slots the decoder gave back
            std::vector<int> out_on_lane(lanes.size(), 0); // slots of the lane the decoder holds
            bool decode_done = false, first = true;
            std::string error;
            // non-blocking: queue the slots the decoder has filled (in order), hand it every free slot to work ahead
            auto service = [&]() {
                DecodeWorker::Done done;
                while (handed > popped && worker.pop(done, 0)) {
                    h_gen.stop();
                    const std::size_t lane = std::size_t(popped % D);
                    h_unit.start();
                    lanes[lane]->CommitSlot(done.n);
                    h_unit.stop();
                    h_batch.stop();
                    out_on_lane[lane]--;
                    ++popped;
                    if (done.n > 0) // (a slot that comes back empty at the end of the stream is not a batch)
                        ++committed;
                    if (done.eof)
                        decode_done = true;
                    if (!done.error.empty() && error.empty())
                        error = done.error;
                }
                while (!decode_done && error.empty()) {
                    const std::size_t lane = std::size_t(handed % D);
                    GpuHighlightAlgo &L = *lanes[lane];
                    if (L.Pending() + out_on_lane[lane] >= L.Depth())
                        break;
                    const GpuHighlightAlgo::Slot slot = L.AcquireSlot();
                    CVVP_ASSERT(slot.pitch >= frame_bytes);
                    long long pre = 0;
                    if (first) { // the frame decoded above is the first slot's first one
                        std::memcpy(slot.frames, a0.data(), frame_bytes);
                        pre = 1;
                        first = false;
                    }
                    h_batch.start();
                    h_gen.start();
                    worker.push(DecodeWorker::Job{slot.frames, slot.pitch, std::min(slot.max_frames, batch_frames), pre});
                    out_on_lane[lane]++;
                    ++handed;
                }
            };
            between_frames = [&]() {
                service();
                if (worker.wants_gil()) { // hand the GIL to the decode thread: it needs it for a moment per frame
                    py::gil_scoped_release nogil;
                    for (int spin = 0; spin < 2000 && worker.wants_gil(); ++spin)
                        std::this_thread::yield();
                }
            };
            while (error.empty()) {
                service();
                if (delivered < committed) {
                    // the oldest batch goes to the tracker: now if it is complete, else once nothing else can move
                    GpuHighlightAlgo &L = *lanes[std::size_t(delivered % D)];
                    const bool idle = decode_done || handed == popped; // the decoder holds no slot: a lane is full
                    if (L.Ready() || idle) {
                        h_consume.start();
                        GpuHighlightAlgo::MaskView v;
                        {
                            py::gil_scoped_release nogil; // other Python threads (and the decoder) run while this waits
                            v = L.NextView();
                        }
                        h_consume.stop();
                        deliver_raw(v.masks, v.pitch, v.n, v.comps, v.ncomps, max_comps, nullptr);
                        L.ReleaseView();
                        ++delivered;
                        continue;
                    }
                } else if (decode_done && handed == popped) {
                    break; // everything decoded, queued and delivered
                }
                // nothing to deliver yet: wait for the decoder (briefly, so that a completed batch is noticed soon)
                py::gil_scoped_release nogil;
                if (handed > popped)
                    worker.wait_done(200);
                else
                    std::this_thread::sleep_for(std::chrono::microseconds(100));
            }
            between_frames = nullptr;
            if (std::getenv("CVVP_TRACK_DEBUG")) {
                auto ms = [](std::chrono::steady_clock::duration d) { return std::chrono::duration<double, std::milli>(d).count(); };
                std::cerr << "[cvvp track] decode thread: read " << ms(worker.t_read) << " ms, GIL wait " << ms(worker.t_gil_wait)
                          << " ms, slot wait " << ms(worker.t_job_wait) << " ms; calling thread: callbacks " << a_unit.ms()
                          << " ms, result wait " << h_consume.ms() << " ms, commits " << h_unit.ms() << " ms; batches " << committed
                          << " of " << batch_frames << " frames\n";
            }
            if (!error.empty())
                throw std::runtime_error(error);
        }
    }
    // one step of the synchronous loop on whichever operator this run uses: insert a batch (null: end of the stream),
    // then hand every mask that has come back to the tracker
    auto step = [&](auto &op, std::unique_ptr<FrameBatch> batch) {
        if (batch) {
            h_unit.start();
            op.Insert(std::move(batch)); // queued on the device; returns before the masks exist
            h_unit.stop();
            h_batch.stop();
        } else {
            op.NotifyNoMoreTokens(); // rolling: the last frames' windows clamp to the frames decoded
        }
        for (;;) {
            h_consume.start();
            std::unique_ptr<FrameBatch> masks = op.TryGetResult();
            h_consume.stop();
            if (!masks)
                break;
            deliver(*masks);
        }
    };
    auto sync_step = [&](std::unique_ptr<FrameBatch> batch) {
        if (roller)
            step(*roller, std::move(batch));
        else
            step(*highlighter, std::move(batch));
    };
    long long consumed = 0;
    bool eof = pipelined; // the pipelined path above has consumed the stream
    while (!eof && consumed < num_frames) {
        h_batch.start();
        h_gen.start();
        auto batch = std::make_unique<FrameBatch>();
        while (batch->n < batch_frames && consumed < num_frames) {
            py::object f = device_prep ? vid.next_decoded() : vid.next();
            if (f.is_none()) {
                eof = true;
                break;
            }
            py::array a = f.cast<py::array>();
            int r, c, ch;
            array_geometry(a, r, c, ch);
            if (!highlighter && !roller) {
                hp.queue_depth = depth;
                hp.max_batch = batch_frames;
                if (device_prep) {
                    CVVP_ASSERT(r == fh && c == fw);
                    hp.source = vid.format_for(r, c, ch);
                    take_channels(ch);
                    CVVP_ASSERT_MSG(hp.source.out_channels() == hp.channels,
                                    "TrackObjects needs single-channel frames: set grayscale or vid_is_grayscale "
                                    "(cv::findContours requires 8UC1)");
                } else {
                    take_channels(ch);
                }
                if (rolling)
                    roller = std::make_unique<GpuRollingHighlightAlgo>(std::move(hp), roll_window, roll_percent);
                else
                    highlighter = std::make_unique<GpuHighlightAlgo>(std::move(hp));
            }
            if (batch->n == 0) {
                batch->rows = r;
                batch->cols = c;
                batch->channels = ch;
                // one allocation per batch: a vector that grows frame by frame re-copies every decoded frame
                batch->data.reserve(std::size_t(std::min(batch_frames, num_frames - consumed)) * r * c * ch);
            }
            if (!device_prep) {
                CVVP_ASSERT_MSG(ch == hp.channels, "TrackObjects needs single-channel frames: set grayscale or "
                                                   "vid_is_grayscale (cv::findContours requires 8UC1)");
                CVVP_ASSERT(r == crop.height && c == crop.width);
            }
            CVVP_ASSERT(r == batch->rows && c == batch->cols && ch == batch->channels);
            const auto *src = static_cast<const std::uint8_t *>(a.data());
            batch->data.insert(batch->data.end(), src, src + std::size_t(r) * c * ch);
            batch->n++;
            ++consumed;
        }
        h_gen.stop();
        if (batch->n == 0)
            break;
        // masks that have come back meanwhile go to the tracker while the device works on the newer batches
        sync_step(std::move(batch));
    }
    if (highlighter || roller) // end of stream: drain in order (token_processing_unit.h:334)
        sync_step(nullptr);
    a_consume.start();
    a_consume.stop();
    if (pack.print_timing_report) { // cv_vid_objecttrack_helpers.cpp:136-143
        std::cout << "Highlight objects timing report:\n" << timing_report(h_batch, h_gen, h_consume, h_unit);
        std::cout << "Assign objects timing report:\n" << timing_report(a_batch, a_gen, a_consume, a_unit);
    }
    if (!any)
        return py::dict{};
    return objects_archive;
}
} // namespace

/// NOTE: cvvidproc_b200/__init__.py re-exports these names exactly like PySources/cvvidproc/__init__.py:3
PYBIND11_MODULE(_core, mod)
{
    mod.doc() = "C++ bindings for processing an opencv video"; // py_bindings.cpp:33

    py::class_<VidBgPack>(mod, "VidBgPack") // py_bindings.cpp:36-60
        .def(py::init([](const std::string &vid_path, const std::string &bg_algo, int max_threads, long long frame_limit,
                         bool grayscale, bool vid_is_grayscale, int crop_x, int crop_y, int crop_width, int crop_height,
                         int token_storage_limit, bool print_timing_report) {
                 return VidBgPack{vid_path, bg_algo, max_threads, frame_limit, grayscale, vid_is_grayscale, crop_x, crop_y,
                                  crop_width, crop_height, token_storage_limit, print_timing_report};
             }),
             py::arg("vid_path"), py::arg("bg_algo") = "hist", py::arg("max_threads") = -1, py::arg("frame_limit") = -1,
             py::arg("grayscale") = false, py::arg("vid_is_grayscale") = false, py::arg("crop_x") = 0, py::arg("crop_y") = 0,
             py::arg("crop_width") = 0, py::arg("crop_height") = 0, py::arg("token_storage_limit") = 10,
             py::arg("print_timing_report") = false);

    mod.def("GetVideoBackground", &GetVideoBackground, "Get the background of an OpenCV video.", py::arg("pack")); // :63-66

    py::class_<HighlightObjectsPack>(mod, "HighlightObjectsPack") // :69-85
        .def(py::init([](py::array background, py::array struct_element, int threshold, int threshold_lo, int threshold_hi,
                         int min_size_hyst, int min_size_threshold, int width_border) {
                 return HighlightObjectsPack{std::move(background), std::move(struct_element), threshold, threshold_lo,
                                             threshold_hi, min_size_hyst, min_size_threshold, width_border};
             }),
             py::arg("background"), py::arg("struct_element"), py::arg("threshold"), py::arg("threshold_lo"),
             py::arg("threshold_hi"), py::arg("min_size_hyst"), py::arg("min_size_threshold"), py::arg("width_border"));

    py::class_<AssignObjectsPack>(mod, "AssignObjectsPack") // :88-95
        .def(py::init([](py::function function, py::dict kwargs) { return AssignObjectsPack{std::move(function), std::move(kwargs)}; }),
             "Expected signature/behavior of input func: \
                next_ID = func(bw_frame, frames_processed, objects_prev, objects_archive, next_ID, kwargs) \
                note: 'kwargs' should be a python dictionary",
             py::arg("function"), py::arg("kwargs"));

    py::class_<VidObjectTrackPack>(mod, "VidObjectTrackPack") // :98-126
        .def(py::init([](const std::string &vid_path, HighlightObjectsPack highlight_objects_pack,
                         AssignObjectsPack assign_objects_pack, int max_threads, long long start_frame, long long frame_limit,
                         bool grayscale, bool vid_is_grayscale, int crop_x, int crop_y, int crop_width, int crop_height,
                         int token_storage_limit, bool print_timing_report) {
                 return VidObjectTrackPack{vid_path, std::move(highlight_objects_pack), std::move(assign_objects_pack),
                                           max_threads, start_frame, frame_limit, grayscale, vid_is_grayscale, crop_x, crop_y,
                                           crop_width, crop_height, token_storage_limit, print_timing_report};
             }),
             py::arg("vid_path"), py::arg("highlight_objects_pack"), py::arg("assign_objects_pack"),
             py::arg("max_threads") = -1, py::arg("start_frame") = 0, py::arg("frame_limit") = -1, py::arg("grayscale") = false,
             py::arg("vid_is_grayscale") = false, py::arg("crop_x") = 0, py::arg("crop_y") = 0, py::arg("crop_width") = 0,
             py::arg("crop_height") = 0, py::arg("token_storage_limit") = 10, py::arg("print_timing_report") = false);

    mod.def("TrackObjects", &TrackObjects, "Track objects in an OpenCV video.", py::arg("pack")); // :129-130
}
