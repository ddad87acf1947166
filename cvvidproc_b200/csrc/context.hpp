// Opaque context behind the C ABI (include/cvvp.h): one CUDA device, its streams/events, the
// device frame stack of the running median job and the pinned staging ring.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/cvvp.h"

namespace cvvp
{
using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct StagingBuf {
    uint8_t *host{nullptr};
    size_t bytes{0};
    cudaEvent_t done{nullptr};
    bool in_flight{false};
};

struct MedianJob {
    bool active{false};
    size_t nelem{0};
    size_t stride{0}; // device frame pitch in bytes (multiple of 128)
    long long capacity{0};
    long long count{0};
    uint8_t *d_stack{nullptr};
    uint8_t *d_out{nullptr};
    size_t d_out_bytes{0};
    size_t d_stack_bytes{0};
    // constant-memory form (median_hist.cu): frames folded into value histograms when the stack cannot grow
    uint32_t *d_hist{nullptr}; // [256][stride] counts, or nullptr
    size_t d_hist_bytes{0};
    long long folded{0};       // frames that live in d_hist only (count = the frames resident in d_stack)
    int percent{50};           // the context's percentile when the job began (cvvp_median_set_percentile)
    // after the first fold the stack is used as two halves: one is filled while the other is being folded
    bool split{false};
    int half{0};
    long long half_cap{0};     // frames per half
    long long base{0};         // first frame slot of the region being filled (0 or half_cap)
    cudaEvent_t ev_fold[2]{nullptr, nullptr}; // the fold that last read half h is complete
};
struct HighlightState; // highlight_state.hpp

// Where the counting rounds of a frame-sharded median push their per-element nibble counts (median_shard.cu):
// element e belongs to rank e / slice, whose receive area for THIS rank's counts starts at dst[e / slice]
// (8 words = 16 u16 counts per element, peer memory over NVLink or local).
constexpr int kMaxShardRanks = 16;
struct ShardPush {
    uint32_t *dst[kMaxShardRanks];
    const uint32_t *sel;   // round 2: per element, the globally selected high nibble in bits 0..3
    const uint32_t *accum; // counts of this rank's earlier frame chunks (8 words per element), or nullptr
    uint32_t slice;
    uint32_t stage; // 1: round 1 stages a tile's count vectors in shared memory and stores them 512 B per warp (peer owners)
    // not NULL: the launch only takes the *tile_count tiles listed in tile_list (128 elements each) instead of all of
    // them -- the two counting rounds behind a window pass recount only the tiles that hold an undecided element
    const uint32_t *tile_list;
    const uint32_t *tile_count;
    // window counting (MODE 3): a source's frame count goes to one header word per owner, not into every record
    uint32_t *hdr[kMaxShardRanks];
    uint32_t nranks;
};
struct MedianShard; // median_shard.cu

// device staging of decoded frames waiting for the preparation kernel (frames.cu), double-buffered
struct RawStage {
    uint8_t *d[2]{nullptr, nullptr};
    size_t cap{0}; // bytes per half
    cudaEvent_t up[2]{nullptr, nullptr};       // H2D of this half complete
    cudaEvent_t consumed[2]{nullptr, nullptr}; // the kernel that read this half is complete
    bool used[2]{false, false};
    int next{0};
    uint8_t *d_out{nullptr}; // result staging of the host-buffer form (cvvp_frames_prepare)
    size_t out_cap{0};
};
struct HighlightQueue; // frame_pipeline.cu
struct RollingStream;  // highlight_rolling.cu
} // namespace cvvp

struct cvvp_ctx {
    int device{0};
    int sm_count{0};
    int cc_major{0};
    int cc_minor{0};
    size_t smem_optin{0};
    cudaStream_t compute{nullptr};
    cudaStream_t copy{nullptr};     // host -> device
    cudaStream_t copy_out{nullptr}; // device -> host (so both directions of the link overlap)
    cudaEvent_t ev_start{nullptr};
    cudaEvent_t ev_stop{nullptr};
    cudaEvent_t ev_copy{nullptr};
    bool have_kernel_time{false};
    long long launches{0};
    std::string err;
    cvvp::EncodeTiledFn encode_tiled{nullptr};
    cvvp::MedianJob med;
    cvvp::HighlightState *hl{nullptr};
    cvvp::MedianShard *shard{nullptr};
    cvvp::MedianShard *big{nullptr}; // internal one-rank job of the two-pass path for long stacks (median.cu)
    std::vector<cvvp::StagingBuf> staging;
    size_t staging_next{0};
    cvvp::RawStage raw;
    cvvp::HighlightQueue *hq{nullptr};
    cvvp::RollingStream *hr{nullptr};
    int percent{50}; // percentile of every background (cvvp_median_set_percentile); jobs take it when they begin
    int polarity{CVVP_POLARITY_DARK}; // object polarity (cvvp_highlight_set_polarity); highlight jobs take it when they begin
    int component_stats{0}; // cvvp_highlight_set_component_stats; highlight jobs take it when they begin
    int channels{1}; // channels of highlight frames (cvvp_highlight_set_channels); highlight jobs take it when they begin
};

namespace cvvp
{
void set_global_error(const char *fmt, ...);
const char *global_error();

int fail(cvvp_ctx *ctx, int code, const char *fmt, ...);

inline size_t round_up(size_t v, size_t a)
{
    return (v + a - 1) / a * a;
}

#define CVVP_CUDA_OK(ctx, expr)                                                                                       \
    do {                                                                                                               \
        cudaError_t _e = (expr);                                                                                       \
        if (_e != cudaSuccess)                                                                                         \
            return ::cvvp::fail((ctx), CVVP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),          \
                                __FILE__, __LINE__);                                                                   \
    } while (0)

// RAII device switch: every ABI call makes its context's device current and restores the caller's.
struct DeviceGuard {
    int prev{-1};
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess)
            prev = -1;
        if (prev != dev)
            cudaSetDevice(dev);
        else
            prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0)
            cudaSetDevice(prev);
    }
};

// median.cu
// percent: the percentile every form selects, sorted[percentile_rank(N, percent)] (median_common.cuh)
int median_launch(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                  uint8_t *d_out, int percent, cudaStream_t stream);
int median_launch_mode(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                       uint8_t *d_out, int mode, int percent, const ShardPush &push, cudaStream_t stream);
// median_pipe.cu
long long median_max_frames();
int median_pipe_launch(cvvp_ctx *ctx, const CUtensorMap &tmap, int log2s, uint8_t *d_out, uint32_t nelem, uint32_t nframes,
                       uint32_t nst, int mode, uint32_t percent, const ShardPush &push, cudaStream_t stream);
// median_hist.cu
size_t median_hist_bytes(size_t frame_stride);
int median_hist_fold(cvvp_ctx *ctx, const uint8_t *d_stack, long long nframes, size_t frame_stride, uint32_t *d_hist,
                     cudaStream_t stream);
int median_hist_select(cvvp_ctx *ctx, const uint32_t *d_hist, size_t frame_stride, size_t nelem, long long total, int percent,
                       uint8_t *d_out, cudaStream_t stream);
// median_shard.cu
void median_shard_release(cvvp_ctx *ctx);
int median_long_stack(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                      uint8_t *d_out, int percent, cudaStream_t stream, int window);
long long median_two_pass_max_frames();
// highlight.cu
void highlight_release(cvvp_ctx *ctx);
int highlight_begin(cvvp_ctx *ctx, const uint8_t *background, int width, int height, const uint8_t *selem, int kw, int kh,
                    int threshold, int threshold_lo, int threshold_hi, int min_size_hyst, int min_size_threshold);
// optional component output of a highlight call: all pointers null = off
struct CcOut {
    cvvp_component *comps{nullptr}; // [frame][max_comps] records of rec_bytes each
    int max_comps{0};
    int *ncomps{nullptr};
    int32_t *labels{nullptr}; // [frame][labels_stride] or nullptr
    size_t labels_stride{0};
    size_t rec_bytes{sizeof(cvvp_component)}; // highlight_device_bg sets the job's (highlight_record_bytes)
};
// bytes of one component record of the context's highlight job: sizeof(cvvp_component_stats) while the job has
// component statistics on (cvvp_highlight_set_component_stats), else sizeof(cvvp_component)
size_t highlight_record_bytes(const cvvp_ctx *ctx);
// the component arguments are complete and the job's path can label (a highlight job must exist)
int highlight_check_cc(cvvp_ctx *ctx, long long n, const CcOut &cc);
// frame f against the background at d_bgs + f * bg_stride (0 = one for all; d_bgs == nullptr: the job's own)
int highlight_device_bg(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride, const uint8_t *d_bgs,
                        size_t bg_stride, uint8_t *d_out, size_t out_stride, const CcOut &cc, cudaStream_t stream);
// channels of the running job's frames (cvvp_highlight_set_channels); 0: no job
int highlight_job_channels(const cvvp_ctx *ctx);
// Colour job: the d planes (highlight_color.cu) of n frames at src + f * frame_stride against the backgrounds at
// d_bgs + f * bg_stride (d_bgs == nullptr: the job's own) -> d_planes + f * pitch.  row_stride == 0: contiguous frames
// of width*height*C bytes; else frame rows row_stride bytes apart whose pixels start at pixel x0 (a crop).
int highlight_color_d(cvvp_ctx *ctx, const uint8_t *src, long long n, size_t frame_stride, size_t row_stride, int x0,
                      const uint8_t *d_bgs, size_t bg_stride, uint8_t *d_planes, size_t pitch, cudaStream_t stream);
// Colour job: the masks (and components) of n d planes of highlight_color_d
int highlight_device_planes(cvvp_ctx *ctx, const uint8_t *d_planes, long long n, size_t pitch, uint8_t *d_out,
                            size_t out_stride, const CcOut &cc, cudaStream_t stream);
// highlight_color.cu: d = max over the channels (2..4) of the polarity's difference, rows of row_len pixels
int color_diff_launch(cvvp_ctx *ctx, int channels, int polarity, const uint8_t *src, long long n, size_t frame_stride,
                      size_t row_stride, int x0, const uint8_t *bg, size_t bg_stride, uint32_t row_len, uint32_t nrows,
                      uint8_t *dst, size_t dst_pitch, cudaStream_t stream);
int highlight_frames_host_cc(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                             size_t out_stride, cvvp_component *comps_out, int max_comps, int *ncomps_out,
                             int32_t *labels_out, size_t labels_stride);
int highlight_set_path(cvvp_ctx *ctx, int path);
int highlight_frames_in_flight(cvvp_ctx *ctx, int *out_frames);
int highlight_frames_host(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                          size_t out_stride);
// frames.cu
size_t frames_out_bytes(const cvvp_frame_format &f);
int frames_check_format(cvvp_ctx *ctx, const cvvp_frame_format *f);
int frames_prepare_launch(cvvp_ctx *ctx, const uint8_t *d_src, long long n, size_t src_stride, size_t src_bytes,
                          const cvvp_frame_format &f, int band_row0, uint8_t *d_dst, size_t dst_stride, cudaStream_t stream);
// frame_pipeline.cu
void raw_stage_release(cvvp_ctx *ctx);
int raw_stage_ensure(cvvp_ctx *ctx, size_t bytes_per_half);
int frames_prepare_host(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format &f,
                        uint8_t *out, size_t out_stride);
int frames_upload_prepare(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format &f,
                          uint8_t *d_dst, size_t dst_stride);
// Shared by the highlight queue and the rolling stream: the results of one batch of up to max_batch frames on their way
// to the host, and the event that marks the end of their download.
struct HlResults {
    size_t npix{0}, pitch{0}; // mask bytes / pitch of the masks on both sides
    int max_comps{0};         // 0: no components
    size_t rec_bytes{0};      // bytes per component record (highlight_record_bytes of the job)
    bool labels{false};
    size_t mask_bytes{0};     // of each pooled mask buffer (pool.hpp)
    uint8_t *h_out{nullptr}, *d_out{nullptr}; // h_*: pinned
    cvvp_component *h_comps{nullptr}, *d_comps{nullptr};
    int *h_ncomps{nullptr}, *d_ncomps{nullptr};
    int32_t *h_labels{nullptr}, *d_labels{nullptr};
    cudaEvent_t down{nullptr};
    long long n{0}; // frames of the batch
};
// false: out of memory (what was allocated stays for hl_results_free)
bool hl_results_alloc(HlResults &r, long long max_batch, size_t npix, size_t pitch, int max_comps, size_t rec_bytes,
                      bool labels);
void hl_results_free(HlResults &r);
// the n frames' component outputs, starting at frame `first` of the batch
CcOut hl_results_cc(const HlResults &r, long long first);
// queues the download of r.n frames after the work on the compute stream: copy_out waits, copies and records `down`
int hl_results_download(cvvp_ctx *ctx, HlResults &r);
// 1: downloaded, 0: not yet, < 0: the batch failed (the message starts with `who`)
int hl_results_ready(cvvp_ctx *ctx, const HlResults &r, const char *who);
// waits for the download; CVVP_OK or the batch's failure
int hl_results_wait(cvvp_ctx *ctx, const HlResults &r, const char *who);
// copies the downloaded batch into the caller's buffers (null comps / ncomps / labels: not wanted)
void hl_results_copy(const HlResults &r, uint8_t *masks, size_t mask_stride, cvvp_component *comps, int *ncomps,
                     int32_t *labels, size_t labels_stride);
void sync_streams(cvvp_ctx *ctx); // copy, compute and copy_out
// A call that failed half-way may leave work of unknown extent queued: drain the streams, keep the error, set the
// stream's `failed` (it refuses further work until it is ended) and return rc.
int drain_after_failure(cvvp_ctx *ctx, bool &failed, int rc);
// Begin-time checks of a stream, in this order: a highlight job exists (*W x *H), the stream has not begun, its own
// arguments (args_rc: the caller's checks, whose message is the last one set), and frames of the format fmt (null:
// prepared frames) prepare to single-channel frames of the job's size.
int highlight_stream_check(cvvp_ctx *ctx, const char *who, bool begun, int args_rc, const cvvp_frame_format *fmt, int *W, int *H);
void highlight_queue_release(cvvp_ctx *ctx);
int highlight_queue_begin(cvvp_ctx *ctx, int depth, long long max_batch, const cvvp_frame_format *fmt, int max_comps);
int highlight_queue_pending(const cvvp_ctx *ctx);
int highlight_queue_submit(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride);
int highlight_queue_ready(cvvp_ctx *ctx);
int highlight_queue_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long *n_out, cvvp_component *comps_out,
                         int *ncomps_out);
int highlight_slot_acquire(cvvp_ctx *ctx, uint8_t **h_frames, size_t *frame_pitch, long long *max_frames);
int highlight_slot_commit(cvvp_ctx *ctx, long long n);
int highlight_queue_next_view(cvvp_ctx *ctx, const uint8_t **h_masks, size_t *mask_pitch, long long *n_out,
                              const cvvp_component **comps, const int **ncomps);
int highlight_queue_view_release(cvvp_ctx *ctx);
// median_roll.cu: backgrounds of outputs [t0, t1) of a rolling-window median; frame i at d_frames + (i % ring) * stride
int median_roll_launch(cvvp_ctx *ctx, const uint8_t *d_frames, long long ring, size_t frame_stride, long long nframes,
                       size_t nelem, int window, int percent, long long t0, long long t1, uint8_t *d_out, size_t out_stride,
                       cudaStream_t stream);
// highlight_rolling.cu
void highlight_rolling_release(cvvp_ctx *ctx);
int highlight_rolling_begin(cvvp_ctx *ctx, int window, long long max_batch, const cvvp_frame_format *fmt, int max_comps,
                            int labels);
int highlight_rolling_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride);
int highlight_rolling_close(cvvp_ctx *ctx);
int highlight_rolling_pending(const cvvp_ctx *ctx);
int highlight_rolling_ready(cvvp_ctx *ctx);
int highlight_rolling_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long max_n, long long *first_index,
                           long long *n_out, cvvp_component *comps_out, int *ncomps_out, int32_t *labels_out,
                           size_t labels_stride);
// highlight.cu: geometry of the running job (false: no job)
bool highlight_geometry(const cvvp_ctx *ctx, int *width, int *height);
// synth.cu
int synth_launch(cvvp_ctx *ctx, uint8_t *d_frames, size_t frame_stride, int width, int height, int row0, int nrows,
                 long long first_frame, long long nframes, uint32_t seed, int ndisks, cudaStream_t stream);
} // namespace cvvp
