// extern "C" entry points of libcvvp_cuda.so (include/cvvp.h): context management, the streaming
// (host-buffer) median job with pinned staging and stream/event pipelining, and the
// device-resident forms used by the benchmark.  No C++ exception leaves this file.
#include "context.hpp"
#include "pool.hpp"

#include <climits>
#include <cstdlib>
#include <cstring>
#include <new>

namespace cvvp
{
namespace
{
thread_local std::string g_err;
constexpr size_t kStagingBytes = size_t(32) << 20; // per pinned staging buffer
constexpr int kStagingBufs = 3;
} // namespace

void set_global_error(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

const char *global_error()
{
    return g_err.c_str();
}

int fail(cvvp_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx)
        ctx->err = buf;
    else
        g_err = buf;
    return code;
}

namespace
{
void release_median(cvvp_ctx *ctx)
{
    MedianJob &m = ctx->med;
    m.active = false;
    m.count = 0;
    m.folded = 0;
    m.split = false;
    m.half = 0;
    m.base = 0;
    // device buffers are kept for reuse by the next job of the same context
}

// Device frame stack of the streaming median job.  While they fit, the job keeps EVERY pushed frame resident (the
// on-chip select needs all of them at once): frames x round_up(nelem, 128) bytes.  The stack is sized EXACTLY to what
// is asked for (the hint of cvvp_median_begin, rounded up to a granule of 16 frames) and grows by half only when more
// frames arrive than were announced; while it grows the old and the new stack coexist, which an exact hint avoids
// altogether.  CVVP_ERR_NOMEM from here is not the end of the job: reserve_frames() below then folds the resident
// frames into value histograms and reuses the stack (the reference's histograms do not depend on the frame count
// either, histogram_median_algo.h:123-126).
int ensure_stack(cvvp_ctx *ctx, long long frames_needed)
{
    MedianJob &m = ctx->med;
    if (frames_needed <= m.capacity)
        return CVVP_OK;
    constexpr long long kGranule = 16;
    long long new_cap = (frames_needed + kGranule - 1) / kGranule * kGranule;
    if (m.capacity > 0 && m.count > 0) { // growing past what was announced: geometric, so pushes stay amortised O(1)
        const long long grown = (m.capacity + m.capacity / 2 + kGranule - 1) / kGranule * kGranule;
        if (grown > new_cap)
            new_cap = grown;
    }
    size_t bytes = size_t(new_cap) * m.stride;
    if (bytes > m.d_stack_bytes) {
        uint8_t *fresh = nullptr;
        if (cudaMalloc(&fresh, bytes) != cudaSuccess) {
            cudaGetLastError();
            // the geometric slack did not fit: retry with exactly what is needed now
            new_cap = (frames_needed + kGranule - 1) / kGranule * kGranule;
            bytes = size_t(new_cap) * m.stride;
            if (bytes <= m.d_stack_bytes || cudaMalloc(&fresh, bytes) != cudaSuccess) {
                cudaGetLastError();
                size_t free_b = 0, total_b = 0;
                cudaMemGetInfo(&free_b, &total_b);
                cudaGetLastError();
                return fail(ctx, CVVP_ERR_NOMEM,
                            "median: cudaMalloc of %zu bytes for a stack of %lld frames x %zu bytes failed (%zu bytes free); the "
                            "job keeps every frame resident, so frames x frame bytes must fit the device",
                            bytes, new_cap, m.stride, free_b);
            }
        }
        if (m.d_stack && m.count > 0) {
            // frames prepared on the device (cvvp_median_push_source) are written by kernels on the compute stream
            CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
            CVVP_CUDA_OK(ctx, cudaMemcpyAsync(fresh, m.d_stack, size_t(m.count) * m.stride, cudaMemcpyDeviceToDevice, ctx->copy));
            CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy));
        }
        if (m.d_stack)
            cudaFree(m.d_stack);
        m.d_stack = fresh;
        m.d_stack_bytes = bytes;
    }
    m.capacity = (long long)(m.d_stack_bytes / m.stride);
    return CVVP_OK;
}

// CVVP_MEDIAN_RESIDENT_MAX=<frames> (development switch, tests): the resident stack holds at most that many frames, so
// that small jobs exercise the constant-memory form
long long resident_limit()
{
    const char *e = getenv("CVVP_MEDIAN_RESIDENT_MAX");
    if (!e || !*e)
        return LLONG_MAX;
    const long long v = atoll(e);
    return v >= 1 ? v : 1;
}

// The frames of the region being filled go into the value histograms (median_hist.cu), asynchronously, and the job
// moves on to the other half of the stack: uploads into one half overlap the fold of the other.  The first fold reads
// the whole stack (it was filled as one region); the halves start behind it.
int spill_resident(cvvp_ctx *ctx)
{
    MedianJob &m = ctx->med;
    if (m.count == 0)
        return CVVP_OK;
    const size_t bytes = median_hist_bytes(m.stride);
    if (m.d_hist_bytes != bytes) {
        if (m.d_hist)
            cudaFree(m.d_hist);
        m.d_hist = nullptr;
        m.d_hist_bytes = 0;
        if (cudaMalloc(&m.d_hist, bytes) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM,
                        "median: the frame stack cannot grow beyond %lld frames and the %zu bytes of value histograms that "
                        "would take their place do not fit the device either",
                        m.capacity, bytes);
        }
        m.d_hist_bytes = bytes;
    }
    for (auto &ev : m.ev_fold)
        if (!ev)
            CVVP_CUDA_OK(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    if (m.folded == 0)
        CVVP_CUDA_OK(ctx, cudaMemsetAsync(m.d_hist, 0, bytes, ctx->compute));
    // uploads still in flight on the copy stream come first (preparation kernels run on the compute stream itself)
    CVVP_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copy, ctx->copy));
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->compute, ctx->ev_copy, 0));
    const int rc = median_hist_fold(ctx, m.d_stack + size_t(m.base) * m.stride, m.count, m.stride, m.d_hist, ctx->compute);
    if (rc != CVVP_OK)
        return rc;
    if (m.split) {
        CVVP_CUDA_OK(ctx, cudaEventRecord(m.ev_fold[m.half], ctx->compute));
        m.half ^= 1;
    } else {
        // the whole stack was one region: both halves are free once this fold is done
        CVVP_CUDA_OK(ctx, cudaEventRecord(m.ev_fold[0], ctx->compute));
        CVVP_CUDA_OK(ctx, cudaEventRecord(m.ev_fold[1], ctx->compute));
        const long long limit = resident_limit();
        const long long eff = m.capacity < limit ? m.capacity : limit;
        m.split = eff >= 2;
        m.half_cap = m.split ? eff / 2 : eff;
        m.half = 0;
    }
    m.base = m.split ? (long long)m.half * m.half_cap : 0;
    m.folded += m.count;
    m.count = 0;
    // the copy stream may write the next region only after the fold that last read it
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy, m.ev_fold[m.half], 0));
    return CVVP_OK;
}

// Room for the next frames of a push: *take <- how many of `want` frames fit behind the resident ones right now
// (at least one).  The stack grows as ensure_stack() allows; when it cannot, the resident frames are folded into the
// value histograms and the stack is reused -- from there on the job's memory no longer depends on the frame count,
// like the reference's (histogram_median_algo.h:123-126).
int reserve_frames(cvvp_ctx *ctx, long long want, long long *take)
{
    MedianJob &m = ctx->med;
    int rc = CVVP_OK;
    if (m.folded > 0) {
        // constant-memory form: the region being filled is a half of the stack (or all of a one-frame stack)
        if (m.half_cap - m.count <= 0 && (rc = spill_resident(ctx)) != CVVP_OK)
            return rc;
        const long long room = m.half_cap - m.count;
        *take = want < room ? want : room;
        return CVVP_OK;
    }
    const long long limit = resident_limit();
    long long need = m.count + want;
    if (need > limit)
        need = limit;
    rc = ensure_stack(ctx, need);
    if (rc == CVVP_ERR_NOMEM && m.capacity == 0) {
        // not even the first allocation fits: take half of what is free beside the histograms
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        cudaGetLastError();
        const size_t hist = median_hist_bytes(m.stride);
        const long long frames = free_b > hist ? (long long)((free_b - hist) / 2 / m.stride) : 0;
        if (frames >= 16)
            rc = ensure_stack(ctx, frames);
    }
    if (rc != CVVP_OK && !(rc == CVVP_ERR_NOMEM && m.capacity > 0))
        return rc;
    long long room = (m.capacity < limit ? m.capacity : limit) - m.count;
    if (room <= 0) {
        if ((rc = spill_resident(ctx)) != CVVP_OK)
            return rc;
        room = m.half_cap;
    }
    *take = want < room ? want : room;
    return CVVP_OK;
}

int ensure_staging(cvvp_ctx *ctx)
{
    if (!ctx->staging.empty())
        return CVVP_OK;
    ctx->staging.resize(kStagingBufs);
    for (auto &b : ctx->staging) {
        if (cudaMallocHost(&b.host, kStagingBytes) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM, "pinned staging allocation failed");
        }
        b.bytes = kStagingBytes;
        CVVP_CUDA_OK(ctx, cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
    }
    return CVVP_OK;
}

bool is_pinned(const void *p)
{
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}
} // namespace
} // namespace cvvp

using namespace cvvp;

namespace cvvp
{
namespace
{
// n frames behind the resident ones (room has been reserved)
int push_piece(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    MedianJob &m = ctx->med;
    int rc = CVVP_OK;
    uint8_t *dst = m.d_stack + size_t(m.base + m.count) * m.stride;
    if (is_pinned(frames)) {
        // DMA straight from the caller's pinned buffer
        if (frame_stride == m.stride && m.stride == m.nelem) {
            CVVP_CUDA_OK(ctx, cudaMemcpyAsync(dst, frames, size_t(n) * m.stride, cudaMemcpyHostToDevice, ctx->copy));
        } else {
            CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(dst, m.stride, frames, frame_stride, m.nelem, size_t(n),
                                                cudaMemcpyHostToDevice, ctx->copy));
        }
    } else {
        // pageable source: stage through the pinned ring, copies overlap the next memcpy
        rc = ensure_staging(ctx);
        if (rc != CVVP_OK)
            return rc;
        const long long per_buf = (long long)(kStagingBytes / m.nelem);
        auto next_buf = [&]() -> StagingBuf * {
            StagingBuf &b = ctx->staging[ctx->staging_next];
            ctx->staging_next = (ctx->staging_next + 1) % ctx->staging.size();
            if (b.in_flight) {
                if (cudaEventSynchronize(b.done) != cudaSuccess)
                    return nullptr;
                b.in_flight = false;
            }
            return &b;
        };
        if (per_buf == 0) {
            // a single frame is larger than a staging buffer (an 8K frame, a 4K colour frame): pieces of the frame
            for (long long i = 0; i < n; ++i) {
                for (size_t off = 0; off < m.nelem; off += kStagingBytes) {
                    const size_t piece = m.nelem - off < kStagingBytes ? m.nelem - off : kStagingBytes;
                    StagingBuf *b = next_buf();
                    if (!b)
                        return fail(ctx, CVVP_ERR_CUDA, "median: waiting for a staging buffer failed");
                    std::memcpy(b->host, frames + size_t(i) * frame_stride + off, piece);
                    CVVP_CUDA_OK(ctx, cudaMemcpyAsync(dst + size_t(i) * m.stride + off, b->host, piece, cudaMemcpyHostToDevice, ctx->copy));
                    CVVP_CUDA_OK(ctx, cudaEventRecord(b->done, ctx->copy));
                    b->in_flight = true;
                }
            }
        }
        for (long long done = 0; per_buf > 0 && done < n;) {
            const long long chunk = (n - done) < per_buf ? (n - done) : per_buf;
            StagingBuf *bp = next_buf();
            if (!bp)
                return fail(ctx, CVVP_ERR_CUDA, "median: waiting for a staging buffer failed");
            StagingBuf &b = *bp;
            for (long long i = 0; i < chunk; ++i)
                std::memcpy(b.host + size_t(i) * m.nelem, frames + size_t(done + i) * frame_stride, m.nelem);
            CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(dst + size_t(done) * m.stride, m.stride, b.host, m.nelem, m.nelem,
                                                size_t(chunk), cudaMemcpyHostToDevice, ctx->copy));
            CVVP_CUDA_OK(ctx, cudaEventRecord(b.done, ctx->copy));
            b.in_flight = true;
            done += chunk;
        }
    }
    m.count += n;
    return CVVP_OK;
}
} // namespace
} // namespace cvvp

extern "C" {

int cvvp_abi_version(void)
{
    return CVVP_ABI_VERSION;
}

int cvvp_ctx_create(int device, cvvp_ctx **out_ctx)
{
    if (!out_ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "cvvp_ctx_create: out_ctx is NULL");
    *out_ctx = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, CVVP_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess)
            device = 0;
    }
    if (device >= ndev)
        return fail(nullptr, CVVP_ERR_INVALID, "device %d out of range (%d devices)", device, ndev);
    cvvp_ctx *ctx = new (std::nothrow) cvvp_ctx();
    if (!ctx)
        return fail(nullptr, CVVP_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    DeviceGuard guard(device);
    cudaDeviceProp prop{};
    int rc = CVVP_OK;
    auto bail = [&](const char *what, cudaError_t err) {
        rc = fail(nullptr, CVVP_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(err));
        cvvp_ctx_destroy(ctx);
        return rc;
    };
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
        return bail("cudaGetDeviceProperties", e);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (prop.major != 10) {
        fail(nullptr, CVVP_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
             prop.major, prop.minor);
        cvvp_ctx_destroy(ctx);
        return CVVP_ERR_UNSUPPORTED;
    }
    if ((e = cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking)) != cudaSuccess)
        return bail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy, cudaStreamNonBlocking)) != cudaSuccess)
        return bail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking)) != cudaSuccess)
        return bail("cudaStreamCreate", e);
    if ((e = cudaEventCreate(&ctx->ev_start)) != cudaSuccess)
        return bail("cudaEventCreate", e);
    if ((e = cudaEventCreate(&ctx->ev_stop)) != cudaSuccess)
        return bail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming)) != cudaSuccess)
        return bail("cudaEventCreate", e);
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres{};
    e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        cudaGetLastError();
        fail(nullptr, CVVP_ERR_CUDA, "cuTensorMapEncodeTiled is not exported by this driver");
        cvvp_ctx_destroy(ctx);
        return CVVP_ERR_CUDA;
    }
    ctx->encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
    *out_ctx = ctx;
    return CVVP_OK;
}

void cvvp_ctx_destroy(cvvp_ctx *ctx)
{
    if (!ctx)
        return;
    DeviceGuard guard(ctx->device);
    if (ctx->compute)
        cudaStreamSynchronize(ctx->compute);
    if (ctx->copy)
        cudaStreamSynchronize(ctx->copy);
    if (ctx->copy_out)
        cudaStreamSynchronize(ctx->copy_out);
    for (auto &b : ctx->staging) {
        if (b.done)
            cudaEventDestroy(b.done);
        if (b.host)
            cudaFreeHost(b.host);
    }
    highlight_queue_release(ctx);
    highlight_rolling_release(ctx);
    highlight_release(ctx);
    raw_stage_release(ctx);
    median_shard_release(ctx);
    if (ctx->med.d_stack)
        cudaFree(ctx->med.d_stack);
    if (ctx->med.d_hist)
        cudaFree(ctx->med.d_hist);
    for (auto &ev : ctx->med.ev_fold)
        if (ev)
            cudaEventDestroy(ev);
    if (ctx->med.d_out)
        cudaFree(ctx->med.d_out);
    if (ctx->ev_start)
        cudaEventDestroy(ctx->ev_start);
    if (ctx->ev_stop)
        cudaEventDestroy(ctx->ev_stop);
    if (ctx->ev_copy)
        cudaEventDestroy(ctx->ev_copy);
    if (ctx->compute)
        cudaStreamDestroy(ctx->compute);
    if (ctx->copy)
        cudaStreamDestroy(ctx->copy);
    if (ctx->copy_out)
        cudaStreamDestroy(ctx->copy_out);
    cudaGetLastError();
    delete ctx;
}

const char *cvvp_last_error(const cvvp_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : global_error();
}

int cvvp_ctx_synchronize(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy));
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy_out));
    for (auto &b : ctx->staging)
        b.in_flight = false;
    return CVVP_OK;
}

void *cvvp_ctx_stream(cvvp_ctx *ctx)
{
    return ctx ? static_cast<void *>(ctx->compute) : nullptr;
}

int cvvp_ctx_device(const cvvp_ctx *ctx)
{
    return ctx ? ctx->device : -1;
}

int cvvp_ctx_sm_count(const cvvp_ctx *ctx)
{
    return ctx ? ctx->sm_count : 0;
}

long long cvvp_ctx_launch_count(const cvvp_ctx *ctx)
{
    return ctx ? ctx->launches : 0;
}

int cvvp_host_alloc(size_t bytes, void **out_ptr)
{
    if (!out_ptr || bytes == 0)
        return fail(nullptr, CVVP_ERR_INVALID, "cvvp_host_alloc: bad arguments");
    *out_ptr = nullptr;
    cudaError_t e = cudaMallocHost(out_ptr, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, CVVP_ERR_NOMEM, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    return CVVP_OK;
}

int cvvp_host_free(void *ptr)
{
    if (!ptr)
        return CVVP_OK;
    cudaError_t e = cudaFreeHost(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, CVVP_ERR_CUDA, "cudaFreeHost failed: %s", cudaGetErrorString(e));
    }
    return CVVP_OK;
}

size_t cvvp_pool_trim(void)
{
    return pool_trim();
}

int cvvp_ctx_copy_to_host(cvvp_ctx *ctx, void *host_dst, const void *device_src, size_t bytes)
{
    if (!ctx || !host_dst || !device_src)
        return fail(ctx, CVVP_ERR_INVALID, "cvvp_ctx_copy_to_host: null argument");
    DeviceGuard guard(ctx->device);
    CVVP_CUDA_OK(ctx, cudaMemcpyAsync(host_dst, device_src, bytes, cudaMemcpyDeviceToHost, ctx->compute));
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->compute));
    return CVVP_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* median                                                                                      */
/* ------------------------------------------------------------------------------------------- */

int cvvp_median_begin(cvvp_ctx *ctx, size_t nelem, long long nframes_hint)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (ctx->med.active)
        return fail(ctx, CVVP_ERR_STATE, "median: a job is already running on this context");
    if (nelem == 0 || nelem >= (1ull << 31))
        return fail(ctx, CVVP_ERR_INVALID, "median: nelem must be in [1, 2^31)");
    DeviceGuard guard(ctx->device);
    MedianJob &m = ctx->med;
    const size_t stride = round_up(nelem, 128);
    if (stride != m.stride) {
        // geometry changed: the old stack cannot be reused as is
        if (m.d_stack)
            cudaFree(m.d_stack);
        m.d_stack = nullptr;
        m.d_stack_bytes = 0;
    }
    if (m.d_hist && m.d_hist_bytes != median_hist_bytes(stride)) {
        cudaFree(m.d_hist);
        m.d_hist = nullptr;
        m.d_hist_bytes = 0;
    }
    m.capacity = 0;
    m.nelem = nelem;
    m.stride = stride;
    m.count = 0;
    m.folded = 0;
    m.split = false;
    m.half = 0;
    m.base = 0;
    m.percent = ctx->percent; // the job keeps the percentile it began with
    if (m.d_out_bytes < stride) {
        if (m.d_out)
            cudaFree(m.d_out);
        m.d_out = nullptr;
        m.d_out_bytes = 0;
        if (cudaMalloc(&m.d_out, stride) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM, "median: cudaMalloc of the result buffer failed");
        }
        m.d_out_bytes = stride;
    }
    if (m.d_stack_bytes >= stride)
        m.capacity = (long long)(m.d_stack_bytes / stride);
    // a hint that does not fit leaves a smaller stack: the job then folds frames into value histograms as it goes
    long long room = 0;
    const int rc = reserve_frames(ctx, nframes_hint > 0 ? nframes_hint : 64, &room);
    if (rc != CVVP_OK)
        return rc;
    m.active = true;
    return CVVP_OK;
}

int cvvp_median_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    MedianJob &m = ctx->med;
    if (!m.active)
        return fail(ctx, CVVP_ERR_STATE, "median: push without begin");
    if (n == 0)
        return CVVP_OK;
    if (!frames || n < 0 || frame_stride < m.nelem)
        return fail(ctx, CVVP_ERR_INVALID, "median: bad push arguments");
    DeviceGuard guard(ctx->device);
    while (n > 0) {
        long long take = 0;
        int rc = reserve_frames(ctx, n, &take);
        if (rc != CVVP_OK)
            return rc;
        if ((rc = push_piece(ctx, frames, take, frame_stride)) != CVVP_OK)
            return rc;
        frames += size_t(take) * frame_stride;
        n -= take;
    }
    return CVVP_OK;
}

long long cvvp_median_count(const cvvp_ctx *ctx)
{
    return ctx ? ctx->med.count + ctx->med.folded : 0;
}

int cvvp_median_stack_device(cvvp_ctx *ctx, const uint8_t **d_frames, size_t *frame_stride, long long *nframes)
{
    if (!ctx || !d_frames || !frame_stride || !nframes)
        return fail(ctx, CVVP_ERR_INVALID, "median: null argument");
    MedianJob &m = ctx->med;
    if (!m.active)
        return fail(ctx, CVVP_ERR_STATE, "median: no job is running");
    if (m.folded > 0)
        return fail(ctx, CVVP_ERR_STATE, "median: %lld frames of this job were folded into value histograms (the stack did "
                                         "not fit the device); the frame stack is no longer complete", m.folded);
    DeviceGuard guard(ctx->device);
    // everything pushed so far is ordered before whatever the caller queues on the compute stream next
    CVVP_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copy, ctx->copy));
    CVVP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->compute, ctx->ev_copy, 0));
    *d_frames = m.d_stack;
    *frame_stride = m.stride;
    *nframes = m.count;
    return CVVP_OK;
}

int cvvp_median_finish(cvvp_ctx *ctx, uint8_t *out)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    MedianJob &m = ctx->med;
    if (!m.active)
        return fail(ctx, CVVP_ERR_STATE, "median: finish without begin");
    if (!out) {
        release_median(ctx);
        return fail(ctx, CVVP_ERR_INVALID, "median: out is NULL");
    }
    if (m.count + m.folded == 0) {
        // the reference publishes an empty Mat when no token was inserted; report it as a state error
        release_median(ctx);
        return fail(ctx, CVVP_ERR_STATE, "median: no frames were pushed");
    }
    DeviceGuard guard(ctx->device);
    int rc = CVVP_OK;
    do {
        cudaError_t e;
        if ((e = cudaEventRecord(ctx->ev_copy, ctx->copy)) != cudaSuccess ||
            (e = cudaStreamWaitEvent(ctx->compute, ctx->ev_copy, 0)) != cudaSuccess ||
            (e = cudaEventRecord(ctx->ev_start, ctx->compute)) != cudaSuccess) {
            rc = fail(ctx, CVVP_ERR_CUDA, "median: stream setup failed: %s", cudaGetErrorString(e));
            break;
        }
        if (m.folded > 0) {
            // constant-memory form: the rest of the stack joins the histograms, the median is read off them
            if ((rc = spill_resident(ctx)) != CVVP_OK)
                break;
            rc = median_hist_select(ctx, m.d_hist, m.stride, m.nelem, m.folded, m.percent, m.d_out, ctx->compute);
        } else {
            rc = median_launch(ctx, m.d_stack, m.count, m.nelem, m.stride, m.d_out, m.percent, ctx->compute);
        }
        if (rc != CVVP_OK)
            break;
        if ((e = cudaEventRecord(ctx->ev_stop, ctx->compute)) != cudaSuccess ||
            (e = cudaMemcpyAsync(out, m.d_out, m.nelem, cudaMemcpyDeviceToHost, ctx->compute)) != cudaSuccess ||
            (e = cudaStreamSynchronize(ctx->compute)) != cudaSuccess) {
            rc = fail(ctx, CVVP_ERR_CUDA, "median: kernel or result copy failed: %s", cudaGetErrorString(e));
            break;
        }
        ctx->have_kernel_time = true;
    } while (false);
    for (auto &b : ctx->staging)
        b.in_flight = false;
    release_median(ctx);
    return rc;
}

int cvvp_median_push_source(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format *fmt)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    MedianJob &m = ctx->med;
    if (!m.active)
        return fail(ctx, CVVP_ERR_STATE, "median: push without begin");
    int rc = frames_check_format(ctx, fmt);
    if (rc != CVVP_OK)
        return rc;
    if (frames_out_bytes(*fmt) != m.nelem)
        return fail(ctx, CVVP_ERR_INVALID, "median: prepared frames have %zu bytes, the job was begun with %zu",
                    frames_out_bytes(*fmt), m.nelem);
    if (n == 0)
        return CVVP_OK;
    const size_t src_frame = size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels);
    if (!frames || n < 0 || frame_stride < src_frame)
        return fail(ctx, CVVP_ERR_INVALID, "median: bad push arguments");
    DeviceGuard guard(ctx->device);
    while (n > 0) {
        long long take = 0;
        if ((rc = reserve_frames(ctx, n, &take)) != CVVP_OK)
            return rc;
        if ((rc = frames_upload_prepare(ctx, frames, take, frame_stride, *fmt, m.d_stack + size_t(m.base + m.count) * m.stride, m.stride)) != CVVP_OK)
            return rc;
        m.count += take;
        frames += size_t(take) * frame_stride;
        n -= take;
    }
    // the caller may reuse `frames` on return: wait for the uploads (not for the kernels) -- a pageable source is
    // already staged at this point, a pinned one is still being read by the copy engine
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy));
    return CVVP_OK;
}

int cvvp_median_abort(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->copy);
    cudaStreamSynchronize(ctx->compute);
    for (auto &b : ctx->staging)
        b.in_flight = false;
    release_median(ctx);
    return CVVP_OK;
}

int cvvp_median_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                       uint8_t *d_out, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return median_launch(ctx, d_frames, nframes, nelem, frame_stride, d_out, ctx->percent, s);
}

int cvvp_median_rolling_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                               int window, long long t0, long long t1, uint8_t *d_out, size_t out_stride, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return median_roll_launch(ctx, d_frames, nframes, frame_stride, nframes, nelem, window, ctx->percent, t0, t1, d_out,
                              out_stride, s);
}

int cvvp_median_set_percentile(cvvp_ctx *ctx, int percent)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (percent < 0 || percent > 100)
        return fail(ctx, CVVP_ERR_INVALID, "median: percentile %d outside [0, 100]", percent);
    // open jobs took the percentile when they began; changing it underneath them would mix two rank rules
    if (ctx->med.active || ctx->shard || ctx->hr)
        return fail(ctx, CVVP_ERR_STATE, "median: a median, sharded or rolling job is open on this context");
    ctx->percent = percent;
    return CVVP_OK;
}

int cvvp_median_percentile(const cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return ctx->percent;
}

int cvvp_median_last_kernel_ms(cvvp_ctx *ctx, float *out_ms)
{
    if (!ctx || !out_ms)
        return fail(ctx, CVVP_ERR_INVALID, "bad arguments");
    if (!ctx->have_kernel_time)
        return fail(ctx, CVVP_ERR_STATE, "no median kernel has been timed on this context");
    DeviceGuard guard(ctx->device);
    CVVP_CUDA_OK(ctx, cudaEventElapsedTime(out_ms, ctx->ev_start, ctx->ev_stop));
    return CVVP_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* highlight                                                                                   */
/* ------------------------------------------------------------------------------------------- */

int cvvp_highlight_begin(cvvp_ctx *ctx, const uint8_t *background, int width, int height, const uint8_t *struct_element,
                         int kw, int kh, int threshold, int threshold_lo, int threshold_hi, int min_size_hyst,
                         int min_size_threshold, int width_border)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    (void)width_border; // accepted and unused, exactly like the reference (FrameAndFill is dead code, :68-71)
    DeviceGuard guard(ctx->device);
    highlight_queue_release(ctx);
    highlight_rolling_release(ctx);
    return highlight_begin(ctx, background, width, height, struct_element, kw, kh, threshold, threshold_lo, threshold_hi,
                           min_size_hyst, min_size_threshold);
}

int cvvp_highlight_set_polarity(cvvp_ctx *ctx, int polarity)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (polarity != CVVP_POLARITY_DARK && polarity != CVVP_POLARITY_BRIGHT && polarity != CVVP_POLARITY_BOTH)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: unknown polarity %d", polarity);
    // an open job, its queue and its rolling stream took the polarity in cvvp_highlight_begin
    if (ctx->hl)
        return fail(ctx, CVVP_ERR_STATE, "highlight: a highlight job is open on this context");
    ctx->polarity = polarity;
    return CVVP_OK;
}

int cvvp_highlight_polarity(const cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return ctx->polarity;
}

int cvvp_highlight_set_channels(cvvp_ctx *ctx, int channels)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (channels < 1 || channels > 4)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: channels must be in 1..4, not %d", channels);
    // an open job, its queue and its rolling stream took the channel count (and their buffers) in cvvp_highlight_begin
    if (ctx->hl)
        return fail(ctx, CVVP_ERR_STATE, "highlight: a highlight job is open on this context");
    ctx->channels = channels;
    return CVVP_OK;
}

int cvvp_highlight_channels(const cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return ctx->channels;
}

int cvvp_highlight_set_component_stats(cvvp_ctx *ctx, int on)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (on != 0 && on != 1)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: component statistics must be 0 or 1, not %d", on);
    // an open job, its queue and its rolling stream took the setting (and their record size) in cvvp_highlight_begin
    if (ctx->hl)
        return fail(ctx, CVVP_ERR_STATE, "highlight: a highlight job is open on this context");
    ctx->component_stats = on;
    return CVVP_OK;
}

int cvvp_highlight_component_stats(const cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return ctx->component_stats;
}

int cvvp_highlight_frames(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                          size_t out_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_frames_host(ctx, frames, n, frame_stride, masks_out, out_stride);
}

int cvvp_highlight_device(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride, uint8_t *d_out,
                          size_t out_stride, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return highlight_device_bg(ctx, d_frames, n, frame_stride, nullptr, 0, d_out, out_stride, CcOut(), s);
}

int cvvp_highlight_device_cc(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride, uint8_t *d_out,
                             size_t out_stride, cvvp_component *d_comps, int max_comps, int *d_ncomps, int32_t *d_labels,
                             size_t labels_stride, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    // components are required here, and their arguments and the path are checked before the frame arguments
    const CcOut cc{d_comps, max_comps, d_ncomps, d_labels, labels_stride};
    const int rc = highlight_check_cc(ctx, n, cc);
    return rc != CVVP_OK ? rc : highlight_device_bg(ctx, d_frames, n, frame_stride, nullptr, 0, d_out, out_stride, cc, s);
}

int cvvp_highlight_device_bg(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride,
                             const uint8_t *d_backgrounds, size_t bg_stride, uint8_t *d_out, size_t out_stride,
                             cvvp_component *d_comps, int max_comps, int *d_ncomps, int32_t *d_labels, size_t labels_stride,
                             void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    // this entry point requires backgrounds: to the internal call a null one means the job's own
    if (!d_backgrounds && ctx->hl)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: bad arguments (null backgrounds)");
    return highlight_device_bg(ctx, d_frames, n, frame_stride, d_backgrounds, bg_stride, d_out, out_stride,
                               CcOut{d_comps, max_comps, d_ncomps, d_labels, labels_stride}, s);
}

int cvvp_highlight_frames_cc(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                             size_t out_stride, cvvp_component *comps_out, int max_comps, int *ncomps_out,
                             int32_t *labels_out, size_t labels_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_frames_host_cc(ctx, frames, n, frame_stride, masks_out, out_stride, comps_out, max_comps, ncomps_out,
                                    labels_out, labels_stride);
}

int cvvp_highlight_end(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    sync_streams(ctx);
    highlight_queue_release(ctx);
    highlight_rolling_release(ctx);
    highlight_release(ctx);
    return CVVP_OK;
}

int cvvp_highlight_set_path(cvvp_ctx *ctx, int path)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return highlight_set_path(ctx, path);
}

int cvvp_highlight_frames_in_flight(cvvp_ctx *ctx, int *out_frames)
{
    if (!ctx || !out_frames)
        return fail(ctx, CVVP_ERR_INVALID, "null argument");
    DeviceGuard guard(ctx->device);
    return highlight_frames_in_flight(ctx, out_frames);
}

/* ------------------------------------------------------------------------------------------- */
/* frame source, asynchronous highlight queue                                                  */
/* ------------------------------------------------------------------------------------------- */

size_t cvvp_frame_format_out_bytes(const cvvp_frame_format *fmt)
{
    return fmt ? frames_out_bytes(*fmt) : 0;
}

int cvvp_frames_prepare_device(cvvp_ctx *ctx, const uint8_t *d_src, long long n, size_t src_stride, const cvvp_frame_format *fmt,
                               uint8_t *d_dst, size_t dst_stride, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    int rc = frames_check_format(ctx, fmt);
    if (rc != CVVP_OK)
        return rc;
    const size_t src_frame = size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels);
    if (!d_src || !d_dst || n < 0 || src_stride < src_frame || dst_stride < frames_out_bytes(*fmt))
        return fail(ctx, CVVP_ERR_INVALID, "frames: bad arguments");
    if (n == 0)
        return CVVP_OK;
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return frames_prepare_launch(ctx, d_src, n, src_stride, size_t(n - 1) * src_stride + src_frame, *fmt, 0, d_dst, dst_stride, s);
}

int cvvp_frames_prepare(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, const cvvp_frame_format *fmt,
                        uint8_t *out, size_t out_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    int rc = frames_check_format(ctx, fmt);
    if (rc != CVVP_OK)
        return rc;
    const size_t src_frame = size_t(fmt->src_width) * size_t(fmt->src_height) * size_t(fmt->src_channels);
    if (!frames || !out || n < 0 || frame_stride < src_frame || out_stride < frames_out_bytes(*fmt))
        return fail(ctx, CVVP_ERR_INVALID, "frames: bad arguments");
    if (n == 0)
        return CVVP_OK;
    DeviceGuard guard(ctx->device);
    return frames_prepare_host(ctx, frames, n, frame_stride, *fmt, out, out_stride);
}

int cvvp_highlight_queue_begin(cvvp_ctx *ctx, int depth, long long max_batch, const cvvp_frame_format *fmt, int max_comps)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_queue_begin(ctx, depth, max_batch, fmt, max_comps);
}

int cvvp_highlight_queue_pending(const cvvp_ctx *ctx)
{
    return ctx ? highlight_queue_pending(ctx) : 0;
}

int cvvp_highlight_submit(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_queue_submit(ctx, frames, n, frame_stride);
}

int cvvp_highlight_queue_ready(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_queue_ready(ctx);
}

int cvvp_highlight_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long *n_out, cvvp_component *comps_out,
                        int *ncomps_out)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_queue_next(ctx, masks_out, out_stride, n_out, comps_out, ncomps_out);
}

int cvvp_highlight_slot_acquire(cvvp_ctx *ctx, uint8_t **h_frames, size_t *frame_pitch, long long *max_frames)
{
    if (!ctx || !h_frames || !frame_pitch)
        return fail(ctx, CVVP_ERR_INVALID, "null argument");
    return highlight_slot_acquire(ctx, h_frames, frame_pitch, max_frames);
}

int cvvp_highlight_slot_commit(cvvp_ctx *ctx, long long n)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_slot_commit(ctx, n);
}

int cvvp_highlight_next_view(cvvp_ctx *ctx, const uint8_t **h_masks, size_t *mask_pitch, long long *n_out,
                             const cvvp_component **comps, const int **ncomps)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_queue_next_view(ctx, h_masks, mask_pitch, n_out, comps, ncomps);
}

int cvvp_highlight_view_release(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    return highlight_queue_view_release(ctx);
}

int cvvp_highlight_queue_end(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    highlight_queue_release(ctx);
    return CVVP_OK;
}

int cvvp_highlight_rolling_begin(cvvp_ctx *ctx, int window, long long max_batch, const cvvp_frame_format *fmt, int max_comps,
                                 int labels)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_rolling_begin(ctx, window, max_batch, fmt, max_comps, labels);
}

int cvvp_highlight_rolling_push(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_rolling_push(ctx, frames, n, frame_stride);
}

int cvvp_highlight_rolling_close(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_rolling_close(ctx);
}

int cvvp_highlight_rolling_pending(const cvvp_ctx *ctx)
{
    return ctx ? highlight_rolling_pending(ctx) : 0;
}

int cvvp_highlight_rolling_ready(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_rolling_ready(ctx);
}

int cvvp_highlight_rolling_next(cvvp_ctx *ctx, uint8_t *masks_out, size_t out_stride, long long max_n, long long *first_index,
                                long long *n_out, cvvp_component *comps_out, int *ncomps_out, int32_t *labels_out,
                                size_t labels_stride)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    return highlight_rolling_next(ctx, masks_out, out_stride, max_n, first_index, n_out, comps_out, ncomps_out, labels_out,
                                  labels_stride);
}

int cvvp_highlight_rolling_end(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    highlight_rolling_release(ctx);
    return CVVP_OK;
}

int cvvp_synth_frames_device(cvvp_ctx *ctx, uint8_t *d_frames, size_t frame_stride, int width, int height, int row0,
                             int nrows, long long first_frame, long long nframes, uint32_t seed, int ndisks, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return synth_launch(ctx, d_frames, frame_stride, width, height, row0, nrows, first_frame, nframes, seed, ndisks, s);
}

} // extern "C"
