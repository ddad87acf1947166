// Constant-memory form of the streaming median job: value histograms per element, for frame stacks that do not fit
// the device -- the direct analogue of HistogramMedianAlgo<T>
// (/root/reference/Sources/ProcessorAlgos/histogram_median_algo.h:116-193: ConsumeVector adds one to
// histogram[element][value], MedianFromHistograms returns the first bin whose cumulative count exceeds N/2), whose
// memory does not depend on the frame count either.
//
// The job normally keeps every frame resident and selects on chip (median_pipe.cu); only when the resident stack
// cannot grow any further does abi.cu FOLD the resident frames into 256 planes of 32-bit counts,
// hist[value][element] (256 x round_up(nelem, 128) x 4 bytes: 2.1 GB for a 1080p grey frame), and reuse the stack for
// the frames that follow.  32-bit counts never saturate (2^32 frames), so there is no bin-width choice to make
// (cv_vid_bg_helpers.cpp:232-253).
//
//   fold   : one thread per four elements walks the resident frames (a 32-bit load per frame, coalesced over the
//            warp) and bumps hist[v][e] -- plain read-modify-write, the thread owns its elements.  A run of equal
//            values costs one update.  Neighbouring elements of a video background have neighbouring values, so the
//            updates of a warp land in few planes.  HBM/L2-bound integer work at about three times the rate of the
//            PCIe link that feeds the job; abi.cu overlaps it with the uploads (two stack halves).
//   select : one thread per element accumulates the 256 planes (coalesced) until the count exceeds k(N, p)
//            (percentile_rank; N/2 at the default p = 50).
#include "context.hpp"
#include "median_common.cuh"

namespace cvvp
{
namespace
{
constexpr int kHistThreads = 256;

__global__ void __launch_bounds__(kHistThreads) median_hist_fold_kernel(const uint8_t *__restrict__ stack, const uint32_t nframes,
                                                                         const size_t frame_stride, const uint32_t nquads,
                                                                         uint32_t *__restrict__ hist, const size_t plane)
{
    const uint32_t q = blockIdx.x * kHistThreads + threadIdx.x;
    if (q >= nquads)
        return;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(stack) + q;
    const size_t words_per_frame = frame_stride / 4u;
    uint32_t *h = hist + 4u * size_t(q);
    // last value and its pending count, per byte lane
    uint32_t last = __ldcs(src);
    uint32_t run[4] = {0, 0, 0, 0};
    for (uint32_t f = 0; f < nframes; ++f) {
        const uint32_t w = __ldcs(src + size_t(f) * words_per_frame);
        const uint32_t diff = w ^ last;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            if ((diff >> (8 * b)) & 0xFFu) {
                h[size_t((last >> (8 * b)) & 0xFFu) * plane + b] += run[b];
                run[b] = 1;
            } else {
                ++run[b];
            }
        }
        last = w;
    }
#pragma unroll
    for (int b = 0; b < 4; ++b)
        h[size_t((last >> (8 * b)) & 0xFFu) * plane + b] += run[b];
}

__global__ void __launch_bounds__(kHistThreads) median_hist_select_kernel(const uint32_t *__restrict__ hist, const size_t plane,
                                                                           const uint32_t nelem, const unsigned long long rank,
                                                                           uint8_t *__restrict__ out)
{
    const uint32_t e = blockIdx.x * kHistThreads + threadIdx.x;
    if (e >= nelem)
        return;
    // first bin whose cumulative count exceeds the rank (N/2 at p = 50: the reference's rule, :160-166)
    unsigned long long cum = 0;
    uint32_t v = 0;
    for (; v < 255u; ++v) {
        cum += __ldcs(hist + size_t(v) * plane + e);
        if (cum > rank)
            break;
    }
    out[e] = uint8_t(v);
}
} // namespace

size_t median_hist_bytes(size_t frame_stride)
{
    return size_t(256) * frame_stride * sizeof(uint32_t);
}

// hist[value * frame_stride + element] += occurrences of `value` at `element` in the nframes resident frames
int median_hist_fold(cvvp_ctx *ctx, const uint8_t *d_stack, long long nframes, size_t frame_stride, uint32_t *d_hist,
                     cudaStream_t stream)
{
    if (nframes <= 0)
        return CVVP_OK;
    if (nframes >= (1ll << 32) || (frame_stride & 3u))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: cannot fold %lld frames of pitch %zu", nframes, frame_stride);
    // every word of the pitch is folded (the pad bytes behind nelem are zero or stale: their counts are never read)
    const uint32_t nquads = uint32_t(frame_stride / 4u);
    const uint32_t grid = (nquads + kHistThreads - 1) / kHistThreads;
    median_hist_fold_kernel<<<grid, kHistThreads, 0, stream>>>(d_stack, uint32_t(nframes), frame_stride, nquads, d_hist, frame_stride);
    CVVP_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches++;
    return CVVP_OK;
}

int median_hist_select(cvvp_ctx *ctx, const uint32_t *d_hist, size_t frame_stride, size_t nelem, long long total, int percent,
                       uint8_t *d_out, cudaStream_t stream)
{
    const uint32_t grid = uint32_t((nelem + kHistThreads - 1) / kHistThreads);
    median_hist_select_kernel<<<grid, kHistThreads, 0, stream>>>(d_hist, frame_stride, uint32_t(nelem),
                                                                  percentile_rank<uint64_t>(uint64_t(total), uint32_t(percent)), d_out);
    CVVP_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches++;
    return CVVP_OK;
}
} // namespace cvvp
