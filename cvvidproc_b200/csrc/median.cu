// Temporal median of a uint8 frame stack on sm_100a -- replaces HistogramMedianAlgo<T>
// (/root/reference/Sources/ProcessorAlgos/histogram_median_algo.h:116-193).
//
// The reference builds a 256-bin histogram per element and returns the first bin whose
// cumulative count exceeds N/2, i.e. sorted[N/2].  Every form here selects sorted[k(N, p)] instead
// (percentile_rank, median_common.cuh), which is sorted[N/2] at the default p = 50.  On B200 a shared-memory histogram costs one
// (atomic) read-modify-write per input byte and cannot keep up with HBM, so this kernel computes
// the same order statistic with an on-chip BIT-SLICED RADIX SELECT:
//
//   tile      = P consecutive elements (P = 128 >> LOG2S) x all N frames, resident on one SM;
//   streaming = a ring of 4 KB TMA boxes (P bytes x 4096/P frames each, zero-filled out of bounds).  There is NO
//               producer warp: each of the 12 transposer warps owns two private ring slots and re-issues the TMA
//               load of its own next stage as soon as its lanes have read a slot (median_pipe.cu), so no "empty"
//               barriers exist and every mbarrier wait is for the direct successor of a fill the warp consumed;
//   transpose = each transposer warp takes one 4 KB stage and turns 4 elements x 32 frame slots per lane into
//               4 elements x 8 bit planes, one word = 32 frames of one bit of one element (a 32x32 bit transpose per
//               lane).  At 128-byte tiles the two byte stages happen in the load: the stage lies 128B-swizzled in
//               shared memory and eight ldmatrix.m16n16.x2.trans.b8 (LDSM.8.MT1616) hand every lane registers that
//               hold four frame slots of ONE element; three shift/LOP3 stages remain.  Planes go to shared memory
//               (swizzled so both the stores and the select loads are bank-conflict free);
//   select    = 8 passes, MSB first: count = popc(alive & ~plane) summed over the element's frame
//               blocks (4..32 threads per element, warp shuffles), compare with the remaining
//               rank, keep the matching half (alive &= plane or ~plane).
//
// Frame order inside a plane word is irrelevant to an order statistic, and zero-filled padding
// frames are accounted for by raising the wanted rank by the number of pad slots, so no masks
// are needed.  HBM traffic is the algorithmic minimum: every input byte is read exactly once.
#include "context.hpp"

#include <cstdlib>

namespace cvvp
{
int median_launch(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                  uint8_t *d_out, int percent, cudaStream_t stream)
{
    if (!d_out)
        return fail(ctx, CVVP_ERR_INVALID, "median: null output pointer");
    // Up to 1024 frames the on-chip select reads every byte once at 128-byte tiles.  Up to 2048 frames it still fits at
    // 64-byte tiles, but TMA boxes of 64-byte rows cap the chip near 3 TB/s (one request per row: about 48 G requests/s
    // whatever the row length, profiles/r1_median_probe_tiles.txt), and a frame stride well beyond a 2 MiB page costs
    // another third there (profiles/r2_median_stride_probe.txt).  Counting passes in chunks of <= 1024 frames at full
    // tile width are faster from about 1300 frames on (1080p x 1500: 0.91 against 1.03 ms; 4K x 1200: 3.1 against
    // 4.3 ms) and reach 16 x 65535 frames (median_shard.cu).  CVVP_MEDIAN_TWO_PASS=0/1 forces either path (tests).
    // Long stacks first try ONE pass of window counting (median_pipe_kernel MODE 3: every 1024-frame launch counts
    // its frames in an 8-value window around its own pilot median; the owner kernel names the median wherever it
    // lies inside every launch's window) and run the two counting passes only over the 128-element tiles that hold an
    // undecided element -- the tile list is built on the device, so the call stays asynchronous.
    // CVVP_MEDIAN_WINDOW=0 skips the window pass (tests hold both to the oracle).
    const char *force = getenv("CVVP_MEDIAN_TWO_PASS");
    const bool long_stride = frame_stride > (5u << 19); // 2.5 MiB
    const bool two_pass = force ? force[0] == '1' : (nframes > 1280 || (nframes > 1024 && long_stride));
    if (two_pass || nframes > median_max_frames()) {
        if (nframes > median_two_pass_max_frames())
            return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: %lld frames exceed the supported maximum (%lld)", nframes,
                        median_two_pass_max_frames());
        const char *win = getenv("CVVP_MEDIAN_WINDOW");
        return median_long_stack(ctx, d_frames, nframes, nelem, frame_stride, d_out, percent, stream, win ? win[0] != '0' : 1);
    }
    return median_launch_mode(ctx, d_frames, nframes, nelem, frame_stride, d_out, 0, percent, ShardPush{}, stream);
}

// mode 0: on-chip select into d_out; modes 1 / 2 / 3: the counting rounds of a frame-sharded job (median_shard.cu).
// percent: the order statistic modes 0 and 3 select (percentile_rank, median_common.cuh)
int median_launch_mode(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                       uint8_t *d_out, int mode, int percent, const ShardPush &push, cudaStream_t stream)
{
    if (!d_frames || nframes <= 0 || nelem == 0)
        return fail(ctx, CVVP_ERR_INVALID, "median: null pointer or empty stack");
    if ((reinterpret_cast<uintptr_t>(d_frames) & 15u) || (frame_stride & 15u) || frame_stride < nelem)
        return fail(ctx, CVVP_ERR_INVALID,
                    "median: device stack must be 16-byte aligned with a frame stride that is a multiple of 16 and >= nelem");
    if (nelem >= (1ull << 31))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: more than 2^31 elements per frame");
    if (percent < 0 || percent > 100)
        return fail(ctx, CVVP_ERR_INVALID, "median: percentile %d outside [0, 100]", percent);
    if (nframes > median_max_frames())
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: %lld frames exceed the on-chip select capacity (%lld)", nframes,
                    median_max_frames());

    // widest tile (smallest LOG2S) whose bit planes fit on chip: P = 128 >> LOG2S elements, 32 << LOG2S frame
    // slots per 4 KB stage, at most 32 stages per tile
    int log2s = 0;
    uint32_t nst = 0;
    if (const char *e = getenv("CVVP_MEDIAN_LOG2S")) // development switch: narrowest tile variant to consider
        log2s = e[0] >= '0' && e[0] <= '3' ? e[0] - '0' : 0;
    for (; log2s <= 3; ++log2s) {
        const long long slots = 32ll << log2s;
        const long long need = (nframes + slots - 1) / slots;
        if (need <= 32) {
            nst = uint32_t(need);
            break;
        }
    }

    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {cuuint64_t(nelem), cuuint64_t(nframes)};
    const cuuint64_t gstride[1] = {cuuint64_t(frame_stride)};
    const cuuint32_t box[2] = {cuuint32_t(128 >> log2s), cuuint32_t(32 << log2s)};
    const cuuint32_t estride[2] = {1, 1};
    const CUresult cr = ctx->encode_tiled(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t *>(d_frames), gdim,
                                          gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                          // 128-byte rows are swizzled for the kernel's transposing matrix loads
                                          log2s == 0 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS)
        return fail(ctx, CVVP_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", int(cr));
    return median_pipe_launch(ctx, tmap, log2s, d_out, uint32_t(nelem), uint32_t(nframes), nst, mode, uint32_t(percent), push, stream);
}
} // namespace cvvp
