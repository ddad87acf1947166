// Rolling temporal median on sm_100a: the background of frame t is the per-element percentile p (the upper median at the
// default p = 50) of a window of W frames centred on t, shifted (not shortened) at both ends of the stream:
//
//   N <= W : every frame's window is all N frames
//   N >  W : s(t) = min(max(t - W/2, 0), N - W), window = frames s(t) .. s(t) + W - 1
//   B_t[e] = min{v : #{window values <= v} > k}  (Weff = min(W, N), k = k(Weff, p) of percentile_rank; k = Weff/2 at
//            p = 50 is the reference's rule, /root/reference/Sources/ProcessorAlgos/histogram_median_algo.h:160-166)
//
// Incremental form.  One CTA owns a tile of kRollE consecutive elements (one thread each) and a chunk of consecutive
// outputs.  Every element keeps a 256-bin histogram of its window on chip with 16-bit counts (W <= 65535, so counts
// never saturate and the result is exact), plus the current median m and lt = #{window values < m}.  The CTA builds
// the histograms once from the W rows of its first window; every later output whose window moves adds the entering
// row and removes the leaving one, updates lt against m and walks m until lt <= k < lt + h[m] holds again (a
// level or two on sensor noise, at most 255 steps on a scene cut).  Outputs whose window does not move (the clamped
// ends) repeat m.
//
// Shared memory: bins are packed two to a 32-bit word, word (b / 2) * kRollE + thread, so the 32 threads of a warp
// always touch 32 different banks whatever values they hold (no conflicts).  128 x 128 x 4 B = 64 KB per CTA: three
// CTAs per SM.  Threads are independent (a thread only ever touches its own column), so there is no barrier.
//
// Bytes: a chunk of C outputs reads (W + 2C) rows of its tile and writes C; chunks are at least W outputs long where
// the output count allows, so reads stay below 3 bytes per output element.  Frames may live in a ring (frame i at
// frames + (i % ring) * stride): the streaming operator of highlight_rolling.cu keeps only W + max_batch frames.
#include "context.hpp"
#include "median_common.cuh"

namespace cvvp
{
namespace
{
constexpr int kRollE = 128;                                        // elements (= threads) per CTA
constexpr int kRollK = 8;                                          // window moves whose loads are issued together
constexpr size_t kRollSmem = size_t(128) * kRollE * sizeof(uint32_t); // 128 bin pairs x kRollE elements

struct RollArgs {
    const uint8_t *frames;
    size_t stride;
    uint32_t ring;      // frames in the ring (frame i lives in slot i % ring)
    long long nframes;  // N: the windows clamp to it
    long long half_w;   // W / 2
    long long weff;     // min(W, N)
    uint32_t rank;      // k(Weff, p): the window's order statistic
    long long t0, t1;   // outputs [t0, t1)
    long long chunk;    // outputs per CTA
    uint8_t *out;       // B_t at out + (t - t0) * out_stride
    size_t out_stride;
    uint32_t nelem;
};

// count of bin b in the thread's packed column
__device__ __forceinline__ uint32_t bin_count(const uint32_t *h, uint32_t b)
{
    return (h[(b >> 1) * kRollE] >> ((b & 1u) * 16u)) & 0xFFFFu;
}

__device__ __forceinline__ void bin_add(uint32_t *h, uint32_t b)
{
    h[(b >> 1) * kRollE] += 1u << ((b & 1u) * 16u);
}

__device__ __forceinline__ void bin_sub(uint32_t *h, uint32_t b)
{
    h[(b >> 1) * kRollE] -= 1u << ((b & 1u) * 16u);
}

__global__ void __launch_bounds__(kRollE) median_roll_kernel(const RollArgs a)
{
    extern __shared__ uint32_t roll_hist[];
    const uint32_t e = blockIdx.x * kRollE + threadIdx.x;
    if (e >= a.nelem)
        return;
    const long long c0 = a.t0 + (long long)blockIdx.y * a.chunk;
    const long long c1 = min(c0 + a.chunk, a.t1);
    if (c0 >= c1)
        return;
    uint32_t *h = roll_hist + threadIdx.x;
#pragma unroll 8
    for (int j = 0; j < 128; ++j)
        h[j * kRollE] = 0;
    const uint8_t *col = a.frames + e;
    // window of the chunk's first output
    const long long s0 = min(max(c0 - a.half_w, 0ll), a.nframes - a.weff);
    uint32_t kl = uint32_t(s0 % a.ring); // slot of the row that leaves at the next move
    uint32_t ke = kl;                    // walks the window's rows; ends on the slot of the row that enters next
    for (long long i = 0; i < a.weff; i += kRollK) {
        uint32_t v[kRollK];
#pragma unroll
        for (int j = 0; j < kRollK; ++j) {
            v[j] = 256u;
            if (i + j < a.weff) {
                v[j] = __ldg(col + size_t(ke) * a.stride);
                ke = ke + 1 == a.ring ? 0u : ke + 1;
            }
        }
#pragma unroll
        for (int j = 0; j < kRollK; ++j)
            if (v[j] < 256u)
                bin_add(h, v[j]);
    }
    const uint32_t rank = a.rank;
    uint32_t m = 0, lt = 0;
    for (uint32_t c = bin_count(h, 0); lt + c <= rank; c = bin_count(h, m)) {
        lt += c;
        ++m;
    }
    uint8_t *dst = a.out + size_t(c0 - a.t0) * a.out_stride + e;
    __stcs(dst, uint8_t(m));
    // the window moves at output t iff 1 <= t - W/2 <= N - Weff
    const long long move_lo = a.half_w + 1, move_hi = a.nframes - a.weff + a.half_w;
    for (long long t = c0 + 1; t < c1; t += kRollK) {
        uint32_t vin[kRollK], vout[kRollK];
        bool mv[kRollK];
#pragma unroll
        for (int j = 0; j < kRollK; ++j) {
            const long long tt = t + j;
            mv[j] = tt < c1 && tt >= move_lo && tt <= move_hi;
            vin[j] = vout[j] = 0;
            if (mv[j]) {
                vin[j] = __ldg(col + size_t(ke) * a.stride);
                vout[j] = __ldg(col + size_t(kl) * a.stride);
                ke = ke + 1 == a.ring ? 0u : ke + 1;
                kl = kl + 1 == a.ring ? 0u : kl + 1;
            }
        }
#pragma unroll
        for (int j = 0; j < kRollK; ++j) {
            if (t + j >= c1)
                break;
            if (mv[j]) {
                bin_add(h, vin[j]);
                bin_sub(h, vout[j]);
                lt = lt + (vin[j] < m) - (vout[j] < m);
                while (lt > rank) {
                    --m;
                    lt -= bin_count(h, m);
                }
                for (uint32_t c = bin_count(h, m); lt + c <= rank; c = bin_count(h, m)) {
                    lt += c;
                    ++m;
                }
            }
            dst += a.out_stride;
            __stcs(dst, uint8_t(m));
        }
    }
}
} // namespace

int median_roll_launch(cvvp_ctx *ctx, const uint8_t *d_frames, long long ring, size_t frame_stride, long long nframes,
                       size_t nelem, int window, int percent, long long t0, long long t1, uint8_t *d_out,
                       size_t out_stride, cudaStream_t stream)
{
    if (window < 1 || window > 65535)
        return fail(ctx, CVVP_ERR_INVALID, "rolling median: window %d outside [1, 65535]", window);
    if (percent < 0 || percent > 100)
        return fail(ctx, CVVP_ERR_INVALID, "rolling median: percentile %d outside [0, 100]", percent);
    if (!d_frames || !d_out || nframes < 1 || nelem == 0 || t0 < 0 || t1 > nframes || t0 > t1)
        return fail(ctx, CVVP_ERR_INVALID, "rolling median: bad arguments (need 0 <= t0 <= t1 <= nframes, nframes >= 1, nelem >= 1)");
    if (frame_stride < nelem || out_stride < nelem)
        return fail(ctx, CVVP_ERR_INVALID, "rolling median: frame_stride %zu and out_stride %zu must be >= nelem %zu", frame_stride,
                    out_stride, nelem);
    if (nelem >= (size_t(1) << 32) || ring < 1 || ring >= (1ll << 32))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "rolling median: frame or ring too large");
    if (t0 == t1)
        return CVVP_OK;
    const long long weff = window < nframes ? window : nframes;
    const long long T = t1 - t0;
    const long long tiles = (long long)((nelem + kRollE - 1) / kRollE);
    // enough CTAs for four waves of three per SM; chunks of at least Weff outputs where the output count allows, so that
    // rebuilding a window costs at most one read per output
    const long long target = 12ll * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    long long nchunks = (target + tiles - 1) / tiles;
    const long long by_window = T / weff > 1 ? T / weff : 1;
    if (nchunks > by_window)
        nchunks = by_window;
    if (nchunks > 65535)
        nchunks = 65535;
    if (nchunks < 1)
        nchunks = 1;
    const long long chunk = (T + nchunks - 1) / nchunks;
    nchunks = (T + chunk - 1) / chunk;
    RollArgs a;
    a.frames = d_frames;
    a.stride = frame_stride;
    a.ring = uint32_t(ring);
    a.nframes = nframes;
    a.half_w = window / 2;
    a.weff = weff;
    a.rank = uint32_t(percentile_rank<uint64_t>(uint64_t(weff), uint32_t(percent)));
    a.t0 = t0;
    a.t1 = t1;
    a.chunk = chunk;
    a.out = d_out;
    a.out_stride = out_stride;
    a.nelem = uint32_t(nelem);
    CVVP_CUDA_OK(ctx, cudaFuncSetAttribute(median_roll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kRollSmem)));
    median_roll_kernel<<<dim3(unsigned(tiles), unsigned(nchunks)), kRollE, kRollSmem, stream>>>(a);
    CVVP_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches++;
    return CVVP_OK;
}
} // namespace cvvp
