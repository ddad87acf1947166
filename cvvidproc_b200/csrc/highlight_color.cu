// Difference image of colour frames (cvvp_highlight_set_channels): frames and backgrounds of C interleaved channels
// (2..4) -> one byte per pixel,
//
//   d(x, y) = max over c of hl_diff(bg_c, f_c, polarity)
//
// written as single-channel planes that the grey highlight kernels (highlight_fused.cu, highlight.cu) then read against
// a zero background in the BRIGHT polarity, where their own difference is max(d - 0, 0) = d.  So the bits phase, Otsu's
// histogram, the per-pixel path and the component statistics see exactly this d without a change to them.
//
// One thread makes 16 pixels.  The aligned path loads them with C 128-bit loads of the frame and C of the background,
// takes the per-channel differences four bytes at a time (VSUBUS4 / VABSDIFF4), regroups the interleaved channels per
// pixel with byte permutes and reduces them with VMAX4, and stores one 128-bit word.  Rows whose frame, background or
// output pointer is not 16-byte aligned, and the last pixels of a row, take a byte path.  A "row" is either the whole
// frame (contiguous frames: one row of width*height pixels) or one image row (the crop of a decoded frame).
#include "highlight_state.hpp"

namespace cvvp
{
namespace
{
template <int POL>
__device__ __forceinline__ uint32_t cdiff_u8x4(uint32_t fr, uint32_t bg)
{
    if (POL == CVVP_POLARITY_DARK)
        return __vsubus4(bg, fr);
    if (POL == CVVP_POLARITY_BRIGHT)
        return __vsubus4(fr, bg);
    return __vabsdiffu4(fr, bg);
}

// the largest channel of each of pixels 4J .. 4J + 3, whose C * 4 interleaved bytes are words J*C .. J*C + C - 1 of v
template <int C, int J>
__device__ __forceinline__ uint32_t max_channels_x4(const uint32_t (&v)[4 * C])
{
    const uint32_t *w = v + J * C;
    if (C == 2) { // [p0c0 p0c1 p1c0 p1c1] [p2c0 p2c1 p3c0 p3c1]
        return __vmaxu4(__byte_perm(w[0], w[1], 0x6420), __byte_perm(w[0], w[1], 0x7531));
    } else if (C == 3) { // [p0c0 p0c1 p0c2 p1c0] [p1c1 p1c2 p2c0 p2c1] [p2c2 p3c0 p3c1 p3c2]
        const uint32_t c0 = __byte_perm(__byte_perm(w[0], w[1], 0x0630), w[2], 0x5210);
        const uint32_t c1 = __byte_perm(__byte_perm(w[0], w[1], 0x0741), w[2], 0x6210);
        const uint32_t c2 = __byte_perm(__byte_perm(w[0], w[1], 0x0052), w[2], 0x7410);
        return __vmaxu4(c0, __vmaxu4(c1, c2));
    } else { // C == 4: word k is pixel k; fold channels 2, 3 onto 0, 1, then the pairs
        const uint32_t m01 = __vmaxu4(__byte_perm(w[0], w[1], 0x5140), __byte_perm(w[0], w[1], 0x7362));
        const uint32_t m23 = __vmaxu4(__byte_perm(w[2], w[3], 0x5140), __byte_perm(w[2], w[3], 0x7362));
        // m01 = [max(p0c0,p0c2) max(p1c0,p1c2) max(p0c1,p0c3) max(p1c1,p1c3)], m23 likewise for p2, p3
        return __vmaxu4(__byte_perm(m01, m23, 0x5410), __byte_perm(m01, m23, 0x7632));
    }
}

// pixel p of row r of frame f: frame at src + f * frame_stride + r * row_stride + x0 * C, background at
// bg + f * bg_stride + r * row_len * C, output at dst + f * dst_pitch + r * row_len
template <int C, int POL>
__global__ void __launch_bounds__(128)
    color_diff_kernel(const uint8_t *__restrict__ src, size_t frame_stride, size_t row_stride, int x0,
                      const uint8_t *__restrict__ bg, size_t bg_stride, uint32_t row_len, uint32_t nrows,
                      uint32_t nframes, uint8_t *__restrict__ dst, size_t dst_pitch)
{
    const uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) * 16u;
    if (p >= row_len)
        return;
    for (uint32_t f = blockIdx.z; f < nframes; f += gridDim.z) {
        for (uint32_t r = blockIdx.y; r < nrows; r += gridDim.y) {
            const uint8_t *fr = src + size_t(f) * frame_stride + size_t(r) * row_stride + size_t(x0) * C;
            const uint8_t *bk = bg + size_t(f) * bg_stride + size_t(r) * row_len * C;
            uint8_t *out = dst + size_t(f) * dst_pitch + size_t(r) * row_len;
            const bool aligned = ((reinterpret_cast<uintptr_t>(fr) | reinterpret_cast<uintptr_t>(bk) |
                                   reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
            if (aligned && p + 16 <= row_len) {
                const uint4 *fv = reinterpret_cast<const uint4 *>(fr + size_t(p) * C);
                const uint4 *bv = reinterpret_cast<const uint4 *>(bk + size_t(p) * C);
                uint4 a[C], b[C];
#pragma unroll
                for (int k = 0; k < C; ++k) {
                    a[k] = __ldg(fv + k);
                    b[k] = __ldg(bv + k);
                }
                uint32_t w[4 * C];
#pragma unroll
                for (int k = 0; k < C; ++k) {
                    w[4 * k + 0] = cdiff_u8x4<POL>(a[k].x, b[k].x);
                    w[4 * k + 1] = cdiff_u8x4<POL>(a[k].y, b[k].y);
                    w[4 * k + 2] = cdiff_u8x4<POL>(a[k].z, b[k].z);
                    w[4 * k + 3] = cdiff_u8x4<POL>(a[k].w, b[k].w);
                }
                *reinterpret_cast<uint4 *>(out + p) =
                    make_uint4(max_channels_x4<C, 0>(w), max_channels_x4<C, 1>(w), max_channels_x4<C, 2>(w),
                               max_channels_x4<C, 3>(w));
            } else {
                const uint32_t p1 = min(p + 16u, row_len);
#pragma unroll 1
                for (uint32_t x = p; x < p1; ++x) {
                    int d = 0;
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        d = max(d, hl_diff(__ldg(bk + size_t(x) * C + c), __ldg(fr + size_t(x) * C + c), POL));
                    out[x] = uint8_t(d);
                }
            }
        }
    }
}

template <int C>
void launch_c(int polarity, dim3 grid, cudaStream_t s, const uint8_t *src, size_t frame_stride, size_t row_stride, int x0,
              const uint8_t *bg, size_t bg_stride, uint32_t row_len, uint32_t nrows, uint32_t nframes, uint8_t *dst,
              size_t dst_pitch)
{
    if (polarity == CVVP_POLARITY_DARK)
        color_diff_kernel<C, CVVP_POLARITY_DARK><<<grid, 128, 0, s>>>(src, frame_stride, row_stride, x0, bg, bg_stride,
                                                                       row_len, nrows, nframes, dst, dst_pitch);
    else if (polarity == CVVP_POLARITY_BRIGHT)
        color_diff_kernel<C, CVVP_POLARITY_BRIGHT><<<grid, 128, 0, s>>>(src, frame_stride, row_stride, x0, bg, bg_stride,
                                                                         row_len, nrows, nframes, dst, dst_pitch);
    else
        color_diff_kernel<C, CVVP_POLARITY_BOTH><<<grid, 128, 0, s>>>(src, frame_stride, row_stride, x0, bg, bg_stride,
                                                                       row_len, nrows, nframes, dst, dst_pitch);
}
} // namespace

int color_diff_launch(cvvp_ctx *ctx, int channels, int polarity, const uint8_t *src, long long n, size_t frame_stride,
                      size_t row_stride, int x0, const uint8_t *bg, size_t bg_stride, uint32_t row_len, uint32_t nrows,
                      uint8_t *dst, size_t dst_pitch, cudaStream_t stream)
{
    if (n <= 0)
        return CVVP_OK;
    const uint32_t groups = (row_len + 15u) / 16u;
    const dim3 grid((groups + 127u) / 128u, nrows < 65535u ? nrows : 65535u, n < 65535 ? unsigned(n) : 65535u);
    const uint32_t nf = uint32_t(n);
    switch (channels) {
    case 2: launch_c<2>(polarity, grid, stream, src, frame_stride, row_stride, x0, bg, bg_stride, row_len, nrows, nf, dst, dst_pitch); break;
    case 3: launch_c<3>(polarity, grid, stream, src, frame_stride, row_stride, x0, bg, bg_stride, row_len, nrows, nf, dst, dst_pitch); break;
    case 4: launch_c<4>(polarity, grid, stream, src, frame_stride, row_stride, x0, bg, bg_stride, row_len, nrows, nf, dst, dst_pitch); break;
    default: return fail(ctx, CVVP_ERR_INVALID, "highlight: %d channels", channels);
    }
    ctx->launches += 1;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return fail(ctx, CVVP_ERR_CUDA, "highlight colour difference: launch failed: %s", cudaGetErrorString(e));
    return CVVP_OK;
}
} // namespace cvvp
