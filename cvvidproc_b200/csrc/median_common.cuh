// Shared helpers of the median kernels: the rank rule of every background, single-LOP3 bit select and the in-register
// 32x32 bit transpose.
#pragma once
#include <cstdint>

namespace cvvp
{
// Rank of percentile `percent` (integer, 0..100) among n values: the result is sorted[k] with
// k = min(n - 1, floor(n * percent / 100)).  percent = 50 gives n / 2, the reference's upper median
// (histogram_median_algo.h:160-166); 0 the minimum, 100 the maximum.  Every kernel and the host code take the rank
// from here.  n = 0 gives 0 (no value to select).  U is the unsigned type of the arithmetic: the host uses 64 bits;
// the kernels use 32, which is exact while n * 100 < 2^32 (their n is at most 16 x 65535 frames) and keeps the
// per-element cost of the owner kernels at that of the n / 2 it replaced (a multiply-high, not a 64-bit division).
template <typename U>
__host__ __device__ __forceinline__ U percentile_rank(U n, uint32_t percent)
{
    static_assert(U(-1) > U(0), "unsigned arithmetic");
    const U k = n * U(percent) / U(100);
    return k < n ? k : (n ? n - U(1) : U(0));
}

// bitwise select: (a & m) | (b & ~m) as ONE LOP3 (ptxas does not fuse the two-mask C expression)
__device__ __forceinline__ uint32_t bitsel(uint32_t a, uint32_t b, uint32_t m)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(d) : "r"(a), "r"(b), "r"(m));
    return d;
}

// The three bit stages of the 32x32 bit transpose: every block of eight words r[8p .. 8p+7] holds one element's 32
// frame slots as bytes (word j, byte k = one frame slot each); afterwards r[8p + b] is bit plane b of that element,
// bit 8k + j = the slot that was byte k of word j.
__device__ __forceinline__ void transpose_bits(uint32_t (&r)[32])
{
#pragma unroll
    for (int h = 0; h < 32; h += 8) {
#pragma unroll
        for (int i = h; i < h + 4; ++i) {
            const uint32_t a = r[i], b = r[i + 4];
            r[i] = bitsel(a, b << 4, 0x0F0F0F0Fu);
            r[i + 4] = bitsel(a >> 4, b, 0x0F0F0F0Fu);
        }
    }
#pragma unroll
    for (int h = 0; h < 32; h += 4) {
#pragma unroll
        for (int i = h; i < h + 2; ++i) {
            const uint32_t a = r[i], b = r[i + 2];
            r[i] = bitsel(a, b << 2, 0x33333333u);
            r[i + 2] = bitsel(a >> 2, b, 0x33333333u);
        }
    }
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        const uint32_t a = r[i], b = r[i + 1];
        r[i] = bitsel(a, b << 1, 0x55555555u);
        r[i + 1] = bitsel(a >> 1, b, 0x55555555u);
    }
}

// The two byte stages: r[i] = the word of frame slot i (4 elements) -> r[8p + j] = element p, slots j, j+8, j+16, j+24.
__device__ __forceinline__ void transpose_bytes(uint32_t (&r)[32])
{
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint32_t a = r[i], b = r[i + 16];
        r[i] = __byte_perm(a, b, 0x5410);
        r[i + 16] = __byte_perm(a, b, 0x7632);
    }
#pragma unroll
    for (int h = 0; h < 32; h += 16) {
#pragma unroll
        for (int i = h; i < h + 8; ++i) {
            const uint32_t a = r[i], b = r[i + 8];
            r[i] = __byte_perm(a, b, 0x6240);
            r[i + 8] = __byte_perm(a, b, 0x7351);
        }
    }
}

// In-register transpose of a 32x32 bit matrix: afterwards r[j] bit i == (old r[i]) bit j.
__device__ __forceinline__ void transpose32(uint32_t (&r)[32])
{
    transpose_bytes(r);
    transpose_bits(r);
}

// High nibbles only: afterwards r[8p + 4 .. 8p + 7] hold bit planes 4..7 of element p (the other entries are
// scratch).  The byte stages are the same as in transpose32; from the 4-bit stage on only the half of every pair that
// carries the high nibbles is computed (160 instead of 256 instructions).  Used by the counting round that needs the
// high nibble alone (median_pipe_kernel MODE 1).
__device__ __forceinline__ void transpose_bits_hi(uint32_t (&r)[32])
{
#pragma unroll
    for (int h = 0; h < 32; h += 8) {
#pragma unroll
        for (int i = h; i < h + 4; ++i)
            r[i + 4] = bitsel(r[i] >> 4, r[i + 4], 0x0F0F0F0Fu); // high nibbles of the pair
    }
#pragma unroll
    for (int h = 4; h < 32; h += 8) { // the high-nibble half of every block of eight
#pragma unroll
        for (int i = h; i < h + 2; ++i) {
            const uint32_t a = r[i], b = r[i + 2];
            r[i] = bitsel(a, b << 2, 0x33333333u);
            r[i + 2] = bitsel(a >> 2, b, 0x33333333u);
        }
#pragma unroll
        for (int i = h; i < h + 4; i += 2) {
            const uint32_t a = r[i], b = r[i + 1];
            r[i] = bitsel(a, b << 1, 0x55555555u);
            r[i + 1] = bitsel(a >> 1, b, 0x55555555u);
        }
    }
}

__device__ __forceinline__ void transpose32_hi(uint32_t (&r)[32])
{
    transpose_bytes(r);
    transpose_bits_hi(r);
}
} // namespace cvvp
