// Temporal-median kernel: on-chip bit-sliced radix select with warp-specialised streaming.
// (Algorithm and reference citations: see median.cu.)
//
//   SELECT warps     (8 or 16)  tile t      : 8 MSB-first passes of popc over bit planes held in shared memory
//   TRANSPOSE warps  (12)       tile t+1    : wait for a 4 KB TMA stage, turn it into bit planes (128-byte tiles: eight
//                                             transposing matrix loads, LDSM.8.MT1616, do the byte stages of the 32x32
//                                             bit transpose in the load path and three shift/LOP3 stages remain;
//                                             narrower tiles: plain loads, two PRMT stages more), store the planes, and
//                                             immediately RE-ISSUE the TMA load of their own next stage into the slot
//                                             they just drained
//
// There is no producer warp: a single thread issuing every TMA box costs ~290 cycles per stage (dependent
// try_wait -> expect_tx -> issue chain) and caps the whole chip near 4 TB/s.  With 12 self-service warps the issue
// work is spread out and the ring needs no "empty" barriers at all: each transposer warp owns two PRIVATE slots
// (stage g of the CTA's global stage sequence goes to warp g % 12, slot g % 24), refills a slot only after its own
// lanes have read it, and therefore always waits for the direct successor of a fill it consumed itself -- the
// condition under which an mbarrier parity wait cannot alias (TMA completions are unordered across slots).
//
// Two buffering modes, chosen by the stage count per tile (nst):
//   nst <= 16 : two plane buffers, 8 select warps  (stages split by parity, JT = ceil(nst/2) <= 8 per thread)
//   nst <= 32 : one plane buffer, 16 select warps  (stages split mod 4,      JT = ceil(nst/4) <= 8 per thread).
//               MODE 0 treats the buffer as a pool of half-stage slots (the four planes of one nibble of one stage):
//               the high-nibble slots of a tile are handed back as soon as those planes are in the selectors'
//               registers, the low-nibble slots four passes later, and the next tile's first / second half of stages
//               goes into them (see "half-slot pool" in the kernel); the 24 ring slots keep HBM streaming meanwhile.
//
// Plane layout per buffer (half-slot pool: per 2 KB slot [byte p][column phi][4 words]):
// [stage][byte p][nibble bh][column phi][4 words = bits 4bh..4bh+3]: a transposer lane
// stores uint4, a select thread loads the four planes of a nibble with one LDS.128.  phi = lane ^ (stage % G)
// (G = 2 or 4 stage classes); the select thread for logical lane L and stage class g reads column L ^ g, which is
// its own lane id ^ (low column bits held in its warp id).  Both patterns touch 8 distinct 16-byte columns per
// quarter-warp: bank-conflict free.
//
// MODE 3 (window counting, see below) hands the single plane buffer back ROW BY ROW: a selector warp bumps the
// monotonic counter rows_free[j] as soon as its lanes hold row j (stages G*j .. G*j + G-1) in registers, and the
// transposer of stage st of the next tile only waits for rows_free[st / G] -- the next tile's transposition runs right
// behind the selectors instead of after them, and monotonic counters cannot alias the way a parity wait can.
//
// Selectors walk through every tile in order, so their planes_full waits are one phase away by induction.  A
// transposer can reach a buffer two fills ahead when tiles are tiny, so before its planes_empty parity wait it
// checks a monotonic shared counter of completed selects; after that the parity wait is at most one phase away.
#include "context.hpp"

#include <cstdlib>

#include "median_common.cuh"
#include "ptx_helpers.cuh"

namespace cvvp
{
namespace
{
constexpr int kTrWarps = 12;
constexpr int kStageBytes = 4096;
constexpr int kStageWords = kStageBytes / 4;
constexpr int kRing = 2 * kTrWarps; // two private slots per transposer warp

// minterm c of three plane words (a = bit 2 of c, b = bit 1, d = bit 0): one LOP3 with the immediate 1 << c
template <int C>
__device__ __forceinline__ uint32_t minterm3(uint32_t a, uint32_t b, uint32_t d)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(d), "n"(1 << C));
    return r;
}

// Counts of the 16 values of one nibble over the 32 frame slots of a plane word, restricted to `mask`:
// acc[c] += count(nibble == 2c) | count(nibble == 2c + 1) << 16.   p3..p0 = the nibble's bit planes, MSB first.
__device__ __forceinline__ void nibble_counts(uint32_t (&acc)[8], uint32_t p3, uint32_t p2, uint32_t p1, uint32_t p0,
                                              uint32_t mask)
{
    const uint32_t m0 = mask & ~p0, m1 = mask & p0;
#define CVVP_MT(C)                                                                                                     \
    {                                                                                                                  \
        const uint32_t t = minterm3<C>(p3, p2, p1);                                                                    \
        acc[C] += __popc(t & m0) + (__popc(t & m1) << 16);                                                             \
    }
    CVVP_MT(0) CVVP_MT(1) CVVP_MT(2) CVVP_MT(3) CVVP_MT(4) CVVP_MT(5) CVVP_MT(6) CVVP_MT(7)
#undef CVVP_MT
}

template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return r;
}

__device__ __forceinline__ uint32_t ld_acquire_shared(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}

__device__ __forceinline__ void red_release_shared_inc(uint32_t *p)
{
    asm volatile("red.release.cta.shared.add.u32 [%0], 1;" ::"r"(smem_u32(p)) : "memory");
}

// A select warp hands plane slots back as soon as it has LOADED them, a transposer warp refills its ring slot as soon
// as it has read it.  The hand-backs are release operations behind a warp barrier, which by the memory model already
// orders the warp's loads before them; the TMA refill, however, is an asynchronous-proxy write issued by one lane
// after generic-proxy reads of all lanes, with only the warp barrier in between.  As a hardening that costs nothing
// measurable (1080p x 1000 frames: 0.363 ms with and without), every hand-back also carries a DATA dependency on the
// loads: `fold` is the XOR of one word of every load, ANDed with a zero the compiler cannot see; the instruction cannot
// issue before the registers are written, and its result (0) is added to the signalled address / the refill's
// destination.  (History: wrong medians once seen at 769 .. 896 frames came from a probe that launched this kernel on
// the library's stream while torch was still generating the input on another; the kernel before this change passes
// tests/test_median_gpu.py::test_every_cta_walks_several_tiles_of_the_single_buffer_mode and tools/stress_median.py
// as well.)
__device__ __forceinline__ uint32_t landed(uint32_t fold, uint32_t opaque_zero)
{
    uint32_t z;
    asm volatile("and.b32 %0, %1, %2;" : "=r"(z) : "r"(fold), "r"(opaque_zero));
    return z;
}

// Every lane of the warp polls a monotonic shared-memory counter until it reaches `need` (acquire).  The loop is
// load + compare + sleep: a polling warp shares its scheduler with working warps, and with one polling lane, a warp
// barrier behind it and the watchdog's timer read in every iteration the pollers issued a tenth of the window
// kernel's instructions.  The watchdog (2 s, trap instead of a hung GPU) looks at the timer once per 4096 polls.
__device__ __forceinline__ void wait_counter(const uint32_t *cnt, uint32_t need)
{
    if (ld_acquire_shared(cnt) >= need)
        return;
    const uint64_t t0 = global_timer_ns();
    for (;;) {
#pragma unroll 1
        for (uint32_t spins = 0; spins < 4096u; ++spins) {
            __nanosleep(32);
            if (ld_acquire_shared(cnt) >= need)
                return;
        }
        if (global_timer_ns() - t0 > 2000000000ull)
            __trap();
    }
}

// One transposing matrix load: two 16 x 16 BYTE tiles (lanes 0..15 / 16..31 name the 16-byte rows of the first / second
// tile) arrive transposed -- lane T holds, of each tile, column T / 4 and column T / 4 + 8, rows 4 (T % 4) .. + 3 packed
// into one register each (layout measured with tools/ldsm_probe.cu).  SASS: LDSM.8.MT1616.
__device__ __forceinline__ void ldsm_t_b8_x2(uint32_t &a0, uint32_t &a1, uint32_t &b0, uint32_t &b1, uint32_t addr)
{
    asm volatile("ldmatrix.sync.aligned.m16n16.x2.trans.shared.b8 {%0, %1, %2, %3}, [%4];"
                 : "=r"(a0), "=r"(a1), "=r"(b0), "=r"(b1)
                 : "r"(addr)
                 : "memory");
}

// Window counting (MODE 3) of one plane row: lo / hi = bit planes 0..3 / 4..7 of one element over 32 frame slots,
// fb[b] = bit b of the window base replicated over the word.  d = v - base is formed bit-sliced (one LOP3 for the
// difference bit, one for the borrow); the final borrow marks the slots below the window (v < base), the OR of
// difference bits 3..7 the slots above it.  acc[c] += count(d == 2c) | count(d == 2c + 1) << 16, below += count(v < base).
// vm masks rows beyond the tile's stage count (they hold garbage).
__device__ __forceinline__ void window_row(uint32_t (&acc)[4], uint32_t &below, const uint4 &lo, const uint4 &hi,
                                           const uint32_t (&fb)[8], uint32_t vm)
{
    const uint32_t a[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    uint32_t d[8];
    uint32_t bw = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        d[b] = lop3<0x96>(a[b], fb[b], bw); // a ^ f ^ borrow
        bw = lop3<0x8E>(a[b], fb[b], bw);   // majority(~a, f, borrow)
    }
    const uint32_t above = lop3<0xFE>(lop3<0xFE>(d[3], d[4], d[5]), d[6], d[7]);
    const uint32_t in = lop3<0x01>(above, bw, ~vm); // ~(above | below | invalid)
    below += __popc(bw & vm);
    const uint32_t m0 = in & ~d[2], m1 = in & d[2];
    acc[0] += __popc(lop3<0x10>(m0, d[1], d[0])) + (__popc(lop3<0x20>(m0, d[1], d[0])) << 16);
    acc[1] += __popc(lop3<0x40>(m0, d[1], d[0])) + (__popc(lop3<0x80>(m0, d[1], d[0])) << 16);
    acc[2] += __popc(lop3<0x10>(m1, d[1], d[0])) + (__popc(lop3<0x20>(m1, d[1], d[0])) << 16);
    acc[3] += __popc(lop3<0x40>(m1, d[1], d[0])) + (__popc(lop3<0x80>(m1, d[1], d[0])) << 16);
}

// LOG2S : log2(32-frame sub-blocks per stage per element); P = 128 >> LOG2S elements per tile
// JT    : stages per select thread (compile time)
// NSELW : select warps, 8 (two stage classes, two plane buffers) or 16 (four stage classes, one plane buffer)
// MODE  : 0 = select the percentile on chip (single-GPU job): rank percentile_rank(nframes, percent), the upper
//             median at percent = 50
//         1 = frame-sharded job, round 1: 16-bin counts of the HIGH nibble of this rank's frames, pushed to the
//             element's owner rank through peer memory
//         2 = round 2: 16-bin counts of the LOW nibble among the frames whose high nibble equals the globally selected
//             one (push.sel[e] & 15), pushed the same way
//         3 = frame-sharded job / long stack in ONE pass over the frames: every element's select threads first pick a
//             PILOT (the same percentile of two of their plane rows: 256 of the launch's <= 1024 frames) on chip, then
//             count all frames in the 8-value window [pilot - 4, pilot + 3] (8 bins) and below it, and push
//             {8 x u16 bins, below | window base << 16} (20 B) to the element's owner (the launch's frame count goes to
//             a header word per owner).  The owner can name the median of
//             ALL sources exactly whenever it lies inside every source's window (shard_window_final_kernel); elements
//             where it does not are flagged and the job falls back to rounds 1 + 2.  (NSELW = 16 only.)
template <int LOG2S, int JT, int NSELW, int MODE>
__global__ void __launch_bounds__((NSELW + kTrWarps) * 32, 1)
    median_pipe_kernel(const __grid_constant__ CUtensorMap tmap, uint8_t *__restrict__ out, const uint32_t nelem,
                       const uint32_t nframes, const uint32_t nst, const uint32_t ntiles, const uint64_t l2_policy,
                       const uint32_t percent, const __grid_constant__ ShardPush push)
{
    constexpr int S = 1 << LOG2S;
    constexpr int P = 128 >> LOG2S;
    constexpr int kSlotsPerStage = 32 * S;
    constexpr int kColBits = 5 - LOG2S;            // word-column bits of a transposer lane id (the rest: sub-block)
    constexpr uint32_t G = NSELW / 4;              // stage classes (st % G) = select threads per (element, sub-block)
    constexpr uint32_t NBUF = (NSELW == 8) ? 2 : 1;
    constexpr uint32_t kBufWords = G * JT * 1024u; // one plane buffer: G*JT stages x 4 KB
    // P == 128: the stage lies in shared memory with TMA's 128-byte swizzle and is read with transposing matrix loads
    // (the byte stages of the transpose happen in the load path instead of 64 PRMTs per lane and stage)
    constexpr bool kLdsm = (LOG2S == 0);
    // MODE 0 with the single plane buffer: the buffer is a pool of 64 half-stage slots (2 KB = the four planes of one
    // nibble of one stage) handed back in two steps, see "half-slot pool" below
    constexpr bool kHalf = (MODE == 0 && NSELW == 16);
    constexpr uint32_t kCap = G * JT;      // stages the plane buffer holds = half-slots per nibble
    constexpr uint32_t kFirst = kCap / 2u; // stages [0, kFirst) of a tile go into the slots that are released first
    static_assert(G == 2 || G == 4, "8 or 16 select warps");
    static_assert((1 << kColBits) >= int(G), "stage classes are encoded in the low column bits");

    extern __shared__ __align__(1024) uint8_t smem[];
    uint32_t *ring = reinterpret_cast<uint32_t *>(smem);                         // kRing x 4 KB
    uint32_t *planes = reinterpret_cast<uint32_t *>(smem + kRing * kStageBytes); // NBUF buffers
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kRing * kStageBytes + NBUF * kBufWords * 4u);
    uint64_t *ring_full = bars;                // [kRing]
    uint64_t *planes_full = bars + kRing;      // [2]
    uint64_t *planes_empty = bars + kRing + 2; // [2]
    volatile uint32_t *sel_done = reinterpret_cast<volatile uint32_t *>(bars + kRing + 4); // [2] selects completed
    uint32_t *rows_free = reinterpret_cast<uint32_t *>(bars + kRing + 4) + 4; // [8] MODE 3: select warps done with row j
    uint32_t *rec_stage = rows_free + 12; // MODE 3, staged push: a tile's 128 records of 5 words (16-byte aligned)

    const uint32_t tid = threadIdx.x;
    const uint32_t warp = tid >> 5;
    const uint32_t lane = tid & 31;

    // tiles of this launch: all of them, or the listed ones (nothing listed: nothing to do, not even barrier set-up)
    const uint32_t *tile_list = MODE != 0 ? push.tile_list : nullptr;
    const uint32_t ntl = tile_list ? min(__ldcg(push.tile_count), ntiles) : ntiles;
    if (ntl == 0u)
        return;
    if (MODE == 3 && blockIdx.x == 0 && tid == 0)
        for (uint32_t r = 0; r < push.nranks; ++r)
            *push.hdr[r] = nframes; // how many frames this source's records count

    if (tid == 0) {
        prefetch_tmap(&tmap);
        for (int i = 0; i < kRing; ++i)
            mbar_init(&ring_full[i], 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&planes_full[i], nst); // one arrival per transposed stage
            mbar_init(&planes_empty[i], NSELW);
            sel_done[i] = 0;
        }
        for (int i = 0; i < 8; ++i)
            rows_free[i] = 0;
        fence_mbar_init();
    }
    __syncthreads();

    // tiles of this CTA, in the order every role walks them: every gridDim.x-th of all tiles, or of the listed ones
    const uint32_t my_tiles = blockIdx.x < ntl ? (ntl - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto tile_at = [&](uint32_t t) {
        const uint32_t idx = blockIdx.x + t * gridDim.x;
        return tile_list ? __ldcg(tile_list + idx) : idx;
    };

    if (warp >= NSELW) {
        // ===================== transposers (self-service TMA) =====================
        const uint32_t w = warp - NSELW;
        const uint32_t total_stages = my_tiles * nst; // global stage sequence of this CTA
        // issue the TMA load of the stage at (tile iteration t, stage s) into this warp's slot for its k-th stage
        // (z: 0, see landed() -- a refill must not be issued before the slot's previous content has been read)
        auto issue = [&](uint32_t k, uint32_t t, uint32_t s, uint32_t z) {
            const uint32_t slot = w + kTrWarps * (k & 1u);
            const uint32_t tile = tile_at(t);
            mbar_arrive_expect_tx(&ring_full[slot], kStageBytes);
            tma_load_2d(ring + size_t(slot) * kStageWords + z, &tmap, &ring_full[slot], int32_t(tile * P),
                        int32_t(s * kSlotsPerStage), l2_policy);
        };
        auto advance = [&](uint32_t &t, uint32_t &s) { // next stage of this warp: global stage number += 12
            s += kTrWarps;
            while (s >= nst) {
                s -= nst;
                ++t;
            }
        };
        // position of this warp's k-th stage: gs = w + 12k -> (ti, st) = (gs / nst, gs % nst), kept incrementally
        uint32_t ti = 0, st = w;
        while (st >= nst) {
            st -= nst;
            ++ti;
        }
        uint32_t ti2 = ti, st2 = st; // look-ahead cursor: the stage that is (re)issued next
        if (lane == 0 && w < total_stages)
            issue(0, ti2, st2, 0u);
        advance(ti2, st2);
        if (lane == 0 && w + kTrWarps < total_stages)
            issue(1, ti2, st2, 0u);
        advance(ti2, st2);

        // byte offsets of this lane's tile row in a swizzled stage, for even and odd loads (see below)
        uint32_t ldsm_off[2];
        {
            const uint32_t m = (lane >> 2) & 3u, i = lane & 3u, pass = lane >> 4;
            for (uint32_t odd = 0; odd < 2; ++odd) {
                const uint32_t f = 4u * ((odd + m) & 1u) + i; // frame slot within the group of eight
                ldsm_off[odd] = f * 128u + (((4u * pass + m) ^ f) << 4);
            }
        }
        uint32_t k = 0;
        for (uint32_t gs = w; gs < total_stages; gs += kTrWarps, ++k) {
            const uint32_t buf = (NBUF == 2) ? (ti & 1u) : 0u;
            const uint32_t q = (NBUF == 2) ? (ti >> 1) : ti; // fill number of this buffer
            const uint32_t slot = w + kTrWarps * (k & 1u);
            mbar_wait(&ring_full[slot], (k >> 1) & 1u);
            uint32_t r[32];
            if constexpr (kLdsm) {
                // load k: tile A = 16-byte chunks 0..3 of the 128-byte frame rows, tile B = chunks 4..7; tile row
                // 4m + i = chunk m of frame slot 8 (k / 2) + 4 ((k + m) & 1) + i.  Lane T (m = T % 4) receives 4 slots
                // of elements 16 (4 pass + m) + T / 4 (+ 8) per load and all 32 slots after the eight loads.  The
                // slot permutation makes rows 0..7 of a tile hit eight different swizzled chunks: no bank conflicts
                // (plain rows: 4-way, measured 3.5x slower).
                const uint32_t sb = smem_u32(ring + size_t(slot) * kStageWords);
#pragma unroll
                for (int kk = 0; kk < 8; ++kk)
                    ldsm_t_b8_x2(r[kk], r[8 + kk], r[16 + kk], r[24 + kk], sb + ldsm_off[kk & 1] + (kk >> 1) * 1024);
            } else {
                const uint32_t *src = ring + size_t(slot) * kStageWords + lane;
#pragma unroll
                for (int i = 0; i < 32; ++i)
                    r[i] = src[i * 32];
            }
            // Every lane has read the slot.  The refill is an asynchronous-proxy write issued by lane 0; its destination
            // carries a data dependency on the loaded words (landed()) so that it cannot be issued before the loads of
            // the whole warp have completed (a warp's load instruction completes for all lanes at once).
            uint32_t fold = 0;
#pragma unroll
            for (int i = 0; i < (kLdsm ? 8 : 32); ++i)
                fold ^= r[i];
            const uint32_t z = landed(fold, nst >> 8);
            __syncwarp(); // refill the slot with this warp's stage k+2
            if (lane == 0 && gs + 2 * kTrWarps < total_stages)
                issue(k, ti2, st2, z);
            advance(ti2, st2);
            if constexpr (kLdsm) {
                if (MODE == 1)
                    transpose_bits_hi(r); // the high-nibble round needs planes 4..7 only
                else
                    transpose_bits(r);
            } else {
                if (MODE == 1)
                    transpose32_hi(r);
                else
                    transpose32(r);
            }
            // r[8*p + b] = bit plane b of this lane's p-th element (elem_of(lane, p)) over its 32 frame slots.
            // Selectors must be done with the previous fill of this buffer.  Pre-check (almost always already
            // true): the fill before that one is finished, which makes the parity wait at most one phase away.
            if constexpr (kHalf) {
                // Half-slot pool.  The selectors of a tile hand back its 32 high-nibble slots as soon as those planes
                // are in their registers (right after planes_full) and the 32 low-nibble slots four passes later.
                // The first half of the NEXT tile's stages (both nibbles) goes into the former, the second half into
                // the latter, so (at 32 stages) 16 stages are stored and 12 more wait transposed in registers while
                // the selectors still work on the current tile.  With C = kCap slots per nibble and F = C / 2 the slot
                // sets repeat with period two:
                //   even tiles: high(s) = s, low(s) = C + s;   odd tiles: s < F: high = s, low = F + s;
                //                                                           s >= F: high = F + s, low = C + s.
                // rows_free[0] / [1] count the select warps that released the high / low slots (monotonic).
                if (ti >= 1u)
                    wait_counter(rows_free + (st < kFirst ? 0 : 1), NSELW * ti);
                const uint32_t odd = ti & 1u;
                const uint32_t hi_slot = st + ((odd && st >= kFirst) ? kFirst : 0u);
                const uint32_t lo_slot = st + ((odd && st < kFirst) ? kFirst : kCap);
                const uint32_t col = lane ^ (st & (G - 1u));
                uint4 *hi = reinterpret_cast<uint4 *>(planes) + hi_slot * 128u + col;
                uint4 *lo = reinterpret_cast<uint4 *>(planes) + lo_slot * 128u + col;
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    lo[p * 32] = make_uint4(r[8 * p + 0], r[8 * p + 1], r[8 * p + 2], r[8 * p + 3]);
                    hi[p * 32] = make_uint4(r[8 * p + 4], r[8 * p + 5], r[8 * p + 6], r[8 * p + 7]);
                }
            } else {
            if constexpr (MODE == 3) {
                // every select warp holds row st / G of the previous tile in registers (monotonic counter: no parity)
                if (q >= 1u)
                    wait_counter(rows_free + st / G, NSELW * q);
            } else {
                if (q >= 2u) {
                    while (sel_done[buf] < NSELW * (q - 1u))
                        __nanosleep(64);
                }
                mbar_wait(&planes_empty[buf], (q & 1u) ^ 1u);
            }
            const uint32_t col = lane ^ (st & (G - 1u));
            uint4 *dst = reinterpret_cast<uint4 *>(planes + buf * kBufWords + st * 1024u) + col;
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                if (MODE != 1)
                    dst[(p * 2 + 0) * 32] = make_uint4(r[8 * p + 0], r[8 * p + 1], r[8 * p + 2], r[8 * p + 3]);
                dst[(p * 2 + 1) * 32] = make_uint4(r[8 * p + 4], r[8 * p + 5], r[8 * p + 6], r[8 * p + 7]);
            }
            } // !kHalf
            __syncwarp();
            if (lane == 0)
                mbar_arrive(&planes_full[buf]);
            advance(ti, st);
        }
        return;
    }

    // ===================== selectors =====================
    // warp = (byte p of the word, cx = low column bits); lane = logical transposer lane id with its low log2(G)
    // bits replaced by the stage class g; this thread owns stages st = G*j + g of element 4c + p, sub-block s
    const uint32_t s_p = warp / G;
    const uint32_t s_cx = warp % G;
    const uint32_t s_g = lane & (G - 1u);
    const uint32_t s_col = lane ^ s_cx;
    const uint32_t s_L = (lane & ~(G - 1u)) | s_cx;
    const uint32_t s_c = s_L & ((32u >> LOG2S) - 1u);
    // element of (transposer lane c, register block p): byte p of word c, or what the matrix loads deliver
    const uint32_t s_elem = kLdsm ? 64u * (s_p >> 1) + 16u * (s_c & 3u) + 8u * (s_p & 1u) + (s_c >> 2) : 4u * s_c + s_p;
    const bool s_writer = (s_g == 0u) && ((lane >> kColBits) == 0u);
    // wanted rank incl. zero pad slots
    const uint32_t k0 = percentile_rank(nframes, percent) + (nst * kSlotsPerStage - nframes);
    const uint32_t zero = nst >> 8; // 0 (nst <= 32), but not to the compiler: see landed()

    for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t tile = tile_at(it);
        const uint32_t buf = (NBUF == 2) ? (it & 1u) : 0u;
        const uint32_t q = (NBUF == 2) ? (it >> 1) : it;
        mbar_wait(&planes_full[buf], q & 1u);
        const uint4 *base = reinterpret_cast<const uint4 *>(planes + buf * kBufWords + s_g * 1024u) + s_p * 64u + s_col;
        if constexpr (MODE == 3) {
            // ---- window counting: pilot median of two plane rows, then 8 bins around it over all rows ----
            static_assert(MODE != 3 || NSELW == 16, "window counting uses the single plane buffer");
            constexpr int JP = JT >= 2 ? 2 : 1; // pilot rows: 0 and JT / 2
            auto pilot_row = [](int i) { return i == 0 ? 0 : JT / 2; };
            const size_t e = size_t(tile) * P + s_elem;
            uint4 plo[JP], phi[JP];
#pragma unroll
            for (int i = 0; i < JP; ++i) {
                plo[i] = base[pilot_row(i) * (G * 256)];
                phi[i] = base[pilot_row(i) * (G * 256) + 32];
            }
            {
                uint32_t fold = 0;
#pragma unroll
                for (int i = 0; i < JP; ++i)
                    fold ^= plo[i].x ^ phi[i].x;
                const uint32_t z = landed(fold, zero);
                __syncwarp();
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < JP; ++i)
                        red_release_shared_inc(rows_free + pilot_row(i) + z);
                }
            }
            // pilot rank: the pilot stages are G*j .. G*j + G-1 of the pilot rows; their real frames and pad slots
            uint32_t p_real = 0, p_slots = 0;
#pragma unroll
            for (int i = 0; i < JP; ++i) {
#pragma unroll
                for (uint32_t g = 0; g < G; ++g) {
                    const uint32_t stg = G * pilot_row(i) + g;
                    if (stg < nst) {
                        const uint32_t f0 = stg * kSlotsPerStage;
                        p_slots += kSlotsPerStage;
                        p_real += nframes > f0 ? min(nframes - f0, uint32_t(kSlotsPerStage)) : 0u;
                    }
                }
            }
            uint32_t med = 0;
            {
                uint32_t alive[JP];
#pragma unroll
                for (int i = 0; i < JP; ++i)
                    alive[i] = (G * pilot_row(i) + s_g) < nst ? 0xFFFFFFFFu : 0u;
                uint32_t k = percentile_rank(p_real, percent) + (p_slots - p_real);
#pragma unroll
                for (int bit = 7; bit >= 0; --bit) {
                    uint32_t cnt = 0;
#pragma unroll
                    for (int i = 0; i < JP; ++i) {
                        const uint4 &q4 = bit >= 4 ? phi[i] : plo[i];
                        const uint32_t wv = (bit & 3) == 0 ? q4.x : (bit & 3) == 1 ? q4.y : (bit & 3) == 2 ? q4.z : q4.w;
                        cnt += __popc(alive[i] & ~wv);
                    }
                    cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 1);
                    cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 2);
                    if (LOG2S >= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 16);
                    if (LOG2S >= 2) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 8);
                    if (LOG2S >= 3) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 4);
                    const bool one = k >= cnt;
                    if (one) {
                        k -= cnt;
                        med |= 1u << bit;
                    }
                    const uint32_t flip = one ? 0u : 0xFFFFFFFFu;
#pragma unroll
                    for (int i = 0; i < JP; ++i) {
                        const uint4 &q4 = bit >= 4 ? phi[i] : plo[i];
                        const uint32_t wv = (bit & 3) == 0 ? q4.x : (bit & 3) == 1 ? q4.y : (bit & 3) == 2 ? q4.z : q4.w;
                        alive[i] &= (wv ^ flip);
                    }
                }
            }
            const uint32_t wbase = med >= 4u ? min(med - 4u, 248u) : 0u; // window = [wbase, wbase + 7]
            uint32_t fb[8];
#pragma unroll
            for (int b = 0; b < 8; ++b)
                fb[b] = 0u - ((wbase >> b) & 1u);
            uint32_t acc[4] = {0, 0, 0, 0};
            uint32_t below = 0;
            // the pilot rows are already in registers
#pragma unroll
            for (int i = 0; i < JP; ++i)
                window_row(acc, below, plo[i], phi[i], fb, (G * pilot_row(i) + s_g) < nst ? 0xFFFFFFFFu : 0u);
            // the other rows: load (one row ahead), hand the row back, count
            constexpr int NR = JT - JP; // rows left
            if constexpr (NR > 0) {
                auto row_of = [](int r) { return r + 1 + (r + 1 >= JT / 2 ? 1 : 0); }; // skips 0 and JT / 2
                uint4 nlo = base[row_of(0) * (G * 256)], nhi = base[row_of(0) * (G * 256) + 32];
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    const int j = row_of(r);
                    const uint4 clo = nlo, chi = nhi;
                    if (r + 1 < NR) {
                        nlo = base[row_of(r + 1) * (G * 256)];
                        nhi = base[row_of(r + 1) * (G * 256) + 32];
                    }
                    const uint32_t z = landed(clo.x ^ chi.x, zero);
                    __syncwarp();
                    if (lane == 0)
                        red_release_shared_inc(rows_free + j + z); // row j was loaded one iteration ago
                    window_row(acc, below, clo, chi, fb, (G * uint32_t(j) + s_g) < nst ? 0xFFFFFFFFu : 0u);
                }
            }
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                uint32_t v = c < 4 ? acc[c] : below;
                v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
                v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
                if (LOG2S >= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, 16);
                if (LOG2S >= 2) v += __shfl_xor_sync(0xFFFFFFFFu, v, 8);
                if (LOG2S >= 3) v += __shfl_xor_sync(0xFFFFFFFFu, v, 4);
                if (c < 4)
                    acc[c] = v;
                else
                    below = v;
            }
            // the zero-filled pad slots were counted as value 0: in bin 0 when the window starts at 0, else below it
            const uint32_t pad = nst * kSlotsPerStage - nframes;
            if (wbase == 0u)
                acc[0] -= pad;
            else
                below -= pad;
            // record of the element: words 0..3 = bins, word 4 = below | window base << 16 (below <= 1024 frames)
            const uint32_t tail = below | (wbase << 16);
            if (push.stage) {
                // Staged push: the tile's 128 records (2560 contiguous bytes in ONE owner's buffer: tiles do not
                // straddle owners) are assembled in shared memory and written 16 bytes per thread.  Storing them
                // straight from the select threads makes every store instruction write scattered 8-byte pieces --
                // poor packets for NVLink once most owners are peers (7 of 8 ranks: 0.65 instead of 0.55 ms).
                if ((lane >> kColBits) == 0u) {
                    if (s_g == 0) {
                        rec_stage[s_elem * 5u + 0u] = acc[0];
                        rec_stage[s_elem * 5u + 1u] = acc[1];
                    } else if (s_g == 1) {
                        rec_stage[s_elem * 5u + 2u] = acc[2];
                        rec_stage[s_elem * 5u + 3u] = acc[3];
                    } else if (s_g == 2) {
                        rec_stage[s_elem * 5u + 4u] = tail;
                    }
                }
                named_bar_sync(1, NSELW * 32);
                const size_t e0 = size_t(tile) * P;
                const uint32_t owner = uint32_t(e0) / push.slice;
                uint32_t *dst = push.dst[owner] + (e0 - size_t(owner) * push.slice) * 5u;
                const uint32_t words = uint32_t(min(size_t(P), size_t(nelem) - e0)) * 5u;
                if (tid < (P * 5u + 3u) / 4u) {
                    if (4u * tid + 4u <= words) {
                        reinterpret_cast<uint4 *>(dst)[tid] = reinterpret_cast<const uint4 *>(rec_stage)[tid];
                    } else {
                        for (uint32_t w = 4u * tid; w < words; ++w)
                            dst[w] = rec_stage[w];
                    }
                }
                named_bar_sync(1, NSELW * 32); // the staging area is rewritten for the next tile
            } else if ((lane >> kColBits) == 0u && e < nelem) {
                const uint32_t owner = uint32_t(e) / push.slice;
                uint32_t *dst = push.dst[owner] + (size_t(e) - size_t(owner) * push.slice) * 5u;
                if (s_g == 0) {
                    dst[0] = acc[0];
                    dst[1] = acc[1];
                } else if (s_g == 1) {
                    dst[2] = acc[2];
                    dst[3] = acc[3];
                } else if (s_g == 2) {
                    dst[4] = tail;
                }
            }
        } else if constexpr (MODE != 0) {
            // ---- frame-sharded job: nibble counts of this rank's frames, pushed to the owner of the element ----
            const size_t e = size_t(tile) * P + s_elem;
            uint32_t acc[8];
#pragma unroll
            for (int c = 0; c < 8; ++c)
                acc[c] = 0;
            uint32_t h = 0;
            if (MODE == 1) {
                uint4 w4[JT];
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    w4[j] = base[j * (G * 256) + 32]; // high-nibble planes
                uint32_t fold = 0;
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    fold ^= w4[j].x;
                const uint32_t z = landed(fold, zero);
                __syncwarp();
                if (lane == 0) {
                    atomicAdd(const_cast<uint32_t *>(sel_done) + buf + z, 1u);
                    mbar_arrive(&planes_empty[buf + z]);
                }
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    if ((G * j + s_g) < nst) // rows >= nst hold garbage
                        nibble_counts(acc, w4[j].w, w4[j].z, w4[j].y, w4[j].x, 0xFFFFFFFFu);
            } else {
                h = e < nelem ? (__ldcg(push.sel + e) & 15u) : 0u;
                const uint32_t f4 = (h & 1u) ? 0u : 0xFFFFFFFFu, f5 = (h & 2u) ? 0u : 0xFFFFFFFFu;
                const uint32_t f6 = (h & 4u) ? 0u : 0xFFFFFFFFu, f7 = (h & 8u) ? 0u : 0xFFFFFFFFu;
                uint32_t eq[JT];
#pragma unroll
                for (int j = 0; j < JT; ++j) {
                    const uint4 w = base[j * (G * 256) + 32];
                    const uint32_t m = (w.x ^ f4) & (w.y ^ f5) & (w.z ^ f6) & (w.w ^ f7); // high nibble == h
                    eq[j] = (G * j + s_g) < nst ? m : 0u;
                }
                uint4 w4[JT];
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    w4[j] = base[j * (G * 256)]; // low-nibble planes
                uint32_t fold = 0;
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    fold ^= w4[j].x ^ eq[j];
                const uint32_t z = landed(fold, zero);
                __syncwarp();
                if (lane == 0) {
                    atomicAdd(const_cast<uint32_t *>(sel_done) + buf + z, 1u);
                    mbar_arrive(&planes_empty[buf + z]);
                }
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    nibble_counts(acc, w4[j].w, w4[j].z, w4[j].y, w4[j].x, eq[j]);
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint32_t v = acc[c];
                v += __shfl_xor_sync(0xFFFFFFFFu, v, 1); // stage classes
                if (G == 4) v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
                if (LOG2S >= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, 16); // sub-blocks
                if (LOG2S >= 2) v += __shfl_xor_sync(0xFFFFFFFFu, v, 8);
                if (LOG2S >= 3) v += __shfl_xor_sync(0xFFFFFFFFu, v, 4);
                acc[c] = v;
            }
            // the zero-filled pad slots were counted as value 0
            if (MODE == 1 || h == 0u)
                acc[0] -= nst * kSlotsPerStage - nframes;
            if (MODE == 1 && LOG2S == 0 && nst >= 2u && push.stage) {
                // Coalesced push.  A warp's elements lie 16 apart, so storing the vectors directly makes every store
                // instruction write eight scattered 32-byte pieces -- poor packets for NVLink when the owner is a
                // peer.  This round never touches the LOW-nibble slots of the plane buffer (the transposers do not
                // fill them, see MODE 1 above), so the tile's 128 count vectors are staged there (8 chunks of 512 B:
                // stage k / 4, byte k % 4 of chunk k) and written out as 16 bytes per lane, 512 contiguous bytes per
                // warp.
                uint4 *stg = reinterpret_cast<uint4 *>(planes + buf * kBufWords);
                auto slot = [](uint32_t el, uint32_t half) { return (el >> 6) * 256u + ((el >> 4) & 3u) * 64u + (el & 15u) * 2u + half; };
                if (G == 4) {
                    const uint2 v = s_g == 0 ? make_uint2(acc[0], acc[1])
                                  : s_g == 1 ? make_uint2(acc[2], acc[3])
                                  : s_g == 2 ? make_uint2(acc[4], acc[5])
                                             : make_uint2(acc[6], acc[7]);
                    reinterpret_cast<uint2 *>(stg)[slot(s_elem, s_g >> 1) * 2u + (s_g & 1u)] = v;
                } else {
                    stg[slot(s_elem, s_g)] = s_g == 0 ? make_uint4(acc[0], acc[1], acc[2], acc[3]) : make_uint4(acc[4], acc[5], acc[6], acc[7]);
                }
                named_bar_sync(1, NSELW * 32);
                for (uint32_t j = tid; j < 256u; j += NSELW * 32u) { // selector threads are tid 0 .. NSELW*32-1
                    const uint32_t el = j >> 1, half = j & 1u;
                    const size_t ee = size_t(tile) * P + el;
                    if (ee < nelem) {
                        uint4 v = stg[slot(el, half)];
                        if (push.accum) {
                            const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(push.accum + ee * 8u + 4u * half));
                            v.x += a.x;
                            v.y += a.y;
                            v.z += a.z;
                            v.w += a.w;
                        }
                        const uint32_t owner = uint32_t(ee) / push.slice;
                        uint32_t *dst = push.dst[owner] + (ee - size_t(owner) * push.slice) * 8u + 4u * half;
                        *reinterpret_cast<uint4 *>(dst) = v;
                    }
                }
                named_bar_sync(1, NSELW * 32); // the staging slots are rewritten for the next tile of this buffer
            } else if ((lane >> kColBits) == 0u && e < nelem) {
                const uint32_t owner = uint32_t(e) / push.slice;
                uint32_t *dst = push.dst[owner] + (size_t(e) - size_t(owner) * push.slice) * 8u;
                // more than one frame chunk on this rank: add the counts of the chunks before this one (packed u16
                // pairs never carry: a rank holds at most 65535 frames)
                const uint32_t *prev = push.accum ? push.accum + size_t(e) * 8u : nullptr;
                if (G == 4) {
                    uint2 v = s_g == 0 ? make_uint2(acc[0], acc[1])
                            : s_g == 1 ? make_uint2(acc[2], acc[3])
                            : s_g == 2 ? make_uint2(acc[4], acc[5])
                                       : make_uint2(acc[6], acc[7]);
                    if (prev) {
                        const uint2 a = __ldcg(reinterpret_cast<const uint2 *>(prev + 2u * s_g));
                        v.x += a.x;
                        v.y += a.y;
                    }
                    *reinterpret_cast<uint2 *>(dst + 2u * s_g) = v;
                } else {
                    uint4 v = s_g == 0 ? make_uint4(acc[0], acc[1], acc[2], acc[3]) : make_uint4(acc[4], acc[5], acc[6], acc[7]);
                    if (prev) {
                        const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(prev + 4u * s_g));
                        v.x += a.x;
                        v.y += a.y;
                        v.z += a.z;
                        v.w += a.w;
                    }
                    *reinterpret_cast<uint4 *>(dst + 4u * s_g) = v;
                }
            }
        } else {
        uint32_t alive[JT];
#pragma unroll
        for (int j = 0; j < JT; ++j)
            alive[j] = (G * j + s_g) < nst ? 0xFFFFFFFFu : 0u; // rows >= nst hold garbage; alive == 0 masks them
        uint32_t k = k0;
        uint32_t med = 0;
#pragma unroll
        for (int bh = 1; bh >= 0; --bh) {
            uint4 w4[JT];
            if constexpr (kHalf) {
                // half-slot pool (see the transposers): this tile's high / low slots of stage 4j + g, then hand them back
                const uint32_t odd = it & 1u;
                const uint4 *hb = reinterpret_cast<const uint4 *>(planes) + s_g * 128u + s_p * 32u + s_col;
#pragma unroll
                for (int j = 0; j < JT; ++j) {
                    const bool first = uint32_t(G * j) + s_g < kFirst;
                    const uint32_t off = bh ? ((odd && !first) ? kFirst : 0u) : ((odd && first) ? kFirst : kCap);
                    w4[j] = hb[(uint32_t(G * j) + off) * 128u];
                }
                uint32_t fold = 0;
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    fold ^= w4[j].x;
                const uint32_t z = landed(fold, zero);
                __syncwarp();
                if (lane == 0)
                    red_release_shared_inc(rows_free + (bh ? 0 : 1) + z);
            } else {
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    w4[j] = base[j * (G * 256) + bh * 32]; // stage G*j+g, nibble bh: 4 planes in one LDS.128
                if (bh == 0) {
                    // every plane word this thread needs is now in registers: hand the buffer back to the transposers
                    uint32_t fold = 0;
#pragma unroll
                    for (int j = 0; j < JT; ++j)
                        fold ^= w4[j].x;
                    const uint32_t z = landed(fold, zero);
                    __syncwarp();
                    if (lane == 0) {
                        atomicAdd(const_cast<uint32_t *>(sel_done) + buf + z, 1u);
                        mbar_arrive(&planes_empty[buf + z]);
                    }
                }
            }
#pragma unroll
            for (int bl = 3; bl >= 0; --bl) {
                uint32_t cnt = 0;
#pragma unroll
                for (int j = 0; j < JT; ++j) {
                    const uint32_t wv = bl == 0 ? w4[j].x : bl == 1 ? w4[j].y : bl == 2 ? w4[j].z : w4[j].w;
                    cnt += __popc(alive[j] & ~wv);
                }
                cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 1); // stage classes
                if (G == 4) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 2);
                if (LOG2S >= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 16); // sub-blocks
                if (LOG2S >= 2) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 8);
                if (LOG2S >= 3) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, 4);
                const bool one = k >= cnt; // fewer than k+1 candidates have a 0 here -> the bit is 1
                if (one) {
                    k -= cnt;
                    med |= 1u << (4 * bh + bl);
                }
                const uint32_t flip = one ? 0u : 0xFFFFFFFFu;
#pragma unroll
                for (int j = 0; j < JT; ++j) {
                    const uint32_t wv = bl == 0 ? w4[j].x : bl == 1 ? w4[j].y : bl == 2 ? w4[j].z : w4[j].w;
                    alive[j] &= (wv ^ flip);
                }
            }
        }
        const size_t e = size_t(tile) * P + s_elem;
        if (s_writer && e < nelem)
            out[e] = uint8_t(med);
        } // MODE == 0
    }
    if (MODE != 0)
        __threadfence_system(); // pushed counts are visible to the peers once this kernel has completed
}

template <int LOG2S, int JT, int NSELW, int MODE>
int launch_pipe_variant(cvvp_ctx *ctx, const CUtensorMap &tmap, uint8_t *d_out, uint32_t nelem, uint32_t nframes,
                        uint32_t nst, uint32_t percent, const ShardPush &push, cudaStream_t stream)
{
    constexpr int P = 128 >> LOG2S;
    constexpr uint32_t G = NSELW / 4;
    constexpr uint32_t NBUF = (NSELW == 8) ? 2 : 1;
    const uint32_t ntiles = (nelem + P - 1) / P;
    const size_t smem_bytes = size_t(kRing) * kStageBytes + size_t(NBUF) * (G * JT * 4096u) + size_t(kRing + 4) * 8 + 16 + 48 + (MODE == 3 ? 2560 : 0);
    if (smem_bytes > ctx->smem_optin)
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: tile does not fit shared memory");
    auto kern = median_pipe_kernel<LOG2S, JT, NSELW, MODE>;
    CVVP_CUDA_OK(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_bytes)));
    const uint32_t grid = ntiles < uint32_t(ctx->sm_count) ? ntiles : uint32_t(ctx->sm_count);
    // P == 128: every line is read exactly once -> evict-first.  P < 128: the neighbouring CTA reads the other part
    // of the line at about the same time and should hit L2.
    const uint64_t policy = (LOG2S == 0) ? kL2EvictFirst : kL2EvictNormal;
    kern<<<grid, (NSELW + kTrWarps) * 32, smem_bytes, stream>>>(tmap, d_out, nelem, nframes, nst, ntiles, policy, percent, push);
    CVVP_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches++;
    return CVVP_OK;
}

template <int LOG2S, int NSELW, int MODE>
int dispatch_jt(cvvp_ctx *ctx, const CUtensorMap &tmap, uint8_t *d_out, uint32_t nelem, uint32_t nframes, uint32_t nst,
                uint32_t percent, const ShardPush &push, cudaStream_t stream)
{
    constexpr uint32_t G = NSELW / 4;
    switch ((nst + G - 1u) / G) {
#define CVVP_JT_CASE(J) \
    case J: return launch_pipe_variant<LOG2S, J, NSELW, MODE>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
        CVVP_JT_CASE(1)
        CVVP_JT_CASE(2)
        CVVP_JT_CASE(3)
        CVVP_JT_CASE(4)
        CVVP_JT_CASE(5)
        CVVP_JT_CASE(6)
        CVVP_JT_CASE(7)
        CVVP_JT_CASE(8)
#undef CVVP_JT_CASE
    default: return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: unsupported stage count %u", nst);
    }
}

template <int LOG2S, int MODE>
int dispatch_bufs(cvvp_ctx *ctx, const CUtensorMap &tmap, uint8_t *d_out, uint32_t nelem, uint32_t nframes, uint32_t nst,
                  uint32_t percent, const ShardPush &push, cudaStream_t stream)
{
    const char *e = getenv("CVVP_MEDIAN_BUFFERS"); // development switch: "1" forces the single-buffer mode
    const bool force_single = e && e[0] == '1';
    if (nst <= 16 && !force_single)
        return dispatch_jt<LOG2S, 8, MODE>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
    return dispatch_jt<LOG2S, 16, MODE>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
}

template <int LOG2S>
int dispatch_mode(cvvp_ctx *ctx, const CUtensorMap &tmap, uint8_t *d_out, uint32_t nelem, uint32_t nframes, uint32_t nst,
                  int mode, uint32_t percent, const ShardPush &push, cudaStream_t stream)
{
    switch (mode) {
    case 0: return dispatch_bufs<LOG2S, 0>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
    case 1: return dispatch_bufs<LOG2S, 1>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
    case 2: return dispatch_bufs<LOG2S, 2>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
    case 3:
        if constexpr (LOG2S == 0)
            return dispatch_jt<0, 16, 3>(ctx, tmap, d_out, nelem, nframes, nst, percent, push, stream);
        else
            return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: window counting takes at most 1024 frames per launch");
    default: return fail(ctx, CVVP_ERR_INVALID, "median: bad kernel mode %d", mode);
    }
}
} // namespace

// Largest frame count the kernel takes: 32 stages x 256 frame slots at P = 16.
long long median_max_frames()
{
    return 32ll * 256ll;
}

int median_pipe_launch(cvvp_ctx *ctx, const CUtensorMap &tmap, int log2s, uint8_t *d_out, uint32_t nelem,
                       uint32_t nframes, uint32_t nst, int mode, uint32_t percent, const ShardPush &push,
                       cudaStream_t stream)
{
    if (nst == 0 || nst > 32)
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median: %u stages exceed the plane buffer", nst);
    switch (log2s) {
    case 0: return dispatch_mode<0>(ctx, tmap, d_out, nelem, nframes, nst, mode, percent, push, stream);
    case 1: return dispatch_mode<1>(ctx, tmap, d_out, nelem, nframes, nst, mode, percent, push, stream);
    case 2: return dispatch_mode<2>(ctx, tmap, d_out, nelem, nframes, nst, mode, percent, push, stream);
    case 3: return dispatch_mode<3>(ctx, tmap, d_out, nelem, nframes, nst, mode, percent, push, stream);
    default: return fail(ctx, CVVP_ERR_INVALID, "median: bad tile variant");
    }
}
} // namespace cvvp
