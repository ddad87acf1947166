// Frame-sharded temporal median across GPUs: the exchange step of BASELINE.json:north_star ("the median shards over
// frame chunks ... before the median select"), fused with the counting kernels over NVLink peer memory.
//
// The reference's analogue is its temporal sharding of the frame range over generator threads
// (/root/reference/Sources/cv_vid_bg_helpers.cpp:84-120) feeding one order-independent histogram
// (histogram_median_algo.h:116-141); the result is the same sorted[N/2] of ALL frames (:160-166) -- in general
// sorted[k(N, p)] for the job's percentile p (percentile_rank, median_common.cuh; the owner kernels below take the rank
// from there, and the window test and the nibble rounds are exact for any rank).
//
// Every rank holds a chunk of the frames (all elements).  Element e is OWNED by rank e / slice.  Instead of
// all-reducing 256-bin histograms (512 B per element), the select is a two-round radix select on nibbles, and
// the counts travel straight from the counting kernel into the owner's memory (reduce-scatter by peer stores):
//
//   phase 0  every rank : 16-bin counts of the HIGH nibble of its frames (median_pipe_kernel MODE 1, the same
//                         TMA -> bit-transpose pipeline as the single-GPU kernel), 32 B per element stored into
//                         owner's  counts1[src rank][e - owner * slice]
//   phase 1  owner      : sums the `world` count vectors, N = their total, k = k(N, p), picks the high nibble h with
//                         cum(h) > k and the residual rank k' = k - cum(< h); stores  sel[e] = h | k' << 8  into
//                         EVERY rank's sel array (4 B per element)
//   phase 2  every rank : 16-bin counts of the LOW nibble among its frames with high nibble == h (MODE 2), pushed
//                         into owner's counts2 the same way
//   phase 3  owner      : sums, picks the low nibble l with cum(l) > k'; stores the result byte h << 4 | l into
//                         EVERY rank's result image (all-gather by peer stores)
//
// ONE-PASS FORM (phases 4 and 5, tried first).  The two rounds above read every frame twice.  Phase 4
// (median_pipe_kernel MODE 3) reads them once: each launch (<= 1024 frames of a rank) picks, per element, a pilot
// median of 256 of its own frames on chip and counts ALL its frames in the 8-value window [pilot - 4, pilot + 3]
// and below it; the 20-byte record {8 x u16 bins, below | window base << 16} goes to the element's owner like the
// nibble counts do (the launch's frame count goes to one header word per owner).  Phase 5 (shard_window_final_kernel, owner): the cumulative count of all sources is exact on the
// intersection [lo - 1, hi] of their windows, so whenever G(lo - 1) <= k < G(hi) the result is the first value
// there with G(v) > k -- the reference's rule (:160-166) at k = N/2 -- and it is stored into every rank's result image.
// Elements whose median lies outside some source's window (sources with very different content) are counted into
// every rank's `unresolved` word and their 128-element tile is flagged on every rank; the job then runs phases
// 10..13 = phases 0..3 restricted to the flagged tiles (the counting kernels walk a compacted tile list, the owner
// kernels skip elements of other tiles), so a handful of flickering pixels costs a few tiles, not a second and third
// pass over the stack.  Phases 0..3 on the whole image stay available (exact for any input on their own).  A video
// background resolves everywhere; the result is bit-identical either way.
//
// Between phases the caller places a cross-rank barrier on the stream (a kernel's peer stores are complete when the
// kernel is; the barrier orders them before the peer's next kernel).  No kernel ever waits for another rank, so ranks
// can also be emulated one after another on a single device (tests).  Traffic per element per rank: 2 x 32 B out,
// 2 x 32 B x (world-1)/world in, + 5 B broadcast -- 8x less than all-reducing 256 x u16 histograms, and the two
// passes over the frames stay at HBM speed.
#include "context.hpp"
#include "median_common.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>

namespace cvvp
{
struct MedianShard {
    int rank{0}, world{1};
    size_t nelem{0};
    uint32_t slice{0};      // elements owned per rank (multiple of 128)
    uint8_t *buf{nullptr};  // one allocation: counts1 | counts2 | sel | result
    size_t bytes{0};
    size_t off_c1{0}, off_c2{0}, off_sel{0}, off_res{0};
    uint8_t *peer[kMaxShardRanks]{}; // base of every rank's buffer as mapped into this process (peer[rank] == buf)
    bool ipc_opened[kMaxShardRanks]{};
    bool attached[kMaxShardRanks]{};
    uint32_t *accum{nullptr}; // [nelem][8 words]: running counts of this rank's frame chunks (allocated on first use)
    int spr{1}; // count slots per rank: a rank with more than 65535 frames pushes one 16-bit count vector per 65535 frames,
                // the owners sum world * spr vectors in 32 bits (world * spr <= kMaxShardRanks)
    int wsubs{1}; // window records per rank (one per launch of <= 1024 frames) the first receive area has room for
    int cslots{1}; // record slots per rank of the first receive area = max(spr, wsubs)
    size_t off_flag{0}; // word 0: elements the window pass left unresolved (summed over all owners); word 1: flagged tiles
    size_t off_tflag{0}; // [ntiles] words: tile holds an undecided element (written by the owners of its elements)
    size_t off_tlist{0}; // [ntiles] words: the flagged tiles, compacted (phase 10)
    size_t off_hdr{0};   // [world * cslots] words: frames counted by the window records of every source slot
    size_t off_bar{0};   // [kMaxShardRanks] words: bar[r] = the last barrier epoch rank r has arrived at (cvvp_median_shard_barrier)
    uint32_t ntiles{0};
    uint32_t epoch{0};   // barriers this rank has issued
    int percent{50};     // the percentile this rank selects (every rank of a job must use the same)
};

// frames one launch of the counting kernel takes at full tile width (128-byte TMA boxes): 32 stages x 32 frames
constexpr long long kChunkFrames = 1024;
constexpr long long kSlotFrames = 65535; // 16-bit counts per slot

namespace
{
struct OwnerArgs {
    const uint32_t *counts; // this rank's receive area of the round: [rank][slot][slice][8 words]
    uint32_t slice, world, rank; // world = vectors / records to sum = ranks x used slots per rank
    uint32_t used, slots;        // slots a rank uses this round / slots per rank in the area
    uint32_t nranks;        // ranks the decisions are broadcast to
    uint32_t owned;         // elements this rank owns
    uint32_t *sel[kMaxShardRanks];    // every rank's sel array
    uint8_t *result[kMaxShardRanks];  // every rank's result image
    uint32_t *flag[kMaxShardRanks];   // window pass: every rank's `unresolved` word
    uint32_t *tflag[kMaxShardRanks];  // window pass: every rank's tile flags
    const uint32_t *tile_list;        // restricted rounds: the flagged tiles and how many there are
    const uint32_t *tile_count;
    const uint32_t *src_frames;       // window pass: frames behind every source slot's records (0: skip the slot)
    uint32_t percent;                 // the job's percentile: rank k(N, percent) of the N frames of all sources
};

// the s-th vector / record of the round lives in slot (s % used) of rank (s / used)
__device__ __forceinline__ size_t src_slot(const OwnerArgs &A, uint32_t s)
{
    return A.used == A.slots ? size_t(s) : size_t(s / A.used) * A.slots + (s % A.used);
}

__device__ __forceinline__ void add_counts(uint32_t (&cnt)[16], const uint32_t *p)
{
    const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(p));
    const uint4 b = __ldcg(reinterpret_cast<const uint4 *>(p) + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        cnt[2 * c] += w[c] & 0xFFFFu;
        cnt[2 * c + 1] += w[c] >> 16;
    }
}

// phase 1 for owned element i
__device__ __forceinline__ void pick_element(const OwnerArgs &A, uint32_t i)
{
    uint32_t cnt[16];
#pragma unroll
    for (int b = 0; b < 16; ++b)
        cnt[b] = 0;
    for (uint32_t src = 0; src < A.world; ++src)
        add_counts(cnt, A.counts + (src_slot(A, src) * A.slice + i) * 8u);
    uint32_t total = 0;
#pragma unroll
    for (int b = 0; b < 16; ++b)
        total += cnt[b];
    // first bin with cumulative count > k(N, p)  (N / 2 at p = 50: the reference's rule, :160-166)
    const uint32_t k = percentile_rank(total, A.percent);
    uint32_t h = 15u, below = 0u, cum = 0u;
    bool found = false;
#pragma unroll
    for (int b = 0; b < 16; ++b) {
        if (!found && cum + cnt[b] > k) {
            h = uint32_t(b);
            below = cum;
            found = true;
        }
        cum += cnt[b];
    }
    if (!found)
        below = total - cnt[15]; // unreachable with exact counts; mirrors the reference's default bin
    const uint32_t v = h | ((k - below) << 8);
    const size_t e = size_t(A.rank) * A.slice + i;
    for (uint32_t r = 0; r < A.nranks; ++r)
        A.sel[r][e] = v;
}

// phase 3 for the owned elements i4 .. i4 + 3 (one 32-bit store of result bytes per rank)
__device__ __forceinline__ void final_group(const OwnerArgs &A, uint32_t i4)
{
    const size_t e0 = size_t(A.rank) * A.slice + i4;
    uint32_t packed = 0;
    const uint32_t n = min(4u, A.owned - i4);
    for (uint32_t q = 0; q < n; ++q) {
        uint32_t cnt[16];
#pragma unroll
        for (int b = 0; b < 16; ++b)
            cnt[b] = 0;
        for (uint32_t src = 0; src < A.world; ++src)
            add_counts(cnt, A.counts + (src_slot(A, src) * A.slice + i4 + q) * 8u);
        const uint32_t s = __ldcg(A.sel[A.rank] + e0 + q);
        const uint32_t h = s & 15u, k = s >> 8;
        uint32_t l = 15u, cum = 0u;
        bool found = false;
#pragma unroll
        for (int b = 0; b < 16; ++b) {
            if (!found && cum + cnt[b] > k) {
                l = uint32_t(b);
                found = true;
            }
            cum += cnt[b];
        }
        packed |= ((h << 4) | l) << (8u * q);
    }
    for (uint32_t r = 0; r < A.nranks; ++r) {
        uint8_t *dst = A.result[r] + e0;
        if (n == 4u) {
            *reinterpret_cast<uint32_t *>(dst) = packed; // e0 is a multiple of 4 (slice % 128 == 0)
        } else {
            for (uint32_t q = 0; q < n; ++q)
                dst[q] = uint8_t(packed >> (8u * q));
        }
    }
}

// phases 1 and 3 over ALL owned elements: one thread per element / per 4 elements
__global__ void __launch_bounds__(256) shard_pick_kernel(const __grid_constant__ OwnerArgs A)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < A.owned)
        pick_element(A, i);
    __threadfence_system();
}

__global__ void __launch_bounds__(256) shard_final_kernel(const __grid_constant__ OwnerArgs A)
{
    const uint32_t i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4u;
    if (i4 < A.owned)
        final_group(A, i4);
    __threadfence_system();
}

// phases 11 and 13: the same over the LISTED tiles only (128 elements each; a tile lies inside one owner's slice).  A
// fixed grid walks the list, so an empty list costs a launch and nothing else.
__global__ void __launch_bounds__(128) shard_pick_listed_kernel(const __grid_constant__ OwnerArgs A)
{
    const uint32_t n = __ldcg(A.tile_count);
    const uint32_t first = A.rank * A.slice;
    for (uint32_t idx = blockIdx.x; idx < n; idx += gridDim.x) {
        const uint32_t e = __ldcg(A.tile_list + idx) * 128u + threadIdx.x;
        if (e >= first && e - first < A.owned)
            pick_element(A, e - first);
    }
    __threadfence_system();
}

__global__ void __launch_bounds__(32) shard_final_listed_kernel(const __grid_constant__ OwnerArgs A)
{
    const uint32_t n = __ldcg(A.tile_count);
    const uint32_t first = A.rank * A.slice;
    for (uint32_t idx = blockIdx.x; idx < n; idx += gridDim.x) {
        const uint32_t e = __ldcg(A.tile_list + idx) * 128u + 4u * threadIdx.x;
        if (e >= first && e - first < A.owned)
            final_group(A, e - first);
    }
    __threadfence_system();
}

// phase 5: window records of every source -> result bytes.  One thread per owned element (a warp reads 640
// consecutive bytes of records per source); four neighbouring lanes pool their bytes into one 32-bit store per rank.
// Record of source slot s for owned element i: 5 words at counts[(s * slice * 8) + i * 5]: words 0..3 = bins 0..7
// (16 bits each), word 4 = frames below the window | window base << 16; src_frames[s] = frames of the source (0: the
// slot is empty and is skipped).
__global__ void __launch_bounds__(256) shard_window_final_kernel(const __grid_constant__ OwnerArgs A)
{
    // The records are read ONCE, coalesced: a group's 256 records of a source are 5120 contiguous bytes, fetched 16 bytes
    // per thread (the next source's while this one is evaluated) and handed out through shared memory.  Windows that
    // intersect lie within 7 values of each other, so counts are kept by position relative to the FIRST source's window
    // (value v at v - base0 + 7, 23 positions); a source further away means an empty intersection.  A block walks over
    // many groups of 256 elements and fences its peer stores once, at the end (one system-wide fence per 256 elements
    // was most of this kernel's time).
    __shared__ uint32_t hist[23][256];
    __shared__ __align__(16) uint32_t stage[2][1280];
    __shared__ uint32_t unresolved;
    const uint32_t tid = threadIdx.x;
    if (tid == 0)
        unresolved = 0;
    // next source slot with frames at or after s (uniform over the block)
    auto next_source = [&](uint32_t s) {
        while (s < A.world && __ldg(A.src_frames + src_slot(A, s)) == 0u)
            ++s;
        return s;
    };
    const uint32_t ngroups = (A.owned + 255u) / 256u;
    for (uint32_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
        __syncthreads(); // the previous group's stage buffers and histogram are no longer read (and `unresolved` is set)
#pragma unroll
        for (int c = 0; c < 23; ++c)
            hist[c][tid] = 0;
        const uint32_t i0 = g * 256u;
        const uint32_t i = i0 + tid;
        const bool mine = i < A.owned;
        const uint32_t nw = min(256u, A.owned - i0) * 5u; // record words of this group per source
        uint4 ra = make_uint4(0, 0, 0, 0), rb = ra;
        auto fetch = [&](uint32_t s) {
            const uint4 *src = reinterpret_cast<const uint4 *>(A.counts + src_slot(A, s) * A.slice * 8u + size_t(i0) * 5u);
            if (4u * tid < nw)
                ra = __ldcg(src + tid);
            if (tid < 64u && 4u * (256u + tid) < nw)
                rb = __ldcg(src + 256u + tid);
        };
        uint32_t total = 0, lo = 0, hi = 255, cum = 0, base0 = 0;
        bool first = true, far = false;
        uint32_t s = next_source(0);
        if (s < A.world)
            fetch(s);
        for (uint32_t buf = 0; s < A.world; buf ^= 1u) {
            uint4 *st4 = reinterpret_cast<uint4 *>(stage[buf]);
            st4[tid] = ra;
            if (tid < 64u)
                st4[256u + tid] = rb;
            __syncthreads(); // (the buffer written two sources ago was read before the previous barrier)
            const uint32_t nfr = __ldg(A.src_frames + src_slot(A, s));
            s = next_source(s + 1u);
            if (s < A.world)
                fetch(s);
            if (mine) {
                const uint32_t *rec = stage[buf] + tid * 5u;
                const uint32_t w[4] = {rec[0], rec[1], rec[2], rec[3]};
                const uint32_t t = rec[4];
                const uint32_t base = t >> 16;
                if (first) {
                    base0 = base;
                    first = false;
                }
                total += nfr;
                lo = max(lo, base);
                hi = min(hi, base + 7u);
                cum += t & 0xFFFFu; // frames below this source's window
                const int off = int(base) - int(base0) + 7;
                if (off < 0 || off > 14) {
                    far = true;
                } else {
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        hist[off + c][tid] += (c & 1) ? (w[c >> 1] >> 16) : (w[c >> 1] & 0xFFFFu);
                }
            }
        }
        uint32_t med = 0;
        bool ok = true;
        if (mine) {
            ok = false;
            // first value with cumulative count > k(N, p)  (N / 2 at p = 50: the reference's rule, :160-166)
            const uint32_t k = percentile_rank(total, A.percent);
            if (total != 0u && !far && lo <= hi) {
                // G(lo - 1) = frames below every window + the counted values <= lo - 1; G is exact up to hi
                const uint32_t p0 = lo - base0 + 7u; // position of value lo
                for (uint32_t pos = 0; pos < p0; ++pos)
                    cum += hist[pos][tid];
                const uint32_t span = hi - lo + 1u;
                if (cum <= k) {
                    for (uint32_t c = 0; c < span; ++c) {
                        cum += hist[p0 + c][tid];
                        if (cum > k) {
                            med = lo + c;
                            ok = true;
                            break;
                        }
                    }
                }
            }
        }
        // four lanes -> one word (owned slices start at multiples of 128 elements, so element i & ~3 is word aligned)
        uint32_t packed = med << (8u * (tid & 3u));
        packed |= __shfl_xor_sync(0xFFFFFFFFu, packed, 1);
        packed |= __shfl_xor_sync(0xFFFFFFFFu, packed, 2);
        if (mine && (tid & 3u) == 0u) {
            const size_t e0 = size_t(A.rank) * A.slice + i;
            const uint32_t n = min(4u, A.owned - i);
            for (uint32_t r = 0; r < A.nranks; ++r) {
                uint8_t *dst = A.result[r] + e0;
                if (n == 4u) {
                    *reinterpret_cast<uint32_t *>(dst) = packed;
                } else {
                    for (uint32_t q = 0; q < n; ++q)
                        dst[q] = uint8_t(packed >> (8u * q));
                }
            }
        }
        if (!ok) {
            atomicAdd(&unresolved, 1u);
            const size_t tile = (size_t(A.rank) * A.slice + i) >> 7; // the 128-element tile of the counting kernels
            for (uint32_t r = 0; r < A.nranks; ++r)
                A.tflag[r][tile] = 1u;
        }
    }
    __syncthreads();
    if (tid == 0 && unresolved != 0u)
        for (uint32_t r = 0; r < A.nranks; ++r)
            atomicAdd_system(A.flag[r], unresolved);
    __threadfence_system();
}

// phase 10, before the restricted counting: flagged tiles -> compact list (one block; *count is zero on entry)
__global__ void __launch_bounds__(1024) shard_tile_list_kernel(const uint32_t *__restrict__ flags, uint32_t ntiles,
                                                               uint32_t *__restrict__ list, uint32_t *__restrict__ count)
{
    for (uint32_t t = threadIdx.x; t < ntiles; t += blockDim.x)
        if (__ldcg(flags + t) != 0u)
            list[atomicAdd(count, 1u)] = t;
}

// window counting: a source slot without frames only tells every owner so
__global__ void shard_empty_slot_kernel(const __grid_constant__ ShardPush push)
{
    if (threadIdx.x < push.nranks)
        *push.hdr[threadIdx.x] = 0u;
    __threadfence_system();
}

// Cross-rank barrier on the stream, for ranks that each have a GPU of their own: lane r tells rank r "I have arrived
// at barrier `epoch`" (a system-scope release store into r's exchange buffer over NVLink) and waits until rank r has
// told this rank the same.  Everything a rank queued before its barrier -- its counting kernel's peer stores, each
// fenced system-wide -- is complete before it signals, so what follows the barrier on any rank sees it.  One warp, a
// few microseconds, where a one-element NCCL all-reduce costs 15-25.  The peers' kernels run on OTHER devices; ranks
// that share a device must not use this (the waiting kernel would keep the other rank's kernel from ever running):
// they take a host-side barrier instead.  A wait of more than 2 s traps.
struct BarrierArgs {
    uint32_t *bar[kMaxShardRanks]; // every rank's flag array
    uint32_t rank, world, epoch;
};

__global__ void __launch_bounds__(32) shard_barrier_kernel(const __grid_constant__ BarrierArgs B)
{
    const uint32_t r = threadIdx.x;
    if (r < B.world) {
        __threadfence_system();
        uint32_t *theirs = B.bar[r] + B.rank;
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(theirs), "r"(B.epoch) : "memory");
        const uint32_t *mine = B.bar[B.rank] + r;
        uint32_t v;
        unsigned long long t0 = 0;
        uint32_t spins = 0;
        for (;;) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
            if (int32_t(v - B.epoch) >= 0)
                break;
            __nanosleep(100);
            if ((++spins & 0xFFu) == 0) {
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                if (t0 == 0)
                    t0 = t;
                else if (t - t0 > 2000000000ull)
                    __trap();
            }
        }
    }
    __syncwarp();
    __threadfence_system();
}

// a rank without frames still owes every owner a (zero) count vector
__global__ void __launch_bounds__(256) shard_zero_push_kernel(const __grid_constant__ ShardPush push, uint32_t nelem)
{
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; // one 16-byte half of an element's counts
    if (i < size_t(nelem) * 2u) {
        const uint32_t e = uint32_t(i >> 1);
        const uint32_t owner = e / push.slice;
        uint32_t *dst = push.dst[owner] + (size_t(e) - size_t(owner) * push.slice) * 8u + 4u * (i & 1u);
        *reinterpret_cast<uint4 *>(dst) = make_uint4(0, 0, 0, 0);
    }
    __threadfence_system();
}

bool all_peers_known(const MedianShard *sh)
{
    for (int r = 0; r < sh->world; ++r)
        if (!sh->peer[r])
            return false;
    return true;
}
} // namespace

static void shard_destroy(cvvp_ctx *ctx, MedianShard *&sh)
{
    if (!sh)
        return;
    cudaStreamSynchronize(ctx->compute);
    for (int r = 0; r < sh->world; ++r)
        if (sh->ipc_opened[r] && sh->peer[r])
            cudaIpcCloseMemHandle(sh->peer[r]);
    if (sh->buf)
        cudaFree(sh->buf);
    if (sh->accum)
        cudaFree(sh->accum);
    cudaGetLastError();
    delete sh;
    sh = nullptr;
}

void median_shard_release(cvvp_ctx *ctx)
{
    shard_destroy(ctx, ctx->shard);
    shard_destroy(ctx, ctx->big);
}

static int shard_create(cvvp_ctx *ctx, size_t nelem, int rank, int world, int spr, int wsubs, MedianShard **out)
{
    MedianShard *sh = new (std::nothrow) MedianShard();
    if (!sh)
        return fail(ctx, CVVP_ERR_NOMEM, "out of host memory");
    sh->percent = ctx->percent; // a sharded job takes the context's percentile when it begins
    sh->rank = rank;
    sh->world = world;
    sh->spr = spr;
    sh->wsubs = wsubs < 1 ? 1 : wsubs;
    sh->cslots = std::max(sh->spr, sh->wsubs);
    sh->nelem = nelem;
    sh->slice = uint32_t(round_up((nelem + size_t(world) - 1) / size_t(world), 128));
    // the first receive area holds the round-1 count vectors (spr per rank) or the window records (wsubs per rank)
    const size_t counts1_bytes = size_t(world) * size_t(sh->cslots) * sh->slice * 32u;
    const size_t counts2_bytes = size_t(world) * size_t(spr) * sh->slice * 32u;
    sh->off_c1 = 0;
    sh->off_c2 = counts1_bytes;
    sh->off_sel = counts1_bytes + counts2_bytes;
    sh->off_res = sh->off_sel + round_up(nelem * 4u, 256);
    sh->ntiles = uint32_t((nelem + 127) / 128);
    sh->off_flag = sh->off_res + round_up(nelem, 256);
    sh->off_tflag = sh->off_flag + 256;
    sh->off_tlist = sh->off_tflag + round_up(size_t(sh->ntiles) * 4u, 256);
    sh->off_hdr = sh->off_tlist + round_up(size_t(sh->ntiles) * 4u, 256);
    sh->off_bar = sh->off_hdr + round_up(size_t(world) * size_t(sh->cslots) * 4u, 256);
    sh->bytes = sh->off_bar + 256;
    if (cudaMalloc(reinterpret_cast<void **>(&sh->buf), sh->bytes) != cudaSuccess) {
        cudaGetLastError();
        const size_t wanted = sh->bytes;
        delete sh;
        return fail(ctx, CVVP_ERR_NOMEM, "median shard: cudaMalloc of %zu bytes of exchange buffers failed", wanted);
    }
    if (cudaMemsetAsync(sh->buf, 0, sh->bytes, ctx->compute) != cudaSuccess ||
        cudaStreamSynchronize(ctx->compute) != cudaSuccess) {
        cudaFree(sh->buf);
        delete sh;
        return fail(ctx, CVVP_ERR_CUDA, "median shard: clearing the exchange buffers failed");
    }
    sh->peer[rank] = sh->buf;
    *out = sh;
    return CVVP_OK;
}

// counting round (phase 0 or 2) of the frames of ONE count slot (at most 65535)
static int shard_count_slot(cvvp_ctx *ctx, MedianShard *sh, int phase, const uint8_t *d_frames, long long nframes,
                            size_t frame_stride, const ShardPush &push, cudaStream_t s)
{
    if (nframes == 0) {
        const size_t n = sh->nelem * 2;
        shard_zero_push_kernel<<<unsigned((n + 255) / 256), 256, 0, s>>>(push, uint32_t(sh->nelem));
        CVVP_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches++;
        return CVVP_OK;
    }
    if (nframes <= kChunkFrames)
        return median_launch_mode(ctx, d_frames, nframes, sh->nelem, frame_stride, nullptr, phase == 0 ? 1 : 2, sh->percent,
                                  push, s);
    // long chunk of frames: several launches at full tile width; the counts of launch c are added to those of
    // launches < c in a local array, the last launch pushes the totals to the owners
    if (!sh->accum && cudaMalloc(reinterpret_cast<void **>(&sh->accum), sh->nelem * 32u) != cudaSuccess) {
        cudaGetLastError();
        sh->accum = nullptr;
        return fail(ctx, CVVP_ERR_NOMEM, "median shard: cudaMalloc of %zu bytes for the running counts failed", sh->nelem * 32u);
    }
    const long long nchunks = (nframes + kChunkFrames - 1) / kChunkFrames;
    long long per = (nframes + nchunks - 1) / nchunks;
    per = (per + 31) / 32 * 32; // whole plane words
    if (per > kChunkFrames)
        per = kChunkFrames;
    for (long long first = 0, c = 0; first < nframes; first += per, ++c) {
        const long long n = nframes - first < per ? nframes - first : per;
        const bool last = first + n >= nframes;
        ShardPush cp = push;
        cp.accum = c == 0 ? nullptr : sh->accum;
        if (!last) { // every element "belongs" to slot 0 = the local running counts
            cp.dst[0] = sh->accum;
            cp.slice = 0x80000000u;
        }
        const int rc = median_launch_mode(ctx, d_frames + size_t(first) * frame_stride, n, sh->nelem, frame_stride, nullptr,
                                          phase == 0 ? 1 : 2, sh->percent, cp, s);
        if (rc != CVVP_OK)
            return rc;
    }
    return CVVP_OK;
}

// Window counting (phase 4) of this rank's frames: launches of <= 1024 frames, each into its own record slot
// (rank * cslots + j) of every owner; slots beyond the launches receive empty records (frame count 0).
static int shard_window_count(cvvp_ctx *ctx, MedianShard *sh, const uint8_t *d_frames, long long nframes, size_t frame_stride,
                              cudaStream_t s)
{
    const long long nsub = nframes == 0 ? 0 : (nframes + kChunkFrames - 1) / kChunkFrames;
    if (nsub > sh->wsubs)
        return fail(ctx, CVVP_ERR_UNSUPPORTED,
                    "median shard: %lld frames need %lld window records per rank, the job was begun with room for %d", nframes,
                    nsub, sh->wsubs);
    long long per = nsub ? (nframes + nsub - 1) / nsub : 0;
    per = (per + 31) / 32 * 32; // whole plane words
    if (per > kChunkFrames)
        per = kChunkFrames;
    // the undecided count, the list length and the tile flags of this job (one contiguous region)
    CVVP_CUDA_OK(ctx, cudaMemsetAsync(sh->buf + sh->off_flag, 0, (sh->off_tflag - sh->off_flag) + size_t(sh->ntiles) * 4u, s));
    for (int j = 0; j < sh->wsubs; ++j) {
        ShardPush push{};
        const size_t slot = size_t(sh->rank) * sh->cslots + size_t(j);
        const size_t off = sh->off_c1 + slot * sh->slice * 32u; // (records take 20 of a slot's 32 bytes per element)
        for (int r = 0; r < sh->world; ++r) {
            push.dst[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + off);
            push.hdr[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + sh->off_hdr) + slot;
        }
        push.nranks = uint32_t(sh->world);
        push.slice = sh->slice;
        {
            // staged push (a tile's records assembled in shared memory, written 16 bytes per thread): pays for its two
            // named barriers per tile once most owners are peers.  CVVP_SHARD_STAGE=0/1 forces it off / on.
            const char *e = getenv("CVVP_SHARD_STAGE");
            push.stage = e ? (e[0] == '1') : (sh->world > 1);
        }
        const long long first = std::min<long long>(nframes, per * j);
        const long long n = std::min<long long>(nframes - first, per);
        if (n <= 0) {
            shard_empty_slot_kernel<<<1, 32, 0, s>>>(push);
            CVVP_CUDA_OK(ctx, cudaGetLastError());
            ctx->launches++;
            continue;
        }
        const int rc = median_launch_mode(ctx, d_frames + size_t(first) * frame_stride, n, sh->nelem, frame_stride, nullptr, 3,
                                          sh->percent, push, s);
        if (rc != CVVP_OK)
            return rc;
    }
    return CVVP_OK;
}

// One phase of a sharded job (see the file header).  d_result: where phase 3 stores this rank's copy of the result
// bytes instead of its own exchange buffer (the one-rank two-pass path writes straight into the caller's image).
static int shard_phase(cvvp_ctx *ctx, MedianShard *sh, int phase, const uint8_t *d_frames, long long nframes,
                       size_t frame_stride, uint8_t *d_result, cudaStream_t s)
{
    // phases 10..13: phases 0..3 restricted to the tiles the window pass flagged
    const bool restricted = phase >= 10 && phase <= 13;
    if (restricted)
        phase -= 10;
    if (!all_peers_known(sh))
        return fail(ctx, CVVP_ERR_STATE, "median shard: not every peer buffer is mapped (import / attach all ranks first)");
    if (nframes < 0)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: negative frame count");
    if (nframes > kSlotFrames * sh->spr)
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median shard: %lld frames on one rank exceed the %d x 16-bit counts (%lld)",
                    nframes, sh->spr, kSlotFrames * sh->spr);
    const uint32_t *tflags = reinterpret_cast<const uint32_t *>(sh->buf + sh->off_tflag);
    uint32_t *tlist = reinterpret_cast<uint32_t *>(sh->buf + sh->off_tlist);
    uint32_t *tcount = reinterpret_cast<uint32_t *>(sh->buf + sh->off_flag) + 1;
    if (phase == 4)
        return shard_window_count(ctx, sh, d_frames, nframes, frame_stride, s);
    if (restricted && phase == 0) {
        CVVP_CUDA_OK(ctx, cudaMemsetAsync(tcount, 0, sizeof(uint32_t), s));
        shard_tile_list_kernel<<<1, 1024, 0, s>>>(tflags, sh->ntiles, tlist, tcount);
        CVVP_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches++;
    }
    if (phase == 0 || phase == 2) {
        // slot j of this rank takes frames [j * 65535, (j + 1) * 65535) (possibly none)
        for (int j = 0; j < sh->spr; ++j) {
            const long long f0 = std::min<long long>(nframes, kSlotFrames * j);
            const long long nf = std::min<long long>(nframes - f0, kSlotFrames);
            ShardPush push{};
            const size_t off = phase == 0 ? sh->off_c1 + (size_t(sh->rank) * sh->cslots + size_t(j)) * sh->slice * 32u
                                          : sh->off_c2 + (size_t(sh->rank) * sh->spr + size_t(j)) * sh->slice * 32u;
            for (int r = 0; r < sh->world; ++r)
                push.dst[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + off);
            push.sel = reinterpret_cast<const uint32_t *>(sh->buf + sh->off_sel);
            push.slice = sh->slice;
            if (restricted) {
                push.tile_list = tlist;
                push.tile_count = tcount;
            }
            {
                const char *e = getenv("CVVP_SHARD_STAGE"); // development switch; default: stage when owners are peers
                push.stage = e ? (e[0] == '1') : (sh->world > 1);
            }
            const int rc = shard_count_slot(ctx, sh, phase, d_frames + size_t(f0) * frame_stride, nf, frame_stride, push, s);
            if (rc != CVVP_OK)
                return rc;
        }
        return CVVP_OK;
    }
    if (phase == 1 || phase == 3 || phase == 5) {
        OwnerArgs A{};
        A.counts = reinterpret_cast<const uint32_t *>(sh->buf + (phase == 3 ? sh->off_c2 : sh->off_c1));
        A.slice = sh->slice;
        // round 1 shares its receive area with the window records: cslots slots per rank, of which it uses spr
        A.used = uint32_t(phase == 5 ? sh->wsubs : sh->spr);
        A.slots = uint32_t(phase == 3 ? sh->spr : sh->cslots);
        A.world = uint32_t(sh->world) * A.used;
        A.tile_list = tlist;
        A.tile_count = tcount;
        A.src_frames = reinterpret_cast<const uint32_t *>(sh->buf + sh->off_hdr);
        A.percent = uint32_t(sh->percent);
        for (int r = 0; r < sh->world; ++r) {
            A.flag[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + sh->off_flag);
            A.tflag[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + sh->off_tflag);
        }
        A.rank = uint32_t(sh->rank);
        A.nranks = uint32_t(sh->world);
        const size_t first = size_t(sh->rank) * sh->slice;
        A.owned = first >= sh->nelem ? 0u : uint32_t(sh->nelem - first < sh->slice ? sh->nelem - first : sh->slice);
        for (int r = 0; r < sh->world; ++r) {
            A.sel[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + sh->off_sel);
            A.result[r] = sh->peer[r] + sh->off_res;
        }
        if (d_result)
            A.result[sh->rank] = d_result;
        if (A.owned == 0)
            return CVVP_OK;
        const unsigned listed_grid = unsigned(std::min<uint32_t>(sh->ntiles, 8u * uint32_t(ctx->sm_count)));
        if (phase == 1 && restricted)
            shard_pick_listed_kernel<<<listed_grid, 128, 0, s>>>(A);
        else if (phase == 3 && restricted)
            shard_final_listed_kernel<<<listed_grid, 32, 0, s>>>(A);
        else if (phase == 1)
            shard_pick_kernel<<<(A.owned + 255) / 256, 256, 0, s>>>(A);
        else if (phase == 3)
            shard_final_kernel<<<((A.owned + 3) / 4 + 255) / 256, 256, 0, s>>>(A);
        else
            {
                const uint32_t groups = (A.owned + 255u) / 256u; // persistent blocks: six fit an SM
                const uint32_t grid = std::min<uint32_t>(groups, uint32_t(ctx->sm_count) * 6u);
                shard_window_final_kernel<<<grid, 256, 0, s>>>(A);
            }
        CVVP_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches++;
        return CVVP_OK;
    }
    return fail(ctx, CVVP_ERR_INVALID, "median shard: phase must be 0..5 or 10..13");
}

long long median_two_pass_max_frames()
{
    return kSlotFrames * kMaxShardRanks;
}

// Single-GPU median of a stack too long for the on-chip select at full tile width: the sharded job with ONE rank.
// window != 0: one pass of window counting first (phases 4, 5); the two counting rounds follow on the stream
// restricted to the tiles that hold an undecided element (phases 10..13; the tile list is built on the device, so
// with nothing undecided they return at once) -- no host round trip, the call stays asynchronous.  window == 0: the
// two counting passes over the whole image only.  Either way two passes
// over the frames in chunks of <= 1024 at 128-byte tiles beat one pass at the 32- or 16-byte tiles the on-chip
// select would need beyond 2048 frames (DESIGN.md section 3).
int median_long_stack(cvvp_ctx *ctx, const uint8_t *d_frames, long long nframes, size_t nelem, size_t frame_stride,
                      uint8_t *d_out, int percent, cudaStream_t stream, int window)
{
    const int spr = int((nframes + kSlotFrames - 1) / kSlotFrames);
    const int wsubs = window ? int((nframes + kChunkFrames - 1) / kChunkFrames) : 1;
    if (ctx->big && (ctx->big->nelem != nelem || ctx->big->spr < spr || ctx->big->wsubs < wsubs))
        shard_destroy(ctx, ctx->big);
    if (!ctx->big) {
        const int rc = shard_create(ctx, nelem, 0, 1, spr, wsubs, &ctx->big);
        if (rc != CVVP_OK)
            return rc;
    }
    ctx->big->percent = percent; // the internal job is reused across calls: it takes each call's percentile
    if ((reinterpret_cast<uintptr_t>(d_out) & 3u) != 0) // the owner kernels store four result bytes at a time
        return fail(ctx, CVVP_ERR_INVALID, "median: the result pointer of a stack that takes the counting path (more than 1024 frames) must be 4-byte aligned");
    if (window) {
        for (int phase = 4; phase <= 5; ++phase) {
            const int rc = shard_phase(ctx, ctx->big, phase, d_frames, nframes, frame_stride, d_out, stream);
            if (rc != CVVP_OK)
                return rc;
        }
    }
    for (int phase = 0; phase < 4; ++phase) {
        const int rc = shard_phase(ctx, ctx->big, phase + (window ? 10 : 0), d_frames, nframes, frame_stride, d_out, stream);
        if (rc != CVVP_OK)
            return rc;
    }
    return CVVP_OK;
}
} // namespace cvvp

using namespace cvvp;

extern "C" {

int cvvp_median_shard_begin(cvvp_ctx *ctx, size_t nelem, int rank, int world)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: a sharded job is already open on this context");
    if (nelem == 0 || nelem >= (1ull << 31))
        return fail(ctx, CVVP_ERR_INVALID, "median shard: nelem must be in [1, 2^31)");
    if (world < 1 || world > kMaxShardRanks || rank < 0 || rank >= world)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: rank %d / world %d out of range (world <= %d)", rank, world,
                    kMaxShardRanks);
    DeviceGuard guard(ctx->device);
    return shard_create(ctx, nelem, rank, world, 1, 1, &ctx->shard);
}

int cvvp_median_shard_begin_frames(cvvp_ctx *ctx, size_t nelem, int rank, int world, long long max_rank_frames)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: a sharded job is already open on this context");
    if (nelem == 0 || nelem >= (1ull << 31))
        return fail(ctx, CVVP_ERR_INVALID, "median shard: nelem must be in [1, 2^31)");
    if (world < 1 || world > kMaxShardRanks || rank < 0 || rank >= world)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: rank %d / world %d out of range (world <= %d)", rank, world,
                    kMaxShardRanks);
    if (max_rank_frames < 1)
        max_rank_frames = 1;
    const long long spr = (max_rank_frames + kSlotFrames - 1) / kSlotFrames;
    if (spr * world > kMaxShardRanks)
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "median shard: %lld frames per rank on %d ranks exceed %d count slots",
                    max_rank_frames, world, kMaxShardRanks);
    DeviceGuard guard(ctx->device);
    return shard_create(ctx, nelem, rank, world, int(spr), int((max_rank_frames + kChunkFrames - 1) / kChunkFrames), &ctx->shard);
}

int cvvp_median_shard_barrier(cvvp_ctx *ctx, void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    MedianShard *sh = ctx->shard;
    if (!sh)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    if (!all_peers_known(sh))
        return fail(ctx, CVVP_ERR_STATE, "median shard: not every peer buffer is mapped (import / attach all ranks first)");
    for (int r = 0; r < sh->world; ++r)
        if (sh->attached[r])
            return fail(ctx, CVVP_ERR_UNSUPPORTED,
                        "median shard: the device barrier is for ranks in processes of their own, one GPU each; ranks attached "
                        "inside one process synchronize their contexts instead");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    BarrierArgs B{};
    for (int r = 0; r < sh->world; ++r)
        B.bar[r] = reinterpret_cast<uint32_t *>(sh->peer[r] + sh->off_bar);
    B.rank = uint32_t(sh->rank);
    B.world = uint32_t(sh->world);
    B.epoch = ++sh->epoch;
    shard_barrier_kernel<<<1, 32, 0, s>>>(B);
    CVVP_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches++;
    return CVVP_OK;
}

int cvvp_median_shard_unresolved(cvvp_ctx *ctx, void *stream, long long *out_elements)
{
    if (!ctx || !out_elements)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: null argument");
    if (!ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    uint32_t v = 0;
    CVVP_CUDA_OK(ctx, cudaMemcpyAsync(&v, ctx->shard->buf + ctx->shard->off_flag, sizeof(v), cudaMemcpyDeviceToHost, s));
    CVVP_CUDA_OK(ctx, cudaStreamSynchronize(s));
    *out_elements = (long long)v;
    return CVVP_OK;
}

int cvvp_median_shard_export(cvvp_ctx *ctx, void *handle_out)
{
    if (!ctx || !handle_out)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: null argument");
    if (!ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    static_assert(sizeof(cudaIpcMemHandle_t) == CVVP_IPC_HANDLE_BYTES, "handle size is part of the ABI");
    DeviceGuard guard(ctx->device);
    cudaIpcMemHandle_t h;
    CVVP_CUDA_OK(ctx, cudaIpcGetMemHandle(&h, ctx->shard->buf));
    std::memcpy(handle_out, &h, sizeof(h));
    return CVVP_OK;
}

int cvvp_median_shard_import(cvvp_ctx *ctx, int peer, const void *handle)
{
    if (!ctx || !handle)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: null argument");
    MedianShard *sh = ctx->shard;
    if (!sh)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    if (peer < 0 || peer >= sh->world || peer == sh->rank)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: bad peer rank %d", peer);
    if (sh->peer[peer])
        return fail(ctx, CVVP_ERR_STATE, "median shard: peer %d is already mapped", peer);
    DeviceGuard guard(ctx->device);
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    CVVP_CUDA_OK(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    sh->peer[peer] = static_cast<uint8_t *>(p);
    sh->ipc_opened[peer] = true;
    return CVVP_OK;
}

int cvvp_median_shard_attach(cvvp_ctx *ctx, int peer, cvvp_ctx *peer_ctx)
{
    if (!ctx || !peer_ctx)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: null argument");
    MedianShard *sh = ctx->shard, *ps = peer_ctx->shard;
    if (!sh || !ps)
        return fail(ctx, CVVP_ERR_STATE, "median shard: both contexts need an open sharded job");
    if (peer < 0 || peer >= sh->world || peer == sh->rank || ps->rank != peer || ps->world != sh->world ||
        ps->nelem != sh->nelem)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: peer context does not describe rank %d of the same job", peer);
    if (sh->peer[peer])
        return fail(ctx, CVVP_ERR_STATE, "median shard: peer %d is already mapped", peer);
    if (peer_ctx->device != ctx->device) {
        DeviceGuard guard(ctx->device);
        int can = 0;
        CVVP_CUDA_OK(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, peer_ctx->device));
        if (!can)
            return fail(ctx, CVVP_ERR_UNSUPPORTED, "median shard: device %d cannot access device %d", ctx->device,
                        peer_ctx->device);
        const cudaError_t e = cudaDeviceEnablePeerAccess(peer_ctx->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            return fail(ctx, CVVP_ERR_CUDA, "cudaDeviceEnablePeerAccess failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
    }
    sh->peer[peer] = ps->buf;
    sh->attached[peer] = true;
    return CVVP_OK;
}

int cvvp_median_shard_phase(cvvp_ctx *ctx, int phase, const uint8_t *d_frames, long long nframes, size_t frame_stride,
                            void *stream)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    if (!ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->compute;
    return shard_phase(ctx, ctx->shard, phase, d_frames, nframes, frame_stride, nullptr, s);
}

int cvvp_median_shard_result(cvvp_ctx *ctx, const uint8_t **d_result)
{
    if (!ctx || !d_result)
        return fail(ctx, CVVP_ERR_INVALID, "median shard: null argument");
    if (!ctx->shard)
        return fail(ctx, CVVP_ERR_STATE, "median shard: no sharded job is open");
    *d_result = ctx->shard->buf + ctx->shard->off_res;
    return CVVP_OK;
}

int cvvp_median_shard_end(cvvp_ctx *ctx)
{
    if (!ctx)
        return fail(nullptr, CVVP_ERR_INVALID, "null context");
    DeviceGuard guard(ctx->device);
    shard_destroy(ctx, ctx->shard);
    return CVVP_OK;
}

} // extern "C"
