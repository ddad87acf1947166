// Fused per-frame highlight kernel for sm_100a -- the product path of the highlight stage.
// Replaces HighlightObjectsAlgo::HighlightObjects (/root/reference/Sources/ProcessorAlgos/highlight_objects_algo.cpp:17-221);
// semantics and reference citations per step: highlight.cu's header and oracle/highlight_model.py.
//
// ONE kernel launch per batch.  A persistent CTA pulls frames from a queue and takes each frame through every step of
// the reference function with block barriers in between, so a frame costs one read of its bytes and one write of its
// mask in HBM (the algorithmic traffic) plus L2-resident scratch:
//
//   bits     frame, background -> three bit images  A = d > th, U = d > hi, L = d > lo   (d = saturating bg - frame)
//            32 pixels per thread from 128-bit loads; the byte compares are SWAR (four pixels per instruction); the
//            object polarity (cvvp_highlight_set_polarity) picks d = bg - frame, frame - bg or |frame - bg| per frame
//   open     erode + dilate on bit rows: one funnel shift + AND/OR per structuring-element tap per 32 pixels
//   label    the nodes of the union-find are the horizontal RUNS of equal bits (a few thousand per 1080p frame, not two
//            million pixels), numbered in raster order by a two-pass block scan, so "smallest id of a component" is
//            still its raster-first pixel; foreground 8-/4-connected, background 4-connected, optional FRAME node
//   hyst     seeds = first runs of the external hi components; marked lo regions are scattered back as bits
//   rso      contour statistics from run geometry: run ends give the horizontal cracks and the convex corners, overlaps
//            with the runs of the neighbouring rows give the vertical cracks; the polygon-area rule, the edge rule and
//            the even-odd nesting parity of the single filled drawContours call decide which bits are cleared
//   fill     background runs that are not connected to the seed corner are set (in place)
//   expand   (A | B) -> 0/255 bytes, 128-bit stores
//
// Scratch is per RESIDENT CTA (a "slot"), not per frame of the batch: 4 bit images and 8 run arrays.  Run-level arrays
// that are touched by atomics are only ever read with ld.global.cg (L2), so a stale L1 line can never be observed.
//
// run record: xinfo[id] = x_start | row << 16 | value << 31   (W <= 65535, H <= 32767; larger frames use highlight.cu)
#include "highlight_state.hpp"
#include "pool.hpp"

#include <climits>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace cvvp
{
namespace
{
// The file is compiled twice (highlight_fused_small.cu includes it with CVVP_HLF_SMALL defined): the same code with
//   1024 threads, 192 KB of dynamic shared memory, one CTA per SM   -- large frames (1080p: 553 us per frame and CTA);
//    256 threads,  48 KB,                          four CTAs per SM -- small frames (512x256), where a 1024-thread CTA
//                                                                      spends its time in block barriers: four frames per
//                                                                      SM overlap each other's barrier and latency stalls.
#ifdef CVVP_HLF_SMALL
#define HLF(name) name##_small
constexpr int NT = 256;
constexpr int kCtasPerSm = 4;
constexpr size_t kDynSmemBytes = 48 * 1024;
#else
#define HLF(name) name##_large
constexpr int NT = 1024; // threads per CTA (one CTA per SM)
constexpr int kCtasPerSm = 1;
constexpr size_t kDynSmemBytes = 192 * 1024; // per CTA; one CTA per SM
#endif
constexpr int NW = NT / 32;
constexpr int kImages = 4;    // A, U (later B), L, Tm
constexpr int kRunArrays = 8; // xinfo0, parent0, xinfo1, parent1, link, st_s, st_e, st_x
constexpr uint32_t kNoLabel = 0xFFFFFFFFu;
constexpr uint32_t kH = 0x80808080u;

struct ThreshSpec {
    uint32_t t4;       // threshold replicated into four bytes (clamped to 0..254)
    uint32_t force_or; // all-ones when the threshold is negative (every pixel passes)
    uint32_t force_and; // zero when the threshold is >= 255 (no pixel passes)
};

// Separable form of the structuring element: its tap rows grouped by their set of column offsets ("patterns").  A
// pattern's horizontal erosion / dilation of a tile row is computed once and shared by every tap row that uses it, so
// the vertical step is a plain AND / OR of words.  (The reference's usual ellipse has two patterns: one tap, and a full
// row.)  Used when there are at most kMaxPat patterns and |dx| <= 31; other elements take the generic tap loop.
constexpr int kMaxPat = 3;
constexpr int kMaxPlanRows = 64;
constexpr int kMaxPlanTaps = 96;

struct MorphPlan {
    int sep;    // 1 = separable path usable
    int npat;   // distinct patterns
    int nrows;  // tap rows
    signed char row_dy[kMaxPlanRows];
    signed char row_pat[kMaxPlanRows];
    signed char pat_ident[kMaxPat];     // pattern == {0}: the tile itself
    unsigned char pat_start[kMaxPat + 1]; // pattern p's offsets are dx[pat_start[p] .. pat_start[p + 1])
    signed char dx[kMaxPlanTaps];
};

struct FusedArgs {
    const uint8_t *frames;
    size_t frame_stride;
    const uint8_t *bg;
    size_t bg_stride; // frame f's background at bg + f * bg_stride (0: one background for every frame)
    uint8_t *out;
    size_t out_stride;
    const int *th_a; // per-frame threshold of branch A (Otsu), or nullptr -> th
    int th, lo, hi, min_th, min_hyst;
    const short2 *offs;
    int noffs;
    int W, H, WW, WWp;
    int wwp_shift;    // log2(WWp) when WWp is a power of two, else -1
    uint32_t nwords;  // H * WWp
    uint32_t cap;     // run-array capacity per slot
    size_t run_words; // run scratch per slot: kRunArrays arrays of cap words + cap / 32 flag words
    uint32_t rstride; // rowoff stride
    uint32_t *bits;
    uint32_t *runs;
    uint32_t *rowoff;
    unsigned *queue; // [0] next frame, [1] CTAs finished
    unsigned nframes;
    int fast_io; // W % 32 == 0 and 16-byte aligned pointers / strides
    int polarity; // CVVP_POLARITY_*: which difference image d the bits phase computes
    uint32_t smem_words; // dynamic shared memory of the CTA, in 32-bit words
    // opening in shared-memory row bands (0 rows = structuring element too large: global-memory taps instead)
    int band_rows, dy_min, dy_max, pad_words;
    int ct_elem; // 0 = run-time plan; 1.. = the structuring element has a compile-time instantiation (open_bands_ct)
    MorphPlan plan;
    // optional component output of the final masks (cvvp_highlight_device_cc): nullptr = off
    cvvp_component *comps; // [frame][max_comps] records of rec_bytes each
    int *ncomps;           // [frame]
    int max_comps;
    int stats;             // 1: the records are cvvp_component_stats (cvvp_highlight_set_component_stats)
    uint32_t rec_bytes;    // sizeof(cvvp_component) or sizeof(cvvp_component_stats)
    int32_t *labels;       // [frame][labels_stride] or nullptr
    size_t labels_stride;
    unsigned long long *prof; // per-phase nanoseconds summed over frames (CVVP_HL_PROF=1), or nullptr
    int debug_stage; // 0 = off; k > 0: write the bit image of intermediate stage k instead of the result (tools/)
};

struct RunSet {
    uint32_t *xinfo;
    uint32_t *parent;
    uint32_t *rowoff; // [H + 1]; rowoff[H] = T
    uint32_t *fbits;  // FRAME flags of the set's roots (one bit per run id)
};

enum ProfPhase {
    kPBits, kPErodeA, kPDilateA, kPExtract, kPMerge, kPFlatten, kPRso, kPFill, kPHyst, kPErodeB, kPDilateB, kPExpand,
    kPCountRuns, kPHook, kPRuns, kPFrames, kPCount
};

struct Shared {
    unsigned long long prof_last;
    unsigned frame;
    uint32_t wsum[NW];
    uint32_t wbase[NW + 1]; // exclusive prefix of wsum (run id of every warp's first run)
    uint32_t T[2];
    int white[2];
    int changed; // remove-small-objects cleared at least one pixel of the current image
};

// ------------------------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// developer aid: thread 0 charges the time since the previous tick to `phase`
__device__ __forceinline__ void prof_tick(const unsigned long long *enabled, unsigned long long *acc, Shared &sh, int phase)
{
    if (enabled && threadIdx.x == 0) {
        const unsigned long long t = global_ns();
        if (phase >= 0)
            atomicAdd(acc + phase, t - sh.prof_last);
        sh.prof_last = t;
    }
}

__device__ __forceinline__ uint32_t ld(const uint32_t *p) { return __ldcg(p); }
__device__ __forceinline__ int ld(const int *p) { return __ldcg(p); }
__device__ __forceinline__ void st(uint32_t *p, uint32_t v) { __stcg(p, v); }
__device__ __forceinline__ void st(int *p, int v) { __stcg(p, v); }

__device__ __forceinline__ uint32_t run_x(uint32_t xi) { return xi & 0xFFFFu; }
__device__ __forceinline__ uint32_t run_y(uint32_t xi) { return (xi >> 16) & 0x7FFFu; }
__device__ __forceinline__ uint32_t run_v(uint32_t xi) { return xi >> 31; }

__device__ __forceinline__ uint32_t valid_mask(const FusedArgs &P, int wx)
{
    const int rem = P.W - 32 * wx;
    return rem >= 32 ? 0xFFFFFFFFu : (rem <= 0 ? 0u : (0xFFFFFFFFu >> (32 - rem)));
}

__device__ __forceinline__ void split(const FusedArgs &P, uint32_t i, int &y, int &wx)
{
    if (P.wwp_shift >= 0) {
        y = int(i >> P.wwp_shift);
        wx = int(i & uint32_t(P.WWp - 1));
    } else {
        y = int(i / uint32_t(P.WWp));
        wx = int(i - uint32_t(y) * uint32_t(P.WWp));
    }
}

__device__ __forceinline__ uint32_t range_mask(int lo, int hi) // bits lo..hi (0 <= lo <= hi <= 31)
{
    return (0xFFFFFFFFu >> (31 - hi)) & (0xFFFFFFFFu << lo);
}

// The parent array of the union-find lives in shared memory while a frame's run count fits (the usual case: a few
// thousand runs), else in the slot's global scratch.  Labels only ever decrease, so a stale read is harmless: every
// link is re-validated by the atomicMin that makes it.
template <bool SM>
struct Par {
    uint32_t *p;
    __device__ __forceinline__ uint32_t get(uint32_t i) const
    {
        return SM ? *reinterpret_cast<volatile uint32_t *>(p + i) : __ldcg(p + i);
    }
    __device__ __forceinline__ void set(uint32_t i, uint32_t v) const
    {
        if (SM)
            *reinterpret_cast<volatile uint32_t *>(p + i) = v;
        else
            __stcg(p + i, v);
    }
    __device__ __forceinline__ uint32_t amin(uint32_t i, uint32_t v) const { return atomicMin(p + i, v); }
};

// find with path halving: every second node of the walked chain is re-linked to its grandparent (atomicMin keeps the
// "labels only decrease" invariant under concurrent unions), so repeated walks of the long vertical chains a frame's
// background produces stay short
template <bool SM>
__device__ __forceinline__ uint32_t uf_find(const Par<SM> &lab, uint32_t x)
{
    for (;;) {
        const uint32_t p = lab.get(x);
        if (p == x)
            return x;
        const uint32_t gp = lab.get(p);
        if (gp == p)
            return p;
        lab.amin(x, gp);
        x = gp;
    }
}

template <bool SM>
__device__ __forceinline__ void uf_union(const Par<SM> &lab, uint32_t a, uint32_t b)
{
    bool done;
    do {
        a = uf_find(lab, a);
        b = uf_find(lab, b);
        if (a < b) {
            const uint32_t old = lab.amin(b, a);
            done = (old == b);
            b = old;
        } else if (b < a) {
            const uint32_t old = lab.amin(a, b);
            done = (old == a);
            a = old;
        } else {
            done = true;
        }
    } while (!done);
}

__device__ __forceinline__ void clear_range(uint32_t *row, int x0, int x1)
{
    for (int w = x0 >> 5; w <= (x1 >> 5); ++w)
        atomicAnd(&row[w], ~range_mask(max(x0, 32 * w) - 32 * w, min(x1, 32 * w + 31) - 32 * w));
}

__device__ __forceinline__ void set_range(uint32_t *row, int x0, int x1)
{
    for (int w = x0 >> 5; w <= (x1 >> 5); ++w)
        atomicOr(&row[w], range_mask(max(x0, 32 * w) - 32 * w, min(x1, 32 * w + 31) - 32 * w));
}

// ------------------------------------------------------------------------------------------------------------------
// bits: d = max(bg - frame, 0) (or another polarity); three thresholds -> three bit images
//                                                             (highlight_objects_algo.cpp:27-30, :100, :117-122)
// ------------------------------------------------------------------------------------------------------------------
// per-byte saturating x - y (SWAR: no carries between bytes)
__device__ __forceinline__ uint32_t sub_sat_u8x4(uint32_t x, uint32_t y)
{
    const uint32_t t = (x | kH) - (y & ~kH);
    const uint32_t ge = (x & ~y) | (~(x ^ y) & t); // byte MSB: x >= y
    const uint32_t diff = t ^ ((x ^ ~y) & kH);
    uint32_t m; // byte MSB -> 0xFF / 0x00 (prmt's sign-replicate mode; __byte_perm masks that selector bit away)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(ge), "r"(0u), "r"(0xba98u));
    return diff & m;
}

// four-bit mask of d > t per byte; d7 = d & 0x7f7f7f7f, th = t4 | 0x80808080
__device__ __forceinline__ uint32_t gt_nibble_top(uint32_t d, uint32_t d7, uint32_t t4, uint32_t th)
{
    const uint32_t t = th - d7;
    const uint32_t ge = (t4 & ~d) | (~(t4 ^ d) & t); // byte MSB: t4 >= d
    return (~ge & kH) * 0x00204081u;                 // bits 28..31 = the four MSBs (lower bits: junk)
}

__device__ __forceinline__ ThreshSpec make_thresh(int t)
{
    ThreshSpec s;
    const int c = t < 0 ? 0 : (t > 254 ? 254 : t);
    s.t4 = uint32_t(c) * 0x01010101u;
    s.force_or = t < 0 ? 0xFFFFFFFFu : 0u;
    s.force_and = t >= 255 ? 0u : 0xFFFFFFFFu;
    return s;
}

// d of four pixels in polarity POL (hl_diff): bg - frame, frame - bg (saturating), or |frame - bg| (VABSDIFF4.U8)
template <int POL>
__device__ __forceinline__ uint32_t diff_u8x4(uint32_t fr, uint32_t bg)
{
    if (POL == CVVP_POLARITY_DARK)
        return sub_sat_u8x4(bg, fr);
    if (POL == CVVP_POLARITY_BRIGHT)
        return sub_sat_u8x4(fr, bg);
    return __vabsdiffu4(fr, bg);
}

// tm: the smallest of the three thresholds (ThreshSpec of it), or force_or != 0 when one of them is negative.  Most
// 32-pixel groups of a frame have no pixel above even the smallest threshold: one compare per four pixels settles all
// three bit words.
template <int POL>
__device__ __forceinline__ void bits_of_32(const uint4 &f0, const uint4 &f1, const uint4 &b0, const uint4 &b1,
                                           const ThreshSpec &ta, const ThreshSpec &tu, const ThreshSpec &tl,
                                           const ThreshSpec &tm, uint32_t &wa, uint32_t &wu, uint32_t &wl)
{
    const uint32_t fr[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
    const uint32_t bk[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    const uint32_t tha = ta.t4 | kH, thu = tu.t4 | kH, thl = tl.t4 | kH, thm = tm.t4 | kH;
    uint32_t d[8];
    uint32_t any = tm.force_or;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        d[k] = diff_u8x4<POL>(fr[k], bk[k]);
        const uint32_t t = thm - (d[k] & ~kH);
        any |= ~((tm.t4 & ~d[k]) | (~(tm.t4 ^ d[k]) & t)) & kH; // byte MSB: d > smallest threshold
    }
    wa = wu = wl = 0;
    if (any != 0u) {
#pragma unroll
        for (int k = 7; k >= 0; --k) { // last group first: each funnel shift pushes the word up by one nibble
            const uint32_t d7 = d[k] & ~kH;
            wa = __funnelshift_l(gt_nibble_top(d[k], d7, ta.t4, tha), wa, 4); // (wa << 4) | top nibble: one SHF
            wu = __funnelshift_l(gt_nibble_top(d[k], d7, tu.t4, thu), wu, 4);
            wl = __funnelshift_l(gt_nibble_top(d[k], d7, tl.t4, thl), wl, 4);
        }
    }
    wa = (wa | ta.force_or) & ta.force_and;
    wu = (wu | tu.force_or) & tu.force_and;
    wl = (wl | tl.force_or) & tl.force_and;
}

// ThreshSpec of the smallest threshold that can still let a pixel pass (see bits_of_32)
__device__ __forceinline__ ThreshSpec min_thresh(int a, int b, int c)
{
    if (a < 0 || b < 0 || c < 0) {
        ThreshSpec s = make_thresh(0);
        s.force_or = 0xFFFFFFFFu; // a negative threshold passes every pixel: no shortcut
        return s;
    }
    return make_thresh(min(a, min(b, c)));
}

// the bits phase in polarity POL; bits_phase picks the instantiation once per frame (P.polarity is uniform)
template <int POL>
__device__ __forceinline__ void bits_phase_pol(const FusedArgs &P, unsigned f, uint32_t *A, uint32_t *U, uint32_t *L)
{
    const int tid = threadIdx.x;
    const uint8_t *fr = P.frames + size_t(f) * P.frame_stride;
    const uint8_t *bg = P.bg + size_t(f) * P.bg_stride;
    const int th_a = P.th_a ? __ldg(P.th_a + f) : P.th;
    if (P.fast_io) {
        const ThreshSpec ta = make_thresh(th_a), tu = make_thresh(P.hi), tl = make_thresh(P.lo);
        const ThreshSpec tm = min_thresh(th_a, P.hi, P.lo);
        // two words per thread per iteration: eight 128-bit loads in flight
        for (uint32_t i0 = tid; i0 < P.nwords; i0 += 2 * NT) {
            const uint32_t i1 = i0 + NT;
            int y0, wx0, y1 = 0, wx1 = P.WW;
            split(P, i0, y0, wx0);
            if (i1 < P.nwords)
                split(P, i1, y1, wx1);
            const bool v0 = wx0 < P.WW, v1 = wx1 < P.WW;
            uint4 fa0, fa1, ba0, ba1, fb0, fb1, bb0, bb1;
            fa0 = fa1 = ba0 = ba1 = fb0 = fb1 = bb0 = bb1 = make_uint4(0, 0, 0, 0);
            if (v0) {
                const size_t o = size_t(y0) * P.W + 32u * wx0;
                fa0 = __ldcs(reinterpret_cast<const uint4 *>(fr + o)); // frames are read once: streaming
                fa1 = __ldcs(reinterpret_cast<const uint4 *>(fr + o + 16));
                ba0 = __ldg(reinterpret_cast<const uint4 *>(bg + o));
                ba1 = __ldg(reinterpret_cast<const uint4 *>(bg + o + 16));
            }
            if (v1) {
                const size_t o = size_t(y1) * P.W + 32u * wx1;
                fb0 = __ldcs(reinterpret_cast<const uint4 *>(fr + o));
                fb1 = __ldcs(reinterpret_cast<const uint4 *>(fr + o + 16));
                bb0 = __ldg(reinterpret_cast<const uint4 *>(bg + o));
                bb1 = __ldg(reinterpret_cast<const uint4 *>(bg + o + 16));
            }
            uint32_t wa = 0, wu = 0, wl = 0;
            if (v0)
                bits_of_32<POL>(fa0, fa1, ba0, ba1, ta, tu, tl, tm, wa, wu, wl);
            A[i0] = wa;
            U[i0] = wu;
            L[i0] = wl;
            if (i1 < P.nwords) {
                wa = wu = wl = 0;
                if (v1)
                    bits_of_32<POL>(fb0, fb1, bb0, bb1, ta, tu, tl, tm, wa, wu, wl);
                A[i1] = wa;
                U[i1] = wu;
                L[i1] = wl;
            }
        }
    } else {
        for (uint32_t i = tid; i < P.nwords; i += NT) {
            int y, wx;
            split(P, i, y, wx);
            uint32_t wa = 0, wu = 0, wl = 0;
            if (wx < P.WW) {
                const size_t o = size_t(y) * P.W;
                const int x1 = min(32 * wx + 32, P.W);
                for (int x = 32 * wx; x < x1; ++x) {
                    const int d = hl_diff(__ldg(bg + o + x), __ldg(fr + o + x), POL);
                    const uint32_t b = 1u << (x & 31);
                    if (d > th_a)
                        wa |= b;
                    if (d > P.hi)
                        wu |= b;
                    if (d > P.lo)
                        wl |= b;
                }
            }
            A[i] = wa;
            U[i] = wu;
            L[i] = wl;
        }
    }
}

__device__ void bits_phase(const FusedArgs &P, unsigned f, uint32_t *A, uint32_t *U, uint32_t *L)
{
    if (P.polarity == CVVP_POLARITY_DARK)
        bits_phase_pol<CVVP_POLARITY_DARK>(P, f, A, U, L);
    else if (P.polarity == CVVP_POLARITY_BRIGHT)
        bits_phase_pol<CVVP_POLARITY_BRIGHT>(P, f, A, U, L);
    else
        bits_phase_pol<CVVP_POLARITY_BOTH>(P, f, A, U, L);
}

// ------------------------------------------------------------------------------------------------------------------
// opening on bit rows (cv::morphologyEx(MORPH_OPEN) :39, :61): taps sorted by (dy, dx); out-of-image samples never win
// ------------------------------------------------------------------------------------------------------------------
template <bool ERODE, bool CG>
__device__ void morph_phase(const FusedArgs &P, const uint32_t *src, uint32_t *dst)
{
    const uint32_t fill = ERODE ? 0xFFFFFFFFu : 0u;
    for (uint32_t i = threadIdx.x; i < P.nwords; i += NT) {
        int y, wx;
        split(P, i, y, wx);
        uint32_t res = 0;
        if (wx < P.WW) {
            auto word = [&](const uint32_t *row, int w) -> uint32_t {
                if (w < 0 || w >= P.WW)
                    return fill;
                uint32_t v = CG ? __ldcg(row + w) : row[w];
                if (ERODE)
                    v |= ~valid_mask(P, w);
                return v;
            };
            uint32_t acc = fill;
            int cur_dy = INT_MIN, cur_q = INT_MIN;
            const uint32_t *row = nullptr;
            uint32_t w0 = fill, w1 = fill;
            for (int k = 0; k < P.noffs; ++k) {
                const short2 o = __ldg(&P.offs[k]);
                if (o.y != cur_dy) {
                    cur_dy = o.y;
                    cur_q = INT_MIN;
                    const int yy = y + o.y;
                    row = (yy >= 0 && yy < P.H) ? src + size_t(yy) * P.WWp : nullptr;
                }
                if (!row)
                    continue;
                const int q = int(o.x) >> 5, r = int(o.x) & 31; // floor division: columns 32*wx + dx .. + 31
                if (q != cur_q) {
                    cur_q = q;
                    w0 = word(row, wx + q);
                    w1 = word(row, wx + q + 1);
                }
                const uint32_t v = r ? __funnelshift_r(w0, w1, r) : w0;
                acc = ERODE ? (acc & v) : (acc | v);
                if (ERODE && acc == 0)
                    break;
            }
            res = acc & valid_mask(P, wx);
        }
        dst[i] = res;
    }
}

// Opening through shared-memory row bands: a band of source rows (plus the halo both steps need) is staged once with
// 128-bit loads, eroded into a second tile and dilated from there straight into `dst` (a different image), so the
// image makes one trip through L2 instead of four and every tap is a shared-memory access.  Tile rows carry
// kPadWords words on both sides so that no tap needs a horizontal bounds test; out-of-image samples are the neutral
// element of each step (all-ones for the erosion's AND, zeros for the dilation's OR).
constexpr int kPadWords = 4; // covers |dx| <= 127 (structuring elements up to 255 wide)

template <bool ERODE>
__device__ __forceinline__ uint32_t morph_word(const short2 *offs, int noffs, const uint32_t *tile, int pitch, int trow_base,
                                               int wx)
{
    uint32_t acc = ERODE ? 0xFFFFFFFFu : 0u;
    int cur_dy = INT_MIN, cur_q = INT_MIN;
    const uint32_t *rowp = tile;
    uint32_t w0 = 0, w1 = 0;
    for (int k = 0; k < noffs; ++k) {
        const short2 o = offs[k];
        if (o.y != cur_dy) {
            cur_dy = o.y;
            cur_q = INT_MIN;
            rowp = tile + (trow_base + o.y) * pitch + kPadWords + wx;
        }
        const int q = int(o.x) >> 5, r = int(o.x) & 31; // floor division: columns 32*wx + dx .. + 31
        if (q != cur_q) {
            cur_q = q;
            w0 = rowp[q];
            w1 = rowp[q + 1];
        }
        const uint32_t v = r ? __funnelshift_r(w0, w1, r) : w0;
        acc = ERODE ? (acc & v) : (acc | v);
        if (ERODE && acc == 0)
            break;
    }
    return acc;
}

__device__ void open_bands(const FusedArgs &P, const short2 *offs, const uint32_t *src, uint32_t *dst, uint32_t *smem)
{
    const int tid = threadIdx.x;
    const int pitch = P.WWp + 2 * kPadWords;
    const int span = P.dy_max - P.dy_min;
    const int BH = P.band_rows;
    const int s_rows_max = BH + 2 * span, e_rows_max = BH + span;
    uint32_t *S = smem;
    uint32_t *E = smem + size_t(s_rows_max) * pitch;
    const int qpr = P.WWp >> 2; // quads per row
    // side pads: written once per call (the tiles alias the union-find's parent array between calls)
    for (int i = tid; i < (s_rows_max + e_rows_max) * 2 * kPadWords; i += NT) {
        const int row = i / (2 * kPadWords), c = i - row * (2 * kPadWords);
        const int col = c < kPadWords ? c : P.WWp + c;
        if (row < s_rows_max)
            S[row * pitch + col] = 0xFFFFFFFFu;
        else
            E[(row - s_rows_max) * pitch + col] = 0u;
    }
    for (int y0 = 0; y0 < P.H; y0 += BH) {
        const int y1 = min(y0 + BH, P.H);
        const int e0 = y0 + P.dy_min, e1 = y1 + P.dy_max; // eroded rows the band's dilation reads
        const int s0 = e0 + P.dy_min, s1 = e1 + P.dy_max; // source rows their erosion reads
        const int srows = s1 - s0, erows = e1 - e0;
        // stage the source rows; invalid columns and out-of-image rows read as set
        for (int i = tid; i < srows * qpr; i += NT) {
            int tr, qc;
            if (P.wwp_shift >= 0) {
                tr = i >> (P.wwp_shift - 2);
                qc = i & (qpr - 1);
            } else {
                tr = i / qpr;
                qc = i - tr * qpr;
            }
            const int r = s0 + tr;
            uint4 v = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            if (r >= 0 && r < P.H) {
                v = __ldcg(reinterpret_cast<const uint4 *>(src + size_t(r) * P.WWp) + qc);
                v.x |= ~valid_mask(P, 4 * qc);
                v.y |= ~valid_mask(P, 4 * qc + 1);
                v.z |= ~valid_mask(P, 4 * qc + 2);
                v.w |= ~valid_mask(P, 4 * qc + 3);
            }
            *reinterpret_cast<uint4 *>(S + tr * pitch + kPadWords + 4 * qc) = v;
        }
        __syncthreads();
        // erode: tile row te <-> image row e0 + te; its taps read S rows te + dy - dy_min
        for (int i = tid; i < erows * P.WWp; i += NT) {
            int te, wx;
            split(P, uint32_t(i), te, wx);
            const int e = e0 + te;
            uint32_t v = 0;
            if (e >= 0 && e < P.H && wx < P.WW)
                v = morph_word<true>(offs, P.noffs, S, pitch, te - P.dy_min, wx) & valid_mask(P, wx);
            E[te * pitch + kPadWords + wx] = v;
        }
        __syncthreads();
        // dilate: output row y0 + ty reads E rows ty + dy - dy_min
        for (int i = tid; i < (y1 - y0) * P.WWp; i += NT) {
            int ty, wx;
            split(P, uint32_t(i), ty, wx);
            uint32_t v = 0;
            if (wx < P.WW)
                v = morph_word<false>(offs, P.noffs, E, pitch, ty - P.dy_min, wx) & valid_mask(P, wx);
            dst[size_t(y0 + ty) * P.WWp + wx] = v;
        }
        __syncthreads();
    }
}

// ---- separable opening (MorphPlan) -----------------------------------------------------------------------------------
// Thread mapping of every step: a thread keeps ONE quad column (qc = tid % quads-per-row) and walks rows r0, r0 + rstep,
// ... of the band, so the row / column split, the column masks and the tile addresses are loop invariants.

// horizontal step of one pattern over `rows` tile rows: dst row = AND / OR over the pattern's dx of (src row shifted)
template <bool ERODE>
__device__ __forceinline__ void morph_rows_h(const FusedArgs &P, int pat, const uint32_t *src, uint32_t *dst, int rows, int pitch,
                                             int qc, int r0, int rstep)
{
    const int k0 = P.plan.pat_start[pat], k1 = P.plan.pat_start[pat + 1];
    const int off = kPadWords + 4 * qc;
    for (int tr = r0; tr < rows; tr += rstep) {
        const uint32_t *row = src + tr * pitch + off;
        const uint4 c = *reinterpret_cast<const uint4 *>(row);
        const uint32_t w[6] = {row[-1], c.x, c.y, c.z, c.w, row[4]};
        uint4 o = make_uint4(0, 0, 0, 0);
        if ((w[0] | w[1] | w[2] | w[3] | w[4] | w[5]) != 0) { // an all-clear neighbourhood stays clear in both steps
            uint32_t acc[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                acc[j] = ERODE ? 0xFFFFFFFFu : 0u;
            for (int k = k0; k < k1; ++k) {
                const int dx = P.plan.dx[k];
                const int sh = dx & 31;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t v = dx < 0 ? __funnelshift_r(w[j], w[j + 1], sh) : __funnelshift_r(w[j + 1], w[j + 2], sh);
                    acc[j] = ERODE ? (acc[j] & v) : (acc[j] | v);
                }
            }
            o = make_uint4(acc[0], acc[1], acc[2], acc[3]);
        }
        *reinterpret_cast<uint4 *>(dst + tr * pitch + off) = o;
    }
}

__device__ __forceinline__ uint4 valid_quad(const FusedArgs &P, int qc)
{
    if (32 * (4 * qc + 4) <= P.W)
        return make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    return make_uint4(valid_mask(P, 4 * qc), valid_mask(P, 4 * qc + 1), valid_mask(P, 4 * qc + 2), valid_mask(P, 4 * qc + 3));
}

// tiles: [0] staged rows, [1 + p] pattern p's horizontal result (erosion, then reused for the dilation), [1 + npat] the
// eroded rows.  All tiles share one geometry (BH + 2 * span rows of `pitch` words).
__device__ void open_bands_sep(const FusedArgs &P, const uint32_t *src, uint32_t *dst, uint32_t *smem)
{
    const int tid = threadIdx.x;
    const int pitch = P.WWp + 2 * kPadWords;
    const int span = P.dy_max - P.dy_min;
    const int BH = P.band_rows;
    const int rows_max = BH + 2 * span;
    const size_t tile_words = size_t(rows_max) * pitch;
    const int npat = P.plan.npat;
    uint32_t *S = smem;
    uint32_t *E = smem + size_t(npat + 1) * tile_words;
    const int qpr = P.WWp >> 2;       // quads per row
    const int rstep = NT / qpr;       // rows in flight per step (threads beyond rstep * qpr idle)
    const int qc = tid % qpr, r0 = tid / qpr >= rstep ? INT_MAX / 2 : tid / qpr;
    const int off = kPadWords + 4 * qc;
    const uint4 vq = valid_quad(P, qc);
    const int nrows = P.plan.nrows;
    // side pads of the staged rows (set) and of the eroded rows (clear); the pattern tiles' pads are never read
    for (int i = tid; i < rows_max * 2 * kPadWords; i += NT) {
        const int row = i / (2 * kPadWords), c = i - row * (2 * kPadWords);
        const int col = c < kPadWords ? c : P.WWp + c;
        S[row * pitch + col] = 0xFFFFFFFFu;
        E[row * pitch + col] = 0u;
    }
    for (int y0 = 0; y0 < P.H; y0 += BH) {
        const int y1 = min(y0 + BH, P.H);
        const int e0 = y0 + P.dy_min, e1 = y1 + P.dy_max; // eroded rows the band's dilation reads
        const int s0 = e0 + P.dy_min, s1 = e1 + P.dy_max; // source rows their erosion reads
        const int srows = s1 - s0, erows = e1 - e0;
        // stage the source rows; invalid columns and out-of-image rows read as set
        for (int tr = r0; tr < srows; tr += rstep) {
            const int r = s0 + tr;
            uint4 v = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            if (r >= 0 && r < P.H) {
                v = __ldcg(reinterpret_cast<const uint4 *>(src + size_t(r) * P.WWp) + qc);
                v.x |= ~vq.x;
                v.y |= ~vq.y;
                v.z |= ~vq.z;
                v.w |= ~vq.w;
            }
            *reinterpret_cast<uint4 *>(S + tr * pitch + off) = v;
        }
        __syncthreads();
        for (int p = 0; p < npat; ++p)
            if (!P.plan.pat_ident[p])
                morph_rows_h<true>(P, p, S, smem + size_t(p + 1) * tile_words, srows, pitch, qc, r0, rstep);
        __syncthreads();
        // erosion, vertical step: eroded tile row te <-> image row e0 + te; tap row k reads tile row te + dy_k - dy_min
        for (int te = r0; te < erows; te += rstep) {
            const int e = e0 + te;
            uint4 acc = make_uint4(0, 0, 0, 0);
            if (e >= 0 && e < P.H) {
                acc = vq;
                for (int k = 0; k < nrows; ++k) {
                    const int pat = P.plan.row_pat[k];
                    const uint32_t *t = smem + (P.plan.pat_ident[pat] ? 0 : size_t(pat + 1) * tile_words);
                    const uint4 v = *reinterpret_cast<const uint4 *>(t + (te + P.plan.row_dy[k] - P.dy_min) * pitch + off);
                    acc.x &= v.x;
                    acc.y &= v.y;
                    acc.z &= v.z;
                    acc.w &= v.w;
                    if ((acc.x | acc.y | acc.z | acc.w) == 0)
                        break;
                }
            }
            *reinterpret_cast<uint4 *>(E + te * pitch + off) = acc;
        }
        __syncthreads();
        // dilation: the pattern tiles are reused for the horizontal results of the eroded rows; an identity pattern
        // reads the eroded rows themselves
        for (int p = 0; p < npat; ++p)
            if (!P.plan.pat_ident[p])
                morph_rows_h<false>(P, p, E, smem + size_t(p + 1) * tile_words, erows, pitch, qc, r0, rstep);
        __syncthreads();
        for (int ty = r0; ty < y1 - y0; ty += rstep) {
            uint4 acc = make_uint4(0, 0, 0, 0);
            for (int k = 0; k < nrows; ++k) {
                const int pat = P.plan.row_pat[k];
                const uint32_t *t = P.plan.pat_ident[pat] ? E : smem + size_t(pat + 1) * tile_words;
                const uint4 v = *reinterpret_cast<const uint4 *>(t + (ty + P.plan.row_dy[k] - P.dy_min) * pitch + off);
                acc.x |= v.x;
                acc.y |= v.y;
                acc.z |= v.z;
                acc.w |= v.w;
            }
            acc.x &= vq.x;
            acc.y &= vq.y;
            acc.z &= vq.z;
            acc.w &= vq.w;
            *reinterpret_cast<uint4 *>(dst + size_t(y0 + ty) * P.WWp + 4 * qc) = acc;
        }
        __syncthreads();
    }
}

// ---- opening with the structuring element known at COMPILE time ---------------------------------------------------------
// With taps that are only known at run time a horizontal step costs ~6 instructions per tap and word (decode the offset,
// pick the word pair, funnel shift, combine) and a vertical step re-derives every tile address from the plan tables:
// the two openings are a fifth of the kernel's instructions.  The structuring elements people actually use are few --
// the reference's only documented one is cv::getStructuringElement(MORPH_ELLIPSE, (4, 4)) (Sources/rand_tests.cpp:42-51,
// :333-342) -- so the common ones are instantiated with their rows as template constants: every row of such an element
// is either the single tap {0} or ONE contiguous range of taps [LO, HI].  The shifts are immediates, three AND / OR
// fold into one LOP3, the row offsets are loop invariants.  Same band structure, same border rule, same result as
// open_bands_sep; elements without an instantiation take that path.
template <int DYMIN_, int NROWS_, int LO_, int HI_, unsigned IDENT_>
struct CtElem {
    static constexpr int dy_min = DYMIN_, nrows = NROWS_, lo = LO_, hi = HI_;
    static constexpr unsigned ident = IDENT_; // bit j: tap row dy_min + j is the single tap {0}; else the range [lo, hi]
};
using CtEllipse4 = CtElem<-2, 4, -2, 1, 0x1u>;  // [[0,0,1,0],[1,1,1,1],[1,1,1,1],[1,1,1,1]]  (cv2 MORPH_ELLIPSE 4x4)
using CtCross3 = CtElem<-1, 3, -1, 1, 0x5u>;    // [[0,1,0],[1,1,1],[0,1,0]]                  (MORPH_ELLIPSE / CROSS 3x3)
using CtRect3 = CtElem<-1, 3, -1, 1, 0x0u>;     // 3x3 of ones
using CtEllipse5 = CtElem<-2, 5, -2, 2, 0x11u>; // [[0,0,1,0,0],[1,1,1,1,1] x 3,[0,0,1,0,0]]  (MORPH_ELLIPSE 5x5)

// horizontal step over the range [E::lo, E::hi]: w[0] = the word left of the quad, w[1..4] = the quad, w[5] = the word right
template <bool ERODE, class E>
__device__ __forceinline__ uint4 ct_hstep(const uint32_t (&w)[6])
{
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t acc = ERODE ? 0xFFFFFFFFu : 0u;
#pragma unroll
        for (int dx = E::lo; dx <= E::hi; ++dx) {
            const uint32_t v = dx == 0 ? w[j + 1] : dx < 0 ? __funnelshift_r(w[j], w[j + 1], 32 + dx) : __funnelshift_r(w[j + 1], w[j + 2], dx);
            acc = ERODE ? (acc & v) : (acc | v);
        }
        o[j] = acc;
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// tiles: S = staged source rows, Ht = horizontal results (of S, later of E), Et = eroded rows; geometry as open_bands_sep
template <class E>
__device__ void open_bands_ct(const FusedArgs &P, const uint32_t *src, uint32_t *dst, uint32_t *smem)
{
    const int tid = threadIdx.x;
    const int pitch = P.WWp + 2 * kPadWords;
    constexpr int span = E::nrows - 1, dy_max = E::dy_min + span;
    const int BH = P.band_rows;
    const int rows_max = BH + 2 * span;
    const size_t tile_words = size_t(rows_max) * pitch;
    uint32_t *S = smem, *Ht = smem + tile_words, *Et = smem + 2 * tile_words;
    const int qpr = P.WWp >> 2;
    const int rstep = NT / qpr;
    const int qc = tid % qpr, r0 = tid / qpr >= rstep ? INT_MAX / 2 : tid / qpr;
    const int off = kPadWords + 4 * qc;
    const uint4 vq = valid_quad(P, qc);
    for (int i = tid; i < rows_max * 2 * kPadWords; i += NT) {
        const int row = i / (2 * kPadWords), c = i - row * (2 * kPadWords);
        const int col = c < kPadWords ? c : P.WWp + c;
        S[row * pitch + col] = 0xFFFFFFFFu;
        Et[row * pitch + col] = 0u;
    }
    for (int y0 = 0; y0 < P.H; y0 += BH) {
        const int y1 = min(y0 + BH, P.H);
        const int e0 = y0 + E::dy_min, e1 = y1 + dy_max;
        const int s0 = e0 + E::dy_min, s1 = e1 + dy_max;
        const int srows = s1 - s0, erows = e1 - e0;
        for (int tr = r0; tr < srows; tr += rstep) {
            const int r = s0 + tr;
            uint4 v = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            if (r >= 0 && r < P.H) {
                v = __ldcg(reinterpret_cast<const uint4 *>(src + size_t(r) * P.WWp) + qc);
                v.x |= ~vq.x;
                v.y |= ~vq.y;
                v.z |= ~vq.z;
                v.w |= ~vq.w;
            }
            *reinterpret_cast<uint4 *>(S + tr * pitch + off) = v;
        }
        __syncthreads();
        // erosion, horizontal step (an all-clear neighbourhood stays clear: the range contains the tap 0)
        for (int tr = r0; tr < srows; tr += rstep) {
            const uint32_t *row = S + tr * pitch + off;
            const uint4 c = *reinterpret_cast<const uint4 *>(row);
            const uint32_t w[6] = {row[-1], c.x, c.y, c.z, c.w, row[4]};
            uint4 o = make_uint4(0, 0, 0, 0);
            if ((w[0] | w[1] | w[2] | w[3] | w[4] | w[5]) != 0)
                o = ct_hstep<true, E>(w);
            *reinterpret_cast<uint4 *>(Ht + tr * pitch + off) = o;
        }
        __syncthreads();
        // erosion, vertical step: eroded tile row te <-> image row e0 + te; tap row j reads tile row te + j
        for (int te = r0; te < erows; te += rstep) {
            const int e = e0 + te;
            uint4 acc = make_uint4(0, 0, 0, 0);
            if (e >= 0 && e < P.H) {
                acc = vq;
#pragma unroll
                for (int j = 0; j < E::nrows; ++j) {
                    const uint32_t *t = ((E::ident >> j) & 1u) ? S : Ht;
                    const uint4 v = *reinterpret_cast<const uint4 *>(t + (te + j) * pitch + off);
                    acc.x &= v.x;
                    acc.y &= v.y;
                    acc.z &= v.z;
                    acc.w &= v.w;
                }
            }
            *reinterpret_cast<uint4 *>(Et + te * pitch + off) = acc;
        }
        __syncthreads();
        // dilation, horizontal step of the eroded rows
        for (int tr = r0; tr < erows; tr += rstep) {
            const uint32_t *row = Et + tr * pitch + off;
            const uint4 c = *reinterpret_cast<const uint4 *>(row);
            const uint32_t w[6] = {row[-1], c.x, c.y, c.z, c.w, row[4]};
            uint4 o = make_uint4(0, 0, 0, 0);
            if ((w[0] | w[1] | w[2] | w[3] | w[4] | w[5]) != 0)
                o = ct_hstep<false, E>(w);
            *reinterpret_cast<uint4 *>(Ht + tr * pitch + off) = o;
        }
        __syncthreads();
        for (int ty = r0; ty < y1 - y0; ty += rstep) {
            uint4 acc = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int j = 0; j < E::nrows; ++j) {
                const uint32_t *t = ((E::ident >> j) & 1u) ? Et : Ht;
                const uint4 v = *reinterpret_cast<const uint4 *>(t + (ty + j) * pitch + off);
                acc.x |= v.x;
                acc.y |= v.y;
                acc.z |= v.z;
                acc.w |= v.w;
            }
            acc.x &= vq.x;
            acc.y &= vq.y;
            acc.z &= vq.z;
            acc.w &= vq.w;
            *reinterpret_cast<uint4 *>(dst + size_t(y0 + ty) * P.WWp + 4 * qc) = acc;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------------
// run extraction.  Warp w owns a contiguous range of 128-bit quads of the bit image; pass 1 counts run starts, a scan
// over the warp totals gives each warp its first id, pass 2 writes the run records.  Returns T (the run count);
// rowoff[H] = T and parent[T] = T (the FRAME node).
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t quad_transitions(const FusedArgs &P, const uint4 &w, uint32_t prev_msb, int wx0, uint32_t t[4])
{
    const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
    const bool row_start = wx0 == 0;
    const bool full = 32 * (wx0 + 4) <= P.W; // all four words lie inside the image: no column masks needed
    const uint32_t any = w.x | w.y | w.z | w.w, all = w.x & w.y & w.z & w.w;
    if (!row_start && ((any == 0 && prev_msb == 0) || (all == 0xFFFFFFFFu && prev_msb == 1 && full))) {
        t[0] = t[1] = t[2] = t[3] = 0;
        return 0;
    }
    uint32_t p = row_start ? (~w.x & 1u) : prev_msb; // x = 0 always starts a run
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        t[k] = ww[k] ^ ((ww[k] << 1) | p);
        p = ww[k] >> 31;
    }
    if (!full) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            t[k] &= valid_mask(P, wx0 + k);
    }
    return __popc(t[0]) + __popc(t[1]) + __popc(t[2]) + __popc(t[3]);
}

constexpr int kQU = 4; // quads (128-bit loads) in flight per lane in the run extraction

// one warp-iteration of the extraction: kQU quads per lane, all loads issued before the first use; bit u of `prevs` is the
// bit that precedes quad u (the MSB of the previous word in raster order)
__device__ __forceinline__ void load_quad_batch(const uint32_t *img, uint32_t qb, uint32_t q1, int lane, uint32_t &carry,
                                                uint4 w[kQU], uint32_t &prevs)
{
#pragma unroll
    for (int u = 0; u < kQU; ++u) {
        const uint32_t q = qb + 32u * u + lane;
        w[u] = make_uint4(0, 0, 0, 0);
        if (q < q1)
            w[u] = __ldcg(reinterpret_cast<const uint4 *>(img) + q);
    }
    prevs = 0;
#pragma unroll
    for (int u = 0; u < kQU; ++u) {
        uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, w[u].w, 1) >> 31;
        if (lane == 0)
            prev = carry;
        carry = __shfl_sync(0xFFFFFFFFu, w[u].w, 31) >> 31;
        prevs |= prev << u;
    }
}

// Where the run-level phases read a labelled run set from.  The slot's global arrays always hold the complete set (run
// records, row offsets and, after the flatten, the roots); while a frame's run count fits, the same three arrays also
// sit in shared memory and every dependent access of the merge / statistics phases stays on the SM.
template <bool SM>
struct View {
    const uint32_t *xinfo;
    const uint32_t *rowoff;
    uint32_t *parent;
    uint32_t *fbits; // one bit per run id: the root of a background region that touches the image border (FRAME)
    __device__ __forceinline__ uint32_t xi(uint32_t i) const { return xinfo[i]; }
    __device__ __forceinline__ uint32_t ro(uint32_t y) const { return rowoff[y]; }
    __device__ __forceinline__ uint32_t par(uint32_t i) const { return Par<SM>{parent}.get(i); }
    // largest j in [a, b) with x_start(j) <= x   (a row's first run starts at 0, so it always exists)
    __device__ __forceinline__ uint32_t at(uint32_t a, uint32_t b, uint32_t x) const
    {
        uint32_t lo = a, hi = b - 1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (run_x(xinfo[mid]) <= x)
                lo = mid;
            else
                hi = mid - 1;
        }
        return lo;
    }
    __device__ __forceinline__ uint32_t end(uint32_t r, uint32_t row_end, int W) const
    {
        return (r + 1 < row_end) ? run_x(xinfo[r + 1]) - 1u : uint32_t(W - 1);
    }
    // root -> does its background region touch the image border (i.e. belong to the FRAME region)?
    __device__ __forceinline__ bool is_frame(uint32_t root) const
    {
        const uint32_t w = SM ? *reinterpret_cast<volatile uint32_t *>(fbits + (root >> 5)) : __ldcg(fbits + (root >> 5));
        return (w >> (root & 31)) & 1u;
    }
    // canonical id of the background region of run j: any region of the FRAME -> T
    __device__ __forceinline__ uint32_t region(uint32_t j, uint32_t T) const
    {
        const uint32_t r = par(j);
        return is_frame(r) ? T : r;
    }
};

// shared-memory copy of a run set: [rowoff: H + 2, padded][xinfo: cap][parent: cap]
struct SmemRuns {
    uint32_t *rowoff, *xinfo, *parent, *fbits;
    uint32_t *stats;  // remove-small-objects statistics: link, st_s, st_e, st_x, `tp` words each (valid when st_ok)
    uint32_t tp;      // array pitch of the current run set: T + 1 rounded up to 4
    uint32_t avail;   // words of the area that starts at rowoff
    uint32_t ro_words;
    bool st_ok;       // the statistics arrays of the current run set also fit
    uint32_t cap; // runs (incl. the FRAME node) the copy can hold; 0 = the row offsets alone do not fit
    uint16_t *qoff; // run extraction: per 128-bit quad, the number of run starts, then their offset inside the owning
                    // warp's range (nullptr: the image has too many quads, the extraction takes the lane-ordered path)
};

__device__ __forceinline__ SmemRuns smem_runs(const FusedArgs &P, uint32_t *smem)
{
    SmemRuns m;
    const uint32_t ro_words = (uint32_t(P.H) + 2 + 3) & ~3u;
    m.rowoff = smem;
    // the quad offsets sit at the end of the dynamic shared memory when they take at most a third of it
    const uint32_t qwords = (((P.nwords >> 2) + 1u) / 2u + 3u) & ~3u;
    uint32_t words = P.smem_words;
    m.qoff = nullptr;
    if (qwords * 3u <= P.smem_words) {
        words -= qwords;
        m.qoff = reinterpret_cast<uint16_t *>(smem + words);
    }
    // cap records + cap parents + cap / 32 + 1 flag words
    m.cap = ro_words + 256 < words ? (((words - ro_words - 4) * 32u) / 65u) & ~31u : 0;
    m.xinfo = smem + ro_words;
    m.parent = m.xinfo + m.cap;
    m.fbits = m.parent + m.cap;
    m.stats = nullptr;
    m.tp = 0;
    m.avail = words;
    m.ro_words = ro_words;
    m.st_ok = false;
    return m;
}

// The arrays behind the run records are placed for the run count T of the set being extracted: parent and the FRAME
// flags always (when they fit: sm_ok), and -- for the usual few thousand runs -- also the four statistics arrays of
// the remove-small-objects step, whose atomics and dependent reads then stay on the SM.
__device__ __forceinline__ bool place_run_arrays(SmemRuns &m, uint32_t T)
{
    const uint32_t tp = (T + 1u + 3u) & ~3u;
    const uint32_t fbw = ((T >> 5) + 1u + 3u) & ~3u;
    m.tp = tp;
    m.parent = m.xinfo + tp;
    m.fbits = m.parent + tp;
    m.stats = m.fbits + fbw;
    const bool sm_ok = m.cap != 0 && m.ro_words + 2u * tp + fbw <= m.avail;
    m.st_ok = sm_ok && m.ro_words + 6u * tp + fbw <= m.avail;
    return sm_ok;
}

// Returns T (the run count).  rowoff[H] = T.  sm_ok <- the set also sits in shared memory.
__device__ uint32_t extract_runs(const FusedArgs &P, Shared &sh, const uint32_t *img, const RunSet &rs, SmemRuns &sm,
                                 bool &sm_ok)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nq = P.nwords >> 2;
    constexpr uint32_t step = 32u * kQU;
    const uint32_t per_warp = ((nq + NW * step - 1) / (NW * step)) * step;
    const uint32_t q0 = min(uint32_t(warp) * per_warp, nq), q1 = min(q0 + per_warp, nq);
    const uint32_t first_carry = (q0 < q1 && q0 > 0) ? (ld(img + 4 * size_t(q0) - 1) >> 31) : 0u;
    // pass 1: count
    {
        uint32_t cnt = 0, carry = first_carry;
        for (uint32_t qb = q0; qb < q1; qb += step) {
            uint4 w[kQU];
            uint32_t prevs;
            load_quad_batch(img, qb, q1, lane, carry, w, prevs);
#pragma unroll
            for (int u = 0; u < kQU; ++u) {
                const uint32_t q = qb + 32u * u + lane;
                if (q < q1) {
                    int y, wx0;
                    split(P, 4 * q, y, wx0);
                    uint32_t t[4];
                    const uint32_t c = quad_transitions(P, w[u], (prevs >> u) & 1u, wx0, t);
                    cnt += c;
                    if (sm.qoff)
                        sm.qoff[q] = uint16_t(c); // at most 128 run starts per quad
                }
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1)
            cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, d);
        if (lane == 0)
            sh.wsum[warp] = cnt;
    }
    __syncthreads();
    prof_tick(P.prof, P.prof, sh, kPCountRuns);
    uint32_t base = 0, T = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        const uint32_t c = sh.wsum[w];
        if (w < warp)
            base += c;
        T += c;
    }
    sm_ok = place_run_arrays(sm, T);
    // the warps' ranges hold at most 65535 runs each (else their 16-bit quad offsets overflow: lane-ordered path)
    bool quick = sm.qoff != nullptr;
#pragma unroll
    for (int w = 0; w < NW; ++w)
        quick = quick && sh.wsum[w] <= 65535u;
    if (quick) {
        // ---- pass 2, work proportional to RUNS: counts -> offsets (per warp, in place), then every thread takes
        // run ids tid, tid + NT, ...: binary search for the quad that holds the run, one 16-byte load of that quad,
        // n-th set bit of its transition words
        if (threadIdx.x <= NW) {
            uint32_t b = 0;
            for (int w = 0; w < NW; ++w)
                if (w < int(threadIdx.x))
                    b += sh.wsum[w];
            sh.wbase[threadIdx.x] = b;
        }
        {
            uint32_t run = 0;
            for (uint32_t qb = q0; qb < q1; qb += 32u) {
                const uint32_t q = qb + lane;
                const uint32_t c = q < q1 ? sm.qoff[q] : 0u;
                uint32_t inc = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                    if (lane >= d)
                        inc += n;
                }
                if (q < q1)
                    sm.qoff[q] = uint16_t(run + inc - c);
                run += __shfl_sync(0xFFFFFFFFu, inc, 31);
            }
        }
        __syncthreads();
        for (uint32_t r = threadIdx.x; r < T; r += NT) {
            uint32_t lo = 0, hi = NW - 1;
            while (lo < hi) { // warp range of run r: largest w with wbase[w] <= r
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (sh.wbase[mid] <= r)
                    lo = mid;
                else
                    hi = mid - 1;
            }
            const uint32_t rel = r - sh.wbase[lo];
            const uint32_t qa = min(lo * per_warp, nq), qz = min(qa + per_warp, nq);
            lo = qa;
            hi = qz - 1;
            while (lo < hi) { // quad of run r: largest q of the range with offset <= rel
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (sm.qoff[mid] <= rel)
                    lo = mid;
                else
                    hi = mid - 1;
            }
            const uint32_t q = lo;
            uint32_t n = rel - sm.qoff[q]; // the run is the n-th run start of its quad
            int y, wx0;
            split(P, 4 * q, y, wx0);
            const uint4 w4 = __ldcg(reinterpret_cast<const uint4 *>(img) + q);
            const uint32_t prev = wx0 == 0 ? 0u : (ld(img + 4 * size_t(q) - 1) >> 31);
            uint32_t t[4];
            quad_transitions(P, w4, prev, wx0, t);
            const uint32_t c0 = __popc(t[0]), c1 = __popc(t[1]), c2 = __popc(t[2]);
            uint32_t k, tk, wk;
            if (n < c0) {
                k = 0, tk = t[0], wk = w4.x;
            } else if (n < c0 + c1) {
                k = 1, tk = t[1], wk = w4.y, n -= c0;
            } else if (n < c0 + c1 + c2) {
                k = 2, tk = t[2], wk = w4.z, n -= c0 + c1;
            } else {
                k = 3, tk = t[3], wk = w4.w, n -= c0 + c1 + c2;
            }
            const uint32_t b = __fns(tk, 0, int(n) + 1);
            const uint32_t x = 32u * (uint32_t(wx0) + k) + b;
            const uint32_t rec = x | (uint32_t(y) << 16) | (((wk >> b) & 1u) << 31);
            rs.xinfo[r] = rec;
            if (sm_ok)
                sm.xinfo[r] = rec;
            if (x == 0) {
                rs.rowoff[y] = r;
                if (sm_ok)
                    sm.rowoff[y] = r;
            }
        }
    } else
    // pass 2 (lane-ordered): fill
    {
        uint32_t carry = first_carry;
        for (uint32_t qb = q0; qb < q1; qb += step) {
            uint4 w[kQU];
            uint32_t prevs;
            load_quad_batch(img, qb, q1, lane, carry, w, prevs);
#pragma unroll
            for (int u = 0; u < kQU; ++u) {
                const uint32_t q = qb + 32u * u + lane;
                uint32_t t[4] = {0, 0, 0, 0};
                uint32_t c = 0;
                int y = 0, wx0 = 0;
                if (q < q1) {
                    split(P, 4 * q, y, wx0);
                    c = quad_transitions(P, w[u], (prevs >> u) & 1u, wx0, t);
                }
                if (__ballot_sync(0xFFFFFFFFu, c != 0) == 0)
                    continue;
                uint32_t inc = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                    if (lane >= d)
                        inc += n;
                }
                uint32_t id = base + inc - c;
                base += __shfl_sync(0xFFFFFFFFu, inc, 31);
                if (c) {
                    if (wx0 == 0) {
                        rs.rowoff[y] = id;
                        if (sm_ok)
                            sm.rowoff[y] = id;
                    }
                    const uint32_t ww[4] = {w[u].x, w[u].y, w[u].z, w[u].w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        uint32_t tt = t[k];
                        while (tt) {
                            const int b = __ffs(tt) - 1;
                            tt &= tt - 1;
                            const uint32_t rec = uint32_t(32 * (wx0 + k) + b) | (uint32_t(y) << 16) | (((ww[k] >> b) & 1u) << 31);
                            rs.xinfo[id] = rec;
                            if (sm_ok)
                                sm.xinfo[id] = rec;
                            ++id;
                        }
                    }
                }
            }
        }
    }
    if (threadIdx.x == 0) {
        rs.rowoff[P.H] = T;
        if (sm_ok)
            sm.rowoff[P.H] = T;
    }
    __syncthreads();
    return T;
}

// ------------------------------------------------------------------------------------------------------------------
// labelling of runs
// ------------------------------------------------------------------------------------------------------------------
// The union-find starts from a FOREST instead of singletons: every run is hooked (plain store, no atomics) to the first
// run of the row above that it touches and that has the same value.  Ids grow in raster order, so a hook always
// points to a smaller id and the "labels only decrease" invariant holds from the start.  Almost every background run
// of a frame touches exactly one background run above it, so the thousands of contended atomicMin calls on the root
// of the background component disappear; only a run's SECOND and later neighbours above need a real union.
template <bool FG8, bool MERGE_FG, bool SM>
__device__ __forceinline__ uint32_t hook_of(const FusedArgs &P, const View<SM> &V, uint32_t r)
{
    const uint32_t xi = V.xi(r);
    const uint32_t s = run_x(xi), y = run_y(xi), v = run_v(xi);
    if ((!MERGE_FG && v) || y == 0)
        return r;
    const uint32_t e = V.end(r, V.ro(y + 1), P.W);
    const uint32_t d = (FG8 && v) ? 1u : 0u; // 8-connected runs may touch diagonally
    const uint32_t a = V.ro(y - 1), b = V.ro(y);
    const uint32_t c0 = s >= d ? s - d : 0u;
    const uint32_t c1 = min(e + d, uint32_t(P.W - 1));
    for (uint32_t j = V.at(a, b, c0); j < b; ++j) {
        const uint32_t xj = V.xi(j);
        if (run_x(xj) > c1)
            break;
        if (run_v(xj) == v)
            return j;
    }
    return r;
}

template <bool FG8, bool FRAME, bool MERGE_FG, bool SM>
__device__ void merge_phase(const FusedArgs &P, const View<SM> &V, uint32_t T)
{
    const Par<SM> par{V.parent};
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        const uint32_t xi = V.xi(r);
        const uint32_t s = run_x(xi), y = run_y(xi), v = run_v(xi);
        if (!MERGE_FG && v)
            continue;
        const uint32_t e = V.end(r, V.ro(y + 1), P.W);
        if (y > 0) {
            const uint32_t d = (FG8 && v) ? 1u : 0u; // 8-connected runs may touch diagonally
            const uint32_t a = V.ro(y - 1), b = V.ro(y);
            const uint32_t c0 = s >= d ? s - d : 0u;
            const uint32_t c1 = min(e + d, uint32_t(P.W - 1));
            bool hooked = false; // the first same-valued neighbour is this run's hook (label_with)
            for (uint32_t j = V.at(a, b, c0); j < b; ++j) {
                const uint32_t xj = V.xi(j);
                if (run_x(xj) > c1)
                    break;
                if (run_v(xj) == v) {
                    if (hooked)
                        uf_union(par, r, j);
                    hooked = true;
                }
            }
        }
    }
}

template <bool FG8, bool FRAME, bool MERGE_FG, bool SM>
__device__ void label_with(const FusedArgs &P, Shared &sh, const RunSet &rs, const View<SM> &V, uint32_t T)
{
    const Par<SM> par{V.parent};
    for (uint32_t r = threadIdx.x; r <= T; r += NT)
        par.set(r, r < T ? hook_of<FG8, MERGE_FG>(P, V, r) : r);
    if (FRAME)
        for (uint32_t i = threadIdx.x; i <= (T >> 5); i += NT) {
            if (SM)
                V.fbits[i] = 0;
            st(rs.fbits + i, 0u);
        }
    __syncthreads();
    // pointer jumping: a hook goes exactly one row up, so the hooked forest is at most H deep (one chain through the
    // background of an empty frame); ceil(log2 H) rounds of parent <- grandparent leave every run pointing at its root
    // and the unions below start from flat trees
    for (int span = 1; span < P.H; span <<= 2) {
        int changed = 0;
        for (uint32_t r = threadIdx.x; r < T; r += NT) {
            uint32_t p = par.get(r);
#pragma unroll
            for (int hop = 0; hop < 3; ++hop) { // three jumps per barrier: up to 8x shallower per round
                const uint32_t gp = par.get(p);
                if (gp == p)
                    break;
                p = gp;
                changed = 1;
            }
            par.set(r, p);
        }
        if (!__syncthreads_or(changed))
            break;
    }
    prof_tick(P.prof, P.prof, sh, kPHook);
    merge_phase<FG8, FRAME, MERGE_FG, SM>(P, V, T);
    __syncthreads();
    prof_tick(P.prof, P.prof, sh, kPMerge);
    // flatten (roots are final: shortening a chain under a concurrent walk is harmless); the slot's global array always
    // receives the roots.  FRAME: instead of a node that every border run is united with (thousands of atomics on
    // one root), the roots of the background regions that touch the image border are flagged.
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        const uint32_t root = uf_find(par, r);
        par.set(r, root);
        if (SM)
            st(rs.parent + r, root);
        if (FRAME) {
            const uint32_t xi = V.xi(r);
            if (!run_v(xi)) {
                const uint32_t y = run_y(xi);
                if (y == 0 || y == uint32_t(P.H - 1) || run_x(xi) == 0 || V.end(r, V.ro(y + 1), P.W) == uint32_t(P.W - 1)) {
                    if (SM)
                        atomicOr(V.fbits + (root >> 5), 1u << (root & 31));
                    atomicOr(rs.fbits + (root >> 5), 1u << (root & 31));
                }
            }
        }
    }
    __syncthreads();
    prof_tick(P.prof, P.prof, sh, kPFlatten);
}

// labels the runs of `img` into run set rs; returns T; sm_ok <- the set is also resident in shared memory
template <bool FG8, bool FRAME, bool MERGE_FG>
__device__ uint32_t label_runs(const FusedArgs &P, Shared &sh, const uint32_t *img, const RunSet &rs, SmemRuns &sm,
                               bool &sm_ok)
{
    const uint32_t T = extract_runs(P, sh, img, rs, sm, sm_ok);
    prof_tick(P.prof, P.prof, sh, kPExtract);
    if (sm_ok)
        label_with<FG8, FRAME, MERGE_FG, true>(P, sh, rs, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T);
    else
        label_with<FG8, FRAME, MERGE_FG, false>(P, sh, rs, View<false>{rs.xinfo, rs.rowoff, rs.parent, rs.fbits}, T);
    if (P.prof && threadIdx.x == 0)
        atomicAdd(P.prof + kPRuns, (unsigned long long)T);
    return T;
}

// ------------------------------------------------------------------------------------------------------------------
// hysteresis (ThresholdImageWithHysteresis :107-144).  U's set is read from the slot's global arrays (the shared-memory
// copy, if any, holds L's set, labelled last).
// ------------------------------------------------------------------------------------------------------------------
template <bool SM>
__device__ void hysteresis_phase(const FusedArgs &P, const View<false> &VU, uint32_t Tu, const View<SM> &VL, uint32_t Tl,
                                 int *marks, uint32_t *out)
{
    for (uint32_t r = threadIdx.x; r <= Tl; r += NT)
        st(marks + r, 0);
    for (uint32_t i = threadIdx.x; i < (P.nwords >> 2); i += NT)
        reinterpret_cast<uint4 *>(out)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < Tu; r += NT) {
        const uint32_t xi = VU.xi(r);
        if (!run_v(xi) || VU.par(r) != r)
            continue; // seeds are the raster-first pixels of the hi components (contour[0])
        const uint32_t s = run_x(xi), y = run_y(xi);
        // RETR_EXTERNAL: the region left of the first pixel (the component's outer background) must be FRAME
        const bool external = (s == 0) || VU.is_frame(VU.par(r - 1));
        if (external) {
            const uint32_t j = VL.at(VL.ro(y), VL.ro(y + 1), s);
            st(marks + VL.par(j), 1);
        }
    }
    __syncthreads();
    // runs of the lower mask whose region holds a seed (both values: the lo > hi quirk)
    for (uint32_t r = threadIdx.x; r < Tl; r += NT) {
        if (!ld(marks + VL.par(r)))
            continue;
        const uint32_t xi = VL.xi(r);
        const uint32_t y = run_y(xi);
        set_range(out + size_t(y) * P.WWp, int(run_x(xi)), int(VL.end(r, VL.ro(y + 1), P.W)));
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------------
// remove small objects (RemoveSmallObjects :146-181), in place on img
// ------------------------------------------------------------------------------------------------------------------
// statistics arrays: shared memory (ST) or the slot's global scratch (read through L2 only: they are hit by atomics)
template <bool ST, typename T_>
__device__ __forceinline__ T_ sld(const T_ *p)
{
    return ST ? *reinterpret_cast<const volatile T_ *>(p) : __ldcg(p);
}
template <bool ST, typename T_>
__device__ __forceinline__ void sst(T_ *p, T_ v)
{
    if (ST)
        *reinterpret_cast<volatile T_ *>(p) = v;
    else
        __stcg(p, v);
}

// is pixel (x, yy) foreground?  Answered from the run set (the runs of a row alternate in value); j <- the run.
template <bool SM>
__device__ __forceinline__ bool fg_at(const FusedArgs &P, const View<SM> &V, int x, int yy, uint32_t &j, uint32_t &row_end)
{
    row_end = V.ro(yy + 1);
    j = V.at(V.ro(yy), row_end, uint32_t(x));
    return run_v(V.xi(j)) != 0u;
}

template <bool SM, bool ST>
__device__ void rso_phase(const FusedArgs &P, uint32_t *img, const View<SM> &V, uint32_t T, uint32_t *link, int *st_s, int *st_e,
                          int *st_x, int min_size, int *changed)
{
    if (threadIdx.x == 0)
        *changed = 0;
    // roots: zero the statistics; link = outer background region (components) / parent component (holes)
    for (uint32_t r = threadIdx.x; r <= T; r += NT) {
        if (r < T && V.par(r) != r)
            continue;
        sst<ST>(st_s + r, 0);
        sst<ST>(st_e + r, 0);
        sst<ST>(st_x + r, 0);
        if (r == T)
            continue;
        const uint32_t xi = V.xi(r);
        const uint32_t s = run_x(xi);
        if (run_v(xi))
            sst<ST>(link + r, s == 0 ? T : V.region(r - 1, T)); // region left of the first pixel
        else
            sst<ST>(link + r, (s == 0 || V.is_frame(r)) ? kNoLabel : V.par(r - 1)); // component left of the hole
    }
    __syncthreads();
    // contour statistics, accumulated on the contour's owner: the component for its outer contour, the hole's
    // background region for a hole contour
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        const uint32_t xi = V.xi(r);
        if (!run_v(xi))
            continue;
        const int s = int(run_x(xi)), y = int(run_y(xi));
        const int e = int(V.end(r, V.ro(y + 1), P.W));
        const uint32_t C = V.par(r);
        const uint32_t bout = sld<ST>(link + C);
        auto owner = [&](uint32_t b) { return b == bout ? C : b; };
        const uint32_t own_l = owner(s == 0 ? T : V.region(r - 1, T));
        const uint32_t own_r = owner(e == P.W - 1 ? T : V.region(r + 1, T));
        // horizontal cracks at the two run ends, and the convex corners there: 2x2 blocks in which a run end is the
        // only foreground pixel
        int xl = 0, xr = 0;
#pragma unroll
        for (int dy = -1; dy <= 1; dy += 2) {
            const int yy = y + dy;
            if (yy < 0 || yy >= P.H) { // outside the image: background on both sides of both run ends
                ++xl;
                ++xr;
                continue;
            }
            uint32_t j, row_end;
            // (s, yy) and its left neighbour: the same run unless that run starts exactly at s
            bool f = fg_at(P, V, s, yy, j, row_end);
            bool fn = s > 0 && (int(run_x(V.xi(j))) < s ? f : !f);
            if (!f && !fn)
                ++xl;
            // (e, yy) and its right neighbour: the same run unless that run ends exactly at e
            f = fg_at(P, V, e, yy, j, row_end);
            fn = e + 1 < P.W && (int(V.end(j, row_end, P.W)) > e ? f : !f);
            if (!f && !fn)
                ++xr;
        }
        if (own_l == own_r) {
            atomicAdd(&st_s[own_l], e + 1 - s);
            atomicAdd(&st_e[own_l], 2);
            if (xl + xr)
                atomicAdd(&st_x[own_l], xl + xr);
        } else {
            atomicAdd(&st_s[own_l], -s);
            atomicAdd(&st_e[own_l], 1);
            atomicAdd(&st_s[own_r], e + 1);
            atomicAdd(&st_e[own_r], 1);
            if (xl)
                atomicAdd(&st_x[own_l], xl);
            if (xr)
                atomicAdd(&st_x[own_r], xr);
        }
        // vertical cracks: columns of this run whose neighbour in the adjacent row is background
        for (int dy = -1; dy <= 1; dy += 2) {
            const int yy = y + dy;
            if (yy < 0 || yy >= P.H) {
                atomicAdd(&st_e[owner(T)], e - s + 1);
                continue;
            }
            const uint32_t a = V.ro(yy), b = V.ro(yy + 1);
            for (uint32_t j = V.at(a, b, uint32_t(s)); j < b; ++j) {
                const uint32_t xj = V.xi(j);
                if (int(run_x(xj)) > e)
                    break;
                if (run_v(xj))
                    continue;
                const int js = max(int(run_x(xj)), s), je = min(int(V.end(j, b, P.W)), e);
                atomicAdd(&st_e[owner(V.region(j, T))], je - js + 1);
            }
        }
    }
    __syncthreads();
    // per root: st_e <- small flag (2*area < 2*min_size; contourArea(c) < min_size, :171)
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        if (V.par(r) != r)
            continue;
        const long long s = sld<ST>(st_s + r);
        const int cracks = sld<ST>(st_e + r);
        const long long len = (long long)cracks - sld<ST>(st_x + r);
        const long long two_a = run_v(V.xi(r)) ? 2 * s - len - 2 : 2 * (s < 0 ? -s : s) + len - 2;
        sst<ST>(st_e + r, (cracks > 0 && two_a < 2ll * min_size) ? 1 : 0);
    }
    __syncthreads();
    // per component: st_x <- parity of the number of consecutive small contours up the nesting chain
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        if (V.par(r) != r || !run_v(V.xi(r)))
            continue;
        int count = 0;
        uint32_t cur = r;
        for (;;) {
            if (!sld<ST>(st_e + cur))
                break;
            ++count;
            const uint32_t b = sld<ST>(link + cur);
            if (b == T)
                break;
            if (!sld<ST>(st_e + b))
                break;
            ++count;
            const uint32_t par = sld<ST>(link + b);
            if (par == kNoLabel)
                break;
            cur = par;
        }
        sst<ST>(st_x + r, count & 1);
    }
    __syncthreads();
    // clear the pixels the single filled drawContours call erases (:178)
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        const uint32_t xi = V.xi(r);
        if (!run_v(xi))
            continue;
        const int s = int(run_x(xi)), y = int(run_y(xi));
        const int e = int(V.end(r, V.ro(y + 1), P.W));
        const uint32_t C = V.par(r);
        uint32_t *row = img + size_t(y) * P.WWp;
        bool cleared = false;
        if (sld<ST>(st_x + C)) {
            clear_range(row, s, e);
            *changed = 1;
            continue;
        }
        const uint32_t bout = sld<ST>(link + C);
        auto is_small = [&](uint32_t b) { return sld<ST>(st_e + (b == bout ? C : b)) != 0; };
        if (is_small(s == 0 ? T : V.region(r - 1, T))) {
            clear_range(row, s, s);
            cleared = true;
        }
        if (is_small(e == P.W - 1 ? T : V.region(r + 1, T))) {
            clear_range(row, e, e);
            cleared = true;
        }
        for (int dy = -1; dy <= 1; dy += 2) {
            const int yy = y + dy;
            if (yy < 0 || yy >= P.H) {
                if (is_small(T)) {
                    clear_range(row, s, e);
                    cleared = true;
                }
                continue;
            }
            const uint32_t a = V.ro(yy), b = V.ro(yy + 1);
            for (uint32_t j = V.at(a, b, uint32_t(s)); j < b; ++j) {
                const uint32_t xj = V.xi(j);
                if (int(run_x(xj)) > e)
                    break;
                if (run_v(xj) || !is_small(V.region(j, T)))
                    continue;
                clear_range(row, max(int(run_x(xj)), s), min(int(V.end(j, b, P.W)), e));
                cleared = true;
            }
        }
        if (cleared)
            *changed = 1;
    }
    __syncthreads();
}

__device__ void rso_dispatch(const FusedArgs &P, uint32_t *img, const RunSet &ra, const SmemRuns &sm, bool sm_ok, uint32_t T,
                             uint32_t *link, int *st_s, int *st_e, int *st_x, int min_size, int *changed)
{
    if (sm_ok && sm.st_ok)
        rso_phase<true, true>(P, img, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T, sm.stats,
                              reinterpret_cast<int *>(sm.stats + sm.tp), reinterpret_cast<int *>(sm.stats + 2 * sm.tp),
                              reinterpret_cast<int *>(sm.stats + 3 * sm.tp), min_size, changed);
    else if (sm_ok)
        rso_phase<true, false>(P, img, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T, link, st_s, st_e, st_x,
                               min_size, changed);
    else
        rso_phase<false, false>(P, img, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, T, link, st_s, st_e, st_x,
                                min_size, changed);
}

// ------------------------------------------------------------------------------------------------------------------
// hole fill (FillHoles :183-221), in place: set every background run that is not connected to the seed corner.
// white <- 1 when the seed pixel itself is set (the flood fill is then a no-op and the result is all 255).
// ------------------------------------------------------------------------------------------------------------------
template <bool SM>
__device__ void fill_phase(const FusedArgs &P, uint32_t *img, const View<SM> &V, uint32_t T, int *white)
{
    // seed = (0,0) if that pixel is set, else the bottom-right corner (follow the code :201-209, not its comment)
    const uint32_t seed = run_v(V.xi(0)) ? 0u : T - 1u;
    if (run_v(V.xi(seed))) {
        if (threadIdx.x == 0)
            *white = 1;
    } else {
        const uint32_t seed_root = V.par(seed);
        for (uint32_t r = threadIdx.x; r < T; r += NT) {
            const uint32_t xi = V.xi(r);
            if (run_v(xi) || V.par(r) == seed_root)
                continue;
            const uint32_t y = run_y(xi);
            set_range(img + size_t(y) * P.WWp, int(run_x(xi)), int(V.end(r, V.ro(y + 1), P.W)));
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------------
// expand: (A | B) -> 0 / 255 bytes (:77)
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t nibble_to_bytes(uint32_t n) // bit j -> byte j = 0xFF
{
    return (((n & 0xFu) * 0x00204081u) & 0x01010101u) * 0xFFu;
}

// 16 mask bits -> 16 bytes of 0 / 255
__device__ __forceinline__ uint4 half_to_bytes(uint32_t h)
{
    return make_uint4(nibble_to_bytes(h), nibble_to_bytes(h >> 4), nibble_to_bytes(h >> 8), nibble_to_bytes(h >> 12));
}

// A warp expands 32 consecutive bit words (1024 pixels) per round.  Lane l does not store the 32 bytes of "its" word
// (that makes every store instruction touch half of 32 sectors); it stores 16-byte chunk l and chunk 32 + l of the
// warp's 1 KB, taking the bits from the lanes that hold those words, so each store instruction writes 512 contiguous
// bytes (whole sectors) whenever the 32 words lie in one image row.
__device__ void expand_phase(const FusedArgs &P, unsigned f, const uint32_t *A, const uint32_t *B, bool white)
{
    uint8_t *dst = P.out + size_t(f) * P.out_stride;
    const int lane = threadIdx.x & 31;
    constexpr int U = 4; // rounds in flight per warp: the loads come from L2
    const uint32_t nround = (P.nwords + 31u) / 32u;
    for (uint32_t r0 = threadIdx.x >> 5; r0 < nround; r0 += U * NW) {
        uint32_t w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t i = (r0 + u * NW) * 32u + lane;
            w[u] = 0xFFFFFFFFu;
            if (!white && i < P.nwords && r0 + u * NW < nround)
                w[u] = ld(A + i) | ld(B + i);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t base = (r0 + u * NW) * 32u;
            if (r0 + u * NW >= nround)
                break; // warp-uniform
            if (P.fast_io) {
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    const int src_lane = 16 * part + (lane >> 1);
                    const uint32_t ws = __shfl_sync(0xFFFFFFFFu, w[u], src_lane);
                    const uint32_t i = base + src_lane;
                    int y, wx;
                    split(P, i, y, wx);
                    if (i < P.nwords && wx < P.WW)
                        __stcs(reinterpret_cast<uint4 *>(dst + size_t(y) * P.W + 32u * wx + 16u * (lane & 1)),
                               half_to_bytes(ws >> (16 * (lane & 1)))); // masks are written once: streaming
                }
            } else {
                const uint32_t i = base + lane;
                int y, wx;
                split(P, i, y, wx);
                if (i < P.nwords && wx < P.WW) {
                    uint8_t *o = dst + size_t(y) * P.W + 32u * wx;
                    const int n = min(32, P.W - 32 * wx);
                    for (int k = 0; k < n; ++k)
                        o[k] = ((w[u] >> k) & 1u) ? 255 : 0;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// components of the final mask (opt-in): what the reference's users compute on the host in their tracker callback with
// cv2.connectedComponentsWithStats(bw_frame, connectivity=8) (assign_objects_algo.h:124-130 hands them bw_frame; the
// in-code note highlight_objects_algo.cpp:152-153 weighs that very call).  8-connected components of the mask, numbered
// 1.. in the raster order of their first pixels (canonical labelling); per component: bounding box, area, first
// pixel, coordinate sums (centroid = sums / area).  The label image is optional (4 bytes per pixel of output).
// ------------------------------------------------------------------------------------------------------------------
// Shape and contrast statistics (cvvp_component_stats) of the foreground runs, added to the records of their components.
// The moments have closed forms per run.  The contrast sums read the run's frame and background bytes: a warp takes its
// 32 runs one at a time and spreads each run's pixels over its lanes (four per lane and step on the 128-bit path), so
// a frame's 1920-pixel runs (the FillHoles all-255 quirk) cost 15 steps, not 1920.  Every lane then adds its own run's
// totals to the record.
template <int POL, bool SM>
__device__ void stats_runs(const FusedArgs &P, unsigned f, const View<SM> &V, uint32_t T, const uint32_t *cidx, uint8_t *recs)
{
    const int lane = threadIdx.x & 31;
    const uint8_t *fr = P.frames + size_t(f) * P.frame_stride;
    const uint8_t *bg = P.bg + size_t(f) * P.bg_stride;
    for (uint32_t rb = threadIdx.x & ~31u; rb < T; rb += NT) { // warp-uniform: runs rb .. rb + 31
        const uint32_t r = rb + lane;
        int s = 0, e = -1, y = 0;
        uint32_t kk = kNoLabel;
        if (r < T) {
            const uint32_t xi = V.xi(r);
            if (run_v(xi)) {
                s = int(run_x(xi)), y = int(run_y(xi));
                e = int(V.end(r, V.ro(y + 1), P.W));
                kk = ld(cidx + V.par(r));
            }
        }
        const bool mine = kk < uint32_t(P.max_comps);
        uint32_t my_sd = 0, my_mn = 0, my_mx = 0;
        unsigned long long my_sdx = 0;
        for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, mine); todo; todo &= todo - 1u) {
            const int src = __ffs(int(todo)) - 1;
            const int rs = __shfl_sync(0xFFFFFFFFu, s, src), re = __shfl_sync(0xFFFFFFFFu, e, src);
            const int ry = __shfl_sync(0xFFFFFFFFu, y, src);
            const uint8_t *frow = fr + size_t(ry) * P.W, *brow = bg + size_t(ry) * P.W;
            uint32_t sd = 0, mn = 255, mx = 0;
            unsigned long long sdx = 0;
            if (P.fast_io) { // rows start 16-byte aligned in both images: aligned words, bytes outside [rs, re] masked
                uint32_t vmn = 0xFFFFFFFFu, vmx = 0;
                for (int w = (rs >> 2) + lane; w <= (re >> 2); w += 32) {
                    const int x0 = 4 * w;
                    uint32_t keep = 0xFFFFFFFFu;
                    if (x0 < rs)
                        keep &= 0xFFFFFFFFu << (8 * (rs - x0));
                    if (x0 + 3 > re)
                        keep &= 0xFFFFFFFFu >> (8 * (x0 + 3 - re));
                    const uint32_t d = diff_u8x4<POL>(__ldg(reinterpret_cast<const uint32_t *>(frow) + w),
                                                      __ldg(reinterpret_cast<const uint32_t *>(brow) + w)) & keep;
                    const uint32_t ws = __dp4a(d, 0x01010101u, 0u);
                    sd += ws;
                    sdx += (unsigned long long)x0 * ws + __dp4a(d, 0x03020100u, 0u);
                    vmn = __vminu4(vmn, d | ~keep);
                    vmx = __vmaxu4(vmx, d);
                }
                mn = min(min(vmn & 0xFFu, (vmn >> 8) & 0xFFu), min((vmn >> 16) & 0xFFu, vmn >> 24));
                mx = max(max(vmx & 0xFFu, (vmx >> 8) & 0xFFu), max((vmx >> 16) & 0xFFu, vmx >> 24));
            } else {
                for (int x = rs + lane; x <= re; x += 32) {
                    const uint32_t d = uint32_t(hl_diff(__ldg(brow + x), __ldg(frow + x), POL));
                    sd += d;
                    sdx += (unsigned long long)d * uint32_t(x);
                    mn = min(mn, d);
                    mx = max(mx, d);
                }
            }
            sd = __reduce_add_sync(0xFFFFFFFFu, sd); // a run's sum of d is below 255 * 65536
            mn = __reduce_min_sync(0xFFFFFFFFu, mn);
            mx = __reduce_max_sync(0xFFFFFFFFu, mx);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
                sdx += __shfl_xor_sync(0xFFFFFFFFu, sdx, o);
            if (lane == src)
                my_sd = sd, my_sdx = sdx, my_mn = mn, my_mx = mx;
        }
        if (mine) {
            cvvp_component_stats *c = reinterpret_cast<cvvp_component_stats *>(recs + size_t(kk) * P.rec_bytes);
            const long long len = e - s + 1, yy = y;
            // sum of x * x over [s, e] = F(e) - F(s - 1), F(n) = n (n + 1) (2n + 1) / 6
            const long long se = e, ss = s - 1;
            const long long sxx = se * (se + 1) * (2 * se + 1) / 6 - ss * (ss + 1) * (2 * ss + 1) / 6;
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_xx), (unsigned long long)sxx);
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_xy), (unsigned long long)(yy * ((s + e) * len / 2)));
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_yy), (unsigned long long)(yy * yy * len));
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_d), (unsigned long long)my_sd);
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_dx), my_sdx);
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_dy), (unsigned long long)yy * my_sd);
            atomicMin(&c->min_d, int(my_mn));
            atomicMax(&c->max_d, int(my_mx));
        }
    }
}

template <bool SM>
__device__ void components_phase(const FusedArgs &P, Shared &sh, unsigned f, const View<SM> &V, uint32_t T, uint32_t *cidx)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // component number of every foreground root = how many foreground roots precede it (ids are in raster order).
    // Threads take contiguous chunks of run ids so that a block scan of the per-thread counts gives the offsets.
    const uint32_t per = (T + NT - 1) / NT;
    const uint32_t r0 = min(threadIdx.x * per, T), r1 = min(r0 + per, T);
    uint32_t cnt = 0;
    for (uint32_t r = r0; r < r1; ++r)
        cnt += (run_v(V.xi(r)) && V.par(r) == r) ? 1u : 0u;
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, d);
        if (lane >= d)
            inc += n;
    }
    if (lane == 31)
        sh.wsum[warp] = inc;
    __syncthreads();
    uint32_t base = 0, total = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        const uint32_t c = sh.wsum[w];
        if (w < warp)
            base += c;
        total += c;
    }
    uint32_t k = base + inc - cnt;
    uint8_t *recs = reinterpret_cast<uint8_t *>(P.comps) + size_t(f) * P.max_comps * P.rec_bytes;
    for (uint32_t r = r0; r < r1; ++r) {
        const uint32_t xi = V.xi(r);
        if (run_v(xi) && V.par(r) == r) {
            st(cidx + r, k);
            if (k < uint32_t(P.max_comps)) {
                cvvp_component c;
                c.x0 = INT_MAX, c.y0 = INT_MAX, c.x1 = -1, c.y1 = -1;
                c.area = 0;
                c.first_x = int(run_x(xi)), c.first_y = int(run_y(xi));
                c.reserved = 0;
                c.sum_x = 0, c.sum_y = 0;
                *reinterpret_cast<cvvp_component *>(recs + size_t(k) * P.rec_bytes) = c;
                if (P.stats) {
                    cvvp_component_stats *cs = reinterpret_cast<cvvp_component_stats *>(recs + size_t(k) * P.rec_bytes);
                    cs->sum_xx = cs->sum_xy = cs->sum_yy = 0;
                    cs->sum_d = cs->sum_dx = cs->sum_dy = 0;
                    cs->min_d = INT_MAX, cs->max_d = INT_MIN;
                }
            }
            ++k;
        }
    }
    if (threadIdx.x == 0)
        P.ncomps[f] = int(total);
    __threadfence_block();
    __syncthreads();
    int32_t *lab = P.labels ? P.labels + size_t(f) * P.labels_stride : nullptr;
    if (lab) { // background = 0 everywhere first
        const uint32_t npix = uint32_t(P.W) * uint32_t(P.H);
        const bool vec = (reinterpret_cast<uintptr_t>(lab) & 15u) == 0;
        const uint32_t n4 = vec ? npix / 4u : 0u;
        for (uint32_t i = threadIdx.x; i < n4; i += NT)
            __stcs(reinterpret_cast<int4 *>(lab) + i, make_int4(0, 0, 0, 0));
        for (uint32_t i = 4u * n4 + threadIdx.x; i < npix; i += NT)
            lab[i] = 0;
        __syncthreads();
    }
    for (uint32_t r = threadIdx.x; r < T; r += NT) {
        const uint32_t xi = V.xi(r);
        if (!run_v(xi))
            continue;
        const int s = int(run_x(xi)), y = int(run_y(xi));
        const int e = int(V.end(r, V.ro(y + 1), P.W));
        const uint32_t kk = ld(cidx + V.par(r));
        if (kk < uint32_t(P.max_comps)) {
            cvvp_component *c = reinterpret_cast<cvvp_component *>(recs + size_t(kk) * P.rec_bytes);
            const int len = e - s + 1;
            atomicAdd(&c->area, len);
            atomicMin(&c->x0, s);
            atomicMax(&c->x1, e);
            atomicMin(&c->y0, y);
            atomicMax(&c->y1, y);
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_x), (unsigned long long)((long long)(s + e) * len / 2));
            atomicAdd(reinterpret_cast<unsigned long long *>(&c->sum_y), (unsigned long long)((long long)y * len));
        }
        if (lab) {
            int32_t *row = lab + size_t(y) * P.W;
            for (int x = s; x <= e; ++x)
                row[x] = int32_t(kk + 1u);
        }
    }
    if (P.stats) { // uniform for the launch
        if (P.polarity == CVVP_POLARITY_DARK)
            stats_runs<CVVP_POLARITY_DARK>(P, f, V, T, cidx, recs);
        else if (P.polarity == CVVP_POLARITY_BRIGHT)
            stats_runs<CVVP_POLARITY_BRIGHT>(P, f, V, T, cidx, recs);
        else
            stats_runs<CVVP_POLARITY_BOTH>(P, f, V, T, cidx, recs);
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------------------------
constexpr int kSmemOffs = 256; // structuring-element taps cached in shared memory

__global__ void __launch_bounds__(NT, kCtasPerSm) highlight_fused_kernel(const FusedArgs P)
{
    extern __shared__ uint4 dyn_smem4[];
    uint32_t *dyn = reinterpret_cast<uint32_t *>(dyn_smem4);
    __shared__ Shared sh;
    __shared__ short2 sh_offs[kSmemOffs];
    const short2 *offs = P.offs;
    if (P.noffs <= kSmemOffs) {
        for (int k = threadIdx.x; k < P.noffs; k += NT)
            sh_offs[k] = P.offs[k];
        offs = sh_offs;
    }
    const size_t slot = blockIdx.x;
    uint32_t *A = P.bits + slot * kImages * size_t(P.nwords);
    uint32_t *U = A + P.nwords, *L = U + P.nwords, *Tm = L + P.nwords;
    uint32_t *rbase = P.runs + slot * P.run_words;
    uint32_t *ro = P.rowoff + slot * 2 * size_t(P.rstride);
    uint32_t *fb = rbase + kRunArrays * size_t(P.cap); // FRAME flag bits of set a (set b is never labelled with FRAME)
    const RunSet ra{rbase, rbase + P.cap, ro, fb};
    const RunSet rb{rbase + 2 * size_t(P.cap), rbase + 3 * size_t(P.cap), ro + P.rstride, fb};
    uint32_t *link = rbase + 4 * size_t(P.cap);
    int *st_s = reinterpret_cast<int *>(rbase + 5 * size_t(P.cap));
    int *st_e = reinterpret_cast<int *>(rbase + 6 * size_t(P.cap));
    int *st_x = reinterpret_cast<int *>(rbase + 7 * size_t(P.cap));
    SmemRuns sm = smem_runs(P, dyn);

    for (;;) {
        if (threadIdx.x == 0) {
            sh.frame = atomicAdd(&P.queue[0], 1u);
            sh.white[0] = sh.white[1] = 0;
        }
        __syncthreads();
        const unsigned f = sh.frame;
        if (f >= P.nframes)
            break;
        prof_tick(P.prof, P.prof, sh, -1);
        bits_phase(P, f, A, U, L);
        __syncthreads();
        prof_tick(P.prof, P.prof, sh, kPBits);
        // debug_stage (CVVP_HL_DEBUG_STAGE): 1 A=d>th, 2 U=d>hi, 3 L=d>lo, 4 A opened, 5 A small removed, 6 A filled,
        // 7 B=hysteresis, 8 B opened, 9 B small removed, 10 B filled
#define CVVP_DEBUG_STAGE(k, img, w)                                                                                    \
    if (P.debug_stage == (k)) {                                                                                        \
        expand_phase(P, f, (img), (img), (w));                                                                         \
        __syncthreads();                                                                                               \
        continue;                                                                                                      \
    }
        CVVP_DEBUG_STAGE(1, A, false)
        CVVP_DEBUG_STAGE(2, U, false)
        CVVP_DEBUG_STAGE(3, L, false)
        // ---- branch A: threshold -> open -> remove small -> fill holes                                  (:35-47)
        if (P.band_rows > 0) {
            if (P.ct_elem == 1)
                open_bands_ct<CtEllipse4>(P, A, Tm, dyn);
            else if (P.ct_elem == 2)
                open_bands_ct<CtCross3>(P, A, Tm, dyn);
            else if (P.ct_elem == 3)
                open_bands_ct<CtRect3>(P, A, Tm, dyn);
            else if (P.ct_elem == 4)
                open_bands_ct<CtEllipse5>(P, A, Tm, dyn);
            else if (P.plan.sep)
                open_bands_sep(P, A, Tm, dyn);
            else
                open_bands(P, offs, A, Tm, dyn);
            uint32_t *t = A;
            A = Tm;
            Tm = t;
        } else {
            morph_phase<true, false>(P, A, Tm);
            __syncthreads();
            prof_tick(P.prof, P.prof, sh, kPErodeA);
            morph_phase<false, false>(P, Tm, A);
            __syncthreads();
        }
        prof_tick(P.prof, P.prof, sh, kPDilateA);
        CVVP_DEBUG_STAGE(4, A, false)
        bool sm_ok;
        uint32_t T = label_runs<true, true, true>(P, sh, A, ra, sm, sm_ok);
        rso_dispatch(P, A, ra, sm, sm_ok, T, link, st_s, st_e, st_x, P.min_th, &sh.changed);
        prof_tick(P.prof, P.prof, sh, kPRso);
        CVVP_DEBUG_STAGE(5, A, false)
        // the hole fill needs the 4-connected background regions of the image: when nothing was cleared they are the
        // ones just labelled, else the image is labelled again
        if (sh.changed)
            T = label_runs<false, false, false>(P, sh, A, ra, sm, sm_ok);
        if (sm_ok)
            fill_phase(P, A, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T, &sh.white[0]);
        else
            fill_phase(P, A, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, T, &sh.white[0]);
        prof_tick(P.prof, P.prof, sh, kPFill);
        CVVP_DEBUG_STAGE(6, A, sh.white[0] != 0)
        // ---- branch B: hysteresis -> open -> remove small -> fill holes                                 (:54-73)
        const uint32_t Tu = label_runs<true, true, true>(P, sh, U, ra, sm, sm_ok);
        const uint32_t Tl = label_runs<false, false, true>(P, sh, L, rb, sm, sm_ok);
        // U's bits are no longer needed: its image now receives the result
        if (sm_ok)
            hysteresis_phase(P, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, Tu, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits},
                             Tl, st_x, U);
        else
            hysteresis_phase(P, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, Tu, View<false>{rb.xinfo, rb.rowoff, rb.parent, rb.fbits},
                             Tl, st_x, U);
        prof_tick(P.prof, P.prof, sh, kPHyst);
        CVVP_DEBUG_STAGE(7, U, false)
        if (P.band_rows > 0) {
            if (P.ct_elem == 1)
                open_bands_ct<CtEllipse4>(P, U, Tm, dyn);
            else if (P.ct_elem == 2)
                open_bands_ct<CtCross3>(P, U, Tm, dyn);
            else if (P.ct_elem == 3)
                open_bands_ct<CtRect3>(P, U, Tm, dyn);
            else if (P.ct_elem == 4)
                open_bands_ct<CtEllipse5>(P, U, Tm, dyn);
            else if (P.plan.sep)
                open_bands_sep(P, U, Tm, dyn);
            else
                open_bands(P, offs, U, Tm, dyn);
            uint32_t *t = U;
            U = Tm;
            Tm = t;
        } else {
            morph_phase<true, true>(P, U, Tm);
            __syncthreads();
            prof_tick(P.prof, P.prof, sh, kPErodeB);
            morph_phase<false, false>(P, Tm, U);
            __syncthreads();
        }
        prof_tick(P.prof, P.prof, sh, kPDilateB);
        CVVP_DEBUG_STAGE(8, U, false)
        T = label_runs<true, true, true>(P, sh, U, ra, sm, sm_ok);
        rso_dispatch(P, U, ra, sm, sm_ok, T, link, st_s, st_e, st_x, P.min_hyst, &sh.changed);
        prof_tick(P.prof, P.prof, sh, kPRso);
        CVVP_DEBUG_STAGE(9, U, false)
        if (sh.changed)
            T = label_runs<false, false, false>(P, sh, U, ra, sm, sm_ok);
        if (sm_ok)
            fill_phase(P, U, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T, &sh.white[1]);
        else
            fill_phase(P, U, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, T, &sh.white[1]);
        prof_tick(P.prof, P.prof, sh, kPFill);
        CVVP_DEBUG_STAGE(10, U, sh.white[1] != 0)
#undef CVVP_DEBUG_STAGE
        // ---- out = 255 * (A | B)                                                                         (:77)
        expand_phase(P, f, A, U, sh.white[0] || sh.white[1]);
        __syncthreads();
        prof_tick(P.prof, P.prof, sh, kPExpand);
        if (P.comps) {
            // final mask as a bit image (A and U are not needed any more), labelled 8-connected
            const bool white = sh.white[0] || sh.white[1];
            for (uint32_t i = threadIdx.x; i < P.nwords; i += NT) {
                int y, wx;
                split(P, i, y, wx);
                Tm[i] = (white ? 0xFFFFFFFFu : (ld(A + i) | ld(U + i))) & valid_mask(P, wx);
            }
            __syncthreads();
            T = label_runs<true, false, true>(P, sh, Tm, ra, sm, sm_ok);
            if (sm_ok)
                components_phase(P, sh, f, View<true>{sm.xinfo, sm.rowoff, sm.parent, sm.fbits}, T, link);
            else
                components_phase(P, sh, f, View<false>{ra.xinfo, ra.rowoff, ra.parent, ra.fbits}, T, link);
        }
        if (P.prof && threadIdx.x == 0)
            atomicAdd(P.prof + kPFrames, 1ull);
    }
    // the last CTA to leave re-arms the queue for the next launch
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned done = atomicAdd(&P.queue[1], 1u);
        if (done == gridDim.x - 1) {
            P.queue[0] = 0;
            P.queue[1] = 0;
            __threadfence();
        }
    }
}

struct FusedGeom {
    int WW, WWp, wwp_shift;
    uint32_t nwords, cap, rstride;
};

// rows per band of the shared-memory opening (0: the tiles do not fit, use the global-memory taps)
int pick_band_rows(const FusedGeom &fg, int dy_min, int dy_max, const MorphPlan &plan)
{
    const int span = dy_max - dy_min;
    const size_t pitch = size_t(fg.WWp) + 2 * kPadWords;
    for (int bh = 128; bh >= 8; bh -= 8) {
        const size_t words = plan.sep ? size_t(plan.npat + 2) * (size_t(bh) + 2 * span) * pitch
                                      : (size_t(bh) * 2 + 3 * size_t(span)) * pitch;
        if (words * sizeof(uint32_t) <= kDynSmemBytes)
            return bh;
    }
    return 0;
}

// taps (sorted by row, then column) -> MorphPlan
MorphPlan make_plan(const std::vector<short2> &offs)
{
    MorphPlan pl;
    memset(&pl, 0, sizeof(pl));
    std::vector<std::vector<int>> pats;
    size_t i = 0;
    int ntaps = 0;
    while (i < offs.size()) {
        const int dy = offs[i].y;
        std::vector<int> dxs;
        for (; i < offs.size() && offs[i].y == dy; ++i) {
            if (offs[i].x < -31 || offs[i].x > 31)
                return pl;
            dxs.push_back(offs[i].x);
        }
        if (dy < -127 || dy > 127 || pl.nrows >= kMaxPlanRows)
            return pl;
        int id = -1;
        for (size_t p = 0; p < pats.size(); ++p)
            if (pats[p] == dxs)
                id = int(p);
        if (id < 0) {
            if (int(pats.size()) >= kMaxPat || ntaps + int(dxs.size()) > kMaxPlanTaps)
                return pl;
            id = int(pats.size());
            pats.push_back(dxs);
            pl.pat_start[id] = (unsigned char)ntaps;
            for (int dx : dxs)
                pl.dx[ntaps++] = (signed char)dx;
            pl.pat_start[id + 1] = (unsigned char)ntaps;
            pl.pat_ident[id] = (dxs.size() == 1 && dxs[0] == 0) ? 1 : 0;
        }
        pl.row_dy[pl.nrows] = (signed char)dy;
        pl.row_pat[pl.nrows] = (signed char)id;
        ++pl.nrows;
    }
    pl.npat = int(pats.size());
    pl.sep = 1;
    return pl;
}

// which compile-time instantiation of the opening (open_bands_ct) an element has: 0 = none
template <class E>
bool matches_ct(const std::vector<short2> &offs)
{
    std::vector<short2> want;
    for (int j = 0; j < E::nrows; ++j) {
        if ((E::ident >> j) & 1u) {
            want.push_back(make_short2(0, short(E::dy_min + j)));
        } else {
            for (int dx = E::lo; dx <= E::hi; ++dx)
                want.push_back(make_short2(short(dx), short(E::dy_min + j)));
        }
    }
    if (want.size() != offs.size())
        return false;
    for (size_t i = 0; i < want.size(); ++i)
        if (want[i].x != offs[i].x || want[i].y != offs[i].y)
            return false;
    return true;
}

int match_ct_elem(const std::vector<short2> &offs)
{
    if (matches_ct<CtEllipse4>(offs))
        return 1;
    if (matches_ct<CtCross3>(offs))
        return 2;
    if (matches_ct<CtRect3>(offs))
        return 3;
    if (matches_ct<CtEllipse5>(offs))
        return 4;
    return 0;
}

FusedGeom fused_geom(const HlGeom &g)
{
    FusedGeom fg;
    fg.WW = (g.W + 31) / 32;
    int wwp = (fg.WW + 3) & ~3;
    int p2 = 4;
    while (p2 < fg.WW)
        p2 <<= 1;
    fg.wwp_shift = -1;
    if (p2 - fg.WW <= fg.WW / 8) { // a power-of-two row pitch replaces the divisions by shifts (<= 12.5 % padding)
        wwp = p2;
        fg.wwp_shift = 0;
        while ((1 << fg.wwp_shift) < p2)
            ++fg.wwp_shift;
    }
    fg.WWp = wwp;
    fg.nwords = uint32_t(g.H) * uint32_t(wwp);
    fg.cap = uint32_t(round_up(size_t(g.npix) + 2, 4));
    fg.rstride = uint32_t(round_up(size_t(g.H) + 2, 4));
    return fg;
}

size_t run_words(const FusedGeom &fg)
{
    return size_t(kRunArrays) * fg.cap + round_up(fg.cap / 32 + 4, 4);
}

size_t slot_bytes(const FusedGeom &fg)
{
    return sizeof(uint32_t) * (size_t(kImages) * fg.nwords + run_words(fg) + 2 * size_t(fg.rstride));
}
} // namespace

int HLF(fused_frames_in_flight)(cvvp_ctx *ctx, HighlightState *st);
int HLF(highlight_fused_batch)(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                               size_t bg_stride, unsigned nb, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                               cudaStream_t stream);

#ifndef CVVP_HLF_SMALL
int fused_frames_in_flight_small(cvvp_ctx *ctx, HighlightState *st);
int highlight_fused_batch_small(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                                size_t bg_stride, unsigned nb, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                                cudaStream_t stream);

bool fused_supports(const HighlightState *st)
{
    return st->g.W <= 65535 && st->g.H <= 32767;
}

void fused_release(HighlightState *st)
{
    FusedScratch &fs = st->fs;
    pool_dev_free(fs.bits, fs.bits_bytes); // parked for the next job of this geometry (pool.hpp)
    pool_dev_free(fs.runs, fs.runs_bytes);
    pool_dev_free(fs.rowoff, fs.rowoff_bytes);
    if (fs.queue)
        cudaFree(fs.queue);
    fs = FusedScratch();
}

// Which build of the kernel a job uses (fixed at its first batch): frames of at most 512x512 pixels take the
// 256-thread CTAs, four to an SM.  CVVP_HL_VARIANT=large|small forces one (tests hold both to the oracle).
static bool use_small(HighlightState *st)
{
    if (st->fused_variant < 0) {
        st->fused_variant = st->g.npix <= 512u * 512u && st->g.W <= 2048 ? 1 : 0;
        if (const char *v = getenv("CVVP_HL_VARIANT")) {
            if (!strcmp(v, "small") && st->g.W <= 8192)
                st->fused_variant = 1;
            else if (!strcmp(v, "large"))
                st->fused_variant = 0;
        }
    }
    return st->fused_variant == 1;
}

int fused_frames_in_flight(cvvp_ctx *ctx, HighlightState *st)
{
    return use_small(st) ? fused_frames_in_flight_small(ctx, st) : fused_frames_in_flight_large(ctx, st);
}

int highlight_fused_batch(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                          size_t bg_stride, unsigned nb, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                          cudaStream_t stream)
{
    return use_small(st) ? highlight_fused_batch_small(ctx, st, in, frame_stride, bg, bg_stride, nb, d_out, out_stride, cc, stream)
                         : highlight_fused_batch_large(ctx, st, in, frame_stride, bg, bg_stride, nb, d_out, out_stride, cc, stream);
}
#endif

// number of frames the kernel keeps in flight = resident CTAs, bounded by a scratch budget
int HLF(fused_frames_in_flight)(cvvp_ctx *ctx, HighlightState *st)
{
    if (st->fs.slots > 0)
        return st->fs.slots;
    int per_sm = 0;
    cudaFuncSetAttribute(highlight_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kDynSmemBytes));
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, highlight_fused_kernel, NT, kDynSmemBytes) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    const FusedGeom fg = fused_geom(st->g);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
        cudaGetLastError();
        free_b = size_t(8) << 30;
    }
    size_t budget = free_b / 4;
    if (budget > (size_t(24) << 30))
        budget = size_t(24) << 30;
    long long slots = (long long)per_sm * ctx->sm_count;
    const long long by_mem = (long long)(budget / slot_bytes(fg));
    if (slots > by_mem)
        slots = by_mem;
    if (const char *ov = getenv("CVVP_HL_SLOTS")) { // developer aid: frames in flight
        const long long v = atoll(ov);
        if (v >= 1 && v <= by_mem)
            slots = v;
    }
    if (slots < 1)
        slots = 1;
    return int(slots);
}

static int ensure_fused(cvvp_ctx *ctx, HighlightState *st)
{
    FusedScratch &fs = st->fs;
    if (fs.slots > 0)
        return CVVP_OK;
    const int slots = HLF(fused_frames_in_flight)(ctx, st);
    const FusedGeom fg = fused_geom(st->g);
    const size_t nb = sizeof(uint32_t) * size_t(slots) * kImages * fg.nwords;
    const size_t nr = sizeof(uint32_t) * size_t(slots) * run_words(fg);
    const size_t no = sizeof(uint32_t) * size_t(slots) * 2 * fg.rstride;
    fs.bits_bytes = nb;
    fs.runs_bytes = nr;
    fs.rowoff_bytes = no;
    if (pool_dev_alloc(reinterpret_cast<void **>(&fs.bits), nb) != cudaSuccess ||
        pool_dev_alloc(reinterpret_cast<void **>(&fs.runs), nr) != cudaSuccess ||
        pool_dev_alloc(reinterpret_cast<void **>(&fs.rowoff), no) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&fs.queue), 2 * sizeof(unsigned)) != cudaSuccess) {
        cudaGetLastError();
        fused_release(st);
        return fail(ctx, CVVP_ERR_NOMEM, "highlight: cudaMalloc of %zu bytes of scratch failed", nb + nr + no);
    }
    if (cudaMemset(fs.queue, 0, 2 * sizeof(unsigned)) != cudaSuccess) {
        fused_release(st);
        return fail(ctx, CVVP_ERR_CUDA, "highlight: queue initialisation failed");
    }
    fs.slots = slots;
    return CVVP_OK;
}

// One batch of nb frames (device pointers), one kernel launch.  Work in flight on a context's highlight scratch must
// be on one stream at a time.
int HLF(highlight_fused_batch)(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                               size_t bg_stride, unsigned nb, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                               cudaStream_t stream)
{
    int rc = ensure_fused(ctx, st);
    if (rc != CVVP_OK)
        return rc;
    const FusedGeom fg = fused_geom(st->g);
    FusedArgs P;
    P.frames = in;
    P.frame_stride = frame_stride;
    P.bg = bg;
    P.bg_stride = bg_stride;
    P.out = d_out;
    P.out_stride = out_stride;
    P.th_a = st->th == -1 ? st->d_th : nullptr;
    P.th = st->th;
    P.lo = st->lo;
    P.hi = st->hi;
    P.min_th = st->min_th;
    P.min_hyst = st->min_hyst;
    P.offs = st->d_offs;
    P.noffs = st->noffs;
    P.W = st->g.W;
    P.H = st->g.H;
    P.WW = fg.WW;
    P.WWp = fg.WWp;
    P.wwp_shift = fg.wwp_shift;
    P.nwords = fg.nwords;
    P.cap = fg.cap;
    P.run_words = run_words(fg);
    P.rstride = fg.rstride;
    P.bits = st->fs.bits;
    P.runs = st->fs.runs;
    P.rowoff = st->fs.rowoff;
    P.queue = st->fs.queue;
    P.nframes = nb;
    P.smem_words = uint32_t(kDynSmemBytes / sizeof(uint32_t));
    P.dy_min = st->dy_min;
    P.dy_max = st->dy_max;
    P.pad_words = kPadWords;
    P.plan = make_plan(st->h_offs);
    if (getenv("CVVP_HL_NO_SEP"))
        P.plan.sep = 0; // developer aid: force the generic tap loop
    P.band_rows = pick_band_rows(fg, st->dy_min, st->dy_max, P.plan);
    // the common structuring elements have compile-time instantiations of the opening (CVVP_HL_NO_CT=1: run-time plan)
    P.ct_elem = (P.plan.sep && P.band_rows > 0 && !getenv("CVVP_HL_NO_CT")) ? match_ct_elem(st->h_offs) : 0;
    auto aligned16 = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    P.polarity = st->polarity;
    P.fast_io = (P.W % 32 == 0) && aligned16(in) && aligned16(d_out) && aligned16(bg) && frame_stride % 16 == 0 &&
                out_stride % 16 == 0 && bg_stride % 16 == 0;
    const char *dbg = getenv("CVVP_HL_DEBUG_STAGE");
    P.debug_stage = dbg ? atoi(dbg) : 0;
    P.comps = cc.comps;
    P.ncomps = cc.ncomps;
    P.max_comps = cc.max_comps;
    P.rec_bytes = uint32_t(cc.rec_bytes);
    P.stats = cc.rec_bytes == sizeof(cvvp_component_stats);
    P.labels = cc.labels;
    P.labels_stride = cc.labels_stride;
    P.prof = nullptr;
    const bool want_prof = getenv("CVVP_HL_PROF") != nullptr;
    if (want_prof && cudaMalloc(reinterpret_cast<void **>(&P.prof), kPCount * sizeof(unsigned long long)) == cudaSuccess)
        cudaMemsetAsync(P.prof, 0, kPCount * sizeof(unsigned long long), stream);
    const unsigned grid = nb < unsigned(st->fs.slots) ? nb : unsigned(st->fs.slots);
    highlight_fused_kernel<<<grid, NT, kDynSmemBytes, stream>>>(P);
    ctx->launches += 1;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return fail(ctx, CVVP_ERR_CUDA, "highlight: kernel launch failed: %s", cudaGetErrorString(e));
    if (P.prof) { // developer aid (CVVP_HL_PROF=1): per-phase time of an average frame, measured by thread 0 of each CTA
        unsigned long long h[kPCount];
        cudaStreamSynchronize(stream);
        cudaMemcpy(h, P.prof, sizeof(h), cudaMemcpyDeviceToHost);
        cudaFree(P.prof);
        static const char *names[] = {"bits", "erodeA", "dilateA", "fill runs(x6)", "merge(x6)", "flatten(x6)", "rso(x2)",
                                      "fill(x2)", "hyst", "erodeB", "dilateB", "expand", "count runs(x6)", "hook(x6)"};
        const double nf = h[kPFrames] ? double(h[kPFrames]) : 1.0;
        double total = 0;
        for (int k = 0; k < kPRuns; ++k)
            total += double(h[k]);
        fprintf(stderr, "[cvvp prof] %llu frames, grid %u, %.1f runs per labelling, %.1f us per frame per CTA\n", h[kPFrames],
                grid, double(h[kPRuns]) / nf / 6.0, total / nf / 1e3);
        for (int k = 0; k < kPRuns; ++k)
            fprintf(stderr, "[cvvp prof]   %-12s %9.1f us  %5.1f %%\n", names[k], double(h[k]) / nf / 1e3,
                    100.0 * double(h[k]) / total);
    }
    return CVVP_OK;
}
} // namespace cvvp
