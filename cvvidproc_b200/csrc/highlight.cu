// Per-frame highlight stage on sm_100a -- replaces HighlightObjectsAlgo::HighlightObjects
// (/root/reference/Sources/ProcessorAlgos/highlight_objects_algo.cpp:17-221).
//
// The reference is a sequence of OpenCV calls (subtract, threshold, morphologyEx, findContours, contourArea,
// drawContours, floodFill).  Contour tracing and flood fills are sequential; here every step is restated with
// connected-component labels and purely local rules (SURVEY.md section 9; executable spec: oracle/highlight_model.py,
// which is held bit-exact to a cv2 restatement of the reference):
//
//   d  = max(bg - frame, 0)                                   (:27-29, saturating, NOT absdiff; other object
//                                                               polarities: hl_diff, cvvp_highlight_set_polarity)
//   A  = fill(rso(open(d > th), min_size_threshold))          (:35-47)
//   B  = fill(rso(open(hyst(d, lo, hi)), min_size_hyst))      (:54-73)
//   out = 255 * (A | B)                                       (:77)
//
//   open  : erode then dilate with the same (unreflected) kernel offsets, anchor (kw/2, kh/2), out-of-image samples
//           ignored                                                                       (cv::morphologyEx :39, :61)
//   ccl   : union-find labelling (label = smallest linear index of the component = its raster-first pixel) of the
//           foreground (8- or 4-connected) AND the background (4-connected) in one label image; optional virtual
//           FRAME node that joins every background region touching the image border
//   hyst  : seeds = raster-first pixels of the EXTERNAL 8-connected components of d > hi (outer background is FRAME);
//           keep the 4-connected equal-value regions of d > lo that contain a seed            (:107-144)
//   rso   : per contour (component, adjacent background region): signed crack sum s, crack count E, convex-corner
//           count Xv -> polygon area 2A = 2s - (E - Xv) - 2 (outer) or 2|s| + (E - Xv) - 2 (hole); zero the pixels
//           on small contours, and the interiors by the even-odd nesting parity of the single filled draw (:146-181)
//   fill  : everything except the 4-connected background region containing the seed corner   (:183-221)
//
// Layout: every kernel takes blockIdx.z = frame of the batch.  Masks are u8 0/1 (npix per frame), label / statistic
// arrays are u32 / i32 with npix + 1 entries per frame (entry npix = the FRAME node).
#include "highlight_state.hpp"
#include "pool.hpp"

#include <cstddef>
#include <new>
#include <vector>

namespace cvvp
{
namespace
{
constexpr uint32_t kNoLabel = 0xFFFFFFFFu;

// ------------------------------------------------------------------------------------------------------------------
// union-find primitives (labels only ever decrease; stale reads are harmless)
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t uf_find(const uint32_t *lab, uint32_t x)
{
    uint32_t p = lab[x];
    while (p != x) {
        x = p;
        p = lab[x];
    }
    return x;
}

__device__ __forceinline__ void uf_union(uint32_t *lab, uint32_t a, uint32_t b)
{
    bool done;
    do {
        a = uf_find(lab, a);
        b = uf_find(lab, b);
        if (a < b) {
            const uint32_t old = atomicMin(&lab[b], a);
            done = (old == b);
            b = old;
        } else if (b < a) {
            const uint32_t old = atomicMin(&lab[a], b);
            done = (old == a);
            a = old;
        } else {
            done = true;
        }
    } while (!done);
}

// ------------------------------------------------------------------------------------------------------------------
// K1: difference + the three thresholds
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    diff_thresh_kernel(const uint8_t *__restrict__ frames, size_t frame_stride, const uint8_t *__restrict__ bg,
                       size_t bg_stride, HlGeom g, int polarity, const int *__restrict__ th_a, int lo, int hi,
                       uint8_t *__restrict__ diff, uint8_t *__restrict__ mask_a, uint8_t *__restrict__ mask_u,
                       uint8_t *__restrict__ mask_l)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const int d = hl_diff(bg[size_t(f) * bg_stride + p], frames[size_t(f) * frame_stride + p], polarity);
    const size_t o = size_t(f) * g.mstride + p;
    if (diff)
        diff[o] = uint8_t(d);
    mask_a[o] = d > th_a[f];
    mask_u[o] = d > hi;
    mask_l[o] = d > lo;
}

// 256-bin histogram of the difference image (only for threshold == -1, Otsu)
__global__ void __launch_bounds__(256)
    diff_hist_kernel(const uint8_t *__restrict__ frames, size_t frame_stride, const uint8_t *__restrict__ bg,
                     size_t bg_stride, HlGeom g, int polarity, unsigned int *__restrict__ hist)
{
    __shared__ unsigned int sh[256];
    const uint32_t f = blockIdx.z;
    sh[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < g.npix; p += gridDim.x * blockDim.x) {
        const int d = hl_diff(bg[size_t(f) * bg_stride + p], frames[size_t(f) * frame_stride + p], polarity);
        atomicAdd(&sh[d], 1u);
    }
    __syncthreads();
    if (sh[threadIdx.x])
        atomicAdd(&hist[f * 256 + threadIdx.x], sh[threadIdx.x]);
}

// OpenCV's Otsu threshold (getThreshVal_Otsu_8u), double arithmetic, first maximum wins (SURVEY.md 9.6)
__global__ void otsu_kernel(const unsigned int *__restrict__ hist, uint32_t npix, int *__restrict__ th_a, int nframes)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes)
        return;
    const unsigned int *h = hist + f * 256;
    const double scale = 1.0 / double(npix);
    double mu = 0;
    for (int i = 0; i < 256; ++i)
        mu += double(i) * double(h[i]);
    mu *= scale;
    double mu1 = 0, q1 = 0, max_sigma = 0;
    int max_val = 0;
    const double eps = 1.1920928955078125e-07; // FLT_EPSILON
    for (int i = 0; i < 256; ++i) {
        const double p_i = double(h[i]) * scale;
        mu1 *= q1;
        q1 += p_i;
        const double q2 = 1.0 - q1;
        if (fmin(q1, q2) < eps || fmax(q1, q2) > 1.0 - eps)
            continue;
        mu1 = (mu1 + double(i) * p_i) / q1;
        const double mu2 = (mu - q1 * mu1) / q2;
        const double sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2);
        if (sigma > max_sigma) {
            max_sigma = sigma;
            max_val = i;
        }
    }
    th_a[f] = max_val;
}

__global__ void fill_int_kernel(int *dst, int value, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        dst[i] = value;
}

// ------------------------------------------------------------------------------------------------------------------
// K3: erode / dilate with an arbitrary structuring element (offsets relative to the anchor)
// ------------------------------------------------------------------------------------------------------------------
template <bool ERODE>
__global__ void __launch_bounds__(256)
    morph_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, HlGeom g, const short2 *__restrict__ offs, int noffs)
{
    const uint32_t f = blockIdx.z;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= g.W)
        return;
    const uint8_t *s = src + size_t(f) * g.mstride;
    bool v = ERODE;
    for (int k = 0; k < noffs; ++k) {
        const int xx = x + offs[k].x, yy = y + offs[k].y;
        if (xx < 0 || yy < 0 || xx >= g.W || yy >= g.H)
            continue; // out-of-image samples never win (erode border = +inf, dilate border = -inf)
        const bool sv = s[yy * g.W + xx] != 0;
        if (ERODE)
            v = v && sv;
        else
            v = v || sv;
    }
    dst[size_t(f) * g.mstride + y * g.W + x] = v;
}

// ------------------------------------------------------------------------------------------------------------------
// K4: dual connected-component labelling
// ------------------------------------------------------------------------------------------------------------------
// init: one warp per image row; label = linear index of the first pixel of the pixel's horizontal run
__global__ void __launch_bounds__(256) ccl_init_kernel(const uint8_t *__restrict__ mask, uint32_t *__restrict__ lab, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (y >= g.H)
        return;
    const uint8_t *m = mask + size_t(f) * g.mstride + size_t(y) * g.W;
    uint32_t *l = lab + size_t(f) * g.lstride + size_t(y) * g.W;
    int carry_v = 3; // differs from every pixel value -> x = 0 starts a run
    int carry_s = 0;
    for (int xb = 0; xb < g.W; xb += 32) {
        const int x = xb + lane;
        const int v = x < g.W ? int(m[x] != 0) : 2;
        int lv = __shfl_up_sync(0xFFFFFFFFu, v, 1);
        if (lane == 0)
            lv = carry_v;
        const unsigned bits = __ballot_sync(0xFFFFFFFFu, v != lv);
        const unsigned mine = bits & (0xFFFFFFFFu >> (31 - lane));
        const int s = mine ? xb + 31 - __clz(mine) : carry_s;
        if (x < g.W)
            l[x] = uint32_t(y) * g.W + s;
        carry_s = __shfl_sync(0xFFFFFFFFu, s, 31);
        carry_v = __shfl_sync(0xFFFFFFFFu, v, 31);
    }
    if (y == 0 && lane == 0)
        lab[size_t(f) * g.lstride + g.npix] = g.npix; // the FRAME node
}

// merge: one union per vertical run overlap (reduced rules derived in DESIGN.md), plus the FRAME node
template <bool FG8, bool FRAME>
__global__ void __launch_bounds__(256) ccl_merge_kernel(const uint8_t *__restrict__ mask, uint32_t *__restrict__ lab, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= g.W)
        return;
    const uint8_t *m = mask + size_t(f) * g.mstride;
    uint32_t *l = lab + size_t(f) * g.lstride;
    const int W = g.W;
    const uint32_t p = uint32_t(y) * W + x;
    const bool v = m[p] != 0;
    // same-class tests; out-of-image neighbours belong to no class
    const bool d_same = x > 0 && (m[p - 1] != 0) == v; // left
    if (y > 0) {
        const bool b_same = (m[p - W] != 0) == v; // up
        const bool a_same = x > 0 && (m[p - W - 1] != 0) == v; // up-left
        if (v && FG8) {
            const bool c_same = x + 1 < W && (m[p - W + 1] != 0) == v; // up-right
            if (b_same) {
                if (!d_same)
                    uf_union(l, p, p - W);
            } else {
                if (a_same && !d_same)
                    uf_union(l, p, p - W - 1);
                if (c_same)
                    uf_union(l, p, p - W + 1);
            }
        } else {
            // 4-connectivity (background always, foreground when !FG8): first column of each vertical overlap
            if (b_same && !(d_same && a_same))
                uf_union(l, p, p - W);
        }
    }
    if (FRAME && !v) {
        // background on the image border belongs to the FRAME region: one union per border run / row end
        const bool top_or_bottom = (y == 0 || y == g.H - 1) && !d_same;
        const bool side = (x == 0) || (x == W - 1);
        if (top_or_bottom || side)
            uf_union(l, p, g.npix);
    }
}

__global__ void __launch_bounds__(256) ccl_flatten_kernel(uint32_t *__restrict__ lab, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > g.npix)
        return;
    uint32_t *l = lab + size_t(f) * g.lstride;
    l[p] = uf_find(l, p);
}

// canonical id of the background region at neighbour position (xx, yy) of a foreground pixel:
// outside the image or inside the FRAME region -> npix (the FRAME id); else the region's label
__device__ __forceinline__ uint32_t bg_id(const uint32_t *l, const HlGeom &g, int xx, int yy, uint32_t frame_root)
{
    if (xx < 0 || yy < 0 || xx >= g.W || yy >= g.H)
        return g.npix;
    const uint32_t r = l[yy * g.W + xx];
    return r == frame_root ? g.npix : r;
}

// ------------------------------------------------------------------------------------------------------------------
// K7: hysteresis
// ------------------------------------------------------------------------------------------------------------------
// lab_u: dual labels of U = d > hi (fg 8-conn, bg 4-conn, FRAME node).  lab_l: 4-conn labels of both values of
// L = d > lo (no FRAME node).  marks[] (u8, indexed by L label) must be zero on entry.
__global__ void __launch_bounds__(256)
    hyst_mark_kernel(const uint8_t *__restrict__ mask_u, const uint32_t *__restrict__ lab_u,
                     const uint32_t *__restrict__ lab_l, uint8_t *__restrict__ marks, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const uint32_t *lu = lab_u + size_t(f) * g.lstride;
    if (!mask_u[size_t(f) * g.mstride + p] || lu[p] != p)
        return; // only raster-first pixels of hi components are seeds (contour[0])
    const int x = int(p % uint32_t(g.W));
    // RETR_EXTERNAL: the component's outer background (left of its first pixel) must be the FRAME region
    const bool external = (x == 0) || (lu[p - 1] == lu[g.npix]);
    if (external)
        marks[size_t(f) * g.mstride + lab_l[size_t(f) * g.lstride + p]] = 1;
}

__global__ void __launch_bounds__(256)
    hyst_apply_kernel(const uint32_t *__restrict__ lab_l, const uint8_t *__restrict__ marks, uint8_t *__restrict__ out, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    out[size_t(f) * g.mstride + p] = marks[size_t(f) * g.mstride + lab_l[size_t(f) * g.lstride + p]];
}

__global__ void __launch_bounds__(256) zero_u8_kernel(uint8_t *__restrict__ dst, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (p < g.mstride)
        *reinterpret_cast<uint4 *>(dst + size_t(f) * g.mstride + p) = make_uint4(0, 0, 0, 0);
}

// ------------------------------------------------------------------------------------------------------------------
// K5/K6: remove small objects
// ------------------------------------------------------------------------------------------------------------------
// per root: zero the contour statistics, record link[] = outer background id (fg roots) / parent component (bg roots)
__global__ void __launch_bounds__(256)
    rso_roots_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, uint32_t *__restrict__ link,
                     int *__restrict__ st_s, int *__restrict__ st_e, int *__restrict__ st_x, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const uint32_t *l = lab + size_t(f) * g.lstride;
    if (l[p] != p)
        return;
    const size_t o = size_t(f) * g.lstride + p;
    st_s[o] = 0;
    st_e[o] = 0;
    st_x[o] = 0;
    const int x = int(p % uint32_t(g.W)), y = int(p / uint32_t(g.W));
    const uint32_t frame_root = l[g.npix];
    if (mask[size_t(f) * g.mstride + p]) {
        link[o] = bg_id(l, g, x - 1, y, frame_root); // b_out(C): region left of the raster-first pixel
    } else {
        // parent component of a hole: the foreground left of the hole's raster-first pixel.  For the FRAME
        // region (or a region touching x == 0) there is no parent.
        link[o] = (p == frame_root || x == 0) ? kNoLabel : l[p - 1];
    }
}

// per foreground pixel: crack sums / counts and convex corners, accumulated on the contour's owner:
// the component itself for its outer contour, the hole's background region for a hole contour
__global__ void __launch_bounds__(256)
    rso_stats_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, const uint32_t *__restrict__ link,
                     int *__restrict__ st_s, int *__restrict__ st_e, int *__restrict__ st_x, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= g.W)
        return;
    const uint8_t *m = mask + size_t(f) * g.mstride;
    const uint32_t p = uint32_t(y) * g.W + x;
    if (!m[p])
        return;
    const uint32_t *l = lab + size_t(f) * g.lstride;
    const size_t fo = size_t(f) * g.lstride;
    const uint32_t C = l[p];
    const uint32_t bout = link[fo + C];
    const uint32_t frame_root = l[g.npix];
    auto fgat = [&](int xx, int yy) { return xx >= 0 && yy >= 0 && xx < g.W && yy < g.H && m[yy * g.W + xx] != 0; };
    const bool fl = fgat(x - 1, y), fr = fgat(x + 1, y), fu = fgat(x, y - 1), fd = fgat(x, y + 1);
    auto owner = [&](uint32_t b) { return b == bout ? C : b; };
    if (!fl) {
        const uint32_t t = owner(bg_id(l, g, x - 1, y, frame_root));
        atomicAdd(&st_s[fo + t], -x);
        atomicAdd(&st_e[fo + t], 1);
    }
    if (!fr) {
        const uint32_t t = owner(bg_id(l, g, x + 1, y, frame_root));
        atomicAdd(&st_s[fo + t], x + 1);
        atomicAdd(&st_e[fo + t], 1);
    }
    if (!fu)
        atomicAdd(&st_e[fo + owner(bg_id(l, g, x, y - 1, frame_root))], 1);
    if (!fd)
        atomicAdd(&st_e[fo + owner(bg_id(l, g, x, y + 1, frame_root))], 1);
    // convex corners: 2x2 blocks in which this pixel is the only foreground pixel (the three background pixels of
    // such a block are 4-connected, so any of them names the region)
    if (!fl && !fu && !fgat(x - 1, y - 1))
        atomicAdd(&st_x[fo + owner(bg_id(l, g, x - 1, y, frame_root))], 1);
    if (!fr && !fu && !fgat(x + 1, y - 1))
        atomicAdd(&st_x[fo + owner(bg_id(l, g, x + 1, y, frame_root))], 1);
    if (!fl && !fd && !fgat(x - 1, y + 1))
        atomicAdd(&st_x[fo + owner(bg_id(l, g, x - 1, y, frame_root))], 1);
    if (!fr && !fd && !fgat(x + 1, y + 1))
        atomicAdd(&st_x[fo + owner(bg_id(l, g, x + 1, y, frame_root))], 1);
}

// per root: small flag (written over st_e): 2*area < 2*min_size
__global__ void __launch_bounds__(256)
    rso_small_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, const int *__restrict__ st_s,
                     int *__restrict__ st_e, const int *__restrict__ st_x, HlGeom g, int min_size)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const size_t o = size_t(f) * g.lstride + p;
    if (lab[o] != p)
        return;
    const long long s = st_s[o];
    const long long len = (long long)st_e[o] - st_x[o]; // chain length
    long long two_a;
    if (mask[size_t(f) * g.mstride + p])
        two_a = 2 * s - len - 2; // outer contour of a component (s > 0)
    else
        two_a = 2 * (s < 0 ? -s : s) + len - 2; // hole contour (s < 0)
    st_e[o] = (st_e[o] > 0 && two_a < 2ll * min_size) ? 1 : 0;
}

// per foreground root: parity of the number of consecutive small contours up the nesting chain (written to st_x)
__global__ void __launch_bounds__(256)
    rso_depth_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, const uint32_t *__restrict__ link,
                     const int *__restrict__ small, int *__restrict__ odd, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const size_t fo = size_t(f) * g.lstride;
    if (lab[fo + p] != p || !mask[size_t(f) * g.mstride + p])
        return;
    int count = 0;
    uint32_t cur = p;
    for (;;) {
        if (!small[fo + cur])
            break;
        ++count;
        const uint32_t b = link[fo + cur];
        if (b == g.npix) // outer background is the FRAME region: top of the chain
            break;
        if (!small[fo + b])
            break;
        ++count;
        const uint32_t par = link[fo + b];
        if (par == kNoLabel)
            break;
        cur = par;
    }
    odd[fo + p] = count & 1;
}

__global__ void __launch_bounds__(256)
    rso_apply_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, const uint32_t *__restrict__ link,
                     const int *__restrict__ small, const int *__restrict__ odd, uint8_t *__restrict__ out, HlGeom g)
{
    const uint32_t f = blockIdx.z;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= g.W)
        return;
    const uint8_t *m = mask + size_t(f) * g.mstride;
    const uint32_t p = uint32_t(y) * g.W + x;
    uint8_t keep = 0;
    if (m[p]) {
        const uint32_t *l = lab + size_t(f) * g.lstride;
        const size_t fo = size_t(f) * g.lstride;
        const uint32_t C = l[p];
        const uint32_t bout = link[fo + C];
        const uint32_t frame_root = l[g.npix];
        bool zero = odd[fo + C] != 0;
        auto edge = [&](int xx, int yy) {
            if (xx >= 0 && yy >= 0 && xx < g.W && yy < g.H && m[yy * g.W + xx] != 0)
                return;
            const uint32_t b = bg_id(l, g, xx, yy, frame_root);
            if (small[fo + (b == bout ? C : b)])
                zero = true;
        };
        edge(x - 1, y);
        edge(x + 1, y);
        edge(x, y - 1);
        edge(x, y + 1);
        keep = zero ? 0 : 1;
    }
    out[size_t(f) * g.mstride + p] = keep;
}

// ------------------------------------------------------------------------------------------------------------------
// K8/K9: hole fill and the final OR
// ------------------------------------------------------------------------------------------------------------------
// lab: labels of `mask` with a 4-connected background (no FRAME node).  filled = 1 everywhere except the background
// region containing the seed corner; all 1 when the seed pixel itself is set.
__global__ void __launch_bounds__(256)
    fill_apply_kernel(const uint8_t *__restrict__ mask, const uint32_t *__restrict__ lab, uint8_t *__restrict__ out, HlGeom g,
                      int accumulate_to_255)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.npix)
        return;
    const uint8_t *m = mask + size_t(f) * g.mstride;
    const uint32_t *l = lab + size_t(f) * g.lstride;
    const uint32_t seed = m[0] ? 0u : g.npix - 1u; // (0,0) if that pixel is set, else the bottom-right corner
    uint8_t v;
    if (m[seed])
        v = 1;
    else
        v = (m[p] != 0) || (l[p] != l[seed]);
    uint8_t *o = out + size_t(f) * g.mstride + p;
    if (accumulate_to_255)
        *o = ((*o != 0) || v) ? 255 : 0;
    else
        *o = v;
}

__global__ void __launch_bounds__(256)
    pack_out_kernel(const uint8_t *__restrict__ src, HlGeom g, uint8_t *__restrict__ dst, size_t dst_stride)
{
    const uint32_t f = blockIdx.z;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < g.npix)
        dst[size_t(f) * dst_stride + p] = src[size_t(f) * g.mstride + p];
}
} // namespace

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
namespace
{
void free_state(HighlightState *s)
{
    if (!s)
        return;
    void *ptrs[] = {s->d_bg, s->d_offs, s->m_a, s->m_u, s->m_l, s->m_t, s->m_out, s->lab0, s->lab1,
                    s->st_s, s->st_e, s->st_x, s->d_th, s->d_hist, s->d_in, s->d_res, s->d_comps, s->d_ncomps, s->d_labels,
                    s->d_cbg};
    for (void *p : ptrs)
        if (p)
            cudaFree(p);
    pool_dev_free(s->d_planes, s->planes_bytes);
    fused_release(s);
    delete s;
}

template <typename T>
int dev_alloc(cvvp_ctx *ctx, T **out, size_t count)
{
    if (cudaMalloc(reinterpret_cast<void **>(out), count * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, CVVP_ERR_NOMEM, "highlight: cudaMalloc of %zu bytes failed", count * sizeof(T));
    }
    return CVVP_OK;
}

struct Launcher {
    cvvp_ctx *ctx;
    cudaStream_t s;
    const HlGeom &g;
    unsigned nb; // frames in this batch
    dim3 per_pixel() const { return dim3((g.npix + 255) / 256, 1, nb); }
    dim3 per_pixel_plus_node() const { return dim3((g.npix + 1 + 255) / 256, 1, nb); }
    dim3 per_row_x() const { return dim3((g.W + 255) / 256, g.H, nb); }
    dim3 per_row_warp() const { return dim3((g.H + 7) / 8, 1, nb); }
};

// labels of `mask`; FG8: foreground 8-connected (else 4); FRAME: virtual frame node
template <bool FG8, bool FRAME>
void run_ccl(const Launcher &L, const uint8_t *mask, uint32_t *lab)
{
    ccl_init_kernel<<<L.per_row_warp(), 256, 0, L.s>>>(mask, lab, L.g);
    ccl_merge_kernel<FG8, FRAME><<<L.per_row_x(), 256, 0, L.s>>>(mask, lab, L.g);
    ccl_flatten_kernel<<<L.per_pixel_plus_node(), 256, 0, L.s>>>(lab, L.g);
    L.ctx->launches += 3;
}

void run_open(const Launcher &L, const HighlightState &st, uint8_t *mask, uint8_t *tmp)
{
    morph_kernel<true><<<L.per_row_x(), 256, 0, L.s>>>(mask, tmp, L.g, st.d_offs, st.noffs);
    morph_kernel<false><<<L.per_row_x(), 256, 0, L.s>>>(tmp, mask, L.g, st.d_offs, st.noffs);
    L.ctx->launches += 2;
}

// mask -> mask with small objects removed (in place; lab0/lab1/stats are scratch)
void run_rso(const Launcher &L, const HighlightState &st, uint8_t *mask, uint8_t *tmp, int min_size)
{
    run_ccl<true, true>(L, mask, st.lab0);
    rso_roots_kernel<<<L.per_pixel(), 256, 0, L.s>>>(mask, st.lab0, st.lab1, st.st_s, st.st_e, st.st_x, L.g);
    rso_stats_kernel<<<L.per_row_x(), 256, 0, L.s>>>(mask, st.lab0, st.lab1, st.st_s, st.st_e, st.st_x, L.g);
    rso_small_kernel<<<L.per_pixel(), 256, 0, L.s>>>(mask, st.lab0, st.st_s, st.st_e, st.st_x, L.g, min_size);
    rso_depth_kernel<<<L.per_pixel(), 256, 0, L.s>>>(mask, st.lab0, st.lab1, st.st_e, st.st_x, L.g);
    rso_apply_kernel<<<L.per_row_x(), 256, 0, L.s>>>(mask, st.lab0, st.lab1, st.st_e, st.st_x, tmp, L.g);
    L.ctx->launches += 5;
    cudaMemcpyAsync(mask, tmp, size_t(L.nb) * L.g.mstride, cudaMemcpyDeviceToDevice, L.s);
}

// out (accumulating) <- fill_holes(mask)
void run_fill(const Launcher &L, const HighlightState &st, const uint8_t *mask, uint8_t *out, bool accumulate)
{
    run_ccl<false, false>(L, mask, st.lab0);
    fill_apply_kernel<<<L.per_pixel(), 256, 0, L.s>>>(mask, st.lab0, out, L.g, accumulate ? 1 : 0);
    L.ctx->launches += 1;
}
} // namespace

void highlight_release(cvvp_ctx *ctx)
{
    free_state(ctx->hl);
    ctx->hl = nullptr;
}

size_t highlight_record_bytes(const cvvp_ctx *ctx)
{
    return ctx->hl && ctx->hl->component_stats ? sizeof(cvvp_component_stats) : sizeof(cvvp_component);
}

int highlight_job_channels(const cvvp_ctx *ctx)
{
    return ctx->hl ? ctx->hl->channels : 0;
}

bool highlight_geometry(const cvvp_ctx *ctx, int *width, int *height)
{
    if (!ctx->hl)
        return false;
    *width = ctx->hl->g.W;
    *height = ctx->hl->g.H;
    return true;
}

int highlight_begin(cvvp_ctx *ctx, const uint8_t *background, int width, int height, const uint8_t *selem, int kw, int kh,
                    int threshold, int threshold_lo, int threshold_hi, int min_size_hyst, int min_size_threshold)
{
    if (!background || !selem || width <= 0 || height <= 0 || kw <= 0 || kh <= 0)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: empty background or structuring element");
    if (kw > 255 || kh > 255)
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "highlight: structuring element larger than 255x255");
    if (size_t(width) * size_t(height) >= (1ull << 31))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "highlight: frame too large");
    highlight_release(ctx);
    HighlightState *st = new (std::nothrow) HighlightState();
    if (!st)
        return fail(ctx, CVVP_ERR_NOMEM, "out of host memory");
    ctx->hl = st;
    st->g.W = width;
    st->g.H = height;
    st->g.npix = uint32_t(width) * uint32_t(height);
    st->g.lstride = (st->g.npix + 1 + 3) & ~3u;
    st->g.mstride = (st->g.npix + 15) & ~15u;
    st->th = threshold;
    st->lo = threshold_lo;
    st->hi = threshold_hi;
    st->min_hyst = min_size_hyst;
    st->min_th = min_size_threshold;
    st->polarity = ctx->polarity; // the job keeps the polarity it began with
    st->channels = ctx->channels; // and its channel count
    if (st->channels > 1) {
        // the grey kernels read the job's d planes against a zero background, where BRIGHT gives max(d - 0, 0) = d
        st->color_polarity = st->polarity;
        st->polarity = CVVP_POLARITY_BRIGHT;
    }
    st->component_stats = ctx->component_stats; // and its component record size (highlight_record_bytes)
    // structuring element -> offsets relative to the anchor (kw/2, kh/2); any non-zero entry is set.  A kernel with
    // no non-zero entry is filtered by OpenCV as if only its element (0,0) were set.
    std::vector<short2> offs;
    const int ax = kw / 2, ay = kh / 2;
    for (int i = 0; i < kh; ++i)
        for (int j = 0; j < kw; ++j)
            if (selem[i * kw + j] != 0)
                offs.push_back(make_short2(short(j - ax), short(i - ay)));
    if (offs.empty())
        offs.push_back(make_short2(short(-ax), short(-ay)));
    st->noffs = int(offs.size());
    st->h_offs = offs;
    st->dy_min = offs.front().y;
    st->dy_max = offs.back().y;
    int rc;
    const bool color = st->channels > 1;
    const size_t bg_bytes = size_t(st->g.npix) * size_t(st->channels);
    if ((rc = dev_alloc(ctx, &st->d_bg, st->g.npix)) != CVVP_OK || (rc = dev_alloc(ctx, &st->d_offs, offs.size())) != CVVP_OK ||
        (color && (rc = dev_alloc(ctx, &st->d_cbg, bg_bytes)) != CVVP_OK)) {
        highlight_release(ctx);
        return rc;
    }
    cudaError_t e;
    if ((e = color ? cudaMemcpy(st->d_cbg, background, bg_bytes, cudaMemcpyHostToDevice) : cudaSuccess) != cudaSuccess ||
        (e = color ? cudaMemset(st->d_bg, 0, st->g.npix) : cudaMemcpy(st->d_bg, background, st->g.npix, cudaMemcpyHostToDevice)) !=
            cudaSuccess ||
        (e = cudaMemcpy(st->d_offs, offs.data(), offs.size() * sizeof(short2), cudaMemcpyHostToDevice)) != cudaSuccess) {
        highlight_release(ctx);
        return fail(ctx, CVVP_ERR_CUDA, "highlight: upload failed: %s", cudaGetErrorString(e));
    }
    return CVVP_OK;
}

static int ensure_batch(cvvp_ctx *ctx, HighlightState *st, int nb)
{
    if (nb <= st->batch_cap)
        return CVVP_OK;
    void **bufs[] = {(void **)&st->m_a, (void **)&st->m_u, (void **)&st->m_l, (void **)&st->m_t, (void **)&st->m_out,
                     (void **)&st->lab0, (void **)&st->lab1, (void **)&st->st_s, (void **)&st->st_e, (void **)&st->st_x};
    for (void **b : bufs) {
        if (*b)
            cudaFree(*b);
        *b = nullptr;
    }
    st->batch_cap = 0;
    const size_t m = size_t(nb) * st->g.mstride, l = size_t(nb) * st->g.lstride;
    int rc;
    if ((rc = dev_alloc(ctx, &st->m_a, m)) || (rc = dev_alloc(ctx, &st->m_u, m)) || (rc = dev_alloc(ctx, &st->m_l, m)) ||
        (rc = dev_alloc(ctx, &st->m_t, m)) || (rc = dev_alloc(ctx, &st->m_out, m)) || (rc = dev_alloc(ctx, &st->lab0, l)) ||
        (rc = dev_alloc(ctx, &st->lab1, l)) || (rc = dev_alloc(ctx, &st->st_s, l)) || (rc = dev_alloc(ctx, &st->st_e, l)) ||
        (rc = dev_alloc(ctx, &st->st_x, l)))
        return rc;
    st->batch_cap = nb;
    return CVVP_OK;
}

// per-frame thresholds of branch A for nb frames -> st->d_th: the constant, or Otsu's per frame (threshold == -1, :89-95)
int highlight_thresholds(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                         size_t bg_stride, unsigned nb, cudaStream_t stream)
{
    if (int(nb) > st->th_cap) {
        // the previous arrays may still be in use by work queued on `stream`
        cudaStreamSynchronize(stream);
        if (st->d_th) cudaFree(st->d_th);
        if (st->d_hist) cudaFree(st->d_hist);
        st->d_th = nullptr;
        st->d_hist = nullptr;
        st->th_cap = 0;
        int rc;
        if ((rc = dev_alloc(ctx, &st->d_th, size_t(nb))) || (rc = dev_alloc(ctx, &st->d_hist, size_t(nb) * 256)))
            return rc;
        st->th_cap = int(nb);
    }
    if (st->th == -1) {
        cudaMemsetAsync(st->d_hist, 0, size_t(nb) * 256 * sizeof(unsigned int), stream);
        diff_hist_kernel<<<dim3(64, 1, nb), 256, 0, stream>>>(in, frame_stride, bg, bg_stride, st->g, st->polarity,
                                                              st->d_hist);
        otsu_kernel<<<(nb + 63) / 64, 64, 0, stream>>>(st->d_hist, st->g.npix, st->d_th, int(nb));
        ctx->launches += 2;
    } else {
        fill_int_kernel<<<(nb + 255) / 256, 256, 0, stream>>>(st->d_th, st->th, int(nb));
        ctx->launches += 1;
    }
    return CVVP_OK;
}

// per-pixel path: frames per launch batch: enough work to fill the GPU, bounded scratch (~37 bytes per pixel per frame)
static int pick_batch(const HighlightState *st, long long n)
{
    const long long by_mem = (3ll << 30) / (37ll * st->g.npix + 64);
    long long b = 32ll * 1024 * 1024 / st->g.npix + 1; // ~32 Mpx per launch: the ~35 launches of a batch amortise
    if (b < 1) b = 1;
    if (b > by_mem) b = by_mem > 0 ? by_mem : 1;
    if (b > 4096) b = 4096;
    if (b > n) b = n;
    return int(b);
}

static int highlight_pixels(cvvp_ctx *ctx, HighlightState *st, const uint8_t *d_frames, long long n, size_t frame_stride,
                            const uint8_t *d_bg, size_t bg_stride, uint8_t *d_out, size_t out_stride, cudaStream_t stream)
{
    const int bcap = pick_batch(st, n);
    int rc = ensure_batch(ctx, st, bcap);
    if (rc != CVVP_OK)
        return rc;
    for (long long done = 0; done < n; done += bcap) {
        const unsigned nb = unsigned(n - done < bcap ? n - done : bcap);
        const uint8_t *in = d_frames + size_t(done) * frame_stride;
        const uint8_t *bg = d_bg + size_t(done) * bg_stride;
        Launcher L{ctx, stream, st->g, nb};
        if ((rc = highlight_thresholds(ctx, st, in, frame_stride, bg, bg_stride, nb, stream)) != CVVP_OK)
            return rc;
        diff_thresh_kernel<<<L.per_pixel(), 256, 0, stream>>>(in, frame_stride, bg, bg_stride, st->g, st->polarity,
                                                              st->d_th, st->lo, st->hi, nullptr, st->m_a, st->m_u,
                                                              st->m_l);
        ctx->launches += 1;
        // ---- branch A: threshold -> open -> remove small -> fill holes
        run_open(L, *st, st->m_a, st->m_t);
        run_rso(L, *st, st->m_a, st->m_t, st->min_th);
        run_fill(L, *st, st->m_a, st->m_out, false);
        // ---- branch B: hysteresis -> open -> remove small -> fill holes
        run_ccl<true, true>(L, st->m_u, st->lab0);
        run_ccl<false, false>(L, st->m_l, st->lab1);
        zero_u8_kernel<<<dim3((st->g.mstride / 16 + 255) / 256, 1, nb), 256, 0, stream>>>(st->m_t, st->g);
        hyst_mark_kernel<<<L.per_pixel(), 256, 0, stream>>>(st->m_u, st->lab0, st->lab1, st->m_t, st->g);
        hyst_apply_kernel<<<L.per_pixel(), 256, 0, stream>>>(st->lab1, st->m_t, st->m_u, st->g);
        ctx->launches += 3;
        run_open(L, *st, st->m_u, st->m_t);
        run_rso(L, *st, st->m_u, st->m_t, st->min_hyst);
        run_fill(L, *st, st->m_u, st->m_out, true); // out = 255 * (A | B)
        pack_out_kernel<<<L.per_pixel(), 256, 0, stream>>>(st->m_out, st->g, d_out + size_t(done) * out_stride, out_stride);
        ctx->launches += 1;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess)
            return fail(ctx, CVVP_ERR_CUDA, "highlight: kernel launch failed: %s", cudaGetErrorString(e));
    }
    return CVVP_OK;
}

static bool use_fused(const HighlightState *st)
{
    return st->path == kPathFused && fused_supports(st);
}

int highlight_set_path(cvvp_ctx *ctx, int path)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    if (path != kPathFused && path != kPathPixel)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: unknown device path %d", path);
    st->path = path;
    return CVVP_OK;
}

int highlight_frames_in_flight(cvvp_ctx *ctx, int *out_frames)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    *out_frames = fused_supports(st) ? fused_frames_in_flight(ctx, st) : 0;
    return CVVP_OK;
}

// n >= 1 validated frames; frame f against the background at d_bg + f * bg_stride (0: one background for all)
static int highlight_run(cvvp_ctx *ctx, HighlightState *st, const uint8_t *d_frames, long long n, size_t frame_stride,
                         const uint8_t *d_bg, size_t bg_stride, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                         cudaStream_t stream)
{
    if (!use_fused(st))
        return highlight_pixels(ctx, st, d_frames, n, frame_stride, d_bg, bg_stride, d_out, out_stride, stream);
    // fused path: one launch per (up to) 2^20 frames; scratch is per resident CTA, not per frame
    const long long bmax = 1ll << 20;
    for (long long done = 0; done < n; done += bmax) {
        const unsigned nb = unsigned(n - done < bmax ? n - done : bmax);
        const uint8_t *in = d_frames + size_t(done) * frame_stride;
        const uint8_t *bg = d_bg + size_t(done) * bg_stride;
        int rc;
        if (st->th == -1 && (rc = highlight_thresholds(ctx, st, in, frame_stride, bg, bg_stride, nb, stream)) != CVVP_OK)
            return rc;
        if ((rc = highlight_fused_batch(ctx, st, in, frame_stride, bg, bg_stride, nb, d_out + size_t(done) * out_stride,
                                        out_stride, cc, stream)) != CVVP_OK)
            return rc;
    }
    return CVVP_OK;
}

// the component outputs of frames [first, ...) of cc
static CcOut cc_from(const CcOut &cc, long long first)
{
    CcOut o = cc;
    if (o.comps)
        o.comps = reinterpret_cast<cvvp_component *>(reinterpret_cast<uint8_t *>(o.comps) +
                                                     size_t(first) * size_t(o.max_comps) * o.rec_bytes);
    if (o.ncomps)
        o.ncomps += first;
    if (o.labels)
        o.labels += size_t(first) * o.labels_stride;
    return o;
}

// Colour job: the d planes of a chunk of frames go into the job's scratch (highlight_color.cu), then the grey path
// runs on them against the zero background.  Chunks hold the frames one launch keeps in flight, so that splitting
// the call costs the kernels no occupancy; at most about 1 GB of scratch.
static int highlight_color_run(cvvp_ctx *ctx, HighlightState *st, const uint8_t *d_frames, long long n, size_t frame_stride,
                               const uint8_t *d_bgs, size_t bg_stride, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                               cudaStream_t stream)
{
    const size_t pitch = round_up(st->g.npix, 128);
    long long chunk = use_fused(st) ? fused_frames_in_flight(ctx, st) : pick_batch(st, n);
    const long long by_mem = (long long)((size_t(1) << 30) / pitch);
    if (chunk > by_mem) chunk = by_mem;
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    if (st->planes_bytes < size_t(chunk) * pitch) {
        // work queued earlier on this stream may still read the old scratch
        CVVP_CUDA_OK(ctx, cudaStreamSynchronize(stream));
        pool_dev_free(st->d_planes, st->planes_bytes);
        st->d_planes = nullptr;
        st->planes_bytes = 0;
        void *p = nullptr;
        if (pool_dev_alloc(&p, size_t(chunk) * pitch) != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CVVP_ERR_NOMEM, "highlight: allocation of %lld difference planes failed", chunk);
        }
        st->d_planes = static_cast<uint8_t *>(p);
        st->planes_bytes = size_t(chunk) * pitch;
    }
    for (long long done = 0; done < n; done += chunk) {
        const long long nb = n - done < chunk ? n - done : chunk;
        int rc = highlight_color_d(ctx, d_frames + size_t(done) * frame_stride, nb, frame_stride, 0, 0,
                                   d_bgs + size_t(done) * bg_stride, bg_stride, st->d_planes, pitch, stream);
        if (rc == CVVP_OK)
            rc = highlight_run(ctx, st, st->d_planes, nb, pitch, st->d_bg, 0, d_out + size_t(done) * out_stride, out_stride,
                               cc_from(cc, done), stream);
        if (rc != CVVP_OK)
            return rc;
    }
    return CVVP_OK;
}

static_assert(sizeof(cvvp_component) == 48, "cvvp_component is part of the C ABI (include/cvvp.h, _cabi.COMPONENT_DTYPE)");
static_assert(sizeof(cvvp_component_stats) == 104 && offsetof(cvvp_component_stats, c) == 0,
              "cvvp_component_stats is part of the C ABI (include/cvvp.h, _cabi.COMPONENT_STATS_DTYPE)");

// [p, p + (n - 1) * p_stride + p_bytes) and [q, q + (n - 1) * q_stride + q_bytes) share a byte
static bool frames_overlap(const uint8_t *p, size_t p_stride, size_t p_bytes, const uint8_t *q, size_t q_stride,
                           size_t q_bytes, long long n)
{
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(p), b0 = reinterpret_cast<uintptr_t>(q);
    const uintptr_t a1 = a0 + size_t(n - 1) * p_stride + p_bytes, b1 = b0 + size_t(n - 1) * q_stride + q_bytes;
    return a0 < b1 && b0 < a1;
}

int highlight_check_cc(cvvp_ctx *ctx, long long n, const CcOut &cc)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    if (!cc.comps || !cc.ncomps || cc.max_comps < 1 || (cc.labels && cc.labels_stride < st->g.npix))
        return fail(ctx, CVVP_ERR_INVALID, "highlight components: bad arguments");
    if (!use_fused(st))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "highlight components: only the fused path labels the final masks");
    if (n > (1ll << 20))
        return fail(ctx, CVVP_ERR_UNSUPPORTED, "highlight components: at most 2^20 frames per call");
    return CVVP_OK;
}

int highlight_device_bg(cvvp_ctx *ctx, const uint8_t *d_frames, long long n, size_t frame_stride, const uint8_t *d_bgs,
                        size_t bg_stride, uint8_t *d_out, size_t out_stride, const CcOut &cc, cudaStream_t stream)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    const size_t fb = size_t(st->g.npix) * size_t(st->channels); // bytes of a frame and of a background
    if (!d_frames || !d_out || n < 0 || frame_stride < fb || out_stride < st->g.npix || (bg_stride != 0 && bg_stride < fb))
        return fail(ctx, CVVP_ERR_INVALID, "highlight: bad arguments (bg_stride must be 0 or at least %zu)", fb);
    const bool want_cc = cc.comps || cc.ncomps || cc.labels;
    if (want_cc) {
        const int rc = highlight_check_cc(ctx, n, cc);
        if (rc != CVVP_OK)
            return rc;
    }
    if (n == 0)
        return CVVP_OK;
    const bool color = st->channels > 1;
    if (!d_bgs) {
        d_bgs = color ? st->d_cbg : st->d_bg;
        bg_stride = 0;
    }
    const size_t np = st->g.npix;
    // a colour job's d is computed chunk by chunk ahead of the masks: a mask must not land on a frame still to be read
    if (color && (frames_overlap(d_out, out_stride, np, d_frames, frame_stride, fb, n) ||
                  frames_overlap(d_out, out_stride, np, d_bgs, bg_stride, fb, n)))
        return fail(ctx, CVVP_ERR_INVALID, "highlight: d_out overlaps the frames or the backgrounds");
    CcOut job_cc = want_cc ? cc : CcOut();
    if (want_cc && st->component_stats) {
        // the statistics read frame and background bytes after the kernel has written the frame's mask
        if (frames_overlap(d_out, out_stride, np, d_frames, frame_stride, np, n) ||
            frames_overlap(d_out, out_stride, np, d_bgs, bg_stride, np, n))
            return fail(ctx, CVVP_ERR_INVALID,
                        "highlight component statistics: d_out overlaps the frames or the backgrounds");
        job_cc.rec_bytes = sizeof(cvvp_component_stats);
    }
    if (color)
        return highlight_color_run(ctx, st, d_frames, n, frame_stride, d_bgs, bg_stride, d_out, out_stride, job_cc, stream);
    return highlight_run(ctx, st, d_frames, n, frame_stride, d_bgs, bg_stride, d_out, out_stride, job_cc, stream);
}

int highlight_color_d(cvvp_ctx *ctx, const uint8_t *src, long long n, size_t frame_stride, size_t row_stride, int x0,
                      const uint8_t *d_bgs, size_t bg_stride, uint8_t *d_planes, size_t pitch, cudaStream_t stream)
{
    const HighlightState *st = ctx->hl;
    if (!d_bgs) {
        d_bgs = st->d_cbg;
        bg_stride = 0;
    }
    const bool rows = row_stride != 0;
    return color_diff_launch(ctx, st->channels, st->color_polarity, src, n, frame_stride, row_stride, x0, d_bgs, bg_stride,
                             rows ? uint32_t(st->g.W) : st->g.npix, rows ? uint32_t(st->g.H) : 1u, d_planes, pitch, stream);
}

int highlight_device_planes(cvvp_ctx *ctx, const uint8_t *d_planes, long long n, size_t pitch, uint8_t *d_out,
                            size_t out_stride, const CcOut &cc, cudaStream_t stream)
{
    HighlightState *st = ctx->hl;
    const bool want_cc = cc.comps || cc.ncomps || cc.labels;
    if (want_cc) {
        const int rc = highlight_check_cc(ctx, n, cc);
        if (rc != CVVP_OK)
            return rc;
    }
    CcOut job_cc = want_cc ? cc : CcOut();
    if (want_cc && st->component_stats)
        job_cc.rec_bytes = sizeof(cvvp_component_stats);
    return highlight_run(ctx, st, d_planes, n, pitch, st->d_bg, 0, d_out, out_stride, job_cc, stream);
}

template <typename T>
static int grow(cvvp_ctx *ctx, T **p, size_t *cap, size_t need)
{
    if (*cap >= need)
        return CVVP_OK;
    if (*p)
        cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    if (cudaMalloc(reinterpret_cast<void **>(p), need * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, CVVP_ERR_NOMEM, "highlight components: cudaMalloc of %zu bytes failed", need * sizeof(T));
    }
    *cap = need;
    return CVVP_OK;
}

// Host-buffer form with components: chunks run one after another (H2D, one kernel launch, D2H); the label images
// quadruple the D2H volume, so this entry point is for callers that want the labels more than the last GB/s.
int highlight_frames_host_cc(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                             size_t out_stride, cvvp_component *comps_out, int max_comps, int *ncomps_out,
                             int32_t *labels_out, size_t labels_stride)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    const size_t np = st->g.npix;
    const size_t fb = np * size_t(st->channels); // bytes of a frame
    if (!frames || !masks_out || !comps_out || !ncomps_out || max_comps < 1 || n < 0 || frame_stride < fb ||
        out_stride < np || (labels_out && labels_stride < np))
        return fail(ctx, CVVP_ERR_INVALID, "highlight components: bad arguments");
    if (n == 0)
        return CVVP_OK;
    const size_t pitch = round_up(fb, 128); // of the frames on the device; the masks keep it too
    long long chunk = fused_supports(st) ? fused_frames_in_flight(ctx, st) : 16;
    if (chunk > n)
        chunk = n;
    int rc;
    if (st->in_bytes < size_t(chunk) * pitch) {
        if (st->d_in) cudaFree(st->d_in);
        if (st->d_res) cudaFree(st->d_res);
        st->d_in = st->d_res = nullptr;
        st->in_bytes = 0;
        if ((rc = dev_alloc(ctx, &st->d_in, 2 * size_t(chunk) * pitch)) || (rc = dev_alloc(ctx, &st->d_res, 2 * size_t(chunk) * pitch)))
            return rc;
        st->in_bytes = size_t(chunk) * pitch;
    }
    const size_t rec = highlight_record_bytes(ctx);
    if ((rc = grow(ctx, &st->d_comps, &st->comps_cap, size_t(chunk) * size_t(max_comps) * rec)) ||
        (rc = grow(ctx, &st->d_ncomps, &st->ncomps_cap, size_t(chunk))) ||
        (labels_out && (rc = grow(ctx, &st->d_labels, &st->labels_cap, size_t(chunk) * np))))
        return rc;
    cudaStream_t s = ctx->compute;
    for (long long done = 0; done < n; done += chunk) {
        const long long nb = n - done < chunk ? n - done : chunk;
        CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(st->d_in, pitch, frames + size_t(done) * frame_stride, frame_stride, fb, size_t(nb),
                                            cudaMemcpyHostToDevice, s));
        rc = highlight_device_bg(ctx, st->d_in, nb, pitch, nullptr, 0, st->d_res, pitch,
                                 CcOut{reinterpret_cast<cvvp_component *>(st->d_comps), max_comps, st->d_ncomps,
                                       labels_out ? st->d_labels : nullptr, np},
                                 s);
        if (rc != CVVP_OK)
            return rc;
        CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(masks_out + size_t(done) * out_stride, out_stride, st->d_res, pitch, np, size_t(nb),
                                            cudaMemcpyDeviceToHost, s));
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(reinterpret_cast<uint8_t *>(comps_out) + size_t(done) * max_comps * rec,
                                          st->d_comps, size_t(nb) * max_comps * rec, cudaMemcpyDeviceToHost, s));
        CVVP_CUDA_OK(ctx, cudaMemcpyAsync(ncomps_out + done, st->d_ncomps, size_t(nb) * sizeof(int), cudaMemcpyDeviceToHost, s));
        if (labels_out)
            CVVP_CUDA_OK(ctx, cudaMemcpy2DAsync(labels_out + size_t(done) * labels_stride, labels_stride * sizeof(int32_t),
                                                st->d_labels, np * sizeof(int32_t), np * sizeof(int32_t), size_t(nb),
                                                cudaMemcpyDeviceToHost, s));
        CVVP_CUDA_OK(ctx, cudaStreamSynchronize(s));
    }
    return CVVP_OK;
}

int highlight_frames_host(cvvp_ctx *ctx, const uint8_t *frames, long long n, size_t frame_stride, uint8_t *masks_out,
                          size_t out_stride)
{
    HighlightState *st = ctx->hl;
    if (!st)
        return fail(ctx, CVVP_ERR_STATE, "highlight: no parameters set (call cvvp_highlight_begin first)");
    const size_t np = st->g.npix;
    const size_t fb = np * size_t(st->channels); // bytes of a frame
    if (!frames || !masks_out || n < 0 || frame_stride < fb || out_stride < np)
        return fail(ctx, CVVP_ERR_INVALID, "highlight: bad arguments");
    if (n == 0)
        return CVVP_OK;
    // chunked, three streams: H2D on `copy`, kernels on `compute`, D2H on `copy_out`, so that both directions of
    // the link stay busy while a chunk is computed.  The device side is far faster than the link, so chunks are
    // sized for the copies (about n/32 frames, at most one frame per resident CTA) rather than for the kernel: the
    // first chunk's upload and the last chunk's download are the only copies that nothing overlaps.
    long long chunk;
    if (use_fused(st)) {
        const long long slots = fused_frames_in_flight(ctx, st);
        chunk = (n + 31) / 32;
        if (chunk < 16) chunk = 16;
        if (chunk > slots) chunk = slots;
        if (chunk > n) chunk = n;
    } else {
        chunk = pick_batch(st, n);
    }
    // device frame pitch: keeps every frame 16-byte aligned (the masks keep the frames' pitch)
    const size_t pitch = round_up(fb, 128);
    const size_t need = size_t(chunk) * pitch;
    if (st->in_bytes < need) {
        if (st->d_in) cudaFree(st->d_in);
        if (st->d_res) cudaFree(st->d_res);
        st->d_in = st->d_res = nullptr;
        st->in_bytes = 0;
        int rc;
        if ((rc = dev_alloc(ctx, &st->d_in, 2 * need)) || (rc = dev_alloc(ctx, &st->d_res, 2 * need)))
            return rc;
        st->in_bytes = need;
    }
    const size_t half = st->in_bytes;
    cudaEvent_t up[2] = {nullptr, nullptr}, kdone[2] = {nullptr, nullptr}, down[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&up[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&kdone[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&down[i], cudaEventDisableTiming);
    }
    int rc = CVVP_OK;
    long long idx = 0;
    for (long long done = 0; done < n && rc == CVVP_OK; done += chunk, ++idx) {
        const long long nb = n - done < chunk ? n - done : chunk;
        const int b = int(idx & 1);
        uint8_t *din = st->d_in + size_t(b) * half;
        uint8_t *dres = st->d_res + size_t(b) * half;
        if (idx >= 2)
            cudaStreamWaitEvent(ctx->copy, kdone[b], 0); // the kernel that read this input half has finished
        cudaError_t e = cudaMemcpy2DAsync(din, pitch, frames + size_t(done) * frame_stride, frame_stride, fb, size_t(nb),
                                          cudaMemcpyHostToDevice, ctx->copy);
        if (e != cudaSuccess) {
            rc = fail(ctx, CVVP_ERR_CUDA, "highlight: H2D failed: %s", cudaGetErrorString(e));
            break;
        }
        cudaEventRecord(up[b], ctx->copy);
        cudaStreamWaitEvent(ctx->compute, up[b], 0);
        if (idx >= 2)
            cudaStreamWaitEvent(ctx->compute, down[b], 0); // this result half's previous masks have left the device
        rc = highlight_device_bg(ctx, din, nb, pitch, nullptr, 0, dres, pitch, CcOut(), ctx->compute);
        if (rc != CVVP_OK)
            break;
        cudaEventRecord(kdone[b], ctx->compute);
        cudaStreamWaitEvent(ctx->copy_out, kdone[b], 0);
        e = cudaMemcpy2DAsync(masks_out + size_t(done) * out_stride, out_stride, dres, pitch, np, size_t(nb),
                              cudaMemcpyDeviceToHost, ctx->copy_out);
        if (e != cudaSuccess) {
            rc = fail(ctx, CVVP_ERR_CUDA, "highlight: D2H failed: %s", cudaGetErrorString(e));
            break;
        }
        cudaEventRecord(down[b], ctx->copy_out);
    }
    cudaError_t e1 = cudaStreamSynchronize(ctx->copy);
    cudaError_t e2 = cudaStreamSynchronize(ctx->compute);
    cudaError_t e3 = cudaStreamSynchronize(ctx->copy_out);
    for (int i = 0; i < 2; ++i) {
        cudaEventDestroy(up[i]);
        cudaEventDestroy(kdone[i]);
        cudaEventDestroy(down[i]);
    }
    if (e1 == cudaSuccess)
        e1 = e2 != cudaSuccess ? e2 : e3;
    if (rc == CVVP_OK && e1 != cudaSuccess)
        rc = fail(ctx, CVVP_ERR_CUDA, "highlight: execution failed: %s", cudaGetErrorString(e1));
    return rc;
}
} // namespace cvvp
