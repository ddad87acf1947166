// State of a highlight job (parameters of TokenProcessorPack<HighlightObjectsAlgo>,
// /root/reference/Sources/ProcessorAlgos/highlight_objects_algo.h:21-32, plus device scratch).  Shared by the two
// device implementations: highlight_fused.cu (the product path: one persistent CTA per frame) and highlight.cu
// (per-pixel kernels: the first implementation, kept as an on-device cross-check and for frames whose geometry the
// run records cannot encode).
#pragma once
#include "context.hpp"

#include <vector>

namespace cvvp
{
struct HlGeom {
    int W, H;
    uint32_t npix;    // W * H
    uint32_t lstride; // label-array stride per frame (npix + 1, padded to 4)
    uint32_t mstride; // mask stride per frame (npix padded to 16)
};

enum HighlightPath { kPathFused = 0, kPathPixel = 1 };

struct FusedScratch {
    int slots{0};            // resident CTAs the scratch was sized for
    uint32_t *bits{nullptr};   // [slots][kFusedImages][nwords]
    uint32_t *runs{nullptr};   // [slots][kFusedRunArrays][cap]
    uint32_t *rowoff{nullptr}; // [slots][2][rstride]
    unsigned *queue{nullptr};  // frame queue counters (one per launch in flight, ring of kQueueRing)
    unsigned queue_next{0};
    size_t bits_bytes{0}, runs_bytes{0}, rowoff_bytes{0}; // sizes of the pooled allocations above (pool.hpp)
};

// d of one pixel in a polarity (CVVP_POLARITY_*): bg - frame, frame - bg, or |frame - bg|, saturated to 0..255
// (highlight_objects_algo.cpp:27-30)
__device__ __forceinline__ int hl_diff(int bg, int fr, int polarity)
{
    const int s = bg - fr;
    return polarity == CVVP_POLARITY_DARK ? max(s, 0) : polarity == CVVP_POLARITY_BRIGHT ? max(-s, 0) : abs(s);
}

struct HighlightState {
    HlGeom g{};
    int th{}, lo{}, hi{}, min_hyst{}, min_th{};
    // polarity of the grey kernels' difference: the context's polarity when the job began (cvvp_highlight_set_polarity),
    // except for a colour job, whose kernels read its d planes against the zero d_bg in BRIGHT (highlight_color.cu)
    int polarity{CVVP_POLARITY_DARK};
    int channels{1};                    // the context's cvvp_highlight_set_channels when the job began
    int color_polarity{CVVP_POLARITY_DARK}; // colour job: the polarity its d planes are computed in
    int component_stats{0}; // the context's cvvp_highlight_set_component_stats when the job began
    int noffs{0};
    int dy_min{0}, dy_max{0}; // row range of the structuring element's taps (offsets are sorted by row, then column)
    int path{kPathFused};
    uint8_t *d_bg{nullptr}; // the background; all zero for a colour job
    uint8_t *d_cbg{nullptr}; // colour job: the background, npix * channels bytes
    // colour job: d planes of a chunk of frames (pooled, pool.hpp).  Like the fused kernel's scratch, it is reused in
    // stream order on the call's stream: work in flight on a context's highlight scratch is on one stream at a time.
    uint8_t *d_planes{nullptr};
    size_t planes_bytes{0};
    short2 *d_offs{nullptr};
    std::vector<short2> h_offs; // host copy of the taps
    // per-pixel path: per-batch work buffers
    int batch_cap{0};
    uint8_t *m_a{nullptr}, *m_u{nullptr}, *m_l{nullptr}, *m_t{nullptr}, *m_out{nullptr};
    uint32_t *lab0{nullptr}, *lab1{nullptr};
    int *st_s{nullptr}, *st_e{nullptr}, *st_x{nullptr};
    // Otsu (threshold == -1): per-frame thresholds of the batch
    int th_cap{0};
    int *d_th{nullptr};
    unsigned int *d_hist{nullptr};
    // fused path
    int fused_variant{-1}; // which build of the fused kernel the job uses: 0 = 1024-thread CTAs, 1 = 256-thread CTAs, -1 = not chosen yet
    FusedScratch fs;
    // staging of the host-buffer component entry point
    uint8_t *d_comps{nullptr}; // component records of the job's size (highlight_record_bytes)
    int *d_ncomps{nullptr};
    int32_t *d_labels{nullptr};
    size_t comps_cap{0}, ncomps_cap{0}, labels_cap{0};
    // staging for the host-buffer entry point
    uint8_t *d_in{nullptr}, *d_res{nullptr};
    size_t in_bytes{0};
};

// highlight.cu
// bg: background of the batch's first frame, frame f's at bg + f * bg_stride (0 = one background for every frame)
int highlight_thresholds(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                         size_t bg_stride, unsigned nb, cudaStream_t stream);
// highlight_fused.cu
bool fused_supports(const HighlightState *st);
void fused_release(HighlightState *st);
int fused_frames_in_flight(cvvp_ctx *ctx, HighlightState *st);
// cc: component output of the final masks (comps == nullptr: off)
int highlight_fused_batch(cvvp_ctx *ctx, HighlightState *st, const uint8_t *in, size_t frame_stride, const uint8_t *bg,
                          size_t bg_stride, unsigned nb, uint8_t *d_out, size_t out_stride, const CcOut &cc,
                          cudaStream_t stream);
} // namespace cvvp
