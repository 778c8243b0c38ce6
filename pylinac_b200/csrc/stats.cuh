// Frame-statistics kernel interface (internal).
#pragma once
#include "common.cuh"

namespace epid {

constexpr int STATS_THREADS = 1024;
constexpr int STATS_MAX_RANKS = 16;
constexpr int STATS_MAX_DIM = 4096;  // rows / columns of the analysed view

// A frame view in HBM: `origin` points at pixel (0,0) of the analysed view (crop is a pointer offset,
// core/image.py:714-745), `pitch` = elements between rows.  If pitch % 8 == 0 the 8-pixel vectors of every row
// share one misalignment (origin address / 2) % 8 and 128-bit loads are legal on the aligned grid.
struct FrameRef {
    const uint16_t* origin;
    int pitch;
    int pad;
};

struct StatsGeom {   // identical for every frame of one launch
    int H, W;        // view size
    int vprp;        // (max) vectors per row, rounded up to a multiple of 32
    int groups;      // row groups handled concurrently = STATS_THREADS / vprp
    // corner boxes of BaseImage.check_inversion (core/image.py:881-894); box <= 0 disables
    int box, rp, cp;
    int nranks;
    uint32_t ranks[STATS_MAX_RANKS];  // 0-based order-statistic indices, ascending not required
};

struct FrameStats {  // per frame, device memory
    uint32_t mn, mx;
    uint32_t npix;
    uint32_t overflow;           // packed-u16 histogram overflowed -> needs the MODE 1 re-run
    unsigned long long sum;
    unsigned long long corner_sum;  // sum over the four corner boxes
    uint32_t ostat[STATS_MAX_RANKS];
};

int make_stats_geom(StatsGeom* g, int H, int W);

// Launches the fast (packed-u16) pass for frames d_frames[0..n) and the exact fallback for frames that overflowed.
// rowsum: [n][H] u32, colsum: [n][W] u32 (may be null).
int launch_frame_stats(epid_ctx* ctx, cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames,
                       int n, FrameStats* d_stats, uint32_t* d_rowsum, uint32_t* d_colsum);
// check_inversion_by_histogram statistics (three percentile pairs in g.ranks): min / max / sum / row / column sums exactly; the decision
// certified from exact counts (FrameStats.overflow = 2 + inverted) or, where the bounds overlap, exact order statistics (overflow = 0)
int launch_frame_stats_inversion(epid_ctx* ctx, cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames, int n, FrameStats* d_stats,
                                 uint32_t* d_rowsum, uint32_t* d_colsum);
// the decision of check_inversion_by_histogram from a FrameStats record of either kind
__device__ __forceinline__ int stats_hist_inverted(const FrameStats& fs, double g_low, double g_mid, double g_high) {
    if (fs.overflow >= 2u) return (int)(fs.overflow - 2u);
    auto lerp = [](double a, double b, double t) { const double d = b - a; double r = a + d * t; if (t >= 0.5) r = b - d * (1.0 - t); return r; };
    const double p_low = lerp((double)fs.ostat[0], (double)fs.ostat[1], g_low);
    const double p_mid = lerp((double)fs.ostat[2], (double)fs.ostat[3], g_mid);
    const double p_high = lerp((double)fs.ostat[4], (double)fs.ostat[5], g_high);
    return fabs(p_mid - p_low) > fabs(p_mid - p_high) ? 1 : 0;
}

}  // namespace epid
