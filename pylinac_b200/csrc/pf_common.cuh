// Shared device-side pieces of the batched PicketFence pipeline (internal; see pf.cu for the stage overview).
#pragma once
#include <cmath>

#include "filters.cuh"
#include "peaks.cuh"
#include "stats.cuh"

namespace epid {

constexpr int PF_P = EPID_PF_MAX_PICKETS;
constexpr int PF_L = EPID_PF_MAX_LEAVES;
constexpr int PROF_THREADS = 256;
constexpr int PROF_MAXN = STATS_MAX_DIM;  // profile length
constexpr int PROF_PEAK_CAP = 512;
constexpr int WIN_WARPS = 4;
constexpr int WIN_CAP_PX = 4096;          // staged pixels per window
constexpr int WIN_MAX_NC = 1024;          // samples along leaf travel
constexpr int WIN_MAX_NR = 64;            // samples across the leaf
constexpr int FIN_THREADS = 256;

struct PctPlan { int prev, next; double gamma; };

// internal status of a frame whose decisions the single-pass front end could not certify (or that _check_for_noise may flag): the
// fast pipeline skips it and the caller re-runs exactly that frame through the exact-histogram pipeline (never visible to callers)
constexpr int PF_STATUS_DEFERRED = 90;

struct PfConst {
    epid_pf_params p;
    int H, W;
    int meas_cap;
    int post_filter;       // stats were taken on an already inverted+filtered copy
    int win2;              // 1: frames the two-kernel window path covers are processed by it (pf_windows2.cu)
    PctPlan lo, hi;        // p0.5 / p99.5 of the frame (ranks live in StatsGeom slots 0..3)
    PctPlan p85[2], p99[2];  // [0]: arrays of length W (np.sum(axis 0)), [1]: length H
};

struct PfFrame {
    int status;
    int noisy;
    int inv;               // pixels are read as g = inv ? mx - v : v - mn
    int corner_inverted;
    int noise_passes;
    uint32_t mn, mx, D;
    uint32_t med2;         // 2 * median(g)
    int orientation;
    int n_pickets;
    int n_inview;
    int todo;              // windows left to the generic kernel (set by k_pf_windows_fast)
    int win2;              // the frame's windows are processed by k_pf_win_medians / k_pf_win_fwxm (set by the former)
    int picket_idx[PF_P];
    double picket_val[PF_P];
    double spacing;
    short inview[PF_L];    // indices into the leaf arrays, reference order
};

struct PfWin { int valid; double l, r; };  // per (in-view leaf, picket)

// two-kernel window path (pf_windows2.cu): what k_pf_win_medians hands to k_pf_win_fwxm
constexpr int PF_W2_NCW = 64;      // travel samples per window
constexpr int PF_W2_NRW = 32;      // rows per window
constexpr int PF_W2_WCAP = 1024;   // windows per frame (in-view leaves x pickets)
constexpr int PF_W2_POOL = PF_W2_WCAP * PF_W2_NCW;     // median samples per frame (bands of neighbouring windows share columns)
struct alignas(16) PfWinRec {              // one per window, 400 bytes
    uint32_t hdr;                          // nc | nr << 16 (signed 16-bit each)
    uint32_t moff;                         // first sample of the window in the frame's median pool
    uint32_t pad[2];
    unsigned long long num[PF_W2_NRW];     // nc * S2 - S1^2 per row (variance numerator along travel)
    uint32_t ext[PF_W2_NRW];               // raw row maximum << 16 | raw row minimum, inside the window
};
static_assert(sizeof(PfWinRec) == 400, "PfWinRec layout");

// numpy _lerp (numpy/lib/_function_base_impl.py): a + (b-a)*t, and b - (b-a)*(1-t) where t >= 0.5
__device__ __forceinline__ double np_lerp(double a, double b, double t) {
    const double d = b - a;
    double r = a + d * t;
    if (t >= 0.5) r = b - d * (1.0 - t);
    return r;
}

// noise flag (_has_noise), corner inversion, D, median in g units for one frame from its statistics.
// check_noise: evaluate the noise criterion (and count noisy frames in counters[0]); post_filter: statistics were taken
// on an already inverted + filtered copy, only D / median are refreshed.
__device__ inline void pf_decide_frame(const PfConst& c, const FrameStats& s, PfFrame& f, int check_noise, int* counters) {
    f.mn = s.mn;
    f.mx = s.mx;
    f.D = s.mx - s.mn;
    if (f.D == 0) { f.status = EPID_PF_FLAT_IMAGE; f.noisy = 0; return; }
    if (!c.post_filter) {
        // _has_noise (picketfence.py:229-238)
        if (check_noise) {
            const double near_min = np_lerp((double)s.ostat[0], (double)s.ostat[1], c.lo.gamma);
            const double near_max = np_lerp((double)s.ostat[2], (double)s.ostat[3], c.hi.gamma);
            const double mnv = (double)s.mn, mxv = (double)s.mx;
            const bool max_is_extreme = mxv > near_max * 1.25;
            const bool min_is_extreme = (mnv < near_min * 0.75) && (fabs(mnv - near_min) > 0.1 * (near_max - near_min));
            f.noisy = (max_is_extreme || min_is_extreme) ? 1 : 0;
            if (f.noisy) atomicAdd(&counters[0], 1);
        }
        // check_inversion(box_size=10, position=(0.01, 0.01)) (core/image.py:881-897)
        const double avg = (double)s.corner_sum / (double)(4 * 10 * 10);
        const double mean = (double)s.sum / (double)s.npix;
        f.corner_inverted = avg > mean ? 1 : 0;
    }
    const int inv = (c.post_filter ? 0 : f.corner_inverted) ^ (c.p.invert ? 1 : 0);
    f.inv = inv;
    // median pair (raw order statistics a <= b) -> g units
    const uint32_t a = s.ostat[4], b = s.ostat[5];
    f.med2 = inv ? (s.mx - b) + (s.mx - a) : (a - s.mn) + (b - s.mn);
}


// bench only: CUDA-event pairs around the frame-streaming kernel of every pipeline pass
struct PfTimers {
    std::vector<cudaEvent_t> ev;
    bool on = false;
    int record(cudaStream_t s) {
        cudaEvent_t e;
        EPID_CUDA(cudaEventCreate(&e));
        EPID_CUDA(cudaEventRecord(e, s));
        ev.push_back(e);
        return EPID_OK;
    }
    float total_ms() {   // call after the stream has been synchronised
        float t = 0;
        for (size_t i = 0; i + 1 < ev.size(); i += 2) { float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); t += ms; }
        return t;
    }
    // stage marks (epid_pf_bench_timed): the time between two consecutive marks is charged to the later mark's stage id
    bool stages = false;
    std::vector<std::pair<int, cudaEvent_t>> marks;
    int mark(cudaStream_t s, int stage) {
        if (!stages) return EPID_OK;
        cudaEvent_t e;
        EPID_CUDA(cudaEventCreate(&e));
        EPID_CUDA(cudaEventRecord(e, s));
        marks.push_back({stage, e});
        return EPID_OK;
    }
    void stage_ms(float* out, int nstages) {   // call after the stream has been synchronised
        for (int k = 0; k < nstages; k++) out[k] = 0.f;
        for (size_t i = 1; i < marks.size(); i++) {
            const int st = marks[i].first;
            if (st < 0 || st >= nstages) continue;
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
            out[st] += ms;
        }
    }
    void destroy() {
        for (auto e : ev) cudaEventDestroy(e);
        ev.clear();
        for (auto& m : marks) cudaEventDestroy(m.second);
        marks.clear();
    }
};
enum { PF_STAGE_START = -1, PF_STAGE_INIT_PILOT = 0, PF_STAGE_STREAM = 1, PF_STAGE_TAIL = 2, PF_STAGE_WINDOWS = 3, PF_STAGE_WINDOWS_GENERIC = 4,
       PF_STAGE_FINALIZE = 5, PF_STAGE_EXACT_FRONT = 6, PF_STAGE_WIN_MEDIANS = 7, PF_STAGE_WIN_FWXM = 8, PF_NSTAGES = 9 };

// pf_windows.cu
int launch_pf_windows_fast(epid_ctx* ctx, cudaStream_t stream, const PfConst* cst, const FrameRef* refs, PfFrame* fr, PfWin* wins, int n);
// pf_windows2.cu
size_t pf_win2_scratch_bytes(int n);       // records followed by the median pools
int launch_pf_windows2(epid_ctx* ctx, cudaStream_t stream, const PfConst* cst, const FrameRef* refs, PfFrame* fr, PfWinRec* recs, PfWin* wins,
                       int n, PfTimers* tm);
// pf_stream.cu
size_t pf_front_scratch_bytes(int n, int H, int W);
// pf_finalize.cu
int launch_pf_finalize(epid_ctx* ctx, cudaStream_t stream, const PfConst* cst, PfFrame* fr, const PfWin* wins, epid_pf_summary* summ,
                       epid_pf_meas* meas, int n, int meas_cap);

// ------------------------------------------------------------------------------------------------ profile / pickets
// r-th smallest (0-based) of src[0..n): value bisection by ONE warp, no block barriers (32 steps, n / 32 compares per lane)
__device__ __forceinline__ uint32_t warp_select_u32(const uint32_t* __restrict__ src, int n, int r) {
    const int lane = threadIdx.x & 31;
    uint32_t lo = 0, hi = 0xffffffffu;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        uint32_t cnt = 0;
        for (int i = lane; i < n; i += 32) cnt += src[i] <= mid ? 1u : 0u;
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (cnt >= (uint32_t)r + 1u) hi = mid; else lo = mid + 1u;
    }
    return lo;
}

// order statistics r_prev <= r_next (adjacent or equal ranks, 0-based) of src[0..n), n <= 1024, by ONE warp: the array lives in
// registers (32 values per lane), the value bisection runs between the array's own minimum and maximum (a sum vector spans ~2^26,
// not 2^32), and the next order statistic is derived from the first: the same value if it occurs often enough, else the smallest
// larger one.
__device__ __forceinline__ void warp_select_pair_u32(const uint32_t* __restrict__ src, int n, int r_prev, int r_next, uint32_t& v_prev,
                                                     uint32_t& v_next) {
    const int lane = threadIdx.x & 31;
    uint32_t x[32];
    uint32_t mnv = 0xffffffffu, mxv = 0;
#pragma unroll
    for (int k = 0; k < 32; k++) {
        const int i = lane + 32 * k;
        x[k] = i < n ? src[i] : 0xffffffffu;      // padding sorts last and is never counted (see below)
        if (i < n) { mnv = min(mnv, x[k]); mxv = max(mxv, x[k]); }
    }
    uint32_t lo = __reduce_min_sync(0xffffffffu, mnv), hi = __reduce_max_sync(0xffffffffu, mxv);
    const uint32_t npad = 32u * 32u - (uint32_t)n;      // padding values equal 0xffffffff: counted only when mid == 0xffffffff
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll
        for (int k = 0; k < 32; k += 4) {
            c0 += x[k] <= mid ? 1u : 0u;
            c1 += x[k + 1] <= mid ? 1u : 0u;
            c2 += x[k + 2] <= mid ? 1u : 0u;
            c3 += x[k + 3] <= mid ? 1u : 0u;
        }
        uint32_t cnt = __reduce_add_sync(0xffffffffu, (c0 + c1) + (c2 + c3));
        if (mid == 0xffffffffu) cnt -= npad;
        if (cnt >= (uint32_t)r_prev + 1u) hi = mid; else lo = mid + 1u;
    }
    v_prev = lo;
    // how many values are <= v_prev, and the smallest value above it
    uint32_t c = 0, above = 0xffffffffu;
#pragma unroll
    for (int k = 0; k < 32; k++) {
        const int i = lane + 32 * k;
        if (i < n) {
            c += x[k] <= lo ? 1u : 0u;
            if (x[k] > lo) above = min(above, x[k]);
        }
    }
    c = __reduce_add_sync(0xffffffffu, c);
    above = __reduce_min_sync(0xffffffffu, above);
    v_next = (c >= (uint32_t)r_next + 1u) ? lo : above;
}

// (p99 - p85) of two arrays at once (np.percentile 'linear'): four independent (array, percentile) selection problems, one per warp
// (each yields the pair of neighbouring order statistics numpy interpolates between).  `sel` : 8 words of shared scratch.
__device__ inline void block_pct_ranges2(const uint32_t* __restrict__ a0, int n0, const PctPlan& p85_0, const PctPlan& p99_0,
                                         const uint32_t* __restrict__ a1, int n1, const PctPlan& p85_1, const PctPlan& p99_1,
                                         uint32_t* sel, double& range0, double& range1) {
    const int wid = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (n0 <= 1024 && n1 <= 1024) {
        for (int s = wid; s < 4; s += nw) {
            const bool second = s >= 2;
            const PctPlan& pp = (s & 1) ? (second ? p99_1 : p99_0) : (second ? p85_1 : p85_0);
            uint32_t va, vb;
            warp_select_pair_u32(second ? a1 : a0, second ? n1 : n0, pp.prev, pp.next, va, vb);
            if (lane == 0) { sel[2 * s] = va; sel[2 * s + 1] = vb; }
        }
    } else {
        for (int s = wid; s < 8; s += nw) {
            const bool second = s >= 4;
            const PctPlan& pp = (s & 2) ? (second ? p99_1 : p99_0) : (second ? p85_1 : p85_0);
            const int r = (s & 1) ? pp.next : pp.prev;
            const uint32_t v = warp_select_u32(second ? a1 : a0, second ? n1 : n0, r);
            if (lane == 0) sel[s] = v;
        }
    }
    __syncthreads();
    range0 = np_lerp((double)sel[2], (double)sel[3], p99_0.gamma) - np_lerp((double)sel[0], (double)sel[1], p85_0.gamma);
    range1 = np_lerp((double)sel[6], (double)sel[7], p99_1.gamma) - np_lerp((double)sel[4], (double)sel[5], p85_1.gamma);
    __syncthreads();
}

// smem needed by pf_profile_block for a block of `threads` threads
__host__ __device__ inline int pf_profile_len(int H, int W) { return ((H > W ? H : W) + 3) & ~3; }
__host__ __device__ inline size_t pf_profile_smem_bytes(int threads, int H, int W) {
    return sizeof(double) * (pf_profile_len(H, W) + 5 * PROF_PEAK_CAP) + sizeof(int) * (5 * PROF_PEAK_CAP + threads + 8) + 64 * sizeof(double);
}

// Orientation, leaf profile, picket search, spacing, leaves in view for ONE frame, executed by the whole block.
// rowsum/colsum: raw pixel sums of THIS frame (rowsum[y] = sum over x); rowsum2/colsum2: clamped sums (may be null if
// the orientation is given).  smraw: pf_profile_smem_bytes(blockDim.x, H, W) bytes of shared memory, 8-byte aligned.
// d_colsum2 / d_rowsum2 > 0: the clamped sums are only known to within [0, d] per element (certified clamp level, see
// pf_stream.cu); the orientation is then decided with that margin and an undecidable frame is counted in counters[1].
__device__ inline void pf_profile_block(const PfConst& c, PfFrame& f, const uint32_t* __restrict__ rowsum,
                                        const uint32_t* __restrict__ colsum, const uint32_t* __restrict__ rowsum2,
                                        const uint32_t* __restrict__ colsum2, unsigned char* smraw, double d_colsum2 = 0.0,
                                        double d_rowsum2 = 0.0, int* counters = nullptr) {
    double* prof = reinterpret_cast<double*>(smraw);                 // max(H, W) doubles (also selection scratch)
    double* w_prom = prof + pf_profile_len(c.H, c.W);
    double* w_wh = w_prom + PROF_PEAK_CAP;
    double* w_lip = w_wh + PROF_PEAK_CAP;
    double* w_rip = w_lip + PROF_PEAK_CAP;
    double* w_skey = w_rip + PROF_PEAK_CAP;
    double* s_red = w_skey + PROF_PEAK_CAP;                          // 32
    double* s_bcast = s_red + 32;                                    // 32 (2 used)
    int* w_idx = reinterpret_cast<int*>(s_bcast + 32);
    int* w_lb = w_idx + PROF_PEAK_CAP;
    int* w_rb = w_lb + PROF_PEAK_CAP;
    int* w_flag = w_rb + PROF_PEAK_CAP;
    int* w_sidx = w_flag + PROF_PEAK_CAP;
    int* w_small = w_sidx + PROF_PEAK_CAP;                           // blockDim.x + 8

    if (f.status != EPID_PF_OK) return;
    const int H = c.H, W = c.W;
    const int tid = threadIdx.x;
    const int NT = blockDim.x;
    const int NW = NT >> 5;

    // ---- orientation (picketfence.py:1501-1526)
    int orient = c.p.orientation;
    if (orient < 0) {
        uint32_t* buf = reinterpret_cast<uint32_t*>(prof);
        double row_range, col_range;   // of np.sum(temp, 0) and np.sum(temp, 1)
        block_pct_ranges2(colsum2, W, c.p85[0], c.p99[0], rowsum2, H, c.p85[1], c.p99[1], buf, row_range, col_range);
        orient = (row_range < col_range) ? 1 : 0;
        if (counters && (d_colsum2 > 0.0 || d_rowsum2 > 0.0)) {
            // every percentile of a sum vector moves by at most its d, so each range moves by at most d (+1: lerp rounding)
            const bool sure_lr = row_range + d_colsum2 + 1.0 < col_range - d_rowsum2;
            const bool sure_ud = row_range - d_colsum2 >= col_range + d_rowsum2 + 1.0;
            if (!sure_lr && !sure_ud) {      // the same in every thread: the frame is re-run by the exact pipeline
                if (threadIdx.x == 0) { atomicAdd(&counters[1], 1); f.status = PF_STATUS_DEFERRED; }
                return;
            }
        }
    }
    // ---- leaf profile: np.mean(image, axis) then / max   (picketfence.py:747-752)
    const int n = orient == 0 ? W : H;
    const int other = orient == 0 ? H : W;
    const uint32_t* raw = orient == 0 ? colsum : rowsum;
    // sum of g along the other axis: inv ? other*mx - raw : raw - other*mn   (exact integers)
    const long long base = (long long)other * (long long)(f.inv ? f.mx : f.mn);
    double lmax = 0.0;
    for (int i = tid; i < n; i += NT) {
        const long long sg = f.inv ? base - (long long)raw[i] : (long long)raw[i] - base;
        const double v = (double)sg;
        prof[i] = v;
        lmax = fmax(lmax, v);
    }
    lmax = warp_max(lmax);
    if ((tid & 31) == 0) s_red[tid >> 5] = lmax;
    __syncthreads();
    if (tid == 0) {
        double m = 0.0;
        for (int i = 0; i < NW; i++) m = fmax(m, s_red[i]);
        s_bcast[0] = m;
    }
    __syncthreads();
    const double pmax = s_bcast[0];
    double lmin = 2.0;
    for (int i = tid; i < n; i += NT) {
        const double v = prof[i] / pmax;
        prof[i] = v;
        lmin = fmin(lmin, v);
    }
    lmin = warp_min(lmin);
    __syncthreads();
    if ((tid & 31) == 0) s_red[tid >> 5] = lmin;
    __syncthreads();
    if (tid == 0) {
        double m = 2.0;
        for (int i = 0; i < NW; i++) m = fmin(m, s_red[i]);
        s_bcast[1] = m;
    }
    __syncthreads();
    const double pmin = s_bcast[1];
    // ---- find_fwxm_peaks(min_distance=0.02, threshold=height_threshold, max_number, peak_sort, required_prominence)
    // _parse_peak_args (core/profile.py:2626-2649): max of the normalised profile is 1.0
    PeakArgs a;
    {
        const double val_range = 1.0 - pmin;
        double thr = c.p.height_threshold;
        if (thr >= 0.0 && thr <= 1.0) thr = pmin + thr * val_range;
        a.hmin = thr;
        a.distance = max((int)(0.02 * (double)n), 1);
        a.pmin = c.p.required_prominence;
        a.wmin = 0.0;
        a.rel_height = 1.0 - 0.5;
        a.max_number = c.p.num_pickets;
        a.sort_by_height = c.p.peak_sort == 1;
    }
    PeakWork w;
    w.cap = PROF_PEAK_CAP;
    w.idx = w_idx; w.prom = w_prom; w.lbase = w_lb; w.rbase = w_rb; w.width_height = w_wh; w.lip = w_lip; w.rip = w_rip;
    w.flag = w_flag; w.skey = w_skey; w.sidx = w_sidx; w.s_small = w_small;
    const int np = block_find_peaks(prof, n, a, w);
    if (tid == 0) {
        f.orientation = orient;
        if (np < 0 || np > PF_P) {
            f.status = EPID_PF_TOO_MANY_PICKETS;
        } else if (np == 0) {
            f.status = EPID_PF_NO_PICKETS;
        } else {
            f.n_pickets = np;
            int sorted[PF_P];
            for (int k = 0; k < np; k++) {
                const double lt = w.lip[k], rt = w.rip[k];
                const int idx = (int)rint(lt + (rt - lt) / 2.0);   // int(round(.)), banker's (core/profile.py:2167)
                f.picket_idx[k] = idx;
                f.picket_val[k] = prof[idx];
                int j = k;
                while (j > 0 && sorted[j - 1] > idx) { sorted[j] = sorted[j - 1]; j--; }
                sorted[j] = idx;
            }
            // picket_spacing = np.median(np.diff(np.sort(peak_idxs)))   (picketfence.py:766-767)
            double spacing = c.p.picket_spacing;
            if (spacing < 0) {
                const int nd = np - 1;
                if (nd <= 0) {
                    spacing = __longlong_as_double(0x7ff8000000000000LL);  // np.median([]) -> nan
                } else {
                    int d[PF_P];
                    for (int k = 0; k < nd; k++) {
                        const int v = sorted[k + 1] - sorted[k];
                        int j = k;
                        while (j > 0 && d[j - 1] > v) { d[j] = d[j - 1]; j--; }
                        d[j] = v;
                    }
                    spacing = (nd & 1) ? (double)d[nd / 2] : ((double)d[nd / 2 - 1] + (double)d[nd / 2]) / 2.0;
                }
            }
            f.spacing = spacing;
            // _leaves_in_view (picketfence.py:888-912)
            const double n_axis = (double)(orient == 0 ? H : W);
            const double ratio = c.p.leaf_analysis_width_ratio;
            double pixel_range = n_axis / 2.0;
            pixel_range -= fmax(c.p.leaf_width_mm[0] * ratio, c.p.leaf_width_mm[c.p.n_leaves - 1] * ratio) * c.p.dpmm;
            int cnt = 0;
            for (int l = 0; l < c.p.n_leaves; l++)
                if (fabs(c.p.leaf_center_mm[l]) < pixel_range / c.p.dpmm) f.inview[cnt++] = (short)l;
            f.n_inview = cnt;
        }
    }
}

}  // namespace epid
