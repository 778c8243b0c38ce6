// Batched Starshot.analyze() on the GPU.  One result per frame; frames never leave HBM between stages.
//
// Reference path reproduced (pylinac v3.46.0):
//   Starshot.analyze / _get_reasonable_start_point / _get_reasonable_wobble / _find_wobble_minimize   starshot.py:197-401
//   StarProfile (CollapsedCircleProfile) / LineManager / calculate_angles                              starshot.py:701-834
//   CircleProfile._radians / x,y_locations / CollapsedCircleProfile._radii / _profile                  core/profile.py:2244-2283, 2405-2483
//   BaseImage.check_inversion_by_histogram / ground / invert / dist2edge_min                           core/image.py:817-852, 899-926
//   find_peaks / MultiProfile.find_fwxm_peaks / FWXMProfile.center_idx                                 core/profile.py:322-327, 602-611, 2143-2176, 2545-2649
//   Line.distance_to                                                                                   core/geometry.py:569-584
// Third-party arithmetic restated here (scipy 1.18.1): ndimage.map_coordinates(order=0, mode='constant') =
// sample at floor(c + 0.5) if 0 <= c <= len - 1 on both axes else 0; ndimage.gaussian_filter = correlate1d with the
// symmetric summation order of NI_Correlate1D and mode='reflect'; signal.find_peaks (peaks.cuh);
// optimize.minimize(method='Nelder-Mead') = _minimize_neldermead (non-adaptive, N = 3, maxiter = maxfun = 600,
// xatol = 1e-4, fatol from the caller, stable ordering of the simplex).
//
// Exactness: after check_inversion_by_histogram + ground (+ invert) the image is an integer map of the uint16 frame,
// f(v) = v - min or max - v; ring samples, their 20-fold sums, column / row maxima and the order statistics behind the
// percentiles are therefore exact integers, and the fp64 profile arithmetic repeats the reference's operation order
// (FMA contraction disabled), so peak indices are bit-exact and the wobble agrees to ~1e-12 px.
//
// Stages:
//   k_frame_stats    exact order statistics of the frame (p4 / p50 / p96) and of its central third (p90)      (stats.cu)
//   k_star_front     inversion decision, central-third column / row maxima, FW80M start point, local maximum
//   k_star_rows      CTA per (frame, candidate row): ring sampling (20 radii, nearest neighbour) -> roll -> gaussian -> ground once per
//                    radius, then per min_peak_height: find_fwxm_peaks -> lines -> Nelder-Mead until a candidate has a verdict
//   k_star_pick      first row in the reference's candidate order that has a verdict = the wobble the serial loop stops at
#include <cmath>

#include "peaks.cuh"
#include "pf_common.cuh"

namespace epid {

constexpr int SS_THREADS = 256;
constexpr int SS_GW_CAP = 192;        // gaussian half-kernel (radius + 1 weights) kept in shared memory: sigma <= 47
constexpr int SS_PEAK_CAP = 512;
constexpr int SS_MAX_PEAKS = EPID_STAR_MAX_PEAKS;
constexpr int SS_MAX_LINES = EPID_STAR_MAX_PEAKS / 2;

struct StarConst {
    epid_star_params p;
    int H, W;
    int top, left, ch, cw;            // central third
    PctPlan p4, p50, p96;             // of the frame
    PctPlan p90;                      // of the central third
    int nmax;                         // capacity of the per-frame profile arrays
    int npad;                         // capacity of the padded (rolled + reflected) copy the gaussian reads: nmax + 2 * filter radius
    int max_sigma;                    // gaussian table covers sigma = 1 .. max_sigma
};

struct StarFrame {
    uint32_t mn, mx;
    int flip;                         // pixels are read as f(v) = flip ? mx - v : v - mn
    int hist_inverted;
    int sx, sy;                       // automatic start point
    double local_max;
};

__device__ __forceinline__ double star_px(const FrameRef& fr, int H, int W, double yc, double xc, uint32_t mn, uint32_t mx, int flip) {
    // scipy.ndimage.map_coordinates(order=0, mode='constant', cval=0)
    if (!(yc >= 0.0 && yc <= (double)(H - 1) && xc >= 0.0 && xc <= (double)(W - 1))) return 0.0;
    const int iy = (int)floor(yc + 0.5), ix = (int)floor(xc + 0.5);
    const uint32_t v = __ldg(fr.origin + (size_t)iy * fr.pitch + ix);
    return (double)(flip ? mx - v : v - mn);
}

// ------------------------------------------------------------------------------------------------ front
__global__ void __launch_bounds__(SS_THREADS)
k_star_front(const StarConst* __restrict__ cc, const FrameRef* __restrict__ frames, const FrameStats* __restrict__ full,
             const FrameStats* __restrict__ central, StarFrame* sf, epid_star_result* __restrict__ res) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const StarConst& c = *cc;
    const int fi = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const FrameRef frf = frames[fi];
    const FrameStats fs = full[fi], cs = central[fi];
    StarFrame& f = sf[fi];
    // ---- check_inversion_by_histogram([4, 50, 96]) (core/image.py:899-926), ground, optional invert
    const int hist_inv = stats_hist_inverted(fs, c.p4.gamma, c.p50.gamma, c.p96.gamma);      // certified from counts or exact percentiles
    const int flip = hist_inv ^ (c.p.invert ? 1 : 0);
    const uint32_t mn = fs.mn, mx = fs.mx;
    // ---- _get_reasonable_start_point (starshot.py:197-227): maxima of the central third along each axis
    const int n_max = c.cw > c.ch ? c.cw : c.ch;
    const int n_al = (n_max + 3) & ~3;
    double* xsum = reinterpret_cast<double*>(smraw);
    double* ysum = xsum + n_al;
    double* w_prom = ysum + n_al;
    double* w_wh = w_prom + SS_PEAK_CAP;
    double* w_lip = w_wh + SS_PEAK_CAP;
    double* w_rip = w_lip + SS_PEAK_CAP;
    double* w_skey = w_rip + SS_PEAK_CAP;
    int* w_idx = reinterpret_cast<int*>(w_skey + SS_PEAK_CAP);
    int* w_lb = w_idx + SS_PEAK_CAP;
    int* w_rb = w_lb + SS_PEAK_CAP;
    int* w_flag = w_rb + SS_PEAK_CAP;
    int* w_sidx = w_flag + SS_PEAK_CAP;
    int* w_small = w_sidx + SS_PEAK_CAP;
    const uint16_t* org = frf.origin + (size_t)c.top * frf.pitch + c.left;
    for (int x = tid; x < c.cw; x += SS_THREADS) {
        uint32_t vmx = 0, vmn = 0xffffu;
        for (int y = 0; y < c.ch; y++) {
            const uint32_t v = __ldg(org + (size_t)y * frf.pitch + x);
            vmx = max(vmx, v);
            vmn = min(vmn, v);
        }
        xsum[x] = (double)(flip ? mx - vmn : vmx - mn);
    }
    for (int y = wid; y < c.ch; y += SS_THREADS / 32) {
        uint32_t vmx = 0, vmn = 0xffffu;
        for (int x = lane; x < c.cw; x += 32) {
            const uint32_t v = __ldg(org + (size_t)y * frf.pitch + x);
            vmx = max(vmx, v);
            vmn = min(vmn, v);
        }
        vmx = warp_max(vmx);
        vmn = warp_min(vmn);
        if (lane == 0) ysum[y] = (double)(flip ? mx - vmn : vmx - mn);
    }
    __syncthreads();
    // FWXMProfile(values, fwxm_height=80).center_idx (core/profile.py:322-327, 602-611)
    PeakArgs a;
    a.hmin = -INFINITY;
    a.distance = 1;
    a.pmin = -1.0;
    a.wmin = 0.0;
    a.rel_height = 1.0 - 80.0 / 100.0;
    a.max_number = 1;
    a.sort_by_height = 0;
    PeakWork w;
    w.cap = SS_PEAK_CAP;
    w.idx = w_idx; w.prom = w_prom; w.lbase = w_lb; w.rbase = w_rb; w.width_height = w_wh; w.lip = w_lip; w.rip = w_rip;
    w.flag = w_flag; w.skey = w_skey; w.sidx = w_sidx; w.s_small = w_small;
    int status = EPID_STAR_OK;
    int pt[2] = {0, 0};
    for (int axis = 0; axis < 2; axis++) {
        const int np = block_find_peaks(axis == 0 ? xsum : ysum, axis == 0 ? c.cw : c.ch, a, w);
        __syncthreads();
        if (np < 1) {
            status = EPID_STAR_NO_START_POINT;          // the reference raises IndexError inside FWXMProfile.field_edge_idx
        } else {
            const double l = w.lip[0], r = w.rip[0];
            pt[axis] = (int)rint(fabs(r - l) / 2.0 + l) + (axis == 0 ? c.left : c.top);   // python round(): half to even
        }
        __syncthreads();
    }
    if (tid == 0) {
        f.mn = mn;
        f.mx = mx;
        f.flip = flip;
        f.hist_inverted = hist_inv;
        f.sx = pt[0];
        f.sy = pt[1];
        // np.percentile(central_array, 90) of the transformed values (sorted ascending = raw descending when flipped)
        double lm;
        if (!flip) lm = np_lerp((double)(cs.ostat[0] - mn), (double)(cs.ostat[1] - mn), c.p90.gamma);
        else lm = np_lerp((double)(mx - cs.ostat[3]), (double)(mx - cs.ostat[2]), c.p90.gamma);
        f.local_max = lm;
        epid_star_result& R = res[fi];
        R.status = mx == mn ? EPID_STAR_FLAT_IMAGE : status;
        R.hist_inverted = hist_inv;
        R.start_x = pt[0];
        R.start_y = pt[1];
        R.local_max = lm;
    }
}

// ------------------------------------------------------------------------------------------------ wobble
struct StarLine { double x1, y1, x2, y2; };

__device__ __forceinline__ double line_distance(const StarLine& l, double px, double py) {
    // Line.distance_to (core/geometry.py:569-584): sqrt(sum(cross(lp2 - lp1, lp1 - p)^2)) / sqrt(sum((lp2 - lp1)^2)), z = 0
    const double ax = l.x2 - l.x1, ay = l.y2 - l.y1;
    const double bx = l.x1 - px, by = l.y1 - py;
    const double cz = ax * by - ay * bx;
    const double num = sqrt(0.0 + 0.0 + cz * cz);
    const double den = sqrt(ax * ax + ay * ay + 0.0);
    return num / den;
}

// max over the lines of the distance to p, evaluated by a whole warp: lane l takes lines l, l + 32, ...; the maximum of the same
// distances as the sequential loop (max is exact and order independent), every lane returns it, so the optimiser below runs
// redundantly but in lock step on all 32 lanes and its objective costs one line instead of nl lines per call
__device__ inline double wobble_objective(const StarLine* lines, int nl, const double* p) {
    const int lane = threadIdx.x & 31;
    double m = -INFINITY;
    for (int i = lane; i < nl; i += 32) m = fmax(m, line_distance(lines[i], p[0], p[1]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    return m;
}

// scipy.optimize._optimize._minimize_neldermead, N = 3 (x, y and the inert z of Point.as_array()), default options + fatol.
// Called by all 32 lanes of one warp (see wobble_objective).
__device__ inline void nelder_mead3(const StarLine* lines, int nl, double x0, double y0, double fatol, double* xout, double* fout) {
    constexpr int N = 3;
    const double xatol = 1e-4;
    const int maxiter = N * 200, maxfun = N * 200;
    double sim[N + 1][N], fsim[N + 1];
    const double start[N] = {x0, y0, 0.0};
    for (int j = 0; j < N; j++) sim[0][j] = start[j];
    for (int k = 0; k < N; k++) {
        for (int j = 0; j < N; j++) sim[k + 1][j] = start[j];
        if (start[k] != 0.0) sim[k + 1][k] = (1 + 0.05) * start[k];
        else sim[k + 1][k] = 0.00025;
    }
    int fcalls = 0;
    auto func = [&](const double* p) { fcalls++; return wobble_objective(lines, nl, p); };
    auto sort_simplex = [&]() {      // np.argsort (stable for these sizes) + np.take
        for (int i = 1; i <= N; i++) {
            const double fv = fsim[i];
            double xv[N];
            for (int j = 0; j < N; j++) xv[j] = sim[i][j];
            int k = i - 1;
            while (k >= 0 && fsim[k] > fv) {
                fsim[k + 1] = fsim[k];
                for (int j = 0; j < N; j++) sim[k + 1][j] = sim[k][j];
                k--;
            }
            fsim[k + 1] = fv;
            for (int j = 0; j < N; j++) sim[k + 1][j] = xv[j];
        }
    };
    for (int k = 0; k <= N; k++) fsim[k] = func(sim[k]);
    sort_simplex();
    int iterations = 1;
    while (fcalls < maxfun && iterations < maxiter) {
        double dx = 0.0, df = 0.0;
        for (int k = 1; k <= N; k++) {
            for (int j = 0; j < N; j++) dx = fmax(dx, fabs(sim[k][j] - sim[0][j]));
            df = fmax(df, fabs(fsim[0] - fsim[k]));
        }
        if (dx <= xatol && df <= fatol) break;
        double xbar[N], xr[N];
        for (int j = 0; j < N; j++) {
            xbar[j] = ((sim[0][j] + sim[1][j]) + sim[2][j]) / N;
            xr[j] = 2.0 * xbar[j] - 1.0 * sim[N][j];
        }
        const double fxr = func(xr);
        bool doshrink = false;
        if (fxr < fsim[0]) {
            double xe[N];
            for (int j = 0; j < N; j++) xe[j] = 3.0 * xbar[j] - 2.0 * sim[N][j];
            const double fxe = func(xe);
            if (fxe < fxr) { for (int j = 0; j < N; j++) sim[N][j] = xe[j]; fsim[N] = fxe; }
            else { for (int j = 0; j < N; j++) sim[N][j] = xr[j]; fsim[N] = fxr; }
        } else if (fxr < fsim[N - 1]) {
            for (int j = 0; j < N; j++) sim[N][j] = xr[j];
            fsim[N] = fxr;
        } else if (fxr < fsim[N]) {
            double xc[N];
            for (int j = 0; j < N; j++) xc[j] = 1.5 * xbar[j] - 0.5 * sim[N][j];
            const double fxc = func(xc);
            if (fxc <= fxr) { for (int j = 0; j < N; j++) sim[N][j] = xc[j]; fsim[N] = fxc; }
            else doshrink = true;
        } else {
            double xcc[N];
            for (int j = 0; j < N; j++) xcc[j] = 0.5 * xbar[j] + 0.5 * sim[N][j];
            const double fxcc = func(xcc);
            if (fxcc < fsim[N]) { for (int j = 0; j < N; j++) sim[N][j] = xcc[j]; fsim[N] = fxcc; }
            else doshrink = true;
        }
        if (doshrink) {
            for (int k = 1; k <= N; k++) {
                for (int j = 0; j < N; j++) sim[k][j] = sim[0][j] + 0.5 * (sim[k][j] - sim[0][j]);
                fsim[k] = func(sim[k]);
            }
        }
        iterations++;
        sort_simplex();
    }
    xout[0] = sim[0][0];
    xout[1] = sim[0][1];
    double fmin_ = fsim[0];
    for (int k = 1; k <= N; k++) fmin_ = fmin(fmin_, fsim[k]);
    *fout = fmin_;
}

// One CTA per (frame, row of the candidate product).  _get_reasonable_wobble (starshot.py:344-376) tries, in this order, the caller's
// (radius, min_peak_height) and then product(append(radius, linspace(0.95, 0.1, 10)), append(min_peak_height, linspace(0.05, 0.95, 10)))
// until a candidate is accepted.  Row 0 = the caller's pair; row r = 1 .. 11 = the r-th radius with its 11 heights.  All candidates
// of a row share the ring samples, the roll, the gaussian and the grounding (only the find_peaks threshold differs), so a row computes
// that profile once; rows are independent, so the rows of a round run in parallel CTAs and every row reports its FIRST candidate
// with a verdict (accepted or hard failure).  k_star_pick then takes the first such row in order, which is the candidate the serial
// loop would have stopped at; best[] (smallest order index with a verdict so far) only lets later candidates stop early.
constexpr int SS_ROWS = 12;
constexpr int SS_ROUND_ROWS = 4;       // rows per round after round 0 (row 0 alone: no speculative work for frames that pass at once)

#ifndef EPID_SS_MIN_CTAS
#define EPID_SS_MIN_CTAS 2      // resident CTAs per SM the row kernel is compiled for (3: 80 registers with ~0.9 KB of spill traffic; variants/)
#endif
__global__ void __launch_bounds__(SS_THREADS, EPID_SS_MIN_CTAS)
k_star_rows(const StarConst* __restrict__ cc, const FrameRef* __restrict__ frames, const StarFrame* __restrict__ sf,
            const double* __restrict__ gauss_w, const int* __restrict__ gauss_off, double* __restrict__ prof_a,
            double* __restrict__ prof_b, double* __restrict__ prof_c, const epid_star_result* __restrict__ res, int row0,
            const int* __restrict__ done, int* __restrict__ best, int* __restrict__ row_verdict, epid_star_result* __restrict__ row_res) {
    __shared__ double s_prom[SS_PEAK_CAP], s_wh[SS_PEAK_CAP], s_lip[SS_PEAK_CAP], s_rip[SS_PEAK_CAP], s_skey[SS_PEAK_CAP];
    __shared__ int s_idx[SS_PEAK_CAP], s_lb[SS_PEAK_CAP], s_rb[SS_PEAK_CAP], s_flag[SS_PEAK_CAP], s_sidx[SS_PEAK_CAP];
    __shared__ int s_small[SS_THREADS + 8];
    __shared__ double s_red[SS_THREADS / 32], s_bc[4];
    __shared__ int s_redi[SS_THREADS / 32], s_ctl[4];
    __shared__ StarLine s_lines[SS_MAX_LINES];
    __shared__ double s_gw[SS_GW_CAP];
    const StarConst& c = *cc;
    const int fi = blockIdx.x;
    const int row = row0 + blockIdx.y;
    if (res[fi].status != EPID_STAR_OK || done[fi]) return;
    epid_star_result& R = row_res[(size_t)fi * SS_ROWS + row];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const FrameRef frf = frames[fi];
    const StarFrame f = sf[fi];
    const int H = c.H, W = c.W;
    const size_t slot = (size_t)fi * gridDim.y + blockIdx.y;
    double* pa = prof_a + slot * c.nmax;
    double* pb = prof_b + slot * c.nmax;
    double* pc = prof_c + slot * c.npad;
    const double dpmm = c.p.dpmm;
    const double fx = c.p.has_start_point ? c.p.start_x : (double)f.sx;
    const double fy = c.p.has_start_point ? c.p.start_y : (double)f.sy;
    PeakWork w;
    w.cap = SS_PEAK_CAP;
    w.idx = s_idx; w.prom = s_prom; w.lbase = s_lb; w.rbase = s_rb; w.width_height = s_wh; w.lip = s_lip; w.rip = s_rip;
    w.flag = s_flag; w.skey = s_skey; w.sidx = s_sidx; w.s_small = s_small;
    const double PI = 3.141592653589793;
    // this row's radius; np.linspace(a, b, 10)[i] = i * step + a, last element = b
    const int ri = row - 1;            // index into append(radius, linspace(0.95, 0.1, 10)); row 0: the caller's radius
    double radius;
    if (row <= 1) radius = c.p.radius;
    else radius = (ri - 1) == 9 ? 0.1 : (double)(ri - 1) * ((0.1 - 0.95) / 9.0) + 0.95;
    const int nheights = row == 0 ? 1 : 11;
    const int order0 = row == 0 ? 0 : 1 + (row - 1) * 11;      // position of the row's first candidate in the serial order
    if (best[fi] < order0) return;                              // an earlier candidate already has a verdict
    int roll = 0;
    int status = EPID_STAR_OK;
    int n;
    double rpx, interval;
    {
        // StarProfile._convert_radius_perc2pix -> dist2edge_min (core/image.py:817-837)
        const double d2e = fmin(fmin((double)H - fy, (double)W - fx), fmin(fy, fx));
        rpx = d2e * radius;
        // CollapsedCircleProfile geometry (core/profile.py:2244-2252, 2446-2455)
        const double r_lo = rpx * (1 - 0.1), r_hi = rpx * (1 + 0.1);
        const double rstep = (r_hi - r_lo) / 19.0;                  // np.linspace(start, stop, 20)
        const double size = PI * r_hi * 2 * 3;
        interval = (2 * PI) / size;
        const double span = ((2 * PI) - interval) / interval;       // np.arange length = ceil((stop - start) / step)
        n = (span > 0.0 && span < 1e9) ? (int)ceil(span) : 0;
        if (n < 3 || n > c.nmax) {
            if (n > c.nmax) status = EPID_STAR_CAPACITY;
            n = 0;
        }
        if (n > 0) {
            // ---- _profile: sum over 20 radii of nearest-neighbour samples / 20
            // The 20 pixel reads of a sample are independent, but behind the bounds test of map_coordinates they were issued one
            // DRAM round trip after the other (the batch does not fit L2): the addresses are clamped instead, all 20 loads are issued
            // back to back, and the test only selects between the pixel and the constant 0 afterwards (same values, same order of sums).
            for (int i = tid; i < n; i += SS_THREADS) {
                const double rad = (double)(n - 1 - i) * interval;   // arange(...)[::-1]
                const double cs = cos(rad), sn = sin(rad);
                uint32_t raw[20];
                bool inside[20];
#pragma unroll
                for (int k = 0; k < 20; k++) {
                    const double rk = k == 19 ? r_hi : (double)k * rstep + r_lo;
                    const double yc = sn * rk + fy, xc = cs * rk + fx;
                    inside[k] = yc >= 0.0 && yc <= (double)(H - 1) && xc >= 0.0 && xc <= (double)(W - 1);
                    const int iy = inside[k] ? (int)floor(yc + 0.5) : 0, ix = inside[k] ? (int)floor(xc + 0.5) : 0;
                    raw[k] = __ldg(frf.origin + (size_t)iy * frf.pitch + ix);
                }
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < 20; k++) acc += inside[k] ? (double)(f.flip ? f.mx - raw[k] : raw[k] - f.mn) : 0.0;
                pa[i] = acc / 20.0;
            }
            __syncthreads();
            // ---- _roll_prof_to_midvalley: first index of the minimum
            double lm = INFINITY;
            int li = 0x7fffffff;
            for (int i = tid; i < n; i += SS_THREADS) {
                const double v = pa[i];
                if (v < lm) { lm = v; li = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double om = __shfl_xor_sync(0xffffffffu, lm, o);
                const int oi = __shfl_xor_sync(0xffffffffu, li, o);
                if (om < lm || (om == lm && oi < li)) { lm = om; li = oi; }
            }
            if (lane == 0) { s_red[wid] = lm; s_redi[wid] = li; }
            __syncthreads();
            if (tid == 0) {
                double m = s_red[0];
                int mi = s_redi[0];
                for (int k = 1; k < SS_THREADS / 32; k++)
                    if (s_red[k] < m || (s_red[k] == m && s_redi[k] < mi)) { m = s_red[k]; mi = s_redi[k]; }
                s_ctl[0] = mi;
            }
            __syncthreads();
            roll = s_ctl[0];
            // ---- filter(size=0.003, kind="gaussian") (core/array_utils.py:106-138): sigma = max(int(round(n * 0.003)), 1)
            int sigma = (int)rint((double)n * 0.003);
            if (sigma < 1) sigma = 1;
            if (sigma > c.max_sigma) { status = EPID_STAR_CAPACITY; sigma = c.max_sigma; }
            const int rad_w = (int)(4.0 * (double)sigma + 0.5);
            const double* __restrict__ gw = gauss_w + gauss_off[sigma];
            auto at = [&](int idx) -> double {      // rolled profile with scipy 'reflect' extension
                while (idx < 0 || idx >= n) {
                    if (idx < 0) idx = -idx - 1;
                    if (idx >= n) idx = 2 * n - 1 - idx;
                }
                int j = idx + roll;
                if (j >= n) j -= n;
                return pa[j];
            };
            // the rolled profile with its reflected margins, laid out contiguously once: the 2 * rad_w + 1 taps of every output sample
            // are then plain coalesced loads (same operands, same order of additions as before)
            for (int l = tid; l < n + 2 * rad_w; l += SS_THREADS) pc[l] = at(l - rad_w);
            __syncthreads();
            // weights of the left half + centre in shared memory; four output samples per thread in flight (independent accumulators:
            // the per-sample order of additions is unchanged, the loads of the four chains overlap)
            const bool gw_sh = rad_w + 1 <= SS_GW_CAP;
            if (gw_sh) for (int k = tid; k <= rad_w; k += SS_THREADS) s_gw[k] = gw[k];
            __syncthreads();
            const double* __restrict__ gwp = gw_sh ? s_gw : gw;
            double tmin = INFINITY;
            for (int l0 = tid; l0 < n; l0 += 4 * SS_THREADS) {
                const int l1 = l0 + SS_THREADS, l2 = l0 + 2 * SS_THREADS, l3 = l0 + 3 * SS_THREADS;
                const bool v1 = l1 < n, v2 = l2 < n, v3 = l3 < n;
                const double* __restrict__ q0 = pc + l0 + rad_w;
                const double* __restrict__ q1 = v1 ? pc + l1 + rad_w : q0;
                const double* __restrict__ q2 = v2 ? pc + l2 + rad_w : q0;
                const double* __restrict__ q3 = v3 ? pc + l3 + rad_w : q0;
                const double gc = gwp[rad_w];
                double t0 = q0[0] * gc, t1 = q1[0] * gc, t2 = q2[0] * gc, t3 = q3[0] * gc;
                for (int ll = -rad_w; ll < 0; ll++) {
                    const double g = gwp[ll + rad_w];
                    t0 += (q0[ll] + q0[-ll]) * g;
                    t1 += (q1[ll] + q1[-ll]) * g;
                    t2 += (q2[ll] + q2[-ll]) * g;
                    t3 += (q3[ll] + q3[-ll]) * g;
                }
                pb[l0] = t0;
                tmin = fmin(tmin, t0);
                if (v1) { pb[l1] = t1; tmin = fmin(tmin, t1); }
                if (v2) { pb[l2] = t2; tmin = fmin(tmin, t2); }
                if (v3) { pb[l3] = t3; tmin = fmin(tmin, t3); }
            }
            tmin = warp_min(tmin);
            if (lane == 0) s_red[wid] = tmin;
            __syncthreads();
            if (tid == 0) {
                double m = s_red[0];
                for (int k = 1; k < SS_THREADS / 32; k++) m = fmin(m, s_red[k]);
                s_bc[0] = m;
            }
            __syncthreads();
            // ---- ground, then the profile maximum (for a ratio threshold)
            const double gmin = s_bc[0];
            double tmax = -INFINITY;
            for (int l = tid; l < n; l += SS_THREADS) {
                const double v = pb[l] - gmin;
                pb[l] = v;
                tmax = fmax(tmax, v);
            }
            tmax = warp_max(tmax);
            __syncthreads();
            if (lane == 0) s_red[wid] = tmax;
            __syncthreads();
            if (tid == 0) {
                double m = s_red[0];
                for (int k = 1; k < SS_THREADS / 32; k++) m = fmax(m, s_red[k]);
                s_bc[1] = m;
            }
            __syncthreads();
        }
    }
    for (int hi = 0; hi < nheights; hi++) {
        const int order = order0 + hi;
        if (hi > 0) {
            // uniform early exit: a candidate before this one has a verdict
            if (tid == 0) s_ctl[0] = atomicMin(&best[fi], 0x7fffffff) < order ? 1 : 0;
            __syncthreads();
            const int stop = s_ctl[0];
            __syncthreads();
            if (stop) return;
        }
        double mph;
        if (row == 0 || hi == 0) mph = c.p.min_peak_height;
        else mph = (hi - 1) == 9 ? 0.95 : (double)(hi - 1) * ((0.95 - 0.05) / 9.0) + 0.05;
        const double min_height = mph * f.local_max;
        const int iterations = order + 1;                          // StarProfile constructions of the serial loop up to this candidate
        int npk = 0;
        if (n > 0) {
            // ---- find_fwxm_peaks(threshold=min_height, min_distance=0.02) / find_peaks (core/profile.py:2050-2176, 2545-2649)
            PeakArgs a;
            double thr = min_height;
            if (thr >= 0.0 && thr <= 1.0) thr = 0.0 + thr * (s_bc[1] - 0.0);       // values.min() == 0 after ground()
            a.hmin = thr;
            a.distance = max((int)(0.02 * (double)n), 1);
            a.pmin = -1.0;
            a.wmin = 0.0;
            a.rel_height = 1.0 - 0.5;
            a.max_number = 0;
            a.sort_by_height = 0;
            npk = block_find_peaks(pb, n, a, w);
            __syncthreads();
            if (npk < 0 || npk > SS_MAX_PEAKS) { status = EPID_STAR_CAPACITY; npk = 0; }
        }
        // ---- lines, wobble, acceptance (warp 0: lane 0 does the scalar bookkeeping, the Nelder-Mead objective uses all lanes)
        if (wid == 0) {
            int verdict = 0;            // 0: next candidate, 1: accepted, 2: hard failure (status)
            int fail = status;
            int nl = 0, do_nm = 0;
            if (lane == 0) {
                if (status == EPID_STAR_OK) {
                    if (npk < 6 || (npk & 1)) {
                        if (!c.p.recursive) { verdict = 2; fail = EPID_STAR_NO_LINES; }
                    } else {
                        double px[SS_MAX_PEAKS], py[SS_MAX_PEAKS];
                        for (int k = 0; k < npk; k++) {
                            int idx;
                            if (c.p.fwhm) idx = (int)rint(s_lip[k] + (s_rip[k] - s_lip[k]) / 2.0);      // int(round(.)), half to even
                            else idx = s_idx[k];
                            R.peak_idx[k] = idx;
                            int j = idx + roll;                                                         // position before the roll
                            if (j >= n) j -= n;
                            const double rad = (double)(n - 1 - j) * interval;
                            px[k] = cos(rad) * rpx + fx;
                            py[k] = sin(rad) * rpx + fy;
                            R.peak_x[k] = px[k];
                            R.peak_y[k] = py[k];
                        }
                        nl = npk / 2;
                        bool near_lines = true;
                        for (int k = 0; k < nl; k++) {
                            s_lines[k].x1 = px[k]; s_lines[k].y1 = py[k];
                            s_lines[k].x2 = px[k + nl]; s_lines[k].y2 = py[k + nl];
                            if (line_distance(s_lines[k], fx, fy) > 10 * dpmm) near_lines = false;    // LineManager raises ValueError
                        }
                        do_nm = near_lines ? 1 : 0;
                    }
                } else {
                    verdict = 2;
                }
            }
            do_nm = __shfl_sync(0xffffffffu, do_nm, 0);
            nl = __shfl_sync(0xffffffffu, nl, 0);
            __syncwarp();
            if (do_nm) {
                double xo[2], fo;
                nelder_mead3(s_lines, nl, fx, fy, 0.001, xo, &fo);
                if (lane == 0) {
                    const double radius_mm = fo / dpmm;
                    // Point.distance_to (core/geometry.py:118-132): sqrt(dx^2 + dy^2 + dz^2)
                    const double ddx = xo[0] - fx, ddy = xo[1] - fy;
                    const bool near_center = sqrt(ddx * ddx + ddy * ddy + 0.0) < 10 * dpmm;
                    if ((radius_mm * 2 < c.p.max_wobble_diameter && near_center) || !c.p.recursive) {
                        verdict = 1;
                        R.n_peaks = npk;
                        R.n_lines = nl;
                        R.iterations = iterations;
                        R.radius_px = rpx;
                        R.profile_len = n;
                        R.wobble_x = xo[0];
                        R.wobble_y = xo[1];
                        R.wobble_radius_px = fo;
                        R.wobble_radius_mm = radius_mm;
                        R.passed = radius_mm * 2 < c.p.tolerance ? 1 : 0;
                        for (int k = 0; k < nl; k++) {     // calculate_angles (starshot.py:817-834)
                            const double m = (s_lines[k].y1 - s_lines[k].y2) / (s_lines[k].x1 - s_lines[k].x2);
                            double phi = atan(m) * (180.0 / PI) - 90;
                            if (phi > 90) phi -= 180;
                            else if (phi <= -90) phi += 180;
                            R.angles[k] = phi;
                        }
                    }
                }
            }
            if (lane == 0) {
                if (verdict == 2) { R.status = fail; R.iterations = iterations; }
                if (verdict != 0) {
                    row_verdict[fi * SS_ROWS + row] = verdict;
                    __threadfence();
                    atomicMin(&best[fi], order);
                }
                s_ctl[2] = verdict;
            }
        }
        __syncthreads();
        const int verdict = s_ctl[2];
        __syncthreads();
        if (verdict != 0) return;
    }
}

// First row (in order) of rows [row0, row0 + nrows) that has a verdict -> the frame's result; after the last round a frame without any
// verdict has exhausted the product: RuntimeError "unable to determine a reasonable wobble" (starshot.py:372-376).
__global__ void __launch_bounds__(128)
k_star_pick(int row0, int nrows, int last_round, const int* __restrict__ row_verdict, const epid_star_result* __restrict__ row_res,
            int* __restrict__ done, epid_star_result* __restrict__ res) {
    const int fi = blockIdx.x;
    if (res[fi].status != EPID_STAR_OK || done[fi]) return;
    int win = -1;
    for (int r = row0; r < row0 + nrows; r++)
        if (row_verdict[fi * SS_ROWS + r] != 0) { win = r; break; }
    __syncthreads();
    if (win < 0) {
        if (last_round && threadIdx.x == 0) { res[fi].status = EPID_STAR_NO_WOBBLE; res[fi].iterations = 1 + 11 * 11; }
        return;
    }
    // the fields the candidate loop fills (iterations .. passed); status / start point / local_max come from k_star_front
    const epid_star_result& S = row_res[(size_t)fi * SS_ROWS + win];
    constexpr int w0 = (int)(offsetof(epid_star_result, iterations) / 4), w1 = (int)(sizeof(epid_star_result) / 4);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&S);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&res[fi]);
    for (int k = w0 + threadIdx.x; k < w1; k += blockDim.x) dst[k] = src[k];
    if (threadIdx.x == 0) {
        if (row_verdict[fi * SS_ROWS + win] == 2) res[fi].status = S.status;
        done[fi] = 1;
    }
}

}  // namespace epid

// ------------------------------------------------------------------------------------------------ circle profiles
// CircleProfile / CollapsedCircleProfile._profile (core/profile.py:2244-2283, 2446-2483) of ONE image: for every sample angle
// radians[i] the sum over `nprof` radii of scipy.ndimage.map_coordinates(image, [y, x], order=0) (nearest neighbour, 0 outside),
// divided by nprof for the collapsed profile.  Also returns x / y locations on the nominal radius.
template <typename T>
__global__ void __launch_bounds__(256)
k_circle_profile(const T* __restrict__ img, int H, int W, double cx, double cy, double radius, double r_lo, double r_hi, int nprof,
                 int collapsed, double first, double delta, int n, int ccw, double* __restrict__ prof, double* __restrict__ xloc,
                 double* __restrict__ yloc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int k = ccw ? n - 1 - i : i;                          // rads[::-1] when counter-clockwise
    const double rad = k == 0 ? first : first + (double)k * delta;   // np.arange: first + i * delta
    const double cs = cos(rad), sn = sin(rad);
    const double rstep = nprof > 1 ? (r_hi - r_lo) / (double)(nprof - 1) : 0.0;
    double acc = 0.0;
    for (int p = 0; p < nprof; p++) {
        const double rk = !collapsed ? radius : (p == nprof - 1 && nprof > 1 ? r_hi : (double)p * rstep + r_lo);
        const double yc = sn * rk + cy, xc = cs * rk + cx;
        double v = 0.0;
        if (yc >= 0.0 && yc <= (double)(H - 1) && xc >= 0.0 && xc <= (double)(W - 1))
            v = (double)img[(size_t)((int)floor(yc + 0.5)) * W + (int)floor(xc + 0.5)];
        acc += v;
    }
    prof[i] = collapsed ? acc / (double)nprof : acc;
    xloc[i] = cs * radius + cx;
    yloc[i] = sn * radius + cy;
}

using namespace epid;

namespace {

PctPlan star_pct_plan(int n, double q_percent) {   // numpy 'linear' virtual index (same arithmetic as pf.cu pct_plan)
    const double q = q_percent / 100.0;
    const double vi = (double)n * q + (1.0 + q * (1.0 - 1.0 - 1.0)) - 1.0;
    double prev = floor(vi);
    PctPlan p;
    p.gamma = vi - prev;
    double next = prev + 1.0;
    if (prev < 0) prev = 0;
    if (next < 0) next = 0;
    if (prev > n - 1) prev = n - 1;
    if (next > n - 1) next = n - 1;
    p.prev = (int)prev;
    p.next = (int)next;
    return p;
}

__global__ void k_star_refs(const uint16_t* base, int n, int H, int W, int top, int left, FrameRef* full, FrameRef* central) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    full[i].origin = base + (size_t)i * H * W;
    full[i].pitch = W;
    full[i].pad = 0;
    central[i].origin = base + (size_t)i * H * W + (size_t)top * W + left;
    central[i].pitch = W;
    central[i].pad = 0;
}

}  // namespace

extern "C" int32_t epid_starshot_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_star_params* p, const double* gauss_weights,
                                         const int32_t* gauss_offsets, int32_t max_sigma, epid_star_result* results) {
    EPID_REQUIRE(ctx && frames && p && gauss_weights && gauss_offsets && results, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(frames->dtype == EPID_U16, EPID_ERR_UNSUPPORTED, "starshot frames must be uint16");
    EPID_REQUIRE(p->dpmm > 0, EPID_ERR_INVALID, "dpmm must be positive");
    EPID_REQUIRE(p->radius >= 0.2 && p->radius <= 0.95, EPID_ERR_INVALID, "radius must be between 0.2 and 0.95");
    EPID_REQUIRE(p->min_peak_height >= 0.05 && p->min_peak_height <= 0.95, EPID_ERR_INVALID, "min_peak_height must be between 0.05 and 0.95");
    EPID_REQUIRE(max_sigma >= 1, EPID_ERR_INVALID, "empty gaussian table");
    EPID_CUDA(cudaSetDevice(ctx->device));
    const int n = frames->n, H = frames->h, W = frames->w;
    EPID_REQUIRE(H >= 9 && W >= 9, EPID_ERR_UNSUPPORTED, "frame too small");
    StarConst hc;
    memset(&hc, 0, sizeof(hc));
    hc.p = *p;
    hc.H = H;
    hc.W = W;
    hc.top = (int)((double)H / 3);
    hc.left = (int)((double)W / 3);
    hc.ch = hc.top * 2 - hc.top;
    hc.cw = hc.left * 2 - hc.left;
    hc.p4 = star_pct_plan(H * W, 4.0);
    hc.p50 = star_pct_plan(H * W, 50.0);
    hc.p96 = star_pct_plan(H * W, 96.0);
    hc.p90 = star_pct_plan(hc.ch * hc.cw, 90.0);
    hc.nmax = 10 * (H > W ? H : W) + 64;
    hc.max_sigma = max_sigma;
    hc.npad = hc.nmax + 2 * (int)(4.0 * max_sigma + 0.5) + 8;
    const size_t gw_count = (size_t)gauss_offsets[max_sigma] + (size_t)(2 * (int)(4.0 * max_sigma + 0.5) + 1);
    // scratch
    size_t o = 0;
    auto sz = [&](size_t b) { const size_t r = o; o += (b + 255) / 256 * 256; return r; };
    const size_t o_cst = sz(sizeof(StarConst)), o_rf = sz(sizeof(FrameRef) * n), o_rc = sz(sizeof(FrameRef) * n);
    const size_t o_sf = sz(sizeof(FrameStats) * n), o_sc = sz(sizeof(FrameStats) * n), o_fr = sz(sizeof(StarFrame) * n);
    const size_t o_res = sz(sizeof(epid_star_result) * n), o_gw = sz(sizeof(double) * gw_count), o_go = sz(sizeof(int) * (max_sigma + 1));
    const size_t o_pa = sz(sizeof(double) * (size_t)n * SS_ROUND_ROWS * hc.nmax), o_pb = sz(sizeof(double) * (size_t)n * SS_ROUND_ROWS * hc.nmax);
    const size_t o_pc = sz(sizeof(double) * (size_t)n * SS_ROUND_ROWS * hc.npad);
    const size_t o_flags = sz(sizeof(int) * (size_t)n * (2 + SS_ROWS));        // done, best, row verdicts
    const size_t o_rows = sz(sizeof(epid_star_result) * (size_t)n * SS_ROWS);
    int rc = ensure_scratch(ctx, o);
    if (rc != EPID_OK) return rc;
    char* base = (char*)ctx->scratch;
    StarConst* d_cst = (StarConst*)(base + o_cst);
    FrameRef* d_rf = (FrameRef*)(base + o_rf);
    FrameRef* d_rc = (FrameRef*)(base + o_rc);
    FrameStats* d_sf = (FrameStats*)(base + o_sf);
    FrameStats* d_sc = (FrameStats*)(base + o_sc);
    StarFrame* d_fr = (StarFrame*)(base + o_fr);
    epid_star_result* d_res = (epid_star_result*)(base + o_res);
    double* d_gw = (double*)(base + o_gw);
    int* d_go = (int*)(base + o_go);
    cudaStream_t st = ctx->stream;
    EPID_CUDA(cudaMemcpyAsync(d_cst, &hc, sizeof(hc), cudaMemcpyHostToDevice, st));
    EPID_CUDA(cudaMemcpyAsync(d_gw, gauss_weights, sizeof(double) * gw_count, cudaMemcpyHostToDevice, st));
    EPID_CUDA(cudaMemcpyAsync(d_go, gauss_offsets, sizeof(int) * (max_sigma + 1), cudaMemcpyHostToDevice, st));
    EPID_CUDA(cudaMemsetAsync(d_res, 0, sizeof(epid_star_result) * n, st));
    k_star_refs<<<(n + 127) / 128, 128, 0, st>>>((const uint16_t*)frames->dptr, n, H, W, hc.top, hc.left, d_rf, d_rc);
    ctx->launches++;
    // exact order statistics: frame (p4, p50, p96) and central third (p90 and its mirror for flipped frames)
    StatsGeom g;
    rc = make_stats_geom(&g, H, W);
    if (rc != EPID_OK) return rc;
    g.nranks = 6;
    g.ranks[0] = hc.p4.prev; g.ranks[1] = hc.p4.next;
    g.ranks[2] = hc.p50.prev; g.ranks[3] = hc.p50.next;
    g.ranks[4] = hc.p96.prev; g.ranks[5] = hc.p96.next;
    g.box = 0;
    rc = launch_frame_stats_inversion(ctx, st, g, d_rf, n, d_sf, nullptr, nullptr);
    if (rc != EPID_OK) return rc;
    StatsGeom gc;
    rc = make_stats_geom(&gc, hc.ch, hc.cw);
    if (rc != EPID_OK) return rc;
    const int nc = hc.ch * hc.cw;
    gc.nranks = 4;
    gc.ranks[0] = hc.p90.prev; gc.ranks[1] = hc.p90.next;
    gc.ranks[2] = nc - 1 - hc.p90.next; gc.ranks[3] = nc - 1 - hc.p90.prev;
    gc.box = 0;
    rc = launch_frame_stats(ctx, st, gc, d_rc, n, d_sc, nullptr, nullptr);
    if (rc != EPID_OK) return rc;
    {
        const int n_max = hc.cw > hc.ch ? hc.cw : hc.ch;
        const int n_al = (n_max + 3) & ~3;
        const size_t smem = sizeof(double) * (size_t)(2 * n_al + 5 * SS_PEAK_CAP) + sizeof(int) * (size_t)(5 * SS_PEAK_CAP + SS_THREADS + 8);
        EPID_SMEM_OPT_IN(ctx, k_star_front, smem);
        k_star_front<<<n, SS_THREADS, smem, st>>>(d_cst, d_rf, d_sf, d_sc, d_fr, d_res);
        ctx->launches++;
    }
    {
        // candidate rows in rounds (see k_star_rows): row 0, then SS_ROUND_ROWS rows at a time; CTAs of settled frames exit at once
        int* d_done = (int*)(base + o_flags);
        int* d_best = d_done + n;
        int* d_verdict = d_best + n;
        epid_star_result* d_rows = (epid_star_result*)(base + o_rows);
        EPID_CUDA(cudaMemsetAsync(d_done, 0, sizeof(int) * (size_t)n, st));
        EPID_CUDA(cudaMemsetAsync(d_best, 0x7f, sizeof(int) * (size_t)n, st));
        EPID_CUDA(cudaMemsetAsync(d_verdict, 0, sizeof(int) * (size_t)n * SS_ROWS, st));
        EPID_CUDA(cudaMemsetAsync(d_rows, 0, sizeof(epid_star_result) * (size_t)n * SS_ROWS, st));
        // rounds: the caller's pair alone (frames that pass at once cost one candidate), the first four radii together (a frame that
        // needs the product usually fails a few whole rows), then two rows at a time: rows after the accepted one are wasted work
        static const int kRound[] = {1, SS_ROUND_ROWS, 2, 2, 3};
        int round = 0;
        for (int row0 = 0; row0 < SS_ROWS; round++) {
            int nrows = kRound[round < 5 ? round : 4];
            if (nrows > SS_ROWS - row0) nrows = SS_ROWS - row0;
            k_star_rows<<<dim3(n, nrows), SS_THREADS, 0, st>>>(d_cst, d_rf, d_fr, d_gw, d_go, (double*)(base + o_pa), (double*)(base + o_pb),
                                                               (double*)(base + o_pc), d_res, row0, d_done, d_best, d_verdict, d_rows);
            k_star_pick<<<n, 128, 0, st>>>(row0, nrows, row0 + nrows >= SS_ROWS ? 1 : 0, d_verdict, d_rows, d_done, d_res);
            ctx->launches += 2;
            row0 += nrows;
            // analyze(recursive=False) usually settles in round 0 (first candidate accepted or NO_LINES); a LineManager ValueError (a line
            // too far from the start point) still moves on to the next candidate in the reference (starshot.py:346-376), so all rounds are
            // enqueued either way -- CTAs of settled frames exit at once
        }
    }
    EPID_CUDA(cudaGetLastError());
    EPID_CUDA(cudaMemcpyAsync(results, d_res, sizeof(epid_star_result) * n, cudaMemcpyDeviceToHost, st));
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("starshot pipeline failed: %s", cudaGetErrorString(e)); return EPID_ERR_CUDA; }
    return EPID_OK;
}

extern "C" int32_t epid_circle_profile(epid_ctx* ctx, const epid_batch* image, double cx, double cy, double radius, double start_angle,
                                       int32_t ccw, double sampling_ratio, int32_t collapsed, double width_ratio, int32_t num_profiles,
                                       int32_t cap, double* profile, double* x_locations, double* y_locations, int32_t* count) {
    EPID_REQUIRE(ctx && image && profile && x_locations && y_locations && count, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(image->n == 1, EPID_ERR_INVALID, "circle profiles are taken from a single image");
    EPID_REQUIRE(image->dtype == EPID_U16 || image->dtype == EPID_F64 || image->dtype == EPID_U8 || image->dtype == EPID_F32,
                 EPID_ERR_UNSUPPORTED, "image dtype not supported");
    EPID_REQUIRE(radius > 0 && sampling_ratio > 0, EPID_ERR_INVALID, "radius and sampling_ratio must be positive");
    EPID_REQUIRE(!collapsed || (num_profiles >= 1 && width_ratio >= 0 && width_ratio <= 1), EPID_ERR_INVALID, "bad band parameters");
    EPID_CUDA(cudaSetDevice(ctx->device));
    const int H = image->h, W = image->w;
    // Array size check of CircleProfile.__init__ (core/profile.py:2228-2230, 2395-2402)
    EPID_REQUIRE(!((double)W < radius + cx || (double)H < radius + cy), EPID_ERR_INVALID, "Array size not large enough to compute profile");
    const double PI = 3.141592653589793;
    const double r_lo = radius * (1 - width_ratio), r_hi = radius * (1 + width_ratio);
    const double rmax = collapsed ? (r_hi > r_lo ? r_hi : r_lo) : radius;     // max(np.linspace(r_lo, r_hi, num))
    const double size = PI * rmax * 2 * sampling_ratio;
    const double interval = (2 * PI) / size;
    const double start = 0 + start_angle, stop = (2 * PI) + start_angle - interval;
    const double span = (stop - start) / interval;                             // np.arange length
    const int n = span > 0 ? (int)ceil(span) : 0;
    EPID_REQUIRE(n >= 1, EPID_ERR_INVALID, "empty profile");
    EPID_REQUIRE(n <= cap, EPID_ERR_INVALID, "output capacity %d too small for %d samples", cap, n);
    const double first = start, delta = (start + interval) - start;           // np.arange fills first + i * (next - first)
    int rc = ensure_scratch(ctx, sizeof(double) * 3 * (size_t)n + 1024);
    if (rc != EPID_OK) return rc;
    double* d_p = (double*)ctx->scratch;
    double* d_x = d_p + n;
    double* d_y = d_x + n;
    const int grid = (n + 255) / 256;
    const int np_ = collapsed ? num_profiles : 1;
    switch (image->dtype) {
        case EPID_U16: k_circle_profile<uint16_t><<<grid, 256, 0, ctx->stream>>>((const uint16_t*)image->dptr, H, W, cx, cy, radius, r_lo, r_hi, np_, collapsed, first, delta, n, ccw, d_p, d_x, d_y); break;
        case EPID_U8: k_circle_profile<uint8_t><<<grid, 256, 0, ctx->stream>>>((const uint8_t*)image->dptr, H, W, cx, cy, radius, r_lo, r_hi, np_, collapsed, first, delta, n, ccw, d_p, d_x, d_y); break;
        case EPID_F32: k_circle_profile<float><<<grid, 256, 0, ctx->stream>>>((const float*)image->dptr, H, W, cx, cy, radius, r_lo, r_hi, np_, collapsed, first, delta, n, ccw, d_p, d_x, d_y); break;
        default: k_circle_profile<double><<<grid, 256, 0, ctx->stream>>>((const double*)image->dptr, H, W, cx, cy, radius, r_lo, r_hi, np_, collapsed, first, delta, n, ccw, d_p, d_x, d_y); break;
    }
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    EPID_CUDA(cudaMemcpyAsync(profile, d_p, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaMemcpyAsync(x_locations, d_x, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaMemcpyAsync(y_locations, d_y, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    *count = n;
    return EPID_OK;
}
