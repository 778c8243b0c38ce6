// Batched PicketFence.analyze() on the GPU.  One result per frame; frames never leave HBM between stages.
//
// Reference path reproduced (pylinac v3.46.0):
//   PFDicomImage.__init__ crop / _check_for_noise / check_inversion      picketfence.py:209-238, core/image.py:868-897
//   PicketFence.__init__ filter / ground / normalize                      picketfence.py:320-323
//   PicketFence.analyze (orientation, picket search, per-leaf windows)    picketfence.py:636-912, 1501-1526
//   MLCValue.get_peak_positions / error / marker_lines                    picketfence.py:1605-1628, 1701-1743
//   Picket.get_fit / dist2cax / skew                                      picketfence.py:1881-1923
//   aggregate results                                                      picketfence.py:439-562, 1313-1363, 1467-1469
//
// Exactness strategy: after ground()+normalize() the reference image is I = g / D with g = v - min (or max - v
// when inverted) and D = max - min, a monotone affine map of the uint16 frame.  Every sum, median, threshold and
// argmax is therefore evaluated EXACTLY on integers (g or 2g), and only the final 1-D profile arithmetic runs
// in fp64 (same operation order as numpy/scipy, FMA contraction disabled).
//
// Stages (all stream-ordered, no host round trip unless a frame is flagged noisy):
//   k_frame_stats   1 read   min/max/sum/row+col sums/corner boxes/exact p0.5,p99.5,median   (stats.cu)
//   k_pf_decide     -        noise flag, corner inversion, D, median in g units
//   k_pf_clamp_sums 1 read   row/col sums of max(2g, 2*median)  (orientation; skipped if orientation is given)
//   k_pf_profile    -        orientation, leaf profile, find_peaks -> pickets, spacing, leaves in view
//   k_pf_windows    ~0.5 read per (leaf, picket) window: validity, median profile, FWHM edges
//   k_pf_finalize   -        leaf-row pruning, per-picket line fit, errors, aggregates
#include <cmath>
#include <condition_variable>
#include <cstdlib>
#include <mutex>
#include <thread>
#include <pthread.h>
#include <sched.h>

// PicketFence profiles have ~1000 samples: find_peaks' 32-sample skip table (peaks.cuh) buys nothing here, and its 9 KB of static shared
// memory cost k_pf_tail a resident CTA per SM (measured: 103 us with the table, 77 us without; profiles/r2m_summary.md)
#define EPID_PK_MAXBLK 2
#include "pf_common.cuh"

namespace epid {

// ------------------------------------------------------------------------------------------------ init
// sel: frame i of this run is frame sel[i] of the batch (per-frame re-run of deferred frames); nullptr: identity
__global__ void k_pf_init(const uint16_t* base, int n, int H0, int W0, int crop, FrameRef* refs, PfFrame* fr, int* counters, const int* __restrict__ sel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { counters[0] = 0; counters[1] = 0; counters[2] = 0; }
    if (i >= n) return;
    refs[i].origin = base + (size_t)(sel ? sel[i] : i) * H0 * W0 + (size_t)crop * W0 + crop;
    refs[i].pitch = W0;
    refs[i].pad = 0;
    PfFrame& f = fr[i];
    f.status = EPID_PF_OK;
    f.noisy = 0;
    f.inv = 0;
    f.corner_inverted = 0;
    f.noise_passes = 0;
    f.n_pickets = 0;
    f.n_inview = 0;
    f.todo = 0;
    f.win2 = 0;
    f.orientation = 0;
}

// ------------------------------------------------------------------------------------------------ decide
// mode 0: first look (noise check only updates `noisy`), mode 1: after a noise-median pass (re-check noise),
// both: corner inversion + median.  post_filter: only D / median, inversion already materialised.
__global__ void k_pf_decide(const PfConst* __restrict__ cc, const FrameStats* __restrict__ st, PfFrame* fr, int n,
                            const int* __restrict__ select, int check_noise, int* counters) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (select && !select[i]) return;
    pf_decide_frame(*cc, st[i], fr[i], check_noise, counters);
}

// ------------------------------------------------------------------------------------------------ clamped sums
// PicketFence.orientation (picketfence.py:1509-1514): temp[temp < median] = median; np.sum(temp, 0); np.sum(temp, 1).
// In 2g units: sum of max(2g, med2).  Same CTA-per-frame streaming structure as k_frame_stats.
__global__ void __launch_bounds__(STATS_THREADS, 1)
k_pf_clamp_sums(const StatsGeom g, const FrameRef* __restrict__ frames, const PfFrame* __restrict__ fr, int nframes,
                uint32_t* __restrict__ rowsum2, uint32_t* __restrict__ colsum2) {
    extern __shared__ uint32_t smem[];
    uint32_t* colpart = smem;                          // STATS_THREADS * 8
    uint32_t* rowsum_sm = colpart + STATS_THREADS * 8; // H
    const int tid = threadIdx.x, lane = tid & 31;
    const int grp = tid / g.vprp, jc = tid - grp * g.vprp;
    const bool active_grp = grp < g.groups;
    for (int fi = blockIdx.x; fi < nframes; fi += gridDim.x) {
        const PfFrame& pf = fr[fi];
        if (pf.status != EPID_PF_OK) continue;
        const FrameRef frf = frames[fi];
        const uint16_t* __restrict__ f = frf.origin;
        const int pitch = frf.pitch;
        const bool aligned = (pitch % 8) == 0;
        const int mis = aligned ? (int)((reinterpret_cast<uintptr_t>(f) >> 1) & 7) : 0;
        const int col_first = jc * 8 - mis;
        uint32_t valid = 0;
        if (active_grp) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int c = col_first + k;
                if (c >= 0 && c < g.W) valid |= 1u << k;
            }
        }
        const bool active = valid != 0;
        const int inv = pf.inv;
        const uint32_t mn = pf.mn, mx = pf.mx, med2 = pf.med2;
        for (int i = tid; i < g.H; i += STATS_THREADS) rowsum_sm[i] = 0;
        __syncthreads();
        uint32_t csum[8];
#pragma unroll
        for (int k = 0; k < 8; k++) csum[k] = 0;
        if (active_grp) {
            constexpr int U = 4;
            for (int r = grp; r < g.H; r += g.groups * U) {
                uint4 q[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int rr = r + u * g.groups;
                    q[u] = make_uint4(0, 0, 0, 0);
                    if (rr < g.H && active) {
                        const uint16_t* rowp = f + (size_t)rr * pitch;
                        if (aligned) {
                            q[u] = ldg_stream16(rowp + col_first);
                        } else {
                            uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
                            for (int k = 0; k < 8; k++)
                                if (valid >> k & 1) w[k >> 1] |= (uint32_t)__ldg(rowp + col_first + k) << ((k & 1) * 16);
                            q[u] = make_uint4(w[0], w[1], w[2], w[3]);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int rr = r + u * g.groups;
                    if (rr >= g.H) break;
                    const uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
                    uint32_t rs = 0;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        if (valid >> k & 1) {
                            const uint32_t v = (w[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
                            const uint32_t g2 = 2u * (inv ? mx - v : v - mn);
                            const uint32_t cl = max(g2, med2);
                            csum[k] += cl;
                            rs += cl;
                        }
                    }
                    rs = warp_sum(rs);
                    if (lane == 0) atomicAdd(&rowsum_sm[rr], rs);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) colpart[tid * 8 + k] = active ? csum[k] : 0u;
        __syncthreads();
        for (int x = tid; x < g.W; x += STATS_THREADS) {
            const int ac = x + mis;
            uint32_t s = 0;
            for (int gg = 0; gg < g.groups; gg++) s += colpart[(gg * g.vprp) * 8 + ac];
            colsum2[(size_t)fi * g.W + x] = s;
        }
        for (int y = tid; y < g.H; y += STATS_THREADS) rowsum2[(size_t)fi * g.H + y] = rowsum_sm[y];
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ profile / pickets
__global__ void __launch_bounds__(PROF_THREADS)
k_pf_profile(const PfConst* __restrict__ cc, PfFrame* fr, const uint32_t* __restrict__ rowsum, const uint32_t* __restrict__ colsum,
             const uint32_t* __restrict__ rowsum2, const uint32_t* __restrict__ colsum2) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int fi = blockIdx.x;
    const PfConst& c = *cc;
    pf_profile_block(c, fr[fi], rowsum + (size_t)fi * c.H, colsum + (size_t)fi * c.W, rowsum2 + (size_t)fi * c.H,
                     colsum2 + (size_t)fi * c.W, smraw);
}

// ------------------------------------------------------------------------------------------------ windows
// One warp per (leaf, picket) window.  Canonical window coordinates: i in [0, nr) across the leaf (the axis the
// median collapses), j in [0, nc) along leaf travel.
__global__ void __launch_bounds__(WIN_WARPS * 32)
k_pf_windows(const PfConst* __restrict__ cc, const FrameRef* __restrict__ frames, PfFrame* fr, PfWin* __restrict__ wins, int todo_only) {
    __shared__ __align__(16) uint16_t s_px[WIN_WARPS][WIN_CAP_PX];     // staged g values; later aliased by the fp64 profile
    __shared__ uint32_t s_m2[WIN_WARPS][WIN_MAX_NC];
    const int fi = blockIdx.y;
    const PfConst& c = *cc;
    PfFrame& f = fr[fi];
    if (f.status != EPID_PF_OK) return;
    if (todo_only && !f.todo) return;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int li = blockIdx.x; li < f.n_inview; li += gridDim.x) {   // in-view leaf slot
    const int H = c.H, W = c.W;
    const int orient = f.orientation;
    const int leaf = f.inview[li];
    const double dpmm = c.p.dpmm;
    const double lw_px = c.p.leaf_width_mm[leaf] * dpmm;
    const double lc_px = c.p.leaf_center_mm[leaf] * dpmm + (orient == 0 ? (double)H / 2.0 : (double)W / 2.0);
    const FrameRef frf = frames[fi];
    const int inv = f.inv;
    const uint32_t mn = f.mn, mx = f.mx;
    const double Dd = (double)f.D;
    uint16_t* px = s_px[wid];
    uint32_t* m2 = s_m2[wid];
    double* xs = reinterpret_cast<double*>(px);

    for (int pk = wid; pk < f.n_pickets; pk += WIN_WARPS) {
        PfWin& out = wins[((size_t)fi * PF_L + li) * PF_P + pk];
        if (todo_only && out.valid != -1) continue;   // already done by k_pf_windows_fast
        const double pidx = (double)f.picket_idx[pk];
        const double spacing = f.spacing;
        // _get_mlc_window (picketfence.py:859-886): python int() truncates toward zero
        int a0 = max((int)(pidx - spacing / 2.0), 0);                                   // along travel
        int a1 = min((int)(pidx + spacing / 2.0), orient == 0 ? W : H);
        int b0 = max((int)(lc_px - lw_px / 2.0), 0);                                    // across the leaf
        int b1 = min((int)(lc_px + lw_px / 2.0), orient == 0 ? H : W);
        const int nc = a1 - a0, nr = b1 - b0;
        if (nc <= 0 || nr <= 0) {           // empty slice: np.max raises ValueError in the reference
            if (lane == 0) { out.valid = 0; out.l = 0; out.r = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            continue;
        }
        if (nc > WIN_MAX_NC || nr > WIN_MAX_NR) {
            if (lane == 0) { out.valid = 0; f.status = EPID_PF_CAPACITY; }
            continue;
        }
        // The window is processed in chunks of `cw` travel samples so that any spacing fits the staging buffer:
        // per chunk, stage g values (canonical layout px[i * cw + jj]), accumulate the validity statistics
        // (max, per-row sum and sum of squares) and take the per-sample median across the leaf.
        const int cw = min(nc, WIN_CAP_PX / nr);
        const int sag = c.p.sag_px;
        const int k1 = (nr - 1) / 2, k2 = nr / 2;
        uint32_t gmax = 0;
        unsigned long long rs1[2] = {0, 0}, rs2[2] = {0, 0};   // row i lives on lane i & 31, slot i >> 5
        uint32_t lmin = 0xffffffffu, lmax = 0;
        for (int j0 = 0; j0 < nc; j0 += cw) {
            const int cn = min(cw, nc - j0);
            __syncwarp();
            // np.roll(sag) folded into the source index
            if (orient == 0) {
                for (int t = lane; t < nr * cn; t += 32) {
                    const int i = t / cn, jj = t - i * cn;
                    int row = b0 + i - sag;
                    row %= H; if (row < 0) row += H;
                    const uint32_t v = __ldg(frf.origin + (size_t)row * frf.pitch + a0 + j0 + jj);
                    const uint32_t g = inv ? mx - v : v - mn;
                    px[i * cn + jj] = (uint16_t)g;
                    gmax = max(gmax, g);
                }
            } else {
                for (int t = lane; t < nr * cn; t += 32) {
                    const int jj = t / nr, i = t - jj * nr;   // lanes run along the memory-contiguous axis
                    int col = b0 + i - sag;
                    col %= W; if (col < 0) col += W;
                    const uint32_t v = __ldg(frf.origin + (size_t)(a0 + j0 + jj) * frf.pitch + col);
                    const uint32_t g = inv ? mx - v : v - mn;
                    px[i * cn + jj] = (uint16_t)g;
                    gmax = max(gmax, g);
                }
            }
            __syncwarp();
            for (int i = 0; i < nr; i++) {
                unsigned long long s1 = 0, s2 = 0;
                for (int jj = lane; jj < cn; jj += 32) {
                    const unsigned long long g = px[i * cn + jj];
                    s1 += g;
                    s2 += g * g;
                }
                s1 = warp_sum(s1);
                s2 = warp_sum(s2);
                if ((i & 31) == lane) { rs1[i >> 5] += s1; rs2[i >> 5] += s2; }
            }
            // np.median(window, axis) -> 2*median per travel sample (picketfence.py:1605-1609)
            for (int jj = lane; jj < cn; jj += 32) {
                uint32_t va = 0, vb = 0;
                for (int i = 0; i < nr; i++) {
                    const uint32_t v = px[i * cn + jj];
                    int rank = 0;
                    for (int i2 = 0; i2 < nr; i2++) {
                        const uint32_t o = px[i2 * cn + jj];
                        rank += (o < v || (o == v && i2 < i)) ? 1 : 0;
                    }
                    if (rank == k1) va = v;
                    if (rank == k2) vb = v;
                }
                const uint32_t m = va + vb;
                m2[j0 + jj] = m;
                lmin = min(lmin, m);
                lmax = max(lmax, m);
            }
        }
        gmax = warp_max(gmax);
        __syncwarp();
        // ---- _is_mlc_peak_in_window (picketfence.py:847-857)
        // std across travel for each i: sqrt(nc*S2 - S1^2) / (nc * D), exact integer numerator
        double sd[2] = {-1.0, -1.0};
#pragma unroll
        for (int sl = 0; sl < 2; sl++) {
            if (sl * 32 + lane < nr) {
                const double num = (double)((unsigned long long)nc * rs2[sl] - rs1[sl] * rs1[sl]);
                sd[sl] = sqrt(num) / ((double)nc * Dd);
            }
        }
        // max and median of the nr std values (rank counting through shuffles)
        double sd_max = fmax(sd[0], sd[1]);
        sd_max = warp_max(sd_max);
        double med_a = 0.0, med_b = 0.0;
        {
            int rank[2] = {0, 0};
            for (int t = 0; t < nr; t++) {
                const double o = __shfl_sync(0xffffffffu, (t >> 5) ? sd[1] : sd[0], t & 31);
#pragma unroll
                for (int sl = 0; sl < 2; sl++) {
                    const int me = sl * 32 + lane;
                    if (me < nr && (o < sd[sl] || (o == sd[sl] && t < me))) rank[sl]++;
                }
            }
            double ca = 0.0, cb = 0.0;
#pragma unroll
            for (int sl = 0; sl < 2; sl++) {
                const int me = sl * 32 + lane;
                if (me < nr) {
                    if (rank[sl] == k1) ca = sd[sl];
                    if (rank[sl] == k2) cb = sd[sl];
                }
            }
            // exactly one lane holds each; sum-reduce to broadcast (others contribute +0.0)
            med_a = warp_sum(ca);
            med_b = warp_sum(cb);
        }
        const double sd_med = (nr & 1) ? med_a : (med_a + med_b) / 2.0;
        const bool above = ((double)gmax / Dd) > c.p.height_threshold * f.picket_val[pk];
        const bool not_edge = sd_max < c.p.edge_threshold * sd_med;
        if (!(above && not_edge)) {
            if (lane == 0) { out.valid = 0; out.l = 0; out.r = 0; }
            __syncwarp();
            continue;
        }
        lmin = warp_min(lmin);
        lmax = warp_max(lmax);
        __syncwarp();
        if (lmax == lmin) {  // flat profile: the reference divides by zero and then finds no peak
            if (lane == 0) { out.valid = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            continue;
        }
        // ---- FWXMProfilePhysical(ground=True, normalization=MAX) (core/profile.py:204-240)
        const double den = (double)(lmax - lmin);
        for (int j = lane; j < nc; j += 32) xs[j] = (double)(m2[j] - lmin) / den;
        __syncwarp();
        // ---- find_peaks(values, fwxm_height=0.5, max_number=1) by prominence (core/profile.py:602-611, 2545-2623)
        double best_prom = -1.0;
        int best_idx = -1, best_lb = 0, best_rb = 0;
        for (int i = 1 + lane; i < nc - 1; i += 32) {
            if (xs[i - 1] < xs[i]) {
                int ahead = i + 1;
                while (ahead < nc - 1 && xs[ahead] == xs[i]) ahead++;
                if (xs[ahead] < xs[i]) {
                    const int p = (i + ahead - 1) / 2;
                    const double xp = xs[p];
                    int k = p, lb = p;
                    double lm = xp;
                    while (k >= 0 && xs[k] <= xp) { if (xs[k] < lm) { lm = xs[k]; lb = k; } k--; }
                    k = p;
                    int rb = p;
                    double rm = xp;
                    while (k <= nc - 1 && xs[k] <= xp) { if (xs[k] < rm) { rm = xs[k]; rb = k; } k++; }
                    const double prom = xp - fmax(lm, rm);
                    if (prom > best_prom || (prom == best_prom && p > best_idx)) { best_prom = prom; best_idx = p; best_lb = lb; best_rb = rb; }
                }
            }
        }
        // warp arg-max by (prominence, index)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double op = __shfl_xor_sync(0xffffffffu, best_prom, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
            const int olb = __shfl_xor_sync(0xffffffffu, best_lb, o);
            const int orb = __shfl_xor_sync(0xffffffffu, best_rb, o);
            if (op > best_prom || (op == best_prom && oi > best_idx)) { best_prom = op; best_idx = oi; best_lb = olb; best_rb = orb; }
        }
        if (best_idx < 0) {
            if (lane == 0) { out.valid = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            __syncwarp();
            continue;
        }
        if (lane == 0) {
            const int p = best_idx;
            const double h = xs[p] - best_prom * 0.5;
            int k = p;
            while (best_lb < k && h < xs[k]) k--;
            double l = (double)k;
            if (xs[k] < h) l += (h - xs[k]) / (xs[k + 1] - xs[k]);
            k = p;
            while (k < best_rb && h < xs[k]) k++;
            double r = (double)k;
            if (xs[k] < h) r -= (h - xs[k]) / (xs[k - 1] - xs[k]);
            out.valid = 1;
            out.l = l;
            out.r = r;
        }
        __syncwarp();
    }
    }   // leaf slots
}

// ------------------------------------------------------------------------------------------------ host side
static PctPlan pct_plan(int n, double q_percent) {
    // numpy 'linear' (numpy/lib/_function_base_impl.py: _compute_virtual_index, _get_indexes, _get_gamma)
    const double q = q_percent / 100.0;
    const double vi = (double)n * q + (1.0 + q * (1.0 - 1.0 - 1.0)) - 1.0;
    double prev = floor(vi);
    double next = prev + 1.0;
    PctPlan p;
    p.gamma = vi - prev;
    if (prev < 0) prev = 0;
    if (next < 0) next = 0;
    if (prev > n - 1) prev = n - 1;
    if (next > n - 1) next = n - 1;
    p.prev = (int)prev;
    p.next = (int)next;
    return p;
}

struct PfWork {   // carved out of ctx->scratch
    FrameRef* refs;
    FrameRef* refs_b;        // ping-pong destination refs for median passes
    ValueMap* maps;
    PfFrame* fr;
    FrameStats* stats;
    uint32_t *rowsum, *colsum, *rowsum2, *colsum2;
    PfWin* wins;
    epid_pf_summary* summ;
    epid_pf_meas* meas;
    PfConst* cst;
    int* counters;           // [0] noisy count
    int* select;             // per-frame flags
    int* sel_idx;            // indices of the deferred frames (k_pf_collect_deferred), count in counters[2]
    void* front;             // partial sums / thresholds of the single-pass front end (pf_stream.cu)
    PfWinRec* winrec;        // records of the two-kernel window path (pf_windows2.cu)
    size_t total;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static void carve(PfWork& w, char* base, int n, int H, int W, int meas_cap) {
    size_t o = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + o : nullptr; o = align_up(o + bytes, 256); return p; };
    w.refs = (FrameRef*)take(sizeof(FrameRef) * n);
    w.refs_b = (FrameRef*)take(sizeof(FrameRef) * n);
    w.maps = (ValueMap*)take(sizeof(ValueMap) * n);
    w.fr = (PfFrame*)take(sizeof(PfFrame) * n);
    w.stats = (FrameStats*)take(sizeof(FrameStats) * n);
    w.rowsum = (uint32_t*)take(sizeof(uint32_t) * (size_t)n * H);
    w.colsum = (uint32_t*)take(sizeof(uint32_t) * (size_t)n * W);
    w.rowsum2 = (uint32_t*)take(sizeof(uint32_t) * (size_t)n * H);
    w.colsum2 = (uint32_t*)take(sizeof(uint32_t) * (size_t)n * W);
    w.wins = (PfWin*)take(sizeof(PfWin) * (size_t)n * PF_L * PF_P);
    w.summ = (epid_pf_summary*)take(sizeof(epid_pf_summary) * n);
    w.meas = (epid_pf_meas*)take(sizeof(epid_pf_meas) * (size_t)n * meas_cap);
    w.cst = (PfConst*)take(sizeof(PfConst));
    w.counters = (int*)take(sizeof(int) * 8);
    w.select = (int*)take(sizeof(int) * n);
    w.sel_idx = (int*)take(sizeof(int) * n);
    w.front = (void*)take(pf_front_scratch_bytes(n, H, W));
    w.winrec = (PfWinRec*)take(pf_win2_scratch_bytes(n));
    w.total = o;
}

__global__ void k_pf_mark_noisy(PfFrame* fr, int n, int* select, ValueMap* maps) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = (fr[i].status == EPID_PF_OK && fr[i].noisy) ? 1 : 0;
    select[i] = s;
    maps[i].inv = 0; maps[i].mn = 0; maps[i].mx = 0;
    if (s) fr[i].noise_passes++;
}

__global__ void k_pf_prepare_filter(PfFrame* fr, int n, int* select, ValueMap* maps, int user_invert) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    select[i] = fr[i].status == EPID_PF_OK ? 1 : 0;
    // materialise check_inversion's invert() only (analyze(invert=True) is applied after normalisation)
    maps[i].inv = fr[i].corner_inverted;
    maps[i].mn = fr[i].mn;
    maps[i].mx = fr[i].mx;
    (void)user_invert;
}

__global__ void k_pf_swap_refs(FrameRef* refs, const FrameRef* refs_b, const int* select, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (select[i]) refs[i] = refs_b[i];
}

__global__ void k_pf_set_dst_refs(FrameRef* refs_b, uint16_t* pool, int n, int H, int Wp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    refs_b[i].origin = pool + (size_t)i * H * Wp;
    refs_b[i].pitch = Wp;
    refs_b[i].pad = 0;
}

// Enqueue the whole pipeline for one device-resident batch on `stream`; results land in w.summ / w.meas (device).
// pf_front.cu
bool pf_front_supported(int H, int W, int pitch);
int launch_pf_front(epid_ctx* ctx, cudaStream_t stream, const PfConst* d_cst, const StatsGeom& g, const FrameRef* refs, int n, PfFrame* fr,
                    FrameStats* stats, int* counters, void* scratch, PfTimers* tm);

// fast == true: fused front kernel (sample-guided exact selection), no host round trip; frames it cannot certify
// (counters[1]) or that _check_for_noise flags (counters[0]) make the caller re-run the batch with fast == false.
__global__ void k_pf_collect_deferred(const PfFrame* __restrict__ fr, int n, int* __restrict__ sel_idx, int* counters, volatile int* host_flag) {
    // ascending list of the deferred frames (one block; n is a few hundred); host_flag: device-mapped page-locked int that
    // receives the count as well, so the host learns it from an event wait without a copy in the stream
    __shared__ int s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool d = i < n && fr[i].status == PF_STATUS_DEFERRED;
        const unsigned b = __ballot_sync(0xffffffffu, d);
        __shared__ int s_w[32];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        if (lane == 0) s_w[wid] = __popc(b);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; k++) off += s_w[k];
        if (d) sel_idx[off + __popc(b & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < (int)(blockDim.x >> 5); k++) t += s_w[k]; s_base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counters[2] = s_base;
        if (host_flag) { *host_flag = s_base; __threadfence_system(); }
    }
}

// ---- certified-noise fast re-run of deferred frames ------------------------------------------------------------------------
// _has_noise() (picketfence.py:229-238) is True as soon as max > 1.25 * p99.5.  With U = the largest integer with 1.25 * U < max,
// "#(pixels > U) <= npix - 1 - rank_next(99.5)" puts both order statistics behind the percentile at or below U, hence
// p99.5 <= U and the criterion holds whatever the minimum does: one exact count certifies the flag.  Such a frame is 3 x 3 median
// filtered like the reference does and handed to the certified fast pipeline as a new frame (which certifies "no noise" on the
// filtered pixels or defers again -> exact pipeline from the raw frame).
constexpr int CA_PARTS = 8;
__global__ void __launch_bounds__(256)
k_pf_count_above(const FrameRef* __restrict__ refs, const PfFrame* __restrict__ raw_fr, const int* __restrict__ sel, int H, int W, int* __restrict__ cnt) {
    const int i = blockIdx.y;
    const FrameRef fr = refs[i];
    const uint32_t mx = raw_fr[sel[i]].mx;
    const uint32_t U = (4u * mx + 4u) / 5u - 1u;            // ceil(0.8 mx) - 1: 1.25 U < mx (exact in binary64)
    const int r0 = (int)((long long)H * blockIdx.x / gridDim.x), r1 = (int)((long long)H * (blockIdx.x + 1) / gridDim.x);
    const int lane = threadIdx.x & 31;
    uint32_t c = 0;
    for (int r = r0 + (int)(threadIdx.x >> 5); r < r1; r += 8) {      // warp per row
        const uint16_t* row = fr.origin + (size_t)r * fr.pitch;
        int head = (int)((8 - ((uintptr_t)row & 7)) & 7) >> 1;        // pixels before the first 8-byte boundary
        if (head > W) head = W;
        if (lane < head) c += (uint32_t)row[lane] > U ? 1u : 0u;
        const int nb = (W - head) >> 2;
        const uint2* b = reinterpret_cast<const uint2*>(row + head);
        for (int j = lane; j < nb; j += 32) {
            const uint2 v = __ldg(b + j);
            c += ((v.x & 0xffffu) > U ? 1u : 0u) + ((v.x >> 16) > U ? 1u : 0u) + ((v.y & 0xffffu) > U ? 1u : 0u) + ((v.y >> 16) > U ? 1u : 0u);
        }
        const int t0 = head + nb * 4;
        if (t0 + lane < W) c += (uint32_t)row[t0 + lane] > U ? 1u : 0u;
    }
    c = warp_sum(c);
    if (lane == 0 && c) atomicAdd(&cnt[i], (int)c);
}

__global__ void k_pf_mark_certified(const int* __restrict__ cnt, int n, int limit, int* __restrict__ select) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) select[i] = cnt[i] <= limit ? 1 : 0;
}

__global__ void k_pf_set_passes(PfFrame* fr, const int* __restrict__ select, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && select[i]) fr[i].noise_passes = 1;
}

// local indices of the frames a re-run deferred again (loc, count in counters[2]) -> batch indices, in place
__global__ void k_pf_compose_sel(int* loc, const int* __restrict__ counters, const int* __restrict__ sel) {
    const int m = counters[2];
    for (int j = threadIdx.x; j < m; j += blockDim.x) loc[j] = sel[loc[j]];
}

__global__ void k_pf_scatter_results(const int* __restrict__ sel_idx, int m, const epid_pf_summary* __restrict__ s_src, const epid_pf_meas* __restrict__ m_src,
                                     epid_pf_summary* __restrict__ s_dst, epid_pf_meas* __restrict__ m_dst, int meas_cap) {
    // rows of the re-run frames back into the batch's result arrays (word copies; both structs are multiples of 4 bytes)
    const int j = blockIdx.x;
    if (j >= m) return;
    const int dst = sel_idx[j];
    const uint32_t* a = reinterpret_cast<const uint32_t*>(s_src + j);
    uint32_t* b = reinterpret_cast<uint32_t*>(s_dst + dst);
    for (int k = threadIdx.x; k < (int)(sizeof(epid_pf_summary) / 4); k += blockDim.x) b[k] = a[k];
    const uint32_t* c = reinterpret_cast<const uint32_t*>(m_src + (size_t)j * meas_cap);
    uint32_t* e = reinterpret_cast<uint32_t*>(m_dst + (size_t)dst * meas_cap);
    for (int k = threadIdx.x; k < (int)(sizeof(epid_pf_meas) / 4) * meas_cap; k += blockDim.x) e[k] = c[k];
}

constexpr int PF_REDO_CHUNK = 64;   // frames per sub-batch of the per-frame re-run

struct PfRedoIn {            // fast re-run of deferred frames (pf_redo_deferred)
    const PfFrame* raw_fr;   // PfFrame records of the batch's fast pass (mx of the raw frame)
    uint16_t* pool;          // room for n filtered frames (H x Wp uint16 each)
};

static int pf_run(epid_ctx* ctx, cudaStream_t stream, const uint16_t* d_frames, int n, int H0, int W0, const epid_pf_params* p,
                  int meas_cap, PfWork& w, uint16_t** pool3, PfTimers* tm, bool fast, const int* d_sel = nullptr,
                  cudaEvent_t front_evt = nullptr, int* host_flag = nullptr, const PfRedoIn* redo = nullptr) {
    const int crop = p->crop_px;
    const int H = H0 - 2 * crop, W = W0 - 2 * crop;
    StatsGeom g;
    int rc = make_stats_geom(&g, H, W);
    if (rc != EPID_OK) return rc;
    PfConst hc;
    memset(&hc, 0, sizeof(hc));
    hc.p = *p;
    hc.H = H;
    hc.W = W;
    hc.meas_cap = meas_cap;
    hc.post_filter = 0;
    hc.win2 = ctx->pf_win2;
    const int npix = H * W;
    hc.lo = pct_plan(npix, 0.5);
    hc.hi = pct_plan(npix, 99.5);
    hc.p85[0] = pct_plan(W, 85.0); hc.p99[0] = pct_plan(W, 99.0);
    hc.p85[1] = pct_plan(H, 85.0); hc.p99[1] = pct_plan(H, 99.0);
    g.nranks = 6;
    g.ranks[0] = hc.lo.prev; g.ranks[1] = hc.lo.next;
    g.ranks[2] = hc.hi.prev; g.ranks[3] = hc.hi.next;
    g.ranks[4] = (npix - 1) / 2; g.ranks[5] = npix / 2;
    g.box = 10;
    g.rp = (int)(0.01 * H) > 1 ? (int)(0.01 * H) : 1;
    g.cp = (int)(0.01 * W) > 1 ? (int)(0.01 * W) : 1;
    if (tm) { rc = tm->mark(stream, PF_STAGE_START); if (rc != EPID_OK) return rc; }
    EPID_CUDA(cudaMemcpyAsync(w.cst, &hc, sizeof(hc), cudaMemcpyHostToDevice, stream));
    const int tb = 128, nb = (n + tb - 1) / tb;
    k_pf_init<<<nb, tb, 0, stream>>>(d_frames, n, H0, W0, crop, w.refs, w.fr, w.counters, d_sel);
    ctx->launches++;
    // bench timers: around the frame-streaming kernel only (k_pf_stream inside launch_pf_front, k_frame_stats otherwise)
    if (fast) {
        if (redo) {      // certify _has_noise() == True by one exact count, filter those frames into the pool (see k_pf_count_above)
            const int Wp = (W + 7) / 8 * 8;
            EPID_CUDA(cudaMemsetAsync(w.sel_idx, 0, sizeof(int) * n, stream));
            k_pf_count_above<<<dim3(CA_PARTS, n), 256, 0, stream>>>(w.refs, redo->raw_fr, d_sel, H, W, w.sel_idx);
            k_pf_mark_certified<<<nb, tb, 0, stream>>>(w.sel_idx, n, npix - 1 - (int)hc.hi.next, w.select);
            k_pf_set_dst_refs<<<nb, tb, 0, stream>>>(w.refs_b, redo->pool, n, H, Wp);
            ctx->launches += 3;
            rc = launch_median_u16(ctx, stream, w.refs, w.refs_b, nullptr, w.select, n, H, W, 3);
            if (rc != EPID_OK) return rc;
            k_pf_swap_refs<<<nb, tb, 0, stream>>>(w.refs, w.refs_b, w.select, n);
            ctx->launches++;
        }
        rc = launch_pf_front(ctx, stream, w.cst, g, w.refs, n, w.fr, w.stats, w.counters, w.front, tm);
        if (rc != EPID_OK) return rc;
        if (redo) { k_pf_set_passes<<<nb, tb, 0, stream>>>(w.fr, w.select, n); ctx->launches++; }
        // which frames were deferred (none on ordinary batches): list + count for the per-frame re-run, known as soon as the front end is done
        k_pf_collect_deferred<<<1, 256, 0, stream>>>(w.fr, n, w.sel_idx, w.counters, host_flag);
        ctx->launches++;
        if (front_evt) EPID_CUDA(cudaEventRecord(front_evt, stream));
    } else {
        if (tm && tm->on) { rc = tm->record(stream); if (rc != EPID_OK) return rc; }
        rc = launch_frame_stats(ctx, stream, g, w.refs, n, w.stats, w.rowsum, w.colsum);
        if (rc == EPID_OK && tm && tm->on) rc = tm->record(stream);
    }
    if (rc != EPID_OK) return rc;
    if (!fast) {
    k_pf_decide<<<nb, tb, 0, stream>>>(w.cst, w.stats, w.fr, n, nullptr, 1, w.counters);
    ctx->launches++;
    // ---- _check_for_noise loop (picketfence.py:221-227): needs the host only to learn whether ANY frame is noisy
    int n_noisy = 0;
    EPID_CUDA(cudaMemcpyAsync(&n_noisy, w.counters, sizeof(int), cudaMemcpyDeviceToHost, stream));
    EPID_CUDA(cudaStreamSynchronize(stream));
    const int Wp = (W + 7) / 8 * 8;
    // the pools live until the end of the API call; re-run sub-batches of different sizes (<= PF_REDO_CHUNK) share them
    const size_t pool_bytes = sizeof(uint16_t) * (size_t)(n < PF_REDO_CHUNK ? PF_REDO_CHUNK : n) * H * Wp + 512;
    int pass = 0;
    uint16_t** pools = pool3;   // [0],[1]: ping-pong for the noise passes, [2]: PicketFence(filter=k)
    auto ensure_pool = [&](int which) -> int {
        if (!pools[which]) {
            cudaError_t e = cudaMalloc(&pools[which], pool_bytes);
            if (e != cudaSuccess) { set_error("cudaMalloc(%zu) for filtered frames failed: %s", pool_bytes, cudaGetErrorString(e)); return EPID_ERR_NOMEM; }
        }
        return EPID_OK;
    };
    int cur_pool = 0;
    while (n_noisy > 0 && pass < 5) {
        rc = ensure_pool(cur_pool);
        if (rc != EPID_OK) return rc;
        k_pf_mark_noisy<<<nb, tb, 0, stream>>>(w.fr, n, w.select, w.maps);
        k_pf_set_dst_refs<<<nb, tb, 0, stream>>>(w.refs_b, pools[cur_pool], n, H, Wp);
        ctx->launches += 2;
        rc = launch_median_u16(ctx, stream, w.refs, w.refs_b, nullptr, w.select, n, H, W, 3);
        if (rc != EPID_OK) return rc;
        k_pf_swap_refs<<<nb, tb, 0, stream>>>(w.refs, w.refs_b, w.select, n);
        ctx->launches++;
        // statistics of the filtered frames only (the others keep theirs): a select-aware re-run over all slots
        // would recompute identical numbers, so run it on all frames -- flagged ones are rare and this keeps
        // one code path.
        EPID_CUDA(cudaMemsetAsync(w.counters, 0, sizeof(int), stream));
        rc = launch_frame_stats(ctx, stream, g, w.refs, n, w.stats, w.rowsum, w.colsum);
        if (rc != EPID_OK) return rc;
        k_pf_decide<<<nb, tb, 0, stream>>>(w.cst, w.stats, w.fr, n, w.select, 1, w.counters);
        ctx->launches++;
        EPID_CUDA(cudaMemcpyAsync(&n_noisy, w.counters, sizeof(int), cudaMemcpyDeviceToHost, stream));
        EPID_CUDA(cudaStreamSynchronize(stream));
        cur_pool ^= 1;
        pass++;
    }
    // ---- optional PicketFence(filter=k) median (picketfence.py:320-321) on the (corner-)inverted image
    if (p->filter_size > 0) {
        rc = ensure_pool(2);
        if (rc != EPID_OK) return rc;
        k_pf_prepare_filter<<<nb, tb, 0, stream>>>(w.fr, n, w.select, w.maps, p->invert);
        k_pf_set_dst_refs<<<nb, tb, 0, stream>>>(w.refs_b, pools[2], n, H, Wp);
        ctx->launches += 2;
        rc = launch_median_u16(ctx, stream, w.refs, w.refs_b, w.maps, w.select, n, H, W, p->filter_size);
        if (rc != EPID_OK) return rc;
        k_pf_swap_refs<<<nb, tb, 0, stream>>>(w.refs, w.refs_b, w.select, n);
        ctx->launches++;
        hc.post_filter = 1;
        EPID_CUDA(cudaMemcpyAsync(w.cst, &hc, sizeof(hc), cudaMemcpyHostToDevice, stream));
        StatsGeom g2 = g;
        g2.box = 0;
        rc = launch_frame_stats(ctx, stream, g2, w.refs, n, w.stats, w.rowsum, w.colsum);
        if (rc != EPID_OK) return rc;
        k_pf_decide<<<nb, tb, 0, stream>>>(w.cst, w.stats, w.fr, n, nullptr, 0, w.counters);
        ctx->launches++;
    }
    // ---- orientation sums
    if (p->orientation < 0) {
        const size_t smem = sizeof(uint32_t) * (size_t)(STATS_THREADS * 8 + H);
        EPID_SMEM_OPT_IN(ctx, k_pf_clamp_sums, 64 * 1024);
        const int grid = n < ctx->sm_count ? n : ctx->sm_count;
        k_pf_clamp_sums<<<grid, STATS_THREADS, smem, stream>>>(g, w.refs, w.fr, n, w.rowsum2, w.colsum2);
        ctx->launches++;
    }
    {
        const size_t smem = pf_profile_smem_bytes(PROF_THREADS, H, W);
        EPID_SMEM_OPT_IN(ctx, k_pf_profile, smem);
        k_pf_profile<<<n, PROF_THREADS, smem, stream>>>(w.cst, w.fr, w.rowsum, w.colsum, w.rowsum2, w.colsum2);
        ctx->launches++;
    }
    if (tm) { rc = tm->mark(stream, PF_STAGE_EXACT_FRONT); if (rc != EPID_OK) return rc; }
    }   // !fast
    {
        // fast path for ordinary window sizes, then the generic kernel for whatever it left marked (valid == -1)
        if (hc.win2) {
            rc = launch_pf_windows2(ctx, stream, w.cst, w.refs, w.fr, w.winrec, w.wins, n, tm);
            if (rc != EPID_OK) return rc;
        }
        rc = launch_pf_windows_fast(ctx, stream, w.cst, w.refs, w.fr, w.wins, n);
        if (rc != EPID_OK) return rc;
        if (tm) { rc = tm->mark(stream, PF_STAGE_WINDOWS); if (rc != EPID_OK) return rc; }
        dim3 grid(p->n_leaves < 8 ? p->n_leaves : 8, n);   // exits at once unless the fast kernel left work (PfFrame.todo)
        k_pf_windows<<<grid, WIN_WARPS * 32, 0, stream>>>(w.cst, w.refs, w.fr, w.wins, 1);
        ctx->launches++;
        if (tm) { rc = tm->mark(stream, PF_STAGE_WINDOWS_GENERIC); if (rc != EPID_OK) return rc; }
    }
    rc = launch_pf_finalize(ctx, stream, w.cst, w.fr, w.wins, w.summ, w.meas, n, meas_cap);
    if (rc != EPID_OK) return rc;
    if (tm) { rc = tm->mark(stream, PF_STAGE_FINALIZE); if (rc != EPID_OK) return rc; }
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

// Per-frame fallback: the m frames the fast pipeline deferred (w.sel_idx, ascending) are re-run by the exact-histogram pipeline in
// sub-batches whose work area lives in ctx->scratch2, and their result rows are scattered into the batch's device result arrays.
static int ensure_scratch2(epid_ctx* ctx, size_t bytes) {
    if (ctx->scratch2_bytes >= bytes) return EPID_OK;
    if (ctx->scratch2) { EPID_CUDA(cudaStreamSynchronize(ctx->stream)); EPID_CUDA(cudaFree(ctx->scratch2)); ctx->scratch2 = nullptr; ctx->scratch2_bytes = 0; }
    cudaError_t e = cudaMalloc(&ctx->scratch2, bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return EPID_ERR_NOMEM; }
    ctx->scratch2_bytes = bytes;
    return EPID_OK;
}

static bool pf_fast_ok(const epid_ctx* ctx, const epid_pf_params* p, int H0, int W0) {
    const int H = H0 - 2 * p->crop_px, W = W0 - 2 * p->crop_px;
    return !ctx->pf_exact_only && p->filter_size == 0 && pf_front_supported(H, W, W0);
}


// Re-run of the m frames the fast pass deferred (w.sel_idx, ascending) on `stream`, in sub-batches whose work area lives in
// ctx->scratch2; result rows are scattered into the batch's device result arrays (after `after`, the event that marks the end of the
// batch's own pass, when the re-run is overlapped with it on another stream).  ctx->pf_fast_redo: first the certified-noise fast
// re-run (pf_run with PfRedoIn), then the exact-histogram pipeline for whatever that deferred again; otherwise exact for all.
static int pf_redo_deferred(epid_ctx* ctx, cudaStream_t stream, const uint16_t* d_frames, int m, int H0, int W0, const epid_pf_params* p,
                            int meas_cap, PfWork& w, uint16_t** pools, cudaEvent_t after = nullptr) {
    const int H = H0 - 2 * p->crop_px, W = W0 - 2 * p->crop_px;
    const int Wp = (W + 7) / 8 * 8;
    const int chunk = m < PF_REDO_CHUNK ? m : PF_REDO_CHUNK;
    const bool fast_redo = ctx->pf_fast_redo && pf_fast_ok(ctx, p, H0, W0);
    PfWork rw;
    carve(rw, nullptr, chunk, H, W, meas_cap);
    const size_t work_bytes = align_up(rw.total, 256);
    const size_t pool_bytes = fast_redo ? align_up(sizeof(uint16_t) * (size_t)chunk * H * Wp + 512, 256) : 0;
    int rc = ensure_scratch2(ctx, work_bytes + pool_bytes);
    if (rc != EPID_OK) return rc;
    carve(rw, (char*)ctx->scratch2, chunk, H, W, meas_cap);
    PfRedoIn rin;
    rin.raw_fr = w.fr;
    rin.pool = (uint16_t*)((char*)ctx->scratch2 + work_bytes);
    bool waited = after == nullptr;
    for (int c0 = 0; c0 < m; c0 += chunk) {
        const int cn = m - c0 < chunk ? m - c0 : chunk;
        int left = fast_redo ? 0 : -1;      // -1: exact pipeline for the whole sub-batch
        if (fast_redo) {
            rc = pf_run(ctx, stream, d_frames, cn, H0, W0, p, meas_cap, rw, pools, nullptr, true, w.sel_idx + c0, nullptr, ctx->h_flags + 1, &rin);
            if (rc != EPID_OK) return rc;
            k_pf_compose_sel<<<1, 64, 0, stream>>>(rw.sel_idx, rw.counters, w.sel_idx + c0);
            ctx->launches++;
            EPID_CUDA(cudaStreamSynchronize(stream));      // the host needs the number of frames that were deferred again
            left = ctx->h_flags[1];
        } else {
            rc = pf_run(ctx, stream, d_frames, cn, H0, W0, p, meas_cap, rw, pools, nullptr, false, w.sel_idx + c0);
            if (rc != EPID_OK) return rc;
            ctx->pf_exact_frames += cn;
        }
        if (!waited) { EPID_CUDA(cudaStreamWaitEvent(stream, after, 0)); waited = true; }
        k_pf_scatter_results<<<cn, 256, 0, stream>>>(w.sel_idx + c0, cn, rw.summ, rw.meas, w.summ, w.meas, meas_cap);
        ctx->launches++;
        if (left > 0) {
            rc = pf_run(ctx, stream, d_frames, left, H0, W0, p, meas_cap, rw, pools, nullptr, false, rw.sel_idx);
            if (rc != EPID_OK) return rc;
            k_pf_scatter_results<<<left, 256, 0, stream>>>(rw.sel_idx, left, rw.summ, rw.meas, w.summ, w.meas, meas_cap);
            ctx->launches++;
            ctx->pf_exact_frames += left;
        }
    }
    ctx->pf_redone_frames += m;
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

// One device-resident batch: the fast pass on `stream`; the host waits for the front end only (ctx->ev_front), reads the number of
// deferred frames from the mapped flag and, if there are any, runs their re-run on ctx->redo_stream while the window / finalize
// stages of the batch are still running; `stream` continues after the re-run's rows have been scattered.
static int pf_run_overlapped(epid_ctx* ctx, cudaStream_t stream, const uint16_t* d_frames, int n, int H0, int W0, const epid_pf_params* p,
                             int meas_cap, PfWork& w, uint16_t** pools, PfTimers* tm, int* n_deferred) {
    int rc = pf_run(ctx, stream, d_frames, n, H0, W0, p, meas_cap, w, pools, tm, true, nullptr, ctx->ev_front, ctx->h_flags);
    if (rc != EPID_OK) return rc;
    EPID_CUDA(cudaEventSynchronize(ctx->ev_front));
    const int m = ctx->h_flags[0];
    if (n_deferred) *n_deferred = m;
    if (m > 0) {
        EPID_CUDA(cudaEventRecord(ctx->ev_main_done, stream));
        rc = pf_redo_deferred(ctx, ctx->redo_stream, d_frames, m, H0, W0, p, meas_cap, w, pools, ctx->ev_main_done);
        if (rc != EPID_OK) { cudaStreamSynchronize(ctx->redo_stream); return rc; }
        EPID_CUDA(cudaEventRecord(ctx->ev_redo_done, ctx->redo_stream));
        EPID_CUDA(cudaStreamWaitEvent(stream, ctx->ev_redo_done, 0));
    }
    return EPID_OK;
}

static int ensure_pinned_ring(epid_ctx* ctx, size_t bytes) {
    if (ctx->pinned_ring_bytes >= bytes) return EPID_OK;
    if (ctx->pinned_ring) { EPID_CUDA(cudaStreamSynchronize(ctx->copy_stream[0])); EPID_CUDA(cudaFreeHost(ctx->pinned_ring)); ctx->pinned_ring = nullptr; ctx->pinned_ring_bytes = 0; }
    cudaError_t e = cudaMallocHost(&ctx->pinned_ring, bytes);
    if (e != cudaSuccess) { set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e)); return EPID_ERR_NOMEM; }
    ctx->pinned_ring_bytes = bytes;
    return EPID_OK;
}

static int pf_validate(const epid_pf_params* p, int H0, int W0, int meas_cap) {
    EPID_REQUIRE(p, EPID_ERR_INVALID, "params is NULL");
    EPID_REQUIRE(p->dpmm > 0, EPID_ERR_INVALID, "dpmm must be positive");
    EPID_REQUIRE(p->crop_px >= 0, EPID_ERR_INVALID, "Pixels to remove must be a positive number");
    EPID_REQUIRE(H0 - 2 * p->crop_px > 0 && W0 - 2 * p->crop_px > 0, EPID_ERR_INVALID,
                 "Too many pixels removed; array is empty. Pass a smaller crop value.");
    EPID_REQUIRE(p->n_leaves > 0 && p->n_leaves <= PF_L, EPID_ERR_INVALID, "n_leaves %d outside 1..%d", p->n_leaves, PF_L);
    EPID_REQUIRE(meas_cap > 0 && meas_cap <= 8192, EPID_ERR_INVALID, "meas_cap %d outside 1..8192", meas_cap);
    EPID_REQUIRE(!(p->action_tolerance >= 0 && p->tolerance < p->action_tolerance), EPID_ERR_INVALID,
                 "Tolerance cannot be lower than the action tolerance");
    EPID_REQUIRE(p->filter_size >= 0 && p->filter_size <= 31, EPID_ERR_UNSUPPORTED, "median filter size %d outside 0..31", p->filter_size);
    return EPID_OK;
}

}  // namespace epid

using namespace epid;

namespace {

}  // namespace
namespace epid { void staging_copy(void* dst, const void* src, size_t bytes); }   // hostcopy.cpp: non-temporal stores
namespace {

// Persistent host threads that copy a pageable chunk into the page-locked staging ring in parallel slices: one thread moves
// ~10 GB/s, the PCIe link takes ~54 GB/s, so a pageable source needs several copy streams to keep the link busy.
class CopyPool {
public:
    static CopyPool& get() {
        static CopyPool p;
        return p;
    }
    void copy(void* dst, const void* src, size_t bytes) {
        const int T = (int)workers_.size();
        if (T == 0 || bytes < (8u << 20)) { staging_copy(dst, src, bytes); return; }
        std::unique_lock<std::mutex> lk(m_);
        dst_ = (char*)dst; src_ = (const char*)src; bytes_ = bytes;
        pending_ = T;
        gen_++;
        cv_.notify_all();
        done_.wait(lk, [&] { return pending_ == 0; });
    }
    int threads() const { return (int)workers_.size(); }

private:
    CopyPool() {
        // measured on the B200 hosts (16 CPUs granted, profiles/r2l_summary.md): 8 / 12 / 14 threads with non-temporal stores reach
        // 72 / 80 / 81 % of the page-locked end-to-end rate; never more threads than the cgroup's CPU quota leaves for the caller
        int T = 12;
        const int hw = (int)std::thread::hardware_concurrency();
        if (hw > 0 && T > hw) T = hw;
        if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
            long long quota = 0, period = 0;
            if (fscanf(f, "%lld %lld", &quota, &period) == 2 && quota > 0 && period > 0) {
                // ranks of one node (torchrun: LOCAL_WORLD_SIZE) share the quota
                int lw = 1;
                if (const char* e = getenv("LOCAL_WORLD_SIZE")) lw = atoi(e) > 0 ? atoi(e) : 1;
                const int q = ((int)(quota / period) - 2) / lw;
                if (T > q) T = q < 2 ? 2 : q;
            }
            fclose(f);
        }
        if (const char* e = getenv("EPID_COPY_THREADS")) { T = atoi(e); if (hw > 0 && T > hw) T = hw; }
        if (T < 0) T = 0;
        for (int i = 0; i < T; i++) workers_.emplace_back([this, i, T] { run(i, T); });
    }
    ~CopyPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; gen_++; }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
    void run(int i, int T) {
        // The caller may have pinned itself to the GPU's NUMA node (parallel.bind_host_to_gpu) for its page-locked buffers; the copy
        // threads inherit that mask.  EPID_COPY_UNBIND=1 lets them run on every CPU the cgroup allows.
        if (const char* e = getenv("EPID_COPY_UNBIND")) {
            if (atoi(e)) {
                cpu_set_t all;
                CPU_ZERO(&all);
                for (int c = 0; c < CPU_SETSIZE; c++) CPU_SET(c, &all);
                pthread_setaffinity_np(pthread_self(), sizeof(all), &all);
            }
        }
        unsigned long long seen = 0;
        for (;;) {
            char* d; const char* s; size_t b;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
                d = dst_; s = src_; b = bytes_;
            }
            const size_t per = ((b + T - 1) / T + 4095) & ~(size_t)4095;
            const size_t o = per * (size_t)i;
            if (o < b) staging_copy(d + o, s + o, b - o < per ? b - o : per);
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0) done_.notify_one();
            }
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    char* dst_ = nullptr;
    const char* src_ = nullptr;
    size_t bytes_ = 0;
    int pending_ = 0;
    unsigned long long gen_ = 0;
    bool stop_ = false;
};

struct PfResultCopy {   // async D2H of one chunk's results + the counters ([2] = number of deferred frames)
    static int enqueue(cudaStream_t st, const PfWork& w, int cnt, int meas_cap, epid_pf_summary* summ, epid_pf_meas* meas, int* counters2) {
        EPID_CUDA(cudaMemcpyAsync(summ, w.summ, sizeof(epid_pf_summary) * cnt, cudaMemcpyDeviceToHost, st));
        EPID_CUDA(cudaMemcpyAsync(meas, w.meas, sizeof(epid_pf_meas) * (size_t)cnt * meas_cap, cudaMemcpyDeviceToHost, st));
        EPID_CUDA(cudaMemcpyAsync(counters2, w.counters, sizeof(int) * 3, cudaMemcpyDeviceToHost, st));
        return EPID_OK;
    }
};

}  // namespace

extern "C" {

int32_t epid_pf_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, epid_pf_summary* summary,
                        epid_pf_meas* meas, int32_t meas_cap) {
    EPID_REQUIRE(ctx && frames && summary && meas, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(frames->dtype == EPID_U16, EPID_ERR_UNSUPPORTED, "picket fence frames must be uint16");
    int rc = pf_validate(p, frames->h, frames->w, meas_cap);
    if (rc != EPID_OK) return rc;
    EPID_CUDA(cudaSetDevice(ctx->device));
    const int n = frames->n, H = frames->h - 2 * p->crop_px, W = frames->w - 2 * p->crop_px;
    PfWork w;
    carve(w, nullptr, n, H, W, meas_cap);
    rc = ensure_scratch(ctx, w.total);
    if (rc != EPID_OK) return rc;
    carve(w, (char*)ctx->scratch, n, H, W, meas_cap);
    uint16_t* pools[3] = {nullptr, nullptr, nullptr};
    const bool fast = pf_fast_ok(ctx, p, frames->h, frames->w);
    // the re-run of deferred frames (if any) overlaps the window stages of the batch on ctx->redo_stream; the exact pipeline defers none
    int m = 0;
    const uint16_t* d_frames = (const uint16_t*)frames->dptr;
    rc = fast ? pf_run_overlapped(ctx, ctx->stream, d_frames, n, frames->h, frames->w, p, meas_cap, w, pools, nullptr, &m)
              : pf_run(ctx, ctx->stream, d_frames, n, frames->h, frames->w, p, meas_cap, w, pools, nullptr, false);
    if (m > 0) ctx->pf_fallbacks++;
    int cnt3[3] = {0, 0, 0};
    if (rc == EPID_OK) rc = PfResultCopy::enqueue(ctx->stream, w, n, meas_cap, summary, meas, cnt3);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc == EPID_OK && e != cudaSuccess) { set_error("PF pipeline failed: %s", cudaGetErrorString(e)); rc = EPID_ERR_CUDA; }
    for (int k = 0; k < 3; k++) if (pools[k]) cudaFree(pools[k]);
    return rc;
}

static int32_t pf_bench_impl(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, int32_t iters, float* total_ms,
                             float* stats_kernel_ms, int64_t* launches, float* stage_ms, int32_t nstages, int64_t* redone) {
    EPID_REQUIRE(ctx && frames && p && iters > 0, EPID_ERR_INVALID, "bad argument");
    EPID_REQUIRE(!stage_ms || nstages >= PF_NSTAGES, EPID_ERR_INVALID, "stage_ms needs %d entries", PF_NSTAGES);
    EPID_REQUIRE(frames->dtype == EPID_U16, EPID_ERR_UNSUPPORTED, "picket fence frames must be uint16");
    const int meas_cap = 1024;
    int rc = pf_validate(p, frames->h, frames->w, meas_cap);
    if (rc != EPID_OK) return rc;
    EPID_CUDA(cudaSetDevice(ctx->device));
    const int n = frames->n, H = frames->h - 2 * p->crop_px, W = frames->w - 2 * p->crop_px;
    PfWork w;
    carve(w, nullptr, n, H, W, meas_cap);
    rc = ensure_scratch(ctx, w.total);
    if (rc != EPID_OK) return rc;
    carve(w, (char*)ctx->scratch, n, H, W, meas_cap);
    uint16_t* pools[3] = {nullptr, nullptr, nullptr};
    const bool fast = pf_fast_ok(ctx, p, frames->h, frames->w);
    const uint16_t* d_frames = (const uint16_t*)frames->dptr;
    cudaEvent_t t0, t1;
    EPID_CUDA(cudaEventCreate(&t0));
    EPID_CUDA(cudaEventCreate(&t1));
    // pass 0: back-to-back passes, no host round trip (what an ordinary batch costs).  If that left deferred frames, pass 1 times
    // the real control flow of epid_pf_analyze: after the front end of every pass the host reads the deferred count and runs the
    // per-frame re-run on ctx->redo_stream, overlapped with the batch's window stages.
    for (int mode = 0; mode < 2; mode++) {
        PfTimers tm;
        tm.on = true;
        tm.stages = stage_ms != nullptr;
        const int64_t l0 = ctx->launches, rd0 = ctx->pf_redone_frames;
        int cnt3[3] = {0, 0, 0};
        EPID_CUDA(cudaStreamSynchronize(ctx->stream));
        EPID_CUDA(cudaEventRecord(t0, ctx->stream));
        for (int it = 0; it < iters && rc == EPID_OK; it++)
            rc = mode == 0 ? pf_run(ctx, ctx->stream, d_frames, n, frames->h, frames->w, p, meas_cap, w, pools, &tm, fast)
                           : pf_run_overlapped(ctx, ctx->stream, d_frames, n, frames->h, frames->w, p, meas_cap, w, pools, &tm, nullptr);
        cudaEventRecord(t1, ctx->stream);
        if (mode == 0) cudaMemcpyAsync(cnt3, w.counters, sizeof(cnt3), cudaMemcpyDeviceToHost, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        if (total_ms) *total_ms = ms;
        if (stats_kernel_ms) *stats_kernel_ms = tm.total_ms();
        if (launches) *launches = ctx->launches - l0;
        if (redone) *redone = ctx->pf_redone_frames - rd0;
        if (stage_ms) tm.stage_ms(stage_ms, PF_NSTAGES);
        tm.destroy();
        if (rc != EPID_OK || !fast || mode == 1 || cnt3[2] == 0) break;
        ctx->pf_fallbacks++;
    }
    cudaEventDestroy(t0); cudaEventDestroy(t1);
    for (int k = 0; k < 3; k++) if (pools[k]) cudaFree(pools[k]);
    return rc;
}

int32_t epid_pf_bench(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, int32_t iters, float* total_ms,
                      float* stats_kernel_ms, int64_t* launches) {
    return pf_bench_impl(ctx, frames, p, iters, total_ms, stats_kernel_ms, launches, nullptr, 0, nullptr);
}

int32_t epid_pf_bench_timed(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, int32_t iters, float* total_ms, float* stage_ms,
                            int32_t nstages, int64_t* launches, int64_t* redone_frames) {
    return pf_bench_impl(ctx, frames, p, iters, total_ms, nullptr, launches, stage_ms, nstages, redone_frames);
}

int32_t epid_pf_analyze_host(epid_ctx* ctx, const uint16_t* frames, int32_t n, int32_t h, int32_t w_, const epid_pf_params* p,
                             epid_pf_summary* summary, epid_pf_meas* meas, int32_t meas_cap) {
    EPID_REQUIRE(ctx && frames && summary && meas, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(n > 0 && h > 0 && w_ > 0, EPID_ERR_INVALID, "empty batch");
    int rc = pf_validate(p, h, w_, meas_cap);
    if (rc != EPID_OK) return rc;
    EPID_CUDA(cudaSetDevice(ctx->device));
    const int H = h - 2 * p->crop_px, W = w_ - 2 * p->crop_px;
    const size_t fbytes = sizeof(uint16_t) * (size_t)h * w_;
    // chunk: ~128 MB of frames, double buffered: small enough that the work left after the last H2D copy (one chunk of
    // compute + its result copy) is short, large enough that the persistent kernels still have several work items per SM
    int chunk = (int)((128u << 20) / fbytes);
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    const int nchunks = (n + chunk - 1) / chunk;
    PfWork wk;
    carve(wk, nullptr, chunk, H, W, meas_cap);
    const size_t work_bytes = align_up(wk.total, 256);
    const size_t buf_bytes = align_up(fbytes * chunk, 256);
    rc = ensure_scratch(ctx, 2 * work_bytes + 2 * buf_bytes + 512);   // slack: 16-byte vector / TMA reads may run a few bytes past the last frame
    if (rc != EPID_OK) return rc;
    // pinned staging for the results of two chunks in flight
    const size_t res_bytes = align_up(sizeof(epid_pf_summary) * chunk, 256) + align_up(sizeof(epid_pf_meas) * (size_t)chunk * meas_cap, 256) + 256;
    rc = ensure_pinned(ctx, 2 * res_bytes);
    if (rc != EPID_OK) return rc;
    char* base = (char*)ctx->scratch;
    PfWork works[2];
    uint16_t* bufs[2];
    epid_pf_summary* h_summ[2];
    epid_pf_meas* h_meas[2];
    int* h_cnt[2];
    for (int s = 0; s < 2; s++) {
        carve(works[s], base + s * work_bytes, chunk, H, W, meas_cap);
        bufs[s] = (uint16_t*)(base + 2 * work_bytes + s * buf_bytes);
        char* r = (char*)ctx->pinned + s * res_bytes;
        h_summ[s] = (epid_pf_summary*)r;
        h_meas[s] = (epid_pf_meas*)(r + align_up(sizeof(epid_pf_summary) * chunk, 256));
        h_cnt[s] = (int*)(r + res_bytes - 256);
    }
    // results go straight into the caller's buffers when those are page-locked (epid_host_alloc / cudaHostRegister): no staging copy
    auto pinned_host = [](const void* ptr) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
        return a.type == cudaMemoryTypeHost;
    };
    const bool direct = pinned_host(summary) && pinned_host(meas);
    // pageable source frames: staged through a page-locked ring, filled by parallel host copies that overlap the previous chunk's DMA
    const bool src_pinned = pinned_host(frames);
    char* ring[2] = {nullptr, nullptr};
    if (!src_pinned) {
        rc = ensure_pinned_ring(ctx, 2 * buf_bytes);
        if (rc != EPID_OK) return rc;
        ring[0] = (char*)ctx->pinned_ring;
        ring[1] = ring[0] + buf_bytes;
    }
    cudaEvent_t copied[2], computed[2];
    for (int s = 0; s < 2; s++) { EPID_CUDA(cudaEventCreateWithFlags(&copied[s], cudaEventDisableTiming)); EPID_CUDA(cudaEventCreateWithFlags(&computed[s], cudaEventDisableTiming)); }
    uint16_t* pools[3] = {nullptr, nullptr, nullptr};
    const bool fast = pf_fast_ok(ctx, p, h, w_);
    auto count_of = [&](int ci) { return (ci == nchunks - 1) ? n - ci * chunk : chunk; };
    auto enqueue_copy = [&](int ci) -> int {
        const int s = ci & 1;
        // the buffer is free once the compute that last used it has finished (finish(ci - 2) already waited for it)
        const uint16_t* src = frames + (size_t)ci * chunk * h * w_;
        if (!src_pinned) {
            // ring slot s was last read by the DMA of chunk ci - 2: its `copied` event has been waited for by the compute stream
            // two iterations ago, but the HOST must see it finished before overwriting the slot
            if (ci >= 2) EPID_CUDA(cudaEventSynchronize(copied[s]));
            CopyPool::get().copy(ring[s], src, fbytes * count_of(ci));
            src = (const uint16_t*)ring[s];
        }
        EPID_CUDA(cudaMemcpyAsync(bufs[s], src, fbytes * count_of(ci), cudaMemcpyHostToDevice, ctx->copy_stream[0]));
        EPID_CUDA(cudaEventRecord(copied[s], ctx->copy_stream[0]));
        return EPID_OK;
    };
    auto enqueue_run = [&](int ci, bool use_fast) -> int {
        const int s = ci & 1, cnt = count_of(ci);
        int r = pf_run(ctx, ctx->stream, bufs[s], cnt, h, w_, p, meas_cap, works[s], pools, nullptr, use_fast);
        if (r != EPID_OK) return r;
        r = PfResultCopy::enqueue(ctx->stream, works[s], cnt, meas_cap, direct ? summary + (size_t)ci * chunk : h_summ[s],
                                  direct ? meas + (size_t)ci * chunk * meas_cap : h_meas[s], h_cnt[s]);
        if (r != EPID_OK) return r;
        EPID_CUDA(cudaEventRecord(computed[s], ctx->stream));
        return EPID_OK;
    };
    auto finish = [&](int ci) -> int {   // wait for chunk ci, re-run its deferred frames exactly, hand the results to the caller
        const int s = ci & 1, cnt = count_of(ci);
        EPID_CUDA(cudaEventSynchronize(computed[s]));
        if (fast && h_cnt[s][2] > 0) {     // re-run exactly the frames the front end deferred, then fetch the chunk's rows again
            ctx->pf_fallbacks++;
            // on the re-run stream: the chunk's own pass has finished, the next chunk's pass keeps ctx->stream busy meanwhile
            cudaStream_t rs = ctx->redo_stream;
            int r = pf_redo_deferred(ctx, rs, bufs[s], h_cnt[s][2], h, w_, p, meas_cap, works[s], pools);
            if (r != EPID_OK) return r;
            r = PfResultCopy::enqueue(rs, works[s], cnt, meas_cap, direct ? summary + (size_t)ci * chunk : h_summ[s],
                                      direct ? meas + (size_t)ci * chunk * meas_cap : h_meas[s], h_cnt[s] + 4);
            if (r != EPID_OK) return r;
            EPID_CUDA(cudaEventRecord(computed[s], rs));
            EPID_CUDA(cudaEventSynchronize(computed[s]));
        }
        if (!direct) {
            memcpy(summary + (size_t)ci * chunk, h_summ[s], sizeof(epid_pf_summary) * cnt);
            memcpy(meas + (size_t)ci * chunk * meas_cap, h_meas[s], sizeof(epid_pf_meas) * (size_t)cnt * meas_cap);
        }
        return EPID_OK;
    };
    rc = enqueue_copy(0);
    for (int ci = 0; ci < nchunks && rc == EPID_OK; ci++) {
        const int s = ci & 1;
        EPID_CUDA(cudaStreamWaitEvent(ctx->stream, copied[s], 0));
        rc = enqueue_run(ci, fast);
        if (rc != EPID_OK) break;
        if (ci >= 1) { rc = finish(ci - 1); if (rc != EPID_OK) break; }
        if (ci + 1 < nchunks) rc = enqueue_copy(ci + 1);
    }
    if (rc == EPID_OK) rc = finish(nchunks - 1);
    cudaStreamSynchronize(ctx->copy_stream[0]);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc == EPID_OK && e != cudaSuccess) { set_error("PF pipeline failed: %s", cudaGetErrorString(e)); rc = EPID_ERR_CUDA; }
    for (int s = 0; s < 2; s++) { cudaEventDestroy(copied[s]); cudaEventDestroy(computed[s]); }
    for (int k = 0; k < 3; k++) if (pools[k]) cudaFree(pools[k]);
    return rc;
}

}  // extern "C"
