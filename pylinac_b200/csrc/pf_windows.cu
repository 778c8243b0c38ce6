// Fast per-(leaf, picket) window kernel of the PicketFence pipeline.
//
// Reference semantics: PicketFence._get_mlc_window / _is_mlc_peak_in_window (picketfence.py:847-886) and
// MLCValue.get_peak_positions (picketfence.py:1605-1628) -> FWXMProfilePhysical.field_edge_idx (core/profile.py:602-611).
//
// One warp per window, 16 windows in flight per CTA (2 CTAs per SM), the windows of a frame spread over gridDim.x CTAs.
//   1. stage the window as exact integers g (ground / invert folded in) into shared memory, canonical layout
//      px[i * S + jj]: i across the leaf (the axis np.median collapses), jj along leaf travel.  Up-Down frames are staged
//      with 128-bit loads on the frame's aligned 8-pixel grid, all loads of a window in flight at once (jj = column - cs,
//      the window starts at jj = off; pixels outside the window are written as 0); the row stride S is even with S/2
//      odd, so "lane = row" accesses are bank-conflict free and a 32-bit load yields two adjacent travel samples;
//   2. validity: lanes own rows -> sum / sum of squares along travel with no shuffles (exact integer variance);
//   3. np.median(window, axis): lanes own PAIRS of travel samples held packed u16x2 in registers and sorted by a fully
//      unrolled Batcher merge-exchange network on VIMNMX.U16x2; the network is instantiated for the exact row count, so
//      every comparator that does not feed the two middle outputs is dead code;
//   4. the 1-D profile (<= 256 samples) is normalised in fp64 and searched for its most prominent peak, FWHM edges by
//      scipy's peak_widths interpolation (warp-parallel search for the crossing, same arithmetic as the reference).
// The CTA's shared memory is split into per-warp slots sized for the frame's largest window (all 16 warps for ordinary
// windows, fewer for very wide ones).  Windows that do not fit at all (nc > 256, nr > 64) are marked valid = -1 and picked up by the
// generic kernel (k_pf_windows in pf.cu) launched right after in "todo" mode.
#include "pf_common.cuh"
#include "pf_win_common.cuh"

namespace epid {

constexpr int W2_WARPS = 16;
constexpr int W2_POOL = 100 * 1024;   // shared memory per CTA, split into per-warp slots sized for the frame's largest window
constexpr int W2_MAXNC = 256;    // travel samples per window on the fast path
constexpr int W2_GRID_X = 12;    // CTAs per frame: a warp takes ~3 windows and prefetches the next one while it analyses the current one (sweep 4..24: flat, 12 best)

// Row statistics of _is_mlc_peak_in_window: max(std) and median(std) over the nr rows, std along travel as
// sqrt(nc*S2 - S1^2) / (nc * D) with an exact integer numerator.  NSL = row slots per lane (1: nr <= 32, 2: nr <= 64).
template <int NSL>
__device__ __forceinline__ void row_std_stats(const uint16_t* __restrict__ px, int S, int nr, int nc, double Dd, int lane,
                                              double& sd_max, double& sd_med, int t0, int t1) {
    double sd[NSL];
#pragma unroll
    for (int sl = 0; sl < NSL; sl++) {
        sd[sl] = -1.0;
        const int i = sl * 32 + lane;
        if (i < nr) {
            const uint32_t* __restrict__ rowp = reinterpret_cast<const uint32_t*>(px + i * S);
            uint32_t s1 = 0;
            unsigned long long s2 = 0;
#pragma unroll 4
            for (int t = t0; t < t1; t++) {  // the words that hold window samples; samples outside the window were staged as zero
                const uint32_t w = rowp[t];
                const uint32_t lo = w & 0xffffu, hi = w >> 16;
                s1 = __dp2a_lo(w, 0x0101u, s1);
                s2 = mad_wide_u32(lo, lo, s2);
                s2 = mad_wide_u32(hi, hi, s2);
            }
            const double num = (double)((unsigned long long)nc * s2 - (unsigned long long)s1 * s1);
            sd[sl] = sqrt(num) / ((double)nc * Dd);
        }
    }
    double m = sd[0];
#pragma unroll
    for (int sl = 1; sl < NSL; sl++) m = fmax(m, sd[sl]);
    sd_max = warp_max(m);
    const int k1 = (nr - 1) / 2, k2 = nr / 2;
    int rank[NSL];
#pragma unroll
    for (int sl = 0; sl < NSL; sl++) rank[sl] = 0;
    for (int t = 0; t < nr; t++) {
        double o;
        if (NSL == 1) o = __shfl_sync(0xffffffffu, sd[0], t);
        else o = __shfl_sync(0xffffffffu, (t >> 5) ? sd[NSL - 1] : sd[0], t & 31);
#pragma unroll
        for (int sl = 0; sl < NSL; sl++) {
            const int me = sl * 32 + lane;
            if (o < sd[sl] || (o == sd[sl] && t < me)) rank[sl]++;
        }
    }
    double ca = 0.0, cb = 0.0;
#pragma unroll
    for (int sl = 0; sl < NSL; sl++) {
        const int me = sl * 32 + lane;
        if (me < nr) {
            if (rank[sl] == k1) ca = sd[sl];
            if (rank[sl] == k2) cb = sd[sl];
        }
    }
    const double med_a = warp_sum(ca);   // exactly one lane holds each; the others contribute +0.0
    const double med_b = warp_sum(cb);
    sd_med = (nr & 1) ? med_a : (med_a + med_b) / 2.0;
}

__global__ void __launch_bounds__(W2_WARPS * 32, 2)
k_pf_windows_fast(const PfConst* __restrict__ cc, const FrameRef* __restrict__ frames, PfFrame* fr, PfWin* __restrict__ wins) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ int s_geo[4];     // status, slot bytes, bytes of the staging part, active warps
    const int fi = blockIdx.y;
    const PfConst& c = *cc;
    PfFrame& f = fr[fi];
    if (f.win2) return;          // the two-kernel window path owns this frame (pf_windows2.cu)
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int H = c.H, W = c.W;
    const double dpmm = c.p.dpmm;
    if (wid == 0) {
        // slot size from the frame's largest possible window (other CTAs may change f.status meanwhile: read it once)
        const int st = f.status;
        double lw = 0.0;
        for (int i = lane; i < f.n_inview; i += 32) lw = fmax(lw, c.p.leaf_width_mm[f.inview[i]] * dpmm);
        lw = warp_max(lw);
        if (lane == 0) {
            const double sp = f.spacing;
            const int nc_max = (sp == sp && sp < 4096.0) ? (int)sp + 2 : 4096;
            const int nr_max = (int)lw + 2;
            const int s_max = ((nc_max + 14) / 8 + 1) * 8 + 2;
            int stage_b = max(nr_max * s_max * 2, nc_max * 8);
            stage_b = (stage_b + 15) & ~15;
            const int slot = stage_b + ((nc_max * 4 + 15) & ~15);
            s_geo[0] = f.win2 ? -1 : st;     // the two-kernel window path owns this frame
            s_geo[1] = slot;
            s_geo[2] = stage_b;
            s_geo[3] = nc_max > W2_MAXNC + 2 ? 0 : min(W2_WARPS, W2_POOL / slot);
        }
    }
    __syncthreads();
    if (s_geo[0] != EPID_PF_OK) return;
    const int np = f.n_pickets;
    const int total = f.n_inview * np;
    const int active = s_geo[3];
    if (active == 0) {           // windows too large for the fast path: all of them go to the generic kernel
        for (int widx = blockIdx.x * blockDim.x + threadIdx.x; widx < total; widx += gridDim.x * blockDim.x) {
            const int li = widx / np, pk = widx - li * np;
            wins[((size_t)fi * PF_L + li) * PF_P + pk].valid = -1;
        }
        if (threadIdx.x == 0) f.todo = 1;
        return;
    }
    if (wid >= active) return;
    const int cap_px = s_geo[2] >> 1;
    uint16_t* px = reinterpret_cast<uint16_t*>(smraw + (size_t)wid * s_geo[1]);
    uint32_t* m2 = reinterpret_cast<uint32_t*>(smraw + (size_t)wid * s_geo[1] + s_geo[2]);
    double* xs = reinterpret_cast<double*>(px);
    const int orient = f.orientation;
    const FrameRef frf = frames[fi];
    const int inv = f.inv;
    const uint32_t mn = f.mn, mx = f.mx;
    const uint32_t MN2 = mn * 0x00010001u, MX2 = mx * 0x00010001u;
    const double Dd = (double)f.D;
    const double spacing = f.spacing;
    const int sag = c.p.sag_px;
    const bool aligned = (frf.pitch & 7) == 0;
    const int mis = (int)((reinterpret_cast<uintptr_t>(frf.origin) >> 1) & 7);

    for (int widx = blockIdx.x * active + wid; widx < total; widx += gridDim.x * active) {
        const int li = widx / np, pk = widx - li * np;
        const int leaf = f.inview[li];
        const double lw_px = c.p.leaf_width_mm[leaf] * dpmm;
        const double lc_px = c.p.leaf_center_mm[leaf] * dpmm + (orient == 0 ? (double)H / 2.0 : (double)W / 2.0);
        PfWin& out = wins[((size_t)fi * PF_L + li) * PF_P + pk];
        const double pidx = (double)f.picket_idx[pk];
        // _get_mlc_window (picketfence.py:859-886): python int() truncates toward zero
        const int a0 = max((int)(pidx - spacing / 2.0), 0);                                   // along travel
        const int a1 = min((int)(pidx + spacing / 2.0), orient == 0 ? W : H);
        const int b0 = max((int)(lc_px - lw_px / 2.0), 0);                                    // across the leaf
        const int b1 = min((int)(lc_px + lw_px / 2.0), orient == 0 ? H : W);
        const int nc = a1 - a0, nr = b1 - b0;
        if (nc <= 0 || nr <= 0) {           // empty slice: np.max raises ValueError in the reference
            if (lane == 0) { out.valid = 0; out.l = 0; out.r = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            continue;
        }
        // staged geometry: sample j of the window lives at jj = j + off of each staged row
        const bool vec = orient == 0 && aligned;
        int S, off, nvec = 0, cs = a0;
        if (vec) {
            cs = a0 - ((a0 + mis) & 7);                       // aligned grid column (view coordinates, may be < 0)
            const int ce = a1 + ((8 - ((a1 + mis) & 7)) & 7);
            nvec = (ce - cs) >> 3;
            off = a0 - cs;
            S = nvec * 8 + 2;
        } else {
            off = 0;
            S = (nc + 1) & ~1;
            if (((S >> 1) & 1) == 0) S += 2;
        }
        if (nc > W2_MAXNC || nr > 64 || nr * S > cap_px || nc * 4 > s_geo[1] - s_geo[2]) {
            if (lane == 0) { out.valid = -1; f.todo = 1; }   // generic kernel
            continue;
        }
        __syncwarp();
        // ---- 1. stage (np.roll(sag) folded into the source index)
        uint32_t gmax = 0;
        if (vec) {
            const int nv_tot = nr * nvec;
            const float inv_nvec = 1.0f / (float)nvec;
            const uint32_t fill = inv ? MX2 : MN2;
            uint32_t gmax2 = 0;
            constexpr int U = 4;
            for (int base = 0; base < nv_tot; base += 32 * U) {
                uint4 q[U];
                int ii[U], jv[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int idx = base + u * 32 + lane;
                    ii[u] = (int)(((float)idx + 0.5f) * inv_nvec);
                    jv[u] = idx - ii[u] * nvec;
                    q[u] = make_uint4(fill, fill, fill, fill);
                    if (idx < nv_tot) {
                        int row = b0 + ii[u] - sag;
                        if (sag) { row %= H; if (row < 0) row += H; }
                        q[u] = ldg_stream16(frf.origin + (size_t)row * frf.pitch + cs + jv[u] * 8);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int idx = base + u * 32 + lane;
                    if (idx >= nv_tot) continue;
                    uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
                    const int col0 = cs + jv[u] * 8;
                    if (col0 < a0 || col0 + 8 > a1) {       // first / last vector: pixels outside the window -> g = 0
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const int c0 = col0 + 2 * k;
                            const uint32_t keep = ((c0 >= a0 && c0 < a1) ? 0xffffu : 0u) | ((c0 + 1 >= a0 && c0 + 1 < a1) ? 0xffff0000u : 0u);
                            w[k] = (w[k] & keep) | (fill & ~keep);
                        }
                    }
                    uint32_t* dst = reinterpret_cast<uint32_t*>(px + ii[u] * S + jv[u] * 8);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t g = inv ? MX2 - w[k] : w[k] - MN2;     // no borrow between halves: mn <= v <= mx
                        gmax2 = __vmaxu2(gmax2, g);
                        dst[k] = g;
                    }
                    if (jv[u] == nvec - 1) dst[4] = 0;      // pad word
                }
            }
            gmax = max(gmax2 & 0xffffu, gmax2 >> 16);
        } else if (orient == 0) {
            for (int i = 0; i < nr; i++) {
                int row = b0 + i - sag;
                if (sag) { row %= H; if (row < 0) row += H; }
                const uint16_t* __restrict__ src = frf.origin + (size_t)row * frf.pitch + a0;
                for (int jj = lane; jj < S; jj += 32) {
                    uint32_t g = 0;
                    if (jj < nc) {
                        const uint32_t v = __ldg(src + jj);
                        g = inv ? mx - v : v - mn;
                        gmax = max(gmax, g);
                    }
                    px[i * S + jj] = (uint16_t)g;
                }
            }
        } else {
            // Left-Right: travel runs along image rows; lanes sweep the (travel, across) index space with 4 loads in flight
            const int tot = nc * nr;
            const float inv_nr = 1.0f / (float)nr;
            constexpr int U = 4;
            for (int base = 0; base < tot; base += 32 * U) {
                uint32_t v[U];
                int ii[U], jj[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int idx = base + u * 32 + lane;
                    jj[u] = (int)(((float)idx + 0.5f) * inv_nr);
                    ii[u] = idx - jj[u] * nr;
                    v[u] = 0;
                    if (idx < tot) {
                        int col = b0 + ii[u] - sag;
                        if (sag) { col %= W; if (col < 0) col += W; }
                        v[u] = __ldg(frf.origin + (size_t)(a0 + jj[u]) * frf.pitch + col);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int idx = base + u * 32 + lane;
                    if (idx >= tot) continue;
                    const uint32_t g = inv ? mx - v[u] : v[u] - mn;
                    gmax = max(gmax, g);
                    px[ii[u] * S + jj[u]] = (uint16_t)g;
                }
            }
            for (int i = lane; i < nr; i += 32)
                for (int jj = nc; jj < S; jj++) px[i * S + jj] = 0;
        }
        {
            // the warp's next window: pull its rows towards L2 / L1 now, so that its staging loads do not wait for HBM
            const int nwidx = widx + gridDim.x * active;
            if (nwidx < total && orient == 0) {
                const int nli = nwidx / np, npk = nwidx - nli * np;
                const int nleaf = f.inview[nli];
                const double nlw = c.p.leaf_width_mm[nleaf] * dpmm;
                const double nlc = c.p.leaf_center_mm[nleaf] * dpmm + (double)H / 2.0;
                const double npidx = (double)f.picket_idx[npk];
                const int na0 = max((int)(npidx - spacing / 2.0), 0), na1 = min((int)(npidx + spacing / 2.0), W);
                const int nb0 = max((int)(nlc - nlw / 2.0), 0), nb1 = min((int)(nlc + nlw / 2.0), H);
                for (int i = lane; i < nb1 - nb0; i += 32) {
                    int row = nb0 + i - sag;
                    if (sag) { row %= H; if (row < 0) row += H; }
                    const uint16_t* ptr = frf.origin + (size_t)row * frf.pitch + na0;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
                    if (na1 - na0 > 56) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr + 64));
                    if (na1 - na0 > 120) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr + 128));
                }
            }
        }
        gmax = warp_max(gmax);
        __syncwarp();
        // ---- 2. _is_mlc_peak_in_window (picketfence.py:847-857): lanes own rows
        double sd_max, sd_med;
        const int t0 = off >> 1, t1 = (off + nc + 1) >> 1;      // words that hold window samples
        if (nr <= 32) row_std_stats<1>(px, S, nr, nc, Dd, lane, sd_max, sd_med, t0, t1);
        else row_std_stats<2>(px, S, nr, nc, Dd, lane, sd_max, sd_med, t0, t1);
        const bool above = ((double)gmax / Dd) > c.p.height_threshold * f.picket_val[pk];
        const bool not_edge = sd_max < c.p.edge_threshold * sd_med;
        if (!(above && not_edge)) {
            if (lane == 0) { out.valid = 0; out.l = 0; out.r = 0; }
            continue;
        }
        // ---- 3. np.median(window, axis) -> 2 * median per travel sample (picketfence.py:1605-1609)
        uint32_t lmin = 0xffffffffu, lmax = 0;
        for (int t = t0 + lane; t < t1; t += 32) {
            const uint2 mm = pair_median_any(px, S, nr, t);
            const uint32_t m_lo = mm.x, m_hi = mm.y;
            const int j0 = 2 * t - off;
            if (j0 >= 0 && j0 < nc) { m2[j0] = m_lo; lmin = min(lmin, m_lo); lmax = max(lmax, m_lo); }
            if (j0 + 1 >= 0 && j0 + 1 < nc) { m2[j0 + 1] = m_hi; lmin = min(lmin, m_hi); lmax = max(lmax, m_hi); }
        }
        lmin = warp_min(lmin);
        lmax = warp_max(lmax);
        __syncwarp();
        if (lmax == lmin) {  // flat profile: the reference divides by zero and then finds no peak
            if (lane == 0) { out.valid = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            continue;
        }
        // ---- 4. FWXMProfilePhysical(ground=True, normalization=MAX) (core/profile.py:204-240); xs aliases px
        const double den = (double)(lmax - lmin);
        for (int j = lane; j < nc; j += 32) xs[j] = (double)(m2[j] - lmin) / den;
        __syncwarp();
        // find_peaks(values, fwxm_height=0.5, max_number=1) by prominence (core/profile.py:602-611, 2545-2623)
        double best_prom = -1.0;
        int best_idx = -1, best_lb = 0, best_rb = 0;
        if (nc <= 128) {
            // xs is a strictly monotone map of the integers m2, so local maxima, nearest higher samples and range minima
            // are found on the integers, warp-wide and without divergent walks.  Candidates are visited from the highest
            // down; a candidate of height h cannot have a prominence above h - min(profile), which ends the search after
            // a few candidates.  The winner is chosen on the fp64 prominences exactly like the sequential formulation.
            uint32_t mv[4], ck[4];
#pragma unroll
            for (int sl = 0; sl < 4; sl++) {
                const int i = lane + 32 * sl;
                mv[sl] = i < nc ? m2[i] : 0u;
                ck[sl] = 0;
                if (i >= 1 && i < nc - 1 && m2[i - 1] < mv[sl]) {
                    int ahead = i + 1;
                    while (ahead < nc - 1 && m2[ahead] == mv[sl]) ahead++;
                    if (m2[ahead] < mv[sl]) ck[sl] = (mv[sl] << 8) | (uint32_t)((i + ahead - 1) / 2);
                }
            }
            int best_int = -1;
            while (true) {
                const uint32_t key = __reduce_max_sync(0xffffffffu, max(max(ck[0], ck[1]), max(ck[2], ck[3])));
                if (key == 0) break;
                const uint32_t hp = key >> 8;
                const int p = (int)(key & 255u);
                if ((int)(hp - lmin) < best_int) break;
                uint32_t gt[4];
#pragma unroll
                for (int sl = 0; sl < 4; sl++) {
                    if (ck[sl] == key) ck[sl] = 0;
                    gt[sl] = __ballot_sync(0xffffffffu, mv[sl] > hp);
                }
                int L = -1, R = nc;       // nearest strictly higher sample on each side
#pragma unroll
                for (int sl = 0; sl < 4; sl++) {
                    const int lo = 32 * sl;
                    uint32_t m = gt[sl];
                    if (p <= lo) m = 0; else if (p < lo + 32) m &= (1u << (p - lo)) - 1u;
                    if (m) L = lo + 31 - __clz(m);
                }
#pragma unroll
                for (int sl = 3; sl >= 0; sl--) {
                    const int lo = 32 * sl;
                    uint32_t m = gt[sl];
                    if (p >= lo + 32) m = 0; else if (p >= lo) m &= ~((2u << (p - lo)) - 1u);
                    if (m) R = lo + __ffs(m) - 1;
                }
                uint32_t lmv = 0xffffffffu, rmv = 0xffffffffu;
#pragma unroll
                for (int sl = 0; sl < 4; sl++) {
                    const int j = lane + 32 * sl;
                    if (j > L && j <= p) lmv = min(lmv, mv[sl]);
                    if (j >= p && j < R && j < nc) rmv = min(rmv, mv[sl]);
                }
                lmv = __reduce_min_sync(0xffffffffu, lmv);
                rmv = __reduce_min_sync(0xffffffffu, rmv);
                // bases: the occurrence of each minimum that is closest to the peak
                int lb = p, rb = p;
#pragma unroll
                for (int sl = 0; sl < 4; sl++) {
                    const int j = lane + 32 * sl;
                    const uint32_t el = __ballot_sync(0xffffffffu, j > L && j <= p && mv[sl] == lmv);
                    if (el) lb = 32 * sl + 31 - __clz(el);
                }
#pragma unroll
                for (int sl = 3; sl >= 0; sl--) {
                    const int j = lane + 32 * sl;
                    const uint32_t er = __ballot_sync(0xffffffffu, j >= p && j < R && j < nc && mv[sl] == rmv);
                    if (er) rb = 32 * sl + __ffs(er) - 1;
                }
                const double prom = xs[p] - fmax(xs[lb], xs[rb]);
                if (prom > best_prom || (prom == best_prom && p > best_idx)) { best_prom = prom; best_idx = p; best_lb = lb; best_rb = rb; }
                best_int = max(best_int, (int)(hp - max(lmv, rmv)));
            }
        } else {
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
    #pragma unroll
            for (int o = 16; o > 0; o >>= 1) {   // warp arg-max by (prominence, index)
                const double op = __shfl_xor_sync(0xffffffffu, best_prom, o);
                const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
                const int olb = __shfl_xor_sync(0xffffffffu, best_lb, o);
                const int orb = __shfl_xor_sync(0xffffffffu, best_rb, o);
                if (op > best_prom || (op == best_prom && oi > best_idx)) { best_prom = op; best_idx = oi; best_lb = olb; best_rb = orb; }
            }
        }
        if (best_idx < 0) {
            if (lane == 0) { out.valid = 0; f.status = EPID_PF_WINDOW_NO_PEAK; }
            continue;
        }
        {
            // scipy _peak_widths: walk from the peak towards each base while the profile is above h; the crossing is
            // searched 32 samples at a time (ballot), the interpolation is the reference's
            const int p = best_idx;
            const double h = xs[p] - best_prom * 0.5;
            int kl = best_lb;
            for (int c0 = p; c0 > best_lb; c0 -= 32) {
                const int k = c0 - lane;
                const bool stop = k > best_lb && !(h < xs[k]);
                const unsigned b = __ballot_sync(0xffffffffu, stop);
                if (b) { kl = c0 - (__ffs(b) - 1); break; }
            }
            double l = (double)kl;
            if (xs[kl] < h) l += (h - xs[kl]) / (xs[kl + 1] - xs[kl]);
            int kr = best_rb;
            for (int c0 = p; c0 < best_rb; c0 += 32) {
                const int k = c0 + lane;
                const bool stop = k < best_rb && !(h < xs[k]);
                const unsigned b = __ballot_sync(0xffffffffu, stop);
                if (b) { kr = c0 + (__ffs(b) - 1); break; }
            }
            double r = (double)kr;
            if (xs[kr] < h) r -= (h - xs[kr]) / (xs[kr - 1] - xs[kr]);
            if (lane == 0) {
                out.valid = 1;
                out.l = l;
                out.r = r;
            }
        }
    }
}

int launch_pf_windows_fast(epid_ctx* ctx, cudaStream_t stream, const PfConst* cst, const FrameRef* refs, PfFrame* fr, PfWin* wins, int n) {
    const size_t smem = W2_POOL;
    EPID_SMEM_OPT_IN(ctx, k_pf_windows_fast, smem);
    dim3 grid(W2_GRID_X, n);
    k_pf_windows_fast<<<grid, W2_WARPS * 32, smem, stream>>>(cst, refs, fr, wins);
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

}  // namespace epid
