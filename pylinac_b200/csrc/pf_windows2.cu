// Two-kernel (leaf, picket) window path of the PicketFence pipeline: integer streaming work and the 1-D analysis are separated so
// that each runs with (nearly) all 32 lanes busy and without CTA barriers.
//
// Reference semantics (unchanged): PicketFence._get_mlc_window / _is_mlc_peak_in_window (picketfence.py:847-886) and
// MLCValue.get_peak_positions (picketfence.py:1605-1628) -> FWXMProfilePhysical.field_edge_idx (core/profile.py:602-611).
//
//   k_pf_win_medians   warp-autonomous.  A task = one leaf x a group of G neighbouring pickets (their windows are column ranges of
//       the same band of rows; G is the largest group whose band fits a staging slot with the leaf's row count).  The band is
//       copied RAW into a per-warp shared-memory slot by one cp.async.bulk (TMA, UBLKCP) per row, issued from warp-uniform
//       operands, completion on an mbarrier; two slots per warp, so the copy of the warp's next task is in flight while it works
//       on the current one.
//       P1  lanes own (picket of the group, row): sum and sum of squares of the row inside the picket's window (IDP.2A on packed
//           pixels, 32-bit partial sums), i.e. the exact integer variance numerator nc * S2 - S1^2 -- invariant under the frame's
//           ground / inversion map, so raw pixels do.  The numerators of a window are then ranked across its lanes (shuffles): only
//           the largest and the two middle ones leave the kernel (max / median of the row standard deviations).
//       P2  lanes own pairs of band columns: median over the rows by register sorting networks on packed u16x2 (VIMNMX.U16x2,
//           comparator lists generated at compile time); the median commutes with the monotone ground / inversion map, which is
//           applied to the result.  The column extremes give the window maximum.  The medians of a band go to the frame's median
//           pool contiguously (columns shared by overlapping windows are computed once).
//   k_pf_win_fwxm      thread per window, 32 windows of a warp in lock step: _is_mlc_peak_in_window from the three numerators and
//       the window maximum (same fp64 expressions as the reference), then the serial integer FWXM analysis of the median profile
//       (window_fwxm: fp64 only for the prominence, the half-height level and the two interpolations).  The profiles are
//       transposed through shared memory ([sample][window], stride 33): coalesced pool reads, conflict-free per-thread walks.
//
// Results are bit-identical to k_pf_windows_fast (same integer quantities, same fp64 expressions; tests/test_gpu_pf.py compares
// them).  Frames this path does not cover (Left-Right orientation, unaligned pitch, windows wider than 64 samples or taller than
// 32 rows, more than 1024 windows) are left to k_pf_windows_fast: this kernel sets PfFrame.win2 for the frames it takes.
#include "pf_common.cuh"
#include "pf_win_common.cuh"
#include "tma.cuh"

namespace epid {

constexpr int WA_WARPS = 8;
// bytes per staging slot: 13 rows x 336 B (three 51-sample windows of a 5 mm leaf at 2.56 px/mm), 3 CTAs / SM.  Measured against
// 6656-byte slots (26 rows x 256 B, 2 CTAs / SM): 0.296 vs 0.317 ms per 512 frames
constexpr int WA_SLOT = 4416;
constexpr int WA_GRID_X = 4;           // CTAs per frame
constexpr int WA_GMAX = 4;             // pickets per task
constexpr int WA_KMAX = 4;             // rows per lane in P1: ceil(32 rows / (32 lanes / 4 pickets))
constexpr int WB_THREADS = 128;
constexpr int WB_ST = 33;              // transposed profile stride (words): [sample][window of the warp]

__device__ __forceinline__ int wa_row_stride_bytes(int nvec) { return (nvec | 1) * 16; }   // odd vector count: rows start 4 banks apart

struct W2Geo {
    int ok, ntasks;
    int nvmax[WA_GMAX + 1];     // widest band (16-byte vectors per row) when pickets are taken g at a time
    int gtot[WA_GMAX + 1];      // median-pool samples of one leaf when pickets are taken g at a time
};

__global__ void __launch_bounds__(WA_WARPS * 32, 3)
k_pf_win_medians(const PfConst* __restrict__ cc, const FrameRef* __restrict__ frames, PfFrame* fr, PfWinRec* __restrict__ recs,
                 uint32_t* __restrict__ pools) {
    extern __shared__ __align__(128) unsigned char smraw[];          // WA_WARPS x 2 slots
    __shared__ __align__(8) unsigned long long s_bar[WA_WARPS][2];
    __shared__ W2Geo s_geo;
    __shared__ int s_a0[PF_P], s_a1[PF_P];
    // per group size / group: first band column (view coordinates), vectors per row, first / one-past-last band word that belongs to
    // a window, offset of the band inside the leaf's part of the median pool
    __shared__ short s_gcs[WA_GMAX + 1][PF_P], s_gnv[WA_GMAX + 1][PF_P], s_gt0[WA_GMAX + 1][PF_P], s_gt1[WA_GMAX + 1][PF_P];
    __shared__ int s_gofs[WA_GMAX + 1][PF_P];
    __shared__ short s_b0[PF_L], s_nr[PF_L];
    __shared__ unsigned char s_lg[PF_L];                              // pickets per task of this leaf
    __shared__ int s_toff[PF_L + 1];                                  // tasks before leaf li
    __shared__ int s_moff[PF_L + 1];                                  // median-pool samples before leaf li
    const int fi = blockIdx.y;
    const PfConst& c = *cc;
    PfFrame& f = fr[fi];
    const int tid = threadIdx.x, lane = tid & 31;
    constexpr bool LDGSTS = false;          // (an LDGSTS loader was measured at the same speed as the TMA row copies: profiles/r2_summary.md)
    const int wid = __shfl_sync(0xffffffffu, tid >> 5, 0);           // warp-uniform for the compiler
    const int H = c.H, W = c.W;
    const FrameRef frf = frames[fi];
    const int mis = (int)((reinterpret_cast<uintptr_t>(frf.origin) >> 1) & 7);
    if (lane == 0) {
        mbar_init(smem_u32(&s_bar[wid][0]), 1);
        mbar_init(smem_u32(&s_bar[wid][1]), 1);
    }
    if (tid == 0) mbar_fence_init();
    // ---- frame geometry: identical in every CTA of the frame (pure function of PfFrame / PfConst)
    const int st = f.status;
    const double sp = f.spacing;
    const int np = f.n_pickets, ninview = f.n_inview;
    const bool pre_ok = c.win2 && st == EPID_PF_OK && f.orientation == 0 && (frf.pitch & 7) == 0 && np >= 1 && np <= PF_P && ninview > 0 &&
                        ninview <= PF_L && sp == sp && sp >= 2.0 && sp < 4096.0 && (long long)ninview * np <= PF_W2_WCAP;
    if (!pre_ok) return;      // uniform across the CTA
    const double dpmm = c.p.dpmm;
    int bad = 0;
    for (int i = tid; i < ninview; i += WA_WARPS * 32) {
        const int leaf = f.inview[i];
        const double lw_px = c.p.leaf_width_mm[leaf] * dpmm;
        const double lc_px = c.p.leaf_center_mm[leaf] * dpmm + (double)H / 2.0;
        const int b0 = max((int)(lc_px - lw_px / 2.0), 0), b1 = min((int)(lc_px + lw_px / 2.0), H);   // _get_mlc_window: int() truncates
        s_b0[i] = (short)b0;
        s_nr[i] = (short)(b1 - b0);
        if (b1 - b0 > PF_W2_NRW) bad = 1;
    }
    if (wid == 0) {
        int a0 = W, a1 = 0;
        if (lane < np) {
            const double pidx = (double)f.picket_idx[lane];
            a0 = max((int)(pidx - sp / 2.0), 0);
            a1 = min((int)(pidx + sp / 2.0), W);
            s_a0[lane] = a0;
            s_a1[lane] = a1;
            if (a1 - a0 > PF_W2_NCW) bad = 1;
        }
        __syncwarp();
        for (int g = 1; g <= WA_GMAX; g++) {       // band of every group of g neighbouring pickets
            const int ng = (np + g - 1) / g;
            int nvec = 0, nsamp = 0;
            if (lane < ng) {
                int lo = W, hi = 0;
                for (int q = 0; q < g && lane * g + q < np; q++) {
                    const int x0 = s_a0[lane * g + q], x1 = s_a1[lane * g + q];
                    if (x1 > x0) { lo = min(lo, x0); hi = max(hi, x1); }
                }
                const bool empty = hi <= lo;
                if (empty) { lo = 0; hi = 8; }
                const int cs = lo - ((lo + mis) & 7);
                const int ce = hi + ((8 - ((hi + mis) & 7)) & 7);
                nvec = (ce - cs) >> 3;
                const int t0 = (lo - cs) >> 1, t1 = empty ? t0 : (hi - cs + 1) >> 1;
                s_gcs[g][lane] = (short)cs;
                s_gnv[g][lane] = (short)nvec;
                s_gt0[g][lane] = (short)t0;
                s_gt1[g][lane] = (short)t1;
                nsamp = 2 * (t1 - t0);
            }
            int inc = nsamp;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            if (lane < ng) s_gofs[g][lane] = inc - nsamp;
            const int nvmax = warp_max(nvec);
            const int tot = __shfl_sync(0xffffffffu, inc, 31);
            if (lane == 0) { s_geo.nvmax[g] = nvmax; s_geo.gtot[g] = tot; }
        }
    }
    bad = __syncthreads_or(bad);
    if (wid == 0) {
        // pickets per task of every leaf: as many as fit a slot with the leaf's row count; running task / pool offsets
        int run = 0, mrun = 0;
        for (int base = 0; base < ninview; base += 32) {
            const int i = base + lane;
            int cnt = 0, msz = 0;
            if (i < ninview) {
                const int nr = s_nr[i];
                int G = 0;
                for (int g = WA_GMAX; g >= 1 && G == 0; g--)
                    if (max(nr, 1) * wa_row_stride_bytes(s_geo.nvmax[g]) <= WA_SLOT) G = g;
                if (G == 0) bad = 1;
                G = max(G, 1);
                s_lg[i] = (unsigned char)G;
                cnt = (np + G - 1) / G;
                msz = s_geo.gtot[G];
            }
            int inc = cnt, minc = msz;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o), u = __shfl_up_sync(0xffffffffu, minc, o);
                if (lane >= o) { inc += t; minc += u; }
            }
            if (i < ninview) { s_toff[i] = run + inc - cnt; s_moff[i] = mrun + minc - msz; }
            run += __shfl_sync(0xffffffffu, inc, 31);
            mrun += __shfl_sync(0xffffffffu, minc, 31);
        }
        if (mrun > PF_W2_POOL) bad = 1;
        bad = __any_sync(0xffffffffu, bad);
        if (lane == 0) {
            s_toff[ninview] = run;
            s_moff[ninview] = mrun;
            s_geo.ntasks = run;
            s_geo.ok = bad ? 0 : 1;
            if (!bad && blockIdx.x == 0) f.win2 = 1;
        }
    }
    __syncthreads();
    if (!s_geo.ok) return;
    const int ntasks = s_geo.ntasks;
    const int inv = f.inv;
    const uint32_t mn = f.mn, mx = f.mx;
    const int sag = c.p.sag_px;
    unsigned char* slot0 = smraw + (size_t)wid * 2 * WA_SLOT;
    const uint32_t bar0 = smem_u32(&s_bar[wid][0]), bar1 = smem_u32(&s_bar[wid][1]);
    PfWinRec* frecs = recs + (size_t)fi * PF_W2_WCAP;
    uint32_t* pool = pools + (size_t)fi * PF_W2_POOL;

    auto leaf_of = [&](int task, int li) { while (s_toff[li + 1] <= task) li++; return li; };     // tasks are visited in ascending order
    auto issue = [&](int task, int li, int sl) {
        const int G = s_lg[li], g = task - s_toff[li];
        const int b0 = s_b0[li], nr = s_nr[li];
        const int nvec = s_gnv[G][g], cs = s_gcs[G][g];
        if (nr <= 0) return;                         // nothing to copy: the consumer does not wait either
        const int RS = wa_row_stride_bytes(nvec);
        if (LDGSTS) {
            const int nv_tot = nr * nvec;
            const float inv_nvec = 1.0f / (float)nvec;
            for (int idx = lane; idx < nv_tot; idx += 32) {
                const int r = (int)(((float)idx + 0.5f) * inv_nvec), v = idx - r * nvec;
                int row = b0 + r - sag;
                if (sag) { row %= H; if (row < 0) row += H; }
                const uint32_t dst = smem_u32(slot0 + (size_t)sl * WA_SLOT + (size_t)r * RS + (size_t)v * 16);
                const void* src = frf.origin + ((ptrdiff_t)row * frf.pitch + cs + v * 8);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
            }
            return;
        }
        const uint32_t bar = sl ? bar1 : bar0;
        const uint32_t bytes = (uint32_t)nvec * 16u;
        if (lane == 0) mbar_expect_tx(bar, (uint32_t)nr * bytes);
        __syncwarp();
        if (lane < nr) {                             // one bulk copy per row, each issued by the lane of that row
            int row = b0 + lane - sag;               // np.roll(sag) folded into the source row
            if (sag) { row %= H; if (row < 0) row += H; }
            tma_load_1d(smem_u32(slot0 + (size_t)sl * WA_SLOT + (size_t)lane * RS), frf.origin + ((ptrdiff_t)row * frf.pitch + cs), bytes, bar);
        }
    };

    const int tstride = gridDim.x * WA_WARPS;
    int task = blockIdx.x * WA_WARPS + wid;
    uint32_t ph0 = 0, ph1 = 0;
    int cur = 0, li = 0, li_next = 0;
    if (task < ntasks) { li = leaf_of(task, 0); issue(task, li, 0); }
    if (LDGSTS) asm volatile("cp.async.commit_group;" ::: "memory");
    for (; task < ntasks; task += tstride, cur ^= 1, li = li_next) {
        if (task + tstride < ntasks) {
            li_next = leaf_of(task + tstride, li);
            issue(task + tstride, li_next, cur ^ 1);     // that slot was released by the __syncwarp at the end of the previous iteration
        }
        if (LDGSTS) asm volatile("cp.async.commit_group;" ::: "memory");      // (possibly empty) group of the next task
        const int G = s_lg[li], g = task - s_toff[li];
        const int nr = s_nr[li];
        const int nvec = s_gnv[G][g], cs = s_gcs[G][g];
        const int RS = wa_row_stride_bytes(nvec);
        const int Gn = min(G, np - g * G);
        const int t_lo = s_gt0[G][g], t_hi = s_gt1[G][g];
        const int boff = s_moff[li] + s_gofs[G][g];                   // the band's first sample in the median pool (even)
        PfWinRec* lrec = frecs + (size_t)li * np + (size_t)g * G;
        if (lane < Gn) {       // header: the shape of the window (empty windows are reported by the analysis kernel) and its samples
            const int a0 = s_a0[g * G + lane], a1 = s_a1[g * G + lane];
            lrec[lane].hdr = ((uint32_t)(uint16_t)(short)max(min(a1 - a0, 32767), -32768)) | ((uint32_t)(uint16_t)(short)nr << 16);
            lrec[lane].moff = (uint32_t)(boff + (a0 - (cs + 2 * t_lo)));
        }
        if (nr <= 0) { __syncwarp(); continue; }
        if (LDGSTS) { asm volatile("cp.async.wait_group 1;" ::: "memory"); __syncwarp(); }      // everything but the newest group has landed
        else if (cur) { mbar_wait(bar1, ph1); ph1 ^= 1u; } else { mbar_wait(bar0, ph0); ph0 ^= 1u; }
        const unsigned char* band = slot0 + (size_t)cur * WA_SLOT;
        // ---- P1: lanes = (picket of the group, row): rows [k * RPI, (k + 1) * RPI) in pass k
        {
            const int RPI = Gn == 1 ? 32 : (Gn == 2 ? 16 : (Gn == 3 ? 10 : 8));
            const int q = Gn == 1 ? 0 : (Gn == 2 ? lane >> 4 : (Gn == 3 ? lane / 10 : lane >> 3));
            const int rr = lane - q * RPI;
            const bool lane_on = q < Gn;
            const int a0 = lane_on ? s_a0[g * G + q] : 0, a1 = lane_on ? s_a1[g * G + q] : 0;
            const bool win_on = lane_on && a1 > a0;
            const int j0 = a0 - cs, j1 = a1 - cs;
            const int wlo = j0 >> 1, whi = (j1 - 1) >> 1;              // first / last word that holds window samples
            uint32_t mfirst = (j0 & 1) ? 0xffff0000u : 0xffffffffu;    // samples outside the window read as zero: sums unchanged
            uint32_t mlast = (j1 & 1) ? 0x0000ffffu : 0xffffffffu;
            if (wlo == whi) { mfirst &= mlast; }
            const unsigned long long ncl = (unsigned long long)(a1 - a0);
            const int nk = (nr + RPI - 1) / RPI;                       // <= WA_KMAX
#pragma unroll
            for (int k = 0; k < WA_KMAX; k++) {
                if (k < nk) {
                    const int r = k * RPI + rr;
                    if (lane_on && r < nr) {
                        unsigned long long numv = 0;
                        uint32_t e = 0x0000ffffu;
                        if (win_on) {
                            const uint32_t* wp = reinterpret_cast<const uint32_t*>(band + (size_t)r * RS);
                            uint32_t s1 = 0, sA = 0, sB = 0, mx2 = 0, mn2 = 0xffffffffu;
                            auto acc = [&](uint32_t x) {
                                // lo^2 + hi^2 = 256 * (lo * (lo >> 8) + hi * (hi >> 8)) + (lo * (lo & 255) + hi * (hi & 255)): two IDP.2A
                                s1 = __dp2a_lo(x, 0x0101u, s1);
                                sA = __dp2a_lo(x, __byte_perm(x, 0u, 0x4431), sA);
                                sB = __dp2a_lo(x, __byte_perm(x, 0u, 0x4420), sB);
                                mx2 = __vmaxu2(mx2, x);
                            };
                            // the masked edge words: zero for the sums and the maximum, all-ones for the minimum
                            const uint32_t xf = wp[wlo];
                            acc(xf & mfirst);
                            mn2 = __vminu2(mn2, xf | ~mfirst);
#pragma unroll 8
                            for (int w = wlo + 1; w < whi; w++) { const uint32_t x = wp[w]; acc(x); mn2 = __vminu2(mn2, x); }
                            if (whi > wlo) { const uint32_t xl = wp[whi]; acc(xl & mlast); mn2 = __vminu2(mn2, xl | ~mlast); }
                            const unsigned long long s2 = ((unsigned long long)sA << 8) + (unsigned long long)sB;
                            numv = ncl * s2 - (unsigned long long)s1 * s1;
                            e = (max(mx2 & 0xffffu, mx2 >> 16) << 16) | min(mn2 & 0xffffu, mn2 >> 16);
                        }
                        lrec[q].num[r] = numv;
                        lrec[q].ext[r] = e;
                    }
                }
            }
        }
        // ---- P2: 2 * median over the rows for every pair of band columns between the group's first and last window
        {
            const uint16_t* px = reinterpret_cast<const uint16_t*>(band);
            const int S = RS >> 1;
            for (int t = t_lo + lane; t < t_hi; t += 32) {
                const uint2 mm = pair_median_any(px, S, nr, t);
                const uint32_t g0 = inv ? 2u * mx - mm.x : mm.x - 2u * mn;
                const uint32_t g1 = inv ? 2u * mx - mm.y : mm.y - 2u * mn;
                *reinterpret_cast<uint2*>(pool + boff + 2 * (t - t_lo)) = make_uint2(g0, g1);
            }
        }
        __syncwarp();       // every lane is done with the slot: the next iteration may overwrite the other one... and this one after it
    }
}

// max, and the two middle order statistics of the nr keys a thread reads through key(i) (i < N slots, slots >= nr padded)
// (an fp64 network on DMNMX pairs -- the numerators are exact as doubles -- measured 25 % slower than this integer one)
template <int N, class F>
__device__ __forceinline__ void rank_keys(F key, int nr, unsigned long long& kmax, unsigned long long& ka, unsigned long long& kb) {
    unsigned long long r[N];
    kmax = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        r[i] = i < nr ? key(i) : ~0ull;
        if (i < nr && r[i] > kmax) kmax = r[i];
    }
    sort_net_u64<N>(r);
    const int k1 = (nr - 1) / 2, k2 = nr / 2;
    ka = 0; kb = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        if (i == k1) ka = r[i];
        if (i == k2) kb = r[i];
    }
}

__global__ void __launch_bounds__(WB_THREADS, 4)
k_pf_win_fwxm(const PfConst* __restrict__ cc, PfFrame* fr, const PfWinRec* __restrict__ recs, const uint32_t* __restrict__ pools,
              PfWin* __restrict__ wins) {
    __shared__ uint32_t s_buf[WB_THREADS / 32][PF_W2_NCW * WB_ST];
    const int fi = blockIdx.y;
    PfFrame& f = fr[fi];
    if (!f.win2) return;
    const PfConst& c = *cc;
    const int np = f.n_pickets;
    const int total = f.n_inview * np;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wbase = blockIdx.x * WB_THREADS + wid * 32;
    if (wbase >= total) return;
    const PfWinRec* frecs = recs + (size_t)fi * PF_W2_WCAP;
    const uint32_t* pool = pools + (size_t)fi * PF_W2_POOL;
    uint32_t* buf = s_buf[wid];
    const int w = wbase + lane;
    const bool active = w < total;
    // ---- this thread's window: header, row extremes and variance numerators straight into registers (independent loads, all
    //      in flight at once; lanes read records 400 bytes apart)
    const PfWinRec& rec = frecs[active ? w : total - 1];
    const uint2 h2 = *reinterpret_cast<const uint2*>(&rec);
    const int my_nc = (int)(short)(h2.x & 0xffffu), my_nr = (int)(short)(h2.x >> 16);
    const uint32_t my_moff = h2.y;
    int li = 0, pk = 0;
    if (active) { li = w / np; pk = w - li * np; }
    PfWin& out = wins[((size_t)fi * PF_L + li) * PF_P + pk];
    bool run = false;
    if (active) {
        if (my_nc <= 0 || my_nr <= 0) {           // empty slice: np.max raises ValueError in the reference
            out.valid = 0; out.l = 0; out.r = 0; f.status = EPID_PF_WINDOW_NO_PEAK;
        } else {
            run = true;
        }
    }
    const int nrr = run ? my_nr : 0;
    const int nr_all = __reduce_max_sync(0xffffffffu, nrr);
    // ---- _is_mlc_peak_in_window (picketfence.py:847-857): std along travel per row = sqrt(num) / (nc * D)
    unsigned long long kmax = 0, ka = 0, kb = 0;
    uint32_t my_vmx = 0, my_vmn = 0xffffu;
    {
        auto key = [&](int i) { return rec.num[i]; };
        if (nr_all <= 16) rank_keys<16>(key, nrr, kmax, ka, kb);       // warp-uniform choice
        else rank_keys<32>(key, nrr, kmax, ka, kb);
#pragma unroll
        for (int i = 0; i < PF_W2_NRW; i++) {
            if (i < nrr) {
                const uint32_t e = rec.ext[i];
                my_vmx = max(my_vmx, e >> 16);
                my_vmn = min(my_vmn, e & 0xffffu);
            }
        }
    }
    if (run) {
        const double Dd = (double)f.D;
        const double dn = (double)my_nc * Dd;
        const double sd_max = sqrt((double)kmax) / dn;
        const double sa = sqrt((double)ka) / dn, sb = sqrt((double)kb) / dn;
        const double sd_med = (my_nr & 1) ? sa : (sa + sb) / 2.0;
        const uint32_t gmax = f.inv ? f.mx - my_vmn : my_vmx - f.mn;
        const bool above = ((double)gmax / Dd) > c.p.height_threshold * f.picket_val[pk];
        const bool not_edge = sd_max < c.p.edge_threshold * sd_med;
        if (!(above && not_edge)) {
            out.valid = 0; out.l = 0; out.r = 0;
            run = false;
        }
    }
    // ---- median profiles of the 32 windows -> [sample][window]
    {
        const int nc_all = __reduce_max_sync(0xffffffffu, run ? my_nc : 0);     // samples beyond a window's own nc are never read
        if (nc_all > 0) {
#pragma unroll 8
            for (int k = 0; k < 32; k++) {
                const uint32_t mo = __shfl_sync(0xffffffffu, my_moff, k);
                const uint32_t v0 = pool[mo + lane];                  // stays inside the frame's pool: moff + 64 <= pool size + slack
                const uint32_t v1 = nc_all > 32 ? pool[mo + lane + 32] : 0u;
                buf[lane * WB_ST + k] = v0;
                if (nc_all > 32) buf[(lane + 32) * WB_ST + k] = v1;
            }
        }
    }
    __syncwarp();
    if (run) {
        double l = 0, r = 0;
        const int v = window_fwxm<WB_ST>(buf + lane, my_nc, l, r);
        out.valid = v;
        if (v) { out.l = l; out.r = r; }
        else f.status = EPID_PF_WINDOW_NO_PEAK;
    }
}

// records of every window + median pools (64 samples of slack behind the last pool: the profile staging reads 64 samples per window)
size_t pf_win2_scratch_bytes(int n) {
    return sizeof(PfWinRec) * (size_t)n * PF_W2_WCAP + 256 + sizeof(uint32_t) * ((size_t)n * PF_W2_POOL + 256);
}

int launch_pf_windows2(epid_ctx* ctx, cudaStream_t stream, const PfConst* cst, const FrameRef* refs, PfFrame* fr, PfWinRec* recs, PfWin* wins,
                       int n, PfTimers* tm) {
    uint32_t* pools = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(recs) + ((sizeof(PfWinRec) * (size_t)n * PF_W2_WCAP + 255) / 256) * 256);
    const size_t smem = (size_t)WA_WARPS * 2 * WA_SLOT;
    EPID_SMEM_OPT_IN(ctx, k_pf_win_medians, smem);
    k_pf_win_medians<<<dim3(WA_GRID_X, n), WA_WARPS * 32, smem, stream>>>(cst, refs, fr, recs, pools);
    ctx->launches++;
    if (tm) { int rc = tm->mark(stream, PF_STAGE_WIN_MEDIANS); if (rc != EPID_OK) return rc; }
    k_pf_win_fwxm<<<dim3(PF_W2_WCAP / WB_THREADS, n), WB_THREADS, 0, stream>>>(cst, fr, recs, pools, wins);
    ctx->launches++;
    if (tm) { int rc = tm->mark(stream, PF_STAGE_WIN_FWXM); if (rc != EPID_OK) return rc; }
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

}  // namespace epid
