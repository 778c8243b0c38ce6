// Fused frame statistics: ONE streaming read of a uint16 frame view produces min, max, sum, row sums,
// column sums, the four check_inversion corner sums and EXACT order statistics (from a 65536-bin histogram
// that never leaves shared memory).
//
// Replaces the reference's numpy passes: array.min()/max() (picketfence.py:231-232, core/image.py:851),
// np.percentile / np.median of the full frame (picketfence.py:233,1510; core/image.py:918-920),
// np.mean(image, axis) (picketfence.py:748-750), corner means (core/image.py:881-896).
//
// Design (B200): one persistent CTA of 1024 threads per SM, one frame per CTA at a time.  Each thread owns a
// fixed 8-pixel column vector (128-bit ld.global.nc.L1::no_allocate, row pitch keeps it 16-byte aligned) and
// strides over rows, so column sums live in registers, row sums are one warp-shuffle reduction + one shared
// atomic per warp-row, and the histogram is 65536 packed 16-bit counters = 128 KB of shared memory updated
// with ATOMS.ADD (1 or 0x10000 into the 32-bit word).  A packed counter can overflow only if > 65535 pixels of
// a frame share one value; that is detected exactly (the decoded bin total then differs from the pixel count)
// and the frame is re-run by the MODE 1 variant (32-bit counters over value>>1 plus a second pass resolving
// the low bit), so results are always exact.
#include "stats.cuh"

namespace epid {

constexpr int HIST_WORDS = 32768;

int make_stats_geom(StatsGeom* g, int H, int W) {
    if (H <= 0 || W <= 0 || H > STATS_MAX_DIM || W > STATS_MAX_DIM) {
        set_error("frame view %d x %d outside the supported range (1..%d)", H, W, STATS_MAX_DIM);
        return EPID_ERR_UNSUPPORTED;
    }
    memset(g, 0, sizeof(*g));
    g->H = H;
    g->W = W;
    const int vpr = (W + 7 + 7) / 8;  // worst-case misalignment of 7 pixels
    g->vprp = (vpr + 31) / 32 * 32;
    g->groups = STATS_THREADS / g->vprp;
    if (g->groups < 1) {
        set_error("frame view too wide (%d)", W);
        return EPID_ERR_UNSUPPORTED;
    }
    return EPID_OK;
}

__device__ __forceinline__ void block_scan_excl_1024(uint32_t v, uint32_t* s_warp, uint32_t& excl, uint32_t& total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = s_warp[lane];
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        s_warp[lane] = winc - w;       // exclusive warp offsets
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    excl = s_warp[wid] + inc - v;
    total = s_warp[32];
    __syncthreads();
}

// MODE 0: packed u16 counters, all 65536 bins.  MODE 1: u32 counters over (v >> 1), low bit resolved by a 2nd pass.
template <int MODE>
__global__ void __launch_bounds__(STATS_THREADS, 1)
k_frame_stats(const StatsGeom g, const FrameRef* __restrict__ frames, int nframes,
              FrameStats* __restrict__ stats, uint32_t* __restrict__ rowsum_out, uint32_t* __restrict__ colsum_out) {
    extern __shared__ uint32_t smem[];
    uint32_t* hist = smem;                                   // HIST_WORDS
    uint32_t* colpart = hist + HIST_WORDS;                   // STATS_THREADS * 8
    uint32_t* s_warp = colpart + STATS_THREADS * 8;          // 40
    uint32_t* s_misc = s_warp + 40;                          // 8 + 3*STATS_MAX_RANKS (even word index: 64-bit atomics)
    uint32_t* rowsum_sm = s_misc + 8 + 3 * STATS_MAX_RANKS;  // H

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int grp = tid / g.vprp;
    const int jc = tid - grp * g.vprp;
    const bool active_grp = grp < g.groups;

    for (int fi = blockIdx.x; fi < nframes; fi += gridDim.x) {
        if (MODE == 1 && stats[fi].overflow == 0) continue;
        const FrameRef fr = frames[fi];
        const uint16_t* __restrict__ f = fr.origin;
        const int pitch = fr.pitch;
        // aligned vector grid of this frame: vector j covers view columns [8j - mis, 8j - mis + 8)
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
        for (int i = tid; i < HIST_WORDS; i += STATS_THREADS) hist[i] = 0;
        for (int i = tid; i < g.H; i += STATS_THREADS) rowsum_sm[i] = 0;
        __syncthreads();

        uint32_t mn = 0xffffu, mx = 0, csum[8];
        unsigned long long tsum = 0;
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
                    if (rr >= g.H) break;  // warp-uniform
                    uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
                    uint32_t rs = 0;
                    if (valid == 0xffu) {
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const uint32_t lo = w[k] & 0xffffu, hi = w[k] >> 16;
                            if (MODE == 0) {
                                atomicAdd(&hist[lo >> 1], (lo & 1) ? 0x10000u : 1u);
                                atomicAdd(&hist[hi >> 1], (hi & 1) ? 0x10000u : 1u);
                            } else {
                                atomicAdd(&hist[lo >> 1], 1u);
                                atomicAdd(&hist[hi >> 1], 1u);
                            }
                            mn = min(mn, min(lo, hi));
                            mx = max(mx, max(lo, hi));
                            csum[2 * k] += lo;
                            csum[2 * k + 1] += hi;
                            rs += lo + hi;
                        }
                    } else if (valid) {
#pragma unroll
                        for (int k = 0; k < 8; k++) {
                            if (valid >> k & 1) {
                                const uint32_t v = (w[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
                                if (MODE == 0)
                                    atomicAdd(&hist[v >> 1], (v & 1) ? 0x10000u : 1u);
                                else
                                    atomicAdd(&hist[v >> 1], 1u);
                                mn = min(mn, v);
                                mx = max(mx, v);
                                csum[k] += v;
                                rs += v;
                            }
                        }
                    }
                    tsum += rs;
                    rs = warp_sum(rs);
                    if (lane == 0) atomicAdd(&rowsum_sm[rr], rs);
                }
            }
        }
        // column partials -> shared
#pragma unroll
        for (int k = 0; k < 8; k++) colpart[tid * 8 + k] = active ? csum[k] : 0u;
        // block reductions of min / max / sum
        mn = warp_min(mn);
        mx = warp_max(mx);
        tsum = warp_sum(tsum);
        __syncthreads();  // (also orders hist / rowsum / colpart writes)
        if (tid == 0) { s_misc[0] = 0xffffu; s_misc[1] = 0; s_misc[2] = 0; s_misc[3] = 0; s_misc[4] = 0; s_misc[5] = 0; }
        __syncthreads();
        if (lane == 0) {
            atomicMin(&s_misc[0], mn);
            atomicMax(&s_misc[1], mx);
            atomicAdd(reinterpret_cast<unsigned long long*>(&s_misc[2]), tsum);
        }
        // corner boxes (core/image.py:881-894): rows [rp, rp+box) and [H-rp-box, H-rp), cols [cp, cp+box) and [W-cp-box, W-cp)
        if (g.box > 0) {
            const int per = g.box * g.box;
            unsigned long long cs = 0;
            for (int i = tid; i < 4 * per; i += STATS_THREADS) {
                const int b = i / per, o = i - b * per;
                const int y = o / g.box, x = o - y * g.box;
                const int rr = ((b & 2) ? g.H - g.rp - g.box : g.rp) + y;
                const int cc = ((b & 1) ? g.W - g.cp - g.box : g.cp) + x;
                if (rr >= 0 && rr < g.H && cc >= 0 && cc < g.W) cs += __ldg(f + (size_t)rr * pitch + cc);
            }
            cs = warp_sum(cs);
            if (lane == 0 && cs) atomicAdd(reinterpret_cast<unsigned long long*>(&s_misc[4]), cs);
        }
        __syncthreads();
        // outputs: sums
        if (colsum_out) {
            for (int x = tid; x < g.W; x += STATS_THREADS) {
                const int ac = x + mis;  // position inside the per-row vector grid
                uint32_t s = 0;
                for (int gg = 0; gg < g.groups; gg++) s += colpart[(gg * g.vprp) * 8 + ac];
                colsum_out[(size_t)fi * g.W + x] = s;
            }
        }
        if (rowsum_out)
            for (int y = tid; y < g.H; y += STATS_THREADS) rowsum_out[(size_t)fi * g.H + y] = rowsum_sm[y];

        // ---- order statistics from the histogram
        uint32_t cnt = 0;
        {
            const uint32_t* hw = hist + tid * 32;
#pragma unroll 8
            for (int i = 0; i < 32; i++) {
                // rotate the start so that the 32 lanes of a warp hit 32 different banks
                const uint32_t w = hw[(i + lane) & 31];
                cnt += (MODE == 0) ? ((w & 0xffffu) + (w >> 16)) : w;
            }
        }
        uint32_t excl, total;
        block_scan_excl_1024(cnt, s_warp, excl, total);
        const uint32_t npix = (uint32_t)g.H * (uint32_t)g.W;
        const bool overflow = (MODE == 0) && (total != npix);
        uint32_t* s_val = s_misc + 8;                       // value (MODE 0) or bin (MODE 1)
        uint32_t* s_off = s_val + STATS_MAX_RANKS;          // MODE 1: rank offset inside the bin
        uint32_t* s_cnt = s_off + STATS_MAX_RANKS;          // MODE 1: count of even values in the bin
        if (!overflow) {
            for (int qi = 0; qi < g.nranks; qi++) {
                const uint32_t k = g.ranks[qi];
                if (k >= excl && k < excl + cnt) {
                    uint32_t acc = excl;
                    const uint32_t* hw = hist + tid * 32;
                    for (int i = 0; i < 32; i++) {
                        const uint32_t w = hw[i];
                        if (MODE == 0) {
                            const uint32_t c0 = w & 0xffffu, c1 = w >> 16;
                            if (k < acc + c0) { s_val[qi] = (tid * 32 + i) * 2; break; }
                            acc += c0;
                            if (k < acc + c1) { s_val[qi] = (tid * 32 + i) * 2 + 1; break; }
                            acc += c1;
                        } else {
                            if (k < acc + w) { s_val[qi] = tid * 32 + i; s_off[qi] = k - acc; s_cnt[qi] = 0; break; }
                            acc += w;
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (MODE == 1 && g.nranks > 0) {
            // second pass: how many pixels equal 2*bin (the even value of each target bin)?
            uint32_t local[STATS_MAX_RANKS];
#pragma unroll
            for (int qi = 0; qi < STATS_MAX_RANKS; qi++) local[qi] = 0;
            for (int i = tid; i < g.H * g.W; i += STATS_THREADS) {
                const int rr = i / g.W, cc = i - rr * g.W;
                const uint32_t v = __ldg(f + (size_t)rr * pitch + cc);
#pragma unroll
                for (int qi = 0; qi < STATS_MAX_RANKS; qi++)
                    if (qi < g.nranks && v == 2u * s_val[qi]) local[qi]++;
            }
#pragma unroll
            for (int qi = 0; qi < STATS_MAX_RANKS; qi++) {
                if (qi < g.nranks) {
                    uint32_t s = warp_sum(local[qi]);
                    if (lane == 0 && s) atomicAdd(&s_cnt[qi], s);
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            FrameStats& o = stats[fi];
            o.mn = s_misc[0];
            o.mx = s_misc[1];
            o.npix = npix;
            o.sum = *reinterpret_cast<unsigned long long*>(&s_misc[2]);
            o.corner_sum = *reinterpret_cast<unsigned long long*>(&s_misc[4]);
            o.overflow = overflow ? 1u : 0u;
            if (!overflow)
                for (int qi = 0; qi < g.nranks; qi++)
                    o.ostat[qi] = (MODE == 0) ? s_val[qi] : (2u * s_val[qi] + (s_off[qi] >= s_cnt[qi] ? 1u : 0u));
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ multi-CTA variant
// The single-CTA kernel above keeps a frame's histogram in shared memory, which ties a frame to one SM (~1 GB/s per frame).  This
// variant spreads a frame over HV_PARTS CTAs: each streams a block of rows with 16-byte loads, merges equal values of a warp
// (__match_any_sync) into a direct-mapped shared-memory cache of histogram bins (first claimant owns a slot, losers go to the global
// histogram; one global atomic per occupied slot at the end), keeps column sums in registers and writes row sums directly; a
// second kernel (one CTA per frame) turns the 65536-bin histogram into min / max / sum / order statistics and adds the column
// partials.  Exact like the single-CTA kernel (32-bit counters, no overflow path).  Views up to 2040 columns.
constexpr int HV_PARTS = 16;
constexpr int HV_THREADS = 256;
constexpr int HV_WARPS = HV_THREADS / 32;
constexpr int HV_SLOTS = 4096;

template <int VPL>
__global__ void __launch_bounds__(HV_THREADS)
k_hist_view(const StatsGeom g, const FrameRef* __restrict__ frames, uint32_t* __restrict__ hist, uint32_t* __restrict__ rowsum_out,
            uint32_t* __restrict__ colpart, int wa) {
    __shared__ uint32_t s_tag[HV_SLOTS];     // value + 1, 0 = free
    __shared__ uint32_t s_cnt[HV_SLOTS];
    extern __shared__ uint32_t s_col[];      // wa column accumulators of the CTA
    const int fi = blockIdx.y, part = blockIdx.x;
    const FrameRef fr = frames[fi];
    const uint16_t* __restrict__ f = fr.origin;
    const int pitch = fr.pitch;
    uint32_t* h = hist + (size_t)fi * 65536;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const bool aligned = (pitch % 8) == 0;
    const int mis = aligned ? (int)((reinterpret_cast<uintptr_t>(f) >> 1) & 7) : 0;
    for (int i = tid; i < HV_SLOTS; i += HV_THREADS) { s_tag[i] = 0; s_cnt[i] = 0; }
    for (int i = tid; i < wa; i += HV_THREADS) s_col[i] = 0;
    __syncthreads();
    auto add = [&](uint32_t v, bool in) {
        const unsigned m = __match_any_sync(0xffffffffu, in ? v : 0x10000u);
        if (in && lane == __ffs(m) - 1) {
            const uint32_t cn = (uint32_t)__popc(m), slot = v & (HV_SLOTS - 1);
            const uint32_t old = atomicCAS(&s_tag[slot], 0u, v + 1u);
            if (old == 0u || old == v + 1u) atomicAdd(&s_cnt[slot], cn);
            else atomicAdd(&h[v], cn);
        }
    };
    const int rp = (g.H + HV_PARTS - 1) / HV_PARTS;
    const int r0 = part * rp, r1 = min(g.H, r0 + rp);
    uint32_t csum[VPL][8];
#pragma unroll
    for (int k = 0; k < VPL; k++)
#pragma unroll
        for (int e = 0; e < 8; e++) csum[k][e] = 0;
    for (int r = r0 + wid; r < r1; r += HV_WARPS) {
        const uint16_t* rowp = f + (size_t)r * pitch;
        uint32_t rs = 0;
        uint4 q[VPL];
        uint32_t valid[VPL];
#pragma unroll
        for (int k = 0; k < VPL; k++) {
            const int col_first = (lane + 32 * k) * 8 - mis;
            uint32_t vm = 0;
#pragma unroll
            for (int e = 0; e < 8; e++) { const int cidx = col_first + e; if (cidx >= 0 && cidx < g.W) vm |= 1u << e; }
            valid[k] = vm;
            q[k] = make_uint4(0, 0, 0, 0);
            if (vm) {
                if (aligned) q[k] = ldg_stream16(rowp + col_first);
                else {
                    uint32_t w4[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int e = 0; e < 8; e++) if (vm >> e & 1) w4[e >> 1] |= (uint32_t)__ldg(rowp + col_first + e) << ((e & 1) * 16);
                    q[k] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < VPL; k++) {
            const uint32_t w4[4] = {q[k].x, q[k].y, q[k].z, q[k].w};
            const bool any = __any_sync(0xffffffffu, valid[k] != 0);
            if (!any) continue;     // warp-uniform
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const uint32_t v = (w4[e >> 1] >> ((e & 1) * 16)) & 0xffffu;
                const bool in = valid[k] >> e & 1;
                add(v, in);
                if (in) { csum[k][e] += v; rs += v; }
            }
        }
        rs = warp_sum(rs);
        if (lane == 0 && rowsum_out) rowsum_out[(size_t)fi * g.H + r] = rs;
    }
    // column partials: registers -> CTA accumulators -> one partial row per (frame, part)
#pragma unroll
    for (int k = 0; k < VPL; k++)
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int ac = (lane + 32 * k) * 8 + e;
            if (ac < wa && csum[k][e]) atomicAdd(&s_col[ac], csum[k][e]);
        }
    __syncthreads();
    if (colpart) for (int i = tid; i < wa; i += HV_THREADS) colpart[((size_t)fi * HV_PARTS + part) * wa + i] = s_col[i];
    for (int i = tid; i < HV_SLOTS; i += HV_THREADS) {
        const uint32_t tg = s_tag[i];
        if (tg) atomicAdd(&h[tg - 1u], s_cnt[i]);
    }
}

__global__ void __launch_bounds__(256)
k_stats_from_hist(const StatsGeom g, const FrameRef* __restrict__ frames, const uint32_t* __restrict__ hist, const uint32_t* __restrict__ colpart,
                  int wa, FrameStats* __restrict__ stats, uint32_t* __restrict__ colsum_out) {
    __shared__ uint32_t s_part[256];
    __shared__ unsigned long long s_wsum[256];
    __shared__ uint32_t s_first, s_last;
    __shared__ unsigned long long s_corner;
    __shared__ uint32_t s_val[STATS_MAX_RANKS];
    const int fi = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const uint32_t* h = hist + (size_t)fi * 65536;
    const FrameRef fr = frames[fi];
    uint32_t cnt = 0, lo_bin = 0xffffffffu, hi_bin = 0;
    unsigned long long ws = 0;
    for (int b = tid * 256; b < (tid + 1) * 256; b++) {
        const uint32_t hb = h[b];
        cnt += hb;
        ws += (unsigned long long)hb * (unsigned)b;
        if (hb) { if (lo_bin == 0xffffffffu) lo_bin = b; hi_bin = b; }
    }
    s_part[tid] = cnt;
    s_wsum[tid] = ws;
    if (tid == 0) { s_first = 0xffffffffu; s_last = 0; s_corner = 0; }
    __syncthreads();
    if (lo_bin != 0xffffffffu) { atomicMin(&s_first, lo_bin); atomicMax(&s_last, hi_bin); }
    uint32_t excl = 0;
    for (int k = 0; k < tid; k++) excl += s_part[k];
    for (int qi = 0; qi < g.nranks; qi++) {
        const uint32_t k = g.ranks[qi];
        if (k >= excl && k < excl + cnt) {
            uint32_t acc = excl;
            for (int b = tid * 256; b < (tid + 1) * 256; b++) {
                const uint32_t hb = h[b];
                if (k < acc + hb) { s_val[qi] = (uint32_t)b; break; }
                acc += hb;
            }
        }
    }
    // corner boxes (core/image.py:881-894)
    if (g.box > 0) {
        const int per = g.box * g.box;
        unsigned long long cs = 0;
        for (int i = tid; i < 4 * per; i += 256) {
            const int b = i / per, o = i - b * per;
            const int y = o / g.box, x = o - y * g.box;
            const int rr = ((b & 2) ? g.H - g.rp - g.box : g.rp) + y;
            const int cc = ((b & 1) ? g.W - g.cp - g.box : g.cp) + x;
            if (rr >= 0 && rr < g.H && cc >= 0 && cc < g.W) cs += __ldg(fr.origin + (size_t)rr * fr.pitch + cc);
        }
        cs = warp_sum(cs);
        if (lane == 0 && cs) atomicAdd(&s_corner, cs);
    }
    // column sums: the parts' partial rows (vector-grid columns) -> view columns
    if (colsum_out && colpart) {
        const bool aligned = (fr.pitch % 8) == 0;
        const int mis = aligned ? (int)((reinterpret_cast<uintptr_t>(fr.origin) >> 1) & 7) : 0;
        for (int x = tid; x < g.W; x += 256) {
            uint32_t sum = 0;
            for (int p = 0; p < HV_PARTS; p++) sum += colpart[((size_t)fi * HV_PARTS + p) * wa + x + mis];
            colsum_out[(size_t)fi * g.W + x] = sum;
        }
    }
    __syncthreads();
    if (tid == 0) {
        unsigned long long tot = 0;
        for (int k = 0; k < 256; k++) tot += s_wsum[k];
        FrameStats& o = stats[fi];
        o.mn = s_first;
        o.mx = s_last;
        o.npix = (uint32_t)g.H * (uint32_t)g.W;
        o.sum = tot;
        o.corner_sum = s_corner;
        o.overflow = 0;
        for (int qi = 0; qi < g.nranks; qi++) o.ostat[qi] = s_val[qi];
    }
}

static int ensure_hist_scratch(epid_ctx* ctx, size_t bytes) {
    if (ctx->hist_bytes >= bytes) return EPID_OK;
    if (ctx->hist_scratch) { EPID_CUDA(cudaStreamSynchronize(ctx->stream)); EPID_CUDA(cudaFree(ctx->hist_scratch)); ctx->hist_scratch = nullptr; ctx->hist_bytes = 0; }
    cudaError_t e = cudaMalloc(&ctx->hist_scratch, bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return EPID_ERR_NOMEM; }
    ctx->hist_bytes = bytes;
    return EPID_OK;
}

template <int VPL>
static int launch_hist_view(cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames, int cn, uint32_t* hist, uint32_t* rowsum,
                            uint32_t* colpart, int wa) {
    k_hist_view<VPL><<<dim3(HV_PARTS, cn), HV_THREADS, sizeof(uint32_t) * wa, stream>>>(g, d_frames, hist, rowsum, colpart, wa);
    return EPID_OK;
}

static int launch_frame_stats_v2(epid_ctx* ctx, cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames, int n, FrameStats* d_stats,
                                 uint32_t* d_rowsum, uint32_t* d_colsum) {
    const int nvec = (g.W + 7 + 7) / 8;
    const int vpl = (nvec + 31) / 32;
    const int wa = vpl * 32 * 8;                 // columns of the vector grid
    const int chunk = n < 256 ? n : 256;
    const size_t hist_b = sizeof(uint32_t) * (size_t)chunk * 65536, col_b = sizeof(uint32_t) * (size_t)chunk * HV_PARTS * wa;
    int rc = ensure_hist_scratch(ctx, hist_b + col_b + 512);
    if (rc != EPID_OK) return rc;
    uint32_t* hist = (uint32_t*)ctx->hist_scratch;
    uint32_t* colpart = d_colsum ? (uint32_t*)((char*)ctx->hist_scratch + (hist_b + 255) / 256 * 256) : nullptr;
    for (int c0 = 0; c0 < n; c0 += chunk) {
        const int cn = n - c0 < chunk ? n - c0 : chunk;
        EPID_CUDA(cudaMemsetAsync(hist, 0, sizeof(uint32_t) * (size_t)cn * 65536, stream));
        uint32_t* rs = d_rowsum ? d_rowsum + (size_t)c0 * g.H : nullptr;
        if (vpl <= 4) rc = launch_hist_view<4>(stream, g, d_frames + c0, cn, hist, rs, colpart, wa);
        else rc = launch_hist_view<8>(stream, g, d_frames + c0, cn, hist, rs, colpart, wa);
        k_stats_from_hist<<<cn, 256, 0, stream>>>(g, d_frames + c0, hist, colpart, wa, d_stats + c0, d_colsum ? d_colsum + (size_t)c0 * g.W : nullptr);
        ctx->launches += 2;
        EPID_CUDA(cudaGetLastError());
    }
    return EPID_OK;
}

// ------------------------------------------------------------------------------------------------ certified inversion statistics
// check_inversion_by_histogram (core/image.py:899-926) needs three percentiles of the frame only to DECIDE |p_mid - p_low| >
// |p_mid - p_high|.  Per-pixel histogram atomics cap the exact path at ~340 GB/s (LSU: ~2 cycles per lane), so FieldAnalysis / Starshot
// get the decision from counts instead, the way pf_stream.cu certifies PicketFence's decisions:
//   k_inv_pilot   CTA per frame: 4096-pixel grid sample, 16-step value bisection -> for each percentile a bracket [tL, tU] of sample order
//                 statistics 5 sigma either side of the rank
//   k_inv_stream  IV_PARTS CTAs per frame, one 16-byte load per lane and vector: exact min / max / sum, row sums, column partials and the
//                 six exact counts #(v < T) by packed u16x2 arithmetic (no atomics in the pixel loop)
//   k_inv_finish  CTA per frame: combines the parts; #(v < tL) <= rank_prev and #(v <= tU) > rank_next PROVE tL <= percentile <= tU; if the
//                 resulting intervals of the two distances do not overlap the decision is certified (FrameStats.overflow = 2 + inverted),
//                 otherwise the frame is listed for the exact histogram path (ostat exact, overflow = 0).
constexpr int IV_PARTS = 16;
constexpr int IV_THREADS = 256;
constexpr int IV_WARPS = IV_THREADS / 32;
constexpr int IV_SAMPLE_ROWS = 16;

struct InvPart {                 // per (frame, part)
    uint32_t cnt[6];
    uint32_t mn, mx;
    unsigned long long total;
};

__global__ void __launch_bounds__(IV_THREADS)
k_inv_pilot(const StatsGeom g, const FrameRef* __restrict__ frames, uint32_t* __restrict__ thr) {
    __shared__ uint32_t b_lo[6], b_hi[6], b_rank[6], b_fix[6];
    __shared__ uint32_t s_cnt[6][IV_WARPS];
    const int fi = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const FrameRef fr = frames[fi];
    const int H = g.H, W = g.W;
    const double npix = (double)H * (double)W;
    const uint32_t S = IV_THREADS * IV_SAMPLE_ROWS;
    uint32_t sv[IV_SAMPLE_ROWS];
    {
        const int col = min(W - 1, (int)(((2LL * tid + 1) * W) / (2 * IV_THREADS)));
#pragma unroll
        for (int i = 0; i < IV_SAMPLE_ROWS; i++) {
            const int row = min(H - 1, (int)(((2LL * i + 1) * H) / (2 * IV_SAMPLE_ROWS)));
            sv[i] = __ldg(fr.origin + (size_t)row * fr.pitch + col);
        }
    }
    if (tid < 6) {
        // lower (even) / upper (odd) sample rank of the bracket: 5 sigma of the binomial sample count around the pixel rank's quantile
        const double q = (double)g.ranks[tid] / npix;
        const double sg = sqrt(q * (1.0 - q) * (double)S);
        const double ctr = q * (double)S;
        const double rr = (tid & 1) ? ctr + 5.0 * sg + 3.0 : ctr - 5.0 * sg - 3.0;
        b_fix[tid] = 0;
        if (rr < 0.0) b_fix[tid] = 1;                      // bracket reaches below the sample: tL = 0
        if (rr > (double)(S - 1)) b_fix[tid] = 2;          // above the sample: tU = 65535
        b_rank[tid] = (uint32_t)fmin(fmax(rr, 0.0), (double)(S - 1));
        b_lo[tid] = 0;
        b_hi[tid] = 65535u;
    }
    __syncthreads();
    // smallest value t with #(sample <= t) > rank = the sample's order statistic, by bisection on the value
    for (int step = 0; step < 16; step++) {
        uint32_t c[6];
#pragma unroll
        for (int t = 0; t < 6; t++) {
            const uint32_t mid = (b_lo[t] + b_hi[t]) >> 1;
            uint32_t cc = 0;
#pragma unroll
            for (int i = 0; i < IV_SAMPLE_ROWS; i++) cc += sv[i] <= mid ? 1u : 0u;
            c[t] = warp_sum(cc);
        }
        if (lane == 0) {
#pragma unroll
            for (int t = 0; t < 6; t++) s_cnt[t][wid] = c[t];
        }
        __syncthreads();
        if (tid < 6) {
            uint32_t tot = 0;
            for (int k = 0; k < IV_WARPS; k++) tot += s_cnt[tid][k];
            const uint32_t mid = (b_lo[tid] + b_hi[tid]) >> 1;
            if (tot > b_rank[tid]) b_hi[tid] = mid; else b_lo[tid] = mid + 1;
        }
        __syncthreads();
    }
    if (tid < 6) {
        uint32_t v = b_hi[tid];
        if (b_fix[tid] == 1) v = 0;
        if (b_fix[tid] == 2) v = 65535u;
        // even: T = tL (count of v < tL); odd: T = tU + 1 (count of v <= tU), 65536 = every pixel
        thr[fi * 6 + tid] = (tid & 1) ? v + 1u : v;
    }
}

template <int VPL, bool COLS>
__global__ void __launch_bounds__(IV_THREADS, COLS ? 2 : 3)
k_inv_stream(const StatsGeom g, const FrameRef* __restrict__ frames, const uint32_t* __restrict__ thr, InvPart* __restrict__ parts,
             uint32_t* __restrict__ rowsum_out, uint32_t* __restrict__ colpart, int wa) {
    extern __shared__ uint32_t s_col[];      // wa column accumulators of the CTA (COLS)
    __shared__ uint32_t s_red[IV_WARPS][8];
    __shared__ unsigned long long s_tot[IV_WARPS];
    const int fi = blockIdx.y, part = blockIdx.x;
    const FrameRef fr = frames[fi];
    const uint16_t* __restrict__ f = fr.origin;
    const int pitch = fr.pitch;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const bool aligned = (pitch % 8) == 0;
    const int mis = aligned ? (int)((reinterpret_cast<uintptr_t>(f) >> 1) & 7) : 0;
    if (COLS) { for (int i = tid; i < wa; i += IV_THREADS) s_col[i] = 0; }
    uint32_t T2[6];
#pragma unroll
    for (int t = 0; t < 6; t++) { const uint32_t T = min(thr[fi * 6 + t], 65535u); T2[t] = T | (T << 16); }
    // validity of the lane's vectors is the same for every row: masks of the pixels inside the view
    uint32_t vmask[VPL][4];
    bool anyv[VPL];
#pragma unroll
    for (int k = 0; k < VPL; k++) {
        const int col_first = (lane + 32 * k) * 8 - mis;
        anyv[k] = false;
#pragma unroll
        for (int h2 = 0; h2 < 4; h2++) {
            uint32_t m = 0;
            if (col_first + 2 * h2 >= 0 && col_first + 2 * h2 < g.W) m |= 0xffffu;
            if (col_first + 2 * h2 + 1 >= 0 && col_first + 2 * h2 + 1 < g.W) m |= 0xffff0000u;
            vmask[k][h2] = m;
            anyv[k] = anyv[k] || m != 0;
        }
    }
    const int rp = (g.H + IV_PARTS - 1) / IV_PARTS;
    const int r0 = part * rp, r1 = min(g.H, r0 + rp);
    uint32_t cnt[6] = {0, 0, 0, 0, 0, 0};
    uint32_t mn2 = 0xffffffffu, mx2 = 0;
    unsigned long long total = 0;
    uint32_t csum[COLS ? VPL : 1][8];
    if (COLS) {
#pragma unroll
        for (int k = 0; k < VPL; k++)
#pragma unroll
            for (int e = 0; e < 8; e++) csum[k][e] = 0;
    }
    for (int r = r0 + wid; r < r1; r += IV_WARPS) {
        const uint16_t* rowp = f + (size_t)r * pitch;
        uint4 q[VPL];
#pragma unroll
        for (int k = 0; k < VPL; k++) {
            q[k] = make_uint4(0, 0, 0, 0);
            if (anyv[k]) {
                const int col_first = (lane + 32 * k) * 8 - mis;
                if (aligned) q[k] = ldg_stream16(rowp + col_first);
                else {
                    uint32_t w4[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int e = 0; e < 8; e++)
                        if ((vmask[k][e >> 1] >> ((e & 1) * 16)) & 1u) w4[e >> 1] |= (uint32_t)__ldg(rowp + col_first + e) << ((e & 1) * 16);
                    q[k] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                }
            }
        }
        uint32_t rs = 0;
#pragma unroll
        for (int k = 0; k < VPL; k++) {
            if (!anyv[k]) continue;
            const uint32_t w4[4] = {q[k].x, q[k].y, q[k].z, q[k].w};
#pragma unroll
            for (int h2 = 0; h2 < 4; h2++) {
                const uint32_t lo = w4[h2] & vmask[k][h2];         // outside the view: 0     (maximum, sums)
                const uint32_t hi = w4[h2] | ~vmask[k][h2];        // outside the view: 65535 (minimum, counts: never < T)
                mn2 = __vminu2(mn2, hi);
                mx2 = __vmaxu2(mx2, lo);
                rs = __dp2a_lo(lo, 0x0101u, rs);
#pragma unroll
                for (int t = 0; t < 6; t++) cnt[t] = __dp2a_lo(__vminu2(__vmaxu2(hi, T2[t]) - hi, 0x00010001u), 0x0101u, cnt[t]);
                if (COLS) {
                    csum[k][2 * h2] = __dp2a_lo(lo, 0x0001u, csum[k][2 * h2]);
                    csum[k][2 * h2 + 1] = __dp2a_lo(lo, 0x0100u, csum[k][2 * h2 + 1]);
                }
            }
        }
        rs = warp_sum(rs);
        total += rs;
        if (lane == 0 && rowsum_out) rowsum_out[(size_t)fi * g.H + r] = rs;
    }
    if (COLS) {
#pragma unroll
        for (int k = 0; k < VPL; k++)
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const int ac = (lane + 32 * k) * 8 + e;
                if (ac < wa && csum[k][e]) atomicAdd(&s_col[ac], csum[k][e]);
            }
    }
    uint32_t mn = min(mn2 & 0xffffu, mn2 >> 16), mx = max(mx2 & 0xffffu, mx2 >> 16);
    mn = warp_min(mn);
    mx = warp_max(mx);
#pragma unroll
    for (int t = 0; t < 6; t++) cnt[t] = warp_sum(cnt[t]);
    if (lane == 0) {
#pragma unroll
        for (int t = 0; t < 6; t++) s_red[wid][t] = cnt[t];
        s_red[wid][6] = mn;
        s_red[wid][7] = mx;
        s_tot[wid] = total;          // every lane holds the warp's row sums
    }
    __syncthreads();
    if (COLS && colpart) for (int i = tid; i < wa; i += IV_THREADS) colpart[((size_t)fi * IV_PARTS + part) * wa + i] = s_col[i];
    if (tid == 0) {
        InvPart o;
        for (int t = 0; t < 6; t++) o.cnt[t] = 0;
        o.mn = 0xffffu; o.mx = 0; o.total = 0;
        for (int k = 0; k < IV_WARPS; k++) {
            for (int t = 0; t < 6; t++) o.cnt[t] += s_red[k][t];
            o.mn = min(o.mn, s_red[k][6]);
            o.mx = max(o.mx, s_red[k][7]);
            o.total += s_tot[k];
        }
        parts[(size_t)fi * IV_PARTS + part] = o;
    }
}

__global__ void __launch_bounds__(256)
k_inv_finish(const StatsGeom g, const FrameRef* __restrict__ frames, const uint32_t* __restrict__ thr, const InvPart* __restrict__ parts,
             const uint32_t* __restrict__ colpart, int wa, FrameStats* __restrict__ stats, uint32_t* __restrict__ colsum_out,
             int* __restrict__ fail_list, int* __restrict__ fail_count) {
    const int fi = blockIdx.x, tid = threadIdx.x;
    const FrameRef fr = frames[fi];
    if (colsum_out && colpart) {
        const bool aligned = (fr.pitch % 8) == 0;
        const int mis = aligned ? (int)((reinterpret_cast<uintptr_t>(fr.origin) >> 1) & 7) : 0;
        for (int x = tid; x < g.W; x += 256) {
            uint32_t sum = 0;
            for (int p = 0; p < IV_PARTS; p++) sum += colpart[((size_t)fi * IV_PARTS + p) * wa + x + mis];
            colsum_out[(size_t)fi * g.W + x] = sum;
        }
    }
    if (tid != 0) return;
    uint32_t cnt[6] = {0, 0, 0, 0, 0, 0}, mn = 0xffffu, mx = 0;
    unsigned long long total = 0;
    for (int p = 0; p < IV_PARTS; p++) {
        const InvPart& o = parts[(size_t)fi * IV_PARTS + p];
        for (int t = 0; t < 6; t++) cnt[t] += o.cnt[t];
        mn = min(mn, o.mn);
        mx = max(mx, o.mx);
        total += o.total;
    }
    const uint32_t npix = (uint32_t)g.H * (uint32_t)g.W;
    bool ok = true;
    double L[3], U[3];
    for (int q = 0; q < 3; q++) {
        const uint32_t TL = thr[fi * 6 + 2 * q], TU = thr[fi * 6 + 2 * q + 1];
        const uint32_t cL = cnt[2 * q], cU = TU >= 65536u ? npix : cnt[2 * q + 1];
        // #(v < TL) <= rank_prev: the order statistic at rank_prev is >= TL; #(v < TU) >= rank_next + 1: the one at rank_next is < TU
        ok = ok && cL <= g.ranks[2 * q] && cU >= g.ranks[2 * q + 1] + 1u;
        L[q] = (double)TL;
        U[q] = (double)TU - 1.0;
    }
    // |p_mid - p_low| = p_mid - p_low, |p_mid - p_high| = p_high - p_mid (percentiles are monotone in q)
    const double a_lo = fmax(0.0, L[1] - U[0]), a_hi = fmax(0.0, U[1] - L[0]);
    const double b_lo = fmax(0.0, L[2] - U[1]), b_hi = fmax(0.0, U[2] - L[1]);
    int code = 0;
    if (ok && a_lo > b_hi) code = 3;            // certainly inverted
    else if (ok && a_hi < b_lo) code = 2;       // certainly not inverted
    FrameStats& o = stats[fi];
    o.mn = mn;
    o.mx = mx;
    o.npix = npix;
    o.sum = total;
    o.corner_sum = 0;
    o.overflow = (uint32_t)code;
    for (int k = 0; k < STATS_MAX_RANKS; k++) o.ostat[k] = 0;
    if (code == 0) fail_list[atomicAdd(fail_count, 1)] = fi;
}

__global__ void k_inv_gather_refs(const FrameRef* __restrict__ frames, const int* __restrict__ list, int m, FrameRef* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[i] = frames[list[i]];
}

__global__ void k_inv_scatter_ostat(const FrameStats* __restrict__ src, const int* __restrict__ list, int m, FrameStats* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    FrameStats& d = dst[list[i]];
    for (int k = 0; k < STATS_MAX_RANKS; k++) d.ostat[k] = src[i].ostat[k];
    d.overflow = 0;
}

template <int VPL>
static void launch_inv_stream(cudaStream_t st, bool cols, const StatsGeom& g, const FrameRef* refs, int n, const uint32_t* thr, InvPart* parts,
                              uint32_t* rowsum, uint32_t* colpart, int wa) {
    if (cols) k_inv_stream<VPL, true><<<dim3(IV_PARTS, n), IV_THREADS, sizeof(uint32_t) * wa, st>>>(g, refs, thr, parts, rowsum, colpart, wa);
    else k_inv_stream<VPL, false><<<dim3(IV_PARTS, n), IV_THREADS, 0, st>>>(g, refs, thr, parts, rowsum, nullptr, wa);
}

// g.ranks = (prev, next) of the low, middle and high percentile; box must be 0.  Returns with d_stats complete: overflow >= 2 carries the
// certified decision (2 + inverted, ostat unused), overflow == 0 exact ostat from the histogram path.  One host round trip (count of the
// uncertified frames).
int launch_frame_stats_inversion(epid_ctx* ctx, cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames, int n, FrameStats* d_stats,
                                 uint32_t* d_rowsum, uint32_t* d_colsum) {
    if (ctx->stats_exact || g.nranks != 6 || g.box > 0 || g.W > 2040 || g.H < IV_SAMPLE_ROWS || g.W < 8)
        return launch_frame_stats(ctx, stream, g, d_frames, n, d_stats, d_rowsum, d_colsum);
    const int nvec = (g.W + 7 + 7) / 8;
    const int vpl = (nvec + 31) / 32;
    const int wa = vpl * 32 * 8;
    size_t o = 0;
    auto sz = [&](size_t b) { const size_t r = o; o += (b + 255) / 256 * 256; return r; };
    const size_t o_thr = sz(sizeof(uint32_t) * 6 * (size_t)n), o_parts = sz(sizeof(InvPart) * (size_t)n * IV_PARTS);
    const size_t o_list = sz(sizeof(int) * ((size_t)n + 1)), o_refs = sz(sizeof(FrameRef) * (size_t)n), o_tmp = sz(sizeof(FrameStats) * (size_t)n);
    const size_t o_col = sz(d_colsum ? sizeof(uint32_t) * (size_t)n * IV_PARTS * wa : 0);
    if (ctx->inv_bytes < o) {
        if (ctx->inv_scratch) { EPID_CUDA(cudaStreamSynchronize(stream)); EPID_CUDA(cudaFree(ctx->inv_scratch)); ctx->inv_scratch = nullptr; ctx->inv_bytes = 0; }
        cudaError_t e = cudaMalloc(&ctx->inv_scratch, o);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", o, cudaGetErrorString(e)); return EPID_ERR_NOMEM; }
        ctx->inv_bytes = o;
    }
    char* base = (char*)ctx->inv_scratch;
    uint32_t* thr = (uint32_t*)(base + o_thr);
    InvPart* parts = (InvPart*)(base + o_parts);
    int* list = (int*)(base + o_list);       // [0] = count, then the frame indices
    FrameRef* refs2 = (FrameRef*)(base + o_refs);
    FrameStats* tmp = (FrameStats*)(base + o_tmp);
    uint32_t* colpart = d_colsum ? (uint32_t*)(base + o_col) : nullptr;
    EPID_CUDA(cudaMemsetAsync(list, 0, sizeof(int), stream));
    k_inv_pilot<<<n, IV_THREADS, 0, stream>>>(g, d_frames, thr);
    const bool cols = d_colsum != nullptr;
    if (vpl <= 4) launch_inv_stream<4>(stream, cols, g, d_frames, n, thr, parts, d_rowsum, colpart, wa);
    else if (vpl <= 6) launch_inv_stream<6>(stream, cols, g, d_frames, n, thr, parts, d_rowsum, colpart, wa);
    else launch_inv_stream<8>(stream, cols, g, d_frames, n, thr, parts, d_rowsum, colpart, wa);
    k_inv_finish<<<n, 256, 0, stream>>>(g, d_frames, thr, parts, colpart, wa, d_stats, d_colsum, list + 1, list);
    ctx->launches += 3;
    EPID_CUDA(cudaGetLastError());
    int m = 0;
    EPID_CUDA(cudaMemcpyAsync(&m, list, sizeof(int), cudaMemcpyDeviceToHost, stream));
    EPID_CUDA(cudaStreamSynchronize(stream));
    ctx->stats_uncertified += m;
    if (m > 0) {       // exact order statistics for the frames whose decision could not be certified
        k_inv_gather_refs<<<(m + 127) / 128, 128, 0, stream>>>(d_frames, list + 1, m, refs2);
        int rc = launch_frame_stats(ctx, stream, g, refs2, m, tmp, nullptr, nullptr);
        if (rc != EPID_OK) return rc;
        k_inv_scatter_ostat<<<(m + 127) / 128, 128, 0, stream>>>(tmp, list + 1, m, d_stats);
        ctx->launches += 2;
        EPID_CUDA(cudaGetLastError());
    }
    return EPID_OK;
}

static size_t stats_smem_bytes(const StatsGeom& g) {
    return sizeof(uint32_t) * (size_t)(HIST_WORDS + STATS_THREADS * 8 + g.H + 40 + 8 + 3 * STATS_MAX_RANKS);
}

int launch_frame_stats(epid_ctx* ctx, cudaStream_t stream, const StatsGeom& g, const FrameRef* d_frames,
                       int n, FrameStats* d_stats, uint32_t* d_rowsum, uint32_t* d_colsum) {
    // multi-CTA histogram path for every view it covers
    if (g.W <= 2040 && g.nranks <= STATS_MAX_RANKS)
        return launch_frame_stats_v2(ctx, stream, g, d_frames, n, d_stats, d_rowsum, d_colsum);
    const size_t smem = stats_smem_bytes(g);
    EPID_SMEM_OPT_IN(ctx, k_frame_stats<0>, 220 * 1024);
    EPID_SMEM_OPT_IN(ctx, k_frame_stats<1>, 220 * 1024);
    const int grid = n < ctx->sm_count ? n : ctx->sm_count;
    k_frame_stats<0><<<grid, STATS_THREADS, smem, stream>>>(g, d_frames, n, d_stats, d_rowsum, d_colsum);
    // exact fallback for frames whose packed counters overflowed (CTAs of other frames exit at once)
    k_frame_stats<1><<<grid, STATS_THREADS, smem, stream>>>(g, d_frames, n, d_stats, d_rowsum, d_colsum);
    ctx->launches += 2;
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

}  // namespace epid
