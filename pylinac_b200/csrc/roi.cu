// Region statistics on device-resident frames.
//
//   epid_roi_stats          RectangleROI.pixels_flat -> mean / std / min / max (core/roi.py:533-706): the pixels of a (possibly
//                           rotated) rectangle given by its four corners, selected like skimage.draw.polygon does -- integer pixel
//                           coordinates inside the polygon or ON its boundary (skimage's point_in_polygon returns non-zero for
//                           edge and vertex hits), clipped to the image.  skimage is not available in the build container: the
//                           rule is restated from its documentation / source as recalled (parity unpinned at that boundary); for
//                           axis-aligned rectangles with integer corners it reduces to a plain slice.
//   epid_weighted_centroid  WeightedCentroid.calculate (metrics/image.py:959-983): sum(idx * a) / sum(a) along both axes.
//   epid_disk_roi_stats     DiskROI median / mean / std / min / max and LowContrastDiskROI.percentile (core/roi.py:103-138, 406-408)
//                           of many disks on many frames: moments plus an exact radix select of the order statistics.
//   epid_disk_roi_pixels    DiskROI.circle_mask / masked_array pixel gathering (core/roi.py:134-150).
//
// One CTA per (frame, ROI).  Integer dtypes accumulate exact 64-bit sums (count, sum, sum of squares, index-weighted sums); float
// dtypes accumulate in fp64.  std = sqrt(mean(|x - mean|^2)) as numpy defines it, evaluated from the exact moments for integers.
#include <algorithm>
#include <cmath>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "roi.cuh"

namespace epid {

constexpr int ROI_THREADS = 256;

template <typename T> struct RoiAcc { using type = double; };
template <> struct RoiAcc<uint8_t> { using type = unsigned long long; };
template <> struct RoiAcc<uint16_t> { using type = unsigned long long; };

struct RoiOut { double count, sum, sumsq, mn, mx, varnum; };   // varnum: exact N * S2 - S1^2 for 8 / 16-bit pixels, else -1

template <typename T>
__global__ void __launch_bounds__(ROI_THREADS)
k_roi_stats(const T* __restrict__ data, int H, int W, int nroi, const double* __restrict__ verts, RoiOut* __restrict__ out) {
    using A = typename RoiAcc<T>::type;
    const int fi = blockIdx.y, ri = blockIdx.x;
    const T* f = data + (size_t)fi * H * W;
    const double* v = verts + (size_t)ri * 8;          // (x, y) x 4
    const double vx[4] = {v[0], v[2], v[4], v[6]}, vy[4] = {v[1], v[3], v[5], v[7]};
    const double xmin = fmin(fmin(vx[0], vx[1]), fmin(vx[2], vx[3])), xmax = fmax(fmax(vx[0], vx[1]), fmax(vx[2], vx[3]));
    const double ymin = fmin(fmin(vy[0], vy[1]), fmin(vy[2], vy[3])), ymax = fmax(fmax(vy[0], vy[1]), fmax(vy[2], vy[3]));
    // skimage.draw._polygon: minr = int(max(0, r.min())), maxr = int(ceil(r.max())), clipped to shape - 1
    const int r0 = (int)fmax(0.0, ymin), r1 = min((int)ceil(ymax), H - 1);
    const int c0 = (int)fmax(0.0, xmin), c1 = min((int)ceil(xmax), W - 1);
    const int bh = r1 - r0 + 1, bw = c1 - c0 + 1;
    A s1 = 0, s2 = 0;
    unsigned long long cnt = 0;
    double mn = INFINITY, mx = -INFINITY;
    if (bh > 0 && bw > 0) {
        for (int i = threadIdx.x; i < bh * bw; i += ROI_THREADS) {
            const int r = r0 + i / bw, c = c0 + i % bw;
            if (!point_in_quad(vx, vy, (double)c, (double)r)) continue;
            const T pv = f[(size_t)r * W + c];
            const A a = (A)pv;
            s1 += a;
            s2 += a * a;
            cnt++;
            mn = fmin(mn, (double)pv);
            mx = fmax(mx, (double)pv);
        }
    }
    __shared__ A sh1[ROI_THREADS], sh2[ROI_THREADS];
    __shared__ unsigned long long shc[ROI_THREADS];
    __shared__ double shmn[ROI_THREADS], shmx[ROI_THREADS];
    sh1[threadIdx.x] = s1; sh2[threadIdx.x] = s2; shc[threadIdx.x] = cnt; shmn[threadIdx.x] = mn; shmx[threadIdx.x] = mx;
    __syncthreads();
    for (int s = ROI_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            sh1[threadIdx.x] += sh1[threadIdx.x + s];
            sh2[threadIdx.x] += sh2[threadIdx.x + s];
            shc[threadIdx.x] += shc[threadIdx.x + s];
            shmn[threadIdx.x] = fmin(shmn[threadIdx.x], shmn[threadIdx.x + s]);
            shmx[threadIdx.x] = fmax(shmx[threadIdx.x], shmx[threadIdx.x + s]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        RoiOut o;
        o.count = (double)shc[0];
        o.sum = (double)sh1[0];
        o.sumsq = (double)sh2[0];
        o.mn = shmn[0];
        o.mx = shmx[0];
        o.varnum = -1.0;
        if (!std::is_floating_point<A>::value && shc[0] > 0) {
            // exact population variance numerator N * S2 - S1^2 in 128-bit integer arithmetic -> fp64 once
            const unsigned __int128 n = shc[0];
            const unsigned __int128 num = n * (unsigned __int128)(unsigned long long)sh2[0] -
                                          (unsigned __int128)(unsigned long long)sh1[0] * (unsigned long long)sh1[0];
            o.varnum = (double)num;
        }
        out[(size_t)fi * nroi + ri] = o;
    }
}

template <typename T>
static int do_roi(epid_ctx* ctx, const epid_batch* b, int nroi, const double* d_verts, RoiOut* d_out) {
    k_roi_stats<T><<<dim3(nroi, b->n), ROI_THREADS, 0, ctx->stream>>>((const T*)b->dptr, b->h, b->w, nroi, d_verts, d_out);
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

// ---------------------------------------------------------------------------------------- weighted centroid
template <typename T>
__global__ void __launch_bounds__(ROI_THREADS)
k_weighted_centroid(const T* __restrict__ data, int H, int W, double* __restrict__ part) {
    // grid (blocks, n): per-block partial sums of a, x * a, y * a (exact for integer pixels), combined on the host side of the C-ABI
    using A = typename RoiAcc<T>::type;
    const int fi = blockIdx.y;
    const T* f = data + (size_t)fi * H * W;
    A s = 0, sx = 0, sy = 0;
    const size_t per = (size_t)H * W;
    for (size_t i = (size_t)blockIdx.x * ROI_THREADS + threadIdx.x; i < per; i += (size_t)gridDim.x * ROI_THREADS) {
        const A a = (A)f[i];
        const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
        s += a;
        sx += a * (A)x;
        sy += a * (A)y;
    }
    __shared__ A sh[3][ROI_THREADS];
    sh[0][threadIdx.x] = s; sh[1][threadIdx.x] = sx; sh[2][threadIdx.x] = sy;
    __syncthreads();
    for (int k = ROI_THREADS / 2; k > 0; k >>= 1) {
        if (threadIdx.x < k) for (int j = 0; j < 3; j++) sh[j][threadIdx.x] += sh[j][threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x < 3) {
        // integer sums travel as two 32-bit halves in doubles (exact), float sums as they are
        double* o = part + ((size_t)fi * gridDim.x + blockIdx.x) * 6;
        const A v = sh[threadIdx.x][0];
        if (std::is_floating_point<A>::value) { o[2 * threadIdx.x] = (double)v; o[2 * threadIdx.x + 1] = 0.0; }
        else {
            const unsigned long long u = (unsigned long long)v;
            o[2 * threadIdx.x] = (double)(u >> 32);
            o[2 * threadIdx.x + 1] = (double)(u & 0xffffffffull);
        }
    }
}

constexpr int WC_BLOCKS = 64;
template <typename T>
static int do_wc(epid_ctx* ctx, const epid_batch* b, double* d_part) {
    k_weighted_centroid<T><<<dim3(WC_BLOCKS, b->n), ROI_THREADS, 0, ctx->stream>>>((const T*)b->dptr, b->h, b->w, d_part);
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    return EPID_OK;
}

// ---------------------------------------------------------------------------------------- disks
// DiskROI.circle_mask / masked_array (core/roi.py:134-150) select their pixels with skimage.draw.disk(center=(y, x), radius[, shape])
// = ellipse(y, x, r, r, shape, rotation=0): bounding box ceil(center - r) .. floor(center + r) (clipped to the image only when shape
// is given), shifted centre = center - box corner, and a box pixel (i, j) is in the disk when ((i - r_org) / r)**2 + ((j - c_org) / r)**2
// < 1, evaluated in fp64 in that order (the build disables FMA contraction).  Without shape, indices in [-dim, -1] wrap to the far edge
// (numpy fancy indexing) and any index outside [-dim, dim - 1] is numpy's IndexError.
struct DiskGeom { int r0, c0, bh, bw; double r_org, c_org, rad; };

static DiskGeom disk_geom(double cy, double cx, double rad, bool clip, int H, int W) {
    const double ext = fabs(rad * 1.0) + rad * 0.0;        // skimage's rotated radius at rotation 0
    int ur = (int)ceil(cy - ext), uc = (int)ceil(cx - ext);
    int lr = (int)floor(cy + ext), lc = (int)floor(cx + ext);
    if (clip) { ur = std::max(ur, 0); uc = std::max(uc, 0); lr = std::min(lr, H - 1); lc = std::min(lc, W - 1); }
    DiskGeom g;
    g.r0 = ur; g.c0 = uc;
    g.bh = std::max(lr - ur + 1, 0); g.bw = std::max(lc - uc + 1, 0);
    g.r_org = cy - (double)ur; g.c_org = cx - (double)uc;
    g.rad = rad;
    return g;
}

__device__ __forceinline__ bool disk_inside(const DiskGeom& g, int i, int j) {
    const double tr = ((double)i - g.r_org) / g.rad, tc = ((double)j - g.c_org) / g.rad;
    return tr * tr + tc * tc < 1.0;
}

// Order-preserving keys for the radix select: 16-bit for 8 / 16-bit pixels, 64-bit otherwise (floats through fp64, -0 folded onto +0
// since numpy orders them as equal; NaN never reaches a selection, see k_disk_roi_stats).
template <typename T> struct DiskKey {
    using K = unsigned long long;
    __host__ __device__ static K of(T v) {
        if (std::is_floating_point<T>::value) {
            double d = (double)v;
            if (d == 0.0) d = 0.0;
            unsigned long long u;
            memcpy(&u, &d, 8);
            return (u >> 63) ? ~u : (u | (1ull << 63));
        }
        return (unsigned long long)(long long)v ^ (1ull << 63);
    }
    __host__ __device__ static T value(K k) {
        if (std::is_floating_point<T>::value) {
            const unsigned long long u = (k >> 63) ? (k & ~(1ull << 63)) : ~k;
            double d;
            memcpy(&d, &u, 8);
            return (T)d;
        }
        return (T)(long long)(k ^ (1ull << 63));
    }
};
template <typename T> struct DiskKey16 {
    using K = unsigned short;
    static constexpr unsigned short flip = std::is_signed<T>::value ? 0x8000 : 0;
    __host__ __device__ static K of(T v) { return (unsigned short)((unsigned short)v ^ flip); }
    __host__ __device__ static T value(K k) { return (T)(unsigned short)(k ^ flip); }
};
template <> struct DiskKey<uint8_t> : DiskKey16<uint8_t> {};
template <> struct DiskKey<uint16_t> : DiskKey16<uint16_t> {};
template <> struct DiskKey<int16_t> : DiskKey16<int16_t> {};

// np.percentile(..., method="linear") index arithmetic for n values: quantile q = p / 100 in the frame's float type (float32 frames keep
// float32, numpy divides by a.dtype.type(100)), virtual index (n - 1) * q, neighbours floor / floor + 1 (both -> n - 1 at or above
// the last index; gamma is then taken against -1, as _get_gamma does).
struct PctIdx { long long lo, hi; double gamma; };
template <bool F32>
__host__ __device__ inline PctIdx pct_index(long long n, double p) {
    PctIdx r;
    if (F32) {
        const float q = (float)p / 100.0f, v = (float)(n - 1) * q;
        long long lo = (long long)floorf(v);
        if (v >= (float)(n - 1)) lo = -1;
        r.gamma = (double)(float)((double)v - (double)lo);
        r.lo = r.hi = lo < 0 ? n - 1 : lo;
        if (lo >= 0) r.hi = lo + 1;
    } else {
        const double q = p / 100.0, v = (double)(n - 1) * q;
        long long lo = (long long)floor(v);
        if (v >= (double)(n - 1)) lo = -1;
        r.gamma = v - (double)lo;
        r.lo = r.hi = lo < 0 ? n - 1 : lo;
        if (lo >= 0) r.hi = lo + 1;
    }
    return r;
}

constexpr int DISK_THREADS = 256;
constexpr size_t DISK_STAGE_BYTES = 64 * 1024;     // keys of one disk staged in shared memory up to this size; larger disks re-read L2
struct DiskOut { double count, sum, m2, mn, mx; int flags, nan; };   // m2: exact N * S2 - S1^2 for 8 / 16-bit pixels, else sum (x - mean)^2

// dynamic shared memory: hist [nrank][256] u32 | want [nrank] u32 | pre [nrank] K | stage [cap] K
template <typename K>
__host__ __device__ inline size_t disk_smem_pre(int nrank) { return ((size_t)nrank * 257 * 4 + 7) / 8 * 8; }
template <typename K>
__host__ __device__ inline size_t disk_smem_stage(int nrank) { return (disk_smem_pre<K>(nrank) + (size_t)nrank * sizeof(K) + 7) / 8 * 8; }

template <typename T, typename K, typename F>
__device__ __forceinline__ void disk_for_each(const T* f, int H, int W, const DiskGeom& g, const K* stage, int staged, F fn) {
    if (stage) {
        for (int k = threadIdx.x; k < staged; k += DISK_THREADS) fn(stage[k]);
        return;
    }
    const int nb = g.bh * g.bw;
    for (int p = threadIdx.x; p < nb; p += DISK_THREADS) {
        const int i = p / g.bw, j = p - i * g.bw;
        if (!disk_inside(g, i, j)) continue;
        int row = g.r0 + i, col = g.c0 + j;
        if (row < 0) row += H;
        if (col < 0) col += W;
        fn(DiskKey<T>::of(f[(size_t)row * W + col]));
    }
}

// One CTA per (frame, disk): exact moments as k_roi_stats (RoiAcc), then a radix select of nrank order statistics on the disk's keys,
// 8 bits per pass, all ranks at once; the keys are staged in shared memory when the disk has at most `cap` pixels, otherwise every
// pass re-evaluates the disk and re-reads its pixels (L2).  Ranks: 0 / 1 the median pair, 2 + 2k / 3 + 2k percentile k's neighbours.
template <typename T>
__global__ void __launch_bounds__(DISK_THREADS)
k_disk_roi_stats(const T* __restrict__ data, int H, int W, int ndisk, const DiskGeom* __restrict__ geom, int npct,
                 const double* __restrict__ pcts, int cap, DiskOut* __restrict__ out, unsigned long long* __restrict__ ost) {
    using A = typename RoiAcc<T>::type;
    using K = typename DiskKey<T>::K;
    const int fi = blockIdx.y, di = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nrank = 2 + 2 * npct;
    const T* f = data + (size_t)fi * H * W;
    const DiskGeom g = geom[di];
    extern __shared__ __align__(8) unsigned char dsm[];
    unsigned* hist = (unsigned*)dsm;
    unsigned* want = hist + nrank * 256;
    K* pre = (K*)(dsm + disk_smem_pre<K>(nrank));
    K* stage = (K*)(dsm + disk_smem_stage<K>(nrank));
    __shared__ unsigned s_staged;
    __shared__ A r1[DISK_THREADS / 32], r2[DISK_THREADS / 32];
    __shared__ double rmn[DISK_THREADS / 32], rmx[DISK_THREADS / 32];
    __shared__ unsigned rc[DISK_THREADS / 32], rnan[DISK_THREADS / 32], rfl[DISK_THREADS / 32];
    __shared__ double s_mean;
    if (tid == 0) s_staged = 0;
    __syncthreads();

    // pass 1: membership, range check, moments, staging (warp-aggregated slots)
    A s1 = 0, s2 = 0;
    unsigned cnt = 0, nan = 0, flags = 0;
    double mn = INFINITY, mx = -INFINITY;
    const int nb = g.bh * g.bw;
    for (int base = 0; base < nb; base += DISK_THREADS) {
        const int p = base + tid;
        bool sel = false;
        K key = 0;
        if (p < nb) {
            const int i = p / g.bw, j = p - i * g.bw;
            if (disk_inside(g, i, j)) {
                int row = g.r0 + i, col = g.c0 + j;
                if (row < -H || row >= H) flags |= 1;
                else if (col < -W || col >= W) flags |= 2;
                else {
                    if (row < 0) row += H;
                    if (col < 0) col += W;
                    const T pv = f[(size_t)row * W + col];
                    const A a = (A)pv;
                    s1 += a;
                    s2 += a * a;
                    cnt++;
                    if (pv != pv) nan++;
                    mn = fmin(mn, (double)pv);
                    mx = fmax(mx, (double)pv);
                    key = DiskKey<T>::of(pv);
                    sel = true;
                }
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        unsigned slot = 0;
        if (lane == 0 && bal) slot = atomicAdd(&s_staged, (unsigned)__popc(bal));
        slot = __shfl_sync(0xffffffffu, slot, 0) + __popc(bal & ((1u << lane) - 1));
        if (sel && slot < (unsigned)cap) stage[slot] = key;
    }
    s1 = warp_sum(s1); s2 = warp_sum(s2); cnt = warp_sum(cnt); nan = warp_sum(nan);
    mn = warp_min(mn); mx = warp_max(mx);
    flags = __reduce_or_sync(0xffffffffu, flags);
    if (lane == 0) { r1[warp] = s1; r2[warp] = s2; rc[warp] = cnt; rnan[warp] = nan; rmn[warp] = mn; rmx[warp] = mx; rfl[warp] = flags; }
    __syncthreads();
    s1 = 0; s2 = 0; cnt = 0; nan = 0; flags = 0; mn = INFINITY; mx = -INFINITY;
    for (int w = 0; w < DISK_THREADS / 32; w++) {
        s1 += r1[w]; s2 += r2[w]; cnt += rc[w]; nan += rnan[w]; flags |= rfl[w];
        mn = fmin(mn, rmn[w]); mx = fmax(mx, rmx[w]);
    }
    DiskOut* o = out + (size_t)fi * ndisk + di;
    if (tid == 0) {
        o->count = (double)cnt; o->sum = (double)s1; o->mn = mn; o->mx = mx; o->flags = (int)flags; o->nan = (int)nan;
        o->m2 = 0.0;
        if (!std::is_floating_point<A>::value && cnt > 0) {
            const unsigned __int128 n = cnt;
            o->m2 = (double)(n * (unsigned __int128)(unsigned long long)s2 - (unsigned __int128)(unsigned long long)s1 * (unsigned long long)s1);
        }
    }
    if (flags || cnt == 0 || nan) return;       // the caller raises, or every statistic is NaN / undefined
    const K* st = cnt <= (unsigned)cap ? stage : nullptr;

    if (std::is_floating_point<A>::value) {     // centred second moment in fp64 (np.std subtracts the mean first)
        if (tid == 0) s_mean = (double)s1 / (double)cnt;
        __syncthreads();
        const double m = s_mean;
        double c2 = 0.0;
        disk_for_each<T>(f, H, W, g, st, (int)cnt, [&](K k) { const double d = (double)DiskKey<T>::value(k) - m; c2 += d * d; });
        c2 = warp_sum(c2);
        if (lane == 0) rmn[warp] = c2;
        __syncthreads();
        if (tid == 0) { double t = 0.0; for (int w = 0; w < DISK_THREADS / 32; w++) t += rmn[w]; o->m2 = t; }
    }

    // radix select of all ranks at once
    if (tid < nrank) {
        const long long n = cnt;
        long long r;
        if (tid < 2) r = tid == 0 ? (n - 1) / 2 : n / 2;
        else {
            const PctIdx q = pct_index<std::is_same<T, float>::value>(n, pcts[(tid - 2) >> 1]);
            r = (tid & 1) ? q.hi : q.lo;
        }
        want[tid] = (unsigned)r;
        pre[tid] = 0;
    }
    for (int shift = 8 * (int)sizeof(K) - 8; shift >= 0; shift -= 8) {
        for (int k = tid; k < nrank * 256; k += DISK_THREADS) hist[k] = 0;
        __syncthreads();
        const K hm = shift + 8 >= 8 * (int)sizeof(K) ? (K)0 : (K)(~(unsigned long long)0 << (shift + 8));
        disk_for_each<T>(f, H, W, g, st, (int)cnt, [&](K k) {
            const unsigned d = (unsigned)(k >> shift) & 255u;
            for (int r = 0; r < nrank; r++)
                if (((k ^ pre[r]) & hm) == 0) atomicAdd(&hist[r * 256 + d], 1u);
        });
        __syncthreads();
        if (tid < nrank) {
            const unsigned* h = hist + tid * 256;
            unsigned w = want[tid], c = 0;
            int d = 0;
            for (; d < 255; d++) {
                if (c + h[d] > w) break;
                c += h[d];
            }
            want[tid] = w - c;
            pre[tid] = (K)(pre[tid] | ((K)d << shift));
        }
        __syncthreads();
    }
    if (tid < nrank) ost[((size_t)fi * ndisk + di) * nrank + tid] = (unsigned long long)pre[tid];
}

// numpy's arithmetic on the selected order statistics: np.median = np.mean of the middle value(s) (float32 frames average in float32,
// everything else in float64), np.percentile = _lerp(a, b, t) with its t >= 0.5 branch, b - a taken in the frame dtype.
template <typename T>
static double np_median(T a, T b, bool odd) {
    if (odd) return (double)a;
    if (std::is_same<T, float>::value) return (double)((float)(a + b) / 2.0f);
    return ((double)a + (double)b) / 2.0;
}
template <typename T>
static double np_lerp(T a, T b, double t) {
    if (std::is_same<T, float>::value) {
        const float fa = (float)a, fb = (float)b, ft = (float)t, d = fb - fa;
        float r = fa + d * ft;
        if (ft >= 0.5f) r = fb - d * (1.0f - ft);
        return (double)r;
    }
    const T d = (T)(b - a);
    double r = (double)a + (double)d * t;
    if (t >= 0.5) r = (double)b - (double)d * (1.0 - t);
    return r;
}

template <typename T>
static int do_disk_stats(epid_ctx* ctx, const epid_batch* b, int ndisk, const DiskGeom* hg, int npct, const double* pcts, double* count,
                         double* mean, double* std, double* mn, double* mx, double* median, double* pct) {
    using K = typename DiskKey<T>::K;
    constexpr bool F32 = std::is_same<T, float>::value;
    for (int k = 0; k < npct; k++) {       // np.percentile's range check, on q in the frame's float type
        const double q = F32 ? (double)((float)pcts[k] / 100.0f) : pcts[k] / 100.0;
        EPID_REQUIRE(q >= 0.0 && q <= 1.0, EPID_ERR_INVALID, "Percentiles must be in the range [0, 100]");
    }
    const int nrank = 2 + 2 * npct;
    long long maxbox = 0;
    for (int d = 0; d < ndisk; d++) maxbox = std::max(maxbox, (long long)hg[d].bh * hg[d].bw);
    const int cap = (int)std::min<long long>(maxbox, DISK_STAGE_BYTES / sizeof(K));
    const size_t smem = disk_smem_stage<K>(nrank) + (size_t)cap * sizeof(K);
    const size_t n = (size_t)b->n * ndisk;
    const size_t ng = sizeof(DiskGeom) * ndisk, np_ = sizeof(double) * std::max(npct, 1), no = sizeof(DiskOut) * n,
                 nk = sizeof(unsigned long long) * n * nrank;
    auto up = [](size_t v) { return (v + 255) / 256 * 256; };
    int rc = ensure_scratch(ctx, up(ng) + up(np_) + up(no) + nk);
    if (rc != EPID_OK) return rc;
    char* s = (char*)ctx->scratch;
    DiskGeom* d_geom = (DiskGeom*)s;
    double* d_pct = (double*)(s + up(ng));
    DiskOut* d_out = (DiskOut*)(s + up(ng) + up(np_));
    unsigned long long* d_ost = (unsigned long long*)(s + up(ng) + up(np_) + up(no));
    EPID_CUDA(cudaMemcpyAsync(d_geom, hg, ng, cudaMemcpyHostToDevice, ctx->stream));
    if (npct) EPID_CUDA(cudaMemcpyAsync(d_pct, pcts, sizeof(double) * npct, cudaMemcpyHostToDevice, ctx->stream));
    EPID_SMEM_OPT_IN(ctx, k_disk_roi_stats<T>, smem);
    k_disk_roi_stats<T><<<dim3(ndisk, b->n), DISK_THREADS, smem, ctx->stream>>>((const T*)b->dptr, b->h, b->w, ndisk, d_geom, npct,
                                                                                 d_pct, cap, d_out, d_ost);
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    std::vector<DiskOut> ho(n);
    std::vector<unsigned long long> hk(n * nrank);
    EPID_CUDA(cudaMemcpyAsync(ho.data(), d_out, no, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaMemcpyAsync(hk.data(), d_ost, nk, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; i++) {
        const DiskOut& o = ho[i];
        if (o.flags) {
            set_error("disk %d: index out of bounds for axis %d with size %d", (int)(i % ndisk), (o.flags & 1) ? 0 : 1,
                      (o.flags & 1) ? b->h : b->w);
            return EPID_ERR_INDEX;
        }
    }
    for (size_t i = 0; i < n; i++) {
        const DiskOut& o = ho[i];
        const long long cnt = (long long)o.count;
        const bool ok = cnt > 0 && o.nan == 0;       // NaN pixels make every numpy statistic NaN
        if (count) count[i] = o.count;
        if (mean) mean[i] = ok ? o.sum / o.count : NAN;
        if (std) std[i] = !ok ? NAN : std::is_floating_point<typename RoiAcc<T>::type>::value ? sqrt(o.m2 / o.count) : sqrt(o.m2) / o.count;
        if (mn) mn[i] = ok ? o.mn : NAN;
        if (mx) mx[i] = ok ? o.mx : NAN;
        const unsigned long long* k = &hk[i * nrank];
        if (median) median[i] = ok ? np_median<T>(DiskKey<T>::value((K)k[0]), DiskKey<T>::value((K)k[1]), cnt & 1) : NAN;
        for (int p = 0; pct && p < npct; p++) {
            double v = NAN;
            if (ok) {
                const PctIdx q = pct_index<F32>(cnt, pcts[p]);
                v = np_lerp<T>(DiskKey<T>::value((K)k[2 + 2 * p]), DiskKey<T>::value((K)k[3 + 2 * p]), q.gamma);
            }
            pct[i * npct + p] = v;
        }
    }
    return EPID_OK;
}

// One disk's pixels in np.nonzero (row-major box) order: values, and the raw (unwrapped) row / column indices skimage returns.
// meta[0] = count, meta[1] = out-of-range flags.  Values are written while the running count is below cap.
template <typename T>
__global__ void __launch_bounds__(DISK_THREADS)
k_disk_roi_pixels(const T* __restrict__ f, int H, int W, DiskGeom g, long long cap, T* __restrict__ vals, int* __restrict__ rows,
                  int* __restrict__ cols, long long* __restrict__ meta) {
    __shared__ unsigned wcnt[DISK_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = g.bh * g.bw;
    long long base = 0;
    unsigned flags = 0;
    for (int chunk = 0; chunk < nb; chunk += DISK_THREADS) {
        const int p = chunk + tid;
        int i = 0, j = 0;
        bool sel = false;
        if (p < nb) {
            i = p / g.bw;
            j = p - i * g.bw;
            sel = disk_inside(g, i, j);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        if (lane == 0) wcnt[warp] = __popc(bal);
        __syncthreads();
        unsigned before = 0, total = 0;
        for (int w = 0; w < DISK_THREADS / 32; w++) {
            before += w < warp ? wcnt[w] : 0;
            total += wcnt[w];
        }
        if (sel) {
            const long long idx = base + before + __popc(bal & ((1u << lane) - 1));
            int row = g.r0 + i, col = g.c0 + j;
            if (row < -H || row >= H) flags |= 1;
            else if (col < -W || col >= W) flags |= 2;
            else if (vals && idx < cap) {
                rows[idx] = row;
                cols[idx] = col;
                if (row < 0) row += H;
                if (col < 0) col += W;
                vals[idx] = f[(size_t)row * W + col];
            }
        }
        base += total;
        __syncthreads();
    }
    flags = __reduce_or_sync(0xffffffffu, flags);
    if (lane == 0) wcnt[warp] = flags;
    __syncthreads();
    if (tid == 0) {
        for (int w = 0; w < DISK_THREADS / 32; w++) flags |= wcnt[w];
        meta[0] = base;
        meta[1] = flags;
    }
}

template <typename T>
static int do_disk_pixels(epid_ctx* ctx, const epid_batch* b, int frame, const DiskGeom& g, long long cap, void* values, int32_t* rows,
                          int32_t* cols, long long* count) {
    const size_t nv = values ? sizeof(T) * cap : 0, ni = values ? sizeof(int) * cap : 0;
    auto up = [](size_t v) { return (v + 255) / 256 * 256; };
    int rc = ensure_scratch(ctx, 256 + up(nv) + 2 * up(ni));
    if (rc != EPID_OK) return rc;
    char* s = (char*)ctx->scratch;
    long long* d_meta = (long long*)s;
    T* d_vals = values ? (T*)(s + 256) : nullptr;
    int* d_rows = (int*)(s + 256 + up(nv));
    int* d_cols = (int*)(s + 256 + up(nv) + up(ni));
    const T* f = (const T*)b->dptr + (size_t)frame * b->h * b->w;
    k_disk_roi_pixels<T><<<1, DISK_THREADS, 0, ctx->stream>>>(f, b->h, b->w, g, cap, d_vals, d_rows, d_cols, d_meta);
    ctx->launches++;
    EPID_CUDA(cudaGetLastError());
    long long meta[2];
    EPID_CUDA(cudaMemcpyAsync(meta, d_meta, sizeof(meta), cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    if (meta[1]) {
        set_error("index out of bounds for axis %d with size %d", (meta[1] & 1) ? 0 : 1, (meta[1] & 1) ? b->h : b->w);
        return EPID_ERR_INDEX;
    }
    *count = meta[0];
    if (values) {
        EPID_REQUIRE(meta[0] <= cap, EPID_ERR_INVALID, "capacity %lld is below the disk's %lld pixels", cap, meta[0]);
        EPID_CUDA(cudaMemcpyAsync(values, d_vals, sizeof(T) * meta[0], cudaMemcpyDeviceToHost, ctx->stream));
        if (rows) EPID_CUDA(cudaMemcpyAsync(rows, d_rows, sizeof(int) * meta[0], cudaMemcpyDeviceToHost, ctx->stream));
        if (cols) EPID_CUDA(cudaMemcpyAsync(cols, d_cols, sizeof(int) * meta[0], cudaMemcpyDeviceToHost, ctx->stream));
        EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return EPID_OK;
}

// centre / radius sanity shared by both disk entry points: finite, and a bounding box that fits 32-bit pixel indices
static int disk_geom_checked(double cx, double cy, double rad, bool clip, int H, int W, DiskGeom* g) {
    EPID_REQUIRE(std::isfinite(cx) && std::isfinite(cy) && std::isfinite(rad), EPID_ERR_INVALID, "disk centre and radius must be finite");
    EPID_REQUIRE(fabs(cx) < 1e8 && fabs(cy) < 1e8 && fabs(rad) < 1e8, EPID_ERR_UNSUPPORTED, "disk outside the supported coordinate range");
    *g = disk_geom(cy, cx, rad, clip, H, W);
    EPID_REQUIRE((long long)g->bh * g->bw < (1ll << 31), EPID_ERR_UNSUPPORTED, "disk bounding box exceeds 2^31 pixels");
    return EPID_OK;
}

}  // namespace epid

using namespace epid;

#define EPID_DISPATCH_ROI(dt, FN, ...)                                              \
    switch (dt) {                                                                   \
        case EPID_U8: rc = FN<uint8_t>(__VA_ARGS__); break;                         \
        case EPID_U16: rc = FN<uint16_t>(__VA_ARGS__); break;                       \
        case EPID_I16: rc = FN<int16_t>(__VA_ARGS__); break;                        \
        case EPID_I32: rc = FN<int32_t>(__VA_ARGS__); break;                        \
        case EPID_I64: rc = FN<long long>(__VA_ARGS__); break;                      \
        case EPID_F32: rc = FN<float>(__VA_ARGS__); break;                          \
        case EPID_F64: rc = FN<double>(__VA_ARGS__); break;                         \
        default: set_error("unknown dtype %d", dt); rc = EPID_ERR_INVALID;          \
    }

extern "C" int32_t epid_roi_stats(epid_ctx* ctx, const epid_batch* b, int32_t nroi, const double* verts_xy, double* count, double* mean,
                                  double* std, double* mn, double* mx) {
    EPID_REQUIRE(ctx && b && verts_xy && nroi > 0 && nroi <= 4096, EPID_ERR_INVALID, "bad argument");
    EPID_CUDA(cudaSetDevice(ctx->device));
    const size_t nv = sizeof(double) * 8 * nroi, no = sizeof(RoiOut) * (size_t)nroi * b->n;
    int rc = ensure_scratch(ctx, nv + no + 512);
    if (rc != EPID_OK) return rc;
    double* d_verts = (double*)ctx->scratch;
    RoiOut* d_out = (RoiOut*)((char*)ctx->scratch + (nv + 255) / 256 * 256);
    EPID_CUDA(cudaMemcpyAsync(d_verts, verts_xy, nv, cudaMemcpyHostToDevice, ctx->stream));
    EPID_DISPATCH_ROI(b->dtype, do_roi, ctx, b, nroi, d_verts, d_out);
    if (rc != EPID_OK) return rc;
    std::vector<RoiOut> h((size_t)nroi * b->n);
    EPID_CUDA(cudaMemcpyAsync(h.data(), d_out, no, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < h.size(); i++) {
        const RoiOut& o = h[i];
        const double n = o.count;
        if (count) count[i] = n;
        const double m = n > 0 ? o.sum / n : NAN;
        if (mean) mean[i] = m;
        if (std) {
            if (!(n > 0)) std[i] = NAN;
            else if (o.varnum >= 0) std[i] = sqrt(o.varnum) / n;   // exact numerator
            else { const double var = o.sumsq / n - m * m; std[i] = var > 0 ? sqrt(var) : 0.0; }
        }
        if (mn) mn[i] = n > 0 ? o.mn : NAN;
        if (mx) mx[i] = n > 0 ? o.mx : NAN;
    }
    return EPID_OK;
}

extern "C" int32_t epid_disk_roi_stats(epid_ctx* ctx, const epid_batch* b, int32_t ndisk, const double* centers_xy, const double* radii,
                                       int32_t npct, const double* percentiles, double* count, double* mean, double* std, double* mn,
                                       double* mx, double* median, double* pct) {
    EPID_REQUIRE(ctx && b && centers_xy && radii && ndisk > 0 && ndisk <= 65535, EPID_ERR_INVALID, "bad argument");
    EPID_REQUIRE(npct >= 0 && npct <= EPID_DISK_MAX_PCT && (npct == 0 || percentiles), EPID_ERR_INVALID,
                 "at most %d percentiles per call", EPID_DISK_MAX_PCT);
    EPID_CUDA(cudaSetDevice(ctx->device));
    std::vector<DiskGeom> g(ndisk);
    for (int d = 0; d < ndisk; d++) {
        const int rc = disk_geom_checked(centers_xy[2 * d], centers_xy[2 * d + 1], radii[d], false, b->h, b->w, &g[d]);
        if (rc != EPID_OK) return rc;
    }
    int rc;
    EPID_DISPATCH_ROI(b->dtype, do_disk_stats, ctx, b, ndisk, g.data(), npct, percentiles, count, mean, std, mn, mx, median, pct);
    return rc;
}

extern "C" int32_t epid_disk_roi_pixels(epid_ctx* ctx, const epid_batch* b, int32_t frame, const double* center_xy, double radius,
                                        int32_t clip, int64_t capacity, void* values, int32_t* rows, int32_t* cols, int64_t* count) {
    EPID_REQUIRE(ctx && b && center_xy && count && capacity >= 0, EPID_ERR_INVALID, "bad argument");
    EPID_REQUIRE(frame >= 0 && frame < b->n, EPID_ERR_INVALID, "frame %d outside the batch of %d", frame, b->n);
    EPID_CUDA(cudaSetDevice(ctx->device));
    DiskGeom g;
    int rc = disk_geom_checked(center_xy[0], center_xy[1], radius, clip != 0, b->h, b->w, &g);
    if (rc != EPID_OK) return rc;
    long long n = 0;
    EPID_DISPATCH_ROI(b->dtype, do_disk_pixels, ctx, b, frame, g, (long long)capacity, values, rows, cols, &n);
    *count = n;
    return rc;
}

extern "C" int32_t epid_weighted_centroid(epid_ctx* ctx, const epid_batch* b, double* cx, double* cy, double* total) {
    EPID_REQUIRE(ctx && b && cx && cy, EPID_ERR_INVALID, "NULL argument");
    EPID_CUDA(cudaSetDevice(ctx->device));
    const size_t np = sizeof(double) * 6 * WC_BLOCKS * (size_t)b->n;
    int rc = ensure_scratch(ctx, np + 256);
    if (rc != EPID_OK) return rc;
    double* d_part = (double*)ctx->scratch;
    EPID_DISPATCH_ROI(b->dtype, do_wc, ctx, b, d_part);
    if (rc != EPID_OK) return rc;
    std::vector<double> h((size_t)6 * WC_BLOCKS * b->n);
    EPID_CUDA(cudaMemcpyAsync(h.data(), d_part, np, cudaMemcpyDeviceToHost, ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    const bool integral = b->dtype == EPID_U8 || b->dtype == EPID_U16;
    for (int fi = 0; fi < b->n; fi++) {
        if (integral) {      // exact 128-bit totals of the 64 block partials, one fp64 division at the end like numpy's
            unsigned __int128 t[3] = {0, 0, 0};
            for (int k = 0; k < WC_BLOCKS; k++) {
                const double* o = &h[((size_t)fi * WC_BLOCKS + k) * 6];
                for (int j = 0; j < 3; j++) t[j] += ((unsigned __int128)(unsigned long long)o[2 * j] << 32) + (unsigned long long)o[2 * j + 1];
            }
            const double s = (double)t[0];
            if (total) total[fi] = s;
            cx[fi] = (double)t[1] / s;
            cy[fi] = (double)t[2] / s;
        } else {
            double t[3] = {0, 0, 0};
            for (int k = 0; k < WC_BLOCKS; k++) for (int j = 0; j < 3; j++) t[j] += h[((size_t)fi * WC_BLOCKS + k) * 6 + 2 * j];
            if (total) total[fi] = t[0];
            cx[fi] = t[1] / t[0];
            cy[fi] = t[2] / t[0];
        }
    }
    return EPID_OK;
}
