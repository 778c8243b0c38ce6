// Element-wise image operators with the reference's dtype semantics (core/array_utils.py:64-102,
// core/image.py:785-815) and the public frame-statistics entry points.
#include <cmath>

#include "filters.cuh"
#include "stats.cuh"

namespace epid {

template <typename T> struct Wide { using type = T; };
template <> struct Wide<uint8_t> { using type = uint32_t; };
template <> struct Wide<uint16_t> { using type = uint32_t; };
template <> struct Wide<int16_t> { using type = int32_t; };

// ---------------------------------------------------------------------------------------- per-frame min / max
constexpr int MM_BLOCKS = 64, MM_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(MM_THREADS) k_minmax_partial(const T* __restrict__ data, size_t per_frame, T* __restrict__ pmin, T* __restrict__ pmax) {
    const int fi = blockIdx.y;
    const T* f = data + (size_t)fi * per_frame;
    T mn = f[0], mx = f[0];
    for (size_t i = (size_t)blockIdx.x * MM_THREADS + threadIdx.x; i < per_frame; i += (size_t)MM_BLOCKS * MM_THREADS) {
        const T v = f[i];
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
    }
    __shared__ T smn[MM_THREADS], smx[MM_THREADS];
    smn[threadIdx.x] = mn;
    smx[threadIdx.x] = mx;
    __syncthreads();
    for (int s = MM_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            const T a = smn[threadIdx.x + s], b = smx[threadIdx.x + s];
            if (a < smn[threadIdx.x]) smn[threadIdx.x] = a;
            if (b > smx[threadIdx.x]) smx[threadIdx.x] = b;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { pmin[fi * MM_BLOCKS + blockIdx.x] = smn[0]; pmax[fi * MM_BLOCKS + blockIdx.x] = smx[0]; }
}

template <typename T>
__global__ void k_minmax_final(const T* __restrict__ pmin, const T* __restrict__ pmax, int n, T* __restrict__ mn, T* __restrict__ mx) {
    const int fi = blockIdx.x * blockDim.x + threadIdx.x;
    if (fi >= n) return;
    T a = pmin[fi * MM_BLOCKS], b = pmax[fi * MM_BLOCKS];
    for (int k = 1; k < MM_BLOCKS; k++) {
        const T x = pmin[fi * MM_BLOCKS + k], y = pmax[fi * MM_BLOCKS + k];
        a = x < a ? x : a;
        b = y > b ? y : b;
    }
    mn[fi] = a;
    mx[fi] = b;
}

// scratch layout for T: [pmin n*64][pmax n*64][mn n][mx n]
template <typename T>
static int frame_minmax(epid_ctx* ctx, const epid_batch* in, T** d_mn, T** d_mx) {
    const int n = in->n;
    const size_t need = sizeof(T) * ((size_t)n * MM_BLOCKS * 2 + (size_t)n * 2) + 64;
    int rc = ensure_scratch(ctx, need);
    if (rc != EPID_OK) return rc;
    T* pmin = (T*)ctx->scratch;
    T* pmax = pmin + (size_t)n * MM_BLOCKS;
    T* mn = pmax + (size_t)n * MM_BLOCKS;
    T* mx = mn + n;
    const size_t per = (size_t)in->h * in->w;
    k_minmax_partial<T><<<dim3(MM_BLOCKS, n), MM_THREADS, 0, ctx->stream>>>((const T*)in->dptr, per, pmin, pmax);
    k_minmax_final<T><<<(n + 127) / 128, 128, 0, ctx->stream>>>(pmin, pmax, n, mn, mx);
    ctx->launches += 2;
    EPID_CUDA(cudaGetLastError());
    *d_mn = mn;
    *d_mx = mx;
    return EPID_OK;
}

// ---------------------------------------------------------------------------------------- maps
enum { OP_INVERT = 0, OP_BITINV = 1, OP_GROUND = 2, OP_THRESH_HI = 3, OP_THRESH_LO = 4 };

template <typename T, int OP>
__global__ void k_map_same(const T* __restrict__ in, T* __restrict__ out, size_t per_frame, const T* __restrict__ mn, const T* __restrict__ mx, double param) {
    const int fi = blockIdx.y;
    const T* f = in + (size_t)fi * per_frame;
    T* o = out + (size_t)fi * per_frame;
    T lo = T(0), hi = T(0);
    if (OP == OP_INVERT || OP == OP_GROUND) { lo = mn[fi]; hi = mx[fi]; }
    using W = typename Wide<T>::type;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_frame; i += (size_t)gridDim.x * blockDim.x) {
        const T v = f[i];
        T r;
        if (OP == OP_INVERT) {
            // -a + max + min evaluated left to right in the array's dtype (modular for integers)
            r = (T)((W)(T)((W)(T)(-(W)v) + (W)hi) + (W)lo);
        } else if (OP == OP_GROUND) {
            r = (T)((W)(T)((W)v - (W)lo) + (W)(T)param);
        } else if (OP == OP_THRESH_HI) {
            r = ((double)v >= param) ? v : T(0);
        } else if (OP == OP_THRESH_LO) {
            r = ((double)v <= param) ? v : T(0);
        } else {
            r = v;
        }
        o[i] = r;
    }
}

template <typename T>
__global__ void k_bitinv(const T* __restrict__ in, T* __restrict__ out, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) out[i] = (T)~in[i];
}

template <typename T, typename O>
__global__ void k_normalize(const T* __restrict__ in, O* __restrict__ out, size_t per_frame, const T* __restrict__ mx, int use_max, double value) {
    const int fi = blockIdx.y;
    const T* f = in + (size_t)fi * per_frame;
    O* o = out + (size_t)fi * per_frame;
    const O den = use_max ? (O)mx[fi] : (O)value;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_frame; i += (size_t)gridDim.x * blockDim.x) o[i] = (O)f[i] / den;
}

template <typename T>
__global__ void k_binarize(const T* __restrict__ in, long long* __restrict__ out, size_t total, double t) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
        out[i] = ((double)in[i] >= t) ? 1 : 0;
}

template <typename T>
__global__ void k_to_double(const T* __restrict__ in, double* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

#define EPID_DISPATCH(dt, FN, ...)                                                  \
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

static dim3 map_grid(const epid_batch* in) {
    size_t per = (size_t)in->h * in->w;
    int bx = (int)((per + 256 * 8 - 1) / (256 * 8));
    if (bx < 1) bx = 1;
    if (bx > 1024) bx = 1024;
    return dim3(bx, in->n);
}

template <typename T>
static int do_invert(epid_ctx* ctx, const epid_batch* in, epid_batch* out) {
    T *mn, *mx;
    int rc = frame_minmax<T>(ctx, in, &mn, &mx);
    if (rc != EPID_OK) return rc;
    k_map_same<T, OP_INVERT><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (T*)out->dptr, (size_t)in->h * in->w, mn, mx, 0.0);
    ctx->launches++;
    return EPID_OK;
}

template <typename T>
static int do_ground(epid_ctx* ctx, const epid_batch* in, epid_batch* out, double value, double* mins) {
    T *mn, *mx;
    int rc = frame_minmax<T>(ctx, in, &mn, &mx);
    if (rc != EPID_OK) return rc;
    k_map_same<T, OP_GROUND><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (T*)out->dptr, (size_t)in->h * in->w, mn, mx, value);
    ctx->launches++;
    if (mins) {
        double* d = nullptr;
        EPID_CUDA(cudaMallocAsync((void**)&d, sizeof(double) * in->n, ctx->stream));
        k_to_double<T><<<(in->n + 127) / 128, 128, 0, ctx->stream>>>(mn, d, in->n);
        ctx->launches++;
        EPID_CUDA(cudaMemcpyAsync(mins, d, sizeof(double) * in->n, cudaMemcpyDeviceToHost, ctx->stream));
        EPID_CUDA(cudaFreeAsync(d, ctx->stream));
    }
    return EPID_OK;
}

template <typename T>
static int do_threshold(epid_ctx* ctx, const epid_batch* in, epid_batch* out, double t, int kind) {
    if (kind == 0)
        k_map_same<T, OP_THRESH_HI><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (T*)out->dptr, (size_t)in->h * in->w, nullptr, nullptr, t);
    else
        k_map_same<T, OP_THRESH_LO><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (T*)out->dptr, (size_t)in->h * in->w, nullptr, nullptr, t);
    ctx->launches++;
    return EPID_OK;
}

template <typename T>
static int do_bitinv(epid_ctx* ctx, const epid_batch* in, epid_batch* out) {
    k_bitinv<T><<<1024, 256, 0, ctx->stream>>>((const T*)in->dptr, (T*)out->dptr, (size_t)in->n * in->h * in->w);
    ctx->launches++;
    return EPID_OK;
}

template <typename T>
static int do_normalize(epid_ctx* ctx, const epid_batch* in, epid_batch* out, int use_max, double value) {
    T *mn = nullptr, *mx = nullptr;
    if (use_max) {
        int rc = frame_minmax<T>(ctx, in, &mn, &mx);
        if (rc != EPID_OK) return rc;
    }
    if (out->dtype == EPID_F32)
        k_normalize<T, float><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (float*)out->dptr, (size_t)in->h * in->w, mx, use_max, value);
    else
        k_normalize<T, double><<<map_grid(in), 256, 0, ctx->stream>>>((const T*)in->dptr, (double*)out->dptr, (size_t)in->h * in->w, mx, use_max, value);
    ctx->launches++;
    return EPID_OK;
}

template <typename T>
static int do_binarize(epid_ctx* ctx, const epid_batch* in, epid_batch* out, double t) {
    k_binarize<T><<<1024, 256, 0, ctx->stream>>>((const T*)in->dptr, (long long*)out->dptr, (size_t)in->n * in->h * in->w, t);
    ctx->launches++;
    return EPID_OK;
}

static int finish(epid_ctx* ctx, int rc, epid_batch** out) {
    if (rc == EPID_OK) {
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { set_error("kernel failed: %s", cudaGetErrorString(e)); rc = EPID_ERR_CUDA; }
    }
    if (rc != EPID_OK && out && *out) { epid_batch_free(*out); *out = nullptr; }
    return rc;
}

// ---------------------------------------------------------------------------------------- statistics API helpers
__global__ void k_refs_from_batch(const uint16_t* base, int n, int H0, int W0, int r0, int c0, FrameRef* refs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    refs[i].origin = base + (size_t)i * H0 * W0 + (size_t)r0 * W0 + c0;
    refs[i].pitch = W0;
    refs[i].pad = 0;
}

__global__ void k_u8_to_u16(const uint8_t* __restrict__ in, uint16_t* __restrict__ out, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) out[i] = in[i];
}

__global__ void k_hist_global(const FrameRef* __restrict__ refs, int H, int W, uint32_t* __restrict__ hist) {
    const FrameRef r = refs[blockIdx.y];
    uint32_t* h = hist + (size_t)blockIdx.y * 65536;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
        const int y = i / W, x = i - y * W;
        atomicAdd(h + __ldg(r.origin + (size_t)y * r.pitch + x), 1u);
    }
}

}  // namespace epid

using namespace epid;

extern "C" {

#define EPID_CHECK_IN(in)                                                          \
    EPID_REQUIRE(ctx && (in) && out, EPID_ERR_INVALID, "NULL argument");           \
    EPID_CUDA(cudaSetDevice(ctx->device));

int32_t epid_invert(epid_ctx* ctx, const epid_batch* in, epid_batch** out) {
    EPID_CHECK_IN(in);
    int rc = epid_batch_alloc(ctx, in->dtype, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    EPID_DISPATCH(in->dtype, do_invert, ctx, in, *out);
    return finish(ctx, rc, out);
}

int32_t epid_bit_invert(epid_ctx* ctx, const epid_batch* in, epid_batch** out) {
    EPID_CHECK_IN(in);
    EPID_REQUIRE(in->dtype != EPID_F32 && in->dtype != EPID_F64, EPID_ERR_INVALID,
                 "The datatype could not be safely inverted. This usually means the array is a float-like datatype. Cast to an integer-like datatype first.");
    int rc = epid_batch_alloc(ctx, in->dtype, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    switch (in->dtype) {
        case EPID_U8: rc = do_bitinv<uint8_t>(ctx, in, *out); break;
        case EPID_U16: rc = do_bitinv<uint16_t>(ctx, in, *out); break;
        case EPID_I16: rc = do_bitinv<int16_t>(ctx, in, *out); break;
        case EPID_I32: rc = do_bitinv<int32_t>(ctx, in, *out); break;
        case EPID_I64: rc = do_bitinv<long long>(ctx, in, *out); break;
        default: rc = EPID_ERR_INVALID;
    }
    return finish(ctx, rc, out);
}

int32_t epid_ground(epid_ctx* ctx, const epid_batch* in, double value, epid_batch** out, double* mins) {
    EPID_CHECK_IN(in);
    const bool is_float = in->dtype == EPID_F32 || in->dtype == EPID_F64;
    EPID_REQUIRE(is_float || value == floor(value), EPID_ERR_UNSUPPORTED, "ground(value) must be integral for integer images");
    int rc = epid_batch_alloc(ctx, in->dtype, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    EPID_DISPATCH(in->dtype, do_ground, ctx, in, *out, value, mins);
    return finish(ctx, rc, out);
}

int32_t epid_normalize(epid_ctx* ctx, const epid_batch* in, int32_t use_max, double value, epid_batch** out) {
    EPID_CHECK_IN(in);
    const int odt = in->dtype == EPID_F32 ? EPID_F32 : EPID_F64;   // numpy: float32 / float32 stays float32, ints -> float64
    int rc = epid_batch_alloc(ctx, odt, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    EPID_DISPATCH(in->dtype, do_normalize, ctx, in, *out, use_max, value);
    return finish(ctx, rc, out);
}

int32_t epid_threshold(epid_ctx* ctx, const epid_batch* in, double t, int32_t kind, epid_batch** out) {
    EPID_CHECK_IN(in);
    int rc = epid_batch_alloc(ctx, in->dtype, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    EPID_DISPATCH(in->dtype, do_threshold, ctx, in, *out, t, kind);
    return finish(ctx, rc, out);
}

int32_t epid_binarize(epid_ctx* ctx, const epid_batch* in, double t, epid_batch** out) {
    EPID_CHECK_IN(in);
    int rc = epid_batch_alloc(ctx, EPID_I64, in->n, in->h, in->w, out);
    if (rc != EPID_OK) return rc;
    EPID_DISPATCH(in->dtype, do_binarize, ctx, in, *out, t);
    return finish(ctx, rc, out);
}

// ---------------------------------------------------------------------------------------- frame statistics
static int stats_prepare(epid_ctx* ctx, const epid_batch* b, int r0, int c0, int vh, int vw, const uint16_t** base, uint16_t** tmp) {
    EPID_REQUIRE(b->dtype == EPID_U16 || b->dtype == EPID_U8, EPID_ERR_UNSUPPORTED, "frame statistics need uint8/uint16 frames");
    EPID_REQUIRE(r0 >= 0 && c0 >= 0 && vh > 0 && vw > 0 && r0 + vh <= b->h && c0 + vw <= b->w, EPID_ERR_INVALID, "view outside the frame");
    *tmp = nullptr;
    if (b->dtype == EPID_U8) {
        const size_t total = (size_t)b->n * b->h * b->w;
        EPID_CUDA(cudaMalloc((void**)tmp, total * 2));
        k_u8_to_u16<<<1024, 256, 0, ctx->stream>>>((const uint8_t*)b->dptr, *tmp, total);
        ctx->launches++;
        *base = *tmp;
    } else {
        *base = (const uint16_t*)b->dptr;
    }
    return EPID_OK;
}

int32_t epid_frame_stats(epid_ctx* ctx, const epid_batch* b, int32_t r0, int32_t c0, int32_t vh, int32_t vw, const double* q_percent,
                         int32_t nq, double* mn, double* mx, double* sum, double* rowsum, double* colsum, double* pct) {
    EPID_REQUIRE(ctx && b, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(nq >= 0 && 2 * nq <= STATS_MAX_RANKS, EPID_ERR_UNSUPPORTED, "at most %d percentiles per call", STATS_MAX_RANKS / 2);
    EPID_CUDA(cudaSetDevice(ctx->device));
    const uint16_t* base;
    uint16_t* tmp;
    int rc = stats_prepare(ctx, b, r0, c0, vh, vw, &base, &tmp);
    if (rc != EPID_OK) return rc;
    StatsGeom g;
    rc = make_stats_geom(&g, vh, vw);
    if (rc != EPID_OK) { if (tmp) cudaFree(tmp); return rc; }
    const int n = b->n;
    const int npix = vh * vw;
    std::vector<double> gam(nq);
    for (int k = 0; k < nq; k++) {
        const double q = q_percent[k] / 100.0;
        EPID_REQUIRE(q >= 0.0 && q <= 1.0, EPID_ERR_INVALID, "Percentiles must be in the range [0, 100]");
        const double vi = (double)npix * q + (1.0 + q * (1.0 - 1.0 - 1.0)) - 1.0;
        double prev = floor(vi), next = prev + 1.0;
        gam[k] = vi - prev;
        if (prev < 0) prev = 0;
        if (next < 0) next = 0;
        if (prev > npix - 1) prev = npix - 1;
        if (next > npix - 1) next = npix - 1;
        g.ranks[2 * k] = (uint32_t)prev;
        g.ranks[2 * k + 1] = (uint32_t)next;
    }
    g.nranks = 2 * nq;
    g.box = 0;
    const size_t bytes = sizeof(FrameRef) * n + sizeof(FrameStats) * n + sizeof(uint32_t) * (size_t)n * (vh + vw) + 1024;
    rc = ensure_scratch(ctx, bytes);
    if (rc != EPID_OK) { if (tmp) cudaFree(tmp); return rc; }
    char* p = (char*)ctx->scratch;
    FrameRef* refs = (FrameRef*)p; p += (sizeof(FrameRef) * n + 255) / 256 * 256;
    FrameStats* st = (FrameStats*)p; p += (sizeof(FrameStats) * n + 255) / 256 * 256;
    uint32_t* d_row = (uint32_t*)p; p += (sizeof(uint32_t) * (size_t)n * vh + 255) / 256 * 256;
    uint32_t* d_col = (uint32_t*)p;
    k_refs_from_batch<<<(n + 127) / 128, 128, 0, ctx->stream>>>(base, n, b->h, b->w, r0, c0, refs);
    ctx->launches++;
    rc = launch_frame_stats(ctx, ctx->stream, g, refs, n, st, d_row, d_col);
    std::vector<FrameStats> hs(n);
    std::vector<uint32_t> hrow, hcol;
    if (rc == EPID_OK) {
        cudaError_t e = cudaMemcpyAsync(hs.data(), st, sizeof(FrameStats) * n, cudaMemcpyDeviceToHost, ctx->stream);
        if (rowsum && e == cudaSuccess) { hrow.resize((size_t)n * vh); e = cudaMemcpyAsync(hrow.data(), d_row, sizeof(uint32_t) * hrow.size(), cudaMemcpyDeviceToHost, ctx->stream); }
        if (colsum && e == cudaSuccess) { hcol.resize((size_t)n * vw); e = cudaMemcpyAsync(hcol.data(), d_col, sizeof(uint32_t) * hcol.size(), cudaMemcpyDeviceToHost, ctx->stream); }
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { set_error("frame stats failed: %s", cudaGetErrorString(e)); rc = EPID_ERR_CUDA; }
    }
    if (tmp) cudaFree(tmp);
    if (rc != EPID_OK) return rc;
    for (int i = 0; i < n; i++) {
        if (mn) mn[i] = hs[i].mn;
        if (mx) mx[i] = hs[i].mx;
        if (sum) sum[i] = (double)hs[i].sum;
        for (int k = 0; k < nq && pct; k++) {
            // numpy _lerp
            const double a = hs[i].ostat[2 * k], bb = hs[i].ostat[2 * k + 1], t = gam[k];
            const double d = bb - a;
            double r = a + d * t;
            if (t >= 0.5) r = bb - d * (1.0 - t);
            pct[(size_t)i * nq + k] = r;
        }
    }
    if (rowsum) for (size_t i = 0; i < hrow.size(); i++) rowsum[i] = hrow[i];
    if (colsum) for (size_t i = 0; i < hcol.size(); i++) colsum[i] = hcol[i];
    return EPID_OK;
}

int32_t epid_frame_histogram(epid_ctx* ctx, const epid_batch* b, int32_t r0, int32_t c0, int32_t vh, int32_t vw, uint32_t* hist) {
    EPID_REQUIRE(ctx && b && hist, EPID_ERR_INVALID, "NULL argument");
    EPID_CUDA(cudaSetDevice(ctx->device));
    const uint16_t* base;
    uint16_t* tmp;
    int rc = stats_prepare(ctx, b, r0, c0, vh, vw, &base, &tmp);
    if (rc != EPID_OK) return rc;
    const int n = b->n;
    const size_t bytes = sizeof(FrameRef) * n + 256 + sizeof(uint32_t) * (size_t)n * 65536;
    rc = ensure_scratch(ctx, bytes);
    if (rc != EPID_OK) { if (tmp) cudaFree(tmp); return rc; }
    FrameRef* refs = (FrameRef*)ctx->scratch;
    uint32_t* d_hist = (uint32_t*)((char*)ctx->scratch + (sizeof(FrameRef) * n + 255) / 256 * 256);
    k_refs_from_batch<<<(n + 127) / 128, 128, 0, ctx->stream>>>(base, n, b->h, b->w, r0, c0, refs);
    cudaMemsetAsync(d_hist, 0, sizeof(uint32_t) * (size_t)n * 65536, ctx->stream);
    k_hist_global<<<dim3(64, n), 256, 0, ctx->stream>>>(refs, vh, vw, d_hist);
    ctx->launches += 2;
    cudaError_t e = cudaMemcpyAsync(hist, d_hist, sizeof(uint32_t) * (size_t)n * 65536, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) { set_error("histogram failed: %s", cudaGetErrorString(e)); return EPID_ERR_CUDA; }
    return EPID_OK;
}

}  // extern "C"
