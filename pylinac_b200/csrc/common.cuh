// Shared internals of libepid (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/epid.h"

namespace epid {

void set_error(const char* fmt, ...);

#define EPID_CUDA(call)                                                                      \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            ::epid::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return EPID_ERR_CUDA;                                                            \
        }                                                                                    \
    } while (0)

#define EPID_REQUIRE(cond, code, ...)              \
    do {                                           \
        if (!(cond)) {                             \
            ::epid::set_error(__VA_ARGS__);        \
            return (code);                         \
        }                                          \
    } while (0)

inline size_t dtype_size(int dt) {
    switch (dt) {
        case EPID_U8: return 1;
        case EPID_U16: case EPID_I16: return 2;
        case EPID_I32: case EPID_F32: return 4;
        case EPID_F64: case EPID_I64: return 8;
    }
    return 0;
}

}  // namespace epid

struct epid_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t hbm_bytes = 0;
    cudaStream_t stream = nullptr;       // main stream
    cudaStream_t copy_stream[2] = {nullptr, nullptr};
    int64_t launches = 0;
    void* nccl_comm = nullptr;           // ncclComm_t
    int nranks = 1, rank = 0;
    // reusable device scratch (grown on demand, freed with the ctx)
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    void* scratch2 = nullptr;            // work area of the per-frame exact re-run (pf.cu)
    size_t scratch2_bytes = 0;
    void* hist_scratch = nullptr;        // histograms + column partials of the multi-CTA frame statistics (stats.cu)
    size_t hist_bytes = 0;
    void* inv_scratch = nullptr;         // thresholds / partials of the certified inversion statistics (stats.cu)
    size_t inv_bytes = 0;
    int stats_exact = 0;                 // 1: FieldAnalysis / Starshot take the exact histogram path for every frame (EPID_OPT_STATS_EXACT)
    int64_t stats_uncertified = 0;       // frames whose inversion decision needed the exact histogram path
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    void* pinned_ring = nullptr;         // page-locked staging ring for pageable source frames (pf.cu)
    size_t pinned_ring_bytes = 0;
    // options / diagnostics (epid_set_option / epid_get_counter)
    int pf_exact_only = 0;               // 1: never use the fused sample-guided front kernel
    int pf_win2 = 1;                     // 1 (default): two-kernel window path for the frames it covers (pf_windows2.cu)
    int64_t pf_fallbacks = 0;            // batches (or chunks) re-run by the exact pipeline
    int64_t pf_redone_frames = 0;        // frames re-run individually (per-frame fallback: certified-noise fast re-run or exact pipeline)
    int64_t pf_exact_frames = 0;         // of those, frames that needed the exact-histogram pipeline
    int pf_fast_redo = 1;                // 1 (default): deferred frames whose noise flag can be certified are median-filtered and re-run by the fast pipeline
    cudaStream_t redo_stream = nullptr;  // high-priority stream of the per-frame re-run
    cudaEvent_t ev_front = nullptr, ev_main_done = nullptr, ev_redo_done = nullptr;
    int* h_flags = nullptr;              // 64 page-locked, device-mapped ints: [0] deferred count written by k_pf_collect_deferred
    // dynamic shared memory opt-ins already made ON THIS DEVICE (cudaFuncSetAttribute is per device; one ctx per device)
    std::unordered_map<const void*, size_t> smem_optin;
};

constexpr size_t EPID_BATCH_PAD = 256;
struct epid_batch {
    epid_ctx* ctx = nullptr;
    int dtype = EPID_U16;
    int n = 0, h = 0, w = 0;
    void* dptr = nullptr;
    void* base = nullptr;   // allocation start: dptr = base + EPID_BATCH_PAD (16-byte vector / TMA reads may touch a few bytes either side)
    bool owns = true;
    size_t bytes() const { return (size_t)n * h * w * epid::dtype_size(dtype); }
};

namespace epid {
int ensure_scratch(epid_ctx* ctx, size_t bytes);   // grows ctx->scratch
int ensure_pinned(epid_ctx* ctx, size_t bytes);

// opt a kernel in to `bytes` of dynamic shared memory on ctx's device (remembered per ctx, i.e. per device)
template <class K>
inline int smem_opt_in(epid_ctx* ctx, K* kernel, size_t bytes) {
    size_t& cur = ctx->smem_optin[(const void*)kernel];
    if (bytes > cur) {
        EPID_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    return EPID_OK;
}
#define EPID_SMEM_OPT_IN(ctx, kernel, bytes) do { int _rc = ::epid::smem_opt_in(ctx, kernel, bytes); if (_rc != EPID_OK) return _rc; } while (0)

// ------------------------------------------------------------------------------------------------ device helpers
#ifdef __CUDACC__
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_min(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
#endif

}  // namespace epid
