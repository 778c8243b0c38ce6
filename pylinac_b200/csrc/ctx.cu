// Context, batch (HBM-resident frames) and host-memory management of libepid.
#include <cstdarg>

#include "common.cuh"

namespace epid {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int ensure_scratch(epid_ctx* ctx, size_t bytes) {
    if (ctx->scratch_bytes >= bytes) return EPID_OK;
    if (ctx->scratch) {
        EPID_CUDA(cudaStreamSynchronize(ctx->stream));
        EPID_CUDA(cudaFree(ctx->scratch));
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMalloc(&ctx->scratch, want);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        return EPID_ERR_NOMEM;
    }
    ctx->scratch_bytes = want;
    return EPID_OK;
}

int ensure_pinned(epid_ctx* ctx, size_t bytes) {
    if (ctx->pinned_bytes >= bytes) return EPID_OK;
    if (ctx->pinned) {
        EPID_CUDA(cudaStreamSynchronize(ctx->stream));
        EPID_CUDA(cudaFreeHost(ctx->pinned));
        ctx->pinned = nullptr;
        ctx->pinned_bytes = 0;
    }
    cudaError_t e = cudaMallocHost(&ctx->pinned, bytes);
    if (e != cudaSuccess) {
        set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return EPID_ERR_NOMEM;
    }
    ctx->pinned_bytes = bytes;
    return EPID_OK;
}

}  // namespace epid

using namespace epid;

extern "C" {

const char* epid_last_error(void) { return g_err; }

int32_t epid_version(void) { return 100; }

int32_t epid_device_count(int32_t* count) {
    if (!count) return EPID_ERR_INVALID;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    *count = n;
    return EPID_OK;
}

int32_t epid_ctx_create(int32_t device, epid_ctx** out) {
    EPID_REQUIRE(out, EPID_ERR_INVALID, "out is NULL");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device is visible; libepid has no CPU fallback");
        return EPID_ERR_NO_DEVICE;
    }
    EPID_REQUIRE(device >= 0 && device < n, EPID_ERR_INVALID, "device %d out of range (have %d)", device, n);
    EPID_CUDA(cudaSetDevice(device));
    epid_ctx* c = new epid_ctx();
    c->device = device;
    cudaDeviceProp prop;
    EPID_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->hbm_bytes = prop.totalGlobalMem;
    EPID_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    EPID_CUDA(cudaStreamCreateWithFlags(&c->copy_stream[0], cudaStreamNonBlocking));
    EPID_CUDA(cudaStreamCreateWithFlags(&c->copy_stream[1], cudaStreamNonBlocking));
    {
        int lo = 0, hi = 0;
        EPID_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        EPID_CUDA(cudaStreamCreateWithPriority(&c->redo_stream, cudaStreamNonBlocking, hi));
        EPID_CUDA(cudaEventCreateWithFlags(&c->ev_front, cudaEventDisableTiming));
        EPID_CUDA(cudaEventCreateWithFlags(&c->ev_main_done, cudaEventDisableTiming));
        EPID_CUDA(cudaEventCreateWithFlags(&c->ev_redo_done, cudaEventDisableTiming));
        EPID_CUDA(cudaHostAlloc((void**)&c->h_flags, 64 * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
        memset(c->h_flags, 0, 64 * sizeof(int));
    }
    *out = c;
    return EPID_OK;
}

int32_t epid_comm_destroy(epid_ctx* ctx);

int32_t epid_ctx_destroy(epid_ctx* ctx) {
    if (!ctx) return EPID_OK;
    cudaSetDevice(ctx->device);
    if (ctx->nccl_comm) epid_comm_destroy(ctx);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->scratch2) cudaFree(ctx->scratch2);
    if (ctx->hist_scratch) cudaFree(ctx->hist_scratch);
    if (ctx->inv_scratch) cudaFree(ctx->inv_scratch);
    if (ctx->pinned_ring) cudaFreeHost(ctx->pinned_ring);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->copy_stream[0]);
    cudaStreamDestroy(ctx->copy_stream[1]);
    if (ctx->redo_stream) { cudaStreamSynchronize(ctx->redo_stream); cudaStreamDestroy(ctx->redo_stream); }
    if (ctx->ev_front) cudaEventDestroy(ctx->ev_front);
    if (ctx->ev_main_done) cudaEventDestroy(ctx->ev_main_done);
    if (ctx->ev_redo_done) cudaEventDestroy(ctx->ev_redo_done);
    if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
    delete ctx;
    return EPID_OK;
}

int32_t epid_sync(epid_ctx* ctx) {
    EPID_REQUIRE(ctx, EPID_ERR_INVALID, "ctx is NULL");
    EPID_CUDA(cudaSetDevice(ctx->device));
    EPID_CUDA(cudaStreamSynchronize(ctx->stream));
    return EPID_OK;
}

int32_t epid_device_info(epid_ctx* ctx, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, size_t* hbm_bytes) {
    EPID_REQUIRE(ctx, EPID_ERR_INVALID, "ctx is NULL");
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (hbm_bytes) *hbm_bytes = ctx->hbm_bytes;
    return EPID_OK;
}

int32_t epid_device_pci_bus_id(int32_t device, char* out, int32_t cap) {
    EPID_REQUIRE(out && cap >= 16, EPID_ERR_INVALID, "output buffer too small");
    EPID_CUDA(cudaDeviceGetPCIBusId(out, cap, device));
    return EPID_OK;
}

int32_t epid_launch_count(epid_ctx* ctx, int64_t* launches) {
    EPID_REQUIRE(ctx && launches, EPID_ERR_INVALID, "NULL argument");
    *launches = ctx->launches;
    return EPID_OK;
}

int32_t epid_set_option(epid_ctx* ctx, int32_t key, int64_t value) {
    EPID_REQUIRE(ctx, EPID_ERR_INVALID, "ctx is NULL");
    switch (key) {
        case EPID_OPT_PF_EXACT_ONLY: ctx->pf_exact_only = value ? 1 : 0; return EPID_OK;
        case EPID_OPT_PF_WIN2: ctx->pf_win2 = value ? 1 : 0; return EPID_OK;
        case EPID_OPT_PF_FAST_REDO: ctx->pf_fast_redo = value ? 1 : 0; return EPID_OK;
        case EPID_OPT_STATS_EXACT: ctx->stats_exact = value ? 1 : 0; return EPID_OK;
    }
    set_error("unknown option %d", key);
    return EPID_ERR_INVALID;
}

int32_t epid_get_counter(epid_ctx* ctx, int32_t key, int64_t* value) {
    EPID_REQUIRE(ctx && value, EPID_ERR_INVALID, "NULL argument");
    switch (key) {
        case EPID_CTR_PF_FALLBACKS: *value = ctx->pf_fallbacks; return EPID_OK;
        case EPID_CTR_PF_REDONE_FRAMES: *value = ctx->pf_redone_frames; return EPID_OK;
        case EPID_CTR_PF_EXACT_FRAMES: *value = ctx->pf_exact_frames; return EPID_OK;
        case EPID_CTR_STATS_UNCERTIFIED: *value = ctx->stats_uncertified; return EPID_OK;
    }
    set_error("unknown counter %d", key);
    return EPID_ERR_INVALID;
}

int32_t epid_host_alloc(size_t bytes, void** out) {
    EPID_REQUIRE(out, EPID_ERR_INVALID, "out is NULL");
    cudaError_t e = cudaMallocHost(out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? EPID_ERR_NO_DEVICE : EPID_ERR_NOMEM;
    }
    return EPID_OK;
}

int32_t epid_host_free(void* p) {
    if (p) cudaFreeHost(p);
    return EPID_OK;
}

int32_t epid_batch_alloc(epid_ctx* ctx, int32_t dtype, int32_t n, int32_t h, int32_t w, epid_batch** out) {
    EPID_REQUIRE(ctx && out, EPID_ERR_INVALID, "NULL argument");
    EPID_REQUIRE(dtype_size(dtype) > 0, EPID_ERR_INVALID, "unknown dtype %d", dtype);
    EPID_REQUIRE(n > 0 && h > 0 && w > 0, EPID_ERR_INVALID, "empty batch (%d x %d x %d)", n, h, w);
    EPID_CUDA(cudaSetDevice(ctx->device));
    epid_batch* b = new epid_batch();
    b->ctx = ctx;
    b->dtype = dtype;
    b->n = n;
    b->h = h;
    b->w = w;
    cudaError_t e = cudaMalloc(&b->base, b->bytes() + 2 * EPID_BATCH_PAD);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu) failed: %s", b->bytes(), cudaGetErrorString(e));
        delete b;
        return EPID_ERR_NOMEM;
    }
    b->dptr = (char*)b->base + EPID_BATCH_PAD;
    *out = b;
    return EPID_OK;
}

int32_t epid_batch_upload(epid_ctx* ctx, const void* host, int32_t dtype, int32_t n, int32_t h, int32_t w, epid_batch** out) {
    EPID_REQUIRE(host, EPID_ERR_INVALID, "host pointer is NULL");
    int rc = epid_batch_alloc(ctx, dtype, n, h, w, out);
    if (rc != EPID_OK) return rc;
    epid_batch* b = *out;
    cudaError_t e = cudaMemcpyAsync(b->dptr, host, b->bytes(), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("H2D copy failed: %s", cudaGetErrorString(e));
        cudaFree(b->base);
        delete b;
        *out = nullptr;
        return EPID_ERR_CUDA;
    }
    return EPID_OK;
}

int32_t epid_batch_write(epid_batch* b, const void* host) {
    EPID_REQUIRE(b && host, EPID_ERR_INVALID, "NULL argument");
    EPID_CUDA(cudaSetDevice(b->ctx->device));
    EPID_CUDA(cudaMemcpyAsync(b->dptr, host, b->bytes(), cudaMemcpyHostToDevice, b->ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return EPID_OK;
}

int32_t epid_batch_download(epid_batch* b, void* host) {
    EPID_REQUIRE(b && host, EPID_ERR_INVALID, "NULL argument");
    EPID_CUDA(cudaSetDevice(b->ctx->device));
    EPID_CUDA(cudaMemcpyAsync(host, b->dptr, b->bytes(), cudaMemcpyDeviceToHost, b->ctx->stream));
    EPID_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return EPID_OK;
}

int32_t epid_batch_free(epid_batch* b) {
    if (!b) return EPID_OK;
    if (b->owns && b->base) {
        cudaSetDevice(b->ctx->device);
        cudaFree(b->base);
    }
    delete b;
    return EPID_OK;
}

int32_t epid_batch_shape(const epid_batch* b, int32_t* dtype, int32_t* n, int32_t* h, int32_t* w) {
    EPID_REQUIRE(b, EPID_ERR_INVALID, "batch is NULL");
    if (dtype) *dtype = b->dtype;
    if (n) *n = b->n;
    if (h) *h = b->h;
    if (w) *w = b->w;
    return EPID_OK;
}

int32_t epid_batch_device_ptr(const epid_batch* b, void** dptr) {
    EPID_REQUIRE(b && dptr, EPID_ERR_INVALID, "NULL argument");
    *dptr = b->dptr;
    return EPID_OK;
}

}  // extern "C"
