// api.cu — context, memory and timing entry points of libjsdrcuda.so.
#include <algorithm>
#include <cstdlib>
#include <memory>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace jsdr {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int upload(jsdr_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    JSDR_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
}

int cuda_failed(cudaError_t e, const char *what, const char *call)
{
    set_error("%s: %s: %s", what, call, cudaGetErrorString(e));
    cudaGetLastError();   // reported: the next launch check must not see it
    return e == cudaErrorMemoryAllocation ? JSDR_ENOMEM : JSDR_ECUDA;
}

}  // namespace jsdr

using namespace jsdr;

extern "C" int jsdr_abi_version(void) { return JSDR_ABI_VERSION; }

extern "C" const char *jsdr_last_error(void) { return g_err; }

extern "C" int jsdr_device_count(int *count)
try {
    JSDR_REQUIRE(count, JSDR_EINVAL, "null argument");
    *count = 0;
    JSDR_CUDA(cudaGetDeviceCount(count));
    return JSDR_OK;
} JSDR_CATCH_ALL

static int ctx_init(jsdr_ctx *ctx);

extern "C" int jsdr_ctx_create(int device, jsdr_ctx **out)
try {
    JSDR_REQUIRE(out, JSDR_EINVAL, "null argument");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        // no CPU fallback by design: the product path is the CUDA path
        set_error("jsdr_ctx_create: no CUDA device (%s)", cudaGetErrorString(e));
        return JSDR_ECUDA;
    }
    JSDR_REQUIRE(device >= 0 && device < count, JSDR_EINVAL, "device index out of range");
    JSDR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    JSDR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("jsdr_ctx_create: device %d is sm_%d%d; this library is built for sm_100a only",
                  device, prop.major, prop.minor);
        return JSDR_EUNSUPPORTED;
    }
    std::unique_ptr<jsdr_ctx> ctx(new jsdr_ctx());
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    JSDR_TRY(ctx_init(ctx.get()));
    *out = ctx.release();
    return JSDR_OK;
} JSDR_CATCH_ALL

static int ctx_init(jsdr_ctx *ctx)
{
    const char *what = "jsdr_ctx_create";
    if (const char *e = getenv("JSDR_L2_PREFETCH")) ctx->l2_prefetch = std::max(0, std::min(atoi(e), 8));   // 0: off, n: n x resident CTAs ahead
    {   // three priorities: the side stream carries the serial, data-independent phase replay and
        // goes first, so that its few CTAs are placed as soon as a slot frees up instead of queueing
        // behind the whole grid of a data kernel; the main stream is in the middle; the auxiliary
        // stream (the pump's FFT when it runs beside the decimator) fills what is left
        int lo = 0, hi = 0;
        JSDR_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        const int mid = (hi < lo) ? lo - 1 : lo;
        JSDR_TRY(ctx->stream.create(mid, what));
        JSDR_TRY(ctx->side.create(hi, what));
        JSDR_TRY(ctx->side2.create(hi, what));
        JSDR_TRY(ctx->aux.create(lo, what));
    }
    JSDR_TRY(ctx->copy_in.create(0, what));
    JSDR_TRY(ctx->copy_out.create(0, what));
    for (int i = 0; i < 16; i++) {
        JSDR_TRY(ctx->ev_chunk_in[i].create(what));
        JSDR_TRY(ctx->ev_chunk_done[i].create(what));
    }
    JSDR_TRY(ctx->ev_t0.create(what, cudaEventDefault));
    JSDR_TRY(ctx->ev_t1.create(what, cudaEventDefault));
    JSDR_TRY(ctx->ev_aux_fork.create(what));
    JSDR_TRY(ctx->ev_aux_join.create(what));
    JSDR_TRY(ctx->ev_fork.create(what));
    JSDR_TRY(ctx->ev_join.create(what));
    return JSDR_OK;
}

extern "C" int jsdr_ctx_destroy(jsdr_ctx *ctx)
try {
    if (!ctx) return JSDR_OK;
    delete ctx;
    cudaGetLastError();
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_ctx_sync(jsdr_ctx *ctx)
try {
    JSDR_REQUIRE(ctx, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaStreamSynchronize(ctx->side));
    JSDR_CUDA(cudaStreamSynchronize(ctx->side2));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->copy_out));
    JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_ctx_launch_count(jsdr_ctx *ctx, int64_t *count)
try {
    JSDR_REQUIRE(ctx && count, JSDR_EINVAL, "null argument");
    *count = ctx->launches;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_ctx_profile(jsdr_ctx *ctx, int enable)
try {
    JSDR_REQUIRE(ctx, JSDR_EINVAL, "null argument");
    if (enable) {                                   // room for every span up front: recording never allocates
        ctx->spans.reserve(jsdr::kMaxProfSpans);
        ctx->free_spans.reserve(jsdr::kMaxProfSpans);
    }
    ctx->profiling = enable != 0;
    return JSDR_OK;
} JSDR_CATCH_ALL

// Sum the event-bracketed durations recorded since the last read, per kernel kind.
extern "C" int jsdr_ctx_profile_read(jsdr_ctx *ctx, double *ms, int64_t *count, int nkinds)
try {
    JSDR_REQUIRE(ctx && ms && count && nkinds >= JSDR_K_COUNT, JSDR_EINVAL, "need room for JSDR_K_COUNT kinds");
    JSDR_TRY(ctx->bind());
    JSDR_TRY(jsdr_ctx_sync(ctx));                   // spans are recorded on every compute stream (bit timing: aux)
    for (int k = 0; k < nkinds; k++) {
        ms[k] = 0.0;
        count[k] = 0;
    }
    int rc = JSDR_OK;
    for (jsdr_prof_span &sp : ctx->spans) {
        float t = 0.f;
        const cudaError_t e = cudaEventElapsedTime(&t, sp.a, sp.b);
        if (e == cudaSuccess) {
            ms[sp.kind] += t;
            count[sp.kind]++;
        } else if (rc == JSDR_OK) {
            set_error("jsdr_ctx_profile_read: %s", cudaGetErrorString(e));
            cudaGetLastError();
            rc = JSDR_ECUDA;
        }
        ctx->free_spans.push_back(std::move(sp));     // every span moves exactly once, error or not
    }
    ctx->spans.clear();
    return rc;
} JSDR_CATCH_ALL

extern "C" int jsdr_host_alloc(jsdr_ctx *ctx, size_t bytes, void **out)
try {
    JSDR_REQUIRE(ctx && out, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_host_free(jsdr_ctx *ctx, void *p)
try {
    JSDR_REQUIRE(ctx, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    if (p) JSDR_CUDA(cudaFreeHost(p));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_dev_alloc(jsdr_ctx *ctx, size_t bytes, void **out)
try {
    JSDR_REQUIRE(ctx && out, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        set_error("jsdr_dev_alloc(%zu): %s", bytes, cudaGetErrorString(e));
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? JSDR_ENOMEM : JSDR_ECUDA;
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_dev_free(jsdr_ctx *ctx, void *p)
try {
    JSDR_REQUIRE(ctx, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    if (p) JSDR_CUDA(cudaFree(p));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_memcpy_h2d(jsdr_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes)
try {
    JSDR_REQUIRE(ctx && (bytes == 0 || (dst_dev && src_host)), JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_memcpy_d2h(jsdr_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes)
try {
    JSDR_REQUIRE(ctx && (bytes == 0 || (dst_host && src_dev)), JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_memset_dev(jsdr_ctx *ctx, void *dst_dev, int value, size_t bytes)
try {
    JSDR_REQUIRE(ctx && dst_dev, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaMemsetAsync(dst_dev, value, bytes, ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_timer_start(jsdr_ctx *ctx)
try {
    JSDR_REQUIRE(ctx, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    JSDR_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_timer_stop_ms(jsdr_ctx *ctx, float *ms)
try {
    JSDR_REQUIRE(ctx && ms, JSDR_EINVAL, "null argument");
    JSDR_TRY(ctx->bind());
    // the timed region ends when the auxiliary stream (bit timing, frames) is done as well; the side
    // stream only ever runs ahead (the next block's phase replay), so it is not waited for
    JSDR_CUDA(cudaEventRecord(ctx->ev_aux_join, ctx->aux));
    JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_aux_join, 0));
    JSDR_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
    JSDR_CUDA(cudaEventSynchronize(ctx->ev_t1));
    JSDR_CUDA(cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return JSDR_OK;
} JSDR_CATCH_ALL
