// common.cuh — shared plumbing for libjsdrcuda.so (context, error reporting,
// streaming load/store helpers).  sm_100a only; there is no CPU fallback.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <exception>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/jsdrcuda.h"

namespace jsdr {

void set_error(const char *fmt, ...);

#define JSDR_CUDA(expr)                                                              \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) {                                                     \
            jsdr::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr,             \
                            cudaGetErrorString(_e));                                 \
            cudaGetLastError(); /* reported: the next launch check must not see it */ \
            return _e == cudaErrorMemoryAllocation ? JSDR_ENOMEM : JSDR_ECUDA;       \
        }                                                                            \
    } while (0)

#define JSDR_REQUIRE(cond, code, msg)                                                \
    do {                                                                             \
        if (!(cond)) {                                                               \
            jsdr::set_error("%s: %s", __func__, msg);                                \
            return code;                                                             \
        }                                                                            \
    } while (0)

#define JSDR_TRY(expr)                                                               \
    do {                                                                             \
        int _rc = (expr);                                                            \
        if (_rc != JSDR_OK) return _rc;                                              \
    } while (0)

// Every entry point is a function-try-block closed by this: the header promises that nothing
// throws across the C boundary (a C++ exception unwinding into a JVM frame ends the process), so a
// failed host allocation (new, std::vector) comes back as a status like every other failure.
#define JSDR_CATCH_ALL                                                               \
    catch (const std::bad_alloc &)                                                   \
    {                                                                                \
        jsdr::set_error("%s: out of host memory", __func__);                         \
        return JSDR_ENOMEM;                                                          \
    }                                                                                \
    catch (const std::exception &e_)                                                 \
    {                                                                                \
        jsdr::set_error("%s: %s", __func__, e_.what());                              \
        return JSDR_EINTERNAL;                                                       \
    }                                                                                \
    catch (...)                                                                      \
    {                                                                                \
        jsdr::set_error("%s: unknown C++ exception", __func__);                      \
        return JSDR_EINTERNAL;                                                       \
    }

// api.cu.  Report a failed CUDA call `call` made for `what` and clear it (as JSDR_CUDA does):
// JSDR_ENOMEM for cudaErrorMemoryAllocation, JSDR_ECUDA for everything else.
int cuda_failed(cudaError_t e, const char *what, const char *call);

// ---- owners of device memory, events and streams ------------------------------------------
// Move-only; the destructor releases what the owner holds.  Acquiring returns a JSDR status and
// reports a failure through cuda_failed, naming `what`.  Every buffer, event and stream a handle
// keeps is one of these, so that a destroy and a failed create release through the same path.

// Device memory with its capacity.
template <class T>
class DevBuf {
public:
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p_(o.p_), cap_(o.cap_) { o.p_ = nullptr, o.cap_ = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept   // what this held is released with `o`
    {
        std::swap(p_, o.p_);
        std::swap(cap_, o.cap_);
        return *this;
    }
    ~DevBuf() { reset(); }
    T *get() const { return p_; }
    explicit operator bool() const { return p_ != nullptr; }
    void reset()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr, cap_ = 0;
    }
    // `bytes` of new memory; what was held is freed first
    int alloc(size_t bytes, const char *what)
    {
        reset();
        void *p = nullptr;
        const cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cuda_failed(e, what, "cudaMalloc");
        p_ = static_cast<T *>(p), cap_ = bytes;
        return JSDR_OK;
    }
    // grow on demand: reallocated (contents lost) only when it holds fewer than `bytes`
    int grow(size_t bytes, const char *what) { return cap_ >= bytes ? JSDR_OK : alloc(bytes, what); }
    // the same, cleared to zeros on `st`
    int alloc_zeroed(size_t bytes, cudaStream_t st, const char *what)
    {
        JSDR_TRY(alloc(bytes, what));
        const cudaError_t e = cudaMemsetAsync(p_, 0, bytes, st);
        return e == cudaSuccess ? JSDR_OK : cuda_failed(e, what, "cudaMemsetAsync");
    }

private:
    T *p_ = nullptr;
    size_t cap_ = 0;
};

inline void release(cudaEvent_t e) { cudaEventDestroy(e); }
inline void release(cudaStream_t s) { cudaStreamDestroy(s); }

// An event or a stream: converts to the runtime's handle, which it keeps owning.
template <class H>
class Owned {
public:
    Owned() = default;
    Owned(Owned &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    Owned &operator=(Owned &&o) noexcept   // what this held is released with `o`
    {
        std::swap(h_, o.h_);
        return *this;
    }
    ~Owned() { reset(); }
    operator H() const { return h_; }
    void reset()
    {
        if (h_) release(h_);
        h_ = nullptr;
    }

protected:
    H h_ = nullptr;
};

struct Event : Owned<cudaEvent_t> {
    int create(const char *what, unsigned flags = cudaEventDisableTiming)
    {
        reset();
        const cudaError_t e = cudaEventCreateWithFlags(&h_, flags);
        return e == cudaSuccess ? JSDR_OK : (h_ = nullptr, cuda_failed(e, what, "cudaEventCreateWithFlags"));
    }
};

struct Stream : Owned<cudaStream_t> {
    int create(int priority, const char *what)   // non-blocking; priority 0 is the runtime's default
    {
        reset();
        const cudaError_t e = cudaStreamCreateWithPriority(&h_, cudaStreamNonBlocking, priority);
        return e == cudaSuccess ? JSDR_OK : (h_ = nullptr, cuda_failed(e, what, "cudaStreamCreateWithPriority"));
    }
};

}  // namespace jsdr

struct jsdr_prof_span {
    int kind;
    jsdr::Event a, b;
};

struct jsdr_ctx {
    int device = 0;
    int sm_count = 0;
    int l2_prefetch = 1;             // FFT: bulk-prefetch the input of the CTA n x (resident CTAs) ahead into L2 (JSDR_L2_PREFETCH=n, 0: off)
    jsdr::Stream stream;             // main stream: data kernels
    jsdr::Stream side;               // side stream: data-independent phase scouts
    jsdr::Stream side2;              // the VCO / bit-phase replay: one short serial chain, beside the tuner scout
    jsdr::Stream aux;                // low priority: work that runs beside the main stream's kernel
    jsdr::Stream copy_in, copy_out;  // host<->device copies of the chunked host path
    jsdr::Event ev_aux_fork, ev_aux_join;
    jsdr::Event ev_chunk_in[16], ev_chunk_done[16];
    jsdr::Event ev_t0, ev_t1;
    jsdr::Event ev_fork, ev_join;
    int64_t launches = 0;
    // per-kernel timing: event pairs recorded around the launches while `profiling` is on
    bool profiling = false;
    std::vector<jsdr_prof_span> spans;       // recorded since the last read
    std::vector<jsdr_prof_span> free_spans;  // event pairs ready for reuse

    int bind() const { return cudaSetDevice(device) == cudaSuccess ? JSDR_OK : JSDR_ECUDA; }
    // the events above may still be pending on any stream; the owners release them after this
    ~jsdr_ctx()
    {
        bind();
        const cudaStream_t all[] = {stream, side, side2, aux, copy_in, copy_out};
        for (cudaStream_t s : all)
            if (s) cudaStreamSynchronize(s);
    }
};

namespace jsdr {

// Function attributes (dynamic shared memory limits, occupancy) are per device: state kept by
// a launch site is indexed by the context's device, so that contexts on different GPUs of one
// process each set their own.
constexpr int kMaxDevices = 64;
// Contexts on different GPUs may be driven from different threads at the same time (the header's
// threading rule), so first-use initialisation is serialised: whoever comes second waits until the
// first has FINISHED (a flag set before the work would let the second thread launch a kernel whose
// shared-memory limit or constant tables are not there yet).
struct PerDeviceFlag {
    std::mutex mu;
    std::atomic<bool> done[kMaxDevices];
    PerDeviceFlag()
    {
        for (auto &d : done) d.store(false, std::memory_order_relaxed);
    }
    template <class F>
    int once(int dev, F &&init)                            // init() -> JSDR status; repeated until it succeeds
    {
        const bool known = dev >= 0 && dev < kMaxDevices;  // unknown device: redo every time
        if (known && done[dev].load(std::memory_order_acquire)) return JSDR_OK;
        std::lock_guard<std::mutex> lock(mu);
        if (known && done[dev].load(std::memory_order_relaxed)) return JSDR_OK;
        const int rc = init();
        if (rc == JSDR_OK && known) done[dev].store(true, std::memory_order_release);
        return rc;
    }
};

// api.cu.  Copy host -> device on the context's main stream and wait for it.
int upload(jsdr_ctx *ctx, void *dst, const void *src, size_t bytes);

// Check the launch that was just made and count it.
static inline int launched(jsdr_ctx *ctx, const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
        return JSDR_ECUDA;
    }
    ctx->launches++;
    return JSDR_OK;
}

// Bracket one kernel launch with CUDA events on its stream when profiling is on.  At most
// kMaxProfSpans launches are kept between two reads (a caller that switches profiling on and never
// reads must not grow event pairs without bound); later launches are simply not timed.
constexpr size_t kMaxProfSpans = 1 << 16;
struct ProfScope {
    jsdr_ctx *ctx;
    cudaStream_t st;
    jsdr_prof_span sp;
    bool on;
    ProfScope(jsdr_ctx *c, int kind, cudaStream_t s)
        : ctx(c), st(s), on(c->profiling && c->spans.size() < kMaxProfSpans && c->spans.size() < c->spans.capacity())
    {
        if (!on) return;
        if (!c->free_spans.empty()) {
            sp = std::move(c->free_spans.back());
            c->free_spans.pop_back();
        } else if (sp.a.create("profiling", cudaEventDefault) != JSDR_OK ||
                   sp.b.create("profiling", cudaEventDefault) != JSDR_OK) {
            on = false;   // this launch is not timed
            return;
        }
        sp.kind = kind;
        cudaEventRecord(sp.a, st);
    }
    ~ProfScope()
    {
        if (!on) return;
        cudaEventRecord(sp.b, st);
        ctx->spans.push_back(std::move(sp));
    }
};

// ---- device helpers -------------------------------------------------------
#ifdef __CUDACC__
// streaming (read-once) global loads: bypass L1 allocation
__device__ __forceinline__ float2 ldg_stream_f2(const float2 *p)
{
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream_u32(const uint32_t *p)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_f32(float *p, float v)
{
    asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v));
}
__device__ __forceinline__ void stg_stream_f2(float2 *p, float2 v)
{
    asm volatile("st.global.cs.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v.x), "f"(v.y));
}

// (float)s / 32767f, correctly rounded, without the generic division.  s/32767 = s*2^-15 repeated
// with period 15 bits, so it never comes within 2^-39 (relative) of a float rounding boundary,
// and 1/32767 split as r_hi + r_lo (two floats, 48 bits) gives the correctly rounded quotient
// in one multiply and one FMA: q = fma(s, r_hi, s*r_lo).  Checked exhaustively against IEEE
// division for all 65536 inputs (tests/test_oracle.py).
__device__ __forceinline__ float s16_over_32767(float x)
{
    const float r_hi = 3.0518509447574615e-05f, r_lo = 2.8422576792141996e-14f;
    return __fmaf_rn(x, r_hi, __fmul_rn(x, r_lo));
}

// One s16le (I, Q) word of the IRawHandler contract to the floats JavaAudio hands its
// IAudioHandlers (JavaAudio.java:281-288): s += (short)ic (16-bit wrap); (float)s/(float)Short.MAX_VALUE
__device__ __forceinline__ float2 s16_iq_to_float2(uint32_t w, int ic, int qc)
{
    const short si = (short)((int)(w & 0xffffu) + ic);
    const short sq = (short)((int)(w >> 16) + qc);
    return make_float2(s16_over_32767((float)si), s16_over_32767((float)sq));
}
#endif

}  // namespace jsdr
