// microbench.cu — the handful of sm_100a numbers DESIGN.md's arguments lean on, measured on the
// device they are about (B200): dependent-chain latencies of the phase replay's instructions,
// per-SM throughput of the pipes the two data kernels sit on, and the rate of small bulk copies.
// Not part of the library.  Build and run (on a GPU box):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o gpurun_out/microbench tools/microbench.cu
//   gpurun_out/microbench > gpurun_out/microbench.txt
// Output is committed as profiles/r02_microbench.txt.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 1; } } while (0)

constexpr int kIters = 4096;

// ---------------------------------------------------------------- latency (one warp, one chain)
__global__ void k_lat_dadd(double *out, long long *cyc, double inc)
{
    double p = out[threadIdx.x];
    long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < kIters; i++) p = __dadd_rn(p, inc);
    long long t1 = clock64();
    out[threadIdx.x] = p;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

__global__ void k_lat_fadd(float *out, long long *cyc, float inc)
{
    float p = out[threadIdx.x];
    long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < kIters; i++) p = __fadd_rn(p, inc);
    long long t1 = clock64();
    out[threadIdx.x] = p;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

// the phase replay's pair: two reference steps in three dependent additions, addends selected by
// two comparisons of the phase before the pair (bpsk.cu phase_step2)
__global__ void k_lat_pair(double *out, long long *cyc, double inc, double th1, double th2)
{
    double p = out[threadIdx.x];
    const double twopi = 6.283185307179586;
    long long t0 = clock64();
#pragma unroll 8
    for (int i = 0; i < kIters; i++) {
        const bool m1 = p > th1, m2 = p > th2;
        const double s2 = m1 ? -twopi : inc;
        const double s3 = m1 ? inc : (m2 ? -twopi : 0.0);
        p = __dadd_rn(__dadd_rn(__dadd_rn(p, inc), s2), s3);
    }
    long long t1 = clock64();
    out[threadIdx.x] = p;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

// float -> double -> multiply -> float, the AM detector's division step (demod_fir.cu k_detect)
__global__ void k_lat_f2f(float *out, long long *cyc, double r)
{
    float a = out[threadIdx.x];
    long long t0 = clock64();
#pragma unroll 8
    for (int i = 0; i < kIters; i++) a = __double2float_rn(__dmul_rn((double)a, r));
    long long t1 = clock64();
    out[threadIdx.x] = a;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

__global__ void k_lat_fdiv(float *out, long long *cyc, float d)
{
    float a = out[threadIdx.x];
    long long t0 = clock64();
#pragma unroll 8
    for (int i = 0; i < kIters; i++) a = __fdiv_rn(a, d);
    long long t1 = clock64();
    out[threadIdx.x] = a;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

// ---------------------------------------------------------------- throughput (whole SM, 8 chains per thread)
template <int OP>
__global__ void __launch_bounds__(1024) k_tput(double *out, long long *cyc, double c)
{
    double a[8];
    float2 f[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        a[k] = out[threadIdx.x] + k;
        f[k] = make_float2((float)a[k], (float)a[k] + 1.f);
    }
    // the interval is first start to last finish over the CTA's warps: with a fixed-latency pipe the
    // scheduler runs some warps well ahead of others, so one warp's own clock pair under-reports
    __shared__ unsigned long long s_t0, s_t1;
    if (threadIdx.x == 0) { s_t0 = ~0ull; s_t1 = 0; }
    __syncthreads();
    long long t0 = clock64();
#pragma unroll 4
    for (int i = 0; i < kIters / 4; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            if (OP == 0) a[k] = __dadd_rn(a[k], c);
            if (OP == 1) a[k] = __dmul_rn(a[k], c);
            if (OP == 2) {
                unsigned long long r, x = *reinterpret_cast<unsigned long long *>(&f[k]);
                asm volatile("fma.rn.f32x2 %0, %1, %1, %1;" : "=l"(r) : "l"(x));
                f[k] = *reinterpret_cast<float2 *>(&r);
            }
            if (OP == 3) a[k] = (double)(__double2float_rn(a[k]) + 1.0f);   // F2F.F32.F64 + FADD + F2F.F64.F32
            if (OP == 4) f[k].x = __shfl_xor_sync(0xffffffffu, f[k].x, 1);
            if (OP == 5) asm volatile("fma.rn.f32 %0, %0, %1, %0;" : "+f"(f[k].x) : "f"(f[k].y));
            if (OP == 6) {                                       // half packed, half scalar: do the two FMA pipes overlap?
                if (k & 1) {
                    asm volatile("fma.rn.f32 %0, %0, %1, %0;" : "+f"(f[k].x) : "f"(f[k].y));
                } else {
                    unsigned long long r, x = *reinterpret_cast<unsigned long long *>(&f[k]);
                    asm volatile("fma.rn.f32x2 %0, %1, %1, %1;" : "=l"(r) : "l"(x));
                    f[k] = *reinterpret_cast<float2 *>(&r);
                }
            }
            if (OP == 7) {                                       // two packed to one scalar
                if (k % 3 == 2) {
                    asm volatile("fma.rn.f32 %0, %0, %1, %0;" : "+f"(f[k].x) : "f"(f[k].y));
                } else {
                    unsigned long long r, x = *reinterpret_cast<unsigned long long *>(&f[k]);
                    asm volatile("fma.rn.f32x2 %0, %1, %1, %1;" : "=l"(r) : "l"(x));
                    f[k] = *reinterpret_cast<float2 *>(&r);
                }
            }
            if (OP == 8) {                                       // packed add (FADD2)
                unsigned long long r, x = *reinterpret_cast<unsigned long long *>(&f[k]);
                asm volatile("add.rn.f32x2 %0, %1, %1;" : "=l"(r) : "l"(x));
                f[k] = *reinterpret_cast<float2 *>(&r);
            }
            if (OP == 9) asm volatile("add.rn.f32 %0, %0, %1;" : "+f"(f[k].x) : "f"(f[k].y));
        }
    }
    long long t1 = clock64();
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&s_t0, (unsigned long long)t0);
        atomicMax(&s_t1, (unsigned long long)t1);
    }
    __syncthreads();
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k] + f[k].x + f[k].y;
    out[threadIdx.x] = s;
    if (threadIdx.x == 0) cyc[blockIdx.x] = (long long)(s_t1 - s_t0);
}

// ---------------------------------------------------------------- small bulk copies
// every lane copies `bytes` from its own row with cp.async.bulk onto one mbarrier per warp, waits,
// repeats: the staging pattern of the period-ring decimator that was measured and dropped (DESIGN.md §9)
__global__ void __launch_bounds__(512) k_bulk(const uint32_t *in, long long row_stride, int bytes, int reps, long long *cyc,
                                              unsigned *sink)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned base = (unsigned)__cvta_generic_to_shared(smem) + warp * (32 * 128 + 16);
    const unsigned mbar = base + 32 * 128;
    if (lane == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    const uint32_t *src = in + ((long long)blockIdx.x * 16 + warp) * 32 * row_stride + (long long)lane * row_stride;
    long long t0 = clock64();
    for (int r = 0; r < reps; r++) {
        if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(32u * bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(base + lane * 128), "l"(src + (long long)r * (bytes / 4)), "r"((unsigned)bytes), "r"(mbar) : "memory");
        asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@!p bra W_%=;\n\t}"
                     ::"r"(mbar), "r"((unsigned)(r & 1)) : "memory");
        __syncwarp();
    }
    long long t1 = clock64();
    if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
    if (sink) sink[blockIdx.x * blockDim.x + threadIdx.x] = *reinterpret_cast<volatile unsigned *>(smem + warp * (32 * 128 + 16) + lane * 128);
}

int main()
{
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("# %s, %d SMs, sm_%d%d, SM clock %.0f MHz (max)\n", prop.name, prop.multiProcessorCount, prop.major, prop.minor, prop.clockRate / 1000.0);
    double *d_out;
    float *d_fout;
    long long *d_cyc, h_cyc[1024];
    CK(cudaMalloc(&d_out, 1024 * sizeof(double)));
    CK(cudaMalloc(&d_fout, 1024 * sizeof(float)));
    CK(cudaMalloc(&d_cyc, 1024 * sizeof(long long)));
    CK(cudaMemset(d_out, 0, 1024 * sizeof(double)));
    CK(cudaMemset(d_fout, 0, 1024 * sizeof(float)));
    auto cyc0 = [&]() { cudaMemcpy(h_cyc, d_cyc, sizeof(long long), cudaMemcpyDeviceToHost); return (double)h_cyc[0]; };

    printf("## dependent-chain latency, one warp (cycles per operation)\n");
    for (int rep = 0; rep < 2; rep++) k_lat_dadd<<<1, 32>>>(d_out, d_cyc, 1e-3);
    CK(cudaDeviceSynchronize());
    printf("DADD                         %6.2f\n", cyc0() / kIters);
    for (int rep = 0; rep < 2; rep++) k_lat_fadd<<<1, 32>>>(d_fout, d_cyc, 1e-3f);
    CK(cudaDeviceSynchronize());
    printf("FADD                         %6.2f\n", cyc0() / kIters);
    CK(cudaMemset(d_out, 0, 1024 * sizeof(double)));
    for (int rep = 0; rep < 2; rep++) k_lat_pair<<<1, 32>>>(d_out, d_cyc, 1.4726215563702154, 4.810563750809371, 3.3379421944391554);
    CK(cudaDeviceSynchronize());
    printf("phase pair (2 steps: 3 DADD + 2 DSETP + 6 FSEL), 1 warp/SM   %6.2f cycles per pair\n", cyc0() / kIters);
    for (int w = 2; w <= 4; w++) {                                   // w warps per sub-partition
        CK(cudaMemset(d_out, 0, 1024 * sizeof(double)));
        for (int rep = 0; rep < 2; rep++) k_lat_pair<<<1, 128 * w>>>(d_out, d_cyc, 1.4726215563702154, 4.810563750809371, 3.3379421944391554);
        CK(cudaDeviceSynchronize());
        printf("phase pair, %d warps per sub-partition                        %6.2f cycles per pair\n", w, cyc0() / kIters);
    }
    CK(cudaMemset(d_fout, 0x3f, 1024 * sizeof(float)));
    for (int rep = 0; rep < 2; rep++) k_lat_f2f<<<1, 32>>>(d_fout, d_cyc, 0.999999);
    CK(cudaDeviceSynchronize());
    printf("F2F.F64.F32 + DMUL + F2F.F32.F64                             %6.2f cycles per step\n", cyc0() / kIters);
    for (int rep = 0; rep < 2; rep++) k_lat_fdiv<<<1, 32>>>(d_fout, d_cyc, 1.0000001f);
    CK(cudaDeviceSynchronize());
    printf("__fdiv_rn (IEEE float division)                              %6.2f cycles per step\n", cyc0() / kIters);

    printf("## throughput, one SM with 1024 threads, 8 independent chains per thread (thread-operations per cycle per SM)\n");
    const char *names[] = {"DADD", "DMUL", "FFMA2 (packed: 2 FMA per lane)", "F2F.F32.F64 + FADD + F2F.F64.F32", "SHFL.BFLY", "FFMA",
                           "4 FFMA2 + 4 FFMA interleaved", "5-6 FFMA2 + 2-3 FFMA interleaved", "FADD2 (packed)", "FADD"};
    for (int op = 0; op < 10; op++) {
        for (int rep = 0; rep < 2; rep++) {
            switch (op) {
            case 0: k_tput<0><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 1: k_tput<1><<<1, 1024>>>(d_out, d_cyc, 1.0000001); break;
            case 2: k_tput<2><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 3: k_tput<3><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 4: k_tput<4><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 5: k_tput<5><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 6: k_tput<6><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 7: k_tput<7><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            case 8: k_tput<8><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            default: k_tput<9><<<1, 1024>>>(d_out, d_cyc, 1e-3); break;
            }
        }
        CK(cudaDeviceSynchronize());
        const double ops = 1024.0 * 8 * (kIters / 4);               // thread-operations in the timed loop
        const double c = cyc0();
        printf("%-34s %8.1f per cycle per SM   (%.0f cycles)\n", names[op], ops / c, c);
    }

    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int th : {32, 128, 512, 1024}) {                               // FFMA again at several occupancies (raw cycles + event time)
        k_tput<5><<<1, th>>>(d_out, d_cyc, 1e-3);
        cudaEventRecord(e0);
        k_tput<5><<<1, th>>>(d_out, d_cyc, 1e-3);
        cudaEventRecord(e1);
        CK(cudaDeviceSynchronize());
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double c = cyc0();
        printf("FFMA, %4d threads: %8.0f cycles (kernel %.1f us by events) for %d FFMA per thread = %.2f warp-instructions per cycle per sub-partition\n", th, c,
               ms * 1e3, 8 * (kIters / 4), (th / 32) * 8.0 * (kIters / 4) / c / (th >= 128 ? 4 : 1));
    }
    for (int th : {128, 1024}) {
        k_tput<0><<<1, th>>>(d_out, d_cyc, 1e-3);
        cudaEventRecord(e0);
        k_tput<0><<<1, th>>>(d_out, d_cyc, 1e-3);
        cudaEventRecord(e1);
        CK(cudaDeviceSynchronize());
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        printf("DADD, %4d threads: %8.0f cycles (kernel %.1f us by events)\n", th, cyc0(), ms * 1e3);
    }
    printf("## small bulk copies: every lane of 16 warps per SM copies B bytes of its own row (cp.async.bulk + mbarrier per warp), waits, repeats\n");
    const int reps = 512;
    const long long row_stride = 1 << 16;                              // words between rows (256 KB)
    uint32_t *d_in;
    const size_t in_words = (size_t)prop.multiProcessorCount * 16 * 32 * row_stride;
    if (cudaMalloc(&d_in, in_words * 4) == cudaSuccess) {
        CK(cudaMemset(d_in, 1, in_words * 4));
        const size_t smem = 16 * (32 * 128 + 16);
        CK(cudaFuncSetAttribute(k_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int bytes : {16, 80, 128}) {
            for (int grid : {1, prop.multiProcessorCount}) {
                for (int rep = 0; rep < 2; rep++) k_bulk<<<grid, 512, smem>>>(d_in, row_stride, bytes, reps, d_cyc, nullptr);
                CK(cudaDeviceSynchronize());
                cudaMemcpy(h_cyc, d_cyc, sizeof(long long) * grid, cudaMemcpyDeviceToHost);
                double mx = 0;
                for (int i = 0; i < grid; i++) mx = h_cyc[i] > mx ? h_cyc[i] : mx;
                printf("B = %3d, %3d SMs busy: %7.1f cycles per round of 512 copies per SM  = one copy per %5.2f cycles per SM, %6.1f GB/s per SM at %.0f MHz\n",
                       bytes, grid, mx / reps, mx / reps / 512.0, 512.0 * bytes / (mx / reps) * prop.clockRate * 1e-6, prop.clockRate / 1000.0);
            }
        }
        cudaFree(d_in);
    } else {
        printf("(not enough memory for the bulk-copy test)\n");
        cudaGetLastError();
    }
    return 0;
}
