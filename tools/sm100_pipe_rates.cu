// Per-SM issue rates of the SIMT instructions the bf16x3 GVP epilogues are made of (sm_100a): FFMA, FFMA2, FADD2,
// MUFU ex2 / rcp alone, and MUFU ex2 mixed with FFMA2.  One CTA of 1024 threads per SM, NCH independent dependency
// chains per thread (enough to cover every pipe's latency); SM cycles from clock64 around the loop, wall time from
// CUDA events.  Built and run by tools/sm100_pipe_rates.py.
#include <cstdio>
#include <cuda_runtime.h>

constexpr int NCH = 8, ITERS = 4096, THREADS = 1024;

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float ex2(float x) { float y; asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp(float x) { float y; asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

enum Op { FFMA, FFMA2, FADD2, EX2, RCP, EX2_FFMA2x2, EX2_FFMA2x4, N_OPS };
static const char* kName[N_OPS] = {"FFMA", "FFMA2", "FADD2", "MUFU.EX2", "MUFU.RCP (+ FADD)", "MUFU.EX2 + 2 FFMA2", "MUFU.EX2 + 4 FFMA2"};
// instructions of each kind per chain per iteration: {FP32-pipe instructions, MUFU instructions}
static const int kFma[N_OPS] = {1, 1, 1, 0, 1, 2, 4}, kMufu[N_OPS] = {0, 0, 0, 1, 1, 1, 1};

template <Op OP>
__global__ void __launch_bounds__(THREADS, 1) pipe_kernel(float* out, long long* cycles, float seed) {
    float s[NCH];
    float2 p[NCH];
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
        s[i] = seed + 1e-3f * (threadIdx.x + i);
        p[i] = make_float2(s[i], 0.5f * s[i]);
    }
    const float2 m = make_float2(0.999f, 0.998f), c = make_float2(1e-3f, 2e-3f);
    __syncthreads();
    const long long t0 = clock64();
    for (int it = 0; it < ITERS; ++it) {
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
            if constexpr (OP == FFMA) s[i] = fmaf(s[i], 0.999f, 1e-3f);
            if constexpr (OP == FFMA2) p[i] = ffma2(p[i], m, c);
            if constexpr (OP == FADD2) p[i] = __fadd2_rn(p[i], c);
            if constexpr (OP == EX2) s[i] = ex2(s[i]);
            if constexpr (OP == RCP) s[i] = rcp(s[i] + 1.0f);   // (+1: ptxas folds rcp(rcp(x)) back to x)
            if constexpr (OP == EX2_FFMA2x2 || OP == EX2_FFMA2x4) {
                s[i] = ex2(s[i]);
                p[i] = ffma2(p[i], m, c);
                p[i] = ffma2(p[i], m, c);
                if constexpr (OP == EX2_FFMA2x4) { p[i] = ffma2(p[i], m, c); p[i] = ffma2(p[i], m, c); }
            }
        }
    }
    __syncthreads();
    const long long t1 = clock64();
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < NCH; ++i) acc += s[i] + p[i].x + p[i].y;
    out[blockIdx.x * THREADS + threadIdx.x] = acc;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

template <Op OP>
static void run(int n_sm, float* out, long long* cyc_d) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    pipe_kernel<OP><<<n_sm, THREADS>>>(out, cyc_d, 0.5f);      // warm-up
    cudaEventRecord(e0);
    pipe_kernel<OP><<<n_sm, THREADS>>>(out, cyc_d, 0.5f);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    long long* cyc = new long long[n_sm];
    cudaMemcpy(cyc, cyc_d, sizeof(long long) * n_sm, cudaMemcpyDeviceToHost);
    long long cmax = 0;
    for (int i = 0; i < n_sm; ++i) cmax = cyc[i] > cmax ? cyc[i] : cmax;
    delete[] cyc;
    const double per_sm = double(THREADS) * ITERS * NCH;      // chain-iterations per SM
    const double fma_ipc = per_sm * kFma[OP] / cmax, mufu_ipc = per_sm * kMufu[OP] / cmax;   // thread-instructions per clock
    printf("%-20s  fp32-pipe %6.1f instr/clk/SM  mufu %5.1f instr/clk/SM  (%lld cycles, %.3f ms, %.0f MHz effective)\n",
           kName[OP], fma_ipc, mufu_ipc, cmax, ms, cmax / (ms * 1e3));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
}

int main() {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, 0) != cudaSuccess) { fprintf(stderr, "no CUDA device\n"); return 1; }
    const int n_sm = prop.multiProcessorCount;
    printf("device %s, %d SMs; one %d-thread CTA per SM, %d chains x %d iterations per thread\n", prop.name, n_sm, THREADS,
           NCH, ITERS);
    float* out;
    long long* cyc;
    cudaMalloc(&out, sizeof(float) * n_sm * THREADS);
    cudaMalloc(&cyc, sizeof(long long) * n_sm);
    run<FFMA>(n_sm, out, cyc);
    run<FFMA2>(n_sm, out, cyc);
    run<FADD2>(n_sm, out, cyc);
    run<EX2>(n_sm, out, cyc);
    run<RCP>(n_sm, out, cyc);
    run<EX2_FFMA2x2>(n_sm, out, cyc);
    run<EX2_FFMA2x4>(n_sm, out, cyc);
    const cudaError_t err = cudaDeviceSynchronize();
    cudaFree(out);
    cudaFree(cyc);
    if (err != cudaSuccess) { fprintf(stderr, "CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
    return 0;
}
