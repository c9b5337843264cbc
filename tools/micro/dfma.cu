// Micro-benchmark: device-wide DFMA (fp64 fused multiply-add) rate on sm_100a -- the FP64 ceiling the double SSIM
// kernels (csrc/ssim_f64.cu) are bound by.  Every thread runs 16 independent DFMA chains; the rate is timed with CUDA
// events over a grid of many waves.  Prints the card name, SM clock, and DFMA/s (1 DFMA = 2 FLOP).
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o dfma dfma.cu && ./dfma
#include <cstdio>
#include <cuda_runtime.h>

constexpr int kChains = 16;

__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double s) {
    double a[kChains];
#pragma unroll
    for (int i = 0; i < kChains; ++i) a[i] = threadIdx.x + i;
    const double b = s, c = s * 0.5;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int i = 0; i < kChains; ++i) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(a[i]) : "d"(b), "d"(c));
    }
    double t = 0;
#pragma unroll
    for (int i = 0; i < kChains; ++i) t += a[i];
    if (t == 12345.678) out[0] = t;   // never true: keeps the chains alive
}

int main() {
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    int clock_khz = 0;
    cudaDeviceGetAttribute(&clock_khz, cudaDevAttrClockRate, 0);
    double* out;
    cudaMalloc(&out, sizeof(double));
    const int threads = 256, iters = 4096;
    const int blocks = prop.multiProcessorCount * 8 * 4;   // 8 resident CTAs of 256 per SM, 4 waves
    dfma_kernel<<<blocks, threads>>>(out, 16, 0.999);      // warm-up
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        dfma_kernel<<<blocks, threads>>>(out, iters, 0.999);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    const double dfma = (double)blocks * threads * iters * 8 * kChains;
    const double rate = dfma / (best * 1e-3);
    printf("{\"device\": \"%s\", \"sms\": %d, \"max_sm_clock_mhz\": %d, \"best_ms\": %.3f, \"dfma_per_s\": %.4e, "
           "\"fp64_tflops\": %.2f, \"dfma_per_clk_per_sm_at_max_clock\": %.1f}\n",
           prop.name, prop.multiProcessorCount, clock_khz / 1000, best, rate, 2 * rate / 1e12,
           rate / (prop.multiProcessorCount * (clock_khz * 1e3)));
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
    cudaFree(out);
    return 0;
}
