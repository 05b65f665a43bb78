// popc_peak.cu -- 32-bit POPC issue rate of this GPU, the denominator of the pair-count kernel's rate
// (pair_counts_kernel: C = popc(H . H^T), bound by POPC issue; bench_configs.py cooccur).
//
// Every thread runs 8 independent chains of acc += __popc(x ^ k), the inner loop of pair_counts_kernel
// (LOP3 + POPC + IADD per word pair), on registers only: nothing touches memory until the sums are stored.
// 8 CTAs of 256 threads per SM, best of several ~50 ms launches.
//
// Prints one JSON line: {"popc_per_s": .., "popc_per_clk_sm": .. (at the device's reported max SM clock), ...}.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o bench_micro/popc_peak bench_micro/popc_peak.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

__global__ void __launch_bounds__(256) popc_kernel(uint32_t seed, int iters, uint32_t *out) {
    uint32_t x[8], acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { x[j] = seed * (threadIdx.x + 17 * j + 1) + blockIdx.x; acc[j] = 0; }
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++)
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] += __popc(x[j] ^ (uint32_t) (i * 16 + u));
    }
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s += acc[j];
    out[(size_t) blockIdx.x * blockDim.x + threadIdx.x] = s;
}

int main() {
    int dev = 0, sms = 0, clk_khz = 0;
    CK(cudaSetDevice(dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CK(cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, dev));
    const int blocks = sms * 8, threads = 256;
    uint32_t *out = nullptr;
    CK(cudaMalloc(&out, (size_t) blocks * threads * 4));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    int iters = 256;
    popc_kernel<<<blocks, threads>>>(1u, iters, out);   // warm-up
    CK(cudaDeviceSynchronize());
    // size one launch to ~50 ms
    CK(cudaEventRecord(a));
    popc_kernel<<<blocks, threads>>>(2u, iters, out);
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    iters = (int) (iters * 50.0 / (ms > 0.01f ? ms : 0.01f));
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(a));
        popc_kernel<<<blocks, threads>>>(3u + rep, iters, out);
        CK(cudaEventRecord(b));
        CK(cudaEventSynchronize(b));
        CK(cudaEventElapsedTime(&ms, a, b));
        const double popc = (double) blocks * threads * iters * 16.0 * 8.0;
        if (popc / (ms * 1e-3) > best) best = popc / (ms * 1e-3);
    }
    CK(cudaGetLastError());
    printf("{\"popc_per_s\": %.6e, \"popc_per_clk_sm\": %.3f, \"sms\": %d, \"max_sm_clock_mhz\": %.0f, \"iters\": %d}\n", best,
           best / sms / (clk_khz * 1e3), sms, clk_khz / 1e3, iters);
    CK(cudaFree(out));
    return 0;
}
