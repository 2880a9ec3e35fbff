// mac64.cu -- throughput of the 32x32->64 multiply-accumulate the RNS basis conversion is made of
// (acc += (u64) y * m, one IMAD.WIDE.U32 with a 64-bit addend; m = m[j][i] of a kernel-parameter
// matrix with a warp-uniform row j that changes every iteration, as in rns_conv_kernel), over the
// whole GPU: 256-thread blocks, grid 8 blocks per SM, 16 terms into 4 independent accumulators
// per thread with distinct y per accumulator (the V = 4 columns of the kernel at S = 16).  Prints one JSON line with the
// multiply-accumulates per second; tools/bench_rns_conv.py compiles and runs it in the same call
// as the conversion rows, as the integer-multiplier ceiling they are compared with.
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o mac64 mac64.cu && ./mac64
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

constexpr int kTerms = 16, kAcc = 4, kRows = 32, kIters = 4096;

struct Mult {
    uint32_t m[kRows][kTerms];
};

__global__ void __launch_bounds__(256) mac_kernel(uint64_t *out, uint32_t seed, const __grid_constant__ Mult p) {
    uint32_t y[kAcc][kTerms];
#pragma unroll
    for (int e = 0; e < kAcc; e++) {
#pragma unroll
        for (int i = 0; i < kTerms; i++) y[e][i] = (threadIdx.x * 2654435761u + (e * kTerms + i) * 40503u + seed) >> 2;
    }
    uint64_t acc[kAcc] = {};
#pragma unroll 1
    for (int it = 0; it < kIters; it++) {
#pragma unroll
        for (int i = 0; i < kTerms; i++) {
#pragma unroll
            for (int e = 0; e < kAcc; e++) {
                acc[e] += (uint64_t) y[e][i] * p.m[it & (kRows - 1)][i];
            }
        }
    }
    uint64_t r = 0;
#pragma unroll
    for (int e = 0; e < kAcc; e++) r ^= acc[e];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

#define CHECK(x)                                                                    \
    do {                                                                            \
        cudaError_t e = (x);                                                        \
        if (e != cudaSuccess) {                                                     \
            fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e));                 \
            return 1;                                                               \
        }                                                                           \
    } while (0)

int main() {
    cudaDeviceProp prop;
    CHECK(cudaGetDeviceProperties(&prop, 0));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    uint64_t *d_out;
    CHECK(cudaMalloc(&d_out, sizeof(uint64_t) * blocks * threads));
    Mult p;
    for (int j = 0; j < kRows; j++) {
        for (int i = 0; i < kTerms; i++) p.m[j][i] = 0x3fffffffu - 977u * (j * kTerms + i);
    }
    cudaEvent_t a, b;
    CHECK(cudaEventCreate(&a));
    CHECK(cudaEventCreate(&b));
    for (int w = 0; w < 3; w++) mac_kernel<<<blocks, threads>>>(d_out, w, p);
    CHECK(cudaEventRecord(a));
    const int reps = 10;
    for (int r = 0; r < reps; r++) mac_kernel<<<blocks, threads>>>(d_out, r, p);
    CHECK(cudaEventRecord(b));
    CHECK(cudaEventSynchronize(b));
    CHECK(cudaGetLastError());
    float ms = 0;
    CHECK(cudaEventElapsedTime(&ms, a, b));
    const double macs = (double) reps * blocks * threads * kIters * kTerms * kAcc;
    printf("{\"mac64_per_s\": %.6e, \"ms\": %.4f, \"blocks\": %d, \"threads\": %d, \"sms\": %d}\n",
           macs / (ms * 1e-3), ms / reps, blocks, threads, prop.multiProcessorCount);
    CHECK(cudaFree(d_out));
    return 0;
}
