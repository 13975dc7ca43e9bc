// stream_mix.cu — streaming bandwidth of a B200 by read : write mix. The Gaussian chain kernel (config 2) reads 12 B and
// writes 52 B per state variable (forward recursion 4 : 24, backward 12 : 24 ... 8 : 28), the copy that defines the roofline
// peak is 1 : 1; the Potts sweep (config 4) reads 5 and writes 4 16-byte vectors per lane.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o stream_mix stream_mix.cu
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cuda_runtime.h>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)
// every thread reads R float2 planes and writes W float2 planes at its element, grid-stride over n elements (8 bytes each)
template <int R, int W>
__global__ void k(const float2* __restrict__ src, float2* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float2 acc = make_float2(1.0f, 2.0f);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float2 v = __ldcs(src + (size_t)r * n + i);
            acc.x += v.x;
            acc.y += v.y;
        }
#pragma unroll
        for (int w = 0; w < W; ++w) __stcs(dst + (size_t)w * n + i, make_float2(acc.x + w, acc.y));
    }
}
// the same with 16-byte elements (two chains per thread would give the chain kernel these)
template <int R, int W>
__global__ void k16(const float4* __restrict__ src, float4* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float4 acc = make_float4(1.0f, 2.0f, 3.0f, 4.0f);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float4 v = __ldcs(src + (size_t)r * n + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
#pragma unroll
        for (int w = 0; w < W; ++w) __stcs(dst + (size_t)w * n + i, make_float4(acc.x + w, acc.y, acc.z, acc.w));
    }
}
int main() {
    const size_t n = (size_t)64 << 20;  // 64 Mi elements of 8 bytes = 512 MiB per plane (the chain planes: 65,536 x 1,024 x 8 B)
    float2 *src, *dst;
    CK(cudaMalloc(&src, n * 8 * 5)); CK(cudaMalloc(&dst, n * 8 * 7));
    CK(cudaMemset(src, 0, n * 8 * 5)); CK(cudaMemset(dst, 0, n * 8 * 7));
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    auto run = [&](const char* name, auto launch, double bytes) {
        for (int i = 0; i < 2; ++i) launch();
        CK(cudaDeviceSynchronize());
        cudaEventRecord(e0);
        const int reps = 5;
        for (int i = 0; i < reps; ++i) launch();
        cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
        printf("%-46s %7.3f ms  %7.1f GB/s\n", name, ms, bytes / ms * 1e-6);
    };
    const int grid = 148 * 16, blk = 256;
    run("read 1 : write 1 (copy)", [&] { k<1, 1><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 2);
    run("read 4 : write 4", [&] { k<4, 4><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 8);
    run("read 1 : write 3", [&] { k<1, 3><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 4);
    run("read 1 : write 4 (chains: 12 B : 52 B)", [&] { k<1, 4><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 5);
    run("read 1 : write 6", [&] { k<1, 6><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 7);
    run("read 2 : write 3 (backward recursion)", [&] { k<2, 3><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 5);
    run("read 0 : write 4 (write only)", [&] { k<0, 4><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 4);
    run("read 4 : write 1", [&] { k<4, 1><<<grid, blk>>>(src, dst, n); }, n * 8.0 * 5);
    const size_t n16 = n / 2;
    const float4* s16 = reinterpret_cast<const float4*>(src);
    float4* d16 = reinterpret_cast<float4*>(dst);
    run("16-byte elements, read 1 : write 1 (copy)", [&] { k16<1, 1><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 2);
    run("16-byte elements, read 4 : write 4", [&] { k16<4, 4><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 8);
    run("16-byte elements, read 1 : write 4", [&] { k16<1, 4><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 5);
    run("16-byte elements, read 2 : write 3", [&] { k16<2, 3><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 5);
    run("16-byte elements, read 1 : write 6", [&] { k16<1, 6><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 7);
    run("16-byte elements, read 5 : write 4 (Potts sweep)", [&] { k16<5, 4><<<grid, blk>>>(s16, d16, n16); }, n16 * 16.0 * 9);
    return 0;
}
