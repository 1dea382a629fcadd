// Rate of the legacy warp-level tensor path on B200: mma.sync.m16n8k8 TF32 (SASS HMMA.1688.F32.TF32), the instruction of the
// AFE_BATCH_MMA_PHASE2 variant of k_fused_mfcc (removed; its code is in commit c5ab662). 8 independent accumulator chains per
// warp, 1 / 2 / 4 warps per scheduler.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o hmma hmma.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
constexpr int ITERS = 4096, CHAINS = 8;
__global__ void __launch_bounds__(512) k(float *out, uint32_t seed)
{
    float c[CHAINS][4];
    for (int i = 0; i < CHAINS; i++) for (int q = 0; q < 4; q++) c[i][q] = 0.f;
    uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, b0 = a0 * 11, b1 = a0 * 13;
    a0 &= 0x3f7fe000u; a1 &= 0x3f7fe000u; a2 &= 0x3f7fe000u; a3 &= 0x3f7fe000u; b0 &= 0x3f7fe000u; b1 &= 0x3f7fe000u;
    for (int it = 0; it < ITERS; it++) {
#pragma unroll
        for (int i = 0; i < CHAINS; i++)
            asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                         : "+f"(c[i][0]), "+f"(c[i][1]), "+f"(c[i][2]), "+f"(c[i][3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
    float s = 0.f;
    for (int i = 0; i < CHAINS; i++) for (int q = 0; q < 4; q++) s += c[i][q];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
int main()
{
    float *d; cudaMalloc(&d, 148 * 512 * 4);
    int clk; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
    for (int w = 1; w <= 4; w *= 2) {
        cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
        k<<<148, 128 * w>>>(d, 1); cudaDeviceSynchronize();
        cudaEventRecord(e0); k<<<148, 128 * w>>>(d, 1); cudaEventRecord(e1); cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        const double cyc = ms * 1e-3 * clk * 1e3 / ((double)ITERS * CHAINS * w);   // per scheduler
        printf("%d warp(s) per scheduler: %.2f cycles per HMMA.1688.F32.TF32 per scheduler = %.1f dense TF32 TFLOP/s on 148 SMs\n", w, cyc,
               2.0 * 16 * 8 * 8 / cyc * 4 * 148 * clk * 1e3 / 1e12);
    }
    printf("status: %s\n", cudaGetErrorString(cudaDeviceSynchronize()));
    return 0;
}
