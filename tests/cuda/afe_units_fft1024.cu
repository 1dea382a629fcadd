// Device unit harness for the 1024-point in-register FFT + magnitude (afe_fft.cuh) as the fused kernel K1 runs it:
// fft_frame_mag<1024, NZ, true, false, PRE>, one frame per warp call. tests/test_fft1024.py compiles this file with the
// library's nvcc flags into a temporary directory and calls the extern "C" entry point through ctypes. It copies with
// cudaMalloc / cudaMemcpy and returns 0, or the cudaError_t of the first failing call.
#include <cuda_runtime.h>
#include <stdint.h>

#include "afe_fft.cuh"

using namespace afe;

#define UNIT_CUDA(expr)                                                                                                 \
    do {                                                                                                                \
        cudaError_t _e = (expr);                                                                                        \
        if (_e != cudaSuccess) return (int)_e;                                                                          \
    } while (0)

// frame f's samples start at pcm + f * 1024 (readable past W), its row at mag + f * 513
template <int NZ, bool PRE>
__global__ void __launch_bounds__(128) k_unit_fft1024(const int16_t *__restrict__ pcm, const float2 *window2, const float2 *tw_a,
                                                      const float2 *tw_p, float *__restrict__ mag, int frames, float pre)
{
    using C = dev::FftCfg<1024>;
    __shared__ float2 scratch[4 * C::SCR];
    __shared__ float s_dump[C::BINS + 3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    dev::LaneConsts<1024, NZ> lc;
    dev::load_lane_consts<1024, NZ>(lc, window2, tw_a, tw_p, lane);
    for (int f0 = blockIdx.x * 4; f0 < frames; f0 += gridDim.x * 4) {
        const int f = f0 + warp;
        const bool act = f < frames;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(pcm + (long long)(act ? f : frames - 1) * 1024);
        dev::fft_frame_mag<1024, NZ, true, false, PRE>(words, lc, scratch + warp * C::SCR,
                                                       act ? mag + (long long)f * C::BINS : s_dump, lane, pre);
    }
}

// pcm: frames * 1024 int16; window2: 512 float2; tw_a: 32 * 16 float2; tw_p: 256 float2; mag: frames * 513 (|2X|)
extern "C" int afe_units_fft1024_mag(int nz, int with_pre, const int16_t *h_pcm, int frames, const float *h_window2,
                                     const float *h_tw_a, const float *h_tw_p, float pre, float *h_mag)
{
    if ((nz != 13 && nz != 16) || frames < 1) return (int)cudaErrorInvalidValue;
    int16_t *pcm = nullptr;
    float2 *w2 = nullptr, *ta = nullptr, *tp = nullptr;
    float *mag = nullptr;
    UNIT_CUDA(cudaMalloc(&pcm, sizeof(int16_t) * frames * 1024));
    UNIT_CUDA(cudaMalloc(&w2, sizeof(float2) * 512));
    UNIT_CUDA(cudaMalloc(&ta, sizeof(float2) * 512));
    UNIT_CUDA(cudaMalloc(&tp, sizeof(float2) * 256));
    UNIT_CUDA(cudaMalloc(&mag, sizeof(float) * frames * 513));
    UNIT_CUDA(cudaMemcpy(pcm, h_pcm, sizeof(int16_t) * frames * 1024, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(w2, h_window2, sizeof(float2) * 512, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(ta, h_tw_a, sizeof(float2) * 512, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(tp, h_tw_p, sizeof(float2) * 256, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemset(mag, 0xff, sizeof(float) * frames * 513)); // NaN: a bin the kernel does not write shows up
    const int grid = (frames + 3) / 4;
    if (nz == 13) {
        if (with_pre) k_unit_fft1024<13, true><<<grid, 128>>>(pcm, w2, ta, tp, mag, frames, pre);
        else k_unit_fft1024<13, false><<<grid, 128>>>(pcm, w2, ta, tp, mag, frames, pre);
    } else {
        if (with_pre) k_unit_fft1024<16, true><<<grid, 128>>>(pcm, w2, ta, tp, mag, frames, pre);
        else k_unit_fft1024<16, false><<<grid, 128>>>(pcm, w2, ta, tp, mag, frames, pre);
    }
    UNIT_CUDA(cudaGetLastError());
    UNIT_CUDA(cudaMemcpy(h_mag, mag, sizeof(float) * frames * 513, cudaMemcpyDeviceToHost));
    UNIT_CUDA(cudaFree(pcm));
    UNIT_CUDA(cudaFree(w2));
    UNIT_CUDA(cudaFree(ta));
    UNIT_CUDA(cudaFree(tp));
    UNIT_CUDA(cudaFree(mag));
    return 0;
}
