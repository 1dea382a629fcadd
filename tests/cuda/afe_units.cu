// Device unit harness for the hand-written numerics shared by the fused kernel K1 and the staged kernels: the packed log
// (afe_mel.cuh) and the in-register FFT + magnitude (afe_fft.cuh). tests/test_kernel_units.py compiles this file with the
// library's nvcc flags into a temporary directory and calls the extern "C" entry points below through ctypes. Every entry
// point copies with cudaMalloc / cudaMemcpy and returns 0, or the cudaError_t of the first failing call.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "afe_fft.cuh"
#include "afe_mel.cuh"

using namespace afe;

#define UNIT_CUDA(expr)                                                                                                 \
    do {                                                                                                                \
        cudaError_t _e = (expr);                                                                                        \
        if (_e != cudaSuccess) return (int)_e;                                                                          \
    } while (0)

// ------------------------------------------------------------------------------------------------ packed log
// Sweep index i in [0, 2 * kPos) names the float pattern i (i < kPos: +0 .. the largest finite float) or
// 0x80000000 + (i - kPos) (-0 .. the most negative finite float). Lane x of mel_log2 gets pattern(i), lane y
// pattern(i + kPos mod 2 kPos), so over a full sweep each lane sees every finite float once.
constexpr uint32_t kPos = 0x7f800000u;
__host__ __device__ inline uint32_t sweep_pattern(unsigned long long i) { return i < kPos ? (uint32_t)i : 0x80000000u + (uint32_t)(i - kPos); }

// error of r in float ulps of ref = log((double)max(x, 1e-30f)); ref == 0 only for x == 1, where r must be 0 too
__device__ inline float ulp_error(float r, double ref)
{
    if (ref == 0.0) return r == 0.f ? 0.f : 3.0e38f;
    int e;
    frexp(ref, &e);                                   // |ref| in [2^(e-1), 2^e): float ulp 2^(e-24)
    return (float)(fabs((double)r - ref) / ldexp(1.0, e - 24));
}

// stats[v]: v = 0 lane x, 1 lane y, 2 scalar mel_log. Per v (4 words): max key ((float error bits << 32) | pattern),
// results != logf(max(x, 1e-30f)) bitwise, clamp mismatches (x <= 1e-30f or NaN not returning f(1e-30f) bit for bit), unused
__device__ inline void account(unsigned long long *acc, uint32_t pat, float r, float clamp_r, bool with_ulp)
{
    const float x = __uint_as_float(pat);
    const float xc = fmaxf(x, 1e-30f);
    if (__float_as_uint(r) != __float_as_uint(logf(xc))) acc[1]++;
    if (!(x > 1e-30f) && __float_as_uint(r) != __float_as_uint(clamp_r)) acc[2]++;
    if (with_ulp) {
        const float err = ulp_error(r, log((double)xc));
        const unsigned long long key = ((unsigned long long)__float_as_uint(err) << 32) | pat;
        if (key > acc[0]) acc[0] = key;
    }
}

__global__ void __launch_bounds__(256) k_log_sweep(unsigned long long begin, unsigned long long end, unsigned long long *stats)
{
    unsigned long long acc[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    const float2 clamp2 = dev::mel_log2<false>(make_float2(1e-30f, 1e-30f));
    const float clamp1 = dev::mel_log<false>(1e-30f);
    for (unsigned long long i = begin + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < end;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long j = i + kPos < 2ull * kPos ? i + kPos : i - kPos;
        const uint32_t px = sweep_pattern(i), py = sweep_pattern(j);
        const float2 r = dev::mel_log2<false>(make_float2(__uint_as_float(px), __uint_as_float(py)));
        // negative inputs all clamp to 1e-30f: their error is the clamp value's, and the clamp check covers them
        account(acc[0], px, r.x, clamp2.x, px < kPos);
        account(acc[1], py, r.y, clamp2.y, py < kPos);
        account(acc[2], px, dev::mel_log<false>(__uint_as_float(px)), clamp1, px < kPos);
    }
    for (int v = 0; v < 3; v++)
        for (int k = 0; k < 3; k++) {
            unsigned long long a = acc[v][k];
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long b = __shfl_xor_sync(0xffffffffu, a, o);
                a = k == 0 ? (a > b ? a : b) : a + b;
            }
            if ((threadIdx.x & 31) == 0) {
                if (k == 0) atomicMax(stats + 4 * v, a);
                else atomicAdd(stats + 4 * v + k, a);
            }
        }
}

// Sweep indices [begin, end) (end <= 2 * 0x7f800000) in launches of `chunk` indices; stats as above, 12 words.
extern "C" int afe_units_log_sweep(unsigned long long begin, unsigned long long end, unsigned long long chunk,
                                   unsigned long long *h_stats)
{
    unsigned long long *d = nullptr;
    UNIT_CUDA(cudaMalloc(&d, 12 * sizeof(unsigned long long)));
    UNIT_CUDA(cudaMemset(d, 0, 12 * sizeof(unsigned long long)));
    for (unsigned long long b = begin; b < end; b += chunk) {
        const unsigned long long e = b + chunk < end ? b + chunk : end;
        k_log_sweep<<<4096, 256>>>(b, e, d);
        UNIT_CUDA(cudaGetLastError());
        UNIT_CUDA(cudaDeviceSynchronize());
    }
    UNIT_CUDA(cudaMemcpy(h_stats, d, 12 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    UNIT_CUDA(cudaFree(d));
    return 0;
}

// Pointwise: out[4 i + 0..3] = mel_log2 lane x (x[i] in lane x, x[n-1-i] in lane y), lane y of the pair whose lane y
// holds x[i], mel_log<false>(x[i]), and the device reference log((double)max(x[i], 1e-30f)) in ref[i].
__global__ void k_log_points(const float *x, int n, float *out, double *ref)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float a = x[i], b = x[n - 1 - i];
    out[4 * i + 0] = dev::mel_log2<false>(make_float2(a, b)).x;
    out[4 * i + 1] = dev::mel_log2<false>(make_float2(b, a)).y;
    out[4 * i + 2] = dev::mel_log<false>(a);
    out[4 * i + 3] = logf(fmaxf(a, 1e-30f));
    ref[i] = log((double)fmaxf(a, 1e-30f));
}

extern "C" int afe_units_log_points(const float *h_x, int n, float *h_out, double *h_ref)
{
    float *dx = nullptr, *dout = nullptr;
    double *dref = nullptr;
    UNIT_CUDA(cudaMalloc(&dx, sizeof(float) * n));
    UNIT_CUDA(cudaMalloc(&dout, sizeof(float) * 4 * n));
    UNIT_CUDA(cudaMalloc(&dref, sizeof(double) * n));
    UNIT_CUDA(cudaMemcpy(dx, h_x, sizeof(float) * n, cudaMemcpyHostToDevice));
    k_log_points<<<(n + 255) / 256, 256>>>(dx, n, dout, dref);
    UNIT_CUDA(cudaGetLastError());
    UNIT_CUDA(cudaMemcpy(h_out, dout, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost));
    UNIT_CUDA(cudaMemcpy(h_ref, dref, sizeof(double) * n, cudaMemcpyDeviceToHost));
    UNIT_CUDA(cudaFree(dx));
    UNIT_CUDA(cudaFree(dout));
    UNIT_CUDA(cudaFree(dref));
    return 0;
}

// ------------------------------------------------------------------------------------------------ FFT + magnitude
// The frame loop of k_fft_mag (afe_stages.cu) with the template arguments of the caller under test; frame f's samples
// start at pcm + f * N2 (N2 samples each, readable past W), its row at mag + f * (N2/2 + 1).
template <int N2, int NZ, bool FAST, bool SCALED, bool PRE>
__global__ void __launch_bounds__(128) k_unit_fft(const int16_t *__restrict__ pcm, const float2 *window2, const float2 *tw_a,
                                                  const float2 *tw_p, float *__restrict__ mag, int frames, float pre)
{
    using C = dev::FftCfg<N2>;
    __shared__ float2 scratch[4 * C::FPW * C::SCR];
    __shared__ float s_dump[C::BINS + 3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lf = lane % C::R, fw = lane / C::R;
    dev::LaneConsts<N2, NZ> lc;
    dev::load_lane_consts<N2, NZ>(lc, window2, tw_a, tw_p, lf);
    const int per_iter = 4 * C::FPW;
    for (int f0 = blockIdx.x * per_iter; f0 < frames; f0 += gridDim.x * per_iter) {
        const int f = f0 + warp * C::FPW + fw;
        const bool act = f < frames;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(pcm + (long long)(act ? f : frames - 1) * N2);
        dev::fft_frame_mag<N2, NZ, FAST, SCALED, PRE>(words, lc, scratch + (warp * C::FPW + fw) * C::SCR,
                                                      act ? mag + (long long)f * C::BINS : s_dump, lf, pre);
    }
}

template <int N2, int NZ, bool FAST, bool SCALED, bool PRE>
static void launch_unit_fft(const int16_t *pcm, const float2 *w2, const float2 *ta, const float2 *tp, float *mag, int frames, float pre)
{
    const int per_iter = 4 * dev::FftCfg<N2>::FPW;
    k_unit_fft<N2, NZ, FAST, SCALED, PRE><<<(frames + per_iter - 1) / per_iter, 128>>>(pcm, w2, ta, tp, mag, frames, pre);
}

// The combinations the library runs, per (N2, NZ):
//   caller 0: K1 without pre-emphasis   fft_frame_mag<N2, NZ, true, false, false>  (afe_fused.cuh, k_fused_mfcc)
//   caller 1: K1 with pre-emphasis      fft_frame_mag<N2, NZ, true, false, true>
//   caller 2: staged route              fft_frame_mag<N2, NZ, false, true, true>   (afe_stages.cu, k_fft_mag)
template <int N2, int NZ>
static int dispatch_unit_fft(int caller, const int16_t *pcm, const float2 *w2, const float2 *ta, const float2 *tp, float *mag,
                             int frames, float pre)
{
    switch (caller) {
    case 0: launch_unit_fft<N2, NZ, true, false, false>(pcm, w2, ta, tp, mag, frames, pre); return 0;
    case 1: launch_unit_fft<N2, NZ, true, false, true>(pcm, w2, ta, tp, mag, frames, pre); return 0;
    case 2: launch_unit_fft<N2, NZ, false, true, true>(pcm, w2, ta, tp, mag, frames, pre); return 0;
    }
    return (int)cudaErrorInvalidValue;
}

// pcm: frames * n2 int16; window2: n2/2 float2; tw_a: (n2/32) * 16 float2; tw_p: n2/4 float2; mag: frames * (n2/2 + 1)
extern "C" int afe_units_fft_mag(int n2, int nz, int caller, const int16_t *h_pcm, int frames, const float *h_window2,
                                 const float *h_tw_a, const float *h_tw_p, float pre, float *h_mag)
{
    if ((n2 != 512 && n2 != 256) || (nz != 13 && nz != 16) || frames < 1) return (int)cudaErrorInvalidValue;
    const size_t M = n2 / 2, R = M / 16, bins = M + 1;
    int16_t *pcm = nullptr;
    float2 *w2 = nullptr, *ta = nullptr, *tp = nullptr;
    float *mag = nullptr;
    UNIT_CUDA(cudaMalloc(&pcm, sizeof(int16_t) * frames * n2));
    UNIT_CUDA(cudaMalloc(&w2, sizeof(float2) * M));
    UNIT_CUDA(cudaMalloc(&ta, sizeof(float2) * R * 16));
    UNIT_CUDA(cudaMalloc(&tp, sizeof(float2) * M / 2));
    UNIT_CUDA(cudaMalloc(&mag, sizeof(float) * frames * bins));
    UNIT_CUDA(cudaMemcpy(pcm, h_pcm, sizeof(int16_t) * frames * n2, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(w2, h_window2, sizeof(float2) * M, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(ta, h_tw_a, sizeof(float2) * R * 16, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemcpy(tp, h_tw_p, sizeof(float2) * M / 2, cudaMemcpyHostToDevice));
    UNIT_CUDA(cudaMemset(mag, 0xff, sizeof(float) * frames * bins)); // NaN: a bin the kernel does not write shows up
    int rc;
    if (n2 == 512) rc = nz == 13 ? dispatch_unit_fft<512, 13>(caller, pcm, w2, ta, tp, mag, frames, pre)
                                 : dispatch_unit_fft<512, 16>(caller, pcm, w2, ta, tp, mag, frames, pre);
    else rc = nz == 13 ? dispatch_unit_fft<256, 13>(caller, pcm, w2, ta, tp, mag, frames, pre)
                       : dispatch_unit_fft<256, 16>(caller, pcm, w2, ta, tp, mag, frames, pre);
    if (rc) return rc;
    UNIT_CUDA(cudaGetLastError());
    UNIT_CUDA(cudaMemcpy(h_mag, mag, sizeof(float) * frames * bins, cudaMemcpyDeviceToHost));
    UNIT_CUDA(cudaFree(pcm));
    UNIT_CUDA(cudaFree(w2));
    UNIT_CUDA(cudaFree(ta));
    UNIT_CUDA(cudaFree(tp));
    UNIT_CUDA(cudaFree(mag));
    return 0;
}
