// Internal declarations shared by the translation units of libafe_cuda.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <stdexcept>

#include "afe_cuda.h"

namespace afe {

void set_error(const std::string &msg);
int fail(const std::string &msg);

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define AFE_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw afe::Error(std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #expr);       \
    } while (0)

// Wrap a C-ABI body: exceptions -> error string + non-zero return.
template <class F> int guarded(F &&f)
{
    try {
        f();
        return 0;
    } catch (const std::exception &e) {
        set_error(e.what());
        return -1;
    }
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        AFE_CUDA(cudaGetDevice(&prev));
        if (prev != dev) AFE_CUDA(cudaSetDevice(dev));
        else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- derived parameter set (MfccBase ctor, mfccbase.cpp:3-31 + MfccCpu ctor, mfcccpu.cpp:94-103)
struct Derived {
    afe_params p;
    int W, S, N2, M, bins;  // bins = N2/2+1
    int nb, C, dct_len, cols, width;
    int l1, l2, D;
    int in_frames_cap, in_cap, frame_cap; // m_input_window_limit, m_input_buffer_size, m_window_limit
    explicit Derived(const afe_params &p);
};

// ---- mean / scale of one column from its statistics (normalizercpu.cpp:31-66): mean s/n; CVN sqrt((n-1)/(s2 - s*(s/n)));
// MINMAX 1/max(|mn-m|,|mx-m|); otherwise 1. The one copy of the rule: K1's cluster and ticket schemes, K2, the Normalizer
// kernels and afe_cmvn_finalize_host all call it, so the device paths agree bit for bit.
__host__ __device__ inline void finalize_column(int norm_type, double n, double s, double s2, float mn, float mx, float &mean,
                                                float &scale)
{
    const float m = (float)(s / n);
    float sc = 1.f;
    if (norm_type == AFE_NORM_CVN) sc = (float)sqrt((n - 1.0) / (s2 - s * (s / n)));
    else if (norm_type == AFE_NORM_MINMAX) sc = 1.f / fmaxf(fabsf(mn - m), fabsf(mx - m));
    mean = m;
    scale = sc;
}

// ---- host tables (afe_host.cpp)
void build_filters(const Derived &d, float alpha, std::vector<int> &edges, std::vector<float> &filters);
void build_dct(const Derived &d, std::vector<float> &dct);
// per-bin (rise, fall) weight pairs + segment edges used by the device mel loop (see afe_mel.cuh)
void build_mel_pairs(const Derived &d, const std::vector<int> &edges, const std::vector<float> &filters,
                     std::vector<float> &pairs /* [bins][2] */);

// ---- device-side constant tables for the in-register FFT (afe_fft.cuh)
struct FftTables {
    float2 *d_tw_a = nullptr;   // [R][16]   exp(-2 pi i n2 k1 / M)
    float2 *d_tw_p = nullptr;   // [M/2]     exp(-2 pi i k / N2)
    int N2 = 0;
    void build(int N2);
    void release();
};

// ---- kernels / launchers (afe_stages.cu)
struct MelTables {              // device copies, rebuilt when alpha changes
    int *d_edges = nullptr;     // [nb+2]
    float *d_pairs = nullptr;   // [bins][2]
    float *d_dct = nullptr;     // [nb][dct_len] (null when ceps_len == 0)
    float *d_window = nullptr;  // [W]
    float2 *d_window2 = nullptr; // [M] (w[2n], w[2n+1]) zero padded
    float alpha_built = -1.f;
    void release();
};
void upload_mel_tables(const Derived &d, float alpha, MelTables &t, cudaStream_t st);
void upload_window(const Derived &d, const float *window, MelTables &t, cudaStream_t st);

// segment + window into float frames [frames][N2] (SegmenterOpenCL::segment_data replacement)
void launch_segment(const int16_t *d_pcm, const float *d_window, float *d_out, int frames, int W, int S, int N2,
                    cudaStream_t st, float pre = 0.f);
// fused segment+window+FFT+|X|/N2 -> d_mag [frames][bins]
void launch_fft_mag(const Derived &d, const FftTables &ft, const MelTables &mt, const int16_t *d_pcm, float *d_mag,
                    int frames, cudaStream_t st, float pre = 0.f);
// mel+log (+DCT) : d_mag [frames][bins] -> d_mel [frames][nb], d_cep [frames][dct_len]
void launch_mel_dct(const Derived &d, const MelTables &mt, const float *d_mag, float *d_mel, float *d_cep, int frames,
                    cudaStream_t st);
// replicate-pad rows: dst[0..lead) = src row 0, dst[lead..lead+rows) = src, dst[..+trail) = last src row
void launch_pad_rows(const float *d_src, float *d_dst, int rows, int dim, int lead, int trail, cudaStream_t st);
// regression deltas, in [rows+2L][dim] -> out [rows][dim]   (DeltaOpenCL::apply replacement)
void launch_delta(const float *d_in, float *d_out, int rows, int dim, int L, cudaStream_t st);
// column statistics in double over rows -> d_stats [dim][4] = sum, sumsq, min, max ; then mean/scale floats
void launch_colstats(const float *d_x, int rows, int dim, int norm_type, float *d_mean, float *d_scale, cudaStream_t st);
void launch_affine(float *d_x, int rows, int dim, int norm_type, const float *d_mean, const float *d_scale,
                   cudaStream_t st);
// running record (sum | sumsq | count | min | max) of a Normalizer: clear, add the rows' column statistics, finalise
void launch_record_reset(double *d_rec, int dim, cudaStream_t st);
void launch_record_accumulate(const float *d_x, int rows, int dim, double *d_rec, cudaStream_t st);
void launch_record_finalize(const double *d_rec, int dim, int norm_type, float *d_mean, float *d_scale, cudaStream_t st);
// interleave [static | delta | acc] rows into d_out [rows][width]
void launch_pack(const float *d_s, const float *d_d1, const float *d_d2, float *d_out, int rows, int cols, int nstreams,
                 cudaStream_t st);

int kernel_launch_count();      // monotonically increasing count of kernel launches by this library
void count_launch(int n = 1);
int sm_count_of(int device);    // cudaDevAttrMultiProcessorCount, cached per device

template <class T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    void alloc(size_t count)
    {
        release();
        n = count;
        AFE_CUDA(cudaMalloc(&p, sizeof(T) * (count > 0 ? count : 1)));
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
};

// ---- Normalizer state (NormalizerCPU / NormalizerOpenCL, normalizercpu.h:7-9): last statistics + a running record.
// record layout (the one all-reduced across ranks): sum[dim] | sumsq[dim] | count | min[dim] | max[dim], doubles
struct NormState {
    int type = AFE_NORM_NONE, dim = 0;
    DevBuf<float> mean, scale;
    DevBuf<double> rec;         // running statistics record, 4*dim+1
    void init(int t, int d);
    int rec_len() const { return 4 * dim + 1; }
    // NormalizerCPU::normalize (normalizercpu.cpp:22-89): block statistics (unless use_last) + affine, in place
    void normalize(float *d_x, int rows, bool use_last, cudaStream_t st);
    void reset_record(cudaStream_t st);
    void accumulate(const float *d_x, int rows, cudaStream_t st);   // record += column statistics of the rows
    void finalize(cudaStream_t st);                                  // record -> mean / scale (normalizercpu.cpp:31-66)
    void apply(float *d_x, int rows, cudaStream_t st);              // (x - mean) [* scale]
};

} // namespace afe

// ---- the C-ABI Normalizer object (afe_stream.cu); afe_batch routes its corpus statistics through one of these
struct afe_normalizer {
    int device = 0;
    cudaStream_t own_st = nullptr, st = nullptr; // st: the stream in use (own, or the owning batch's)
    afe::NormState ns;
};
