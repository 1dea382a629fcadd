// Stage kernels behind the streaming objects (SegmenterCuda / MfccCuda / DeltaCuda / NormalizerCuda): one kernel per
// reference stage with device buffers in between, mirroring the OpenCL classes' structure (SURVEY §2.1) with the
// CPU classes' numerics. The throughput path is the fused kernel in afe_fused.cuh; these serve the block-wise
// ParamBase API where a block is small and the spectrum must persist across apply() calls (VTLN sweeps).
#include <cfloat>
#include <mutex>

#include "afe_internal.h"
#include "afe_fft.cuh"
#include "afe_mel.cuh"

namespace afe {

int sm_count_of(int device)
{
    static std::mutex mu;
    static int cache[64] = {0};
    std::lock_guard<std::mutex> lock(mu);
    if (device < 0 || device >= 64) device = 0;
    if (!cache[device]) AFE_CUDA(cudaDeviceGetAttribute(&cache[device], cudaDevAttrMultiProcessorCount, device));
    return cache[device];
}
// grid cap of the grid-stride stage kernels: `per_sm` CTAs per SM of the current device
static int grid_cap(int per_sm)
{
    int dev = 0;
    AFE_CUDA(cudaGetDevice(&dev));
    return sm_count_of(dev) * per_sm;
}

// ------------------------------------------------------------------------------------------------ segmenter
// out[N2*f + j] = window[j] * pcm[f*S + j] (j < W), 0 beyond   — segmentercpu.cpp:17-28 / segmenter.cl:1-22
// pre != 0: per-frame pre-emphasis before the window, x[j] - pre * x[j-1] with x[-1] := x[0] (not in the reference)
__device__ __forceinline__ float windowed_sample(const int16_t *__restrict__ frame, const float *__restrict__ window, int j, float pre)
{
    const float x = (float)frame[j];
    if (pre == 0.f) return __fmul_rn(window[j], x);
    const float xp = (float)frame[j > 0 ? j - 1 : 0];
    return fmaf(xp, __fmul_rn(window[j], -pre), __fmul_rn(x, window[j]));
}

__global__ void k_segment(const int16_t *__restrict__ pcm, const float *__restrict__ window, float *__restrict__ out,
                          int frames, int W, int S, int N2, float pre)
{
    const long long n = (long long)frames * N2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int f = (int)(i / N2), j = (int)(i - (long long)f * N2);
        out[i] = j < W ? windowed_sample(pcm + (long long)f * S, window, j, pre) : 0.f;
    }
}
void launch_segment(const int16_t *d_pcm, const float *d_window, float *d_out, int frames, int W, int S, int N2,
                    cudaStream_t st, float pre)
{
    if (frames <= 0) return;
    const long long n = (long long)frames * N2;
    const int grid = (int)std::min<long long>((n + 255) / 256, grid_cap(16));
    k_segment<<<grid, 256, 0, st>>>(d_pcm, d_window, d_out, frames, W, S, N2, pre);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ------------------------------------------------------------------------------------------------ FFT + magnitude
// Fast path (N2 = 256/512, even S): the same in-register FFT as the fused kernel, PCM read straight from global.
template <int N2, int NZ>
__global__ void __launch_bounds__(128) k_fft_mag(const int16_t *__restrict__ pcm, const float2 *window2, const float2 *tw_a,
                                                 const float2 *tw_p, float *__restrict__ mag, int frames, int S, float pre)
{
    using C = dev::FftCfg<N2>;
    __shared__ float2 scratch[4 * C::FPW * C::SCR];
    __shared__ float s_dump[C::BINS + 3]; // magnitude row of padding frames
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lf = lane % C::R, fw = lane / C::R;
    dev::LaneConsts<N2, NZ> lc;
    dev::load_lane_consts<N2, NZ>(lc, window2, tw_a, tw_p, lf);
    const int per_iter = 4 * C::FPW;
    for (int f0 = blockIdx.x * per_iter; f0 < frames; f0 += gridDim.x * per_iter) {
        const int f = f0 + warp * C::FPW + fw;
        const bool act = f < frames;
        const int fc = act ? f : frames - 1;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(pcm + (long long)fc * S);
        dev::fft_frame_mag<N2, NZ, false>(words, lc, scratch + (warp * C::FPW + fw) * C::SCR,
                                          act ? mag + (long long)f * C::BINS : s_dump, lf, pre);
    }
}

// Generic path: any power-of-two N2 <= 4096, any W/S. One CTA per frame, radix-2 Stockham in shared memory.
__global__ void k_fft_mag_generic(const int16_t *__restrict__ pcm, const float *__restrict__ window,
                                  float *__restrict__ mag, int frames, int W, int S, int N2, float pre)
{
    extern __shared__ float2 sm[]; // 2 * N2
    float2 *a = sm, *b = sm + N2;
    for (int f = blockIdx.x; f < frames; f += gridDim.x) {
        for (int j = threadIdx.x; j < N2; j += blockDim.x)
            a[j] = make_float2(j < W ? windowed_sample(pcm + (long long)f * S, window, j, pre) : 0.f, 0.f);
        __syncthreads();
        // Stockham autosort, radix 2: stage with half-size l, stride m
        for (int l = N2 / 2, m = 1; l >= 1; l >>= 1, m <<= 1) {
            for (int i = threadIdx.x; i < N2 / 2; i += blockDim.x) {
                const int j = i / m, k = i - j * m; // j in [0,l), k in [0,m)
                float sn, cs;
                sincospif(-(float)j / (float)l, &sn, &cs); // exp(-i pi j / l)
                const float2 c0 = a[k + j * m], c1 = a[k + j * m + l * m];
                const float2 d = make_float2(c0.x - c1.x, c0.y - c1.y);
                b[k + 2 * j * m] = make_float2(c0.x + c1.x, c0.y + c1.y);
                b[k + 2 * j * m + m] = make_float2(d.x * cs - d.y * sn, d.x * sn + d.y * cs);
            }
            __syncthreads();
            float2 *t = a; a = b; b = t;
        }
        for (int j = threadIdx.x; j <= N2 / 2; j += blockDim.x)
            mag[(long long)f * (N2 / 2 + 1) + j] = sqrtf(a[j].x * a[j].x + a[j].y * a[j].y) / (float)N2;
        __syncthreads();
    }
}

void launch_fft_mag(const Derived &d, const FftTables &ft, const MelTables &mt, const int16_t *d_pcm, float *d_mag,
                    int frames, cudaStream_t st, float pre)
{
    if (frames <= 0) return;
    const bool fast = (d.N2 == 512 || d.N2 == 256) && d.S % 2 == 0 && ft.N2 == d.N2 &&
                      (reinterpret_cast<uintptr_t>(d_pcm) & 3) == 0;
    if (fast) {
        const int R = d.M / 16, per_iter = 4 * (32 / R);
        const int grid = std::min((frames + per_iter - 1) / per_iter, grid_cap(8));
        const bool pruned = d.W <= 26 * R;
        if (d.N2 == 512) {
            if (pruned) k_fft_mag<512, 13><<<grid, 128, 0, st>>>(d_pcm, mt.d_window2.p, ft.d_tw_a.p, ft.d_tw_p.p, d_mag, frames, d.S, pre);
            else k_fft_mag<512, 16><<<grid, 128, 0, st>>>(d_pcm, mt.d_window2.p, ft.d_tw_a.p, ft.d_tw_p.p, d_mag, frames, d.S, pre);
        } else {
            if (pruned) k_fft_mag<256, 13><<<grid, 128, 0, st>>>(d_pcm, mt.d_window2.p, ft.d_tw_a.p, ft.d_tw_p.p, d_mag, frames, d.S, pre);
            else k_fft_mag<256, 16><<<grid, 128, 0, st>>>(d_pcm, mt.d_window2.p, ft.d_tw_a.p, ft.d_tw_p.p, d_mag, frames, d.S, pre);
        }
    } else {
        if (d.N2 > 4096) throw Error("window_size above 4096 is not supported");
        const int threads = std::max(32, std::min(256, d.N2 / 2));
        k_fft_mag_generic<<<std::min(frames, grid_cap(8)), threads, sizeof(float2) * 2 * d.N2, st>>>(d_pcm, mt.d_window.p, d_mag,
                                                                                                 frames, d.W, d.S, d.N2, pre);
    }
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ------------------------------------------------------------------------------------------------ mel + log + DCT
// one thread per frame; tables broadcast from shared memory
__global__ void k_mel_dct(const float *__restrict__ mag, const int *__restrict__ edges, const float2 *__restrict__ pairs,
                          const float *__restrict__ dct, float *__restrict__ mel, float *__restrict__ cep, int frames,
                          int bins, int nb, int dct_len)
{
    extern __shared__ unsigned char sm_raw[];
    int *s_edges = reinterpret_cast<int *>(sm_raw);
    float2 *s_pairs = reinterpret_cast<float2 *>(sm_raw + ((nb + 2) * 4 + 15) / 16 * 16);
    float *s_dct = reinterpret_cast<float *>(s_pairs + bins);
    for (int i = threadIdx.x; i < nb + 2; i += blockDim.x) s_edges[i] = edges[i];
    for (int i = threadIdx.x; i < bins; i += blockDim.x) s_pairs[i] = pairs[i];
    for (int i = threadIdx.x; i < nb * dct_len; i += blockDim.x) s_dct[i] = dct[i];
    __syncthreads();
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= frames) return;
    const float *row = mag + (long long)f * bins;
    // pass 1: log-mel energies (always kept: FBANK output and the reference's m_mel_energies)
    dev::mel_dct_frame<1, false>(row, s_edges, s_pairs, nullptr, nb, 0, mel + (long long)f * nb);
    // pass 2: cepstra, k ascending fp32 accumulation (mfcccpu.cpp:222-232)
    if (dct_len > 0) {
        const float *e = mel + (long long)f * nb;
        for (int j = 0; j < dct_len; j++) {
            float s = 0.f;
            for (int k = 0; k < nb; k++) s = fmaf(e[k], s_dct[k * dct_len + j], s);
            cep[(long long)f * dct_len + j] = s;
        }
    }
}
void launch_mel_dct(const Derived &d, const MelTables &mt, const float *d_mag, float *d_mel, float *d_cep, int frames,
                    cudaStream_t st)
{
    if (frames <= 0) return;
    const int dl = d.C > 0 ? d.dct_len : 0;
    const size_t sm = ((d.nb + 2) * 4 + 15) / 16 * 16 + (size_t)d.bins * 8 + (size_t)d.nb * dl * 4;
    if (sm > 200 * 1024) throw Error("mel/DCT tables do not fit in shared memory");
    AFE_CUDA(cudaFuncSetAttribute(k_mel_dct, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    k_mel_dct<<<(frames + 63) / 64, 64, sm, st>>>(d_mag, mt.d_edges.p, reinterpret_cast<const float2 *>(mt.d_pairs.p), mt.d_dct.p,
                                                  d_mel, d_cep, frames, d.bins, d.nb, dl);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ------------------------------------------------------------------------------------------------ delta
__global__ void k_pad_rows(const float *__restrict__ src, float *__restrict__ dst, int rows, int dim, int lead, int trail)
{
    const int total = (lead + rows + trail) * dim;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int r = i / dim - lead;
        const int c = i % dim;
        r = r < 0 ? 0 : (r >= rows ? rows - 1 : r);
        dst[i] = src[r * dim + c];
    }
}
void launch_pad_rows(const float *d_src, float *d_dst, int rows, int dim, int lead, int trail, cudaStream_t st)
{
    const int total = (lead + rows + trail) * dim;
    if (total <= 0) return;
    k_pad_rows<<<std::min((total + 255) / 256, grid_cap(8)), 256, 0, st>>>(d_src, d_dst, rows, dim, lead, trail);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// out[i][j] = sum_l l*(in[i+L+l][j] - in[i+L-l][j]) / (2 sum l^2)   — deltacpu.cpp:16-30 / delta.cl:6-34
__global__ void k_delta(const float *__restrict__ in, float *__restrict__ out, int rows, int dim, int L)
{
    const int total = rows * dim;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int r = i / dim, c = i % dim;
        float num = 0.f, den = 0.f;
        for (int l = 1; l <= L; l++) {
            num = __fadd_rn(num, __fmul_rn((float)l, __fsub_rn(in[(r + L + l) * dim + c], in[(r + L - l) * dim + c])));
            den = __fadd_rn(den, (float)(l * l));
        }
        out[i] = __fdiv_rn(num, __fmul_rn(2.f, den));
    }
}
void launch_delta(const float *d_in, float *d_out, int rows, int dim, int L, cudaStream_t st)
{
    const int total = rows * dim;
    if (total <= 0) return;
    k_delta<<<std::min((total + 255) / 256, grid_cap(8)), 256, 0, st>>>(d_in, d_out, rows, dim, L);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ------------------------------------------------------------------------------------------------ normalizer
// Replaces norm.cl kernelSum + kernelFinalizeSum with the CPU class' double statistics (normalizercpu.cpp:31-66).
// Statistics of column c over the CTA (256 threads): rows strided over threads, double accumulation, fixed-order tree:
// deterministic. Every thread gets the totals.
__device__ __forceinline__ void block_column_stats(const float *__restrict__ x, int rows, int dim, int c, double &sum,
                                                   double &sumsq, float &mn, float &mx)
{
    __shared__ double s_sum[256], s_sq[256];
    __shared__ float s_mn[256], s_mx[256];
    const int t = threadIdx.x;
    double s = 0.0, s2 = 0.0;
    float lo = FLT_MAX, hi = -FLT_MAX;
    for (int r = t; r < rows; r += blockDim.x) {
        const float v = x[(long long)r * dim + c];
        s += (double)v;
        s2 += (double)__fmul_rn(v, v);
        lo = fminf(lo, v); hi = fmaxf(hi, v);
    }
    s_sum[t] = s; s_sq[t] = s2; s_mn[t] = lo; s_mx[t] = hi;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (t < o) {
            s_sum[t] += s_sum[t + o]; s_sq[t] += s_sq[t + o];
            s_mn[t] = fminf(s_mn[t], s_mn[t + o]); s_mx[t] = fmaxf(s_mx[t], s_mx[t + o]);
        }
        __syncthreads();
    }
    sum = s_sum[0]; sumsq = s_sq[0]; mn = s_mn[0]; mx = s_mx[0];
}

// one CTA per column -> the column's mean / scale
__global__ void k_colstats(const float *__restrict__ x, int rows, int dim, int norm_type, float *__restrict__ mean,
                           float *__restrict__ scale)
{
    const int c = blockIdx.x;
    double s, s2;
    float mn, mx;
    block_column_stats(x, rows, dim, c, s, s2, mn, mx);
    if (threadIdx.x == 0) finalize_column(norm_type, (double)rows, s, s2, mn, mx, mean[c], scale[c]);
}
void launch_colstats(const float *d_x, int rows, int dim, int norm_type, float *d_mean, float *d_scale, cudaStream_t st)
{
    if (rows <= 0 || dim <= 0) return;
    k_colstats<<<dim, 256, 0, st>>>(d_x, rows, dim, norm_type, d_mean, d_scale);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ---- running record of a Normalizer (the statistics that corpus-level CMVN all-reduces): sum | sumsq | count | min | max
__global__ void k_record_reset(double *rec, int dim)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < dim) { rec[c] = 0.0; rec[dim + c] = 0.0; rec[2 * dim + 1 + c] = (double)FLT_MAX; rec[3 * dim + 1 + c] = -(double)FLT_MAX; }
    if (c == 0) rec[2 * dim] = 0.0;
}
// one CTA per column, same reduction as k_colstats; the column's totals are ADDED to the record (calls are stream ordered)
__global__ void k_record_accumulate(const float *__restrict__ x, int rows, int dim, double *__restrict__ rec)
{
    const int c = blockIdx.x;
    double s, s2;
    float mn, mx;
    block_column_stats(x, rows, dim, c, s, s2, mn, mx);
    if (threadIdx.x == 0) {
        rec[c] += s; rec[dim + c] += s2;
        rec[2 * dim + 1 + c] = fmin(rec[2 * dim + 1 + c], (double)mn);
        rec[3 * dim + 1 + c] = fmax(rec[3 * dim + 1 + c], (double)mx);
        if (c == 0) rec[2 * dim] += (double)rows;
    }
}
__global__ void k_record_finalize(const double *__restrict__ rec, int dim, int norm_type, float *__restrict__ mean,
                                  float *__restrict__ scale)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= dim) return;
    finalize_column(norm_type, rec[2 * dim], rec[c], rec[dim + c], (float)rec[2 * dim + 1 + c], (float)rec[3 * dim + 1 + c],
                    mean[c], scale[c]);
}
void launch_record_reset(double *d_rec, int dim, cudaStream_t st)
{
    k_record_reset<<<(dim + 127) / 128, 128, 0, st>>>(d_rec, dim);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}
void launch_record_accumulate(const float *d_x, int rows, int dim, double *d_rec, cudaStream_t st)
{
    if (rows <= 0 || dim <= 0) return;
    k_record_accumulate<<<dim, 256, 0, st>>>(d_x, rows, dim, d_rec);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}
void launch_record_finalize(const double *d_rec, int dim, int norm_type, float *d_mean, float *d_scale, cudaStream_t st)
{
    k_record_finalize<<<(dim + 127) / 128, 128, 0, st>>>(d_rec, dim, norm_type, d_mean, d_scale);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

void NormState::init(int t, int d)
{
    type = t; dim = d;
    mean.alloc(d); scale.alloc(d); rec.alloc(4 * (size_t)d + 1);
}
void NormState::normalize(float *d_x, int rows, bool use_last, cudaStream_t st)   // normalizercpu.cpp:22-89
{
    if (type == AFE_NORM_NONE || rows <= 0) return;
    if (!use_last) launch_colstats(d_x, rows, dim, type, mean.p, scale.p, st);
    launch_affine(d_x, rows, dim, type, mean.p, scale.p, st);
}
void NormState::reset_record(cudaStream_t st) { launch_record_reset(rec.p, dim, st); }
void NormState::accumulate(const float *d_x, int rows, cudaStream_t st) { launch_record_accumulate(d_x, rows, dim, rec.p, st); }
void NormState::finalize(cudaStream_t st) { launch_record_finalize(rec.p, dim, type, mean.p, scale.p, st); }
void NormState::apply(float *d_x, int rows, cudaStream_t st)
{
    if (type == AFE_NORM_NONE || rows <= 0) return;
    launch_affine(d_x, rows, dim, type, mean.p, scale.p, st);
}

__global__ void k_affine(float *__restrict__ x, int rows, int dim, int norm_type, const float *__restrict__ mean,
                         const float *__restrict__ scale)
{
    const long long total = (long long)rows * dim;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % dim);
        const float v = __fsub_rn(x[i], mean[c]);
        x[i] = norm_type == AFE_NORM_CMN ? v : __fmul_rn(v, scale[c]);
    }
}
void launch_affine(float *d_x, int rows, int dim, int norm_type, const float *d_mean, const float *d_scale, cudaStream_t st)
{
    const long long total = (long long)rows * dim;
    if (total <= 0) return;
    k_affine<<<(int)std::min<long long>((total + 255) / 256, grid_cap(8)), 256, 0, st>>>(d_x, rows, dim, norm_type, d_mean, d_scale);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

// ------------------------------------------------------------------------------------------------ output packing
__global__ void k_pack(const float *__restrict__ s, const float *__restrict__ d1, const float *__restrict__ d2,
                       float *__restrict__ out, int rows, int cols, int nstreams)
{
    const int width = cols * nstreams, total = rows * width;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int r = i / width, c = i % width, k = c / cols, cc = c % cols;
        const float *src = k == 0 ? s : (k == 1 ? d1 : d2);
        out[i] = src[r * cols + cc];
    }
}
void launch_pack(const float *d_s, const float *d_d1, const float *d_d2, float *d_out, int rows, int cols, int nstreams,
                 cudaStream_t st)
{
    const int total = rows * cols * nstreams;
    if (total <= 0) return;
    k_pack<<<std::min((total + 255) / 256, grid_cap(8)), 256, 0, st>>>(d_s, d_d1, d_d2, d_out, rows, cols, nstreams);
    AFE_CUDA(cudaGetLastError());
    count_launch();
}

} // namespace afe
