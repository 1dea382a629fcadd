// Host-side logic of libafe_cuda.so: error handling, derived parameters and the tables the kernels consume.
// Tables are built on the host with the reference's float/double expression order (mfcccpu.cpp:24-60,118-136)
// so that filter edges and weights are bit-identical to the CPU path; they are uploaded once per alpha.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>

#include "afe_internal.h"

namespace afe {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
int fail(const std::string &msg) { g_error = msg; return -1; }
const char *last_error_cstr() { return g_error.c_str(); }

static int ceil_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }   // mfcccpu.cpp:10-20

static int est_windows(int samples, int W, int S)                             // parambase.cpp:16-19 (float arithmetic)
{
    return (int)std::floor(float(samples - (W - S)) / S);
}

Derived::Derived(const afe_params &prm) : p(prm)
{
    if (p.window_size < 2 || p.shift < 1) throw Error("invalid window_size/shift");
    if (p.num_banks < 1) throw Error("invalid num_banks");
    if (p.ceps_len < 0) throw Error("invalid ceps_len");
    if (p.norm < AFE_NORM_NONE || p.norm > AFE_NORM_MINMAX) throw Error("invalid norm type");
    if (p.dyn < AFE_DYN_NONE || p.dyn > AFE_DYN_ACC) throw Error("invalid dyn type");
    W = p.window_size; S = p.shift;
    N2 = ceil_pow2(W); M = N2 / 2; bins = M + 1;
    nb = p.num_banks; C = p.ceps_len;
    dct_len = p.want_c0 ? C + 1 : C;                       // mfccbase.cpp:28
    cols = C > 0 ? dct_len : nb;                           // mfccbase.cpp:35
    l1 = p.dyn != AFE_DYN_NONE ? p.delta_l1 : 0;           // mfccbase.cpp:26-27
    l2 = p.dyn == AFE_DYN_ACC ? p.delta_l2 : 0;
    if (l1 < 0 || l2 < 0) throw Error("invalid delta sizes");
    if (p.dyn != AFE_DYN_NONE && l1 < 1) throw Error("delta_l1 must be >= 1 when dyn != NONE");
    if (p.dyn == AFE_DYN_ACC && l2 < 1) throw Error("delta_l2 must be >= 1 when dyn == ACC");
    D = l1 + l2;
    width = cols * (p.dyn == AFE_DYN_ACC ? 3 : p.dyn == AFE_DYN_DELTA ? 2 : 1);
    in_frames_cap = est_windows(p.input_buffer_size, W, S);  // parambase.cpp:12-13
    in_cap = in_frames_cap * S + W - S;
    frame_cap = in_frames_cap + 2 + (p.dyn != AFE_DYN_NONE ? 3 * D : 0); // mfcccpu.cpp:95-103
}

static inline float hz2mel(float f) { return 1127 * logf(f / 700 + 1); }     // mfcccpu.cpp:21
static inline float mel2hz(float f) { return 700 * (expf(f / 1127) - 1); }   // mfcccpu.cpp:22

void build_filters(const Derived &d, float alpha, std::vector<int> &edges, std::vector<float> &filters)
{
    const int nb = d.nb, N2 = d.N2;
    const float sr = d.p.sample_rate;
    std::vector<float> cent(nb + 2);
    edges.assign(nb + 2, 0);
    filters.assign(2 * (size_t)N2, 0.f);
    const float mlo = hz2mel(d.p.low_freq), mhi = hz2mel(d.p.high_freq);
    for (int i = 0; i < nb + 2; i++) {
        float f = mel2hz(i / float(nb + 1) * (mhi - mlo) + mlo);
        float o = 2 * (float)M_PI * f / sr;
        o = o + 2 * atanf(((1 - alpha) * sinf(o)) / (1 - (1 - alpha) * cosf(o)));   // VTLN bilinear warp, mfcccpu.cpp:36-37
        cent[i] = sr * o / (2 * (float)M_PI);
        edges[i] = (int)floor(cent[i] * N2 / sr + 0.5);
    }
    for (int i = 0; i < nb; i++) {
        const float cl = cent[i], cc = cent[i + 1], cr = cent[i + 2];
        const int il = (int)floor(N2 * cl / sr + 0.5), ir = (int)floor(N2 * cr / sr + 0.5);
        for (int j = il; j < ir; j++) {
            if (j < 0 || j >= N2) continue;
            float up = (j * sr / (N2) - cl) / (cc - cl);
            float dn = (j * sr / (N2) - cr) / (cc - cr);
            filters[(size_t)(i % 2) * N2 + j] = std::fmax(0.0f, std::fmin(up, dn));
        }
    }
}

void build_dct(const Derived &d, std::vector<float> &dct)
{
    dct.assign((size_t)d.nb * (d.dct_len > 0 ? d.dct_len : 1), 0.f);
    if (d.C <= 0) return;
    const float lift = d.p.lift_coef;
    const float nf = (float)sqrt(2.0 / d.nb);
    for (int k = 0; k < d.nb; k++)
        for (int i = 1; i <= d.C; i++) {
            float lifter = (1 + lift / 2 * sinf((float)M_PI * (float)i / lift));
            dct[(size_t)d.dct_len * k + i - 1] = lifter * nf * cosf((float)M_PI * i * (k + 0.5f) / d.nb);
        }
    if (d.p.want_c0)
        for (int k = 0; k < d.nb; k++) dct[(size_t)d.dct_len * k + d.C] = nf;
}

// The reference sweeps bins edges[0]..edges[nb+1] once with two running sums (even / odd filters), closing filter
// b when the sweep reaches edges[b+2] (mfcccpu.cpp:192-220). Bin j in segment i = [edges[i], edges[i+1]) therefore feeds
// the RISING side of filter i (row i%2) and the FALLING side of filter i-1 (row (i+1)%2). pairs[j] = (rise, fall).
void build_mel_pairs(const Derived &d, const std::vector<int> &edges, const std::vector<float> &filters,
                     std::vector<float> &pairs)
{
    pairs.assign((size_t)d.bins * 2, 0.f);
    for (int i = 0; i <= d.nb; i++)
        for (int j = edges[i]; j < edges[i + 1]; j++) {
            if (j < 0 || j >= d.bins) continue;
            pairs[2 * (size_t)j + 0] = filters[(size_t)(i % 2) * d.N2 + j];
            pairs[2 * (size_t)j + 1] = filters[(size_t)((i + 1) % 2) * d.N2 + j];
        }
}

} // namespace afe

using namespace afe;

extern "C" {

const char *afe_last_error(void) { return afe::last_error_cstr(); }
int afe_abi_version(void) { return AFE_ABI_VERSION; }

int afe_estimated_window_count(int samples, int window_size, int shift) { return est_windows(samples, window_size, shift); }

int afe_output_width(const afe_params *p)
{
    try { return Derived(*p).width; } catch (const std::exception &e) { set_error(e.what()); return -1; }
}

int afe_fft_size(int window_size) { return ceil_pow2(window_size); }

void afe_make_window(float *window, int W)
{
    for (int i = 0; i < W; i++) window[i] = (float)(0.56f - 0.46f * cos((2.0f * M_PI * i) / W)) / 32768.f;
}

int afe_build_filters(const afe_params *p, float alpha, int *edges, float *filters)
{
    return guarded([&] {
        Derived d(*p);
        std::vector<int> e; std::vector<float> f;
        build_filters(d, alpha, e, f);
        memcpy(edges, e.data(), sizeof(int) * e.size());
        memcpy(filters, f.data(), sizeof(float) * f.size());
    });
}

int afe_build_dct(const afe_params *p, float *dct)
{
    return guarded([&] {
        Derived d(*p);
        if (d.C <= 0) throw Error("ceps_len == 0: no DCT matrix");
        std::vector<float> m;
        build_dct(d, m);
        memcpy(dct, m.data(), sizeof(float) * m.size());
    });
}

// stats record: sum[w], sumsq[w], count, min[w], max[w]. Formulas: normalizercpu.cpp:31-66.
int afe_cmvn_finalize_host(int norm_type, int width, const double *stats, float *mean, float *scale)
{
    return guarded([&] {
        const int w = width;
        const double n = stats[2 * (size_t)w];
        if (!(n >= 1)) throw Error("cmvn finalize: empty statistics");
        for (int c = 0; c < w; c++)
            finalize_column(norm_type, n, stats[c], stats[w + c], (float)stats[2 * w + 1 + c], (float)stats[3 * w + 1 + c],
                            mean[c], scale[c]);
    });
}

// Contiguous utterance ranges balanced by sample count (prefix sums): rank r gets [starts[r], starts[r+1]).
int afe_shard_utterances(const int64_t *len, int n_utts, int n_ranks, int *starts)
{
    return guarded([&] {
        if (n_ranks < 1 || n_utts < 0) throw Error("shard: invalid arguments");
        std::vector<int64_t> off((size_t)n_utts + 1, 0);
        for (int u = 0; u < n_utts; u++) {
            if (len[u] < 0) throw Error("shard: negative length");
            off[u + 1] = off[u] + len[u];
        }
        const int64_t total = off[n_utts];
        starts[0] = 0;
        int u = 0;
        for (int r = 1; r < n_ranks; r++) {
            const int64_t target = (int64_t)((__int128)total * r / n_ranks);
            while (u < n_utts && off[u + 1] - target <= target - off[u]) u++; // boundary nearest to the target
            if (u < starts[r - 1]) u = starts[r - 1];
            starts[r] = u;
        }
        starts[n_ranks] = n_utts;
    });
}

// Time sharding of ONE stream over ranks (SURVEY §8 f4): rank r produces the frames [first[r], first[r] + count[r]) and needs the
// samples [sample_begin[r], sample_begin[r] + sample_count[r]), i.e. its frames plus D frames of context on each side
// (the (W - S) + 2 D S sample halo of segmentercpu.cpp:69-73, 90-92). local_first[r] = index of its first frame inside that range.
int afe_shard_stream(int64_t total_samples, int window_size, int shift, int delta_frames, int n_ranks, int64_t *sample_begin,
                     int64_t *sample_count, int64_t *first, int *count, int *local_first)
{
    return guarded([&] {
        if (n_ranks < 1 || window_size < 2 || shift < 1 || delta_frames < 0) throw Error("shard_stream: invalid arguments");
        const int64_t T = total_samples >= window_size ? (total_samples - (window_size - shift)) / shift : 0;
        if (T < (int64_t)n_ranks * (2 * delta_frames + 1)) throw Error("shard_stream: stream too short for this many ranks");
        for (int r = 0; r < n_ranks; r++) {
            const int64_t f0 = T * r / n_ranks, f1 = T * (r + 1) / n_ranks;
            const int64_t c0 = std::max<int64_t>(0, f0 - delta_frames), c1 = std::min<int64_t>(T, f1 + delta_frames);
            first[r] = f0; count[r] = (int)(f1 - f0);
            local_first[r] = (int)(f0 - c0);
            sample_begin[r] = c0 * shift;
            sample_count[r] = (c1 - c0 - 1) * shift + window_size;
        }
    });
}

} // extern "C"
