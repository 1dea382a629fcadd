// Batch extractor (afe_batch_*): planning, launch of the fused kernel K1, statistics finalize K2 and the normalise
// pass K3. Corpus-level statistics are owned by a Normalizer object (afe_batch_normalizer): the batch reduces its
// per-tile records into the Normalizer's record, the Normalizer all-reduces it over NCCL, the batch normalises with it.
#include <algorithm>
#include <atomic>
#include <memory>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "afe_internal.h"
#include "afe_fused_host.h"
#include "afe_nccl.h"

namespace afe {

// ------------------------------------------------------------------------------------------------ FFT tables
void FftTables::build(int n2)
{
    N2 = n2;
    const int M = n2 / 2, R = M / 16;
    std::vector<float2> a((size_t)R * 16), p((size_t)M / 2);
    for (int l = 0; l < R; l++)
        for (int k1 = 0; k1 < 16; k1++) {
            const double ang = -2.0 * M_PI * (double)(l * k1) / (double)M;
            a[(size_t)l * 16 + k1] = make_float2((float)cos(ang), (float)sin(ang));
        }
    for (int k = 0; k < M / 2; k++) {
        const double ang = -2.0 * M_PI * (double)k / (double)n2;
        p[k] = make_float2((float)cos(ang), (float)sin(ang));
    }
    d_tw_a.upload(a);
    d_tw_p.upload(p);
}

void upload_mel_tables(const Derived &d, float alpha, MelTables &t, cudaStream_t st)
{
    std::vector<int> edges; std::vector<float> filters, pairs, dct;
    build_filters(d, alpha, edges, filters);
    for (int i = 0; i + 1 < (int)edges.size(); i++)
        if (edges[i + 1] < edges[i]) throw Error("mel filter edges are not monotonic");
    if (edges.front() < 0 || edges.back() > d.M) throw Error("mel filterbank exceeds the Nyquist bin (check low_freq/high_freq)");
    build_mel_pairs(d, edges, filters, pairs);
    if (!t.d_edges.p) t.d_edges.alloc(d.nb + 2);
    if (!t.d_pairs.p) t.d_pairs.alloc(2 * d.bins);
    // pageable source + stream-ordered copy: cudaMemcpyAsync from pageable memory stages synchronously, safe with locals
    AFE_CUDA(cudaMemcpyAsync(t.d_edges.p, edges.data(), sizeof(int) * (d.nb + 2), cudaMemcpyHostToDevice, st));
    AFE_CUDA(cudaMemcpyAsync(t.d_pairs.p, pairs.data(), sizeof(float) * 2 * d.bins, cudaMemcpyHostToDevice, st));
    if (d.C > 0 && !t.d_dct.p) {
        build_dct(d, dct);
        t.d_dct.alloc(dct.size());
        AFE_CUDA(cudaMemcpyAsync(t.d_dct.p, dct.data(), sizeof(float) * dct.size(), cudaMemcpyHostToDevice, st));
    }
    AFE_CUDA(cudaStreamSynchronize(st));
    t.alpha_built = alpha;
}

void upload_window(const Derived &d, const float *window, MelTables &t, cudaStream_t st)
{
    if (!t.d_window.p) t.d_window.alloc(d.W);
    if (!t.d_window2.p) t.d_window2.alloc(d.M);
    std::vector<float> w2((size_t)d.N2, 0.f);
    memcpy(w2.data(), window, sizeof(float) * d.W);
    AFE_CUDA(cudaMemcpyAsync(t.d_window.p, window, sizeof(float) * d.W, cudaMemcpyHostToDevice, st));
    AFE_CUDA(cudaMemcpyAsync(t.d_window2.p, w2.data(), sizeof(float) * d.N2, cudaMemcpyHostToDevice, st));
    AFE_CUDA(cudaStreamSynchronize(st));
}

// ------------------------------------------------------------------------------------------------ K2 / K3
// stats record per group: [sum[w], sumsq[w], count, min[w], max[w]]  (4w+1 doubles)
__global__ void __launch_bounds__(256) k_reduce_partials(const double *__restrict__ partials, const int *__restrict__ tile_begin,
                                  const double *__restrict__ counts, int width, double *__restrict__ stats)
{
    // the canonical summation order of dev::group_total, so that K2 and the in-kernel schemes agree bit for bit
    extern __shared__ double s_seg[];
    const int g = blockIdx.x, c = threadIdx.x;
    double s0, s1, lo, hi;
    dev::group_total(partials, width, tile_begin[g], tile_begin[g + 1] - tile_begin[g], threadIdx.x, blockDim.x, s_seg,
                     c < width ? c : 0, s0, s1, lo, hi);
    if (c >= width) return;
    double *o = stats + (long long)g * (4 * width + 1);
    o[c] = s0; o[width + c] = s1; o[2 * width + 1 + c] = lo; o[3 * width + 1 + c] = hi;
    if (c == 0) o[2 * width] = counts[g];
}

// Corpus scope has ONE group over all tiles: two deterministic levels instead of one serial loop.
// level 1: block j sums tiles j, j+gridDim.x, ... -> scratch[j][width][4]; level 2 = k_reduce_partials over the scratch.
__global__ void __launch_bounds__(128) k_reduce_partials_level1(const double *__restrict__ partials, int n_tiles, int width,
                                         double *__restrict__ scratch)
{
    const int c = threadIdx.x;
    if (c >= width) return;
    double s0, s1, lo, hi;
    dev::sum_records(partials, width, c, blockIdx.x, n_tiles, s0, s1, lo, hi, gridDim.x);
    double *o = scratch + ((long long)blockIdx.x * width + c) * 4;
    o[0] = s0; o[1] = s1; o[2] = lo; o[3] = hi;
}

// mean / scale per group and column (normalizercpu.cpp:31-66). With norm_after_dyn == 0 the reference normalises the
// statics before the deltas are taken, which equals scaling delta columns by the static column's scale (mean 0).
__global__ void k_finalize_stats(const double *__restrict__ stats, int width, int cols, int norm_type, int norm_after_dyn,
                                 float *__restrict__ mean, float *__restrict__ scale)
{
    const int g = blockIdx.x, c = threadIdx.x;
    if (c >= width) return;
    const double *o = stats + (long long)g * (4 * width + 1);
    const double n = o[2 * width];
    const int src = norm_after_dyn ? c : (c % cols);
    float m, sc;
    finalize_column(norm_type, n, o[src], o[width + src], (float)o[2 * width + 1 + src], (float)o[3 * width + 1 + src], m, sc);
    if (!norm_after_dyn && c >= cols) m = 0.f;
    mean[(long long)g * width + c] = m;
    scale[(long long)g * width + c] = sc;
}

// K3: in-place (x - mean) [* scale] over one tile's rows (dev::normalise_tile_rows). HBM / L2 bound: 8 B per float.
__global__ void k_normalize_tiles(float *__restrict__ out, const Tile *__restrict__ tiles, int width, int norm_type,
                                  const float *__restrict__ mean, const float *__restrict__ scale)
{
    extern __shared__ float s_ms[]; // mean[width] | scale[width]
    dev::normalise_tile_rows(out, tiles[blockIdx.x], width, norm_type, mean, scale, s_ms);
}

static std::atomic<int> g_launches{0};
int kernel_launch_count() { return g_launches.load(); }
void count_launch(int n) { g_launches.fetch_add(n); }

// ------------------------------------------------------------------------------------------------ K1 launch table
#define AFE_DECL_INST(k) cudaError_t fused_launch_##k(const FusedLaunch &); int fused_max_clusters_##k(const FusedLaunch &);
#define AFE_FOR_EACH_INST(X) X(0) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) \
    X(18) X(19) X(20) X(21) X(22) X(23) X(24) X(25) X(26) X(27) X(28) X(29) X(30) X(31) X(32) X(33) X(34) X(35) X(36) X(37) \
    X(38) X(39) X(40) X(41) X(42) X(43) X(44) X(45) X(46) X(47) X(48) X(49) X(50) X(51) X(52) X(53) X(54) X(55) X(56) X(57) \
    X(58) X(59) X(60) X(61) X(62) X(63)
AFE_FOR_EACH_INST(AFE_DECL_INST)
#undef AFE_DECL_INST

cudaError_t launch_fused_variant(int key, const FusedLaunch &fl)
{
    typedef cudaError_t (*fn_t)(const FusedLaunch &);
#define AFE_ENTRY(k) fused_launch_##k,
    static const fn_t table[kFusedVariants] = {AFE_FOR_EACH_INST(AFE_ENTRY)};
#undef AFE_ENTRY
    if (key < 0 || key >= kFusedVariants) return cudaErrorInvalidValue;
    return table[key](fl);
}
int fused_variant_max_clusters(int key, const FusedLaunch &fl)
{
    typedef int (*fn_t)(const FusedLaunch &);
#define AFE_ENTRY(k) fused_max_clusters_##k,
    static const fn_t table[kFusedVariants] = {AFE_FOR_EACH_INST(AFE_ENTRY)};
#undef AFE_ENTRY
    if (key < 0 || key >= kFusedVariants) return -1;
    return table[key](fl);
}

// ------------------------------------------------------------------------------------------------ FusedEngine
std::string fused_unsupported_reason(const Derived &d)
{
    if (d.N2 != 1024 && d.N2 != 512 && d.N2 != 256) return "fused path supports 256/512/1024-point FFTs (window_size 129..1024)";
    if (d.S % 2) return "fused path needs an even shift";
    if (d.C > 0 && d.dct_len > kMaxCepsWide) return "fused path supports ceps_len + c0 <= 48";
    if (d.width > 128) return "fused path supports output width <= 128";
    if (d.nb > kMaxBanksWide) return "fused path supports num_banks <= 128";
    // 128 banks x 48 DCT columns of constant-bank tables would not fit the kernel parameter list
    if (d.C > 0 && d.dct_len > 16 && d.nb > kMaxBanks) return "fused path supports ceps_len + c0 <= 16 with more than 64 banks";
    if (d.C > 0 && d.dct_len > 16 && d.N2 == 1024) return "fused path supports ceps_len + c0 <= 16 with 1024-point FFTs";
    if (d.W > 26 * (d.M / 16) && d.W > d.N2) return "window longer than the FFT";
    return "";
}

// Mel weights + DCT matrix as a by-value kernel parameter (constant bank). Per filter b: bins [edges[b], edges[b+2]) with
// weights filters[b%2][bin] — the per-filter form of the reference's two-running-sums sweep (mfcccpu.cpp:192-220).
template <int NB, int NC, int NBINS>
static void build_mel_const(const Derived &d, float alpha, MelConstT<NB, NC, NBINS> &mc)
{
    std::vector<int> edges; std::vector<float> filters, dct;
    build_filters(d, alpha, edges, filters);
    for (int i = 0; i + 1 < (int)edges.size(); i++)
        if (edges[i + 1] < edges[i]) throw Error("mel filter edges are not monotonic");
    if (edges.front() < 0 || edges.back() > d.M) throw Error("mel filterbank exceeds the Nyquist bin (check low_freq/high_freq)");
    if (d.bins > NBINS) throw Error("FFT bins exceed the mel table capacity");
    memset(&mc, 0, sizeof mc);
    int off4 = 0;
    const float scale = 0.5f / (float)d.N2; // the kernel stores |2X|; scaling by a power of two commutes with rounding
    for (int w = 0; w < 8; w++) {           // warp class w owns the filters w, w + 8, ...: their lists are contiguous
        mc.wstart[w] = (short)off4;
        for (int b = w; b < d.nb; b += 8) {
            const int j0 = edges[b], j1 = edges[b + 2], s4 = j0 & ~3, n8 = std::max(1, (j1 - s4 + 7) / 8);
            if (off4 + 2 * n8 > MelConstT<NB, NC, NBINS>::kWl4) throw Error("mel weight list exceeds the kernel-parameter budget");
            if (s4 + 8 * n8 > mag_stride(d.N2) + 16) throw Error("mel filter too wide for the fused kernel");
            mc.desc[b] = (s4 / 4) | (n8 << 16);
            float *wt = reinterpret_cast<float *>(mc.wl4 + off4);
            for (int j = j0; j < j1; j++) wt[j - s4] = filters[(size_t)(b % 2) * d.N2 + j] * scale;
            off4 += 2 * n8;
        }
    }
    if (d.C > 0) {
        if (d.dct_len > NC) throw Error("DCT exceeds the kernel-parameter budget");
        build_dct(d, dct);
        for (int k = 0; k < d.nb; k++)
            for (int j = 0; j < d.dct_len; j++) reinterpret_cast<float *>(mc.dct4[k])[j] = dct[(size_t)k * d.dct_len + j];
    }
}

FusedEngine::FusedEngine(const Derived &dd, int dev) : d(dd), device(dev)
{
    const std::string why = fused_unsupported_reason(d);
    if (!why.empty()) throw Error(why);
    sm_count = sm_count_of(dev);
    fft.build(d.N2);
    const int nfw = (d.nb + 7) / 8;  // filters per warp (8 warps): instantiated for 3, 5, 8 and 16
    kf = nfw <= 3 ? 3 : nfw <= 5 ? 5 : nfw <= 8 ? 8 : 16;
    if (d.C > 0 && d.dct_len > 16) { nc = kMaxCepsWide; kf = nfw <= 5 ? 5 : 8; } // wide DCT: KF = 5 (<= 40 banks) or 8
    if (d.N2 == 1024) ctas_per_sm = 1; // the 66 KB magnitude tile (__launch_bounds__(256, 1) in k_fused_mfcc)
    const int ns = d.width / d.cols;
    auto layout = [&](int tc, int nout) {
        FusedSmem l = d.N2 == 1024 ? fused_smem_layout<1024>(8, d.S, d.cols, tc, nout, d.l2, ns)
                      : d.N2 == 512 ? fused_smem_layout<512>(8, d.S, d.cols, tc, nout, d.l2, ns)
                                    : fused_smem_layout<256>(8, d.S, d.cols, tc, nout, d.l2, ns);
        if (nc > 16) l.total += lm_tile_bytes(kf); // the wide DCT's log-mel tile follows everything else
        return l;
    };
    if ((kf == 16 && d.C == 0) || (nc > 16 && d.D == 0)) {
        // 65..128-column log-mel, and the wide DCT without deltas (D = 0, see k_fused_mfcc): the kernel writes each
        // 32-frame round's rows as soon as they are computed, so the cepstra buffer holds one round and the tile size is
        // not bound by shared memory
        tc_max = kRoundFrames; nout_max = 512;
    } else if (nc > 16) {
        // wide DCT with deltas: the largest whole-round cepstra tile that keeps 2 CTAs per SM (41 + c0 with deltas and
        // delta-deltas: 128 frames)
        const int tc_min = kRoundFrames * ((2 * d.D + 1 + kRoundFrames - 1) / kRoundFrames + 1);
        int tc = 512;
        while (tc > tc_min && layout(tc, tc - 2 * d.D).total > kSmemTwoCtas) tc -= kRoundFrames;
        tc_max = tc; nout_max = tc - 2 * d.D;
    } else if (d.N2 == 1024) {
        // 1024 points: the 66 KB magnitude tile already limits K1 to one CTA per SM, so the cepstra tile is the largest
        // whole-round tile, up to 512 frames, that fits one CTA's shared memory
        const int tc_min = kRoundFrames * ((2 * d.D + 1 + kRoundFrames - 1) / kRoundFrames + 1);
        int tc = 512;
        while (tc > tc_min && layout(tc, tc - 2 * d.D).total > kSmemOneCta) tc -= kRoundFrames;
        tc_max = tc; nout_max = tc - 2 * d.D;
    } else {
        // tile geometry (2 CTAs per SM): the cepstra tile holds up to 512 frames (<= 27 KB of shared memory)
        int tc = 512;
        tc = std::min(tc, (6912 / d.cols) / kRoundFrames * kRoundFrames);
        tc = std::max(tc, kRoundFrames * ((2 * d.D + 1 + kRoundFrames - 1) / kRoundFrames + 1));
        tc_max = tc; nout_max = tc - 2 * d.D;
    }
    L = layout(tc_max, nout_max);
    if (L.total > kSmemOneCta) throw Error("fused kernel shared-memory budget exceeded");
    // phase-3 scratch of the default regression and the clustered scheme (k_fused_mfcc): row-group records at off_mags,
    // the tile's record at +25 KB, mean / scale at +30 KB, all below the cepstra
    const int rp = kMaxFusedThreads / d.cols;
    if (rp * d.width * 32 > 25 * 1024 || d.width * 32 > 5 * 1024 || L.off_mags + 30 * 1024 + 2 * d.width * 4 > L.off_cep)
        throw Error("fused kernel phase-3 scratch does not fit its shared-memory slots");
    const int R = d.M / 16;
    pruned = d.W <= 26 * R;            // window tail is zero from n1 = 13 on (400/512 and 200/256 both qualify)
}

void FusedEngine::set_window(const float *window, cudaStream_t st)
{
    upload_window(d, window, mel, st);
    window_set = true;
}
void FusedEngine::ensure_mel(float alpha)
{
    if (mc_alpha == alpha) return;
    if (d.N2 == 1024 && kf == 16) build_mel_const(d, alpha, mc_wide1024);
    else if (d.N2 == 1024) build_mel_const(d, alpha, mc1024);
    else if (nc > 16) build_mel_const(d, alpha, mc_ceps);
    else if (kf == 16) build_mel_const(d, alpha, mc_wide);
    else build_mel_const(d, alpha, mc);
    mc_alpha = alpha;
}
std::string FusedEngine::kernel_label() const
{
    const int k = launch_key();
    char buf[96];
    snprintf(buf, sizeof buf, "k_fused_mfcc<%d,%d,8,%d,%s%s>", fused_key_n2(k), fused_key_nz(k), fused_key_kf(k),
             fused_key_pre(k) ? "true" : "false", fused_key_nc(k) > 16 ? ",48" : "");
    return buf;
}

int FusedEngine::latency_tile(int n_out) const
{
    const int target = std::max(1, ctas_per_sm * sm_count);
    const int want = (n_out + target - 1) / target;                          // rows per tile for ~2 tiles per SM
    const int rounds = std::max(2, (want + 2 * d.D + kRoundFrames - 1) / kRoundFrames);
    return std::max(1, std::min(nout_max, rounds * kRoundFrames - 2 * d.D));
}

void FusedEngine::plan_uniform(int T, int t_first, int n_out, int nout_cap, int &ntile, int &nout) const
{
    const int cap = nout_cap > 0 ? std::min(nout_cap, nout_max) : nout_max;
    // number of tiles: fewest 32-frame rounds (the halo of D frames per side is recomputed by every tile)
    int best_cost = 1 << 30;
    ntile = (n_out + cap - 1) / cap;
    for (int cand = ntile; cand <= ntile + 3; cand++) {
        const int no = (n_out + cand - 1) / cand;
        int cost = 0;
        for (int t0 = t_first; t0 < t_first + n_out; t0 += no) {
            const int c0 = std::max(0, t0 - d.D), c1 = std::min(T, t0 + std::min(no, t_first + n_out - t0) + d.D);
            cost += (c1 - c0 + kRoundFrames - 1) / kRoundFrames;
        }
        if (cost < best_cost) { best_cost = cost; ntile = cand; }
    }
    nout = (n_out + ntile - 1) / ntile;
    ntile = (n_out + nout - 1) / nout;
}

int FusedEngine::plan_rows(std::vector<Tile> &tiles, long long pcm_off, long long out_row0, int T, int t_first, int n_out,
                           int group, int nout_cap) const
{
    if (n_out <= 0) return 0;
    int count, nout;
    plan_uniform(T, t_first, n_out, nout_cap, count, nout);
    const int first = (int)tiles.size();
    for (int t0 = t_first; t0 < t_first + n_out; t0 += nout) {
        Tile tl;
        tl.pcm_off = pcm_off; tl.out_row0 = out_row0; tl.T = T; tl.t0 = t0;
        tl.nout = std::min(nout, t_first + n_out - t0); tl.group = group;
        tl.tile0 = first; tl.ntiles = count; tl.flags = 0; tl.pad_ = 0;
        tiles.push_back(tl);
    }
    return count;
}

FusedArgs FusedEngine::base_args(int q1, const int16_t *pcm, bool tma_ok) const
{
    FusedArgs a{};
    a.pcm = pcm;
    a.use_tma = tma_ok && d.S % 8 == 0 && (reinterpret_cast<uintptr_t>(pcm) & 15) == 0 ? 1 : 0;
    a.window2 = mel.d_window2.p; a.tw_a = fft.d_tw_a.p; a.tw_p = fft.d_tw_p.p;
    a.norm_type = d.p.norm; a.norm_after_dyn = d.p.norm_after_dyn;
    a.W = d.W; a.S = d.S; a.nb = d.nb; a.dct_len = d.C > 0 ? d.dct_len : 0; a.cols = d.cols; a.width = d.width;
    a.l1 = d.l1; a.l2 = d.l2; a.nstreams = d.width / d.cols;
    a.q1 = d.D > 0 ? q1 : 0;
    a.tc_max = tc_max;
    a.pre = pre;
    float den1 = 0, den2 = 0;
    for (int l = 1; l <= d.l1; l++) den1 += l * l;   // float accumulation like deltacpu.cpp:26
    for (int l = 1; l <= d.l2; l++) den2 += l * l;
    a.rden1 = den1 > 0 ? 1.f / (2 * den1) : 0.f;
    a.rden2 = den2 > 0 ? 1.f / (2 * den2) : 0.f;
#ifdef AFE_DEVTOOLS
    { const char *dbg = getenv("AFE_DEBUG_SKIP"); a.debug_skip = dbg ? atoi(dbg) : 0; }
#endif
    return a;
}

// A clustered launch needs all CTAs of a cluster co-scheduled (111 KB of shared memory each). On a partitioned device
// (MIG / MPS slices, fewer GPCs) that can be impossible: probe once per cluster size and let the caller use the ticket scheme.
bool FusedEngine::cluster_schedulable(int cluster, const FusedArgs &a, cudaStream_t st)
{
    if (cluster < 1 || cluster > 4) return false;
    if (cluster_probe[cluster] < 0) {
        FusedLaunch fl{a, L, mel_const(), cluster, cluster, st};
        const int n = fused_variant_max_clusters(fused_key(d.N2, pruned ? 13 : 16, kf, false, nc), fl); // same footprint with and without pre-emphasis
        cluster_probe[cluster] = n > 0 ? n : 0;
    }
    return cluster_probe[cluster] > 0;
}

void FusedEngine::launch(const FusedArgs &a, int grid, int cluster, cudaStream_t st)
{
    if (!window_set) throw Error("set_window must be called before running");
    FusedLaunch fl{a, L, mel_const(), grid, cluster, st};
    const cudaError_t e = launch_fused_variant(launch_key(), fl);
    if (e != cudaSuccess) {
        cudaGetLastError();
        throw Error(std::string("CUDA error: ") + cudaGetErrorString(e) + " at k_fused_mfcc launch" + (cluster > 0 ? " (clustered)" : ""));
    }
    count_launch();
}

void FusedNormState::alloc(int n_groups, size_t n_tiles, int width)
{
    partials.alloc(4 * (size_t)width * n_tiles);
    counters.alloc(n_groups + 1); flags.alloc(n_groups);
    AFE_CUDA(cudaMemset(counters.p, 0, sizeof(int) * (n_groups + 1)));
    AFE_CUDA(cudaMemset(flags.p, 0, sizeof(unsigned) * n_groups));
    epoch = 0;
    mean.alloc((size_t)width * n_groups); scale.alloc((size_t)width * n_groups);
}

void FusedEngine::launch_roles(FusedArgs a, int ntiles, FusedNormState &ns, cudaStream_t st)
{
    a.counters = ns.counters.p; a.work_counter = ns.counters.p + ns.counters.n - 1;
    a.flags = ns.flags.p; a.epoch = ++ns.epoch; a.ntiles_launch = ntiles;
    a.g_mean = ns.mean.p; a.g_scale = ns.scale.p;
    launch(a, ntiles + std::min(ntiles, ctas_per_sm * sm_count), 0, st);
}

void FusedEngine::launch_clustered(FusedArgs a, int grid, int cluster, FusedNormState &ns, cudaStream_t st)
{
    a.cluster_norm = 1;
    try {
        launch(a, grid, cluster, st);
    } catch (const Error &) {
        cluster_probe[cluster] = 0; // the clustered launch was refused (nothing ran): no more tries at this size
        a.cluster_norm = 0;
        launch_ticket(a, grid, ns, st);
    }
}

} // namespace afe

using namespace afe;

// ================================================================================================== afe_batch
struct NormalizerDestroy {
    void operator()(afe_normalizer *n) const { afe_normalizer_destroy(n); }
};

struct afe_batch {
    Derived d;
    int device;
    Stream own_stream, s_in, s_out;         // s_in / s_out: the copy streams of run_host, created by its first call
    std::vector<Event> ev_in, ev_k;
    cudaStream_t stream = nullptr;          // the stream in use: own_stream or the caller's
    std::unique_ptr<FusedEngine> eng;
    float alpha = 1.f;
    int scope = AFE_STATS_REFERENCE_BLOCK, flags = 0;
    struct Plan {                           // everything afe_batch_plan derives, replaced as a whole by it
        int n_utts = 0, n_tiles = 0, n_groups = 0;
        bool aligned = false;               // every utterance starts on a 16-byte boundary
        std::vector<int64_t> sample_off, sample_len, frame_off;
        std::vector<int> h_tile_begin;      // [n_utts+1] first tile of every utterance
        int64_t pcm_extent = 0;
        int corpus_blocks = 0;              // level-1 blocks of the corpus reduction (2 per SM)
        int max_tiles_per_utt = 0;
        DevBuf<Tile> tiles;
        DevBuf<int> tile_begin, scratch_begin;
        DevBuf<double> counts, scratch;
        DevBuf<double> group_stats;         // per-utterance scopes: the statistics records
        FusedNormState norm;                // also K2's partials and K3's mean / scale
        std::unique_ptr<afe_normalizer, NormalizerDestroy> cnorm; // corpus scope: the Normalizer that owns the record
        double *stats() const { return cnorm ? cnorm->ns.rec.p : group_stats.p; } // [n_groups][4 * width + 1]
    } plan;
    // One tile normalising its whole utterance is right for short utterances and a serial bottleneck for long ones:
    // up to 8 tiles -> clusters / ticket scheme; more -> the role scheme (normaliser CTAs, one per tile, same launch).
    bool fuse_norm() const { return !(flags & AFE_BATCH_UNFUSED_NORM); }
    bool long_scheme() const { return plan.max_tiles_per_utt > 8; }
    int last_launches = 0;
    // device staging for run_host (grow-only)
    DevBuf<int16_t> pcm_stage;
    DevBuf<float> out_stage;

    explicit afe_batch(const afe_params &p, int dev) : d(p), device(dev) {}
};

// Tiles [t0, t1) (whole utterances) through K1. With fused normalisation:
//  * the default regression and utterances of 1..4 tiles: runs of equal tile count become ONE clustered launch each
//    (cluster = utterance, statistics through distributed shared memory), at most kMaxClusterRuns launches;
//  * other batches whose utterances have at most 8 tiles: the ticket scheme (last tile normalises through L2), one launch;
//  * batches with longer utterances: the role scheme (2 x tiles CTAs, the second half normalises a tile each), one launch.
constexpr int kMaxClusterRuns = 8;
constexpr int kMaxClusterTiles = 4; // utterances of up to 4 tiles (~20 s) form a cluster; longer ones keep the ticket scheme
static void run_extract(afe_batch *b, const int16_t *d_pcm, float *d_out, int t0 = 0, int t1 = -1, bool fuse_norm = false)
{
    afe_batch::Plan &pl = b->plan;
    if (!pl.tiles.p) throw Error("afe_batch_plan must be called before running");
    if (t1 < 0) t1 = pl.n_tiles;
    if (t1 <= t0) return;
    FusedEngine &eng = *b->eng;
    eng.ensure_mel(b->alpha);
    const Derived &d = b->d;
    const bool want_stats = d.p.norm != AFE_NORM_NONE;
    FusedArgs a = eng.base_args((b->flags & AFE_BATCH_Q1_EXACT) ? 1 : 0, d_pcm, pl.aligned && !(b->flags & AFE_BATCH_NO_TMA));
    a.out = d_out; a.tiles = pl.tiles.p; a.tile_base = t0;
    if (want_stats) eng.set_stats(a, pl.norm, d.p.norm_after_dyn && b->scope == AFE_STATS_REFERENCE_BLOCK ? 1 : 2);
    if (!(fuse_norm && want_stats)) { eng.launch_plain(a, t1 - t0, b->stream); b->last_launches++; return; }
    if (b->long_scheme()) { eng.launch_roles(a, t1 - t0, pl.norm, b->stream); b->last_launches++; return; }
    if (!(b->flags & AFE_BATCH_NO_CLUSTER) && eng.default_regression()) {
        struct Run { int t0, t1, cluster; };
        std::vector<Run> runs;
        const std::vector<int> &tb = pl.h_tile_begin;
        const int u0 = (int)(std::lower_bound(tb.begin(), tb.end(), t0) - tb.begin());
        bool schedulable = true;
        for (int u = u0; u < pl.n_utts && tb[u] < t1 && (int)runs.size() <= kMaxClusterRuns; u++) {
            const int nt = tb[u + 1] - tb[u], cl = nt <= kMaxClusterTiles ? nt : 0;
            if (cl > 0 && !eng.cluster_schedulable(cl, a, b->stream)) { schedulable = false; break; }
            if (!runs.empty() && runs.back().cluster == cl) runs.back().t1 = tb[u + 1];
            else runs.push_back({tb[u], tb[u + 1], cl});
        }
        if (schedulable && (int)runs.size() <= kMaxClusterRuns && !runs.empty() && runs.front().t0 == t0 && runs.back().t1 == t1) {
            for (const Run &r : runs) {
                a.tile_base = r.t0;
                if (r.cluster > 0) eng.launch_clustered(a, r.t1 - r.t0, r.cluster, pl.norm, b->stream);
                else eng.launch_ticket(a, r.t1 - r.t0, pl.norm, b->stream);
                b->last_launches++;
            }
            return;
        }
    }
    eng.launch_ticket(a, t1 - t0, pl.norm, b->stream);
    b->last_launches++;
}

static void run_reduce(afe_batch *b, int g0 = 0, int g1 = -1)
{
    const afe_batch::Plan &pl = b->plan;
    if (g1 < 0) g1 = pl.n_groups;
    if (g1 <= g0) return;
    const int w = b->d.width;
    if (b->scope == AFE_STATS_CORPUS && pl.n_tiles > 2 * pl.corpus_blocks) {
        k_reduce_partials_level1<<<pl.corpus_blocks, 128, 0, b->stream>>>(pl.norm.partials.p, pl.n_tiles, w, pl.scratch.p);
        AFE_CUDA(cudaGetLastError());
        k_reduce_partials<<<1, 256, dev::kSegs * w * 4 * sizeof(double), b->stream>>>(pl.scratch.p, pl.scratch_begin.p, pl.counts.p, w, pl.stats());
        AFE_CUDA(cudaGetLastError());
        count_launch(2); b->last_launches += 2;
        return;
    }
    k_reduce_partials<<<g1 - g0, 256, dev::kSegs * w * 4 * sizeof(double), b->stream>>>(pl.norm.partials.p, pl.tile_begin.p + g0, pl.counts.p + g0, w,
                                                                                       pl.stats() + (size_t)g0 * (4 * w + 1));
    AFE_CUDA(cudaGetLastError());
    count_launch(); b->last_launches++;
}

static void run_normalize(afe_batch *b, float *d_out, int t0 = 0, int t1 = -1, int g0 = 0, int g1 = -1)
{
    const Derived &d = b->d;
    const afe_batch::Plan &pl = b->plan;
    if (t1 < 0) t1 = pl.n_tiles;
    if (g1 < 0) g1 = pl.n_groups;
    if (t1 <= t0 || g1 <= g0) return;
    const size_t w = d.width;
    k_finalize_stats<<<g1 - g0, 128, 0, b->stream>>>(pl.stats() + (size_t)g0 * (4 * w + 1), d.width, d.cols, d.p.norm,
                                                      d.p.norm_after_dyn, pl.norm.mean.p + g0 * w, pl.norm.scale.p + g0 * w);
    AFE_CUDA(cudaGetLastError());
    // Tile::group is absolute, so mean / scale keep their base
    k_normalize_tiles<<<t1 - t0, 256, 2 * d.width * sizeof(float), b->stream>>>(d_out, pl.tiles.p + t0, d.width, d.p.norm,
                                                                              pl.norm.mean.p, pl.norm.scale.p);
    AFE_CUDA(cudaGetLastError());
    count_launch(2); b->last_launches += 2;
}

extern "C" {

int afe_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { set_error(std::string("CUDA error: ") + cudaGetErrorString(e)); return 0; }
    return n;
}

int afe_build_flags(void)
{
#ifdef AFE_DEVTOOLS
    return 1;
#else
    return 0;
#endif
}

int afe_batch_create(const afe_params *p, int cuda_device, afe_batch **out)
{
    *out = nullptr;
    return guarded([&] {
        if (afe_device_count() <= cuda_device) throw Error("no usable CUDA device " + std::to_string(cuda_device) + " (the product has no CPU fallback)");
        DeviceGuard g(cuda_device);
        std::unique_ptr<afe_batch> b(new afe_batch(*p, cuda_device));
        const std::string why = fused_unsupported_reason(b->d);
        if (!why.empty()) throw Error(why + "; use the streaming object");
        b->own_stream.create();
        b->stream = b->own_stream;
        b->eng.reset(new FusedEngine(b->d, cuda_device));
        *out = b.release();
    });
}

void afe_batch_destroy(afe_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    cudaStreamSynchronize(b->stream);
    delete b;
}

int afe_batch_set_window(afe_batch *b, const float *window)
{
    return guarded([&] { DeviceGuard g(b->device); b->eng->set_window(window, b->stream); });
}

int afe_batch_set_alpha(afe_batch *b, float alpha) { b->alpha = alpha; return 0; }

int afe_batch_set_preemphasis(afe_batch *b, float coefficient)
{
    return guarded([&] {
        if (!(coefficient >= 0.f && coefficient < 1.f)) throw Error("pre-emphasis coefficient must be in [0, 1)");
        b->eng->pre = coefficient;
    });
}

int afe_batch_set_options(afe_batch *b, int stats_scope, int flags)
{
    return guarded([&] {
        if (stats_scope < AFE_STATS_REFERENCE_BLOCK || stats_scope > AFE_STATS_CORPUS) throw Error("invalid stats scope");
        // the per-group row counts, the group table and the corpus Normalizer are laid down by afe_batch_plan from the scope
        if (b->plan.tiles.p && stats_scope != b->scope) throw Error("set the statistics scope before afe_batch_plan");
        const int known = AFE_BATCH_Q1_EXACT | AFE_BATCH_NO_TMA | AFE_BATCH_UNFUSED_NORM | AFE_BATCH_NO_CLUSTER;
        if (flags & ~known) throw Error("unknown batch flag bits " + std::to_string(flags & ~known));
        b->scope = stats_scope; b->flags = flags; // every flag is read at run time
    });
}

int afe_batch_set_stream(afe_batch *b, void *cuda_stream)
{
    b->stream = cuda_stream ? (cudaStream_t)cuda_stream : b->own_stream;
    if (b->plan.cnorm) b->plan.cnorm->st = b->stream;
    return 0;
}

static int plan_impl(afe_batch *b, const int64_t *off, const int64_t *len, const int *seg_first, const int *seg_rows, int n_utts,
                     int64_t *total_frames);

int afe_batch_plan(afe_batch *b, const int64_t *off, const int64_t *len, int n_utts, int64_t *total_frames)
{
    return plan_impl(b, off, len, nullptr, nullptr, n_utts, total_frames);
}

// Segments of longer streams (time sharding, SURVEY §8 f4): entry u covers the samples [off, off + len) = T frames of context and
// produces only the rows of its frames [first_frame[u], first_frame[u] + n_frames[u]); the frames in front of / behind that range
// are real context for the deltas (no edge replication except where the segment touches the end of its sample range).
int afe_batch_plan_segments(afe_batch *b, const int64_t *off, const int64_t *len, const int *first_frame, const int *n_frames,
                            int n_segments, int64_t *total_frames)
{
    if (!first_frame || !n_frames) return fail("plan_segments: null segment arrays");
    return plan_impl(b, off, len, first_frame, n_frames, n_segments, total_frames);
}

static int plan_impl(afe_batch *b, const int64_t *off, const int64_t *len, const int *seg_first, const int *seg_rows, int n_utts,
                     int64_t *total_frames)
{
    return guarded([&] {
        const Derived &d = b->d;
        if (n_utts < 1) throw Error("plan: no utterances");
        DeviceGuard g(b->device);
        b->plan = {};
        const FusedEngine &eng = *b->eng;
        // built aside and installed whole, so that a plan that fails here leaves the batch unplanned
        afe_batch::Plan pl;
        pl.n_utts = n_utts;
        pl.sample_off.assign(off, off + n_utts);
        pl.sample_len.assign(len, len + n_utts);
        pl.h_tile_begin.assign(n_utts + 1, 0);
        pl.frame_off.assign(n_utts + 1, 0);
        std::vector<Tile> tiles;
        std::vector<double> counts;
        const bool corpus = b->scope == AFE_STATS_CORPUS;
        if (seg_first && d.p.norm != AFE_NORM_NONE && !corpus)
            throw Error("plan_segments: normalisation over segments needs the CORPUS statistics scope");
        pl.aligned = true;
        double corpus_count = 0;
        // Wave balancing for small batches (a single long stream, a handful of files): with fewer than ~8 waves of CTAs the
        // tail of a partly filled last wave costs a whole tile time, so pick the tile size for which
        // waves x rounds-per-tile is smallest (config 5: 720 tiles x 16 rounds -> 4 full waves x 10 rounds).
        int nout_cap = 0;
        {
            int64_t total = 0, longest = 0;
            for (int u = 0; u < n_utts; u++) {
                const int64_t T = std::max<int64_t>(0, (len[u] - (d.W - d.S)) / d.S);
                total += T; longest = std::max(longest, T);
            }
            const int slots = eng.ctas_per_sm * eng.sm_count;
            const int64_t tiles_default = (total + eng.nout_max - 1) / eng.nout_max;
            // only batches that hold a long utterance (more than 8 tiles: the role scheme anyway); batches of short
            // utterances keep the large tiles, whose 1..4-tile utterances normalise inside a thread-block cluster
            if (longest > 8 * (int64_t)eng.nout_max && tiles_default <= 8 * (int64_t)slots) {
                const int w0 = (int)((tiles_default + slots - 1) / slots);
                int best_cost = w0 * ((eng.nout_max + 2 * d.D + kRoundFrames - 1) / kRoundFrames);
                for (int w = w0; w <= w0 + 3; w++) {
                    const int cap = (int)std::min<int64_t>(eng.nout_max, std::max<int64_t>(1, (total + (int64_t)w * slots - 1) / ((int64_t)w * slots)));
                    const int rounds = std::max(2, (cap + 2 * d.D + kRoundFrames - 1) / kRoundFrames);
                    if (w * rounds < best_cost) { best_cost = w * rounds; nout_cap = std::max(1, std::min(eng.nout_max, rounds * kRoundFrames - 2 * d.D)); }
                }
            }
        }
        for (int u = 0; u < n_utts; u++) {
            const int64_t n = len[u];
            if (n < 0 || n > 0x7fffffff || off[u] < 0) throw Error("plan: invalid utterance offset/length");
            pl.pcm_extent = std::max<int64_t>(pl.pcm_extent, off[u] + n);
            if (off[u] % 2) throw Error("plan: utterance offsets must be even (32-bit PCM word loads)");
            if (off[u] % 8) pl.aligned = false;
            // parambase.cpp:16-19 evaluates in float32, which is inexact above 2^24 samples: never let it exceed the
            // exact count (the extra frame would lie outside the utterance)
            const int T = std::min(afe_estimated_window_count((int)n, d.W, d.S), (int)std::max<int64_t>(0, (n - (d.W - d.S)) / d.S));
            if (T <= 2 * d.D || T < 1) throw Error("Can't process data, window count is too small"); // segmentercpu.cpp:65-66
            const int t_first = seg_first ? seg_first[u] : 0, rows = seg_rows ? seg_rows[u] : T;
            if (t_first < 0 || rows < 1 || t_first + rows > T) throw Error("plan_segments: segment outside its frames");
            pl.frame_off[u + 1] = pl.frame_off[u] + rows;
            pl.h_tile_begin[u] = (int)tiles.size();
            const int ntile = eng.plan_rows(tiles, off[u], pl.frame_off[u] - t_first, T, t_first, rows, corpus ? 0 : u, nout_cap);
            pl.max_tiles_per_utt = std::max(pl.max_tiles_per_utt, ntile);
            const double cnt = seg_first ? rows : !d.p.norm_after_dyn ? T : (b->scope == AFE_STATS_REFERENCE_BLOCK ? T - d.D : T);
            if (corpus) corpus_count += cnt; else counts.push_back(cnt);
        }
        if (corpus) counts.push_back(corpus_count);
        pl.h_tile_begin[n_utts] = (int)tiles.size();
        pl.n_tiles = (int)tiles.size();
        pl.n_groups = corpus ? 1 : n_utts;
        pl.corpus_blocks = 2 * eng.sm_count;
        pl.tiles.upload(tiles);
        if (d.p.norm != AFE_NORM_NONE) {
            const size_t w = d.width;
            pl.tile_begin.upload(corpus ? std::vector<int>{0, pl.n_tiles} : pl.h_tile_begin); // first tile of every group
            pl.counts.upload(counts);
            pl.norm.alloc(pl.n_groups, tiles.size(), d.width);
            if (corpus) {
                // the corpus record lives in a Normalizer of dim = width (all three streams in one record)
                afe_normalizer *n = nullptr;
                if (afe_normalizer_create(d.p.norm, d.width, b->device, &n) != 0) throw Error(afe_last_error());
                pl.cnorm.reset(n);
                n->st = b->stream;
                pl.scratch.alloc(4 * w * pl.corpus_blocks);
                pl.scratch_begin.upload({0, pl.corpus_blocks});
            } else
                pl.group_stats.alloc((4 * w + 1) * pl.n_groups);
        }
        if (total_frames) *total_frames = pl.frame_off[n_utts];
        b->plan = std::move(pl);
    });
}

int afe_batch_frame_offsets(const afe_batch *b, int64_t *fo)
{
    memcpy(fo, b->plan.frame_off.data(), sizeof(int64_t) * b->plan.frame_off.size());
    return 0;
}
int afe_batch_num_tiles(const afe_batch *b) { return b->plan.n_tiles; }
int afe_batch_kernel_launches(const afe_batch *b) { return b->last_launches; }
const char *afe_batch_kernel_name(const afe_batch *b)
{
    static thread_local std::string name;
    name = b->eng ? b->eng->kernel_label() : "k_fused_mfcc";
    return name.c_str();
}
afe_normalizer *afe_batch_normalizer(afe_batch *b) { return b->plan.cnorm.get(); }

int afe_batch_extract_device(afe_batch *b, const int16_t *d_pcm, float *d_out)
{
    return guarded([&] { DeviceGuard g(b->device); b->last_launches = 0; run_extract(b, d_pcm, d_out); });
}

int afe_batch_run_device(afe_batch *b, const int16_t *d_pcm, float *d_out)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        if (b->scope == AFE_STATS_CORPUS && b->d.p.norm != AFE_NORM_NONE)
            throw Error("corpus statistics need the two-pass sequence: extract_device, corpus_stats, allreduce, normalize_device");
        b->last_launches = 0;
        const bool fuse = b->fuse_norm();
        run_extract(b, d_pcm, d_out, 0, -1, fuse);   // per-utterance scopes: normalised inside the one launch
        if (b->d.p.norm != AFE_NORM_NONE && !fuse) { run_reduce(b); run_normalize(b, d_out); }
    });
}

int afe_batch_corpus_stats(afe_batch *b, double **d_stats, int *stats_len)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        if (b->d.p.norm == AFE_NORM_NONE) throw Error("corpus_stats: norm is NONE");
        run_reduce(b);
        if (d_stats) *d_stats = b->plan.stats();
        if (stats_len) *stats_len = (4 * b->d.width + 1) * b->plan.n_groups;
    });
}

int afe_batch_set_corpus_stats(afe_batch *b, const double *h_stats, int stats_len)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        if (b->d.p.norm == AFE_NORM_NONE) throw Error("set_corpus_stats: norm is NONE");
        if (stats_len != (4 * b->d.width + 1) * b->plan.n_groups) throw Error("set_corpus_stats: wrong length");
        AFE_CUDA(cudaMemcpyAsync(b->plan.stats(), h_stats, sizeof(double) * stats_len, cudaMemcpyHostToDevice, b->stream));
        AFE_CUDA(cudaStreamSynchronize(b->stream));
    });
}

int afe_batch_normalize_device(afe_batch *b, float *d_out)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        if (b->d.p.norm == AFE_NORM_NONE) return;
        run_normalize(b, d_out);
    });
}

int afe_batch_synchronize(afe_batch *b)
{
    return guarded([&] { DeviceGuard g(b->device); AFE_CUDA(cudaStreamSynchronize(b->stream)); });
}

// End to end with host buffers. h_pcm / h_out should be pinned for full PCIe speed (pageable memory works too).
// The shard is cut into utterance chunks and pipelined over three streams: H2D of chunk c+1, the kernels of
// chunk c and D2H of chunk c-1 overlap (PCIe is full duplex), so the call is bound by max(H2D, D2H) instead of their sum.
int afe_batch_run_host(afe_batch *b, const int16_t *h_pcm, float *h_out)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        const Derived &d = b->d;
        const afe_batch::Plan &pl = b->plan;
        if (!pl.tiles.p) throw Error("afe_batch_plan must be called before running");
        if (b->scope == AFE_STATS_CORPUS && d.p.norm != AFE_NORM_NONE)
            throw Error("run_host: corpus statistics need the two-pass device sequence");
        const size_t n_samples = (size_t)pl.pcm_extent;
        const size_t pcm_len = n_samples + 16, out_len = (size_t)pl.frame_off.back() * d.width;
        if (pcm_len > b->pcm_stage.n) b->pcm_stage.alloc(pcm_len);
        if (out_len > b->out_stage.n) b->out_stage.alloc(out_len);
        if (!b->s_in) { b->s_in.create(); b->s_out.create(); }
        // chunks are contiguous in samples only when the utterances are packed in increasing order
        bool ordered = true;
        for (int u = 0; u + 1 < pl.n_utts; u++) ordered = ordered && pl.sample_off[u] + pl.sample_len[u] <= pl.sample_off[u + 1];
        const int n_chunks = ordered ? std::max(1, std::min(32, pl.n_utts / 8)) : 1;
        while ((int)b->ev_in.size() < n_chunks) {
            Event e1, e2;
            e1.create(); e2.create();
            b->ev_in.push_back(std::move(e1)); b->ev_k.push_back(std::move(e2));
        }
        b->last_launches = 0;
        const bool norm = d.p.norm != AFE_NORM_NONE;
        for (int c = 0; c < n_chunks; c++) {
            const int u0 = (int)((int64_t)pl.n_utts * c / n_chunks), u1 = (int)((int64_t)pl.n_utts * (c + 1) / n_chunks);
            if (u1 <= u0) continue;
            const int64_t s0 = n_chunks == 1 ? 0 : pl.sample_off[u0];
            const int64_t s1 = n_chunks == 1 ? (int64_t)n_samples : pl.sample_off[u1 - 1] + pl.sample_len[u1 - 1];
            AFE_CUDA(cudaMemcpyAsync(b->pcm_stage.p + s0, h_pcm + s0, (size_t)(s1 - s0) * 2, cudaMemcpyHostToDevice, b->s_in));
            AFE_CUDA(cudaEventRecord(b->ev_in[c], b->s_in));
            AFE_CUDA(cudaStreamWaitEvent(b->stream, b->ev_in[c], 0));
            const int t0 = pl.h_tile_begin[u0], t1 = pl.h_tile_begin[u1];
            const bool fuse = b->fuse_norm();
            run_extract(b, b->pcm_stage.p, b->out_stage.p, t0, t1, fuse);
            if (norm && !fuse) { run_reduce(b, u0, u1); run_normalize(b, b->out_stage.p, t0, t1, u0, u1); }
            AFE_CUDA(cudaEventRecord(b->ev_k[c], b->stream));
            AFE_CUDA(cudaStreamWaitEvent(b->s_out, b->ev_k[c], 0));
            const size_t r0 = (size_t)pl.frame_off[u0] * d.width, r1 = (size_t)pl.frame_off[u1] * d.width;
            AFE_CUDA(cudaMemcpyAsync(h_out + r0, b->out_stage.p + r0, (r1 - r0) * 4, cudaMemcpyDeviceToHost, b->s_out));
        }
        AFE_CUDA(cudaStreamSynchronize(b->s_out));
        AFE_CUDA(cudaStreamSynchronize(b->stream));
    });
}

} // extern "C"
