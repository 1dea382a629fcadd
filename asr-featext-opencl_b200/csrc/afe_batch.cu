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
    release();
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
    AFE_CUDA(cudaMalloc(&d_tw_a, a.size() * sizeof(float2)));
    AFE_CUDA(cudaMalloc(&d_tw_p, p.size() * sizeof(float2)));
    AFE_CUDA(cudaMemcpy(d_tw_a, a.data(), a.size() * sizeof(float2), cudaMemcpyHostToDevice));
    AFE_CUDA(cudaMemcpy(d_tw_p, p.data(), p.size() * sizeof(float2), cudaMemcpyHostToDevice));
}
void FftTables::release()
{
    if (d_tw_a) cudaFree(d_tw_a);
    if (d_tw_p) cudaFree(d_tw_p);
    d_tw_a = d_tw_p = nullptr;
}

void MelTables::release()
{
    if (d_edges) cudaFree(d_edges);
    if (d_pairs) cudaFree(d_pairs);
    if (d_dct) cudaFree(d_dct);
    if (d_window) cudaFree(d_window);
    if (d_window2) cudaFree(d_window2);
    d_edges = nullptr; d_pairs = nullptr; d_dct = nullptr; d_window = nullptr; d_window2 = nullptr;
    alpha_built = -1.f;
}

void upload_mel_tables(const Derived &d, float alpha, MelTables &t, cudaStream_t st)
{
    std::vector<int> edges; std::vector<float> filters, pairs, dct;
    build_filters(d, alpha, edges, filters);
    for (int i = 0; i + 1 < (int)edges.size(); i++)
        if (edges[i + 1] < edges[i]) throw Error("mel filter edges are not monotonic");
    if (edges.front() < 0 || edges.back() > d.M) throw Error("mel filterbank exceeds the Nyquist bin (check low_freq/high_freq)");
    build_mel_pairs(d, edges, filters, pairs);
    if (!t.d_edges) AFE_CUDA(cudaMalloc(&t.d_edges, sizeof(int) * (d.nb + 2)));
    if (!t.d_pairs) AFE_CUDA(cudaMalloc(&t.d_pairs, sizeof(float) * 2 * d.bins));
    // pageable source + stream-ordered copy: cudaMemcpyAsync from pageable memory stages synchronously, safe with locals
    AFE_CUDA(cudaMemcpyAsync(t.d_edges, edges.data(), sizeof(int) * (d.nb + 2), cudaMemcpyHostToDevice, st));
    AFE_CUDA(cudaMemcpyAsync(t.d_pairs, pairs.data(), sizeof(float) * 2 * d.bins, cudaMemcpyHostToDevice, st));
    if (d.C > 0 && !t.d_dct) {
        build_dct(d, dct);
        AFE_CUDA(cudaMalloc(&t.d_dct, sizeof(float) * dct.size()));
        AFE_CUDA(cudaMemcpyAsync(t.d_dct, dct.data(), sizeof(float) * dct.size(), cudaMemcpyHostToDevice, st));
    }
    AFE_CUDA(cudaStreamSynchronize(st));
    t.alpha_built = alpha;
}

void upload_window(const Derived &d, const float *window, MelTables &t, cudaStream_t st)
{
    if (!t.d_window) AFE_CUDA(cudaMalloc(&t.d_window, sizeof(float) * d.W));
    if (!t.d_window2) AFE_CUDA(cudaMalloc(&t.d_window2, sizeof(float2) * d.M));
    std::vector<float> w2((size_t)d.N2, 0.f);
    memcpy(w2.data(), window, sizeof(float) * d.W);
    AFE_CUDA(cudaMemcpyAsync(t.d_window, window, sizeof(float) * d.W, cudaMemcpyHostToDevice, st));
    AFE_CUDA(cudaMemcpyAsync(t.d_window2, w2.data(), sizeof(float) * d.N2, cudaMemcpyHostToDevice, st));
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
    X(18) X(19) X(20) X(21) X(22) X(23)
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
    if (d.N2 != 512 && d.N2 != 256) return "fused path supports 256/512-point FFTs (window_size 129..512)";
    if (d.S % 2) return "fused path needs an even shift";
    if (d.dct_len > 16) return "fused path supports ceps_len + c0 <= 16";
    if (d.width > 128) return "fused path supports output width <= 128";
    if (d.nb > kMaxBanks) return "fused path supports num_banks <= 64";
    if (d.W > 26 * (d.M / 16) && d.W > d.N2) return "window longer than the FFT";
    return "";
}

// Mel weights + DCT matrix as a by-value kernel parameter (constant bank). Per filter b: bins [edges[b], edges[b+2]) with
// weights filters[b%2][bin] — the per-filter form of the reference's two-running-sums sweep (mfcccpu.cpp:192-220).
static void build_mel_const(const Derived &d, float alpha, MelConst &mc)
{
    std::vector<int> edges; std::vector<float> filters, dct;
    build_filters(d, alpha, edges, filters);
    for (int i = 0; i + 1 < (int)edges.size(); i++)
        if (edges[i + 1] < edges[i]) throw Error("mel filter edges are not monotonic");
    if (edges.front() < 0 || edges.back() > d.M) throw Error("mel filterbank exceeds the Nyquist bin (check low_freq/high_freq)");
    memset(&mc, 0, sizeof mc);
    int off4 = 0;
    const float scale = 0.5f / (float)d.N2; // the kernel stores |2X|; scaling by a power of two commutes with rounding
    for (int w = 0; w < 8; w++) {           // warp class w owns the filters w, w + 8, ...: their lists are contiguous
        mc.wstart[w] = (short)off4;
        for (int b = w; b < d.nb; b += 8) {
            const int j0 = edges[b], j1 = edges[b + 2], s4 = j0 & ~3, n8 = std::max(1, (j1 - s4 + 7) / 8);
            if (off4 + 2 * n8 > kMaxWl4) throw Error("mel weight list exceeds the kernel-parameter budget");
            if (s4 + 8 * n8 > kMagStride + 16) throw Error("mel filter too wide for the fused kernel");
            mc.desc[b] = (s4 / 4) | (n8 << 16);
            float *wt = reinterpret_cast<float *>(mc.wl4 + off4);
            for (int j = j0; j < j1; j++) wt[j - s4] = filters[(size_t)(b % 2) * d.N2 + j] * scale;
            off4 += 2 * n8;
        }
    }
    if (d.C > 0) {
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
    // tile geometry (2 CTAs per SM): the cepstra tile holds up to 512 frames (<= 27 KB of shared memory)
    int tc = 512;
    tc = std::min(tc, (6912 / d.cols) / kRoundFrames * kRoundFrames);
    tc = std::max(tc, kRoundFrames * ((2 * d.D + 1 + kRoundFrames - 1) / kRoundFrames + 1));
    tc_max = tc; nout_max = tc - 2 * d.D;
    const int ns = d.width / d.cols;
    L = d.N2 == 512 ? fused_smem_layout<512>(8, d.S, d.cols, tc_max, nout_max, d.l2, ns)
                    : fused_smem_layout<256>(8, d.S, d.cols, tc_max, nout_max, d.l2, ns);
    if (L.total > 227 * 1024) throw Error("fused kernel shared-memory budget exceeded");
    const int R = d.M / 16;
    pruned = d.W <= 26 * R;            // window tail is zero from n1 = 13 on (400/512 and 200/256 both qualify)
    const int kf = (d.nb + 7) / 8;     // filters per warp (8 warps): instantiated for 3, 5 and 8
    key = (d.N2 == 512 ? 0 : 6) + (pruned ? 0 : 3) + (kf <= 3 ? 0 : kf <= 5 ? 1 : 2);
}
FusedEngine::~FusedEngine() { fft.release(); mel.release(); }

void FusedEngine::set_window(const float *window, cudaStream_t st)
{
    upload_window(d, window, mel, st);
    window_set = true;
}
void FusedEngine::ensure_mel(float alpha)
{
    if (mc_alpha != alpha) { build_mel_const(d, alpha, mc); mc_alpha = alpha; }
}
std::string FusedEngine::kernel_label() const
{
    const int kf = (d.nb + 7) / 8;
    char buf[96];
    snprintf(buf, sizeof buf, "k_fused_mfcc<%d,%d,8,%d,%s>", d.N2, pruned ? 13 : 16, kf <= 3 ? 3 : kf <= 5 ? 5 : 8,
             pre != 0.f ? "true" : "false");
    return buf;
}

int FusedEngine::latency_tile(int n_out) const
{
    const int target = std::max(1, 2 * sm_count);
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

FusedArgs FusedEngine::base_args(int q1, bool use_tma) const
{
    FusedArgs a{};
    a.window2 = mel.d_window2; a.tw_a = fft.d_tw_a; a.tw_p = fft.d_tw_p;
    a.norm_type = d.p.norm; a.norm_after_dyn = d.p.norm_after_dyn;
    a.W = d.W; a.S = d.S; a.nb = d.nb; a.dct_len = d.C > 0 ? d.dct_len : 0; a.cols = d.cols; a.width = d.width;
    a.l1 = d.l1; a.l2 = d.l2; a.nstreams = d.width / d.cols;
    a.q1 = d.D > 0 ? q1 : 0;
    a.use_tma = use_tma ? 1 : 0;
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
        FusedLaunch fl{a, L, &mc, cluster, cluster, st};
        const int n = fused_variant_max_clusters(key, fl); // same footprint with and without pre-emphasis
        cluster_probe[cluster] = n > 0 ? n : 0;
    }
    return cluster_probe[cluster] > 0;
}

void FusedEngine::launch(const FusedArgs &a, int grid, int cluster, cudaStream_t st)
{
    if (!window_set) throw Error("set_window must be called before running");
    FusedLaunch fl{a, L, &mc, grid, cluster, st};
    const cudaError_t e = launch_fused_variant(key + (a.pre != 0.f ? 12 : 0), fl);
    if (e != cudaSuccess) {
        cudaGetLastError();
        throw Error(std::string("CUDA error: ") + cudaGetErrorString(e) + " at k_fused_mfcc launch" + (cluster > 0 ? " (clustered)" : ""));
    }
    count_launch();
}

} // namespace afe

using namespace afe;

// ================================================================================================== afe_batch
struct afe_batch {
    Derived d;
    int device;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::unique_ptr<FusedEngine> eng;
    float alpha = 1.f;
    int scope = AFE_STATS_REFERENCE_BLOCK, flags = 0;
    // plan
    int n_utts = 0, n_tiles = 0, n_groups = 0;
    bool aligned = false;
    std::vector<int64_t> sample_off, sample_len, frame_off;
    std::vector<int> h_tile_begin;          // [n_utts+1] first tile of every utterance
    cudaStream_t s_in = nullptr, s_out = nullptr;
    std::vector<cudaEvent_t> ev_in, ev_k;
    int64_t pcm_extent = 0;
    Tile *d_tiles = nullptr;
    int *d_tile_begin = nullptr;
    double *d_counts = nullptr, *d_partials = nullptr, *d_stats = nullptr, *d_scratch = nullptr;
    int *d_counters = nullptr;      // [n_groups] arrival tickets + [1] role tickets of the long-utterance scheme
    unsigned *d_flags = nullptr;    // [n_groups]
    unsigned epoch = 0;
    int *d_scratch_begin = nullptr;
    float *d_mean = nullptr, *d_scale = nullptr;
    int corpus_blocks = 0;          // level-1 blocks of the corpus reduction (2 per SM)
    afe_normalizer *cnorm = nullptr; // corpus scope: the Normalizer that owns the record (d_stats aliases its buffer)
    int max_tiles_per_utt = 0;
    // One tile normalising its whole utterance is right for short utterances and a serial bottleneck for long ones:
    // up to 8 tiles -> clusters / ticket scheme; more -> the role scheme (normaliser CTAs, one per tile, same launch).
    bool fuse_norm() const { return !(flags & AFE_BATCH_UNFUSED_NORM); }
    bool long_scheme() const { return max_tiles_per_utt > 8; }
    int last_launches = 0;
    // host staging for run_host
    int16_t *d_pcm_stage = nullptr; float *d_out_stage = nullptr;
    size_t pcm_stage_bytes = 0, out_stage_bytes = 0;

    explicit afe_batch(const afe_params &p, int dev) : d(p), device(dev) {}
    void free_plan()
    {
        if (d_tiles) cudaFree(d_tiles);
        if (d_tile_begin) cudaFree(d_tile_begin);
        if (d_counts) cudaFree(d_counts);
        if (d_partials) cudaFree(d_partials);
        if (d_stats && !cnorm) cudaFree(d_stats);
        if (d_scratch) cudaFree(d_scratch);
        if (d_counters) cudaFree(d_counters);
        if (d_flags) cudaFree(d_flags);
        if (d_scratch_begin) cudaFree(d_scratch_begin);
        if (d_mean) cudaFree(d_mean);
        if (d_scale) cudaFree(d_scale);
        if (cnorm) { cnorm->st = nullptr; afe_normalizer_destroy(cnorm); cnorm = nullptr; }
        d_tiles = nullptr; d_tile_begin = nullptr; d_counts = d_partials = d_stats = d_scratch = nullptr;
        d_counters = nullptr; d_flags = nullptr; d_scratch_begin = nullptr; d_mean = d_scale = nullptr;
    }
};

static FusedArgs make_fused_args(afe_batch *b, const int16_t *d_pcm, float *d_out, bool want_stats, int t0)
{
    const Derived &d = b->d;
    const bool tma = b->aligned && !(b->flags & AFE_BATCH_NO_TMA) && (reinterpret_cast<uintptr_t>(d_pcm) & 15) == 0;
    FusedArgs a = b->eng->base_args((b->flags & AFE_BATCH_Q1_EXACT) ? 1 : 0, tma);
    a.pcm = d_pcm; a.out = d_out; a.tiles = b->d_tiles; a.tile_base = t0;
    a.partials = want_stats ? b->d_partials : nullptr;
    if (!want_stats) a.stats_rows_mode = 0;
    else if (!d.p.norm_after_dyn) a.stats_rows_mode = 2;
    else a.stats_rows_mode = b->scope == AFE_STATS_REFERENCE_BLOCK ? 1 : 2;
    a.stats_kind = !want_stats ? 0 : (d.p.norm == AFE_NORM_CMN ? 1 : d.p.norm == AFE_NORM_CVN ? 2 : 3);
    return a;
}

// Tiles [t0, t1) (whole utterances) through K1. With fused normalisation:
//  * the default regression and utterances of 1..4 tiles: runs of equal tile count become ONE clustered launch each
//    (cluster = utterance, statistics through distributed shared memory), at most kMaxClusterRuns launches;
//  * other batches whose utterances have at most 8 tiles: the ticket scheme (last tile normalises through L2), one launch;
//  * batches with longer utterances: the role scheme (2 x tiles CTAs, the second half normalises a tile each), one launch.
constexpr int kMaxClusterRuns = 8;
constexpr int kMaxClusterTiles = 4; // utterances of up to 4 tiles (~20 s) form a cluster; longer ones keep the ticket scheme
static void run_extract(afe_batch *b, const int16_t *d_pcm, float *d_out, int t0 = 0, int t1 = -1, bool fuse_norm = false)
{
    if (t1 < 0) t1 = b->n_tiles;
    if (t1 <= t0) return;
    if (!b->d_tiles) throw Error("afe_batch_plan must be called before running");
    FusedEngine &eng = *b->eng;
    eng.ensure_mel(b->alpha);
    const Derived &d = b->d;
    const bool want_stats = d.p.norm != AFE_NORM_NONE;
    FusedArgs a = make_fused_args(b, d_pcm, d_out, want_stats, t0);
    auto launch = [&](const FusedArgs &args, int grid, int cluster) { eng.launch(args, grid, cluster, b->stream); b->last_launches++; };
    if (!(fuse_norm && want_stats)) { launch(a, t1 - t0, 0); return; }
    if (b->long_scheme()) {
        a.counters = b->d_counters; a.work_counter = b->d_counters + b->n_groups;
        a.flags = b->d_flags; a.epoch = ++b->epoch; a.ntiles_launch = t1 - t0;
        a.g_mean = b->d_mean; a.g_scale = b->d_scale;
        launch(a, (t1 - t0) + std::min(t1 - t0, 2 * eng.sm_count), 0); // + one wave of normaliser roles
        return;
    }
    const bool cluster_ok = !(b->flags & AFE_BATCH_NO_CLUSTER) && d.width == 3 * d.cols && d.l1 == 3 && d.l2 == 3;
    if (cluster_ok) {
        struct Run { int t0, t1, cluster; };
        std::vector<Run> runs;
        const int u0 = (int)(std::lower_bound(b->h_tile_begin.begin(), b->h_tile_begin.end(), t0) - b->h_tile_begin.begin());
        bool schedulable = true;
        for (int u = u0; u < b->n_utts && b->h_tile_begin[u] < t1 && (int)runs.size() <= kMaxClusterRuns; u++) {
            const int nt = b->h_tile_begin[u + 1] - b->h_tile_begin[u], cl = nt <= kMaxClusterTiles ? nt : 0;
            if (cl > 0 && !eng.cluster_schedulable(cl, a, b->stream)) { schedulable = false; break; }
            if (!runs.empty() && runs.back().cluster == cl) runs.back().t1 = b->h_tile_begin[u + 1];
            else runs.push_back({b->h_tile_begin[u], b->h_tile_begin[u + 1], cl});
        }
        if (schedulable && (int)runs.size() <= kMaxClusterRuns && !runs.empty() && runs.front().t0 == t0 && runs.back().t1 == t1) {
            for (const Run &r : runs) {
                FusedArgs ar = a;
                ar.tile_base = r.t0;
                if (r.cluster > 0) { ar.cluster_norm = 1; ar.counters = nullptr; }
                else ar.counters = b->d_counters;
                try {
                    launch(ar, r.t1 - r.t0, r.cluster);
                } catch (const Error &) {
                    if (r.cluster == 0) throw;
                    // the clustered launch was refused (nothing ran): this run takes the ticket scheme instead
                    eng.cluster_probe[r.cluster] = 0;
                    ar.cluster_norm = 0; ar.counters = b->d_counters;
                    launch(ar, r.t1 - r.t0, 0);
                }
            }
            return;
        }
    }
    a.counters = b->d_counters;
    launch(a, t1 - t0, 0);
}

static void run_reduce(afe_batch *b, int g0 = 0, int g1 = -1)
{
    if (g1 < 0) g1 = b->n_groups;
    if (g1 <= g0) return;
    const int w = b->d.width;
    if (b->scope == AFE_STATS_CORPUS && b->n_tiles > 2 * b->corpus_blocks) {
        k_reduce_partials_level1<<<b->corpus_blocks, 128, 0, b->stream>>>(b->d_partials, b->n_tiles, w, b->d_scratch);
        AFE_CUDA(cudaGetLastError());
        k_reduce_partials<<<1, 256, dev::kSegs * w * 4 * sizeof(double), b->stream>>>(b->d_scratch, b->d_scratch_begin, b->d_counts, w, b->d_stats);
        AFE_CUDA(cudaGetLastError());
        count_launch(2); b->last_launches += 2;
        return;
    }
    k_reduce_partials<<<g1 - g0, 256, dev::kSegs * w * 4 * sizeof(double), b->stream>>>(b->d_partials, b->d_tile_begin + g0, b->d_counts + g0, w,
                                                                                       b->d_stats + (size_t)g0 * (4 * w + 1));
    AFE_CUDA(cudaGetLastError());
    count_launch(); b->last_launches++;
}

static void run_normalize(afe_batch *b, float *d_out, int t0 = 0, int t1 = -1, int g0 = 0, int g1 = -1)
{
    const Derived &d = b->d;
    if (t1 < 0) t1 = b->n_tiles;
    if (g1 < 0) g1 = b->n_groups;
    if (t1 <= t0 || g1 <= g0) return;
    const size_t w = d.width;
    k_finalize_stats<<<g1 - g0, 128, 0, b->stream>>>(b->d_stats + (size_t)g0 * (4 * w + 1), d.width, d.cols, d.p.norm,
                                                      d.p.norm_after_dyn, b->d_mean + g0 * w, b->d_scale + g0 * w);
    AFE_CUDA(cudaGetLastError());
    // Tile::group is absolute, so mean / scale keep their base
    k_normalize_tiles<<<t1 - t0, 256, 2 * d.width * sizeof(float), b->stream>>>(d_out, b->d_tiles + t0, d.width, d.p.norm,
                                                                              b->d_mean, b->d_scale);
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
        std::unique_ptr<afe_batch> b(new afe_batch(*p, cuda_device));
        const std::string why = fused_unsupported_reason(b->d);
        if (!why.empty()) throw Error(why + "; use the streaming object");
        DeviceGuard g(cuda_device);
        AFE_CUDA(cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking));
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
    b->free_plan();
    b->eng.reset();
    if (b->d_pcm_stage) cudaFree(b->d_pcm_stage);
    if (b->d_out_stage) cudaFree(b->d_out_stage);
    if (b->own_stream) cudaStreamDestroy(b->own_stream);
    if (b->s_in) cudaStreamDestroy(b->s_in);
    if (b->s_out) cudaStreamDestroy(b->s_out);
    for (auto e : b->ev_in) cudaEventDestroy(e);
    for (auto e : b->ev_k) cudaEventDestroy(e);
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
        if (b->d_tiles && stats_scope != b->scope) throw Error("set the statistics scope before afe_batch_plan");
        const int known = AFE_BATCH_Q1_EXACT | AFE_BATCH_NO_TMA | AFE_BATCH_UNFUSED_NORM | AFE_BATCH_NO_CLUSTER;
        if (flags & ~known) throw Error("unknown batch flag bits " + std::to_string(flags & ~known));
        b->scope = stats_scope; b->flags = flags; // every flag is read at run time
    });
}

int afe_batch_set_stream(afe_batch *b, void *cuda_stream)
{
    b->stream = cuda_stream ? (cudaStream_t)cuda_stream : b->own_stream;
    if (b->cnorm) b->cnorm->st = b->stream;
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
        b->free_plan();
        const FusedEngine &eng = *b->eng;
        b->n_utts = n_utts;
        b->sample_off.assign(off, off + n_utts);
        b->sample_len.assign(len, len + n_utts);
        b->h_tile_begin.assign(n_utts + 1, 0);
        b->max_tiles_per_utt = 0;
        b->pcm_extent = 0;
        b->frame_off.assign(n_utts + 1, 0);
        std::vector<Tile> tiles;
        std::vector<int> tile_begin;
        std::vector<double> counts;
        const bool corpus = b->scope == AFE_STATS_CORPUS;
        if (seg_first && d.p.norm != AFE_NORM_NONE && !corpus)
            throw Error("plan_segments: normalisation over segments needs the CORPUS statistics scope");
        bool aligned = d.S % 8 == 0;
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
            const int slots = 2 * eng.sm_count;
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
            b->pcm_extent = std::max<int64_t>(b->pcm_extent, off[u] + n);
            if (off[u] % 2) throw Error("plan: utterance offsets must be even (32-bit PCM word loads)");
            if (off[u] % 8) aligned = false;
            // parambase.cpp:16-19 evaluates in float32, which is inexact above 2^24 samples: never let it exceed the
            // exact count (the extra frame would lie outside the utterance)
            const int T = std::min(afe_estimated_window_count((int)n, d.W, d.S), (int)std::max<int64_t>(0, (n - (d.W - d.S)) / d.S));
            if (T <= 2 * d.D || T < 1) throw Error("Can't process data, window count is too small"); // segmentercpu.cpp:65-66
            const int t_first = seg_first ? seg_first[u] : 0, rows = seg_rows ? seg_rows[u] : T;
            if (t_first < 0 || rows < 1 || t_first + rows > T) throw Error("plan_segments: segment outside its frames");
            b->frame_off[u + 1] = b->frame_off[u] + rows;
            b->h_tile_begin[u] = (int)tiles.size();
            if (!corpus) tile_begin.push_back((int)tiles.size());
            const int ntile = eng.plan_rows(tiles, off[u], b->frame_off[u] - t_first, T, t_first, rows, corpus ? 0 : u, nout_cap);
            b->max_tiles_per_utt = std::max(b->max_tiles_per_utt, ntile);
            const double cnt = seg_first ? rows : !d.p.norm_after_dyn ? T : (b->scope == AFE_STATS_REFERENCE_BLOCK ? T - d.D : T);
            if (corpus) corpus_count += cnt; else counts.push_back(cnt);
        }
        if (corpus) { tile_begin.push_back(0); counts.push_back(corpus_count); }
        tile_begin.push_back((int)tiles.size());
        b->h_tile_begin[n_utts] = (int)tiles.size();
        b->aligned = aligned;
        b->n_tiles = (int)tiles.size();
        b->n_groups = corpus ? 1 : n_utts;
        b->corpus_blocks = 2 * eng.sm_count;
        AFE_CUDA(cudaMalloc(&b->d_tiles, sizeof(Tile) * tiles.size()));
        AFE_CUDA(cudaMemcpy(b->d_tiles, tiles.data(), sizeof(Tile) * tiles.size(), cudaMemcpyHostToDevice));
        if (d.p.norm != AFE_NORM_NONE) {
            const size_t w = d.width;
            AFE_CUDA(cudaMalloc(&b->d_tile_begin, sizeof(int) * tile_begin.size()));
            AFE_CUDA(cudaMemcpy(b->d_tile_begin, tile_begin.data(), sizeof(int) * tile_begin.size(), cudaMemcpyHostToDevice));
            AFE_CUDA(cudaMalloc(&b->d_counts, sizeof(double) * counts.size()));
            AFE_CUDA(cudaMemcpy(b->d_counts, counts.data(), sizeof(double) * counts.size(), cudaMemcpyHostToDevice));
            AFE_CUDA(cudaMalloc(&b->d_partials, sizeof(double) * 4 * w * tiles.size()));
            if (corpus) {
                // the corpus record lives in a Normalizer of dim = width (all three streams in one record)
                if (afe_normalizer_create(d.p.norm, d.width, b->device, &b->cnorm) != 0) throw Error(afe_last_error());
                b->cnorm->st = b->stream;
                b->d_stats = b->cnorm->ns.rec.p;
                const int sb[2] = {0, b->corpus_blocks};
                AFE_CUDA(cudaMalloc(&b->d_scratch, sizeof(double) * 4 * w * b->corpus_blocks));
                AFE_CUDA(cudaMalloc(&b->d_scratch_begin, sizeof(sb)));
                AFE_CUDA(cudaMemcpy(b->d_scratch_begin, sb, sizeof(sb), cudaMemcpyHostToDevice));
            } else
                AFE_CUDA(cudaMalloc(&b->d_stats, sizeof(double) * (4 * w + 1) * b->n_groups));
            AFE_CUDA(cudaMalloc(&b->d_counters, sizeof(int) * (b->n_groups + 1)));
            AFE_CUDA(cudaMemset(b->d_counters, 0, sizeof(int) * (b->n_groups + 1)));
            AFE_CUDA(cudaMalloc(&b->d_flags, sizeof(unsigned) * b->n_groups));
            AFE_CUDA(cudaMemset(b->d_flags, 0, sizeof(unsigned) * b->n_groups));
            b->epoch = 0;
            AFE_CUDA(cudaMalloc(&b->d_mean, sizeof(float) * w * b->n_groups));
            AFE_CUDA(cudaMalloc(&b->d_scale, sizeof(float) * w * b->n_groups));
        }
        if (total_frames) *total_frames = b->frame_off[n_utts];
    });
}

int afe_batch_frame_offsets(const afe_batch *b, int64_t *fo)
{
    memcpy(fo, b->frame_off.data(), sizeof(int64_t) * b->frame_off.size());
    return 0;
}
int afe_batch_num_tiles(const afe_batch *b) { return b->n_tiles; }
int afe_batch_kernel_launches(const afe_batch *b) { return b->last_launches; }
const char *afe_batch_kernel_name(const afe_batch *b)
{
    static thread_local std::string name;
    name = b->eng ? b->eng->kernel_label() : "k_fused_mfcc";
    return name.c_str();
}
afe_normalizer *afe_batch_normalizer(afe_batch *b) { return b->cnorm; }

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
        if (d_stats) *d_stats = b->d_stats;
        if (stats_len) *stats_len = (4 * b->d.width + 1) * b->n_groups;
    });
}

int afe_batch_set_corpus_stats(afe_batch *b, const double *h_stats, int stats_len)
{
    return guarded([&] {
        DeviceGuard g(b->device);
        if (b->d.p.norm == AFE_NORM_NONE) throw Error("set_corpus_stats: norm is NONE");
        if (stats_len != (4 * b->d.width + 1) * b->n_groups) throw Error("set_corpus_stats: wrong length");
        AFE_CUDA(cudaMemcpyAsync(b->d_stats, h_stats, sizeof(double) * stats_len, cudaMemcpyHostToDevice, b->stream));
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
        if (!b->d_tiles) throw Error("afe_batch_plan must be called before running");
        if (b->scope == AFE_STATS_CORPUS && d.p.norm != AFE_NORM_NONE)
            throw Error("run_host: corpus statistics need the two-pass device sequence");
        const size_t n_samples = (size_t)b->pcm_extent;
        const size_t pcm_bytes = n_samples * 2 + 32, out_bytes = (size_t)b->frame_off.back() * d.width * 4;
        if (pcm_bytes > b->pcm_stage_bytes) {
            if (b->d_pcm_stage) cudaFree(b->d_pcm_stage);
            AFE_CUDA(cudaMalloc(&b->d_pcm_stage, pcm_bytes));
            b->pcm_stage_bytes = pcm_bytes;
        }
        if (out_bytes > b->out_stage_bytes) {
            if (b->d_out_stage) cudaFree(b->d_out_stage);
            AFE_CUDA(cudaMalloc(&b->d_out_stage, out_bytes));
            b->out_stage_bytes = out_bytes;
        }
        if (!b->s_in) {
            AFE_CUDA(cudaStreamCreateWithFlags(&b->s_in, cudaStreamNonBlocking));
            AFE_CUDA(cudaStreamCreateWithFlags(&b->s_out, cudaStreamNonBlocking));
        }
        // chunks are contiguous in samples only when the utterances are packed in increasing order
        bool ordered = true;
        for (int u = 0; u + 1 < b->n_utts; u++) ordered = ordered && b->sample_off[u] + b->sample_len[u] <= b->sample_off[u + 1];
        const int n_chunks = ordered ? std::max(1, std::min(32, b->n_utts / 8)) : 1;
        while ((int)b->ev_in.size() < n_chunks) {
            cudaEvent_t e1, e2;
            AFE_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            AFE_CUDA(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            b->ev_in.push_back(e1); b->ev_k.push_back(e2);
        }
        b->last_launches = 0;
        const bool norm = d.p.norm != AFE_NORM_NONE;
        for (int c = 0; c < n_chunks; c++) {
            const int u0 = (int)((int64_t)b->n_utts * c / n_chunks), u1 = (int)((int64_t)b->n_utts * (c + 1) / n_chunks);
            if (u1 <= u0) continue;
            const int64_t s0 = n_chunks == 1 ? 0 : b->sample_off[u0];
            const int64_t s1 = n_chunks == 1 ? (int64_t)n_samples : b->sample_off[u1 - 1] + b->sample_len[u1 - 1];
            AFE_CUDA(cudaMemcpyAsync(b->d_pcm_stage + s0, h_pcm + s0, (size_t)(s1 - s0) * 2, cudaMemcpyHostToDevice, b->s_in));
            AFE_CUDA(cudaEventRecord(b->ev_in[c], b->s_in));
            AFE_CUDA(cudaStreamWaitEvent(b->stream, b->ev_in[c], 0));
            const int t0 = b->h_tile_begin[u0], t1 = b->h_tile_begin[u1];
            const bool fuse = b->fuse_norm();
            run_extract(b, b->d_pcm_stage, b->d_out_stage, t0, t1, fuse);
            if (norm && !fuse) { run_reduce(b, u0, u1); run_normalize(b, b->d_out_stage, t0, t1, u0, u1); }
            AFE_CUDA(cudaEventRecord(b->ev_k[c], b->stream));
            AFE_CUDA(cudaStreamWaitEvent(b->s_out, b->ev_k[c], 0));
            const size_t r0 = (size_t)b->frame_off[u0] * d.width, r1 = (size_t)b->frame_off[u1] * d.width;
            AFE_CUDA(cudaMemcpyAsync(h_out + r0, b->d_out_stage + r0, (r1 - r0) * 4, cudaMemcpyDeviceToHost, b->s_out));
        }
        AFE_CUDA(cudaStreamSynchronize(b->s_out));
        AFE_CUDA(cudaStreamSynchronize(b->stream));
    });
}

} // extern "C"
