// Host side of the fused kernel K1, shared by the batch extractor (afe_batch.cu) and the streaming object (afe_stream.cu):
// tables, shared-memory layout, tile planning and the launch (plain, clustered, or the long-utterance role scheme).
#pragma once
#include <vector>

#include "afe_internal.h"
#include "afe_fused_launch.h"

namespace afe {

// Why the fused kernel cannot serve a parameter set (empty string: it can). Everything else runs the staged kernels.
std::string fused_unsupported_reason(const Derived &d);

struct FusedEngine {
    Derived d;
    int device = 0, sm_count = 0;
    FftTables fft;
    MelTables mel;               // window tables only (the mel weights travel in `mc`)
    MelConst mc;
    float mc_alpha = -1.f;
    bool pruned = false;         // zero-padded window tail: the first FFT layer is pruned (NZ = 13)
    bool window_set = false;
    float pre = 0.f;             // pre-emphasis coefficient
    FusedSmem L{};
    int tc_max = 0, nout_max = 0, key = 0;
    int cluster_probe[5] = {-1, -1, -1, -1, -1}; // max active clusters per cluster size (lazy; 0 = not schedulable)

    explicit FusedEngine(const Derived &dd, int dev);
    ~FusedEngine();
    FusedEngine(const FusedEngine &) = delete;
    FusedEngine &operator=(const FusedEngine &) = delete;

    void set_window(const float *window, cudaStream_t st);
    void ensure_mel(float alpha);   // rebuilds the constant-bank tables when alpha changed (refresh_filters, mfcccpu.cpp:24-60)
    std::string kernel_label() const; // the instantiation that runs, e.g. "k_fused_mfcc<512,13,8,5,false>"
    // Tiles for the output rows [t_first, t_first + n_out) of a sequence of T frames whose PCM starts at sample pcm_off;
    // output row of frame t = out_row0 + t. Appends to `tiles`; returns the number of tiles added.
    // nout_cap: largest tile (output frames), 0 = as large as the kernel's cepstra buffer allows (best throughput for big
    // batches); the streaming object passes a smaller one so that a single block spreads over the whole GPU.
    int plan_rows(std::vector<Tile> &tiles, long long pcm_off, long long out_row0, int T, int t_first, int n_out, int group,
                  int nout_cap = 0) const;
    // the split plan_rows makes: ntile tiles of nout output frames each (the last one shorter)
    void plan_uniform(int T, int t_first, int n_out, int nout_cap, int &ntile, int &nout) const;
    int latency_tile(int n_out) const; // nout_cap that cuts n_out rows into about two tiles per SM (whole 32-frame rounds)
    // Arguments common to every launch; the caller fills pcm/out/tiles and the statistics / normalisation fields.
    FusedArgs base_args(int flags_q1, bool use_tma) const;
    bool cluster_schedulable(int cluster, const FusedArgs &a, cudaStream_t st);
    void launch(const FusedArgs &a, int grid, int cluster, cudaStream_t st);
};

} // namespace afe
