// Host side of the fused kernel K1, shared by the batch extractor (afe_batch.cu) and the streaming object (afe_stream.cu):
// tables, shared-memory layout, tile planning and the launch (plain, clustered, or the long-utterance role scheme).
#pragma once
#include <vector>

#include "afe_internal.h"
#include "afe_fused_launch.h"

namespace afe {

// Why the fused kernel cannot serve a parameter set (empty string: it can). Everything else runs the staged kernels.
std::string fused_unsupported_reason(const Derived &d);

// Device state of K1's in-kernel normalisation for n_groups groups over n_tiles tiles. The counters reset themselves in
// the kernel; the flags hold the epoch of the last role launch, so the epoch lives with them.
struct FusedNormState {
    DevBuf<double> partials;     // [n_tiles][width][4] per-tile statistics records
    DevBuf<int> counters;        // [n_groups] arrival tickets + [1] role tickets of the long-utterance scheme
    DevBuf<unsigned> flags;      // [n_groups]
    unsigned epoch = 0;
    DevBuf<float> mean, scale;   // [n_groups][width] finalised statistics
    void alloc(int n_groups, size_t n_tiles, int width); // zeroes counters and flags, resets epoch
};

struct FusedEngine {
    Derived d;
    int device = 0, sm_count = 0;
    FftTables fft;
    MelTables mel;               // window tables only (the mel weights travel in `mc` / `mc_wide`)
    MelConst mc;                 // up to 64 banks
    MelConstWide mc_wide;        // 65..128 banks (KF = 16)
    MelConstCeps mc_ceps;        // ceps_len + c0 = 17..48 (NC = 48, up to 64 banks)
    MelConst1024 mc1024;         // 1024 points, up to 64 banks
    MelConstWide1024 mc_wide1024; // 1024 points, 65..128 banks
    float mc_alpha = -1.f;
    bool pruned = false;         // zero-padded window tail: the first FFT layer is pruned (NZ = 13)
    bool window_set = false;
    float pre = 0.f;             // pre-emphasis coefficient
    FusedSmem L{};
    int tc_max = 0, nout_max = 0;
    int kf = 0;                  // filters per warp of the instantiation: 3, 5, 8 or 16
    int nc = 16;                 // DCT column capacity of the instantiation: 16 or 48
    int ctas_per_sm = 2;         // resident CTAs per SM the tile planning counts on: 1 at 1024 points (DESIGN §4)

    explicit FusedEngine(const Derived &dd, int dev);

    void set_window(const float *window, cudaStream_t st);
    void ensure_mel(float alpha);   // rebuilds the constant-bank tables when alpha changed (refresh_filters, mfcccpu.cpp:24-60)
    int launch_key() const { return fused_key(d.N2, pruned ? 13 : 16, kf, pre != 0.f, nc); }
    const void *mel_const() const
    {
        if (d.N2 == 1024) return kf == 16 ? (const void *)&mc_wide1024 : (const void *)&mc1024;
        return nc > 16 ? (const void *)&mc_ceps : kf == 16 ? (const void *)&mc_wide : (const void *)&mc;
    }
    // the instantiation that runs, e.g. "k_fused_mfcc<512,13,8,5,false>" or, with NC = 48, "k_fused_mfcc<512,13,8,5,false,48>"
    std::string kernel_label() const;
    // Tiles for the output rows [t_first, t_first + n_out) of a sequence of T frames whose PCM starts at sample pcm_off;
    // output row of frame t = out_row0 + t. Appends to `tiles`; returns the number of tiles added.
    // nout_cap: largest tile (output frames), 0 = as large as the kernel's cepstra buffer allows (best throughput for big
    // batches); the streaming object passes a smaller one so that a single block spreads over the whole GPU.
    int plan_rows(std::vector<Tile> &tiles, long long pcm_off, long long out_row0, int T, int t_first, int n_out, int group,
                  int nout_cap = 0) const;
    // the split plan_rows makes: ntile tiles of nout output frames each (the last one shorter)
    void plan_uniform(int T, int t_first, int n_out, int nout_cap, int &ntile, int &nout) const;
    int latency_tile(int n_out) const; // nout_cap that cuts n_out rows into about two tiles per SM (whole 32-frame rounds)
    // Arguments common to every launch; the caller fills out / tiles and the statistics / normalisation fields. The PCM is
    // staged with TMA when tma_ok (the caller's utterances start 16-byte aligned), S % 8 == 0 and pcm is 16-byte aligned.
    FusedArgs base_args(int flags_q1, const int16_t *pcm, bool tma_ok) const;
    // K1 writes per-tile statistics records (rows_mode, count: FusedArgs::stats_rows_mode / stats_count)
    void set_stats(FusedArgs &a, FusedNormState &ns, int rows_mode, int count = 0) const
    {
        a.partials = ns.partials.p; a.stats_rows_mode = rows_mode; a.stats_count = count;
        a.stats_kind = d.p.norm == AFE_NORM_CMN ? 1 : d.p.norm == AFE_NORM_CVN ? 2 : 3;
    }
    // deltas and delta-deltas with the default regression windows: the only shape the clustered scheme serves
    bool default_regression() const { return d.width == 3 * d.cols && d.l1 == 3 && d.l2 == 3; }
    bool cluster_schedulable(int cluster, const FusedArgs &a, cudaStream_t st);

    // One launch each. The in-kernel normalisation schemes (see FusedArgs) take their state from `ns`.
    void launch_plain(const FusedArgs &a, int grid, cudaStream_t st) { launch(a, grid, 0, st); } // none, or use_last
    // a group's last tile normalises it
    void launch_ticket(FusedArgs a, int grid, FusedNormState &ns, cudaStream_t st) { a.counters = ns.counters.p; launch(a, grid, 0, st); }
    void launch_roles(FusedArgs a, int ntiles, FusedNormState &ns, cudaStream_t st); // + one wave of normaliser CTAs
    // one thread-block cluster of `cluster` tiles per group; a refused launch runs the ticket scheme instead
    void launch_clustered(FusedArgs a, int grid, int cluster, FusedNormState &ns, cudaStream_t st);

private:
    int cluster_probe[5] = {-1, -1, -1, -1, -1}; // max active clusters per cluster size (lazy; 0 = not schedulable)
    void launch(const FusedArgs &a, int grid, int cluster, cudaStream_t st);
};

} // namespace afe
