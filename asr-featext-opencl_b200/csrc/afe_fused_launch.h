// Launch interface of the fused kernel's instantiations. k_fused_mfcc<N2, NZ, 8, KF, PRE[, NC]> is instantiated for 64
// parameter sets, one per translation unit (afe_fused_inst.cu compiled with -DAFE_INST_KEY=0..63) so that they build in parallel.
#pragma once
#include "afe_fused.cuh"

namespace afe {

struct FusedLaunch {
    FusedArgs a;
    FusedSmem L;
    const void *mc;      // MelConstFor<N2, KF, NC>: MelConst, MelConstWide, MelConstCeps, MelConst1024 or MelConstWide1024
    int grid;            // CTAs
    int cluster;         // 0: plain launch; 1..: thread-block cluster size (one cluster = the tiles of one utterance)
    cudaStream_t st;
};

// keys 0..23:  (N2 == 512 ? 0 : 6) + (pruned first layer, NZ = 13 ? 0 : 3) + (KF: 3 -> 0, 5 -> 1, 8 -> 2) + (pre-emphasis ? 12 : 0)
// keys 24..31: 24 + (N2 == 512 ? 0 : 2) + (NZ == 13 ? 0 : 1) + (pre-emphasis ? 4 : 0), KF = 16 (65..128 banks)
// keys 32..47: 32 + (N2 == 512 ? 0 : 4) + (NZ == 13 ? 0 : 2) + (KF == 5 ? 0 : 1) + (pre-emphasis ? 8 : 0), NC = 48
//              (ceps_len + c0 = 17..48)
// keys 48..63: 48 + (NZ == 13 ? 0 : 4) + (KF: 3 -> 0, 5 -> 1, 8 -> 2, 16 -> 3) + (pre-emphasis ? 8 : 0), N2 = 1024
//              (window_size 513..1024); every key but 32..47 has NC = 16
constexpr int kFusedVariants = 64;
constexpr int fused_key(int n2, int nz, int kf, bool pre, int nc = 16)
{
    return n2 == 1024  ? 48 + (nz == 13 ? 0 : 4) + (kf == 3 ? 0 : kf == 5 ? 1 : kf == 8 ? 2 : 3) + (pre ? 8 : 0)
           : nc > 16   ? 32 + (n2 == 512 ? 0 : 4) + (nz == 13 ? 0 : 2) + (kf == 5 ? 0 : 1) + (pre ? 8 : 0)
           : kf == 16 ? 24 + (n2 == 512 ? 0 : 2) + (nz == 13 ? 0 : 1) + (pre ? 4 : 0)
                      : (n2 == 512 ? 0 : 6) + (nz == 13 ? 0 : 3) + (kf == 3 ? 0 : kf == 5 ? 1 : 2) + (pre ? 12 : 0);
}
constexpr int fused_key_n2(int key)
{
    return key >= 48   ? 1024
           : key >= 32 ? ((key - 32) % 8 < 4 ? 512 : 256)
           : key >= 24 ? ((key - 24) % 4 < 2 ? 512 : 256)
                       : key % 12 < 6 ? 512 : 256;
}
constexpr int fused_key_nz(int key)
{
    return key >= 48   ? ((key - 48) % 8 < 4 ? 13 : 16)
           : key >= 32 ? ((key - 32) % 4 < 2 ? 13 : 16)
           : key >= 24 ? ((key - 24) % 2 == 0 ? 13 : 16)
                       : key % 6 < 3 ? 13 : 16;
}
constexpr int fused_key_kf(int key)
{
    return key >= 48   ? ((key - 48) % 4 == 0 ? 3 : (key - 48) % 4 == 1 ? 5 : (key - 48) % 4 == 2 ? 8 : 16)
           : key >= 32 ? ((key - 32) % 2 == 0 ? 5 : 8)
           : key >= 24 ? 16
                       : key % 3 == 0 ? 3 : key % 3 == 1 ? 5 : 8;
}
constexpr bool fused_key_pre(int key)
{
    return key >= 48 ? key >= 56 : key >= 32 ? key >= 40 : key >= 24 ? key >= 28 : key >= 12;
}
constexpr int fused_key_nc(int key) { return key >= 32 && key < 48 ? kMaxCepsWide : 16; }
cudaError_t launch_fused_variant(int key, const FusedLaunch &fl);
// occupancy probe for the cluster path (cudaOccupancyMaxActiveClusters); < 0 on error
int fused_variant_max_clusters(int key, const FusedLaunch &fl);

} // namespace afe
