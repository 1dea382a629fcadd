// Launch interface of the fused kernel's instantiations. k_fused_mfcc<N2, NZ, 8, KF, PRE> is instantiated for 24 parameter
// sets, one per translation unit (afe_fused_inst.cu compiled with -DAFE_INST_KEY=0..23) so that they build in parallel.
#pragma once
#include "afe_fused.cuh"

namespace afe {

struct FusedLaunch {
    FusedArgs a;
    FusedSmem L;
    const MelConst *mc;
    int grid;            // CTAs
    int cluster;         // 0: plain launch; 1..: thread-block cluster size (one cluster = the tiles of one utterance)
    cudaStream_t st;
};

// key = (N2 == 512 ? 0 : 6) + (pruned first layer, NZ = 13 ? 0 : 3) + (KF: 3 -> 0, 5 -> 1, 8 -> 2) + (pre-emphasis ? 12 : 0)
constexpr int kFusedVariants = 24;
cudaError_t launch_fused_variant(int key, const FusedLaunch &fl);
// occupancy probe for the cluster path (cudaOccupancyMaxActiveClusters); < 0 on error
int fused_variant_max_clusters(int key, const FusedLaunch &fl);

} // namespace afe
