// One instantiation of the fused kernel per translation unit: nvcc -DAFE_INST_KEY=<0..63> (see the Makefile).
#include <atomic>

#include "afe_internal.h"
#include "afe_fused_launch.h"

#ifndef AFE_INST_KEY
#error "compile with -DAFE_INST_KEY=0..63"
#endif

namespace afe {

namespace {
constexpr bool kPre = fused_key_pre(AFE_INST_KEY); // per-frame pre-emphasis in the load
constexpr int kN2 = fused_key_n2(AFE_INST_KEY);
constexpr int kNZ = fused_key_nz(AFE_INST_KEY);
constexpr int kKF = fused_key_kf(AFE_INST_KEY);
constexpr int kNC = fused_key_nc(AFE_INST_KEY);
static_assert(fused_key(kN2, kNZ, kKF, kPre, kNC) == AFE_INST_KEY, "key encoding and decoding disagree");
using Mel = MelConstFor<kN2, kKF, kNC>;

void fill(cudaLaunchConfig_t &cfg, cudaLaunchAttribute &attr, const FusedLaunch &fl)
{
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = dim3(fl.grid); cfg.blockDim = dim3(32 * 8); cfg.dynamicSmemBytes = fl.L.total; cfg.stream = fl.st;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = fl.cluster > 0 ? fl.cluster : 1; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = fl.cluster > 0 ? 1 : 0;
}
} // namespace

#define AFE_CAT2(a, b) a##b
#define AFE_CAT(a, b) AFE_CAT2(a, b)

// cudaFuncSetAttribute is a slow, serialising call: once per device and shared-memory size, not per launch
static cudaError_t ensure_smem_attr(int bytes)
{
    static std::atomic<int> done[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) dev = 63;
    if (done[dev].load(std::memory_order_acquire) >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(k_fused_mfcc<kN2, kNZ, 8, kKF, kPre, kNC>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done[dev].store(bytes, std::memory_order_release);
    return e;
}

cudaError_t AFE_CAT(fused_launch_, AFE_INST_KEY)(const FusedLaunch &fl)
{
    auto kern = k_fused_mfcc<kN2, kNZ, 8, kKF, kPre, kNC>;
    cudaError_t e = ensure_smem_attr(fl.L.total);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg; cudaLaunchAttribute attr;
    fill(cfg, attr, fl);
    return cudaLaunchKernelEx(&cfg, kern, fl.a, fl.L, *static_cast<const Mel *>(fl.mc));
}

int AFE_CAT(fused_max_clusters_, AFE_INST_KEY)(const FusedLaunch &fl)
{
    auto kern = k_fused_mfcc<kN2, kNZ, 8, kKF, kPre, kNC>;
    if (ensure_smem_attr(fl.L.total) != cudaSuccess) return -1;
    cudaLaunchConfig_t cfg; cudaLaunchAttribute attr;
    fill(cfg, attr, fl);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return -1; }
    return n;
}

} // namespace afe
