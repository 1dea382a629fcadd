// K1: the fused hot-path kernel.  int16 PCM -> window -> real FFT -> |X|/N2 -> mel+log -> DCT -> delta/delta-delta
// -> feature rows (+ per-tile column statistics, + per-utterance normalisation): one HBM read of PCM and one HBM write
// of features per frame.
//
// Work item = (utterance, tile of `nout` output frames). A CTA (8 warps, 2 CTAs per SM; 1 at 1024 points) computes the cepstra of its tile
// plus a halo of D = l1+l2 frames on each side (clamped at the utterance edges, where the reference replicates the edge
// frame, mfcccpu.cpp:243-254) in rounds of 32 frames:
//   stage 0  each warp stages the PCM of ITS 4 frames with one cp.async.bulk (TMA, SASS UBLKCP) into its own buffer,
//            completion on its own mbarrier; the next round's copy is issued as soon as this round's FFTs are done
//   phase 1  each warp: 4/FPW calls of the in-register FFT + magnitude (afe_fft.cuh, packed FP32) -> mags[32][260] (CTA
//            shared; [32][516] at 1024 points). Frame f lives in row mag_row(f): the two adjacent frames of one call land
//            4 rows = 16 banks apart, and the 8 frames of a quarter warp occupy 8 consecutive rows, so phase 2's "lane =
//            frame" 128-bit reads (row stride 65 or 129 chunks = 1 mod 8) are conflict free
//   phase 2  mel + log + DCT, ONE THREAD PER FRAME, warp w owning the filters b = w (mod 8). The triangular weights and
//            the DCT matrix are kernel parameters, i.e. constant-bank operands (LDCU.64 -> uniform-register operand of
//            FFMA2): they cost no shared-memory bandwidth (v3/v4 re-loaded weights per lane: 116 of 245 smem wavefronts
//            per frame, profiles/r01_v3_k_fused_summary.txt). Accumulation per filter runs in ascending-bin order
//            (mfcccpu.cpp:192-220) in four chains. Per-warp partial cepstra are summed in a fixed order -> cep[tile][cols].
//   phase 3  default regression (l1 = l2 = 3): one register-blocked pass computes delta / delta-delta, writes the rows and
//            keeps column sums / sums of squares (double) / min / max -> per-tile record (dev::phase3_l3). Otherwise:
//            delta rows through shared memory, then coalesced row writes.
//   norm     the last tile of an utterance to finish reduces the records and normalises the utterance in place (L2).
// Two CTA barriers per 32 frames (v1 serialised phase 2 on one warp and lost 39 % of its issue slots at the barrier,
// profiles/r01_v1_k_fused_summary.txt). A warp-specialised persistent variant was measured 1.6 % slower in round 1
// (profiles/r01_ws_vs_generic.txt) and removed.
// Replaces, for whole utterances: segmenter.cl, AppleFFT fft0, mfcc.cl kernelTranspose+kernelFilter, DCT.cl,
// delta.cl and norm.cl:kernelSum (SURVEY §2.1).
#pragma once
#include <cfloat>

#include "afe_fft.cuh"
#include "afe_internal.h"
#include "afe_mel.cuh"

namespace afe {

struct Tile {
    long long pcm_off;   // first sample of the utterance in the packed PCM buffer
    long long out_row0;  // output row of the utterance's frame 0
    int T;               // frames in the utterance
    int t0;              // first output frame of this tile
    int nout;            // output frames of this tile
    int group;           // statistics group (utterance index, or 0 for corpus scope)
    int tile0;           // index of the utterance's first tile
    int ntiles;          // tiles of the utterance
    int flags;           // kTileNoStats | kTileQ1All
    int pad_;
};
constexpr int kTileNoStats = 1; // the tile's rows do not enter the group's statistics (speculative flush rows of a stream block)
constexpr int kTileQ1All = 2;   // every row of the tile takes its static D rows early (FusedArgs::q1 == 2 for this tile only)

constexpr int kMaxBanks = 64;      // bank capacity of the instantiations with KF <= 8 (up to 64 banks)
constexpr int kMaxBanksWide = 128; // bank capacity of the KF = 16 instantiations (65..128 banks)
// floats per magnitude row (16-byte aligned rows, an odd number of 16-byte chunks): 257 bins up to 512 points, 513 at 1024
__host__ __device__ constexpr int mag_stride(int n2) { return n2 == 1024 ? 516 : 260; }
// row of frame f (0..31) of a round: pair k = f>>1 -> rows 8*(k>>2) + (k&3) and +4
__host__ __device__ constexpr int mag_row(int f) { return 8 * (f >> 3) + ((f >> 1) & 3) + 4 * (f & 1); }

// Mel / DCT tables for up to NB banks, NC DCT columns and NBINS magnitude bins, passed BY VALUE as a kernel parameter
// (constant bank): indexed with warp-uniform indices only, read with 128-bit constant loads. Weight lists are zero padded
// to a multiple of 4 bins; DCT rows to NC columns. NB = 64: 7 KB; NB = 128: 16 KB; NB = 64 with NC = 48: 17 KB; 513 bins
// (1024 points): 11 KB with NB = 64, 18 KB with NB = 128 (the parameter list must stay under 32 764 bytes, see below).
template <int NB, int NC = 16, int NBINS = 257>
struct MelConstT {
    static constexpr int kBanks = NB;
    static constexpr int kCols = NC;
    static constexpr int kWl4 = (2 * NBINS + 10 * NB + 3) / 4; // every bin feeds a rising and a falling side; lists start on
                                                              // a multiple of 4 bins and are padded to whole 8-bin chunks
    float4 wl4[kWl4];            // weights of filter b: 2*n8[b] float4 = bins 4*fchunk[b] + 8*i + {0..7}, i < n8[b]. The lists
                                 // of the filters of one warp class (b = w, w + 8, w + 16, ...) are CONTIGUOUS from
                                 // wstart[w], in that order, so phase 2 walks them with one running offset. The weights
                                 // carry the 0.5/N2 magnitude scale (an exact power of two), see fft_frame_mag
    float4 dct4[NB][NC / 4];     // [nb][NC]
    int desc[NB];                // fchunk[b] (first 4-bin chunk = edges[b] / 4; leading weights are zero) | n8[b] << 16
    short wstart[8];             // first float4 of warp class w (8 warps per CTA)
};
constexpr int kMaxCepsWide = 48; // DCT column capacity of the wide-DCT instantiations (ceps_len + c0 = 17..48, <= 64 banks)
using MelConst = MelConstT<kMaxBanks>;
using MelConstWide = MelConstT<kMaxBanksWide>;
using MelConstCeps = MelConstT<kMaxBanks, kMaxCepsWide>;
using MelConst1024 = MelConstT<kMaxBanks, 16, 513>;
using MelConstWide1024 = MelConstT<kMaxBanksWide, 16, 513>;
// the constant-bank tables of k_fused_mfcc<N2, .., KF, .., NC>
template <int N2, int KF, int NC>
using MelConstFor = MelConstT<(KF <= 8 ? kMaxBanks : kMaxBanksWide), NC, (N2 == 1024 ? 513 : 257)>;

struct FusedArgs {
    const int16_t *pcm;
    float *out;
    const Tile *tiles;
    const float2 *window2, *tw_a, *tw_p;
    double *partials;    // [ntiles][width][4] or nullptr (indexed by absolute tile number)
    int *counters;       // [groups] arrival tickets for the fused normalisation (self-resetting), or nullptr
    int cluster_norm;    // 1: the launch is clustered, one cluster = the tiles of ONE utterance; the tiles exchange their
                         // statistics records through distributed shared memory and write normalised rows directly
    int tile_base;       // absolute index of this launch's first tile
    int norm_type, norm_after_dyn;
#ifdef AFE_DEVTOOLS
    int debug_skip;      // timing experiments only (tools build, -DAFE_DEVTOOLS): 1 skip FFT calls, 2 skip mel/DCT, 4 skip phase 3
#endif
    int W, S, nb, dct_len, cols, width, l1, l2, nstreams;
    int q1;              // 1: reproduce the single-block flush quirk Q1 for the last D rows of an utterance; 2: for EVERY row of
                         // the tile (the streaming object's flush block after a single set_input, mfcccpu.cpp:439)
    int use_tma;
    int stats_rows_mode; // 0: no stats, 1: rows < T-D, 2: all rows of the utterance, 3: the output rows of the group's tiles
                         // (a block of the streaming object: stats_count rows, normalizercpu.cpp:22-30)
    int stats_count;     // mode 3: rows of the whole group
    int use_last;        // 1: no statistics; normalise with g_mean / g_scale of the tile's group (use_last_stats, mfcccpu.cpp:389)
    float *g_mean, *g_scale; // [groups][width] finalised mean / scale: exported by whoever finalises a group (when non-null),
                         // read by use_last tiles and by the normaliser roles of the long-utterance scheme
    // long utterances (more than 8 tiles): the launch carries 2 * ntiles_launch CTAs that take their role from a ticket:
    // the first ntiles_launch tickets extract a tile each, the others wait for their tile's group to be finalised
    // (flags[group] == epoch, set by the group's last tile) and normalise that tile's rows in place through L2
    int *work_counter;   // self-resetting ticket counter, or nullptr
    unsigned *flags;     // [groups]
    unsigned epoch;
    int ntiles_launch;
    float pre;           // pre-emphasis coefficient applied per frame before the window (0: none, the reference's behaviour)
    // A block of the streaming object needs no tile table in memory: blk_ntiles > 0 describes its tiles (all of blk_nout
    // output frames, the last one shorter) and, with blk_spec, one more tile holding the D rows a flush() right after this
    // block would return (right edge replicated, no statistics): see dev::load_tile.
    int blk_ntiles, blk_T, blk_t_first, blk_n_out, blk_nout, blk_spec, blk_spec_q1;
    int stats_kind;      // 0: none, 1: sums (CMN), 2: + sums of squares (CVN), 3: + min/max (MINMAX)
    int tc_max;          // capacity (frames) of the cepstra tile
    float rden1, rden2;  // 1 / (2*sum(l^2))
};

constexpr int kRoundFrames = 32; // frames per CTA round; WARPS (4 or 8) warps share them, 32/WARPS frames each
constexpr int kMaxFusedThreads = 256;
// Wide-DCT instantiations: phase 2 leaves the round's log-mel values in a tile [32 frames][8 KF + 4 floats] that follows the
// rest of the dynamic shared memory (FusedSmem::total includes it). A row is an odd number of 16-byte chunks, so the DCT's
// "lane = frame" 128-bit reads are conflict free.
__host__ __device__ constexpr int lm_stride(int kf) { return 8 * kf + 4; }
__host__ __device__ constexpr int lm_tile_bytes(int kf) { return kRoundFrames * lm_stride(kf) * 4; }

struct FusedSmem {
    int off_mbar, off_mags, off_part, off_warp, warp_bytes, w_pcm, w_scratch, pcm_bytes, off_dhat, off_dd, off_red,
        off_cep, total;
};

// CUDA 12.1+ accepts kernel parameter lists of up to 32 764 bytes; the widest ones are (FusedArgs, FusedSmem, MelConstWide),
// (FusedArgs, FusedSmem, MelConstCeps) and (FusedArgs, FusedSmem, MelConstWide1024)
static_assert(sizeof(FusedArgs) + sizeof(FusedSmem) + sizeof(MelConstWide) + 16 <= 32764, "K1 kernel parameters too large");
static_assert(sizeof(FusedArgs) + sizeof(FusedSmem) + sizeof(MelConstCeps) + 16 <= 32764, "K1 kernel parameters too large");
static_assert(sizeof(FusedArgs) + sizeof(FusedSmem) + sizeof(MelConstWide1024) + 16 <= 32764, "K1 kernel parameters too large");

inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// dynamic shared memory of one CTA when 2 CTAs share an SM (sm_100: 228 KB per SM, 1 KB reserved per CTA, and the few
// bytes of k_fused_mfcc's static shared variables)
constexpr int kSmemTwoCtas = 113 * 1024 - 64;
// the most dynamic shared memory one CTA may take: the 227 KB opt-in limit of a block holds dynamic AND static shared
// memory, and k_fused_mfcc's static shared variables take 128 bytes (ptxas -v); 256 bytes are set aside for them
constexpr int kSmemOneCta = 227 * 1024 - 256;

template <int N2>
FusedSmem fused_smem_layout(int kFusedWarps, int S, int cols, int tc_max, int nout_max, int l2, int nstreams)
{
    using C = dev::FftCfg<N2>;
    const int kWarpFrames = kRoundFrames / kFusedWarps;
    FusedSmem L;
    int o = 0;
    L.off_mbar = o; o += align_up(kFusedWarps * 8, 16);           // one mbarrier per warp, never aliased
    L.off_mags = o; o += align_up((kRoundFrames * mag_stride(N2) + 16) * 4, 16); // [32][260 | 516] + pad for whole-chunk reads
    // per-warp staging [pcm]; then the FFT exchange tiles [scratch], which phase 2 reuses for the partial cepstra
    L.pcm_bytes = align_up(((kWarpFrames - 1) * S + N2) * 2, 16) + 16;
    L.w_pcm = 0;
    L.warp_bytes = L.pcm_bytes;
    o = align_up(o, 128);
    L.off_warp = o; o += kFusedWarps * L.warp_bytes;
    o = align_up(o, 128);
    const int scratch = kFusedWarps * align_up(C::FPW * C::SCR * 8, 16);
    const int part = kFusedWarps * 4 * kRoundFrames * 16;          // float4 [warp][c4][frame]
    L.w_scratch = align_up(C::FPW * C::SCR * 8, 16);               // bytes per warp
    L.off_part = o; o += scratch > part ? scratch : part;
    // phase 3 reuses everything between off_mags and off_cep: [delta rows | delta-delta rows | reduction scratch]
    const int dhat = nstreams >= 2 ? align_up((nout_max + 2 * l2) * cols * 4, 16) : 0;
    const int dd = nstreams >= 3 ? align_up(nout_max * cols * 4, 16) : 0;
    L.off_dhat = L.off_mags;
    L.off_dd = L.off_dhat + dhat;
    L.off_red = L.off_dd + dd;
    const int phase3_end = L.off_red + kMaxFusedThreads * 4 * 8;
    if (phase3_end > o) o = align_up(phase3_end, 128);
    L.off_cep = o; o += align_up(tc_max * cols * 4, 16);
    L.total = o;
    return L;
}

namespace dev {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    // bounded: a TMA that never completes must trap (error to the host), never hang the GPU
    for (uint32_t spin = 0; spin < (1u << 24); spin++) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) return;
    }
    __trap();
}
// 1-D bulk async copy global -> shared through the TMA engine, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float4 lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// keeps a value in its register: the compiler cannot rematerialise the expression it came from
__device__ __forceinline__ uint32_t opaque(uint32_t v)
{
    asm volatile("" : "+r"(v));
    return v;
}

// ---- thread-block clusters: barrier over all CTAs of the cluster, read of a peer CTA's shared memory (DSMEM)
__device__ __forceinline__ void cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_size()
{
    uint32_t n;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(n));
    return n;
}
__device__ __forceinline__ double ld_peer_f64(const double *local, uint32_t rank)
{
    uint32_t peer;
    double v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(peer) : "r"(smem_u32(local)), "r"(rank));
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(peer) : "memory");
    return v;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// The tile's record of column c: its rp row-group records rec[g][width][4] (sum, sumsq, min, max) summed in group order,
// stored to dst(). The destination address is formed after the loop: computed by the caller and held across it, it changed
// ptxas' register allocation and schedule of the whole epilogue.
template <class Dst>
__device__ __forceinline__ void sum_row_groups(const double *rec, int rp, int width, int c, Dst dst)
{
    double s0 = 0.0, s1 = 0.0, lo = (double)FLT_MAX, hi = -(double)FLT_MAX;
    for (int g = 0; g < rp; g++) {
        const double *p = rec + (g * width + c) * 4;
        s0 += p[0]; s1 += p[1];
        lo = fmin(lo, p[2]); hi = fmax(hi, p[3]);
    }
    double *d = dst();
    d[0] = s0; d[1] = s1; d[2] = lo; d[3] = hi;
}

} // namespace dev

namespace dev {

// regression numerator sum_l l*(p[+l*stride] - p[-l*stride]); L == 3 (the reference's default l1 = l2 = 3) is unrolled
__device__ __forceinline__ float delta_num(const float *p, int stride, int L)
{
    if (L == 3) {
        float num = p[stride] - p[-stride];
        num = fmaf(2.f, p[2 * stride] - p[-2 * stride], num);
        return fmaf(3.f, p[3 * stride] - p[-3 * stride], num);
    }
    float num = 0.f;
    for (int l = 1; l <= L; l++) num = fmaf((float)l, p[l * stride] - p[-l * stride], num);
    return num;
}

// rows out + column statistics of one thread's column. KIND: 0 none, 1 sums, 2 + sums of squares, 3 + min/max
template <int KIND>
__device__ __forceinline__ void write_rows(float *__restrict__ orow, const float *__restrict__ src, int r_off, int rpp, int nout,
                                           int rq, int rs, int cols, int width, int D, double &sum, double &sumsq, float &mn,
                                           float &mx)
{
    const int ostep = rpp * width, sstep = rpp * cols;
    orow += r_off * width;
    src += r_off * cols;
    for (int r = r_off; r < nout; r += rpp, orow += ostep, src += sstep) {
        const float sval = *src;
        // Q1 shifts only what is WRITTEN for the flushed rows; the reference takes its statistics on the first
        // block's own statics (mfcccpu.cpp:274 / :383-384), i.e. always un-shifted
        *orow = r >= rq ? src[-D * cols] : sval;
        if (KIND >= 1 && r < rs) { // normalizercpu.cpp:31-66: double sums of float values / float products
            sum += (double)sval;
            if (KIND >= 2) sumsq += (double)__fmul_rn(sval, sval);
            if (KIND >= 3) { mn = fminf(mn, sval); mx = fmaxf(mx, sval); }
        }
    }
}

// Phase 3 for the reference's default regression (l1 = l2 = 3, static + delta + delta-delta): ONE pass, one barrier.
// A task = (column c, block of R consecutive output rows). The thread loads the R + 12 cepstra of its column that the
// block depends on (edge frames replicated by clamping, mfcccpu.cpp:243-254), computes the R + 6 extended-axis deltas
// and the R delta-deltas in registers (same operation order as delta_num), writes the three streams of its rows and
// keeps the column statistics. 1.5 shared-memory loads per output value instead of 7, no delta rows in shared memory,
// and the tile's rows leave as 13-float runs that L2 merges into full sectors.
// s_red3: [rp][width][4] doubles, reduced in group order by the caller (deterministic).
// MODE 0: write the raw rows and keep the statistics (the tile's record is reduced by the caller)
// MODE 1: statistics only  \ a tile that holds a WHOLE utterance (k_fused_ws) takes the statistics first and then writes
// MODE 2: write (v - mean) * scale, no statistics  / normalised rows directly: no second trip through L2
// norm3: mean[3] | scale[3] of this thread's three columns (MODE 2 only)
// KIND (statistics: 0 none, 1 sums, 2 + sums of squares, 3 + min/max) is a run-time, warp-uniform argument: one copy of
// the unrolled block code per MODE keeps the kernel's epilogue small (8 template copies were 6 400 instructions).
template <int MODE>
__device__ __forceinline__ void phase3_l3(const int KIND, const FusedArgs &a, const Tile &tl, const float *__restrict__ s_cep,
                                          int c0f, int c1f, double *__restrict__ s_red3, int tid, int nthreads, int rs,
                                          const float *norm3 = nullptr)
{
    constexpr int R = 8;
    const int cols = a.cols, width = a.width, T = tl.T, t0 = tl.t0, nout = tl.nout;
    const int rp = nthreads / cols, g = tid / cols, c = tid - g * cols;
    if (g >= rp) return;
    const int q1 = (tl.flags & kTileQ1All) ? 2 : a.q1;
    const int rq = q1 ? (q1 == 2 ? 0 : max(0, T - 6 - t0)) : nout; // first row written with the static of 6 rows earlier (Q1)
    const float rden1 = a.rden1, rden2 = a.rden2;
    double sum[3] = {0.0, 0.0, 0.0}, sumsq[3] = {0.0, 0.0, 0.0};
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    float nm[3] = {0.f, 0.f, 0.f}, ns[3] = {1.f, 1.f, 1.f};
    if (MODE == 2) {
#pragma unroll
        for (int k = 0; k < 3; k++) { nm[k] = norm3[k]; ns[k] = norm3[3 + k]; }
    }
    const bool cmn = a.norm_type == AFE_NORM_CMN;
    float *obase = a.out + (tl.out_row0 + t0) * (long long)width + c;
    for (int r0 = g * R; r0 < (MODE == 1 ? rs : nout); r0 += rp * R) {
        float x[R + 12], dh[R + 6];
#pragma unroll
        for (int i = 0; i < R + 12; i++) // cepstra of frames t0 + r0 - 6 + i; rows past the tile only feed unused results
            x[i] = s_cep[(clampi(t0 + r0 - 6 + i, c0f, c1f - 1) - c0f) * cols + c];
#pragma unroll
        for (int j = 0; j < R + 6; j++) { // extended-axis delta at frame t0 + r0 - 3 + j (deltacpu.cpp:25)
            float num = x[j + 4] - x[j + 2];
            num = fmaf(2.f, x[j + 5] - x[j + 1], num);
            num = fmaf(3.f, x[j + 6] - x[j], num);
            dh[j] = __fmul_rn(num, rden1); // rounded like the stored delta row of the reference: never contracted into the
                                           // differences below
        }
        float *orow = obase + (long long)r0 * width;
#pragma unroll
        for (int r = 0; r < R; r++, orow += width) {
            const int row = r0 + r;
            if (row >= nout) break;
            float num = dh[r + 4] - dh[r + 2];
            num = fmaf(2.f, dh[r + 5] - dh[r + 1], num);
            num = fmaf(3.f, dh[r + 6] - dh[r], num);
            const float v[3] = {x[r + 6], dh[r + 3], __fmul_rn(num, rden2)};
            if (MODE == 0) {
                orow[0] = row >= rq ? x[r] : v[0];
                orow[cols] = v[1];
                orow[2 * cols] = v[2];
            } else if (MODE == 2) { // same operations as the in-place normaliser: v - m, or (v - m) * scale
                const float w0 = row >= rq ? x[r] : v[0];
                orow[0] = cmn ? w0 - nm[0] : (w0 - nm[0]) * ns[0];
                orow[cols] = cmn ? v[1] - nm[1] : (v[1] - nm[1]) * ns[1];
                orow[2 * cols] = cmn ? v[2] - nm[2] : (v[2] - nm[2]) * ns[2];
            }
            if (MODE != 2 && KIND >= 1 && row < rs) { // normalizercpu.cpp:31-66: double sums of float values / float products
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    sum[k] += (double)v[k];
                    if (KIND >= 2) sumsq[k] += (double)__fmul_rn(v[k], v[k]);
                    if (KIND >= 3) { mn[k] = fminf(mn[k], v[k]); mx[k] = fmaxf(mx[k], v[k]); }
                }
            }
        }
    }
    if (MODE != 2) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            double *p = s_red3 + ((g * width) + k * cols + c) * 4;
            p[0] = sum[k]; p[1] = sumsq[k]; p[2] = (double)mn[k]; p[3] = (double)mx[k];
        }
    }
}

} // namespace dev

namespace dev {
__device__ __forceinline__ Tile load_tile(const FusedArgs &a, int idx)
{
    if (a.blk_ntiles == 0) return a.tiles[idx];
    const int D = a.l1 + a.l2;
    Tile tl;
    tl.pcm_off = 0; tl.out_row0 = -(long long)a.blk_t_first; tl.T = a.blk_T; tl.group = 0; tl.tile0 = 0;
    tl.ntiles = a.blk_ntiles + a.blk_spec; tl.pad_ = 0;
    if (idx < a.blk_ntiles) {
        tl.t0 = a.blk_t_first + idx * a.blk_nout;
        tl.nout = min(a.blk_nout, a.blk_t_first + a.blk_n_out - tl.t0);
        tl.flags = 0;
    } else { // rows [T - D, T): what flush() would return if the stream ended with this block (mfcccpu.cpp:373-390)
        tl.t0 = a.blk_T - D; tl.nout = D;
        tl.flags = kTileNoStats | (a.blk_spec_q1 ? kTileQ1All : 0);
    }
    return tl;
}

// Canonical order in which the per-tile statistics records of one group are summed (every scheme - cluster, ticket, role
// scheme, K2 - must produce the same bits): up to kSeqTiles tiles strictly in tile order; more tiles in kSegs segments of
// consecutive tiles, each summed in tile order, the segment sums then added in segment order.
constexpr int kSeqTiles = 32, kSegs = 6;
__host__ __device__ inline int seg_len(int ntiles) { return ntiles <= kSeqTiles ? ntiles : (ntiles + kSegs - 1) / kSegs; }

static __device__ unsigned g_opaque_zero = 0; // never written

// sum of the records [t_begin, t_end) of column c, tile order; partials: [tile][width][4] = sum, sumsq, min, max.
// Eight records (sixteen 16-byte loads) are in flight before the first add: the records come from L2, and a loop that
// loads and adds one record at a time costs a full L2 round trip per tile (163 us for 1169 tiles, profiles/r02_c5_launches.csv).
// PLAIN (weak) loads on purpose: ptxas keeps `ld.global.cg` / __ldcg loads next to their consumers (measured: two loads in
// flight), while it batches ordinary loads. They are correct here: every caller reads the records after the synchronising
// pattern "ticket atomic -> __syncthreads -> __threadfence" (or in a later kernel), which orders them after the writers'
// "stores -> __threadfence -> ticket atomic" and drops stale L1 lines.
__device__ __forceinline__ void sum_records(const double *__restrict__ partials, int width, int c, int t_begin, int t_end,
                                            double &s0, double &s1, double &lo, double &hi, int tstep = 1)
{
    s0 = 0.0; s1 = 0.0; lo = (double)FLT_MAX; hi = -(double)FLT_MAX;
    constexpr int U = 8;
    const size_t stride = (size_t)width * 4 * tstep;   // records t_begin, t_begin + tstep, ... below t_end
    const double *p = partials + ((size_t)t_begin * width + c) * 4;
    const int last = t_end - 1;
    const unsigned z = *reinterpret_cast<volatile unsigned *>(&g_opaque_zero); // a zero neither NVVM nor ptxas can see through
    for (int t = t_begin; t < t_end; t += U * tstep, p += U * stride) {
        double2 a[U], b[U];
        // unconditional loads (a record past the end re-reads the last valid one and is discarded below): predicated loads
        // share the predicate registers with the min / max compares and ptxas then serialises them (two L2 round trips per
        // four records in the first version of this loop)
#pragma unroll
        for (int k = 0; k < U; k++) {
            const double2 *q = reinterpret_cast<const double2 *>(t + k * tstep <= last ? p + k * stride : p);
            a[k] = q[0];
            b[k] = q[1];
        }
        // All sixteen loads must be ISSUED before the first add. ptxas schedules each load right in front of its consumer
        // (load, add, load, add: an L2 round trip per record) and looks through empty asm barriers, so the first summand is
        // made to depend on every loaded word through an OR with `z`, a zero the compiler cannot see (bits unchanged).
        unsigned all = 0;
#pragma unroll
        for (int k = 0; k < U; k++)
            all |= (unsigned)__double2hiint(a[k].x) | (unsigned)__double2hiint(a[k].y) | (unsigned)__double2hiint(b[k].x) |
                   (unsigned)__double2hiint(b[k].y);
        a[0].x = __hiloint2double(__double2hiint(a[0].x) | (int)(all & z), __double2loint(a[0].x));
#pragma unroll
        for (int k = 0; k < U; k++) {
            const bool ok = t + k * tstep <= last; // tile order; adding 0.0 / comparing with the identity changes no bits
            s0 += ok ? a[k].x : 0.0; s1 += ok ? a[k].y : 0.0;
            lo = fmin(lo, ok ? b[k].x : (double)FLT_MAX); hi = fmax(hi, ok ? b[k].y : -(double)FLT_MAX);
        }
    }
}

// Group total of column c in the canonical order. Called by threads tid < kSegs * width of ONE CTA (thread = (segment,
// column)); s_seg: kSegs * width * 4 doubles of shared memory. Contains __syncthreads: every thread of the CTA must call it.
// The result is valid in threads tid < width.
__device__ __forceinline__ void group_total(const double *__restrict__ partials, int width, int tile0, int ntiles, int tid,
                                            int nthreads, double *s_seg, int c_of_tid, double &s0, double &s1, double &lo, double &hi)
{
    if (ntiles <= kSeqTiles) { // short groups: plain tile order, no exchange (c_of_tid: the column this thread finalises)
        if (tid < width) sum_records(partials, width, c_of_tid, tile0, tile0 + ntiles, s0, s1, lo, hi);
        return;
    }
    const int len = seg_len(ntiles);
    for (int i = tid; i < kSegs * width; i += nthreads) {
        const int seg = i / width, c = i - seg * width;
        const int b = min(ntiles, seg * len), e = min(ntiles, b + len);
        double a0, a1, l, h;
        sum_records(partials, width, c, tile0 + b, tile0 + e, a0, a1, l, h);
        double *o = s_seg + (size_t)i * 4;
        o[0] = a0; o[1] = a1; o[2] = l; o[3] = h;
    }
    __syncthreads();
    if (tid < width) {
        s0 = 0.0; s1 = 0.0; lo = (double)FLT_MAX; hi = -(double)FLT_MAX;
        for (int seg = 0; seg < kSegs; seg++) {
            const double *o = s_seg + ((size_t)seg * width + c_of_tid) * 4;
            s0 += o[0]; s1 += o[1];
            lo = fmin(lo, o[2]); hi = fmax(hi, o[3]);
        }
    }
}

// In-place (x - mean) [* scale] over one tile's rows, 128-bit accesses on the 16-byte aligned body of the tile's contiguous
// region; columns tracked incrementally (no division in the loop). Used by K3 (k_normalize_tiles) and by the normaliser
// roles of the long-utterance scheme, so both give the same bits. s_ms: 2 * width floats of shared memory.
__device__ __forceinline__ void normalise_tile_rows(float *__restrict__ out, const Tile &tl, int width, int norm_type,
                                                    const float *__restrict__ mean, const float *__restrict__ scale, float *s_ms)
{
    float *base = out + (tl.out_row0 + tl.t0) * (long long)width;
    const int n = tl.nout * width;
    for (int i = threadIdx.x; i < width; i += blockDim.x) {
        s_ms[i] = __ldcg(mean + (long long)tl.group * width + i);
        s_ms[width + i] = norm_type == AFE_NORM_CMN ? 1.f : __ldcg(scale + (long long)tl.group * width + i);
    }
    __syncthreads();
    const float *m = s_ms, *sc = s_ms + width;
    const bool cmn = norm_type == AFE_NORM_CMN;
    const int head = min(n, (int)(((16 - (reinterpret_cast<uintptr_t>(base) & 15)) & 15) >> 2));
    const int n4 = (n - head) >> 2, tail0 = head + 4 * n4;
    if ((int)threadIdx.x < head) {
        const int i = threadIdx.x;
        const float v = __ldcg(base + i) - m[i % width];
        base[i] = cmn ? v : v * sc[i % width];
    }
    if ((int)threadIdx.x < n - tail0) {
        const int i = tail0 + threadIdx.x, c = i % width;
        const float v = __ldcg(base + i) - m[c];
        base[i] = cmn ? v : v * sc[c];
    }
    float4 *p4 = reinterpret_cast<float4 *>(base + head);
    int c = (head + 4 * (int)threadIdx.x) % width;
    const int cstep = (4 * (int)blockDim.x) % width;
    constexpr int U = 4; // loads in flight per thread: the rows come from L2 (~300 cycles away)
    const int bd = blockDim.x;
    for (int j = threadIdx.x; j < n4; j += U * bd) {
        float4 v[U];
#pragma unroll
        for (int k = 0; k < U; k++)
            if (j + k * bd < n4) v[k] = __ldcg(p4 + j + k * bd);
#pragma unroll
        for (int k = 0; k < U; k++) {
            if (j + k * bd < n4) {
                int c1 = c + 1; if (c1 >= width) c1 -= width;
                int c2 = c1 + 1; if (c2 >= width) c2 -= width;
                int c3 = c2 + 1; if (c3 >= width) c3 -= width;
                float4 w = v[k];
                w.x -= m[c]; w.y -= m[c1]; w.z -= m[c2]; w.w -= m[c3];
                if (!cmn) { w.x *= sc[c]; w.y *= sc[c1]; w.z *= sc[c2]; w.w *= sc[c3]; }
                p4[j + k * bd] = w;
            }
            c += cstep; if (c >= width) c -= width;
        }
    }
}

// Normaliser role of the long-utterance scheme: wait (bounded) until the tile's group is finalised, then normalise the tile.
__device__ __forceinline__ void normalise_role(const FusedArgs &a, const Tile tl, float *s_ms)
{
    if (threadIdx.x == 0) {
        // The flag is set by the group's last extracting CTA, which holds an earlier ticket and is therefore running or
        // done: the wait always ends. Bounded all the same (a lost flag must trap, never hang the GPU).
        unsigned v = 0;
        for (unsigned spin = 0; spin < (1u << 26); spin++) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(a.flags + tl.group) : "memory");
            if (v == a.epoch) break;
            __nanosleep(128);
        }
        if (v != a.epoch) __trap();
    }
    __syncthreads();
    normalise_tile_rows(a.out, tl, a.width, a.norm_type, a.g_mean, a.g_scale, s_ms);
}
} // namespace dev

// KF = filters per warp in phase 2 (ceil(num_banks / WARPS), rounded up to 3, 5, 8 or 16): up to 8 the phase is unrolled
// KF times, so a tight bound keeps the round loop inside the instruction cache. KF = 16 (65..128 banks) runs the warp's
// filters in passes of 4: 16 unrolled filters do not fit the register budget of 2 CTAs per SM.
// NC = DCT column capacity. NC = 16: every warp keeps the partial cepstra of its filter class, warps 0-3 sum them.
// NC = 48 (ceps_len + c0 = 17..48, KF = 5 or 8): phase 2 writes log-mel values to a tile and, after barrier B, warps 0-3
// compute the DCT split by column (12 each, lane = frame), in ascending bank order, straight into s_cep.
// N2 = 1024: the 66 KB magnitude tile leaves room for one CTA per SM (DESIGN §4), which may use up to 255 registers.
template <int N2, int NZ, int kFusedWarps, int KF, bool PRE, int NC = 16>
__global__ void __launch_bounds__(32 * kFusedWarps, N2 == 1024 ? 1 : 2)
k_fused_mfcc(const FusedArgs a, const FusedSmem L, const __grid_constant__ MelConstFor<N2, KF, NC> mc)
{
    constexpr bool FAST = false; // MUFU log approximation: measured in round 1, not shipped
    constexpr bool kWideDct = NC > 16;
    static_assert(!kWideDct || KF <= 8, "the wide DCT serves up to 64 banks");
    static_assert(!kWideDct || N2 <= 512, "the wide DCT serves up to 512 points");
    constexpr int kMagStride = mag_stride(N2);
    // warps of the wide DCT and columns per warp: with 4, warps 4-7 run ahead into the next round's FFTs (DESIGN §4)
    constexpr int kDctWarps = 4, kDctCols = NC / kDctWarps;
    using C = dev::FftCfg<N2>;
    constexpr int kFusedThreads = 32 * kFusedWarps, kWarpFrames = kRoundFrames / kFusedWarps;
    constexpr int R = C::R, FPW = C::FPW, SCR = C::SCR;
    static_assert(kWarpFrames % FPW == 0, "a warp's frames must fill whole FFT calls");
    extern __shared__ __align__(128) unsigned char smem[];
    float *s_mags = reinterpret_cast<float *>(smem + L.off_mags);
    float *s_cep = reinterpret_cast<float *>(smem + L.off_cep);

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0); // warp-uniform for the compiler: constant-bank indexing
    const int lf = lane % R, fw = lane / R;
    unsigned char *wbase = smem + L.off_warp + warp * L.warp_bytes;
    uint64_t *w_mbar = reinterpret_cast<uint64_t *>(smem + L.off_mbar) + warp;
    unsigned char *w_pcm = wbase + L.w_pcm;
    float2 *w_scratch = reinterpret_cast<float2 *>(smem + L.off_part + warp * L.w_scratch); // aliased by s_part in phase 2

    int tile_local = blockIdx.x;
    if (a.work_counter) { // long-utterance scheme: roles by ticket, so that a waiting CTA can only wait for RUNNING ones
        __shared__ int s_role;
        if (tid == 0) {
            const int t = atomicAdd(a.work_counter, 1);
            if (t == (int)gridDim.x - 1) *a.work_counter = 0; // every ticket of this launch is out: ready for the next
            s_role = t;
        }
        __syncthreads();
        tile_local = s_role;
        if (tile_local >= a.ntiles_launch) {
            // normaliser role j of n_norm = gridDim.x - ntiles_launch: tiles j, j + n_norm, ...
            const int n_norm = (int)gridDim.x - a.ntiles_launch;
            for (int j = tile_local - a.ntiles_launch; j < a.ntiles_launch; j += n_norm) {
                dev::normalise_role(a, dev::load_tile(a, a.tile_base + j), reinterpret_cast<float *>(smem));
                __syncthreads();
            }
            return;
        }
    }
    const int tile_idx = a.tile_base + tile_local;
    const Tile tl = dev::load_tile(a, tile_idx);
    const int q1 = (tl.flags & kTileQ1All) ? 2 : a.q1;
    const int D = a.l1 + a.l2, cols = a.cols;
    const int c0f = max(0, tl.t0 - D), c1f = min(tl.T, tl.t0 + tl.nout + D);
    const int ncomp = c1f - c0f;
    const int nrounds = (ncomp + kRoundFrames - 1) / kRoundFrames;
    // this warp's frames of round r: [r*32 + warp*8, +8)
    const int16_t *wpcm = a.pcm + tl.pcm_off + (long long)(c0f + warp * kWarpFrames) * a.S;
    auto warp_frames = [&](int r) { return min(kWarpFrames, ncomp - r * kRoundFrames - warp * kWarpFrames); };
    auto issue_tma = [&](int r) { // lane 0 only; nothing to copy when the warp has no frame in round r
        const int nf = warp_frames(r);
        if (nf <= 0) return;
        const uint32_t bytes = (uint32_t)((((nf - 1) * a.S + a.W) * 2 + 15) & ~15);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        dev::mbar_expect_tx(w_mbar, bytes);
        dev::tma_bulk_g2s(w_pcm, wpcm + (long long)r * kRoundFrames * a.S, bytes, w_mbar);
    };
    if (a.use_tma && lane == 0) {
        dev::mbar_init(w_mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue_tma(0); // overlaps the constant loads below
    }
    dev::LaneConsts<N2, NZ> lc;
    dev::load_lane_consts<N2, NZ>(lc, a.window2, a.tw_a, a.tw_p, lf);
    // phase 2 reads whole 8-bin chunks: up to 11 floats past a filter's end, i.e. into the next row (or the pad) with a
    // ZERO weight. Rows of frames that are never computed (short tiles) must therefore hold finite numbers.
    for (int i = tid; i < (kRoundFrames * kMagStride + 16) / 4; i += kFusedThreads)
        reinterpret_cast<float4 *>(s_mags)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();

    // shared-memory address of this lane's magnitude row in phase 2 (lane = frame of the round), pinned in a register
    const uint32_t mrow_s = dev::opaque(dev::smem_u32(s_mags) + mag_row(lane) * kMagStride * 4);
    uint32_t parity = 0;
    // Log-mel rows of 65..128 columns (KF = 16 and no DCT; their width <= 128 leaves no room for deltas, so D = 0): the
    // cepstra buffer holds ONE round and each round's rows are written, and their statistics kept, right after phase 2.
    // A whole-tile buffer would allow 64-frame tiles only (2 CTAs per SM); this keeps tiles of up to 512 frames.
    // The wide DCT without deltas (D = 0) does the same; its cepstra are complete only after the DCT that follows barrier B,
    // so a round's rows leave after the next round's barrier A (the last round's after the loop).
    const bool round_rows = (KF > 8 && a.dct_len == 0) || (kWideDct && D == 0);
    int wr_next = tid / a.width; // next row of this thread: rows tid / width + k * (256 / width), ascending (write_rows)
    double wr_sum = 0.0, wr_sumsq = 0.0;
    float wr_mn = FLT_MAX, wr_mx = -FLT_MAX;
    // wide DCT: rows [f0, f0 + nfr) of the tile, held in s_cep[0 .. nfr) (c0f = t0: no halo)
    auto write_round_rows = [&](int f0, int nfr) {
        if (tid >= kFusedThreads / a.width * a.width) return;
        const int wr_rpp = kFusedThreads / a.width, wr_col = tid - tid / a.width * a.width;
        const int wr_rs = (tl.flags & kTileNoStats) ? 0
                          : a.stats_rows_mode == 3 ? tl.nout
                          : a.stats_rows_mode == 0 ? 0
                                                    : min(tl.nout, max(0, (a.stats_rows_mode == 1 ? tl.T - D : tl.T) - tl.t0));
        float *orow = a.out + (tl.out_row0 + tl.t0 + f0) * (long long)a.width + wr_col;
        const float *src = s_cep + wr_col;
        const int r0 = wr_next - f0, rs = wr_rs - f0;
        switch (a.stats_kind) {
        case 0: dev::write_rows<0>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
        case 1: dev::write_rows<1>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
        case 2: dev::write_rows<2>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
        default: dev::write_rows<3>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
        }
        while (wr_next < f0 + nfr) wr_next += wr_rpp;
    };
    for (int r = 0; r < nrounds; r++) {
        const int f0 = r * kRoundFrames;            // first frame of the round (tile-local)
        const int nfr = min(kRoundFrames, ncomp - f0); // live frames of the round
        const int nfw = warp_frames(r);              // live frames of this warp
        // ---- stage 0 + phase 1 (skipped by warps without a live frame in a short last round)
        if (nfw > 0) {
            if (a.use_tma) {
                dev::mbar_wait(w_mbar, parity);
                parity ^= 1;
            } else {
                // plain staging (any alignment): the warp's samples, 32-bit words when the source allows
                const int16_t *src = wpcm + (long long)f0 * a.S;
                const int n = (nfw - 1) * a.S + a.W;
                int16_t *dst = reinterpret_cast<int16_t *>(w_pcm);
                if ((reinterpret_cast<uintptr_t>(src) & 3) == 0) {
                    const uint32_t *s32 = reinterpret_cast<const uint32_t *>(src);
                    uint32_t *d32 = reinterpret_cast<uint32_t *>(dst);
                    for (int i = lane; i < n / 2; i += 32) d32[i] = __ldg(s32 + i);
                    if ((n & 1) && lane == 0) dst[n - 1] = src[n - 1];
                } else
                    for (int i = lane; i < n; i += 32) dst[i] = src[i];
                __syncwarp();
            }
#pragma unroll
            for (int it = 0; it < kWarpFrames / FPW; it++) {
                if (it * FPW >= nfw) break;
#ifdef AFE_DEVTOOLS
                if (a.debug_skip & 1) break;
#endif
                const int fl = it * FPW + fw;                    // frame within the warp's 8 (adjacent frames per call)
                const int fr = warp * kWarpFrames + fl;          // frame within the round
                const uint32_t *words = reinterpret_cast<const uint32_t *>(w_pcm) + ((fl * a.S) >> 1);
                dev::fft_frame_mag<N2, NZ, true, false, PRE>(words, lc, w_scratch + fw * SCR, s_mags + mag_row(fr) * kMagStride, lf, a.pre);
            }
            // the staging buffer is free again: prefetch this warp's next round while phase 2 runs
            if (a.use_tma && lane == 0 && r + 1 < nrounds) issue_tma(r + 1);
        }
        __syncthreads(); // A: all magnitudes of the round are in shared memory
        if (kWideDct && round_rows && r > 0) write_round_rows(f0 - kRoundFrames, kRoundFrames);

        // ---- phase 2: lane = frame of the round, warp = filter class (filters warp, warp + WARPS, ...).
        //      Three unrolled passes over the warp's <= KF filters - sums, logs, DCT - so that the independent filters'
        //      long dependency chains (accumulation, logf) interleave instead of running back to back.
#ifdef AFE_DEVTOOLS
        if (lane < nfr && !(a.debug_skip & 2)) {
#else
        if (lane < nfr) {
#endif
            constexpr int KP = KF <= 8 && !(kWideDct && KF == 8) ? KF : 4; // filters per pass
            int woff = mc.wstart[warp]; // running float4 offset into this warp class's weight lists (uniform)
            float2 cep[8];              // DCT accumulators, carried across passes
#pragma unroll
            for (int c = 0; c < 8; c++) cep[c] = make_float2(0.f, 0.f);
            const int npass = KP == KF ? 1 : ((a.nb - warp + kFusedWarps - 1) / kFusedWarps + KP - 1) / KP;
#pragma unroll 1
            for (int kb = 0; kb < npass * KP; kb += KP) { // filter slots kb .. kb + KP - 1 (b < 8 * KF always)
                float es[KP];
                // the first 8-bin chunk of every filter of this pass is loaded up front (2*KP independent 128-bit loads in
                // flight): 40 of the 89 chunks of the 40-filter bank, so most filters never wait for shared memory
                int dsc[KP];
                float4 mf0[KP], mf1[KP];
#pragma unroll
                for (int k = 0; k < KP; k++) {
                    const int b = warp + (kb + k) * kFusedWarps;
                    dsc[k] = b < a.nb ? mc.desc[b] : 0;
                    const uint32_t maddr = mrow_s + ((dsc[k] & 0xffff) << 4);
                    mf0[k] = dev::lds128(maddr);
                    mf1[k] = dev::lds128(maddr + 16);
                }
#pragma unroll
                for (int k = 0; k < KP; k++) {
                    // four chains (bins 0,1 | 2,3 of every 4-bin group) in two register pairs: FFMA2, ascending bins in each
                    float2 acc0 = make_float2(0.f, 0.f), acc1 = acc0;
                    int n8 = dsc[k] >> 16;       // 0 for a slot past num_banks (warp uniform), else >= 1
                    if (n8 > 0) {
                        uint32_t maddr = mrow_s + ((dsc[k] & 0xffff) << 4);
                        float4 m0 = mf0[k], m1 = mf1[k];
                        for (;;) {
                            const float4 w0 = mc.wl4[woff], w1 = mc.wl4[woff + 1];
                            acc0 = __ffma2_rn(make_float2(m0.x, m0.y), make_float2(w0.x, w0.y), acc0);
                            acc1 = __ffma2_rn(make_float2(m0.z, m0.w), make_float2(w0.z, w0.w), acc1);
                            acc0 = __ffma2_rn(make_float2(m1.x, m1.y), make_float2(w1.x, w1.y), acc0);
                            acc1 = __ffma2_rn(make_float2(m1.z, m1.w), make_float2(w1.z, w1.w), acc1);
                            woff += 2;
                            if (--n8 == 0) break;
                            maddr += 32;
                            m0 = dev::lds128(maddr);
                            m1 = dev::lds128(maddr + 16);
                        }
                    }
                    const float2 t = __fadd2_rn(acc0, acc1);
                    es[k] = t.x + t.y;
                }
                // logs two at a time (packed); a filter slot past num_banks holds 0 -> log(1e-30), never used
#pragma unroll
                for (int k = 0; k + 1 < KP; k += 2) {
                    const float2 e2 = dev::mel_log2<FAST>(make_float2(es[k], es[k + 1]));
                    es[k] = e2.x; es[k + 1] = e2.y;
                }
                if (KP & 1) es[KP - 1] = dev::mel_log<FAST>(es[KP - 1]);
                if (kWideDct) {
                    // every slot, also those past num_banks (the finite log(1e-30), against zero DCT rows): the DCT reads
                    // whole 4-bank chunks
                    float *lrow = reinterpret_cast<float *>(smem + L.total - lm_tile_bytes(KF)) + lane * lm_stride(KF) + warp;
#pragma unroll
                    for (int k = 0; k < KP; k++) lrow[(kb + k) * kFusedWarps] = es[k];
                } else if (a.dct_len > 0) {
                    // no branch on b < num_banks: the DCT rows of the slots past it are zero (MelConst is zero filled) and their
                    // es is the finite log(1e-30), so the straight-line code lets the constant loads run ahead of the FMAs
                    // (6.23 -> 6.15 ms)
#pragma unroll
                    for (int k = 0; k < KP; k++) {
                        const int b = warp + (kb + k) * kFusedWarps;
                        const float2 e2 = make_float2(es[k], es[k]);
#pragma unroll
                        for (int c4 = 0; c4 < 4; c4++) {
                            const float4 d4 = mc.dct4[b][c4];
                            cep[2 * c4 + 0] = __ffma2_rn(e2, make_float2(d4.x, d4.y), cep[2 * c4 + 0]);
                            cep[2 * c4 + 1] = __ffma2_rn(e2, make_float2(d4.z, d4.w), cep[2 * c4 + 1]);
                        }
                    }
                    // partial cepstra of this filter class -> the exchange tile of the warp that will sum column group c4
                    if (kb + KP == npass * KP) {
#pragma unroll
                        for (int c4 = 0; c4 < 4; c4++)
                            reinterpret_cast<float4 *>(smem + L.off_part + c4 * L.w_scratch)[warp * kRoundFrames + lane] =
                                make_float4(cep[2 * c4].x, cep[2 * c4].y, cep[2 * c4 + 1].x, cep[2 * c4 + 1].y);
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < KP; k++)
                        if (warp + (kb + k) * kFusedWarps < a.nb) s_cep[((round_rows ? 0 : f0) + lane) * cols + warp + (kb + k) * kFusedWarps] = es[k];
                }
            }
        }
        __syncthreads(); // B: partial cepstra are complete; the magnitudes may be overwritten
        // (the same code as write_round_rows, written out: called through the lambda, it compiled to a different schedule
        // for the KF = 16 instantiations)
        if (!kWideDct && round_rows && tid < kFusedThreads / a.width * a.width) {
            // this round's rows [f0, f0 + nfr) (c0f = t0: no halo); the next round's phase 2 overwrites s_cep only after
            // barrier A, which every thread reaches after its writes. Values recomputed per round: fewer live registers.
            const int wr_rpp = kFusedThreads / a.width, wr_col = tid - tid / a.width * a.width;
            const int wr_rs = (tl.flags & kTileNoStats) ? 0
                              : a.stats_rows_mode == 3 ? tl.nout
                              : a.stats_rows_mode == 0 ? 0
                                                        : min(tl.nout, max(0, (a.stats_rows_mode == 1 ? tl.T - D : tl.T) - tl.t0));
            float *orow = a.out + (tl.out_row0 + tl.t0 + f0) * (long long)a.width + wr_col;
            const float *src = s_cep + wr_col;
            const int r0 = wr_next - f0, rs = wr_rs - f0;
            switch (a.stats_kind) {
            case 0: dev::write_rows<0>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
            case 1: dev::write_rows<1>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
            case 2: dev::write_rows<2>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
            default: dev::write_rows<3>(orow, src, r0, wr_rpp, nfr, nfr, rs, cols, a.width, 0, wr_sum, wr_sumsq, wr_mn, wr_mx); break;
            }
            while (wr_next < f0 + nfr) wr_next += wr_rpp;
        }
        if (kWideDct) {
            // warp w (< kDctWarps) computes columns kDctCols*w .. +kDctCols of every frame from the log-mel tile, one FFMA2
            // chain per column pair in ascending bank order. The log-mel tile is rewritten only after the next barrier A,
            // and s_cep is read (next round's rows, phase 3) only after a barrier: none is needed here.
            if (warp < kDctWarps && kDctCols * warp < a.dct_len && lane < nfr) {
                const float4 *lrow = reinterpret_cast<const float4 *>(smem + L.total - lm_tile_bytes(KF)) + lane * (lm_stride(KF) / 4);
                float2 acc[kDctCols / 2];
#pragma unroll
                for (int j = 0; j < kDctCols / 2; j++) acc[j] = make_float2(0.f, 0.f);
                const int nb4 = (a.nb + 3) >> 2;
#pragma unroll 2
                for (int b4 = 0; b4 < nb4; b4++) {
                    const float4 e = lrow[b4];
                    const float ev[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const float2 e2 = make_float2(ev[i], ev[i]);
                        const float2 *drow = reinterpret_cast<const float2 *>(mc.dct4[4 * b4 + i]) + warp * (kDctCols / 2);
#pragma unroll
                        for (int j = 0; j < kDctCols / 2; j++) acc[j] = __ffma2_rn(e2, drow[j], acc[j]);
                    }
                }
                float *crow = s_cep + ((round_rows ? 0 : f0) + lane) * cols + kDctCols * warp;
#pragma unroll
                for (int j = 0; j < kDctCols / 2; j++) {
                    if (kDctCols * warp + 2 * j < a.dct_len) crow[2 * j] = acc[j].x;
                    if (kDctCols * warp + 2 * j + 1 < a.dct_len) crow[2 * j + 1] = acc[j].y;
                }
            }
        } else if (a.dct_len > 0 && warp < 4) {
            // warp w (< 4) sums columns 4w..4w+3 of every frame over the filter classes, in a fixed order. The partials
            // sit in ITS OWN exchange tile, so no CTA barrier is needed before the next round's FFTs reuse that memory.
            // (Spreading this sum over all 8 warps was measured 6 % SLOWER, tools/gpu_ab.sh: warps 4-7 running ahead
            // into the next round's FFTs is what keeps FMA-bound FFT work and LSU-bound mel work mixed on the SM.)
            if (lane < nfr) {
                const float4 *part = reinterpret_cast<const float4 *>(w_scratch);
                float4 t = part[lane];
#pragma unroll
                for (int w2 = 1; w2 < kFusedWarps; w2++) {
                    const float4 u = part[w2 * kRoundFrames + lane];
                    t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
                }
                float *crow = s_cep + (f0 + lane) * cols + 4 * warp;
                if (4 * warp + 0 < a.dct_len) crow[0] = t.x;
                if (4 * warp + 1 < a.dct_len) crow[1] = t.y;
                if (4 * warp + 2 < a.dct_len) crow[2] = t.z;
                if (4 * warp + 3 < a.dct_len) crow[3] = t.w;
            }
            __syncwarp();
        }
    }
    __syncthreads(); // all cepstra of the tile are in shared memory
    if (kWideDct && round_rows) write_round_rows((nrounds - 1) * kRoundFrames, ncomp - (nrounds - 1) * kRoundFrames);

    // ---- phase 3: every thread owns ONE column (c = tid % cols / col = tid % width) and strides over rows, so the loops
    //      are uniform (no integer division, no stream-dependent branch inside them).
    float *s_dhat = reinterpret_cast<float *>(smem + L.off_dhat);
    float *s_dd = reinterpret_cast<float *>(smem + L.off_dd);
    double *s_red = reinterpret_cast<double *>(smem + L.off_red);
    const int T = tl.T, t0 = tl.t0, nout = tl.nout, l1 = a.l1, l2 = a.l2;
#ifdef AFE_DEVTOOLS
    if (a.debug_skip & 4) return;
#endif
    // ownership of the generic row writer and of the fused normalisation: thread = (row group r_off, output column col)
    const int width = a.width;
    const int rpp = kFusedThreads / width; // rows per pass (width <= 128 enforced by the host)
    const bool active = tid < rpp * width;
    const int r_off = tid / width, col = tid - r_off * width;
    const int strm = col / cols, c = col - strm * cols;
    const int n_stats = a.stats_rows_mode == 1 ? T - D : a.stats_rows_mode == 2 ? T : a.stats_rows_mode == 3 ? a.stats_count : 0;
    // source of this thread's column: src[r * cols]; statics of the Q1 rows come from D rows earlier
    const float *src = strm == 0 ? s_cep + (t0 - c0f) * cols + c : strm == 1 ? s_dhat + l2 * cols + c : s_dd + c;
    const int rq = (q1 && strm == 0) ? (q1 == 2 ? 0 : max(0, T - D - t0)) : nout; // first row written with the shifted static
    const int rs = (tl.flags & kTileNoStats) ? 0 : a.stats_rows_mode == 3 ? nout : min(nout, max(0, n_stats - t0)); // rows [0, rs) enter the statistics
    const bool fast3 = a.nstreams == 3 && l1 == 3 && l2 == 3;
    if (fast3 && a.use_last) {
        // flush block of the streaming object: the previous block's statistics (mfcccpu.cpp:389), rows written normalised
        const int cc = tid % cols;
        const float *gm = a.g_mean + (long long)tl.group * width, *gs = a.g_scale + (long long)tl.group * width;
        const float norm3[6] = {gm[cc], gm[cols + cc], gm[2 * cols + cc], gs[cc], gs[cols + cc], gs[2 * cols + cc]};
        dev::phase3_l3<2>(0, a, tl, s_cep, c0f, c1f, nullptr, tid, kFusedThreads, rs, norm3);
    } else if (fast3 && a.cluster_norm) {
        // One cluster = the tiles of one utterance (cluster rank = tile number). Statistics first (MODE 1), records
        // exchanged through distributed shared memory and summed in tile order - the order of the ticket scheme below and
        // of K2, so the results are bitwise the same -, then every tile writes its rows already normalised (MODE 2):
        // the features make ONE trip to HBM and none back through L2.
        double *s_red3 = reinterpret_cast<double *>(smem + L.off_mags);
        double *s_rec = reinterpret_cast<double *>(smem + L.off_mags + 25 * 1024);
        float *s_mean = reinterpret_cast<float *>(smem + L.off_mags + 30 * 1024), *s_scale = s_mean + width;
        dev::phase3_l3<1>(a.stats_kind, a, tl, s_cep, c0f, c1f, s_red3, tid, kFusedThreads, rs);
        __syncthreads();
        if (tid < width) dev::sum_row_groups(s_red3, kFusedThreads / cols, width, tid, [&] { return s_rec + tid * 4; });
        dev::cluster_sync(); // every tile's record is in its CTA's shared memory
        if (tid < width) {   // normalizercpu.cpp:31-66
            const double *rec = s_rec + (a.norm_after_dyn ? tid : tid % cols) * 4;
            const uint32_t ncta = dev::cluster_size();
            double s0 = 0.0, s1 = 0.0, lo = (double)FLT_MAX, hi = -(double)FLT_MAX;
            for (uint32_t t = 0; t < ncta; t++) {
                s0 += dev::ld_peer_f64(rec, t); s1 += dev::ld_peer_f64(rec + 1, t);
                lo = fmin(lo, dev::ld_peer_f64(rec + 2, t)); hi = fmax(hi, dev::ld_peer_f64(rec + 3, t));
            }
            float m, sc;
            finalize_column(a.norm_type, (double)n_stats, s0, s1, (float)lo, (float)hi, m, sc);
            if (!a.norm_after_dyn && tid >= cols) m = 0.f;
            s_mean[tid] = m; s_scale[tid] = sc;
            if (a.g_mean && tile_idx == tl.tile0) { // every tile holds the same values: the group's first tile exports them
                a.g_mean[(long long)tl.group * width + tid] = m;
                a.g_scale[(long long)tl.group * width + tid] = sc;
            }
        }
        __syncthreads();
        {
            const int cc = tid % cols;
            const float norm3[6] = {s_mean[cc], s_mean[cols + cc], s_mean[2 * cols + cc],
                                    s_scale[cc], s_scale[cols + cc], s_scale[2 * cols + cc]};
            dev::phase3_l3<2>(0, a, tl, s_cep, c0f, c1f, s_red3, tid, kFusedThreads, rs, norm3);
        }
        dev::cluster_sync(); // no CTA leaves while a peer may still read its record
    } else if (fast3) {
        // default regression: deltas, rows and statistics in one register-blocked pass (dev::phase3_l3)
        double *s_red3 = reinterpret_cast<double *>(smem + L.off_mags);
        dev::phase3_l3<0>(a.stats_kind, a, tl, s_cep, c0f, c1f, s_red3, tid, kFusedThreads, rs);
        if (a.partials) {
            __syncthreads();
            if (tid < width)
                dev::sum_row_groups(s_red3, kFusedThreads / cols, width, tid, [&] { return a.partials + ((long long)tile_idx * width + tid) * 4; });
        }
    } else {
        if (a.nstreams >= 2) {
            // 3a: delta on the extended axis u in [t0-l2, t0+nout+l2), edge frames replicated (clamped index)
            const int rp = kFusedThreads / cols, rl = tid / cols, c = tid - rl * cols;
            const int nd = nout + 2 * l2;
            if (rl < rp) {
                for (int i = rl; i < nd; i += rp) {
                    const int u = t0 - l2 + i;
                    float num;
                    if (u - l1 >= 0 && u + l1 <= T - 1) // interior: no edge replication needed
                        num = dev::delta_num(s_cep + (u - c0f) * cols + c, cols, l1);
                    else {
                        num = 0.f;
                        for (int l = 1; l <= l1; l++) {
                            const float hi = s_cep[(dev::clampi(u + l, 0, T - 1) - c0f) * cols + c];
                            const float lo = s_cep[(dev::clampi(u - l, 0, T - 1) - c0f) * cols + c];
                            num = fmaf((float)l, hi - lo, num); // deltacpu.cpp:25
                        }
                    }
                    s_dhat[i * cols + c] = num * a.rden1;
                }
            }
            __syncthreads();
            if (a.nstreams >= 3) { // 3b: delta-delta of the extended delta rows
                if (rl < rp)
                    for (int r = rl; r < nout; r += rp)
                        s_dd[r * cols + c] = dev::delta_num(s_dhat + (r + l2) * cols + c, cols, l2) * a.rden2;
                __syncthreads();
            }
        }

        // 3c: rows out (coalesced: consecutive threads write consecutive floats), column statistics
        double sum = 0.0, sumsq = 0.0;
        float mn = FLT_MAX, mx = -FLT_MAX;
        if (round_rows) { // rows already written round by round
            sum = wr_sum; sumsq = wr_sumsq; mn = wr_mn; mx = wr_mx;
        } else if (active) {
            float *orow = a.out + (tl.out_row0 + t0) * (long long)width + col;
            switch (a.stats_kind) {
            case 0: dev::write_rows<0>(orow, src, r_off, rpp, nout, rq, rs, cols, width, D, sum, sumsq, mn, mx); break;
            case 1: dev::write_rows<1>(orow, src, r_off, rpp, nout, rq, rs, cols, width, D, sum, sumsq, mn, mx); break;
            case 2: dev::write_rows<2>(orow, src, r_off, rpp, nout, rq, rs, cols, width, D, sum, sumsq, mn, mx); break;
            default: dev::write_rows<3>(orow, src, r_off, rpp, nout, rq, rs, cols, width, D, sum, sumsq, mn, mx); break;
            }
        }
        if (a.partials) {
            s_red[tid * 4 + 0] = sum;
            s_red[tid * 4 + 1] = sumsq;
            s_red[tid * 4 + 2] = (double)mn;
            s_red[tid * 4 + 3] = (double)mx;
            __syncthreads();
            if (tid < width)
                dev::sum_row_groups(s_red, rpp, width, tid, [&] { return a.partials + ((long long)tile_idx * width + tid) * 4; });
        }
        if (a.use_last) {
            // flush block of the streaming object, generic regression: the rows just written are normalised in place with
            // the previous block's statistics (mfcccpu.cpp:389)
            __syncthreads();
            dev::normalise_tile_rows(a.out, tl, width, a.norm_type, a.g_mean, a.g_scale, reinterpret_cast<float *>(smem + L.off_dhat));
        }
    }

    // ---- fused normalisation (per-utterance statistics scopes): the LAST tile of an utterance to finish reduces the
    //      utterance's per-tile partials in tile order (deterministic, whoever is last), finalises mean / scale
    //      (normalizercpu.cpp:31-66) and normalises the utterance's rows in place while they are still L2 resident.
    //      Replaces K2 + K3 (three launches and one extra HBM round trip of the features).
    if (a.counters) {
        __shared__ int s_last;
        float *s_mean = reinterpret_cast<float *>(smem + L.off_dhat), *s_scale = s_mean + width;
        __threadfence(); // rows + partial record of this tile are visible device-wide before the ticket is taken
        __syncthreads();
        if (tid == 0) {
            const int ticket = atomicAdd(a.counters + tl.group, 1);
            s_last = ticket == tl.ntiles - 1;
            if (s_last) a.counters[tl.group] = 0; // ready for the next launch
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            double s0, s1, lo, hi;
            {
                // records of the group's tiles in the canonical order (segments in parallel for long utterances)
                double *s_seg = reinterpret_cast<double *>(smem + L.off_mags + 1024); // clear of s_mean / s_scale
                const int src_col = a.norm_after_dyn ? tid : tid % cols;
                dev::group_total(a.partials, width, tl.tile0, tl.ntiles, tid, kFusedThreads, s_seg, tid < width ? src_col : 0, s0, s1, lo, hi);
            }
            if (tid < width) {
                float m, sc;
                finalize_column(a.norm_type, (double)n_stats, s0, s1, (float)lo, (float)hi, m, sc);
                if (!a.norm_after_dyn && tid >= cols) m = 0.f;
                s_mean[tid] = m; s_scale[tid] = sc;
                if (a.g_mean) {
                    a.g_mean[(long long)tl.group * width + tid] = m;
                    a.g_scale[(long long)tl.group * width + tid] = sc;
                }
            }
            if (a.work_counter) {
                // long utterance: the normaliser roles take it from here (one per tile, all SMs) instead of this one CTA
                __threadfence();
                __syncthreads();
                if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(a.flags + tl.group), "r"(a.epoch) : "memory");
                return;
            }
            __syncthreads();
            if (active) { // same (row group, column) ownership as the row writer: no division in the loop
                // rows of the group = first tile's t0 .. last tile's end (the whole utterance, or a block of a stream)
                const Tile tf = dev::load_tile(a, tl.tile0), tz = dev::load_tile(a, tl.tile0 + tl.ntiles - 1);
                const int rb = tf.t0, re = tz.t0 + tz.nout;
                float *o = a.out + (tl.out_row0 + rb) * (long long)width + col;
                const float m = s_mean[col], sc = a.norm_type == AFE_NORM_CMN ? 1.f : s_scale[col];
                const bool cmn = a.norm_type == AFE_NORM_CMN;
                const int step = rpp * width;
                o += r_off * width;
                int r = rb + r_off;
                constexpr int U = 8; // loads in flight per thread: the rows come from L2, ~300 cycles away
                for (; r + (U - 1) * rpp < re; r += U * rpp, o += U * step) {
                    float v[U];
#pragma unroll
                    for (int k = 0; k < U; k++) v[k] = __ldcg(o + k * step);
#pragma unroll
                    for (int k = 0; k < U; k++) o[k * step] = cmn ? v[k] - m : (v[k] - m) * sc;
                }
                for (; r < re; r += rpp, o += step) *o = cmn ? __ldcg(o) - m : (__ldcg(o) - m) * sc;
            }
        }
    }
}

} // namespace afe
