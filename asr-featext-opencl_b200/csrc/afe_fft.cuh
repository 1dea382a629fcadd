// In-register batched real FFT (256/512/1024 point) + magnitude, replacing clfft.cpp / AppleFFT and mfcc.cl:kernelTranspose.
//
// An N2-point real frame is transformed as an M = N2/2 point complex FFT of z[n] = x[2n] + i*x[2n+1] (one 32-bit
// shared-memory word holds both int16 samples), M = 16*R:
//   R lanes cooperate on one frame (R = 32 for N2 = 1024, 16 for 512, 8 for 256), so a warp transforms 32/R frames at once.
//   stage A   lane n2 holds z[R*n1 + n2], n1 = 0..15, and runs a radix-16 butterfly (4x4) entirely in registers
//   twiddle   * exp(-2 pi i n2 k1 / M) from per-lane registers
//   exchange  one trip through a padded shared-memory tile S[k1][n2] (the only data exchange of the transform)
//   stage B   R-point FFT over n2 (radix-16, or two radix-8) in registers -> Z[k1 + 16 k2]
//   split     X[k], X[M-k] from Z[k] (own registers) and Z[M-k] (one warp shuffle from the mirror lane) -> |X| row
// R = 32 (1024 points): the 32-point FFT over n2 = a + 16 b is split by decimation in frequency. Lane pairs (a, a + 16)
// run the radix-2 butterfly over b BEFORE the exchange, after one swap of 8 values through __shfl_xor_sync(.., 16):
// lanes with b = 1 load their odd-n1 window pairs negated, which rotates their stage-A outputs by 8 slots, so every lane
// keeps the same slots (its own half of k1) and sends the same slots (the other half). The exchange tile then holds row
// k1 + 16 d = 16 values over a, and stage B is one radix-16 per lane -> Z[lane + 32 c]: the split is the R = 16 one.
// The index maps are modelled and checked against numpy.fft.rfft in tools/fft_model.py / tests/test_host_logic.py.
// Reference semantics: fftwf r2c unnormalised (mfcccpu.cpp:114,189), v = sqrt(re^2+im^2)/N2 (mfcccpu.cpp:203).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace afe {
namespace dev {

constexpr float kC1 = 0.92387953251128674f; // cos(pi/8)
constexpr float kS1 = 0.38268343236508977f; // sin(pi/8)
constexpr float kR2 = 0.70710678118654752f; // sqrt(1/2)

// ---- packed FP32 arithmetic (sm_100a FADD2 / FMUL2 / FFMA2): one instruction works on a (re, im) register pair, and
// the operand modifiers of those instructions swap the halves (.LO_HI), negate either half (.NP / .PN) or broadcast a
// scalar (.F32) for free. A complex add, a multiplication by +-i folded into an add, and half of a complex product
// are therefore ONE issue slot each; this kernel is bound by issue slots, not by the FP32 pipe
// (tools/ubench/f32x2.cu: FADD2 + 1 ALU op runs 1.33x faster than 2 FADD + 1 ALU op on B200).
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 add_mi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(b.y, -b.x)); } // a - i*b
__device__ __forceinline__ float2 add_pi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.y, b.x)); } // a + i*b
__device__ __forceinline__ float2 cmul(float2 a, float2 b) // a*b.x + (i*a)*b.y
{
    return __ffma2_rn(make_float2(-a.y, a.x), make_float2(b.y, b.y), __fmul2_rn(a, make_float2(b.x, b.x)));
}

// forward 4-point DFT, natural order in and out: 8 packed instructions
__device__ __forceinline__ void fft4(float2 &a0, float2 &a1, float2 &a2, float2 &a3)
{
    const float2 s02 = cadd(a0, a2), d02 = csub(a0, a2), s13 = cadd(a1, a3), d13 = csub(a1, a3);
    a0 = cadd(s02, s13);
    a2 = csub(s02, s13);
    a1 = add_mi(d02, d13);
    a3 = add_pi(d02, d13);
}

// (x+iy) * exp(-i pi/4), * (-i), * exp(-3 i pi/4)
__device__ __forceinline__ float2 mul_w8_1(float2 v) { return __fmul2_rn(add_mi(v, v), make_float2(kR2, kR2)); }
__device__ __forceinline__ float2 mul_mi(float2 v) { return make_float2(v.y, -v.x); } // folds into the consumer's operand modifiers
__device__ __forceinline__ float2 mul_w8_3(float2 v) { return __fmul2_rn(add_pi(v, v), make_float2(-kR2, -kR2)); }

// forward 16-point DFT in registers. Input natural order; output X[k] lands in slot 4*(k%4) + k/4.
__device__ __forceinline__ void fft16(float2 (&x)[16])
{
#pragma unroll
    for (int b = 0; b < 4; b++) fft4(x[b], x[4 + b], x[8 + b], x[12 + b]);
    // slot 4c+b *= W16^(b*c)
    x[5] = cmul(x[5], make_float2(kC1, -kS1));   // W^1
    x[6] = mul_w8_1(x[6]);                       // W^2
    x[7] = cmul(x[7], make_float2(kS1, -kC1));   // W^3
    x[9] = mul_w8_1(x[9]);                       // W^2
    x[10] = mul_mi(x[10]);                       // W^4
    x[11] = mul_w8_3(x[11]);                     // W^6
    x[13] = cmul(x[13], make_float2(kS1, -kC1)); // W^3
    x[14] = mul_w8_3(x[14]);                     // W^6
    x[15] = cmul(x[15], make_float2(-kC1, kS1)); // W^9
#pragma unroll
    for (int c = 0; c < 4; c++) fft4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
}
__host__ __device__ constexpr int pos16(int k) { return 4 * (k % 4) + k / 4; }

// forward 8-point DFT on x[o..o+7]. Output X[k] lands in slot o + 2*(k%4) + k/4.
template <int O> __device__ __forceinline__ void fft8(float2 (&x)[16])
{
    fft4(x[O + 0], x[O + 2], x[O + 4], x[O + 6]);
    fft4(x[O + 1], x[O + 3], x[O + 5], x[O + 7]);
    x[O + 3] = mul_w8_1(x[O + 3]);
    x[O + 5] = mul_mi(x[O + 5]);
    x[O + 7] = mul_w8_3(x[O + 7]);
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const float2 a = x[O + 2 * c], b = x[O + 2 * c + 1];
        x[O + 2 * c] = cadd(a, b);
        x[O + 2 * c + 1] = csub(a, b);
    }
}
__host__ __device__ constexpr int pos8(int k) { return 2 * (k % 4) + k / 4; }

template <int N2> struct FftCfg {
    static_assert(N2 == 1024 || N2 == 512 || N2 == 256, "in-register FFT supports 256, 512 and 1024 points");
    static constexpr int M = N2 / 2;         // complex length
    static constexpr int R = M / 16;         // lanes per frame
    static constexpr int FPW = 32 / R;       // frames per warp
    // padded row stride of the exchange tile (float2 units): 16 rows of R values, or at 1024 points 32 rows of 16 values
    static constexpr int RS = R == 32 ? 17 : R + 1;
    static constexpr int SCR = R == 32 ? 32 * RS : 16 * RS + (R == 8 ? 1 : 0); // per-frame scratch (float2 units), >= M
    static constexpr int BINS = M + 1;
};

// forward 16-point DFT whose inputs x[NZ..15] are known to be zero (zero-padded window tail): prunes the first
// radix-4 layer. NZ >= 13 keeps x[0..12]; anything else falls back to the full butterfly.
template <int NZ> __device__ __forceinline__ void fft16_in(float2 (&x)[16])
{
    if (NZ == 13) {
        fft4(x[0], x[4], x[8], x[12]);
#pragma unroll
        for (int b = 1; b < 4; b++) { // a3 == 0: s13 = d13 = a1
            const float2 a0 = x[b], a1 = x[4 + b], a2 = x[8 + b];
            const float2 s02 = cadd(a0, a2), d02 = csub(a0, a2);
            x[b] = cadd(s02, a1);
            x[8 + b] = csub(s02, a1);
            x[4 + b] = add_mi(d02, a1);
            x[12 + b] = add_pi(d02, a1);
        }
        x[5] = cmul(x[5], make_float2(kC1, -kS1));
        x[6] = mul_w8_1(x[6]);
        x[7] = cmul(x[7], make_float2(kS1, -kC1));
        x[9] = mul_w8_1(x[9]);
        x[10] = mul_mi(x[10]);
        x[11] = mul_w8_3(x[11]);
        x[13] = cmul(x[13], make_float2(kS1, -kC1));
        x[14] = mul_w8_3(x[14]);
        x[15] = cmul(x[15], make_float2(-kC1, kS1));
#pragma unroll
        for (int c = 0; c < 4; c++) fft4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
    } else
        fft16(x);
}

// Per-lane constants kept in registers for the whole kernel (shared memory bandwidth is the scarce resource here,
// profiles/r01_v4b_8x4_k_fused_summary.txt): window pairs, exchange twiddles, split twiddles.
// R = 32, lane = a + 16 b: b = 1 negates win[n1] for odd n1 and takes twa[j] for k1 = (j + 8) % 16; twb = (-1)^b W32^a.
template <int N2, int NZ> struct LaneConsts {
    float2 win[NZ]; // (w[2n], w[2n+1]) for n = R*n1 + lane, n1 < NZ (zero beyond)
    float2 twa[16]; // exp(-2 pi i lane*k1 / M)
    float2 twp[8];  // exp(-2 pi i (lane + R*m) / N2)
    float2 twb;     // R = 32 only: twiddle of the radix-2 difference
};

template <int N2, int NZ>
__device__ __forceinline__ void load_lane_consts(LaneConsts<N2, NZ> &lc, const float2 *__restrict__ window2,
                                                 const float2 *__restrict__ tw_a, const float2 *__restrict__ tw_p, int lf)
{
    using C = FftCfg<N2>;
    if (C::R == 32) {
        const int b = lf >> 4;
#pragma unroll
        for (int n1 = 0; n1 < NZ; n1++) {
            const float2 w = window2[C::R * n1 + lf];
            lc.win[n1] = b && (n1 & 1) ? make_float2(-w.x, -w.y) : w;
        }
#pragma unroll
        for (int j = 0; j < 16; j++) lc.twa[j] = tw_a[lf * 16 + ((j + 8 * b) & 15)];
        const float2 t = tw_a[(lf & 15) * 32 + 8]; // exp(-2 pi i 16 a / M) = W32^a
        lc.twb = b ? make_float2(-t.x, -t.y) : t;
    } else {
#pragma unroll
        for (int n1 = 0; n1 < NZ; n1++) lc.win[n1] = window2[C::R * n1 + lf];
#pragma unroll
        for (int k1 = 0; k1 < 16; k1++) lc.twa[k1] = tw_a[lf * 16 + k1];
    }
#pragma unroll
    for (int m = 0; m < 8; m++) lc.twp[m] = tw_p[lf + C::R * m];
}

template <bool FAST> __device__ __forceinline__ float mag_sqrt(float x)
{
    if (FAST) {
        float r;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
        return r;
    }
    return sqrtf(x);
}

// One frame per R-lane group; ALL 32 lanes of the warp must call (uses __syncwarp). Branch free.
//   words    : the frame's PCM as 32-bit words (2 int16 each), readable for NZ*R words; samples beyond W meet a 0 window
//   NZ       : leading n1 slots that can be non-zero (13 when W <= 26*R, else 16)
//   lc       : this lane's window pairs and twiddles (registers)
//   scratch  : this frame's exchange tile, FftCfg::SCR float2
//   mag_out  : BINS floats (always written; padding frames point at a row nobody reads)
//   SCALED   : true -> |X|/N2 (reference value); false -> |2X| (= 2*N2 times that; the caller folds the exact
//              power-of-two factor 0.5/N2 into its mel weights)
//   PRE      : compile the pre-emphasis variant of the load (taken when pre != 0); false keeps the reference path free of it
template <int N2, int NZ, bool FAST, bool SCALED = true, bool PRE = true>
__device__ __forceinline__ void fft_frame_mag(const uint32_t *words, const LaneConsts<N2, NZ> &lc, float2 *scratch,
                                              float *mag_out, int lf, float pre = 0.f)
{
    using C = FftCfg<N2>;
    constexpr int M = C::M, R = C::R, RS = C::RS;
    float2 x[16];
    if (!PRE || pre == 0.f) { // the reference has no pre-emphasis (segmentercpu.cpp:21-27), this is its path
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) {
            if (n1 < NZ) {
                const uint32_t w = words[R * n1 + lf];
                const float2 wn = lc.win[n1];
                const float lo = (float)(int)(short)(w & 0xffffu);
                const float hi = (float)((int)w >> 16);
                x[n1] = __fmul2_rn(make_float2(lo, hi), wn);
            } else
                x[n1] = make_float2(0.f, 0.f);
        }
    } else {
        // per-frame pre-emphasis y[j] = x[j] - pre * x[j-1], y[0] = (1 - pre) * x[0] (HTK / Kaldi convention), then the
        // window: w[j] * x[j] + (-pre * w[j]) * x[j-1]
        const float2 mp = make_float2(-pre, -pre);
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) {
            if (n1 < NZ) {
                const int idx = R * n1 + lf;
                const uint32_t w = words[idx], wp = words[idx > 0 ? idx - 1 : 0];
                const float2 wn = lc.win[n1];
                const float lo = (float)(int)(short)(w & 0xffffu);
                const float hi = (float)((int)w >> 16);
                const float prev = idx > 0 ? (float)((int)wp >> 16) : lo;
                x[n1] = __ffma2_rn(make_float2(prev, lo), __fmul2_rn(wn, mp), __fmul2_rn(make_float2(lo, hi), wn));
            } else
                x[n1] = make_float2(0.f, 0.f);
        }
    }
    fft16_in<NZ>(x);
    if (R == 32) {
        // twiddle; keep slots j < 8 (k1 = 8 b + j), swap slots 8 + j with lane ^ 16; radix 2 over b -> S[k1 + 16 d][a]
        float2 v[16];
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = cmul(x[pos16(j)], lc.twa[j]);
        float2 *row = scratch + (lf >> 4) * 8 * RS + (lf & 15);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            float2 got;
            got.x = __shfl_xor_sync(0xffffffffu, v[8 + j].x, 16);
            got.y = __shfl_xor_sync(0xffffffffu, v[8 + j].y, 16);
            row[j * RS] = cadd(v[j], got);
            row[(16 + j) * RS] = cmul(csub(v[j], got), lc.twb);
        }
    } else {
        // twiddle + exchange: S[k1][n2]
#pragma unroll
        for (int k1 = 0; k1 < 16; k1++) {
            float2 v = x[pos16(k1)];
            if (k1 > 0) v = cmul(v, lc.twa[k1]);
            scratch[k1 * RS + lf] = v;
        }
    }
    __syncwarp();
    if (R >= 16) { // R = 32: row lf holds the 16 values over a
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) x[n2] = scratch[lf * RS + n2];
        fft16(x);
    } else {
#pragma unroll
        for (int n2 = 0; n2 < 8; n2++) {
            x[n2] = scratch[lf * RS + n2];
            x[8 + n2] = scratch[(lf + 8) * RS + n2];
        }
        fft8<0>(x);
        fft8<8>(x);
    }
    __syncwarp();
    // Real split without another trip through shared memory: lane lf finalises the bins k = lf + R*m, m = 0..7, and
    // their mirrors M-k. Z[k] is already in its registers; Z[M-k] lives in lane (R-lf)%R of the same frame:
    //   R = 16, 32: slot 15-m                      (lane 0 pairs with itself: Z[M-Rm] = its own slot 16-m; Z[M] := Z[0])
    //   R =  8: the other 8-point group, slot 7-m/2 (lane 0: same group; group 0 pairs with slot 8-m/2)
    // so every lane sends 8 complex values through one shuffle each way.
    float2 za[8], zb[8];
    const int src = (threadIdx.x & 31 & ~(R - 1)) | ((R - lf) & (R - 1));
#pragma unroll
    for (int m = 0; m < 8; m++) {
        float2 own, send, self;
        if (R >= 16) {
            own = x[pos16(m)];
            send = x[pos16(15 - m)];
            self = m == 0 ? x[pos16(0)] : x[pos16(16 - m)];
        } else {
            own = (m & 1) ? x[8 + pos8(m >> 1)] : x[pos8(m >> 1)];
            send = (m & 1) ? x[pos8(7 - (m >> 1))] : x[8 + pos8(7 - (m >> 1))];
            self = (m & 1) ? x[8 + pos8(7 - (m >> 1))] : (m == 0 ? x[pos8(0)] : x[pos8(8 - (m >> 1))]);
        }
        float2 got;
        got.x = __shfl_sync(0xffffffffu, send.x, src);
        got.y = __shfl_sync(0xffffffffu, send.y, src);
        za[m] = own;
        zb[m] = lf == 0 ? self : got;
    }
    const float scale = 0.5f / (float)N2; // |2X| * 0.5/N2 == |X|/N2 exactly (powers of two)
    float *mf = mag_out + lf, *mr = mag_out + (M - lf);
#pragma unroll
    for (int m = 0; m < 8; m++) {
        const float2 a = za[m], b = zb[m];
        const float2 w = lc.twp[m];
        const float2 c = __fadd2_rn(a, make_float2(b.x, -b.y));  // a + conj(b)
        const float2 d = __fadd2_rn(a, make_float2(-b.x, b.y));  // a - conj(b)
        const float2 p = cmul(d, w);
        const float2 x1 = add_mi(c, p), x2 = add_pi(c, p);       // 2 X[k], 2 conj(X[M-k])
        const float x1r = x1.x, x1i = x1.y, x2r = x2.x, x2i = x2.y;
        const float v1 = mag_sqrt<FAST>(x1r * x1r + x1i * x1i), v2 = mag_sqrt<FAST>(x2r * x2r + x2i * x2i);
        mf[R * m] = SCALED ? v1 * scale : v1;
        mr[-R * m] = SCALED ? v2 * scale : v2;
    }
    if (lf == 0) {
        const float2 a = R >= 16 ? x[pos16(8)] : x[pos8(4)]; // X[M/2] = conj(Z[M/2]): k1 = 0, k2 = M/32 (R = 32: c = 8)
        const float vm = mag_sqrt<FAST>(a.x * a.x + a.y * a.y);
        mag_out[M / 2] = SCALED ? vm * (1.0f / (float)N2) : vm + vm;
    }
    __syncwarp();
}

} // namespace dev
} // namespace afe
