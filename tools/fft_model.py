"""NumPy model of the in-kernel real FFT (asr-featext-opencl_b200/csrc/afe_fft.cuh): same lane/slot index maps.

N2-point real FFT = M=N2/2 complex FFT of z[n]=x[2n]+i x[2n+1], M = 16*R (R = lanes per frame, 32, 16 or 8):
  stage A  : lane n2 holds z[R*n1+n2], n1=0..15 -> radix-16 over n1 (4x4, output k1 at slot 4*(k1%4)+k1//4)
  twiddle  : * exp(-2 pi i n2 k1 / M)
  exchange : S[k1][n2] through shared memory
  stage B  : R-point FFT over n2 for each k1 -> Z[k1+16*k2]
  split    : X[k], X[M-k] from Z[k], Z[M-k]; k=0 -> X[0], X[M]; k=M/2 separately
R = 32 (1024 points, rfft_model_1024): lane n2 = a + 16 b. Lanes with b = 1 negate their odd-n1 window pairs, so their
radix-16 output slot of k1 holds k1 + 8 (mod 16); each lane then keeps the slots of its own half of k1 (8 b + j, j < 8),
swaps the other half with lane n2 ^ 16 and runs the radix-2 butterfly over b (the twiddle W32^a on the difference, negated
in lanes b = 1) before the exchange. Exchange row k1 + 16 d holds the 16 values over a; its lane runs a radix-16 over a and
holds Z[lane + 32 c] at slot pos16(c): the real split is the R = 16 one with R = 32.
Used by tests/test_host_logic.py and tests/test_fft1024.py to pin the decompositions against numpy.fft.rfft.
"""
import numpy as np


def fft4(a0, a1, a2, a3):
    s02, d02, s13, d13 = a0 + a2, a0 - a2, a1 + a3, a1 - a3
    return s02 + s13, d02 - 1j * d13, s02 - s13, d02 + 1j * d13


def fft16_slots(x):
    """x: list of 16 complex (natural order). Returns list y with y[4*(k%4)+k//4] = X[k]."""
    x = list(x)
    for b in range(4):
        x[b], x[4 + b], x[8 + b], x[12 + b] = fft4(x[b], x[4 + b], x[8 + b], x[12 + b])
    for c in range(1, 4):
        for b in range(1, 4):
            x[4 * c + b] = x[4 * c + b] * np.exp(-2j * np.pi * b * c / 16)
    for c in range(4):
        x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3] = fft4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3])
    return x


def fft8_slots(x):
    """y[2*(k%4)+k//4] = X[k]"""
    x = list(x)
    for b in range(2):
        x[b], x[2 + b], x[4 + b], x[6 + b] = fft4(x[b], x[2 + b], x[4 + b], x[6 + b])
    for c in range(1, 4):
        x[2 * c + 1] = x[2 * c + 1] * np.exp(-2j * np.pi * c / 8)
    for c in range(4):
        x[2 * c], x[2 * c + 1] = x[2 * c] + x[2 * c + 1], x[2 * c] - x[2 * c + 1]
    return x


def pos16(k):
    return 4 * (k % 4) + k // 4


def pos8(k):
    return 2 * (k % 4) + k // 4


def rfft_model(x):
    N2 = len(x)
    M = N2 // 2
    R = M // 16
    assert R in (8, 16)
    z = x[0::2] + 1j * x[1::2]
    # stage A + twiddle, per lane n2
    S = np.zeros((16, R), complex)
    for n2 in range(R):
        y = fft16_slots([z[R * n1 + n2] for n1 in range(16)])
        for k1 in range(16):
            S[k1, n2] = y[pos16(k1)] * np.exp(-2j * np.pi * n2 * k1 / M)
    # stage B
    Z = np.zeros(M, complex)
    for lane in range(R):
        for k1 in ([lane] if R == 16 else [lane, lane + 8]):
            if R == 16:
                y = fft16_slots(list(S[k1, :]))
                for k2 in range(16):
                    Z[k1 + 16 * k2] = y[pos16(k2)]
            else:
                y = fft8_slots(list(S[k1, :]))
                for k2 in range(8):
                    Z[k1 + 16 * k2] = y[pos8(k2)]
    # split; magnitudes of 2*X
    X = np.zeros(M + 1, complex)
    for lane in range(R):
        for m in range(8):
            k = lane + R * m
            a, b = Z[k], Z[(M - k) % M]
            w = np.exp(-2j * np.pi * k / N2)
            sr, si = a.real + b.real, a.imag - b.imag
            dr, di = a.real - b.real, a.imag + b.imag
            pr, pi = dr * w.real - di * w.imag, dr * w.imag + di * w.real
            X[k] = 0.5 * complex(sr + pi, si - pr)
            X[M - k] = 0.5 * complex(sr - pi, -(si + pr))
    X[M // 2] = np.conj(Z[M // 2])
    return X


def rfft_model_1024(x):
    N2 = len(x)
    assert N2 == 1024
    M, R = N2 // 2, 32
    z = x[0::2] + 1j * x[1::2]
    # stage A per lane n2 = a + 16 b: odd-n1 inputs of lanes b = 1 negated (their window pairs), radix 16 over n1
    V = np.zeros((R, 16), complex)               # V[n2][j]: the value lane n2 keeps in logical slot j
    for n2 in range(R):
        b = n2 >> 4
        y = fft16_slots([z[R * n1 + n2] * (-1 if b and n1 % 2 else 1) for n1 in range(16)])
        for j in range(16):
            k1 = (j + 8 * b) % 16                # slot pos16(j) holds X[k1]
            V[n2, j] = y[pos16(j)] * np.exp(-2j * np.pi * n2 * k1 / M)
    # lane pair (a, a + 16): slots j < 8 kept, slots 8 + j swapped; butterfly over b; exchange S[k1 + 16 d][a]
    S = np.zeros((32, 16), complex)
    for n2 in range(R):
        a, b = n2 & 15, n2 >> 4
        t = (-1 if b else 1) * np.exp(-2j * np.pi * a / 32)
        for j in range(8):
            own, got = V[n2, j], V[n2 ^ 16, 8 + j]
            k1 = 8 * b + j
            S[k1, a] = own + got
            S[k1 + 16, a] = (own - got) * t
    # stage C: lane L runs radix 16 over a on row L -> Z[L + 32 c] at slot pos16(c)
    Z = np.zeros(M, complex)
    for L in range(R):
        y = fft16_slots(list(S[L, :]))
        for c in range(16):
            Z[L + 32 * c] = y[pos16(c)]
    # split: lane L finalises k = L + 32 m, m < 8, and M - k (the R = 16 rule with R = 32)
    X = np.zeros(M + 1, complex)
    for lane in range(R):
        for m in range(8):
            k = lane + R * m
            a, b = Z[k], Z[(M - k) % M]
            w = np.exp(-2j * np.pi * k / N2)
            c, d = a + np.conj(b), a - np.conj(b)
            p = d * w
            X[k] = 0.5 * (c - 1j * p)
            X[M - k] = np.conj(0.5 * (c + 1j * p))
    X[M // 2] = np.conj(Z[M // 2])
    return X


if __name__ == "__main__":
    rng = np.random.default_rng(0)
    for N2 in (512, 256):
        x = rng.standard_normal(N2)
        err = np.abs(rfft_model(x) - np.fft.rfft(x)).max()
        print(N2, err)
        assert err < 1e-10
    x = rng.standard_normal(1024)
    err = np.abs(rfft_model_1024(x) - np.fft.rfft(x)).max()
    print(1024, err)
    assert err < 1e-10
