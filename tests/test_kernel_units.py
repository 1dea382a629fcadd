"""Device unit tests of the hand-written numerics under the fused kernel K1 and the staged kernels, each against a float64
reference of the same operation: the packed log dev::mel_log2 (afe_mel.cuh) over every finite float, and the in-register
FFT + magnitude dev::fft_frame_mag (afe_fft.cuh) in every instantiation the library runs.

The end-to-end feature comparisons cannot see these errors: a relative error of 1e-5 in every mel energy moves c0 by
about 9e-5 at 40 banks, inside their 5e-4 tolerance. tests/cuda/afe_units.cu is compiled here with the library's nvcc
flags into a temporary directory (never into the tree) and called through ctypes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "cuda", "afe_units.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# asr-featext-opencl_b200/Makefile: NVFLAGS, run from the repository root
NVFLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC,-Wall",
           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "asr-featext-opencl_b200", "csrc")]
ENTRY_POINTS = ("afe_units_log_sweep", "afe_units_log_points", "afe_units_fft_mag")

POS_FINITE = 0x7f800000                   # bit patterns 0 .. 0x7f7fffff: +0 .. the largest finite float
CLAMP = np.float32(1e-30)


@pytest.fixture(scope="module")
def units_so(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("afe_units") / "libafe_units.so")
    r = subprocess.run([NVCC, *NVFLAGS, "-shared", "-o", so, SRC], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return so


@pytest.fixture(scope="module")
def units(units_so):
    L = C.CDLL(units_so)
    u64p, fp, dp = C.POINTER(C.c_ulonglong), C.POINTER(C.c_float), C.POINTER(C.c_double)
    L.afe_units_log_sweep.restype, L.afe_units_log_sweep.argtypes = C.c_int, [C.c_ulonglong] * 3 + [u64p]
    L.afe_units_log_points.restype, L.afe_units_log_points.argtypes = C.c_int, [fp, C.c_int, fp, dp]
    L.afe_units_fft_mag.restype = C.c_int
    L.afe_units_fft_mag.argtypes = [C.c_int] * 3 + [C.POINTER(C.c_short), C.c_int, fp, fp, fp, C.c_float, fp]
    return L


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def test_unit_harness_compiles(units_so):
    """CPU-only: the harness still compiles against the current headers and exports its entry points."""
    L = C.CDLL(units_so)
    for name in ENTRY_POINTS:
        getattr(L, name)


# ---------------------------------------------------------------------------------------------- packed log
def f32_ulp(ref):
    """Float ulp at float64 values ref (ref != 0): 2^(e-24) for |ref| in [2^(e-1), 2^e)."""
    _, e = np.frexp(ref)
    return np.ldexp(1.0, e - 24)


def log_points(units, x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros((len(x), 4), np.float32)
    ref = np.zeros(len(x), np.float64)
    assert units.afe_units_log_points(_ptr(x, C.c_float), len(x), _ptr(out, C.c_float), _ptr(ref, C.c_double)) == 0
    return out, ref


@pytest.mark.gpu
def test_packed_log_sweep_every_finite_float(units):
    """mel_log2<false> in both lanes, and mel_log<false>, over every finite float bit pattern (2 * 0x7f800000 inputs,
    2^31 of them non-negative) against log((double)fmaxf(x, 1e-30f)) on the device.

    Measured on a B200: max error 0.8697 ulp in both lanes, at x = 1.5580899 (0x3fc76f7d); 720652 results differ from
    logf's (whose own maximum here is 0.8642 ulp). The whole sweep takes about a second. Every input <= 1e-30f (+-0,
    denormals, negative numbers) returns exactly the value for 1e-30f."""
    stats = np.zeros(12, np.uint64)
    assert units.afe_units_log_sweep(0, 2 * POS_FINITE, 1 << 28, _ptr(stats, C.c_ulonglong)) == 0
    names = ("mel_log2 lane x", "mel_log2 lane y", "mel_log")
    worst = {}
    for v, name in enumerate(names):
        key, differ, clamp_bad = (int(s) for s in stats[4 * v:4 * v + 3])
        err = float(np.uint32(key >> 32).view(np.float32))
        arg = np.uint32(key & 0xffffffff).view(np.float32)
        worst[name] = err
        print(f"{name}: max error {err:.4f} ulp at x = {arg!r} ({key & 0xffffffff:#010x}); {differ} results differ from "
              f"logf; {clamp_bad} clamp mismatches")
        assert clamp_bad == 0, name
        assert err <= 1.0, name
    assert stats[4 * 2 + 1] == 0                   # mel_log<false> is logf after the clamp
    assert worst["mel_log2 lane x"] == worst["mel_log2 lane y"]


@pytest.mark.gpu
def test_packed_log_clamp_and_nan(units):
    """x <= 1e-30f and NaN: fmaxf returns the other operand for a NaN, so every such input gives log(1e-30f) =
    -69.0776 exactly, in both lanes and in the scalar form."""
    bits = np.array([0x00000000, 0x80000000, 0x00000001, 0x007fffff, 0x00800000, 0x80000001, 0xbf800000, 0xff7fffff,
                     0xff800000, 0x7fc00000, 0x7f800001, 0xffc00000, 0xffffffff, 0x7fffffff], np.uint32)
    x = np.concatenate([bits.view(np.float32), [CLAMP, np.nextafter(CLAMP, np.float32(0))]]).astype(np.float32)
    out, _ = log_points(units, x)
    (c_out,), _ = log_points(units, np.array([CLAMP], np.float32))
    for col in range(3):
        np.testing.assert_array_equal(out[:, col].view(np.uint32), np.full(len(x), c_out[col].view(np.uint32)))
    assert abs(float(c_out[0]) - np.log(np.float64(CLAMP))) <= f32_ulp(np.log(np.float64(CLAMP)))
    up, _ = log_points(units, np.array([1e-29], np.float32))
    assert up[0, 0] > c_out[0]


@pytest.mark.gpu
def test_packed_log_random_against_numpy(units):
    """Host-side check of the sweep's device reference and of the ulp bound: 4 M random finite floats (uniform bit
    patterns and log-uniform values), every power of two and the float neighbours of the mantissa split points 2/3 and
    4/3 in every binade, against NumPy's float64 np.log."""
    rng = np.random.default_rng(20261020)
    x = [rng.integers(0, POS_FINITE, 2_000_000, dtype=np.uint32).view(np.float32),
         np.exp(rng.uniform(np.log(1e-30), np.log(3e38), 2_000_000)).astype(np.float32)]
    e = np.arange(-126, 128, dtype=np.float64)
    x.append(np.ldexp(np.float32(1), e.astype(np.int32)).astype(np.float32))
    for split in (np.float32(2 / 3), np.float32(4 / 3)):
        base = np.ldexp(np.float64(split), e.astype(np.int32)[:-1]).astype(np.float32)
        for k in range(-3, 4):
            x.append((base.view(np.int32) + k).view(np.float32))
    x = np.concatenate(x).astype(np.float32)
    x = x[np.isfinite(x)]
    out, dev_ref = log_points(units, x)
    ref = np.log(np.maximum(x, CLAMP).astype(np.float64))
    np.testing.assert_array_less(np.abs(dev_ref - ref), 2 * np.spacing(np.abs(ref)) + 1e-300)
    np.testing.assert_array_equal(out[:, 0].view(np.uint32), out[:, 1].view(np.uint32))   # the lanes agree
    np.testing.assert_array_equal(out[:, 2].view(np.uint32), out[:, 3].view(np.uint32))   # mel_log == logf
    nz = ref != 0
    err = np.abs(out[nz, 0].astype(np.float64) - ref[nz]) / f32_ulp(ref[nz])
    assert np.all(out[~nz, 0] == 0)
    print(f"packed log, {len(x)} points: max error {err.max():.4f} ulp at x = {x[nz][err.argmax()]!r}")
    assert err.max() <= 1.0


# ---------------------------------------------------------------------------------------------- FFT + magnitude
SHAPES = {(512, 13): (400, 401, 416), (512, 16): (417, 480, 512), (256, 13): (129, 200, 208), (256, 16): (209, 256)}
# caller -> (label, SCALED, preemphasis coefficients run through it); see afe_units.cu:dispatch_unit_fft
CALLERS = {0: ("k1", False, (0.0,)), 1: ("k1pre", False, (0.97,)), 2: ("staged", True, (0.0, 0.97))}
# max_k |mag_k - ref_k| <= TAU[N2] * ||ref||_2 per frame. Worst measured on a B200 over the 12 instantiations and these
# inputs: 1.71e-7 at 512 points, 2.78e-7 at 256 points (the pre-emphasis load). A relative 1e-5 error in one tw_a entry
# moves a bin by about 1e-5 / R of the frame's norm (R = N2 / 32 lanes share a twiddle column): 6.3e-7 at 512 points,
# 8.9e-7 at 256; one tw_p entry: 3e-6. TAU sits between the two, 2.3x and 2.2x the worst error seen.
TAU = {512: 4e-7, 256: 6e-7}


def fft_tables(n2):
    """FftTables::build (afe_batch.cu:18-37): the same double expressions, rounded to float."""
    M = n2 // 2
    R = M // 16
    lk = (np.arange(R)[:, None] * np.arange(16)[None, :]).astype(np.float64).ravel()
    ang = -2.0 * np.pi * lk / M
    tw_a = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    ang = -2.0 * np.pi * np.arange(M // 2, dtype=np.float64) / n2
    tw_p = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    return tw_a, tw_p


def window2(window, n2):
    """upload_window (afe_batch.cu:78-87): the float window zero-padded to N2, read as (w[2n], w[2n+1]) pairs."""
    w2 = np.zeros(n2, np.float32)
    w2[:len(window)] = window
    return w2


def fft_inputs(W, n2, rng):
    """Frames of n2 int16 samples; samples from W on are random and must not leak through the zero window tail."""
    full = lambda: rng.integers(-32768, 32768, n2).astype(np.int16)
    frames = []

    def add(x):
        f = full()
        f[:W] = x
        frames.append(f)
    n = np.arange(W)
    for i in range(32):                                              # uniform over the full range, -32768 included
        x = full()[:W]
        x[(7 * i) % W] = -32768
        add(x)
    for half in (1, 5, 25, 64):                                       # full-scale square waves
        add(np.where((n // half) % 2 == 0, 32767, -32768))
    add(np.full(W, 32767))                                            # DC
    add(np.full(W, -32768))
    for m in range(W):                                                # an impulse in every load slot (lane, n1)
        x = np.zeros(W, np.int16)
        x[m] = 32767 if m % 2 else -32768
        add(x)
    for k in range(n2 // 2 + 1):                                      # a cosine at every bin: every real-split slot
        add(np.round(30000 * np.cos(2 * np.pi * k * n / n2)))
    add(np.zeros(W, np.int16))                                        # zeros: exactly 0 (must stay the last frame)
    return np.stack(frames)


def fft_reference(frames, W, window, n2, pre, scaled):
    """float64 rfft of the float32 window times the PCM, pre-emphasis as oracle/oracle_np.py:mfcc defines it."""
    x = frames[:, :W].astype(np.float64)
    if pre:
        x = x - np.float64(np.float32(pre)) * np.concatenate([x[:, :1], x[:, :-1]], axis=1)
    fr = np.zeros((len(frames), n2))
    fr[:, :W] = x * window.astype(np.float64)
    mag = np.abs(np.fft.rfft(fr, axis=1))
    return mag / n2 if scaled else 2.0 * mag


def run_fft(units, n2, nz, caller, frames, w2, tw_a, tw_p, pre):
    frames = np.ascontiguousarray(frames, np.int16)
    mag = np.zeros((len(frames), n2 // 2 + 1), np.float32)
    rc = units.afe_units_fft_mag(n2, nz, caller, _ptr(frames, C.c_short), len(frames), _ptr(w2, C.c_float),
                                 _ptr(np.ascontiguousarray(tw_a), C.c_float), _ptr(np.ascontiguousarray(tw_p), C.c_float),
                                 float(pre), _ptr(mag, C.c_float))
    assert rc == 0, f"CUDA error {rc}"
    return mag


def normwise_error(mag, ref):
    """per frame max_k |mag_k - ref_k| / ||ref||_2 (frames with ref == 0 excluded)"""
    nrm = np.sqrt((ref * ref).sum(1))
    err = np.abs(mag.astype(np.float64) - ref).max(1)
    live = nrm > 0
    return err[live] / nrm[live]


@pytest.mark.gpu
@pytest.mark.parametrize("caller", sorted(CALLERS), ids=[CALLERS[c][0] for c in sorted(CALLERS)])
@pytest.mark.parametrize("n2,nz", sorted(SHAPES), ids=[f"{a}-{b}" for a, b in sorted(SHAPES)])
def test_fft_frame_mag_against_float64(units, n2, nz, caller):
    """fft_frame_mag<N2, NZ, FAST, SCALED, PRE> as K1 (|2X|, sqrt.approx) and the staged route (|X|/N2, sqrtf) run it,
    on random full-range PCM, square waves, DC, an impulse at every position < W and a cosine at every bin, at the
    reference window for every W of the shape: max_k |mag_k - ref_k| <= TAU[N2] * ||ref||_2 per frame, all-zero frames give
    exactly 0.

    Sensitivity: one tw_a entry or one tw_p entry off by a relative 1e-5 - a change the end-to-end tolerance cannot see -
    fails the same comparison."""
    import afe_loader
    afe = afe_loader.load()
    label, scaled, pres = CALLERS[caller]
    tw_a, tw_p = fft_tables(n2)
    rng = np.random.default_rng(n2 * 100 + nz)
    worst, worst_pa, worst_pp = 0.0, np.inf, np.inf
    for W in SHAPES[(n2, nz)]:
        window = afe.make_window(W)
        w2 = window2(window, n2)
        frames = fft_inputs(W, n2, rng)
        for pre in pres:
            ref = fft_reference(frames, W, window, n2, pre, scaled)
            mag = run_fft(units, n2, nz, caller, frames, w2, tw_a, tw_p, pre)
            assert np.isfinite(mag).all()
            assert np.all(mag[-1] == 0), "all-zero frame"
            e = normwise_error(mag, ref)
            worst = max(worst, float(e.max()))
            assert e.max() <= TAU[n2], f"W={W} pre={pre}: normwise error {e.max():.3g} > {TAU[n2]} (frame {e.argmax()})"
            # sensitivity: a twiddle of each table off by a relative 1e-5
            for table, k, sink in ((tw_a, 16 + 1, "a"), (tw_p, 1, "p")):
                bad = table.copy()
                bad[k] *= np.float32(1 + 1e-5)
                args = (bad, tw_p) if sink == "a" else (tw_a, bad)
                eb = normwise_error(run_fft(units, n2, nz, caller, frames, w2, *args, pre), ref).max()
                if sink == "a":
                    worst_pa = min(worst_pa, float(eb))
                else:
                    worst_pp = min(worst_pp, float(eb))
    print(f"fft_frame_mag<{n2},{nz}> {label}: worst normwise error {worst:.3g}; perturbed tw_a {worst_pa:.3g}, "
          f"tw_p {worst_pp:.3g} (tau {TAU[n2]})")
    assert worst_pa > TAU[n2] and worst_pp > TAU[n2]
