"""1024-point FFTs (windows of 513 to 1024 samples: 22.05, 24 and 32 kHz audio with 25 ms windows, and the 1024 / 256 TTS
mel front end) through the fused kernel K1 in the batch extractor: the 1024-point index map of tools/fft_model.py against
numpy, the filterbank tables, the in-register FFT fft_frame_mag<1024, ..> against a float64 rfft, the sixteen
instantiations k_fused_mfcc<1024, NZ, 8, KF, PRE> end to end against the CPU oracle and the float64 NumPy restatement,
every normalisation route and statistics scope, segments, the streaming object (which keeps its staged route at 1024
points), the C++ driver, and the refusals.

Pre-emphasis entries start at 300 Hz, as PRE_LOW in test_fused_instantiations does: pre-emphasis attenuates the lowest bands
by 25 dB or more, where an fp32 FFT is 3e-4 off in the log."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from common import afe, assert_close, compare, run_batch, synth_utterances, to_afe_params

sys.path.insert(0, os.path.join(ol.ROOT, "oracle"))
sys.path.insert(0, os.path.join(ol.ROOT, "tools"))
import fft_model  # noqa: E402
import oracle_np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
BIG = 1 << 22
PRE = 0.97
R22 = dict(sample_rate=22050.0, low_freq=64.0, high_freq=11025.0)
R24 = dict(sample_rate=24000.0, low_freq=64.0, high_freq=12000.0)
R32 = dict(sample_rate=32000.0, low_freq=64.0, high_freq=16000.0)
PRE_LOW = dict(low_freq=300.0)
LOGMEL = dict(ceps_len=0, want_c0=0, dyn="none")
MFCC13 = dict(ceps_len=13, want_c0=1, dyn="acc")   # 13 + c0, delta + acceleration: 42 columns

# (NZ, KF, PRE) -> parameters (CMN unless named). NZ = 13 for W <= 832 (26 lanes x 32), KF from the bank count:
# 3 up to 24 banks, 5 up to 40, 8 up to 64, 16 up to 128
KEYS1024 = {
    (13, 3, False): dict(R22, window_size=551, shift=220, num_banks=23, **MFCC13),
    (13, 5, False): dict(R24, window_size=600, shift=240, num_banks=40, **MFCC13, norm="cvn"),
    (13, 8, False): dict(R32, window_size=800, shift=320, num_banks=64, **MFCC13, norm="none"),
    (13, 16, False): dict(R32, window_size=832, shift=320, num_banks=80, **LOGMEL),
    (16, 3, False): dict(R32, window_size=833, shift=320, num_banks=24, ceps_len=12, want_c0=1, dyn="delta", norm="minmax"),
    (16, 5, False): dict(R22, window_size=1024, shift=256, num_banks=25, **MFCC13),
    (16, 8, False): dict(R22, window_size=1024, shift=256, num_banks=41, **LOGMEL, norm="none"),
    (16, 16, False): dict(R22, window_size=1024, shift=256, num_banks=128, **LOGMEL),
    (13, 3, True): dict(R22, **PRE_LOW, window_size=513, shift=220, num_banks=24, **MFCC13),
    (13, 5, True): dict(R24, **PRE_LOW, window_size=600, shift=240, num_banks=25, **LOGMEL),
    (13, 8, True): dict(R22, **PRE_LOW, window_size=551, shift=220, num_banks=64, **MFCC13, norm="cvn"),
    (13, 16, True): dict(R24, **PRE_LOW, window_size=600, shift=240, num_banks=65, **LOGMEL, norm="minmax"),
    (16, 3, True): dict(R32, **PRE_LOW, window_size=900, shift=320, num_banks=20, **MFCC13),
    (16, 5, True): dict(R32, **PRE_LOW, window_size=1024, shift=320, num_banks=40, **MFCC13, norm="none"),
    (16, 8, True): dict(R22, **PRE_LOW, window_size=1000, shift=256, num_banks=48, **LOGMEL),
    (16, 16, True): dict(R24, **PRE_LOW, window_size=1024, shift=240, num_banks=80, **LOGMEL, high_freq=8000.0),
}
KEYS = sorted(KEYS1024)


def key_id(k):
    return "k_fused_mfcc<1024,{},8,{},{}>".format(k[0], k[1], "true" if k[2] else "false")


def params_of(key):
    return ol.default_params(**dict(dict(norm="cmn"), **KEYS1024[key]))


def test_key_table_covers_every_new_instantiation():
    assert len(KEYS) == 16
    for nz, kf, pre in KEYS:
        p = params_of((nz, kf, pre))
        W, nb = p["window_size"], p["num_banks"]
        assert 513 <= W <= 1024
        assert (W <= 832) == (nz == 13)
        nfw = (nb + 7) // 8
        assert kf == (3 if nfw <= 3 else 5 if nfw <= 5 else 8 if nfw <= 8 else 16)
        assert ol.width_of(p) <= 128 and ol.cols_of(p) <= 128


# ---------------------------------------------------------------------------------------------- host only
def test_fft_model_1024_matches_numpy_rfft():
    """The lane / slot index maps of the 1024-point in-register FFT (tools/fft_model.py:rfft_model_1024) are an exact
    restatement of the real FFT: random, impulse and single-bin inputs against numpy.fft.rfft."""
    rng = np.random.default_rng(1024)
    xs = [rng.standard_normal(1024) for _ in range(4)]
    for m in (0, 1, 31, 32, 511, 512, 1023):
        x = np.zeros(1024)
        x[m] = 1.0
        xs.append(x)
    for k in (0, 1, 16, 255, 256, 257, 511, 512):
        xs.append(np.cos(2 * np.pi * k * np.arange(1024) / 1024))
    for x in xs:
        ref = np.fft.rfft(x)
        assert np.abs(fft_model.rfft_model_1024(x) - ref).max() <= 1e-10 * max(1.0, np.abs(ref).max())


def lib_filter_rows(p, alpha):
    """The library's filterbank as a [num_banks][bins] matrix (afe_build_filters: edges + the two interleaved weight rows)."""
    edges, filt = afe.build_filters(to_afe_params(p, BIG), alpha)
    filt = np.asarray(filt).reshape(2, -1)
    rows = np.zeros((p["num_banks"], 513))
    for b in range(p["num_banks"]):
        for j in range(edges[b], min(edges[b + 2], 513)):
            rows[b, j] = filt[b % 2][j]
    return np.asarray(edges), rows


@pytest.mark.parametrize("alpha", [1.0, 0.9, 1.1])
@pytest.mark.parametrize("key", KEYS, ids=key_id)
def test_filters_1024_match_numpy(key, alpha):
    """Host only: at 1024 points the edges equal the float64 restatement's, the weights agree to float32 rounding, and the
    all-zero filters are the same ones."""
    p = params_of(key)
    edges, rows = lib_filter_rows(p, alpha)
    _, want_edges, want = oracle_np.mel_tables(p["num_banks"], 1024, p["sample_rate"], p["low_freq"], p["high_freq"], alpha)
    np.testing.assert_array_equal(edges, want_edges)
    np.testing.assert_allclose(rows, want, atol=3e-5)
    np.testing.assert_array_equal(rows.max(1) == 0, want.max(1) == 0)


# ---------------------------------------------------------------------------------------------- FFT unit (device)
SRC = os.path.join(HERE, "cuda", "afe_units_fft1024.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# asr-featext-opencl_b200/Makefile: NVFLAGS, run from the repository root
NVFLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC,-Wall",
           "-I", os.path.join(ol.ROOT, "include"), "-I", os.path.join(ol.ROOT, "asr-featext-opencl_b200", "csrc")]


@pytest.fixture(scope="module")
def units_so(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("afe_units_fft1024") / "libafe_units_fft1024.so")
    r = subprocess.run([NVCC, *NVFLAGS, "-shared", "-o", so, SRC], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return so


@pytest.fixture(scope="module")
def units(units_so):
    L = C.CDLL(units_so)
    fp = C.POINTER(C.c_float)
    L.afe_units_fft1024_mag.restype = C.c_int
    L.afe_units_fft1024_mag.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_short), C.c_int, fp, fp, fp, C.c_float, fp]
    return L


def test_fft1024_harness_compiles(units_so):
    """CPU-only: the 1024-point harness compiles for sm_100a with the library's flags and exports its entry point."""
    C.CDLL(units_so).afe_units_fft1024_mag


def fft_tables():
    """FftTables::build(1024) (afe_batch.cu): the same double expressions, rounded to float."""
    lk = (np.arange(32)[:, None] * np.arange(16)[None, :]).astype(np.float64).ravel()
    ang = -2.0 * np.pi * lk / 512
    tw_a = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    ang = -2.0 * np.pi * np.arange(256, dtype=np.float64) / 1024
    tw_p = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    return tw_a, tw_p


def fft_inputs(W, rng):
    """Frames of 1024 int16 samples; samples from W on are random and must not leak through the zero window tail."""
    full = lambda: rng.integers(-32768, 32768, 1024).astype(np.int16)
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
    for half in (1, 5, 25, 64, 200):                                  # full-scale square waves
        add(np.where((n // half) % 2 == 0, 32767, -32768))
    add(np.full(W, 32767))                                            # DC
    add(np.full(W, -32768))
    for m in range(W):                                                # an impulse in every load slot (lane, n1)
        x = np.zeros(W, np.int16)
        x[m] = 32767 if m % 2 else -32768
        add(x)
    for k in range(513):                                              # a cosine at every bin: every real-split slot
        add(np.round(30000 * np.cos(2 * np.pi * k * n / 1024)))
    add(np.zeros(W, np.int16))                                        # zeros: exactly 0 (must stay the last frame)
    return np.stack(frames)


def fft_reference(frames, W, window, pre):
    """float64 |2X| of the float32 window times the PCM, pre-emphasis as oracle/oracle_np.py:mfcc defines it."""
    x = frames[:, :W].astype(np.float64)
    if pre:
        x = x - np.float64(np.float32(pre)) * np.concatenate([x[:, :1], x[:, :-1]], axis=1)
    fr = np.zeros((len(frames), 1024))
    fr[:, :W] = x * window.astype(np.float64)
    return 2.0 * np.abs(np.fft.rfft(fr, axis=1))


def run_fft(units, nz, with_pre, frames, w2, tw_a, tw_p, pre):
    frames = np.ascontiguousarray(frames, np.int16)
    mag = np.zeros((len(frames), 513), np.float32)
    ptr = lambda a: np.ascontiguousarray(a).ctypes.data_as(C.POINTER(C.c_float))
    rc = units.afe_units_fft1024_mag(nz, int(with_pre), frames.ctypes.data_as(C.POINTER(C.c_short)), len(frames), ptr(w2),
                                     ptr(tw_a), ptr(tw_p), float(pre), mag.ctypes.data_as(C.POINTER(C.c_float)))
    assert rc == 0, f"CUDA error {rc}"
    return mag


def normwise_error(mag, ref):
    """per frame max_k |mag_k - ref_k| / ||ref||_2 (frames with ref == 0 excluded)"""
    nrm = np.sqrt((ref * ref).sum(1))
    err = np.abs(mag.astype(np.float64) - ref).max(1)
    live = nrm > 0
    return err[live] / nrm[live]


SHAPES = {13: (513, 551, 600, 800, 832), 16: (833, 900, 1024)}
# max_k |mag_k - ref_k| <= TAU * ||ref||_2 per frame; the numbers behind it are in the docstring below
TAU = 3e-7


@pytest.mark.gpu
@pytest.mark.parametrize("with_pre", [False, True], ids=["k1", "k1pre"])
@pytest.mark.parametrize("nz", [13, 16])
def test_fft1024_frame_mag_against_float64(units, nz, with_pre):
    """fft_frame_mag<1024, NZ, true, false, PRE> as K1 runs it (|2X|, sqrt.approx), on random full-range PCM, square waves,
    DC, an impulse at every position < W and a cosine at every bin, at the reference window for every W of the shape:
    max_k |mag_k - ref_k| <= TAU * ||ref||_2 per frame; all-zero frames give exactly 0.

    Sensitivity: one tw_a entry or one tw_p entry off by a relative 1e-5 fails the same comparison. Measured on a B200
    (1000 W): worst error 2.07e-7 over the four instantiations (NZ = 16, no pre-emphasis); a perturbed tw_a entry gives at
    least 4.44e-7, a perturbed tw_p entry at least 3.02e-6. TAU = 3e-7 sits between them, 1.45x the worst error seen. The
    pruned instantiation gives the same bits as the unpruned one for every W <= 832."""
    import afe_loader
    afe_ = afe_loader.load()
    tw_a, tw_p = fft_tables()
    rng = np.random.default_rng(1000 + nz)
    worst, worst_pa, worst_pp = 0.0, np.inf, np.inf
    failures = []
    for W in SHAPES[nz]:
        window = afe_.make_window(W)
        w2 = np.zeros(1024, np.float32)
        w2[:W] = window
        frames = fft_inputs(W, rng)
        for pre in ((PRE,) if with_pre else (0.0,)):
            ref = fft_reference(frames, W, window, pre)
            mag = run_fft(units, nz, with_pre, frames, w2, tw_a, tw_p, pre)
            assert np.isfinite(mag).all()
            assert np.all(mag[-1] == 0), "all-zero frame"
            e = normwise_error(mag, ref)
            worst = max(worst, float(e.max()))
            if e.max() > TAU:
                failures.append(f"W={W} pre={pre}: normwise error {e.max():.3g} > {TAU} (frame {e.argmax()})")
            if nz == 13:
                np.testing.assert_array_equal(run_fft(units, 16, with_pre, frames, w2, tw_a, tw_p, pre), mag,
                                              err_msg=f"W={W}: pruned and unpruned FFTs differ")
            for table, k, sink in ((tw_a, 16 + 1, "a"), (tw_p, 1, "p")):
                bad = table.copy()
                bad[k] *= np.float32(1 + 1e-5)
                args = (bad, tw_p) if sink == "a" else (tw_a, bad)
                eb = float(normwise_error(run_fft(units, nz, with_pre, frames, w2, *args, pre), ref).max())
                if sink == "a":
                    worst_pa = min(worst_pa, eb)
                else:
                    worst_pp = min(worst_pp, eb)
    print(f"fft_frame_mag<1024,{nz}> pre={with_pre}: worst normwise error {worst:.3g}; perturbed tw_a {worst_pa:.3g}, "
          f"tw_p {worst_pp:.3g} (tau {TAU})")
    assert not failures, failures
    assert worst_pa > TAU and worst_pp > TAU


# ---------------------------------------------------------------------------------------------- end to end (device)
def ragged_utterances(p, seed):
    """8 utterances: exactly 2D+1 frames, 2D+2, a few rounds, and several tiles; odd sample remainders."""
    W, S = p["window_size"], p["shift"]
    D = (p["delta_l1"] if p["dyn"] else 0) + (p["delta_l2"] if p["dyn"] == ol.DYN["acc"] else 0)
    frames = [2 * D + 1, 2 * D + 2, 33, 100, 511, 530, 1200, 2100]
    rem = [0, 3, S - 1, 1, S // 2 + 1, 0, 7, S - 3]
    return [synth_utterances(1, W - S + S * t + r, seed=seed + i, sr=p["sample_rate"])[0]
            for i, (t, r) in enumerate(zip(frames, rem))]


def pack(utts, phase):
    """Concatenate with every start at 8k + phase samples (phase 0: the 16-byte alignment the TMA staging path needs)."""
    offs, pos, chunks = [], phase, [np.zeros(phase, np.int16)]
    for u in utts:
        offs.append(pos)
        chunks.append(u)
        pad = (-(pos + len(u) - phase)) % 8
        chunks.append(np.zeros(pad, np.int16))
        pos += len(u) + pad
    chunks.append(np.zeros(16, np.int16))
    return np.concatenate(chunks), np.array(offs, np.int64), np.array([len(u) for u in utts], np.int64)


def run(p, utts, flags, pre, phase=0, alpha=1.0):
    b = afe.BatchMfcc(to_afe_params(p, BIG), 0, flags=flags, preemphasis=pre, alpha=alpha)
    try:
        pcm, offs, lens = pack(utts, phase)
        b.plan(offs, lens)
        out = b.run_host(pcm)
        fo = b.frame_offsets
        return b.kernel_name, [out[fo[i]:fo[i + 1]] for i in range(len(utts))]
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key", KEYS, ids=key_id)
def test_fft1024_instantiation_end_to_end(oracle, key):
    """Ragged utterances through the named instantiation with AFE_BATCH_Q1_EXACT: against the CPU oracle without
    pre-emphasis, against oracle_np.mfcc(q1=True) with it; plain staging from misaligned starts is bitwise the TMA path
    (S % 8 != 0 stages plainly in both runs)."""
    p = params_of(key)
    pre = PRE if key[2] else 0.0
    utts = ragged_utterances(p, seed=10 * key[0] + key[1] + (1000 if key[2] else 0))
    name, got = run(p, utts, afe.BATCH_Q1_EXACT, pre)
    assert name == key_id(key)
    if key[2]:
        for i, (g, u) in enumerate(zip(got, utts)):
            w = oracle_np.mfcc(u, dict(p, preemphasis=pre), q1=True).astype(np.float32)
            compare(g, w, p, f"{name} utt {i} vs float64")
    else:
        want = oracle.extract(p, utts, sample_limit=BIG)[0]
        for i, (g, w) in enumerate(zip(got, want)):
            compare(g, w, p, f"{name} utt {i} vs oracle")
            compare(g, oracle_np.mfcc(utts[i], p, q1=True).astype(np.float32), p, f"{name} utt {i} vs float64")
    _, plain = run(p, utts, afe.BATCH_Q1_EXACT | afe.BATCH_NO_TMA, pre, phase=2)
    for i, (a, b) in enumerate(zip(got, plain)):
        np.testing.assert_array_equal(a, b, err_msg=f"{name} utt {i}: plain staging differs from TMA")


# the four arms of tools/fft1024_bench.py and a few more
SETS = {
    "mfcc22k": dict(R22, window_size=551, shift=220, num_banks=40, **MFCC13),
    "logmel80_24k": dict(R24, window_size=600, shift=240, num_banks=80, **LOGMEL),
    "tts80_22k": dict(R22, window_size=1024, shift=256, num_banks=80, **LOGMEL, high_freq=8000.0),
    "mfcc32k": dict(R32, window_size=800, shift=320, num_banks=64, **MFCC13),
    "mfcc32k_1024": dict(R32, window_size=1024, shift=320, num_banks=30, ceps_len=15, want_c0=1, dyn="none"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["none", "cmn", "cvn", "minmax"])
@pytest.mark.parametrize("name", sorted(SETS))
def test_fft1024_normalisations_and_vtln(oracle, name, norm):
    """Every normalisation at alpha 1.0, 0.9 and 1.1 (VTLN-warped banks fill the weight list differently): reference-block
    scope against the CPU oracle, utterance scope against the float64 restatement with statistics over all rows."""
    p = ol.default_params(**dict(SETS[name], norm=norm))
    utts = synth_utterances(6, 120000, seed=61, sr=p["sample_rate"], ragged=True)
    for alpha in (1.0, 0.9, 1.1):
        q = dict(p, alpha=alpha)
        got = run_batch(q, utts, flags=afe.BATCH_Q1_EXACT)
        want = oracle.extract(q, utts, sample_limit=BIG)[0]
        for i in range(len(utts)):
            compare(got[i], want[i], q, f"{name} utt {i} alpha {alpha}")
    got = run_batch(p, utts, stats_scope=afe.STATS_UTTERANCE)
    for i, u in enumerate(utts):
        T = ol.total_frames(len(u), p)
        compare(got[i], oracle_np.mfcc(u, p, stats_rows=T).astype(np.float32), p, f"{name} utt {i} utterance scope")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mfcc22k", "logmel80_24k", "tts80_22k", "mfcc32k"])
@pytest.mark.parametrize("norm", ["cmn", "cvn"])
def test_fft1024_normalisation_routes_bitwise_equal(name, norm):
    """Cluster (MFCC with the default regression), ticket (AFE_BATCH_NO_CLUSTER) and role schemes (an utterance of more
    than 8 tiles) and K2 + K3 (AFE_BATCH_UNFUSED_NORM) give the same bits."""
    p = ol.default_params(**dict(SETS[name], norm=norm))
    sr = int(p["sample_rate"])
    short = synth_utterances(12, 4 * sr, seed=71, sr=sr, ragged=True)
    long_ = synth_utterances(3, 12 * sr, seed=72, sr=sr)
    very_long = synth_utterances(1, 60 * sr, seed=73, sr=sr)       # > 8 tiles of <= 512 frames
    for utts in (short + long_, short + very_long):
        a = run_batch(p, utts)
        b = run_batch(p, utts, flags=afe.BATCH_NO_CLUSTER)
        c = run_batch(p, utts, flags=afe.BATCH_UNFUSED_NORM)
        for i in range(len(utts)):
            np.testing.assert_array_equal(a[i], b[i])
            np.testing.assert_array_equal(a[i], c[i])


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_fft1024_corpus_scope(oracle, norm):
    """extract -> corpus_stats -> set_corpus_stats -> normalize: the raw rows equal the oracle's and the normalised ones the
    NumPy restatement of normalizercpu.cpp over the whole corpus."""
    p = ol.default_params(**dict(SETS["tts80_22k"], norm=norm))
    utts = synth_utterances(12, 100000, seed=81, sr=22050.0, ragged=True)
    w = ol.width_of(p)
    b = afe.BatchMfcc(to_afe_params(p, BIG), 0, stats_scope=afe.STATS_CORPUS)
    pcm, offs, lens = afe.pack_utterances(utts)
    total = b.plan(offs, lens)
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * w * 4)
    try:
        b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
        ptr, n = b.corpus_stats()
        b.synchronize()
        stats = np.zeros(n, np.float64)
        afe._check(afe.lib().afe_memcpy_d2h(0, stats.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), stats.nbytes))
        raw = d_out.download((total, w), np.float32)
        b.set_corpus_stats(stats)
        b.normalize_device(d_out.ptr.value)
        b.synchronize()
        got = d_out.download((total, w), np.float32)
        fo = b.frame_offsets
    finally:
        b.close(); d_pcm.free(); d_out.free()
    want_raw = oracle.extract(dict(p, norm=ol.NORM["none"]), utts, sample_limit=BIG)[0]
    for i in range(len(utts)):
        assert_close(raw[fo[i]:fo[i + 1]], want_raw[i], dict(p, norm=ol.NORM["none"]), f"raw utt {i}")
    x = raw.astype(np.float64)
    mu = x.mean(0)
    if norm == "cmn":
        want = x - mu
    elif norm == "cvn":
        want = (x - mu) * np.sqrt((len(x) - 1) / ((x * x).sum(0) - x.sum(0) ** 2 / len(x)))
    else:
        want = (x - mu) / np.maximum(np.abs(x.min(0) - mu), np.abs(x.max(0) - mu))
    np.testing.assert_allclose(got, want, atol=2e-5 if norm != "cvn" else 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mfcc22k", "tts80_22k"])
def test_fft1024_time_sharded_segments_equal_whole_stream(name):
    """One stream cut by time into 3 segments (afe_batch_plan_segments, D frames of context per side): bitwise the rows
    of the whole stream without normalisation."""
    p = ol.default_params(**dict(SETS[name], norm="none"))
    W, S, w = p["window_size"], p["shift"], ol.width_of(p)
    D = 6 if p["dyn"] == ol.DYN["acc"] else 0
    x = synth_utterances(1, 22050 * 40 + 77, seed=91, sr=22050.0)[0]
    whole = run_batch(p, [x], stats_scope=afe.STATS_UTTERANCE)[0]
    sh = afe.shard_stream(len(x), W, S, D, 3)
    parts = []
    for r in range(3):
        b = afe.BatchMfcc(to_afe_params(p, BIG), 0, stats_scope=afe.STATS_CORPUS)
        seg = np.ascontiguousarray(x[sh["sample_begin"][r]:sh["sample_begin"][r] + sh["sample_count"][r]])
        pcm, offs, lens = afe.pack_utterances([seg])
        total = b.plan_segments(offs, lens, [sh["local_first"][r]], [sh["count"][r]])
        d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
        d_out = afe.DeviceBuffer(total * w * 4)
        try:
            b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
            b.synchronize()
            parts.append(d_out.download((total, w), np.float32))
        finally:
            b.close(); d_pcm.free(); d_out.free()
    np.testing.assert_array_equal(np.concatenate(parts), whole)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mfcc22k", "logmel80_24k", "tts80_22k"])
def test_fft1024_batch_against_streaming_object(name):
    """The streaming object keeps its staged kernels at 1024 points (uses_fused_kernel is false); the batch extractor's
    K1 output agrees with it within the stated tolerance."""
    p = ol.default_params(**SETS[name])
    m = afe.MfccCuda(to_afe_params(p, BIG))
    assert not m.uses_fused_kernel
    m.close()
    x = synth_utterances(1, int(p["sample_rate"]) * 20 + 123, seed=97, sr=p["sample_rate"])[0]
    staged = afe.extract_stream(to_afe_params(p, BIG), x)
    batch = run_batch(p, [x], flags=afe.BATCH_Q1_EXACT)[0]
    compare(batch, staged, p, f"{name}: batch vs streaming object")


@pytest.mark.gpu
def test_fft1024_driver_batch_mode_at_22k(tmp_path):
    """afe_extract --sample-rate 22050 --window-size 25 --shift 10 (W = 551, S = 220): --batch 1 runs K1 and agrees with
    the driver's streaming mode on a generated WAV."""
    import struct
    exe = os.path.join(ol.ROOT, "asr-featext-opencl_b200", "afe_extract")
    if not os.path.exists(exe):
        pytest.skip("afe_extract not built")
    pcm = synth_utterances(1, 22050 * 6 + 31, seed=5, sr=22050.0)[0]
    data = np.ascontiguousarray(pcm, "<i2").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, 22050, 44100, 2, 16)
    wav = str(tmp_path / "a22k.wav")
    open(wav, "wb").write(hdr + b"data" + struct.pack("<I", len(data)) + data)
    opts = ["--sample-rate", "22050", "--window-size", "25", "--shift", "10", "--banks", "40", "--high-freq", "11025"]
    outs = {}
    for mode, extra in (("batch", ["--batch", "1"]), ("stream", [])):
        txt = str(tmp_path / f"{mode}.txt")
        r = subprocess.run([exe] + opts + extra + [wav, txt], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                           timeout=120)
        assert r.returncode == 0, r.stderr
        lines = open(txt).read().splitlines()
        outs[mode] = (lines, np.array([[float(v) for v in l.strip("| ").split(" | ")] for l in lines]))
    (bl, b), (sl, s) = outs["batch"], outs["stream"]
    assert len(bl) == len(sl) == (len(pcm) - (551 - 220)) // 220
    assert [l.split(" | ")[0] for l in bl] == [l.split(" | ")[0] for l in sl]
    assert np.abs(b[:, 1:] - s[:, 1:]).max() < 5e-4


# Parameter sets whose cepstra tile fills one CTA's shared memory to the last 256 bytes the budget leaves for K1's static
# shared variables: with the whole 227 KB opt-in limit as the dynamic budget their launches were refused by the driver
EDGE = {
    "logmel64_22k_s176": dict(R22, window_size=1024, shift=176, num_banks=64, **LOGMEL, norm="none"),
    "logmel60_delta_32k_s314": dict(R32, window_size=800, shift=314, num_banks=60, ceps_len=0, want_c0=0, dyn="delta"),
    "logmel50_24k_s260": dict(R24, window_size=600, shift=260, num_banks=50, **LOGMEL),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EDGE))
def test_fft1024_largest_tiles_fit_one_cta(oracle, name):
    """The largest cepstra tiles the 1024-point layout allows launch and match the CPU oracle."""
    p = ol.default_params(**dict(dict(norm="cmn"), **EDGE[name]))
    utts = synth_utterances(6, 200000, seed=41, sr=p["sample_rate"], ragged=True)
    got = run_batch(p, utts, flags=afe.BATCH_Q1_EXACT)
    want = oracle.extract(p, utts, sample_limit=BIG)[0]
    for i in range(len(utts)):
        compare(got[i], want[i], p, f"{name} utt {i}")


@pytest.mark.gpu
def test_fft1024_refusals_name_the_limit():
    """1025-sample windows (2048-point FFTs) and 17 cepstral columns at 1024 points stay outside K1: afe_batch_create
    refuses them, naming the limit."""
    with pytest.raises(afe.AfeError, match="256/512/1024-point FFTs"):
        afe.BatchMfcc(afe.make_params(sample_rate=32000.0, window_size=1025, shift=320, high_freq=16000.0), 0)
    with pytest.raises(afe.AfeError, match="ceps_len \\+ c0 <= 16 with 1024-point FFTs"):
        afe.BatchMfcc(afe.make_params(sample_rate=22050.0, window_size=551, shift=220, high_freq=11025.0, num_banks=40,
                                      ceps_len=16, want_c0=1), 0)
