"""Filterbanks of 65 to 128 banks (80- and 128-band log-mel, MFCC from wide banks) through the fused kernel K1: the eight
KF = 16 instantiations k_fused_mfcc<N2, NZ, 8, 16, PRE>, every normalisation route, corpus scope, time-sharded segments and
the streaming object, against the CPU oracle and the float64 NumPy restatement; and the parameter sets K1 still refuses.

Low-frequency edges: 64 Hz (the reference's default) unless pre-emphasis is on. Pre-emphasis attenuates the lowest bands
by 25 dB or more, where an fp32 FFT is 3e-4 off in the log (see PRE_LOW in test_fused_instantiations): those entries start
at 300 Hz. Their banks also have no filter whose float32 weights differ from the float64 ones by more than 2e-5 of the
filter's sum, so the float64 comparison measures the kernel and not the weight tables."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import oracle_lib as ol
from common import afe, assert_close, compare, run_batch, synth_utterances, to_afe_params

sys.path.insert(0, os.path.join(ol.ROOT, "oracle"))
import oracle_np  # noqa: E402

BIG = 1 << 22
PRE = 0.97
K16 = dict(sample_rate=16000.0, low_freq=64.0, high_freq=8000.0, shift=160)
K8 = dict(sample_rate=8000.0, low_freq=64.0, high_freq=4000.0, shift=80)
PRE_LOW = dict(low_freq=300.0)
LOGMEL = dict(ceps_len=0, want_c0=0, dyn="none")
MFCC13 = dict(ceps_len=13, want_c0=1, dyn="acc")   # 13 + c0, delta + acceleration: 42 columns

# (N2, NZ, 16, PRE) -> parameters (CMN unless named)
WIDE = {
    (512, 13, 16, False): dict(K16, window_size=400, num_banks=80, **LOGMEL),
    (512, 16, 16, False): dict(K16, window_size=512, num_banks=128, **LOGMEL),      # zero-width filters from 64 Hz
    (256, 13, 16, False): dict(K8, window_size=200, num_banks=80, **MFCC13, norm="cvn"),
    (256, 16, 16, False): dict(K8, window_size=256, num_banks=96, **LOGMEL, norm="none"),
    (512, 13, 16, True): dict(K16, **PRE_LOW, window_size=416, num_banks=80, **LOGMEL),
    (512, 16, 16, True): dict(K16, **PRE_LOW, window_size=480, num_banks=80, **MFCC13),
    (256, 13, 16, True): dict(K8, **PRE_LOW, window_size=208, num_banks=65, **MFCC13, norm="minmax"),
    (256, 16, 16, True): dict(K8, **PRE_LOW, window_size=209, num_banks=65, **LOGMEL),
}
KEYS = sorted(WIDE)


def key_id(k):
    return "k_fused_mfcc<{},{},8,{},{}>".format(k[0], k[1], k[2], "true" if k[3] else "false")


def params_of(key):
    return ol.default_params(**dict(dict(norm="cmn"), **WIDE[key]))


def lib_filter_rows(p, alpha):
    """The library's filterbank as a [num_banks][bins] matrix (afe_build_filters: edges + the two interleaved weight rows)."""
    edges, filt = afe.build_filters(to_afe_params(p, BIG), alpha)
    n2 = 1 << (p["window_size"] - 1).bit_length()
    filt = np.asarray(filt).reshape(2, -1)
    rows = np.zeros((p["num_banks"], n2 // 2 + 1))
    for b in range(p["num_banks"]):
        for j in range(edges[b], min(edges[b + 2], n2 // 2 + 1)):
            rows[b, j] = filt[b % 2][j]
    return np.asarray(edges), rows


def test_wide_table_covers_every_new_key():
    assert len(KEYS) == 8
    for n2, nz, kf, pre in KEYS:
        p = params_of((n2, nz, kf, pre))
        W = p["window_size"]
        assert 1 << (W - 1).bit_length() == n2
        assert (W <= 26 * n2 // 32) == (nz == 13)
        assert 8 < (p["num_banks"] + 7) // 8 <= 16
        assert ol.width_of(p) <= 128


BANKS = {"80@16k": dict(K16, num_banks=80, window_size=400), "128@16k": dict(K16, num_banks=128, window_size=512),
         "80@8k": dict(K8, num_banks=80, window_size=200), "128@8k": dict(K8, num_banks=128, window_size=256)}


@pytest.mark.parametrize("alpha", [1.0, 0.9, 1.1])
@pytest.mark.parametrize("bank", sorted(BANKS))
def test_wide_filters_match_numpy(bank, alpha):
    """Host only: edges equal the float64 restatement's, weights agree to float32 rounding, and the filters whose weights
    are all zero (narrow low bands of the 128-band banks) are the same ones, so their energy takes the 1e-30 log clamp in
    both."""
    p = ol.default_params(**BANKS[bank])
    edges, rows = lib_filter_rows(p, alpha)
    n2 = 1 << (p["window_size"] - 1).bit_length()
    _, want_edges, want = oracle_np.mel_tables(p["num_banks"], n2, p["sample_rate"], p["low_freq"], p["high_freq"], alpha)
    np.testing.assert_array_equal(edges, want_edges)
    np.testing.assert_allclose(rows, want, atol=3e-5)
    np.testing.assert_array_equal(rows.max(1) == 0, want.max(1) == 0)
    if bank == "128@16k" and alpha == 1.0:
        assert (rows.max(1) == 0).any()


def test_wide_banks_carry_zero_width_filters_where_the_gpu_tests_expect_them():
    """The GPU parameter sets below include the zero-width filter case (128 banks from 64 Hz at 16 kHz)."""
    _, rows = lib_filter_rows(params_of((512, 16, 16, False)), 1.0)
    assert (rows.max(1) == 0).sum() >= 1


# ---------------------------------------------------------------------------------------------- GPU
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


def run(p, utts, flags, pre, phase=0):
    b = afe.BatchMfcc(to_afe_params(p, BIG), 0, flags=flags, preemphasis=pre)
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
def test_wide_instantiation_end_to_end(oracle, key):
    """Ragged utterances through the named KF = 16 instantiation with AFE_BATCH_Q1_EXACT: against the CPU oracle without
    pre-emphasis, against oracle_np.mfcc(q1=True) with it; plain staging from misaligned starts is bitwise the TMA path."""
    p = params_of(key)
    pre = PRE if key[3] else 0.0
    utts = ragged_utterances(p, seed=key[0] + 10 * key[1] + (1000 if key[3] else 0))
    name, got = run(p, utts, afe.BATCH_Q1_EXACT, pre)
    assert name == key_id(key)
    if key[3]:
        for i, (g, u) in enumerate(zip(got, utts)):
            w = oracle_np.mfcc(u, dict(p, preemphasis=pre), q1=True).astype(np.float32)
            compare(g, w, p, f"{name} utt {i} vs float64")
    else:
        want = oracle.extract(p, utts, sample_limit=BIG)[0]
        for i, (g, w) in enumerate(zip(got, want)):
            compare(g, w, p, f"{name} utt {i} vs oracle")
    _, plain = run(p, utts, afe.BATCH_Q1_EXACT | afe.BATCH_NO_TMA, pre, phase=2)
    for i, (a, b) in enumerate(zip(got, plain)):
        np.testing.assert_array_equal(a, b, err_msg=f"{name} utt {i}: plain staging differs from TMA")


SETS = {
    "logmel80-none": dict(num_banks=80, **LOGMEL, norm="none"),
    "logmel80-cmn": dict(num_banks=80, **LOGMEL, norm="cmn"),
    "logmel80-cvn": dict(num_banks=80, **LOGMEL, norm="cvn"),
    "logmel80-minmax": dict(num_banks=80, **LOGMEL, norm="minmax"),
    "logmel128-cmn": dict(num_banks=128, **LOGMEL, norm="cmn"),
    "logmel128-none-zero-width": dict(num_banks=128, window_size=512, **LOGMEL, norm="none"),
    "mfcc13-80-acc": dict(num_banks=80, **MFCC13, norm="cmn"),
    "logmel80-8k": dict(K8, window_size=200, num_banks=80, **LOGMEL, norm="cmn"),
    "mfcc13-80-8k": dict(K8, window_size=200, num_banks=80, **MFCC13, norm="cvn"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SETS))
def test_wide_parameter_sets_match_oracle(oracle, name):
    """80- and 128-band log-mel under every normalisation, 13 + c0 from 80 banks with deltas, 80 banks at 8 kHz / 256,
    each at alpha 1.0, 0.9 and 1.1 (VTLN-warped banks fill the constant-bank weight list differently)."""
    p = ol.default_params(**SETS[name])
    utts = synth_utterances(10, 90000, seed=61, sr=p["sample_rate"], ragged=True)
    for alpha in (1.0, 0.9, 1.1):
        q = dict(p, alpha=alpha)
        got = run_batch(q, utts, flags=afe.BATCH_Q1_EXACT)
        want = oracle.extract(q, utts, sample_limit=BIG)[0]
        for i in range(len(utts)):
            compare(got[i], want[i], q, f"{name} utt {i} alpha {alpha}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mfcc13-80-acc", "logmel80-cmn", "logmel128-cvn", "logmel80-minmax"])
def test_wide_normalisation_routes_bitwise_equal(name):
    """Cluster (MFCC from 80 banks, default regression), ticket and role schemes (log-mel: the role scheme from an utterance
    of more than 8 tiles) and K2 + K3 (AFE_BATCH_UNFUSED_NORM) give the same bits."""
    p = ol.default_params(**(SETS[name] if name in SETS else dict(num_banks=128, **LOGMEL, norm="cvn")))
    short = synth_utterances(12, 60000, seed=71, ragged=True)
    long_ = synth_utterances(3, 200000, seed=72)
    very_long = synth_utterances(1, 900000, seed=73)        # 5623 frames: > 8 tiles of <= 512 frames
    for utts in (short + long_, short + very_long):
        a = run_batch(p, utts)
        b = run_batch(p, utts, flags=afe.BATCH_NO_CLUSTER)
        c = run_batch(p, utts, flags=afe.BATCH_UNFUSED_NORM)
        for i in range(len(utts)):
            np.testing.assert_array_equal(a[i], b[i])
            np.testing.assert_array_equal(a[i], c[i])


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_wide_corpus_scope(oracle, norm):
    """extract -> corpus_stats -> set_corpus_stats (the record as the all-reduce would return it) -> normalize: equals the
    NumPy restatement of normalizercpu.cpp over the whole corpus, and the raw rows equal the oracle's."""
    p = ol.default_params(num_banks=80, **LOGMEL, norm=norm)
    utts = synth_utterances(16, 70000, seed=81, ragged=True)
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
def test_wide_time_sharded_segments_equal_whole_stream():
    """One 80-band log-mel stream cut by time into 3 segments (afe_batch_plan_segments): bitwise the rows of the whole
    stream without normalisation."""
    p = ol.default_params(num_banks=80, **LOGMEL, norm="none")
    x = synth_utterances(1, 16000 * 40 + 77, seed=91)[0]
    whole = run_batch(p, [x], stats_scope=afe.STATS_UTTERANCE)[0]
    sh = afe.shard_stream(len(x), 400, 160, 0, 3)
    parts = []
    for r in range(3):
        b = afe.BatchMfcc(to_afe_params(p, BIG), 0, stats_scope=afe.STATS_CORPUS)
        seg = np.ascontiguousarray(x[sh["sample_begin"][r]:sh["sample_begin"][r] + sh["sample_count"][r]])
        pcm, offs, lens = afe.pack_utterances([seg])
        total = b.plan_segments(offs, lens, [sh["local_first"][r]], [sh["count"][r]])
        d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
        d_out = afe.DeviceBuffer(total * 80 * 4)
        try:
            b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
            b.synchronize()
            parts.append(d_out.download((total, 80), np.float32))
        finally:
            b.close(); d_pcm.free(); d_out.free()
    np.testing.assert_array_equal(np.concatenate(parts), whole)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["logmel80-cmn", "logmel80-none", "mfcc13-80-acc", "logmel128-cmn"])
def test_wide_streaming_object(oracle, name):
    """The streaming object runs wide banks on K1 (one launch per block): blocks of 16 000 / 100 000 / 330 000 samples and
    the whole file against the reference fed the same blocks; the staged route (AFE_OPT_STAGED_KERNELS) stays within the
    same tolerance."""
    p = ol.default_params(**SETS[name])
    m = afe.MfccCuda(to_afe_params(p, 16000))
    assert m.uses_fused_kernel
    m.close()
    x = synth_utterances(1, 16000 * 30 + 123, seed=97)[0]
    for limit in (16000, 100000, 330000, 1 << 20):
        got = afe.extract_stream(to_afe_params(p, limit), x)
        want = oracle.extract(p, [x], sample_limit=limit)[0][0]
        compare(got, want, p, f"{name} limit={limit}")
    staged = afe.extract_stream(to_afe_params(p, 100000), x, staged=True)
    want = oracle.extract(p, [x], sample_limit=100000)[0][0]
    compare(staged, want, p, f"{name} staged")


@pytest.mark.gpu
def test_wide_refusals_name_the_limit():
    """129 banks, and 80-band log-mel with deltas (160 columns), stay outside K1: afe_batch_create refuses them."""
    with pytest.raises(afe.AfeError, match="num_banks <= 128"):
        afe.BatchMfcc(afe.make_params(num_banks=129, ceps_len=12), 0)
    with pytest.raises(afe.AfeError, match="output width <= 128"):
        afe.BatchMfcc(afe.make_params(num_banks=80, ceps_len=0, want_c0=0, dyn=1), 0)
    m = afe.MfccCuda(afe.make_params(input_buffer_size=BIG, num_banks=129, ceps_len=12))
    assert not m.uses_fused_kernel
    m.close()
