"""MFCC with 17 to 48 cepstral columns (ceps_len + c0; 40-coefficient high-resolution MFCC, speaker-ID front ends) through
the fused kernel K1: the sixteen wide-DCT instantiations k_fused_mfcc<N2, NZ, 8, KF, PRE, 48>, every normalisation route,
corpus scope, time-sharded segments and the streaming object, against the CPU oracle and the float64 NumPy restatement;
and the parameter sets K1 still refuses.

Pre-emphasis entries start their banks at 300 Hz, for the reason given in test_fused_instantiations (PRE_LOW)."""
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


def mf(ceps, c0, dyn):
    return dict(ceps_len=ceps, want_c0=c0, dyn=dyn)


# (N2, NZ, KF, PRE) -> parameters (CMN unless named). KF = 5 serves up to 40 banks, KF = 8 41..64 banks. No CVN without
# deltas here: the ragged set's first utterance is then one frame, whose CVN scale is 0/0 in float64 but, from float
# products, finite in the reference and the kernel (CVN without deltas: SETS, against the reference).
WIDE = {
    (512, 13, 5, False): dict(K16, window_size=400, num_banks=40, **mf(39, 1, "none")),
    (512, 13, 8, False): dict(K16, window_size=401, num_banks=64, **mf(47, 1, "none")),
    (512, 16, 5, False): dict(K16, window_size=512, num_banks=23, **mf(20, 1, "acc"), norm="cvn"),
    (512, 16, 8, False): dict(K16, window_size=480, num_banks=48, **mf(41, 1, "acc")),
    (256, 13, 5, False): dict(K8, window_size=200, num_banks=30, **mf(29, 1, "delta"), norm="minmax"),
    (256, 13, 8, False): dict(K8, window_size=129, num_banks=41, **mf(40, 0, "none"), norm="none"),
    (256, 16, 5, False): dict(K8, window_size=256, num_banks=40, **mf(24, 1, "acc")),
    (256, 16, 8, False): dict(K8, window_size=209, num_banks=41, **mf(16, 1, "acc")),
    (512, 13, 5, True): dict(K16, **PRE_LOW, window_size=416, num_banks=40, **mf(39, 1, "none")),
    (512, 13, 8, True): dict(K16, **PRE_LOW, window_size=400, num_banks=56, **mf(30, 0, "delta")),
    (512, 16, 5, True): dict(K16, **PRE_LOW, window_size=417, num_banks=36, **mf(19, 1, "acc"), norm="minmax"),
    (512, 16, 8, True): dict(K16, **PRE_LOW, window_size=512, num_banks=64, **mf(40, 1, "none")),
    (256, 13, 5, True): dict(K8, **PRE_LOW, window_size=208, num_banks=24, **mf(20, 1, "acc")),
    (256, 13, 8, True): dict(K8, **PRE_LOW, window_size=200, num_banks=41, **mf(30, 1, "delta")),
    (256, 16, 5, True): dict(K8, **PRE_LOW, window_size=209, num_banks=40, **mf(39, 1, "none")),
    (256, 16, 8, True): dict(K8, **PRE_LOW, window_size=256, num_banks=41, **mf(41, 1, "none")),
}
KEYS = sorted(WIDE)


def key_id(k):
    return "k_fused_mfcc<{},{},8,{},{},48>".format(k[0], k[1], k[2], "true" if k[3] else "false")


def params_of(key):
    return ol.default_params(**dict(dict(norm="cmn"), **WIDE[key]))


def test_wide_cepstra_table_covers_every_new_key():
    assert len(KEYS) == 16 == len({key_id(k) for k in KEYS})
    for n2, nz, kf, pre in KEYS:
        p = params_of((n2, nz, kf, pre))
        W = p["window_size"]
        assert 1 << (W - 1).bit_length() == n2
        assert (W <= 26 * n2 // 32) == (nz == 13)
        assert (5 if (p["num_banks"] + 7) // 8 <= 5 else 8) == kf and p["num_banks"] <= 64
        assert 16 < ol.cols_of(p) <= 48
        assert ol.width_of(p) <= 128


@pytest.mark.parametrize("key", KEYS, ids=key_id)
def test_wide_cepstra_filters_match_numpy(key):
    """Host only: the filter edges are strictly increasing and equal the float64 restatement's."""
    p = params_of(key)
    edges, _ = afe.build_filters(to_afe_params(p, BIG))
    assert np.all(np.diff(edges) > 0), edges
    _, want, _ = oracle_np.mel_tables(p["num_banks"], key[0], p["sample_rate"], p["low_freq"], p["high_freq"])
    np.testing.assert_array_equal(edges, want)


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
        return b.kernel_name, b.num_tiles, [out[fo[i]:fo[i + 1]] for i in range(len(utts))]
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key", KEYS, ids=key_id)
def test_wide_cepstra_instantiation_end_to_end(oracle, key):
    """Ragged utterances through the named wide-DCT instantiation with AFE_BATCH_Q1_EXACT: against the CPU oracle and
    oracle_np.mfcc(q1=True) without pre-emphasis, against the latter only with it; plain staging from misaligned starts
    is bitwise the TMA path."""
    p = params_of(key)
    pre = PRE if key[3] else 0.0
    utts = ragged_utterances(p, seed=key[0] + 10 * key[1] + key[2] + (1000 if key[3] else 0))
    name, ntiles, got = run(p, utts, afe.BATCH_Q1_EXACT, pre)
    assert name == key_id(key)
    assert ntiles > len(utts)  # the longest utterances take several tiles
    for i, (g, u) in enumerate(zip(got, utts)):
        w = oracle_np.mfcc(u, dict(p, preemphasis=pre), q1=True).astype(np.float32)
        compare(g, w, p, f"{name} utt {i} vs float64")
    if not key[3]:
        want = oracle.extract(p, utts, sample_limit=BIG)[0]
        for i, (g, w) in enumerate(zip(got, want)):
            compare(g, w, p, f"{name} utt {i} vs oracle")
    _, _, plain = run(p, utts, afe.BATCH_Q1_EXACT | afe.BATCH_NO_TMA, pre, phase=2)
    for i, (a, b) in enumerate(zip(got, plain)):
        np.testing.assert_array_equal(a, b, err_msg=f"{name} utt {i}: plain staging differs from TMA")


HIRES = dict(num_banks=40, **mf(39, 1, "none"))
SETS = {
    "hires39-none": dict(HIRES, norm="none"),
    "hires39-cmn": dict(HIRES, norm="cmn"),
    "hires39-cvn": dict(HIRES, norm="cvn"),
    "hires39-minmax": dict(HIRES, norm="minmax"),
    "hires40-none": dict(num_banks=40, **mf(40, 1, "none"), norm="none"),
    "hires40-cmn": dict(num_banks=40, **mf(40, 1, "none"), norm="cmn"),
    "hires40-cvn": dict(num_banks=40, **mf(40, 1, "none"), norm="cvn"),
    "hires40-minmax": dict(num_banks=40, **mf(40, 1, "none"), norm="minmax"),
    "mfcc20-acc": dict(num_banks=40, **mf(20, 1, "acc"), norm="cvn"),
    "ceps30-delta": dict(num_banks=40, **mf(30, 0, "delta"), norm="cmn"),
    "ceps41-acc": dict(num_banks=48, **mf(41, 1, "acc"), norm="cmn"),
    "ceps47-64": dict(num_banks=64, **mf(47, 1, "none"), norm="cmn"),
    "mfcc24-8k": dict(K8, window_size=200, num_banks=40, **mf(24, 1, "acc"), norm="cmn"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SETS))
def test_wide_cepstra_parameter_sets_match_oracle(oracle, name):
    """High-resolution MFCC under every normalisation, 20 + c0 with deltas and delta-deltas, 30 cepstra with deltas,
    41 + c0 with both (126 columns), 47 + c0 from 64 banks, 8 kHz with a 256-point FFT; each at alpha 1.0, 0.9 and 1.1."""
    p = ol.default_params(**SETS[name])
    utts = synth_utterances(10, 90000, seed=62, sr=p["sample_rate"], ragged=True)
    for alpha in (1.0, 0.9, 1.1):
        q = dict(p, alpha=alpha)
        got = run_batch(q, utts, flags=afe.BATCH_Q1_EXACT)
        want = oracle.extract(q, utts, sample_limit=BIG)[0]
        for i in range(len(utts)):
            compare(got[i], want[i], q, f"{name} utt {i} alpha {alpha}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mfcc20-acc", "ceps41-acc", "hires40-cmn", "hires39-minmax", "ceps30-delta"])
def test_wide_cepstra_normalisation_routes_bitwise_equal(name):
    """Cluster (default regression: utterances of 1 to 4 tiles), ticket (AFE_BATCH_NO_CLUSTER), role scheme (an utterance
    of more than 8 tiles) and K2 + K3 (AFE_BATCH_UNFUSED_NORM) give the same bits."""
    p = ol.default_params(**SETS[name])
    short = synth_utterances(12, 60000, seed=71, ragged=True)
    long_ = synth_utterances(3, 200000, seed=72)
    very_long = synth_utterances(1, 900000, seed=73)        # 5623 frames: more than 8 tiles of <= 512 frames
    for utts in (short + long_, short + very_long):
        a = run_batch(p, utts)
        b = run_batch(p, utts, flags=afe.BATCH_NO_CLUSTER)
        c = run_batch(p, utts, flags=afe.BATCH_UNFUSED_NORM)
        for i in range(len(utts)):
            np.testing.assert_array_equal(a[i], b[i])
            np.testing.assert_array_equal(a[i], c[i])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hires40-cvn", "mfcc20-acc", "hires39-minmax"])
def test_wide_cepstra_corpus_scope(oracle, name):
    """extract -> corpus_stats -> set_corpus_stats (the record as the all-reduce would return it) -> normalize: equals the
    NumPy restatement of normalizercpu.cpp over the whole corpus, and the raw rows equal the oracle's."""
    p = ol.default_params(**SETS[name])
    norm = {v: k for k, v in ol.NORM.items()}[p["norm"]]
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
    # without AFE_BATCH_Q1_EXACT the last D rows keep their own statics, where the reference repeats earlier ones (Q1)
    D = (p["delta_l1"] if p["dyn"] else 0) + (p["delta_l2"] if p["dyn"] == ol.DYN["acc"] else 0)
    want_raw = oracle.extract(dict(p, norm=ol.NORM["none"]), utts, sample_limit=BIG)[0]
    for i in range(len(utts)):
        assert_close(raw[fo[i]:fo[i + 1] - D], want_raw[i][:len(want_raw[i]) - D], dict(p, norm=ol.NORM["none"]), f"raw utt {i}")
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
@pytest.mark.parametrize("name", ["hires40-none", "mfcc20-acc"])
def test_wide_cepstra_time_sharded_segments_equal_whole_stream(name):
    """One stream cut by time into 3 segments (afe_batch_plan_segments): bitwise the rows of the whole stream without
    normalisation (for deltas, the segments' context frames stand in for the neighbours)."""
    p = ol.default_params(**dict(SETS[name], norm="none"))
    w = ol.width_of(p)
    x = synth_utterances(1, 16000 * 40 + 77, seed=91)[0]
    whole = run_batch(p, [x], stats_scope=afe.STATS_UTTERANCE)[0]
    D = (p["delta_l1"] if p["dyn"] else 0) + (p["delta_l2"] if p["dyn"] == ol.DYN["acc"] else 0)
    sh = afe.shard_stream(len(x), 400, 160, D, 3)
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
@pytest.mark.parametrize("name", ["hires40-cmn", "hires39-none", "mfcc20-acc", "ceps41-acc"])
def test_wide_cepstra_streaming_object(oracle, name):
    """The streaming object runs wide DCTs on K1 (one launch per block, with the speculative flush tile and the use_last
    flush): blocks of 16 000 / 100 000 / 330 000 samples and the whole file against the reference fed the same blocks;
    the staged route (AFE_OPT_STAGED_KERNELS) stays within the same tolerance."""
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
def test_wide_cepstra_refusals_name_the_limit():
    """ceps_len + c0 = 49, and 17 cepstral columns from 65 banks, stay outside K1: afe_batch_create refuses them and the
    streaming object runs them on the staged kernels."""
    too_many = afe.make_params(input_buffer_size=BIG, num_banks=64, ceps_len=48, want_c0=1)
    wide_banks = afe.make_params(input_buffer_size=BIG, num_banks=65, ceps_len=16, want_c0=1)
    with pytest.raises(afe.AfeError, match=r"ceps_len \+ c0 <= 48"):
        afe.BatchMfcc(too_many, 0)
    with pytest.raises(afe.AfeError, match=r"ceps_len \+ c0 <= 16 with more than 64 banks"):
        afe.BatchMfcc(wide_banks, 0)
    for ap in (too_many, wide_banks):
        m = afe.MfccCuda(ap)
        assert not m.uses_fused_kernel
        m.close()
