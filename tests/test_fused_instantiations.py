"""Every instantiation of the fused kernel K1, k_fused_mfcc<N2, NZ, 8, KF, PRE>, end to end against the CPU oracle and
the float64 NumPy restatement, plus signal edges (silence, full-scale squares, DC, a tone at sr/4) for every
normalisation kind.

The instantiation key (afe_batch.cu, FusedEngine): N2 in {512, 256}; NZ = 13 (pruned first FFT layer) when
W <= 26 * N2 / 32, else 16; KF = ceil(num_banks / 8) rounded up to 3, 5 or 8; PRE = a non-zero pre-emphasis
coefficient. Each parameter set below is chosen to land on one key, with windows on both sides of the pruning cut-off,
odd windows (the last 32-bit PCM word holds a single sample) and bank counts on both sides of the KF cut-offs."""
import os
import sys

import numpy as np
import pytest

import oracle_lib as ol
from common import afe, assert_close, compare, synth_utterances, to_afe_params

sys.path.insert(0, os.path.join(ol.ROOT, "oracle"))
import oracle_np  # noqa: E402

BIG = 1 << 22
PRE = 0.97
K16 = dict(sample_rate=16000.0, low_freq=64.0, high_freq=8000.0, shift=160)
K8 = dict(sample_rate=8000.0, low_freq=64.0, high_freq=4000.0, shift=80)
FBANK_DELTA = dict(ceps_len=0, want_c0=0, dyn="delta")
# Pre-emphasis attenuates the lowest bands by 25 dB or more: with filters from 64 Hz their energies sit 60 dB below the
# frame's, where any fp32 FFT (pocketfft's included) is 3e-4 off in the log. The pre-emphasis entries start at 300 Hz.
PRE_LOW = dict(low_freq=300.0)

# (N2, NZ, KF, PRE) -> parameters; unnamed fields: 12 cepstra + c0, delta + acceleration (3 + 3), CMN
INSTANTIATIONS = {
    (512, 13, 3, False): dict(K16, window_size=400, num_banks=20),
    (512, 13, 5, False): dict(K16, window_size=401, num_banks=25, **FBANK_DELTA),
    (512, 13, 8, False): dict(K16, window_size=416, num_banks=64, ceps_len=15, norm="minmax"),
    (512, 13, 3, True): dict(K16, **PRE_LOW, window_size=416, num_banks=24),
    (512, 13, 5, True): dict(K16, **PRE_LOW, window_size=400, num_banks=40, norm="cvn"),
    (512, 13, 8, True): dict(K16, **PRE_LOW, window_size=401, num_banks=41, **FBANK_DELTA),
    (512, 16, 3, False): dict(K16, window_size=417, num_banks=24, norm="cvn"),
    (512, 16, 5, False): dict(K16, window_size=480, num_banks=40, ceps_len=0, want_c0=0),
    (512, 16, 8, False): dict(K16, window_size=512, num_banks=41),
    (512, 16, 3, True): dict(K16, **PRE_LOW, window_size=512, num_banks=20),
    (512, 16, 5, True): dict(K16, **PRE_LOW, window_size=417, num_banks=25, norm="minmax"),
    (512, 16, 8, True): dict(K16, **PRE_LOW, window_size=480, num_banks=64, **FBANK_DELTA),
    (256, 13, 3, False): dict(K8, window_size=200, num_banks=20),
    (256, 13, 5, False): dict(K8, window_size=129, num_banks=25, **FBANK_DELTA),
    (256, 13, 8, False): dict(K8, window_size=208, num_banks=41, norm="cvn"),
    (256, 13, 3, True): dict(K8, **PRE_LOW, window_size=208, num_banks=24, norm="minmax"),
    (256, 13, 5, True): dict(K8, **PRE_LOW, window_size=200, num_banks=40),
    (256, 13, 8, True): dict(K8, **PRE_LOW, window_size=129, num_banks=41, **FBANK_DELTA),
    (256, 16, 3, False): dict(K8, window_size=209, num_banks=20, norm="minmax"),
    (256, 16, 5, False): dict(K8, window_size=256, num_banks=40),
    (256, 16, 8, False): dict(K8, window_size=209, num_banks=41, **FBANK_DELTA),
    (256, 16, 3, True): dict(K8, **PRE_LOW, window_size=256, num_banks=24),
    (256, 16, 5, True): dict(K8, **PRE_LOW, window_size=209, num_banks=25, ceps_len=15, norm="cvn"),
    (256, 16, 8, True): dict(K8, **PRE_LOW, window_size=256, num_banks=41),
}
KEYS = sorted(INSTANTIATIONS)


def key_id(k):
    return "k_fused_mfcc<{},{},8,{},{}>".format(k[0], k[1], k[2], "true" if k[3] else "false")


def params_of(key):
    return ol.default_params(**dict(dict(norm="cmn", dyn="acc"), **INSTANTIATIONS[key]))


def test_instantiation_table_covers_every_key():
    assert len(KEYS) == 24 == len({key_id(k) for k in KEYS})
    for n2, nz, kf, _ in KEYS:
        p = params_of((n2, nz, kf, _))
        W = p["window_size"]
        assert 1 << (W - 1).bit_length() == n2
        assert (W <= 26 * n2 // 32) == (nz == 13)
        c = (p["num_banks"] + 7) // 8
        assert (3 if c <= 3 else 5 if c <= 5 else 8) == kf
        assert ol.width_of(p) <= 128


@pytest.mark.parametrize("key", KEYS, ids=key_id)
def test_instantiation_filters_match_numpy(key):
    """Host only: the library's filter edges are strictly increasing (no empty filter) and equal the float64
    restatement's, so a disagreement at float64 rounding cannot pose as a kernel error below."""
    p = params_of(key)
    edges, _ = afe.build_filters(to_afe_params(p, BIG))
    assert np.all(np.diff(edges) > 0), edges
    _, want, _ = oracle_np.mel_tables(p["num_banks"], key[0], p["sample_rate"], p["low_freq"], p["high_freq"])
    np.testing.assert_array_equal(edges, want)


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
def test_instantiation_end_to_end(oracle, key):
    """One batch of ragged utterances through the named instantiation with AFE_BATCH_Q1_EXACT, against the CPU oracle
    (no pre-emphasis: the reference has none) and against oracle_np.mfcc(q1=True); the plain staging path (utterance
    starts at 2 mod 8 samples, so odd windows store a single-sample tail word) gives the same bits as the TMA path."""
    p = params_of(key)
    pre = PRE if key[3] else 0.0
    utts = ragged_utterances(p, seed=key[0] + 10 * key[1] + key[2] + (1000 if key[3] else 0))
    name, got = run(p, utts, afe.BATCH_Q1_EXACT, pre)
    assert name == key_id(key)
    worst = [0.0, 0.0]
    if not key[3]:
        want = oracle.extract(p, utts, sample_limit=BIG)[0]
        for i, (g, w) in enumerate(zip(got, want)):
            worst[0] = max(worst[0], *assert_close(g, w, p, f"{name} utt {i} vs oracle"))
    for i, (g, u) in enumerate(zip(got, utts)):
        w = oracle_np.mfcc(u, dict(p, preemphasis=pre), q1=True).astype(np.float32)
        worst[1] = max(worst[1], *assert_close(g, w, p, f"{name} utt {i} vs float64"))
    print(f"{name}: worst max-abs vs oracle {worst[0]:.3g}, vs float64 {worst[1]:.3g}")
    _, plain = run(p, utts, afe.BATCH_Q1_EXACT | afe.BATCH_NO_TMA, pre, phase=2)
    for i, (a, b) in enumerate(zip(got, plain)):
        np.testing.assert_array_equal(a, b, err_msg=f"{name} utt {i}: plain staging differs from TMA")


@pytest.mark.gpu
@pytest.mark.parametrize("key", [k for k in KEYS if k[1] == 16], ids=key_id)
def test_unpruned_instantiation_streaming(oracle, key):
    """The streaming object runs the unpruned instantiations too: blocks of 16000 samples against the reference class
    fed the same blocks, or (pre-emphasis, no normalisation) against the float64 restatement."""
    p = params_of(key)
    x = synth_utterances(1, 61111, seed=7, sr=p["sample_rate"])[0]
    m = afe.MfccCuda(to_afe_params(p, 16000))
    assert m.uses_fused_kernel
    m.close()
    if key[3]:
        p = dict(p, norm=ol.NORM["none"])
        got = afe.extract_stream(to_afe_params(p, 16000), x, preemphasis=PRE)
        want = oracle_np.mfcc(x, dict(p, preemphasis=PRE)).astype(np.float32)
    else:
        got = afe.extract_stream(to_afe_params(p, 16000), x)
        want = oracle.extract(p, [x], sample_limit=16000)[0][0]
    e = assert_close(got, want, p, key_id(key) + " stream")
    print(f"{key_id(key)} stream: worst max-abs {max(e):.3g}")


# ---------------------------------------------------------------------------------------------- signal edges
EDGE_CONFIGS = {"config2": dict(window_size=400, shift=160, num_banks=23),
                "config5": dict(window_size=200, shift=80, num_banks=20, sample_rate=8000.0, high_freq=4000.0)}


def edge_signals(sr, n):
    speech = synth_utterances(3, n, seed=99, sr=sr)
    t = np.arange(n)
    sq = np.where((t // 20) % 2 == 0, 32767, -32767).astype(np.int16)
    sq_min = np.where((t // 10) % 2 == 0, 32767, -32768).astype(np.int16)
    lead = speech[0].copy()
    lead[:n // 3] = 0
    mid = speech[1].copy()
    mid[n // 3:n // 2] = 0
    return {
        "zeros": np.zeros(n, np.int16),
        "zero-lead": lead,
        "zero-middle": mid,
        "square+-32767": sq,
        "square-32768": sq_min,
        "dc": np.full(n, 12000, np.int16),
        "dc-offset": np.clip(speech[2].astype(np.int32) + 9000, -32768, 32767).astype(np.int16),
        "tone-sr/4": np.round(20000 * np.cos(np.pi * t / 2)).astype(np.int16),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["none", "cmn", "cvn", "minmax"])
@pytest.mark.parametrize("cfg", sorted(EDGE_CONFIGS))
def test_signal_edges_match_oracle(oracle, cfg, norm):
    """Silence, silence before and inside speech, full-scale squares (+-32767 and 32767 / -32768), DC, a DC offset
    and a tone at exactly sr/4 through K1 against the reference. Silent or periodic utterances give constant columns,
    where CVN and MINMAX divide by zero in the reference: there the result must be non-finite in the same places.

    CVN of an exactly constant column is 0 * sqrt((n-1) / (sumsq - sum^2/n)), where the variance is the float rounding
    error of v*v: its sign follows the last bit of v, so the reference gives NaN or 0 column by column. There either is
    accepted, from both."""
    p = ol.default_params(norm=norm, dyn="acc", **EDGE_CONFIGS[cfg])
    sig = edge_signals(p["sample_rate"], int(p["sample_rate"]) * 2 + 37)
    names = list(sig)
    _, got = run(p, [sig[k] for k in names], afe.BATCH_Q1_EXACT, 0.0)
    want = oracle.extract(p, [sig[k] for k in names], sample_limit=BIG)[0]
    raw = oracle.extract(dict(p, norm=ol.NORM["none"]), [sig[k] for k in names], sample_limit=BIG)[0]
    for k, g, w, r in zip(names, got, want, raw):
        if norm == "cvn":
            const = np.ptp(r, axis=0) == 0
            for x, who in ((g, "result"), (w, "reference")):
                assert np.all(~np.isfinite(x[:, const]) | (x[:, const] == 0)), f"{cfg} {k}: {who} in a constant column"
            g, w = np.where(const, np.nan, g), np.where(const, np.nan, w)
        compare(g, w, p, f"{cfg} {norm} {k}")
