"""GPU tier (`-m gpu`): the CUDA path, called through the C ABI (ctypes), against the pinned CPU oracle on the same
inputs. Tolerances are stated in tests/common.py:tolerances (SURVEY §7). Nothing here reads /root/reference."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from common import afe, assert_close, run_batch, synth_utterances, to_afe_params
from golden_io import load_golden, load_pcm

pytestmark = pytest.mark.gpu

BIG = 1 << 22


def oracle_extract(oracle, p, utts, sample_limit):
    return oracle.extract(p, utts, sample_limit=sample_limit)[0]


# ---------------------------------------------------------------------------------------------- streaming object
@pytest.mark.parametrize("case", sorted(load_golden().keys()))
def test_stream_object_matches_golden_and_oracle(oracle, case):
    """MfccCuda driven like the reference driver drives ParamBase, block sizes as in the golden case."""
    g = load_golden()[case]
    p, pcm = g["params"], load_pcm()[g["utt"]]
    limit = g["sample_limit"] if g["sample_limit"] > 0 else len(pcm)
    got = afe.extract_stream(to_afe_params(p, limit), pcm, alpha=p["alpha"])
    assert got.shape == (g["frames"], g["width"])
    assert_close(got[g["rows"]], g["feats"], p, case + " vs golden")
    want = oracle_extract(oracle, p, [pcm], g["sample_limit"])[0]
    assert_close(got, want, p, case + " vs oracle")


def test_stream_fix_flush_statics_option(oracle):
    """AFE_OPT_FIX_FLUSH_STATICS: single block + flush gives the streamed (intended) statics for the last D rows."""
    pcm = load_pcm()["a1"]
    p = ol.default_params(dyn="acc")
    want = oracle_extract(oracle, p, [pcm], 0)[0]           # 2 set_input calls -> no Q1
    got = afe.extract_stream(to_afe_params(p, BIG), pcm, fix_flush_statics=True)
    assert_close(got, want, p, "fixed flush")
    exact = afe.extract_stream(to_afe_params(p, BIG), pcm)  # default: reference-exact (Q1)
    assert_close(exact, oracle_extract(oracle, p, [pcm], BIG)[0], p, "q1 exact")


def test_stream_vtln_sweep_reuses_spectrum(oracle):
    """set_alpha + repeated apply() after ONE set_input (ASR_OCL.cpp:236-243): the spectrum must persist."""
    pcm = load_pcm()["sample1"]
    p = ol.default_params(dyn="acc", norm="cmn")
    m = afe.MfccCuda(to_afe_params(p, BIG))
    m.set_window(afe.make_window(400))
    ref = ol.RefMfcc(oracle, BIG, p)
    ref.set_window(oracle.window(400))
    n = m.get_input_buffer_size()
    assert n == ref.get_input_buffer_size()
    wc = m.set_input(pcm[:n])
    assert wc == ref.set_input(pcm[:n])
    for alpha in (0.9, 1.0, 1.1):
        m.set_alpha(alpha); ref.set_alpha(alpha)
        m.apply(); ref.apply()
        assert_close(m.get_output_data(wc), ref.get_output_data(wc), p, f"alpha={alpha}")
    m.close(); ref.close()


def test_stream_error_behaviour():
    p = afe.make_params(input_buffer_size=16000, dyn=2)
    m = afe.MfccCuda(p)
    m.set_window(afe.make_window(400))
    assert m.get_input_buffer_size() == 98 * 160 + 240                    # parambase.cpp:12-13
    with pytest.raises(afe.AfeError, match="buffer is too small"):       # mfcccpu.cpp:338-339
        m.set_input(np.zeros(m.get_input_buffer_size() + 1, np.int16))
    with pytest.raises(afe.AfeError, match="window count is too small"):  # segmentercpu.cpp:65-66
        m.set_input(np.zeros(400 + 160 * 5, np.int16))
    m.reset()
    assert m.set_input(np.zeros(m.get_input_buffer_size(), np.int16)) == 98 - 6
    m.apply()
    with pytest.raises(afe.AfeError, match="Window count too high"):      # mfcccpu.cpp:429-430
        m.get_output_data(10_000)
    assert m.flush() == 6
    assert m.flush() == 0                                                 # idempotent (mfcccpu.cpp:350-352)
    m.close()


def test_stream_refuses_where_the_reference_overruns_its_buffer():
    """W > 2S without deltas: carry-over (W - S + leftover) + a full block exceeds the reference's buffer of
    (est(limit) + 2) * S + W - S samples and SegmenterCPU::set_input overruns its heap (segmentercpu.cpp:41,76-78; found by
    tools/fuzz_gpu.py, confirmed under AddressSanitizer). The object raises the reference's buffer error instead."""
    p = ol.default_params(window_size=480, shift=124, num_banks=32, low_freq=120.0, high_freq=6800.0, ceps_len=13)
    x = synth_utterances(1, 41312, seed=1033)[0]
    with pytest.raises(afe.AfeError, match="buffer is too small"):
        afe.extract_stream(to_afe_params(p, 16000), x)
    got = afe.extract_stream(to_afe_params(p, BIG), x)          # one block: fine
    assert got.shape[0] == (len(x) - (480 - 124)) // 124 and np.isfinite(got).all()


def test_stream_reset_makes_handle_reusable(oracle):
    pcm = load_pcm()
    p = ol.default_params(dyn="acc", norm="cmn")
    m = afe.MfccCuda(to_afe_params(p, BIG))
    m.set_window(afe.make_window(400))
    for name in ("a1", "sample1"):
        rows = []
        wc = m.set_input(pcm[name]); m.apply(); rows.append(m.get_output_data(wc))
        wc = m.flush(); m.apply(); rows.append(m.get_output_data(wc))
        assert_close(np.concatenate(rows), oracle_extract(oracle, p, [pcm[name]], BIG)[0], p, name)
        m.reset()
    m.close()


def test_stream_generic_fft_sizes(oracle):
    """window sizes whose ceil2 is neither 256 nor 512 take the generic shared-memory FFT kernel."""
    pcm = load_pcm()["sample1"]
    for W, S in ((100, 40), (640, 160), (1024, 256)):
        p = ol.default_params(window_size=W, shift=S, dyn="acc")
        got = afe.extract_stream(to_afe_params(p, BIG), pcm, window=oracle.window(W))
        want = oracle_extract(oracle, p, [pcm], BIG)[0]
        assert_close(got, want, p, f"W={W}")


# ---------------------------------------------------------------------------------------------- stage objects
def test_segmenter_cuda_bit_exact_and_state(oracle):
    pcm = load_pcm()["a1"]
    W, S, D, limit = 400, 160, 6, 120
    seg = afe.SegmenterCuda(W, S, limit, D)
    seg.set_window(afe.make_window(W))
    ref = oracle.segmenter_create(W, S, limit, D)
    win = oracle.window(W)
    oracle.segmenter_set_window(ref, win.ctypes.data_as(C.POINTER(C.c_float)))
    buf = np.zeros((limit, 512), np.float32)
    pos = 0
    for n in (16000, 16000, 7000, 16000):
        blk = np.ascontiguousarray(pcm[pos:pos + n]); pos += n
        wc, nd = seg.set_input(blk)
        rwc, rnd = C.c_int(0), C.c_int(0)
        buf[:] = 0
        assert oracle.segmenter_set_input(ref, blk.ctypes.data_as(C.POINTER(C.c_short)), buf.ctypes.data_as(C.POINTER(C.c_float)),
                                          n, C.byref(rwc), C.byref(rnd)) == 0
        assert (wc, nd) == (rwc.value, rnd.value)
        assert seg.get_remaining_samples() == oracle.segmenter_remaining_samples(ref)
        assert seg.get_samples() == oracle.segmenter_samples(ref)
        assert seg.was_flushed() == bool(oracle.segmenter_was_flushed(ref))
        np.testing.assert_array_equal(seg.frames(nd), buf[:nd])          # one fp32 multiply per sample: bit-exact
    wc, nd = seg.flush()
    rwc, rnd = C.c_int(0), C.c_int(0)
    buf[:] = 0
    oracle.segmenter_flush(ref, buf.ctypes.data_as(C.POINTER(C.c_float)), C.byref(rwc), C.byref(rnd))
    assert (wc, nd) == (rwc.value, rnd.value) and seg.is_flushed()
    np.testing.assert_array_equal(seg.frames(nd), buf[:nd])
    oracle.segmenter_destroy(ref)
    seg.close()


@pytest.mark.parametrize("L", [1, 2, 3])
def test_delta_cuda_bit_exact(oracle, L):
    rng = np.random.default_rng(L)
    rows, dim = 257, 13
    x = rng.standard_normal((rows + 2 * L, dim)).astype(np.float32) * 10
    want = np.zeros((rows, dim), np.float32)
    fp = C.POINTER(C.c_float)
    oracle.delta_apply(x.ctypes.data_as(fp), want.ctypes.data_as(fp), dim, rows, L)
    d = afe.DeltaCuda(dim, rows, L)
    np.testing.assert_array_equal(d.apply(x, rows), want)                # unfused mul/add/div like the CPU: bit-exact
    d.close()


@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_normalizer_cuda(oracle, norm):
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((1000, 39)) * 4 + 11).astype(np.float32)
    want = x.copy()
    h = oracle.normalizer_create(ol.NORM[norm], 39)
    oracle.normalizer_normalize(h, want.ctypes.data_as(C.POINTER(C.c_float)), 1000, 0)
    n = afe.NormalizerCuda(ol.NORM[norm], 39)
    got = n.normalize(x)
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-6)             # double stats, summation order differs
    tail = x[:9].copy()
    oracle.normalizer_normalize(h, tail.ctypes.data_as(C.POINTER(C.c_float)), 9, 1)
    np.testing.assert_allclose(n.normalize(x[:9], use_last_stats=True), tail, rtol=0, atol=2e-6)
    oracle.normalizer_destroy(h)
    n.close()


# ---------------------------------------------------------------------------------------------- fused batch path
SOUNDFILES = ["a0001", "a1", "a2", "a3", "a4", "a5"]


@pytest.mark.parametrize("flags", [0, afe.BATCH_NO_TMA, afe.BATCH_UNFUSED_NORM], ids=["tma", "plain-loads", "unfused-norm"])
def test_batch_config2_soundfiles_q1_exact(oracle, flags):
    """BASELINE config 2: a0001 + a1..a5, 23 mel, 12+c0, delta+delta-delta, per-utterance CMN, one block per
    utterance. AFE_BATCH_Q1_EXACT == the reference driver with its default sample_limit (single set_input + flush)."""
    pcm = load_pcm()
    p = ol.default_params(norm="cmn", dyn="acc")
    utts = [pcm[n] for n in SOUNDFILES]
    got = run_batch(p, utts, flags=afe.BATCH_Q1_EXACT | flags)
    want = oracle_extract(oracle, p, utts, BIG)
    assert [len(g) for g in got] == [711, 504, 1011, 1517, 2023, 2529]
    for n, g, w in zip(SOUNDFILES, got, want):
        assert_close(g, w, p, n)
    G = load_golden()
    for n in SOUNDFILES:
        gold = G[f"c2_{n}_single"]
        assert_close(got[SOUNDFILES.index(n)][gold["rows"]], gold["feats"], p, n + " golden")


def test_batch_config2_intended_semantics(oracle):
    """Without the Q1 flag the last D rows carry their own statics == the reference fed in >= 2 blocks."""
    pcm = load_pcm()
    p = ol.default_params(norm="cmn", dyn="acc")
    # a0001 and a2 are exactly frame aligned, so the reference would take them in ONE set_input even with
    # sample_limit = N (Q1 again); three trailing zero samples force the second, frame-less block without adding a frame
    utts = [np.concatenate([pcm[n], np.zeros(3, np.int16)]) for n in SOUNDFILES]
    got = run_batch(p, utts)
    want = oracle_extract(oracle, p, utts, 0)
    for n, g, w in zip(SOUNDFILES, got, want):
        assert_close(g, w, p, n)


def test_batch_unfused_variants(oracle):
    """K2 + K3 kernels (AFE_BATCH_UNFUSED_NORM) for CVN / MINMAX / norm-before-dyn."""
    G = load_golden()
    for case in ("v_a1_cvn", "v_a1_minmax", "v_a1_norm_before_dyn"):
        g = G[case]
        got = run_batch(g["params"], [load_pcm()[g["utt"]]], flags=afe.BATCH_Q1_EXACT | afe.BATCH_UNFUSED_NORM)[0]
        assert_close(got[g["rows"]], g["feats"], g["params"], case + " unfused")


@pytest.mark.parametrize("case", ["c1_sample1", "c1_sample1_acc", "c3_a1_40mel", "c3_a1_40mel_nonorm", "v_a1_cvn",
                                  "v_a1_minmax", "v_a1_delta_only", "v_a1_l1_2_l2_1", "v_a1_norm_before_dyn",
                                  "v_a1_fbank", "v_a1_nolifter_noc0", "v_a1_alpha090", "v_a1_alpha112", "c5_a1_8k"])
def test_batch_variants_match_golden(oracle, case):
    g = load_golden()[case]
    p, pcm = g["params"], load_pcm()[g["utt"]]
    got = run_batch(p, [pcm], flags=afe.BATCH_Q1_EXACT)[0]
    assert_close(got[g["rows"]], g["feats"], p, case + " vs golden")
    assert_close(got, oracle_extract(oracle, p, [pcm], BIG)[0], p, case + " vs oracle")


def test_batch_config3_synthetic_subset(oracle):
    """BASELINE config 3 on a 64-utterance subset (BASELINE.md §3): synthetic 16 kHz, 10 s, 40 mel, 13 MFCC + d + dd, CMN."""
    p = ol.default_params(num_banks=40, norm="cmn", dyn="acc")
    utts = synth_utterances(64, 160000)
    got = run_batch(p, utts, flags=afe.BATCH_Q1_EXACT)
    want = oracle_extract(oracle, p, utts, BIG)
    worst = (0.0, 0.0)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == (998, 39)
        e = assert_close(g, w, p, f"utt {i}")
        worst = max(worst, e)
    print("config3 subset worst (static, delta) abs err:", worst)


def test_batch_config5_telephony_long_stream(oracle):
    """BASELINE config 5 shape (8 kHz, 256-pt FFT, 20 mel, fused deltas) on a 60 s stream: many tiles with halos."""
    p = ol.default_params(window_size=200, shift=80, num_banks=20, sample_rate=8000.0, high_freq=4000.0, dyn="acc")
    x = synth_utterances(1, 480000, seed=5, sr=8000.0)[0]
    got = run_batch(p, [x], flags=afe.BATCH_Q1_EXACT)[0]
    want = oracle_extract(oracle, p, [x], BIG)[0]
    assert got.shape == (5998, 39)
    assert_close(got, want, p, "8k stream")
    pc = dict(p, norm=ol.NORM["cmn"])
    assert_close(run_batch(pc, [x], flags=afe.BATCH_Q1_EXACT)[0], oracle_extract(oracle, pc, [x], BIG)[0], pc, "8k cmn")


def test_batch_ragged_and_edge_lengths(oracle):
    """Ragged batch incl. the shortest legal utterance (T = 2D+1), a tile-boundary length and an odd sample count."""
    p = ol.default_params(norm="cmn", dyn="acc")
    D = 6
    # (+k samples: not frame aligned, so the oracle with sample_limit = N needs a second set_input -> no Q1)
    lens = [240 + 160 * (2 * D + 1) + 5, 240 + 160 * 244 + 1, 240 + 160 * 245 + 77, 240 + 160 * 489 + 3, 50001,
            240 + 160 * 32 + 8]
    utts = [synth_utterances(1, n, seed=n)[0] for n in lens]
    got = run_batch(p, utts)
    want = oracle_extract(oracle, p, utts, 0)
    for n, g, w in zip(lens, got, want):
        assert_close(g, w, p, f"len {n}")
    with pytest.raises(afe.AfeError, match="window count is too small"):
        run_batch(p, [np.zeros(240 + 160 * 2 * D, np.int16)])


def test_batch_is_deterministic_and_order_independent():
    """Size-independent properties at a larger size: bitwise repeatable; rows of an utterance do not depend on its
    neighbours or on the staging path (TMA bulk copy vs plain loads)."""
    p = ol.default_params(num_banks=40, norm="cmn", dyn="acc")
    utts = synth_utterances(96, 160000, seed=11, ragged=True)
    a = run_batch(p, utts)
    b = run_batch(p, utts)
    c = run_batch(p, utts[::-1])[::-1]
    d = run_batch(p, utts, flags=afe.BATCH_NO_TMA)
    e = run_batch(p, utts, flags=afe.BATCH_UNFUSED_NORM)   # separate K2/K3 kernels == in-kernel normalisation, bitwise
    for i in range(len(utts)):
        np.testing.assert_array_equal(a[i], b[i])
        np.testing.assert_array_equal(a[i], c[i])
        np.testing.assert_array_equal(a[i], d[i])
        np.testing.assert_array_equal(a[i], e[i])


@pytest.mark.parametrize("cfg", [dict(num_banks=40), dict(num_banks=23), dict(num_banks=64),
                                 dict(num_banks=20, window_size=200, shift=80, sample_rate=8000.0, high_freq=4000.0),
                                 dict(num_banks=40, ceps_len=0, want_c0=0), dict(num_banks=26, ceps_len=15, want_c0=1)])
def test_batch_filterbank_shapes_match_oracle(oracle, cfg):
    """Phase 2 of the fused kernel (mel sums, logs, DCT) against the reference's CPU classes for all three filters-per-warp
    instantiations (20 to 64 banks), 256- and 512-point FFTs, FBANK output and 16 DCT columns, VTLN-warped banks and ragged
    lengths; the handle names the instantiation that runs."""
    p = ol.default_params(norm="cmn", dyn="acc", **cfg)
    utts = synth_utterances(10, 60000, seed=51, sr=p["sample_rate"], ragged=True)
    for alpha in (1.0, 0.9):
        q = dict(p, alpha=alpha)
        got = run_batch(q, utts, flags=afe.BATCH_Q1_EXACT)
        want = oracle_extract(oracle, q, utts, BIG)
        for i in range(len(utts)):
            assert_close(got[i], want[i], q, f"utt {i} alpha {alpha}")
    bm = afe.BatchMfcc(to_afe_params(p, BIG), 0)
    try:
        kf = (p["num_banks"] + 7) // 8
        n2 = 512 if p["window_size"] > 256 else 256
        assert bm.kernel_name == f"k_fused_mfcc<{n2},13,8,{3 if kf <= 3 else 5 if kf <= 5 else 8},false>", bm.kernel_name
    finally:
        bm.close()


def test_batch_refuses_unknown_flags():
    """Flag bits outside AFE_BATCH_Q1_EXACT | NO_TMA | UNFUSED_NORM | NO_CLUSTER fail loudly instead of being ignored
    (64 selected the tensor-core phase 2 before ABI 3)."""
    with pytest.raises(afe.AfeError, match="unknown batch flag bits 64"):
        afe.BatchMfcc(afe.make_params(), 0, flags=64)


@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_batch_cluster_normalisation_equals_ticket_scheme(norm):
    """Fused normalisation inside a thread-block cluster (one cluster = the 1 or 2 tiles of an utterance, statistics
    records exchanged through distributed shared memory, rows written already normalised) against the ticket scheme
    (AFE_BATCH_NO_CLUSTER: last tile normalises in place through L2) and against K2 + K3: bitwise equal. Batches of
    2-tile utterances, of 1-tile utterances, length-sorted mixed (two runs) and with 3-tile (cluster of 3) and 6-tile
    (ticket scheme) utterances."""
    p = ol.default_params(num_banks=40, norm=norm, dyn="acc")
    long_ = synth_utterances(40, 160000, seed=31)
    short = synth_utterances(40, 60000, seed=32)
    three = synth_utterances(2, 250000, seed=33)          # 3 tiles: cluster of 3
    four = synth_utterances(2, 320000, seed=35)           # 4 tiles: cluster of 4 (the largest)
    six = synth_utterances(1, 450000, seed=34)            # 6 tiles: ticket scheme
    for utts in (long_, short, short + long_, short + three + four + long_ + six):
        for extra in (0, afe.BATCH_Q1_EXACT):
            a = run_batch(p, utts, flags=extra)
            b = run_batch(p, utts, flags=extra | afe.BATCH_NO_CLUSTER)
            c = run_batch(p, utts, flags=extra | afe.BATCH_UNFUSED_NORM)
            for i in range(len(utts)):
                np.testing.assert_array_equal(a[i], b[i])
                np.testing.assert_array_equal(a[i], c[i])


def test_batch_linearity_property():
    """Without log the path would be linear; with it, scaling the PCM by 2 shifts every log-mel by ln 2, i.e. adds
    ln2 * sum_k M[k][j] to cepstrum j and leaves deltas unchanged (checked on c0: sqrt(2/nb)*nb*ln 2)."""
    p = ol.default_params(num_banks=40, dyn="acc")
    x = synth_utterances(4, 80000, seed=3)
    half = [(u // 2 * 1).astype(np.int16) for u in x]
    dbl = [(h * 2).astype(np.int16) for h in half]
    a, b = run_batch(p, half), run_batch(p, dbl)
    shift = np.sqrt(2.0 / 40) * 40 * np.log(2.0)
    for u, v in zip(a, b):
        np.testing.assert_allclose(v[:, 12] - u[:, 12], shift, atol=2e-4)
        np.testing.assert_allclose(v[:, 13:], u[:, 13:], atol=2e-4)


def test_batch_equals_stream_object():
    """The batch extractor, the streaming object on the fused kernel and the streaming object on the staged kernels
    (AFE_OPT_STAGED_KERNELS) are three routes to the same arithmetic."""
    pcm = load_pcm()["a3"]
    p = ol.default_params(norm="cvn", dyn="acc")
    a = run_batch(p, [pcm], flags=afe.BATCH_Q1_EXACT)[0]
    b = afe.extract_stream(to_afe_params(p, BIG), pcm)
    c = afe.extract_stream(to_afe_params(p, BIG), pcm, staged=True)
    np.testing.assert_allclose(a, b, atol=2e-6)   # same kernel, same tiles up to the block structure
    np.testing.assert_allclose(a, c, atol=2e-4)


# ---------------------------------------------------------------------------------------------- streaming object on K1
def test_stream_object_runs_the_fused_kernel():
    """One launch of k_fused_mfcc per apply(); parameter sets it does not cover fall back to the staged kernels."""
    m = afe.MfccCuda(afe.make_params(input_buffer_size=BIG, norm=1, dyn=2))
    assert m.uses_fused_kernel
    m.set_window(afe.make_window(400))
    pcm = load_pcm()["a1"]
    wc = m.set_input(pcm); m.apply(); m.get_output_data(wc)
    assert m.kernel_launches == 1
    wc = m.flush(); m.apply(); m.get_output_data(wc)
    assert m.kernel_launches == 1            # the flush rows were computed speculatively by the block's launch
    m.reset()
    wc = m.set_input(pcm); m.set_alpha(0.9); m.apply(); m.get_output_data(wc)
    wc = m.flush(); m.set_alpha(1.0); m.apply(); m.get_output_data(wc)
    assert m.kernel_launches == 3            # alpha changed before the flush: the speculation is discarded, one more launch
    m.close()
    for kw in (dict(window_size=640), dict(shift=161), dict(norm=1, dyn=2, norm_after_dyn=0)):
        m = afe.MfccCuda(afe.make_params(input_buffer_size=BIG, **kw))
        assert not m.uses_fused_kernel
        m.close()


@pytest.mark.parametrize("norm", ["none", "cmn", "cvn", "minmax"])
@pytest.mark.parametrize("dyn,l1,l2", [("acc", 3, 3), ("acc", 2, 1), ("delta", 2, 2), ("none", 3, 3)])
def test_stream_fused_blocks_match_oracle(oracle, norm, dyn, l1, l2):
    """Every block shape of the state machine through K1: first / middle / flush blocks, 1 tile, several tiles (cluster,
    ticket scheme) and more than 8 tiles (role scheme), all regressions, against the reference class fed the same blocks."""
    pcm = np.concatenate([load_pcm()["a5"], load_pcm()["a4"]])   # 45.5 s
    p = ol.default_params(norm=norm, dyn=dyn, delta_l1=l1, delta_l2=l2)
    for limit in (16000, 100000, 330000, 1 << 20):               # ~100 / 623 / 2061 / 4556-frame blocks
        got = afe.extract_stream(to_afe_params(p, limit), pcm)
        want = oracle_extract(oracle, p, [pcm], limit)[0]
        assert_close(got, want, p, f"limit={limit}")


def test_stream_fused_equals_staged_bitwise_structure():
    """Fused and staged routes on the same blocks (golden streamed case c2_a1_stream16k parameters): within one rounding
    of each other, and the fused route is bitwise repeatable."""
    pcm = load_pcm()["a3"]
    p = ol.default_params(norm="cmn", dyn="acc")
    a = afe.extract_stream(to_afe_params(p, 16000), pcm)
    b = afe.extract_stream(to_afe_params(p, 16000), pcm)
    c = afe.extract_stream(to_afe_params(p, 16000), pcm, staged=True)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_allclose(a, c, atol=1e-4)


def test_stream_short_utterances(oracle):
    """Utterances of D+1 .. 2D+2 frames (ADVICE r1: the first-block arithmetic of segmentercpu.cpp:69-73 runs out of its
    buffer below 2D frames): below 2D frames the reference's own error, from 2D on the reference's rows."""
    p = ol.default_params(dyn="acc")
    D = 6
    for T in range(D + 1, 2 * D + 3):
        x = synth_utterances(1, 240 + 160 * T, seed=T)[0]
        if T < 2 * D:
            with pytest.raises(afe.AfeError, match="window count is too small"):
                afe.extract_stream(to_afe_params(p, BIG), x)
        else:
            got = afe.extract_stream(to_afe_params(p, BIG), x)
            want = oracle_extract(oracle, p, [x], BIG)[0]
            assert got.shape == (T, 39)
            assert_close(got, want, p, f"T={T}")


def test_preemphasis_against_numpy_and_zero_is_identity():
    """Pre-emphasis is NOT in the reference (segmentercpu.cpp:21-27): coefficient 0 is bit-identical to the default path;
    0.97 matches the NumPy float64 restatement (oracle/oracle_np.py) on the batch, fused-stream and staged-stream routes."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import oracle_np
    pcm = load_pcm()["a1"]
    p = ol.default_params(num_banks=40, norm="cmn", dyn="acc")
    ap = to_afe_params(p, BIG)

    def batch(pre):
        b = afe.BatchMfcc(ap, 0, preemphasis=pre)
        x, offs, lens = afe.pack_utterances([pcm])
        b.plan(offs, lens)
        out = b.run_host(np.concatenate([x, np.zeros(16, np.int16)]))
        b.close()
        return out

    base = run_batch(p, [pcm])[0]
    np.testing.assert_array_equal(batch(0.0), base)
    want = oracle_np.mfcc(pcm, dict(p, preemphasis=0.97)).astype(np.float32)
    assert np.abs(want - base).max() > 0.5                       # it does something
    assert_close(batch(0.97), want, p, "batch pre-emphasis")
    # streamed in two blocks (no Q1): fused and staged routes
    limit = 50000
    fused = afe.extract_stream(to_afe_params(p, limit), pcm, preemphasis=0.97)
    staged = afe.extract_stream(to_afe_params(p, limit), pcm, preemphasis=0.97, staged=True)
    assert_close(fused, staged, p, "fused vs staged pre-emphasis")
    p0 = ol.default_params(num_banks=40, dyn="acc")
    got = afe.extract_stream(to_afe_params(p0, limit), pcm, preemphasis=0.97)
    assert_close(got, oracle_np.mfcc(pcm, dict(p0, preemphasis=0.97)).astype(np.float32), p0, "stream pre-emphasis")


# ---------------------------------------------------------------------------------------------- corpus CMVN
def test_corpus_cmvn_many_tiles_two_level_reduction():
    """> 592 tiles: the corpus statistics take the two-level reduction; must equal NumPy on the raw features."""
    p = ol.default_params(norm="cvn", dyn="acc")
    utts = synth_utterances(700, 6000, seed=33, ragged=True)
    utts = [u for u in utts if len(u) >= 240 + 160 * 14]
    ap = to_afe_params(p, BIG)
    b = afe.BatchMfcc(ap, 0, stats_scope=afe.STATS_CORPUS)
    pcm, offs, lens = afe.pack_utterances(utts)
    total = b.plan(offs, lens)
    assert b.num_tiles > 592
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * 39 * 4)
    b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
    b.synchronize()
    raw = d_out.download((total, 39), np.float32).astype(np.float64)
    b.corpus_stats()
    b.normalize_device(d_out.ptr.value)
    b.synchronize()
    got = d_out.download((total, 39), np.float32)
    n = len(raw)
    want = (raw - raw.mean(0)) * np.sqrt((n - 1) / ((raw * raw).sum(0) - raw.sum(0) ** 2 / n))
    np.testing.assert_allclose(got, want, atol=2e-5)
    b.close(); d_pcm.free(); d_out.free()


@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_corpus_cmvn_two_shards_equal_one(norm):
    """Corpus statistics: (a) one batch; (b) two 'ranks' over disjoint utterance shards whose statistics records are
    merged as the NCCL all-reduce merges them (sum | min | max) — must agree, and match NumPy on the raw features."""
    p = ol.default_params(num_banks=40, norm=norm, dyn="acc")
    utts = synth_utterances(24, 48000, seed=21, ragged=True)
    w = ol.width_of(p)

    def two_pass(shard, merged=None):
        ap = to_afe_params(p, BIG)
        b = afe.BatchMfcc(ap, 0, stats_scope=afe.STATS_CORPUS)
        pcm, offs, lens = afe.pack_utterances(shard)
        total = b.plan(offs, lens)
        d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
        d_out = afe.DeviceBuffer(total * w * 4)
        b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
        ptr, n = b.corpus_stats()
        b.synchronize()
        stats = np.zeros(n, np.float64)
        afe._check(afe.lib().afe_memcpy_d2h(0, stats.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), stats.nbytes))
        raw = d_out.download((total, w), np.float32)
        if merged is not None:
            b.set_corpus_stats(merged)
        b.normalize_device(d_out.ptr.value)
        b.synchronize()
        out = d_out.download((total, w), np.float32)
        b.close(); d_pcm.free(); d_out.free()
        return raw, stats, out

    raw, stats, one = two_pass(utts)
    ra, sa, _ = two_pass(utts[:10])
    rb, sb, _ = two_pass(utts[10:])
    merged = np.concatenate([sa[:2 * w + 1] + sb[:2 * w + 1], np.minimum(sa[2 * w + 1:3 * w + 1], sb[2 * w + 1:3 * w + 1]),
                             np.maximum(sa[3 * w + 1:], sb[3 * w + 1:])])
    np.testing.assert_allclose(merged[:2 * w + 1], stats[:2 * w + 1], rtol=1e-12)
    np.testing.assert_array_equal(merged[2 * w + 1:], stats[2 * w + 1:])
    _, _, oa = two_pass(utts[:10], merged)
    _, _, ob = two_pass(utts[10:], merged)
    np.testing.assert_allclose(np.concatenate([oa, ob]), one, atol=1e-6)
    # NumPy restatement of normalizercpu.cpp:31-66 over the whole corpus
    x = raw.astype(np.float64)
    mu = x.mean(0)
    if norm == "cmn":
        want = x - mu
    elif norm == "cvn":
        want = (x - mu) * np.sqrt((len(x) - 1) / ((x * x).sum(0) - x.sum(0) ** 2 / len(x)))
    else:
        want = (x - mu) / np.maximum(np.abs(x.min(0) - mu), np.abs(x.max(0) - mu))
    np.testing.assert_allclose(one, want, atol=2e-5 if norm != "cvn" else 1e-5)
    mean, scale = afe.cmvn_finalize_host(ol.NORM[norm], w, stats)
    np.testing.assert_allclose(mean, mu, atol=1e-5)


# ---------------------------------------------------------------------------------------------- Normalizer-owned corpus verbs
@pytest.mark.parametrize("norm", ["cmn", "cvn", "minmax"])
def test_normalizer_corpus_verbs(norm):
    """reset -> accumulate (3 blocks) -> finalize -> apply == NumPy over the concatenation (normalizercpu.cpp:31-66);
    two Normalizers over disjoint blocks whose records are merged like the all-reduce merges them give the same rows."""
    rng = np.random.default_rng(5)
    blocks = [(rng.standard_normal((n, 39)) * 3 + 7).astype(np.float32) for n in (700, 1, 1299)]
    x = np.concatenate(blocks).astype(np.float64)
    mu = x.mean(0)
    if norm == "cmn":
        want = x - mu
    elif norm == "cvn":
        want = (x - mu) * np.sqrt((len(x) - 1) / ((x * x).sum(0) - x.sum(0) ** 2 / len(x)))
    else:
        want = (x - mu) / np.maximum(np.abs(x.min(0) - mu), np.abs(x.max(0) - mu))
    n = afe.NormalizerCuda(ol.NORM[norm], 39)
    assert n.stats_len == 4 * 39 + 1
    n.reset()
    for b in blocks:
        n.accumulate(b)
    rec = n.get_stats()
    assert rec[2 * 39] == len(x)
    np.testing.assert_allclose(rec[:39], x.sum(0), rtol=1e-12)
    np.testing.assert_array_equal(rec[2 * 39 + 1:3 * 39 + 1], x.min(0))
    np.testing.assert_array_equal(rec[3 * 39 + 1:], x.max(0))
    n.finalize()
    got = np.concatenate([n.apply(b) for b in blocks])
    np.testing.assert_allclose(got, want, atol=3e-6)
    # two "ranks": merge the records by hand (sum | min | max), push the merged record into both
    a, b = afe.NormalizerCuda(ol.NORM[norm], 39), afe.NormalizerCuda(ol.NORM[norm], 39)
    a.reset(); b.reset()
    a.accumulate(blocks[0]); b.accumulate(blocks[1]); b.accumulate(blocks[2])
    ra, rb = a.get_stats(), b.get_stats()
    w = 39
    merged = np.concatenate([ra[:2 * w + 1] + rb[:2 * w + 1], np.minimum(ra[2 * w + 1:3 * w + 1], rb[2 * w + 1:3 * w + 1]),
                             np.maximum(ra[3 * w + 1:], rb[3 * w + 1:])])
    a.set_stats(merged); b.set_stats(merged)
    a.finalize(); b.finalize()
    got2 = np.concatenate([a.apply(blocks[0]), b.apply(blocks[1]), b.apply(blocks[2])])
    np.testing.assert_allclose(got2, got, atol=1e-6)
    for h in (n, a, b):
        h.close()


def test_batch_routes_corpus_statistics_through_its_normalizer():
    """afe_batch_normalizer(): the record the batch reduces into IS the Normalizer's (scope CORPUS); other scopes have none."""
    p = ol.default_params(num_banks=40, norm="cvn", dyn="acc")
    utts = synth_utterances(12, 48000, seed=2, ragged=True)
    ap = to_afe_params(p, BIG)
    b = afe.BatchMfcc(ap, 0, stats_scope=afe.STATS_CORPUS)
    pcm, offs, lens = afe.pack_utterances(utts)
    total = b.plan(offs, lens)
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * 39 * 4)
    b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
    ptr, n = b.corpus_stats()
    b.synchronize()
    raw = d_out.download((total, 39), np.float32).astype(np.float64)
    rec = b.corpus_record()
    assert len(rec) == n == 4 * 39 + 1 and rec[2 * 39] == total
    np.testing.assert_allclose(rec[:39], raw.sum(0), rtol=1e-12)
    with pytest.raises(afe.AfeError, match="statistics scope"):
        b.set_options(afe.STATS_UTTERANCE, 0)                    # ADVICE r1: the plan depends on the scope
    b.close(); d_pcm.free(); d_out.free()
    b2 = afe.BatchMfcc(ap, 0, stats_scope=afe.STATS_UTTERANCE)
    b2.plan(offs, lens)
    with pytest.raises(afe.AfeError, match="no corpus Normalizer"):
        b2.normalizer
    b2.close()


# ---------------------------------------------------------------------------------------------- BASELINE config 5 at full size
@pytest.mark.parametrize("norm", ["none", "cmn"])
def test_config5_full_size_one_hour_stream(oracle, norm):
    """BASELINE configs[4] at its real size: ONE 8 kHz stream of 28 800 000 samples (1 hour), 256-point FFT, 20 mel, fused
    deltas -> 359 998 frames in 720 tiles. With CMN the statistics are final only after the last tile: the role scheme
    (one launch: extracting CTAs + one normalising CTA per tile) must equal the K2 + K3 kernels bit for bit, and both the
    reference's CPU path."""
    p = ol.default_params(window_size=200, shift=80, num_banks=20, sample_rate=8000.0, high_freq=4000.0, dyn="acc", norm=norm)
    x = synth_utterances(1, 28_800_000, seed=55, sr=8000.0)[0]
    ap = to_afe_params(p, BIG)
    b = afe.BatchMfcc(ap, 0, flags=afe.BATCH_Q1_EXACT)
    pcm, offs, lens = afe.pack_utterances([x])
    assert b.plan(offs, lens) == 359_998
    assert b.num_tiles >= 700
    got = b.run_host(np.concatenate([pcm, np.zeros(16, np.int16)]))
    launches = b.kernel_launches
    b.close()
    assert launches == 1                                          # also with CMN: no K2 / K3
    want = oracle_extract(oracle, p, [x], 1 << 25)[0]            # one set_input + flush (Q1), like the default driver
    assert_close(got, want, p, "1-hour stream " + norm)
    if norm != "none":
        u = run_batch(p, [x], flags=afe.BATCH_Q1_EXACT | afe.BATCH_UNFUSED_NORM)[0]
        np.testing.assert_array_equal(got, u)


def test_long_utterances_role_scheme_equals_unfused():
    """Batches with utterances of more than 8 tiles take the role scheme: bitwise equal to K2 + K3, repeatable, for every
    normalisation kind, mixed with short utterances, with Q1."""
    for norm in ("cmn", "cvn", "minmax"):
        p = ol.default_params(num_banks=40, norm=norm, dyn="acc")
        utts = synth_utterances(3, 900000, seed=41, ragged=True) + synth_utterances(10, 100000, seed=42, ragged=True) + \
            synth_utterances(1, 1500000, seed=43)
        for extra in (0, afe.BATCH_Q1_EXACT):
            a = run_batch(p, utts, flags=extra)
            a2 = run_batch(p, utts, flags=extra)
            c = run_batch(p, utts, flags=extra | afe.BATCH_UNFUSED_NORM)
            for i in range(len(utts)):
                np.testing.assert_array_equal(a[i], a2[i])
                np.testing.assert_array_equal(a[i], c[i])


# ---------------------------------------------------------------------------------------------- N > 1 on hardware
def _two_rank_worker(rank, world, port, q):
    """One process per GPU (torch.distributed only rendezvous): extract -> corpus record -> afe_normalizer_allreduce (NCCL) ->
    normalise, on a sample-balanced utterance shard."""
    import os
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    import afe_loader, oracle_lib as ol
    from common import synth_utterances, to_afe_params
    afe = afe_loader.load()
    try:
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        p = ol.default_params(num_banks=40, norm="cvn", dyn="acc")
        utts = synth_utterances(31, 64000, seed=77, ragged=True)
        lens_all = np.array([len(u) for u in utts], np.int64)
        starts = afe.shard_utterances(lens_all, world)
        mine = utts[starts[rank]:starts[rank + 1]]
        idb = [None]
        if rank == 0:
            raw = (C.c_char * 128)()
            afe._check(afe.lib().afe_nccl_get_unique_id(raw))
            idb = [bytes(raw.raw)]
        dist.broadcast_object_list(idb, 0)
        comm = C.c_void_p()
        afe._check(afe.lib().afe_nccl_comm_init(idb[0], world, rank, rank, C.byref(comm)))
        b = afe.BatchMfcc(to_afe_params(p, 1 << 22), rank, stats_scope=afe.STATS_CORPUS)
        pcm, offs, lens = afe.pack_utterances(mine)
        total = b.plan(offs, lens)
        d_pcm = afe.DeviceBuffer(pcm.nbytes + 64, rank); d_pcm.upload(pcm)
        d_out = afe.DeviceBuffer(total * 39 * 4, rank)
        b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
        b.corpus_stats()
        b.synchronize()
        local = b.corpus_record()
        b.allreduce(comm.value)
        b.synchronize()
        merged = b.corpus_record()
        b.normalize_device(d_out.ptr.value)
        b.synchronize()
        out = d_out.download((total, 39), np.float32)
        b.close(); d_pcm.free(); d_out.free()
        afe.lib().afe_nccl_comm_destroy(comm)
        q.put((rank, int(starts[rank]), int(starts[rank + 1]), local, merged, out))
        dist.destroy_process_group()
    except Exception as e:  # surfaces in the parent
        q.put((rank, "error", repr(e)))


def test_corpus_cmvn_nccl_two_gpus_equal_one():
    """SURVEY §4 pin 5 on hardware: 2 ranks over afe_nccl_* / afe_normalizer_allreduce on 2 GPUs == 1 GPU over the whole
    corpus, rows within 1e-6; the all-reduced record is sum / min / max of the local ones EXACTLY (catches a wrong NCCL
    reduction enum). Skipped unless >= 2 GPUs are visible."""
    if afe.lib().afe_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import multiprocessing as mp
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = [q.get(timeout=600) for _ in procs]
    for pr in procs:
        pr.join(60)
    for r in res:
        assert r[1] != "error", r
    res.sort(key=lambda r: r[0])
    w = 39
    l0, l1, m0, m1 = res[0][3], res[1][3], res[0][4], res[1][4]
    np.testing.assert_array_equal(m0, m1)
    np.testing.assert_array_equal(m0[:2 * w + 1], l0[:2 * w + 1] + l1[:2 * w + 1])       # ncclSum on doubles, 2 ranks: exact
    np.testing.assert_array_equal(m0[2 * w + 1:3 * w + 1], np.minimum(l0[2 * w + 1:3 * w + 1], l1[2 * w + 1:3 * w + 1]))
    np.testing.assert_array_equal(m0[3 * w + 1:], np.maximum(l0[3 * w + 1:], l1[3 * w + 1:]))
    # one GPU over the whole corpus
    p = ol.default_params(num_banks=40, norm="cvn", dyn="acc")
    utts = synth_utterances(31, 64000, seed=77, ragged=True)
    b = afe.BatchMfcc(to_afe_params(p, BIG), 0, stats_scope=afe.STATS_CORPUS)
    pcm, offs, lens = afe.pack_utterances(utts)
    total = b.plan(offs, lens)
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * 39 * 4)
    b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
    b.corpus_stats()
    b.normalize_device(d_out.ptr.value)
    b.synchronize()
    one = d_out.download((total, 39), np.float32)
    rec = b.corpus_record()
    b.close(); d_pcm.free(); d_out.free()
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == len(utts)
    two = np.concatenate([res[0][5], res[1][5]])
    assert rec[2 * w] == m0[2 * w]
    np.testing.assert_allclose(m0[:2 * w], rec[:2 * w], rtol=1e-13)
    np.testing.assert_array_equal(m0[2 * w + 1:], rec[2 * w + 1:])
    np.testing.assert_allclose(two, one, rtol=0, atol=1e-6)


# ---------------------------------------------------------------------------------------------- f4: one stream, sharded by time
def _run_stream_shard(p, x, sh, r, device=0, merged=None):
    """Rank r of a time-sharded stream on `device`: raw rows, record, (normalised rows when `merged` is given)."""
    b = afe.BatchMfcc(to_afe_params(p, BIG), device, stats_scope=afe.STATS_CORPUS)
    seg = np.ascontiguousarray(x[sh["sample_begin"][r]:sh["sample_begin"][r] + sh["sample_count"][r]])
    pcm, offs, lens = afe.pack_utterances([seg])
    total = b.plan_segments(offs, lens, [sh["local_first"][r]], [sh["count"][r]])
    assert total == sh["count"][r]
    w = ol.width_of(p)
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64, device); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * w * 4, device)
    b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
    rec = None
    if p["norm"]:
        b.corpus_stats(); b.synchronize()
        rec = b.corpus_record()
        if merged is not None:
            b.set_corpus_stats(merged)
            b.normalize_device(d_out.ptr.value)
    b.synchronize()
    out = d_out.download((total, w), np.float32)
    b.close(); d_pcm.free(); d_out.free()
    return out, rec


@pytest.mark.parametrize("norm", ["none", "cmn", "cvn"])
def test_stream_time_sharded_equals_whole_stream(oracle, norm):
    """SURVEY §8 f4: ONE stream cut by time into 3 'ranks' (afe_shard_stream: frames + D frames of real context per side),
    records merged like the all-reduce merges them. Without normalisation the rows are BITWISE those of the whole stream on one
    GPU (frames do not depend on the cut); with stream-level CMN / CVN they agree to a rounding of the statistics, and both
    match the reference's CPU classes (which see the stream in one block)."""
    x = np.concatenate([load_pcm()["a5"], load_pcm()["a3"], load_pcm()["a0001"]])      # 47.6 s of speech
    p = ol.default_params(norm=norm, dyn="acc")
    whole = run_batch(p, [x], stats_scope=afe.STATS_UTTERANCE)[0]                      # statistics over all rows, no Q1
    sh = afe.shard_stream(len(x), 400, 160, 6, 3)
    parts = [_run_stream_shard(p, x, sh, r) for r in range(3)]
    if norm == "none":
        np.testing.assert_array_equal(np.concatenate([o for o, _ in parts]), whole)
    else:
        w = 39
        recs = [rec for _, rec in parts]
        merged = np.concatenate([sum(r[:2 * w + 1] for r in recs), np.minimum.reduce([r[2 * w + 1:3 * w + 1] for r in recs]),
                                 np.maximum.reduce([r[3 * w + 1:] for r in recs])])
        assert merged[2 * w] == len(whole)
        got = np.concatenate([_run_stream_shard(p, x, sh, r, merged=merged)[0] for r in range(3)])
        np.testing.assert_allclose(got, whole, rtol=0, atol=2e-6 if norm == "cmn" else 2e-5)
    # and the whole-stream rows are the reference's (two set_input calls: no Q1; statistics over T - D rows there -> compare raw)
    if norm == "none":
        assert_close(whole, oracle_extract(oracle, p, [np.concatenate([x, np.zeros(3, np.int16)])], 0)[0], p, "whole stream")


def _stream_shard_worker(rank, world, port, q):
    import os
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    import afe_loader, oracle_lib as ol
    from common import synth_utterances
    afe = afe_loader.load()
    try:
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        p = ol.default_params(window_size=200, shift=80, num_banks=20, sample_rate=8000.0, high_freq=4000.0, dyn="acc", norm="cmn")
        x = synth_utterances(1, 2_400_000, seed=91, sr=8000.0)[0]                      # 5 minutes at 8 kHz
        sh = afe.shard_stream(len(x), 200, 80, 6, world)
        idb = [None]
        if rank == 0:
            raw = (C.c_char * 128)()
            afe._check(afe.lib().afe_nccl_get_unique_id(raw))
            idb = [bytes(raw.raw)]
        dist.broadcast_object_list(idb, 0)
        comm = C.c_void_p()
        afe._check(afe.lib().afe_nccl_comm_init(idb[0], world, rank, rank, C.byref(comm)))
        from common import to_afe_params
        b = afe.BatchMfcc(to_afe_params(p, 1 << 22), rank, stats_scope=afe.STATS_CORPUS)
        seg = np.ascontiguousarray(x[sh["sample_begin"][rank]:sh["sample_begin"][rank] + sh["sample_count"][rank]])
        pcm, offs, lens = afe.pack_utterances([seg])
        total = b.plan_segments(offs, lens, [sh["local_first"][rank]], [sh["count"][rank]])
        d_pcm = afe.DeviceBuffer(pcm.nbytes + 64, rank); d_pcm.upload(pcm)
        d_out = afe.DeviceBuffer(total * 39 * 4, rank)
        b.extract_device(d_pcm.ptr.value, d_out.ptr.value)
        b.corpus_stats()
        b.allreduce(comm.value)
        b.normalize_device(d_out.ptr.value)
        b.synchronize()
        out = d_out.download((total, 39), np.float32)
        b.close(); d_pcm.free(); d_out.free()
        afe.lib().afe_nccl_comm_destroy(comm)
        q.put((rank, out))
        dist.destroy_process_group()
    except Exception as e:
        q.put((rank, "error", repr(e)))


def test_stream_time_sharded_nccl_two_gpus():
    """f4 on hardware: a 5-minute 8 kHz stream cut in two, one half per GPU, stream-level CMN through afe_normalizer_allreduce
    == the whole stream on one GPU within 1e-6. Skipped unless >= 2 GPUs are visible."""
    if afe.lib().afe_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import multiprocessing as mp
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_stream_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = [q.get(timeout=600) for _ in procs]
    for pr in procs:
        pr.join(60)
    for r in res:
        assert r[1] is not None and not (isinstance(r[1], str) and r[1] == "error"), r
    res.sort(key=lambda r: r[0])
    p = ol.default_params(window_size=200, shift=80, num_banks=20, sample_rate=8000.0, high_freq=4000.0, dyn="acc", norm="cmn")
    x = synth_utterances(1, 2_400_000, seed=91, sr=8000.0)[0]
    whole = run_batch(p, [x], stats_scope=afe.STATS_UTTERANCE)[0]
    np.testing.assert_allclose(np.concatenate([res[0][1], res[1][1]]), whole, rtol=0, atol=1e-6)
