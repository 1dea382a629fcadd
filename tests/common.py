"""Shared helpers for the parity tests."""
import numpy as np

import afe_loader
import oracle_lib as ol

afe = afe_loader.load()


def to_afe_params(p, input_buffer_size):
    """oracle parameter dict (oracle_lib.default_params) -> afe_params"""
    q = {k: v for k, v in p.items() if k != "alpha"}
    return afe.make_params(input_buffer_size=input_buffer_size, **q)


def synth_utterances(n_utts, n_samples, seed=1234, sr=16000.0, ragged=False):
    """SURVEY §8(d) config-3 generator: x = clip(round(3000*N(0,1) + 8000*sin(2*pi*f_u*t)), +-32767), f_u ~ U[100, 3800]."""
    rng = np.random.default_rng(seed)
    out = []
    for u in range(n_utts):
        n = n_samples if not ragged else int(rng.integers(n_samples // 3, n_samples + 1))
        f = rng.uniform(100.0, 3800.0)
        t = np.arange(n) / sr
        x = 3000.0 * rng.standard_normal(n) + 8000.0 * np.sin(2 * np.pi * f * t)
        out.append(np.clip(np.round(x), -32767, 32767).astype(np.int16))
    return out


def tolerances(p):
    """Stated floating-point tolerances (SURVEY §7): max |gpu - oracle| per stream.

    fp32 FFT + fused multiply-adds vs the oracle's fp32 radix-2 shim and unfused libm path; c0 is ~ -80..-90 so 1 ulp
    there is 7.6e-6. The oracle's own libm-flavour noise floor is 3e-5 .. 4e-5 (float vs double libm, SURVEY Q11)."""
    if p["norm"] == ol.NORM["cvn"]:
        return dict(static=1e-3, delta=1e-3)
    if p["norm"] == ol.NORM["minmax"]:
        return dict(static=2e-4, delta=2e-4)
    return dict(static=5e-4, delta=2e-4)


def assert_close(got, want, p, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    cols = ol.cols_of(p)
    tol = tolerances(p)
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    assert np.isfinite(got).all(), what
    e_static = err[:, :cols].max() if err.size else 0.0
    e_dyn = err[:, cols:].max() if err.shape[1] > cols else 0.0
    rel = (err / np.maximum(np.abs(want), 1.0)).max() if err.size else 0.0
    assert e_static <= tol["static"], f"{what}: static max-abs {e_static:.3g} > {tol['static']}"
    assert e_dyn <= tol["delta"], f"{what}: delta max-abs {e_dyn:.3g} > {tol['delta']}"
    assert rel <= 2e-4 or p["norm"] in (ol.NORM["cvn"],), f"{what}: max rel {rel:.3g}"
    return e_static, e_dyn


def compare(got, want, p, what):
    """assert_close, except that where the REFERENCE is not finite (MINMAX / CVN over a constant column, e.g. an empty filter
    or a silent utterance: scale = 1/0) the result only has to be non-finite in the same places."""
    bad = ~np.isfinite(want)
    if bad.any():
        assert got.shape == want.shape, (what, got.shape, want.shape)
        assert np.array_equal(bad, ~np.isfinite(got)), f"{what}: non-finite entries differ from the reference's"
        got, want = np.where(bad, 0.0, got).astype(np.float32), np.where(bad, 0.0, want).astype(np.float32)
    return assert_close(got, want, p, what)


def run_batch(p, utts, stats_scope=0, flags=0, alpha=None, host=True):
    """Features of a list of utterances through the fused batch path; returns list of [T,width] arrays."""
    ap = to_afe_params(p, 1 << 22)
    b = afe.BatchMfcc(ap, 0, stats_scope=stats_scope, flags=flags, alpha=p.get("alpha", 1.0) if alpha is None else alpha)
    try:
        pcm, offs, lens = afe.pack_utterances(utts)
        b.plan(offs, lens)
        out = b.run_host(np.concatenate([pcm, np.zeros(16, np.int16)]))
        fo = b.frame_offsets
        return [out[fo[i]:fo[i + 1]] for i in range(len(utts))]
    finally:
        b.close()


def ref_alpha_sweep(oracle, pcm, p, limit, alphas):
    """The reference driver's VTLN sweep (ASR_OCL.cpp:227-301) on the reference's own objects: per block ONE set_input, then
    set_alpha -> apply -> get_output_data per alpha (so the flush block is normalised with the LAST alpha's statistics).
    -> list of [T, width] arrays, one per alpha."""
    ref = ol.RefMfcc(oracle, limit, p)
    ref.set_window(oracle.window(p["window_size"]))
    n = ref.get_input_buffer_size()
    rows = [[] for _ in alphas]

    def emit(wc):
        for k, a in enumerate(alphas):
            ref.set_alpha(a)
            ref.apply()
            rows[k].append(ref.get_output_data(wc))
    for pos in range(0, len(pcm), n):
        wc = ref.set_input(pcm[pos:pos + n])
        if wc > 0:
            emit(wc)
    wc = ref.flush()
    if wc > 0:
        emit(wc)
    ref.close()
    return [np.concatenate(r) for r in rows]
