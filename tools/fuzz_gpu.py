#!/usr/bin/env python
"""Randomised parity sweep on a GPU box: random parameter sets (window / shift / FFT size, filterbank, cepstra or log-mel,
regression widths, normalisation kind and order, VTLN alpha, pre-set block sizes) x ragged utterances, the fused batch path and
the streaming object against the reference's own CPU classes (oracle/_ref, or the C port). The fixed cases live in tests/; this
looks for parameter corners they do not name. Usage (under gpurun): python tools/fuzz_gpu.py [n_cases] [seed]
`python tools/fuzz_gpu.py schemes [n] [seed]`: bitwise equality of the normalisation / staging routes on random ragged batches.
Prints one line per failure and a summary; exit code 1 when any case is out of tolerance."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as ol  # noqa: E402
from common import afe, compare, run_batch, synth_utterances, to_afe_params  # noqa: E402


def random_params(rng):
    sr = float(rng.choice([8000.0, 16000.0, 16000.0, 22050.0, 24000.0, 32000.0]))
    W = int(rng.choice([200, 256, 320, 400, 401, 480, 512, 150, 130]))
    if sr == 8000.0:
        W = min(W, 256) if rng.random() < 0.7 else W
    if sr > 16000.0:  # 1024-point FFTs: 25 ms windows and the 1024 / 256 TTS shape
        W = int(rng.choice([513, 551, 600, 800, 832, 833, 1000, 1024]))
    S = int(rng.integers(max(2, W // 5), W // 2 + 1))
    if rng.random() < 0.85:
        S -= S % 2
    nb = int(rng.choice([8, 12, 20, 23, 24, 26, 32, 40, 41, 48, 64, 72, 80, 96, 128]))
    ceps = int(rng.choice([0, 8, 12, 12, 12, 13, 15, 16, 19, 23, 29, 39, 40, 47]))
    if W > 512:
        ceps = min(ceps, 15)  # the batch extractor serves up to 16 columns at 1024 points
    c0 = int(rng.integers(0, 2))
    dyn = int(rng.integers(0, 3))
    cols = ceps + c0 if ceps > 0 else nb
    if cols * (dyn + 1) > 128:
        dyn = 0 if cols > 64 else 1
    return ol.default_params(window_size=W, shift=S, num_banks=nb, sample_rate=sr, low_freq=float(rng.choice([0.0, 64.0, 120.0])),
                             high_freq=float(sr / 2 * rng.choice([1.0, 0.95, 0.85])), ceps_len=ceps, want_c0=c0,
                             lift_coef=float(rng.choice([22.0, 1.0, 16.0])) if ceps > 0 else 22.0,  # 0 divides by zero in the reference (mfcccpu.cpp:127)
                             norm=int(rng.integers(0, 4)), dyn=dyn, delta_l1=int(rng.integers(1, 5)), delta_l2=int(rng.integers(1, 5)),
                             norm_after_dyn=int(rng.random() < 0.75), alpha=float(rng.choice([1.0, 1.0, 0.9, 1.08])))


def reference_blocking_is_memory_safe(p, n, limit):
    """The reference's SegmenterCPU copies carry-over + block into a buffer of (est(limit) + 2 [+ 3D]) * S + W - S samples without
    a bound check (segmentercpu.cpp:41,76-78): for some (W, S, limit) the second block overruns it. This library throws "buffer is
    too small" there; the oracle would corrupt its heap, so such blockings are not compared."""
    W, S = p["window_size"], p["shift"]
    D = p["delta_l1"] + p["delta_l2"] if p["dyn"] else 0
    est = lambda m: int(np.floor(np.float32(m - (W - S)) / np.float32(S)))
    cap = (est(limit) + 2 + (3 * D if p["dyn"] else 0)) * S + W - S
    pos, remaining, first = 0, 0, True
    while pos < n:
        m = min(limit, n - pos)
        if first:
            wc = est(m) - D
            if wc <= 0 or wc < D or m > cap:
                return False
            remaining = m - ((wc - D) * S + W - S) + W - S
            first = False
        else:
            if remaining + m > cap:
                return False
            total = remaining + m
            wc = max(0, est(total) - 2 * D)
            remaining = total - (wc * S + W - S) + W - S
        pos += m
    return True


def isolated(fn, *args):
    """Run an oracle call in a forked child: the reference has heap overruns of its own on odd parameter sets (Q4 and the
    one above); a child that dies or hangs means 'the reference cannot answer', not a parity failure."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    parent, child = ctx.Pipe(duplex=False)

    def work():
        try:
            child.send(("ok", fn(*args)))
        except Exception as e:  # noqa: BLE001
            child.send(("err", str(e)))
    pr = ctx.Process(target=work)
    pr.start()
    child.close()
    res = parent.recv() if parent.poll(120) else ("dead", "no answer")
    pr.join(5)
    if pr.is_alive():
        pr.kill()
    if pr.exitcode not in (0, None) and res[0] == "ok":
        res = ("dead", f"exit code {pr.exitcode}")
    if res[0] != "ok":
        raise RuntimeError(res[1])
    return res[1]


def schemes(n_cases, seed):
    """Internal consistency: the same random batch (ragged lengths from the minimum to 30 s, so clusters of 1-4 tiles, the ticket
    scheme and the role scheme all occur) through every normalisation route and staging path must give the SAME BITS."""
    rng = np.random.default_rng(seed)
    fails, done, skipped = [], 0, 0
    for case in range(n_cases):
        p = random_params(rng)
        p["norm"] = int(rng.integers(1, 4))
        if p["shift"] % 2:
            p["shift"] += 1
        D = p["delta_l1"] + p["delta_l2"] if p["dyn"] else 0
        n_min = p["window_size"] + p["shift"] * (2 * D + 4)
        lens = [n_min, int(rng.integers(n_min, 20000)), int(rng.integers(20000, 200000)), int(rng.integers(100000, 480000)),
                int(rng.integers(n_min, 60000)), int(rng.integers(200000, 330000))]
        rng.shuffle(lens)
        utts = [synth_utterances(1, n, seed=5000 + 10 * case + i, sr=p["sample_rate"])[0] for i, n in enumerate(lens)]
        scope = int(rng.integers(0, 2))
        try:
            base = run_batch(p, utts, stats_scope=scope)
            for name, fl in (("no_cluster", afe.BATCH_NO_CLUSTER), ("unfused", afe.BATCH_UNFUSED_NORM), ("no_tma", afe.BATCH_NO_TMA),
                             ("q1", afe.BATCH_Q1_EXACT)):
                other = run_batch(p, utts, stats_scope=scope, flags=fl)
                for i, (a, b) in enumerate(zip(base, other)):
                    same = np.array_equal(a, b, equal_nan=True) if name != "q1" else np.array_equal(a[:max(0, len(a) - D)], b[:max(0, len(b) - D)], equal_nan=True)
                    if not same:
                        fails.append(f"schemes case {case} {name} utt {i} (len {lens[i]}) differs: {p}")
            done += 1
        except afe.AfeError as e:
            if "fused path" in str(e) or "mel filter" in str(e) or "window" in str(e):
                skipped += 1
            else:
                fails.append(f"schemes case {case}: {e} {p}")
    for f in fails:
        print("FAIL", f)
    print(f"fuzz schemes: {done} batches x 5 routes, {skipped} skipped, {len(fails)} failures, seed {seed}")
    return 1 if fails else 0


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "schemes":
        return schemes(int(sys.argv[2]) if len(sys.argv) > 2 else 60, int(sys.argv[3]) if len(sys.argv) > 3 else 11)
    n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 120
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    oracle = ol.RefLib("ref" if ol.available("ref") else "port")
    fails, skipped, done, worst = [], 0, 0, 0.0
    for case in range(n_cases):
        p = random_params(rng)
        D = p["delta_l1"] + p["delta_l2"] if p["dyn"] else 0
        n_min = p["window_size"] + p["shift"] * (2 * D + 4)
        utts = synth_utterances(3, int(rng.integers(n_min + 4000, 60000)), seed=1000 + case, sr=p["sample_rate"], ragged=False)
        utts[1] = utts[1][:max(n_min, len(utts[1]) // 3)]
        utts[2] = utts[2][:n_min]                                       # the shortest utterance the path accepts
        edges, _ = afe.build_filters(to_afe_params(p, 1 << 22), p["alpha"])
        if np.any(np.diff(edges) <= 0):
            # more filters than bins: empty filters give log(1e-30) = -69 and cepstra of +-50, where the reference's own float /
            # double flavours already differ by 2.6e-4 (absolute tolerances are stated for speech-range features)
            skipped += 1
            continue
        tag = f"case {case} {dict((k, p[k]) for k in ('window_size', 'shift', 'num_banks', 'sample_rate', 'ceps_len', 'want_c0', 'norm', 'dyn', 'delta_l1', 'delta_l2', 'norm_after_dyn', 'alpha'))}"
        try:
            want = isolated(lambda: oracle.extract(p, utts, sample_limit=1 << 22)[0])
        except Exception as e:  # the reference itself rejects the set (or dies on it)
            skipped += 1
            continue
        # (a) fused batch path, single block + flush semantics
        try:
            got = run_batch(p, utts, flags=afe.BATCH_Q1_EXACT)
            for i, (g, w) in enumerate(zip(got, want)):
                e = compare(g, w, p, f"{tag} batch utt {i}")
                worst = max(worst, e[0], e[1])
            done += 1
        except afe.AfeError as e:
            if "fused path" in str(e) or "mel filter" in str(e) or "window" in str(e):
                skipped += 1
            else:
                fails.append(f"{tag}: batch error {e}")
        except AssertionError as e:
            fails.append(str(e))
        # (b) streaming object, blocks of `limit` samples
        limit = int(rng.choice([1 << 22, 16000, 30011]))
        if not reference_blocking_is_memory_safe(p, len(utts[0]), limit):
            skipped += 1
            continue
        try:
            want_s = isolated(lambda: oracle.extract(p, utts[:1], sample_limit=limit)[0][0])
            got_s = afe.extract_stream(to_afe_params(p, limit), utts[0], alpha=p["alpha"])
            e = compare(got_s, want_s, p, f"{tag} stream limit {limit}")
            worst = max(worst, e[0], e[1])
            done += 1
        except afe.AfeError as e:
            fails.append(f"{tag}: stream error {e}")
        except AssertionError as e:
            fails.append(str(e))
        except Exception as e:  # the reference rejects the blocking (e.g. first block too short)
            skipped += 1
    for f in fails:
        print("FAIL", f)
    print(f"fuzz: {done} comparisons, {skipped} skipped, {len(fails)} failures, worst max-abs {worst:.3g}, seed {seed}, oracle {oracle.kind}")
    return 1 if fails else 0


if __name__ == "__main__":
    sys.exit(main())
