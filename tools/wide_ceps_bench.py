"""Device-resident throughput of wide DCTs (ceps_len + c0 = 17..48) through the fused kernel K1, next to config 3.

One GPU, one process. Every arm runs the config-3 shape: N seeded synthetic 10 s utterances at 16 kHz (W=400, S=160,
512-point FFT), PCM and features resident on the device, per-utterance CMN inside K1 (afe_batch_run_device), timed with
CUDA events over --steps steps after --warmup steps. Arms, alternated --reps times:
  config3        40 banks, 12 cepstra + c0, delta + delta-delta (39 columns): the reference point
  hires40        40 banks, 39 cepstra + c0, no deltas (40 columns): high-resolution MFCC
  hires40_acc    40 banks, 40 cepstra + c0, delta + delta-delta (123 columns)
  mfcc20_acc     40 banks, 20 cepstra + c0, delta + delta-delta (63 columns), CVN instead of CMN
Then hires40 through the streaming object on --stream-utts of the utterances (0: skipped), host to host, once on the
staged kernels (AFE_OPT_STAGED_KERNELS, the route such parameter sets took before K1 covered them) and once on K1.
Prints one JSON line (also written to --out when given); the card's name and power limit are read with nvidia-smi in
the same run. Nothing is written elsewhere.

    python tools/wide_ceps_bench.py [--utts 10000] [--steps 10] [--warmup 2] [--reps 2] [--stream-utts 256]
                                    [--arms config3,hires40,...] [--out F]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (the config-3 geometry and its device-side PCM generator)

G = bench.CFG16
ARMS = {
    "config3": dict(num_banks=40),
    "hires40": dict(num_banks=40, ceps_len=39, want_c0=1, dyn=0),
    "hires40_acc": dict(num_banks=40, ceps_len=40, want_c0=1),
    "mfcc20_acc": dict(num_banks=40, ceps_len=20, want_c0=1, norm=2),
}


def params(**kw):
    p = bench.params_dict(G, norm=1)
    p.update(kw)
    return p


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip()


def width_of(p):
    cols = p["ceps_len"] + p["want_c0"] if p["ceps_len"] > 0 else p["num_banks"]
    return cols * (1, 2, 3)[p["dyn"]]


def time_arm(torch, afe, p, pcm, offs, lens, n_utts, steps, warmup, stream):
    T = bench.frames_of(G["n"], G)
    w = width_of(p)
    out = torch.empty((n_utts * T * w,), dtype=torch.float32, device="cuda")
    q = {k: v for k, v in p.items() if k != "alpha"}
    b = afe.BatchMfcc(afe.make_params(input_buffer_size=1 << 22, **q), 0)
    try:
        b.set_stream(stream.cuda_stream)
        assert b.plan(offs, lens) == n_utts * T
        for _ in range(warmup):
            b.run_device(pcm.data_ptr(), out.data_ptr())
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(stream)
        for i in range(steps):
            b.run_device(pcm.data_ptr(), out.data_ptr())
            ev[i + 1].record(stream)
        stream.synchronize()
        ms = ev[0].elapsed_time(ev[-1]) / steps
        res = dict(kernel=b.kernel_name, tiles=b.num_tiles, launches=b.kernel_launches, width=w, ms_per_step=round(ms, 4),
                   frames_per_s=n_utts * T / (ms * 1e-3))
    finally:
        b.close()
    assert torch.isfinite(out[: min(out.numel(), 1 << 24)]).all().item()
    del out
    return res


def time_stream(afe, p, utts, staged):
    q = {k: v for k, v in p.items() if k != "alpha"}
    ap = afe.make_params(input_buffer_size=G["n"], **q)
    afe.extract_stream(ap, utts[0], staged=staged)                      # warm-up (module load, allocations)
    t0 = time.perf_counter()
    frames = sum(len(afe.extract_stream(ap, u, staged=staged)) for u in utts)
    dt = time.perf_counter() - t0
    return dict(utterances=len(utts), frames=frames, seconds=round(dt, 4), frames_per_s=frames / dt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--stream-utts", type=int, default=256)
    ap.add_argument("--arms", default=",".join(ARMS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    names = args.arms.split(",")
    assert names[0] == "config3" and all(n in ARMS for n in names), "arms: config3 first, then any of " + ", ".join(ARMS)

    import torch
    import afe_loader
    afe = afe_loader.load()
    if not torch.cuda.is_available() or afe.lib().afe_device_count() < 1:
        sys.exit("wide_ceps_bench: needs a CUDA device")
    n = G["n"]
    pcm = bench.synth_device(torch, "cuda", args.utts, G, seed=1234)
    offs = np.arange(args.utts, dtype=np.int64) * n
    lens = np.full(args.utts, n, np.int64)
    stream = torch.cuda.Stream()
    arms = {k: [] for k in names}
    for _ in range(args.reps):
        for name in names:
            kw = ARMS[name]
            arms[name].append(time_arm(torch, afe, params(**kw), pcm, offs, lens, args.utts, args.steps, args.warmup, stream))
    summary = {}
    for name, runs in arms.items():
        v = [r["frames_per_s"] for r in runs]
        summary[name] = dict(runs[0], frames_per_s=max(v), frames_per_s_runs=[round(x) for x in v],
                             spread=round((max(v) - min(v)) / max(v), 4), ms_per_step=min(r["ms_per_step"] for r in runs))
        summary[name]["frames_per_s"] = round(summary[name]["frames_per_s"])
    base = summary["config3"]["frames_per_s"]
    for name in names:
        summary[name]["vs_config3"] = round(summary[name]["frames_per_s"] / base, 3)
    k = min(args.stream_utts, args.utts)
    line = dict(
        tool="tools/wide_ceps_bench.py", card=card(),
        workload=f"{args.utts} synthetic 10 s utterances at 16 kHz (seed 1234, the config-3 generator), W=400/S=160, "
                 f"512-point FFT, per-utterance CMN (mfcc20_acc: CVN), device-resident, {args.steps} timed steps after "
                 f"{args.warmup} warm-up, {args.reps} alternating repetitions (best reported, spread = (max - min) / max)",
        unit="frames/s", arms=summary)
    if k > 0:
        utts = pcm[: k * n].view(k, n).cpu().numpy()
        del pcm
        hires = params(**ARMS["hires40"])
        stream_staged = time_stream(afe, hires, list(utts), staged=True)
        stream_fused = time_stream(afe, hires, list(utts), staged=False)
        line["stream_hires40"] = dict(note=f"streaming object, one 10 s utterance per stream, host to host, {k} utterances",
                                      staged_kernels=stream_staged, fused_k1=stream_fused,
                                      k1_over_staged=round(stream_fused["frames_per_s"] / stream_staged["frames_per_s"], 2))
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
