"""Device-resident throughput of 1024-point FFTs (windows of 513..1024 samples) through the fused kernel K1, next to config 3.

One GPU, one process. Every arm runs N seeded synthetic 10 s utterances at its sample rate (the config-3 generator), PCM
and features resident on the device (afe_batch_run_device), timed with CUDA events over --steps steps after --warmup
steps. Arms, alternated --reps times:
  config3        16 kHz, W=400, S=160, 512 points, 40 banks, 12 + c0 + delta + delta-delta, CMN: the reference point
  mfcc22k        22.05 kHz, W=551, S=220, 40 banks, 12 + c0 + delta + delta-delta, CMN (S % 8 != 0: plain staging)
  logmel80_24k   24 kHz, W=600, S=240, 80-band log-mel, CMN
  tts80_22k      22.05 kHz, W=1024, S=256, 80-band log-mel to 8 kHz, no normalisation (unpruned first FFT layer)
  mfcc32k        32 kHz, W=800, S=320, 64 banks, 12 + c0 + delta + delta-delta, CVN
Prints one JSON line (also written to --out when given) with frames/s and audio-hours/s per arm; the card's name and
power limit are read with nvidia-smi in the same run. Nothing is written elsewhere.

    python tools/fft1024_bench.py [--utts 10000] [--steps 10] [--warmup 2] [--reps 2] [--arms config3,mfcc22k,...] [--out F]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (the config-3 geometry and its device-side PCM generator)


def geom(sr, W, S, nb, hi):
    return dict(sr=sr, W=W, S=S, nb=nb, hi=hi, n=10 * sr)


# arm -> (geometry, parameter overrides)
ARMS = {
    "config3": (bench.CFG16, dict(norm=1)),
    "mfcc22k": (geom(22050, 551, 220, 40, 11025.0), dict(norm=1)),
    "logmel80_24k": (geom(24000, 600, 240, 80, 12000.0), dict(norm=1, ceps_len=0, want_c0=0, dyn=0)),
    "tts80_22k": (geom(22050, 1024, 256, 80, 8000.0), dict(norm=0, ceps_len=0, want_c0=0, dyn=0)),
    "mfcc32k": (geom(32000, 800, 320, 64, 16000.0), dict(norm=2)),
}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip()


def width_of(p):
    cols = p["ceps_len"] + p["want_c0"] if p["ceps_len"] > 0 else p["num_banks"]
    return cols * (1, 2, 3)[p["dyn"]]


def time_arm(torch, afe, name, n_utts, steps, warmup, stream):
    g, kw = ARMS[name]
    p = bench.params_dict(g, norm=kw.get("norm", 1))
    p.update(kw)
    pcm = bench.synth_device(torch, "cuda", n_utts, g, seed=1234)
    n = g["n"]
    offs = np.arange(n_utts, dtype=np.int64) * n
    lens = np.full(n_utts, n, np.int64)
    T = bench.frames_of(n, g)
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
        res = dict(kernel=b.kernel_name, tiles=b.num_tiles, launches=b.kernel_launches, W=g["W"], S=g["S"], sr=g["sr"],
                   width=w, ms_per_step=round(ms, 4), frames_per_s=n_utts * T / (ms * 1e-3),
                   audio_hours_per_s=n_utts * n / g["sr"] / 3600.0 / (ms * 1e-3))
    finally:
        b.close()
    assert torch.isfinite(out[: min(out.numel(), 1 << 24)]).all().item()
    del out, pcm
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--arms", default=",".join(ARMS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    names = args.arms.split(",")
    assert names[0] == "config3" and all(n in ARMS for n in names), "arms: config3 first, then any of " + ", ".join(ARMS)

    import torch
    import afe_loader
    afe = afe_loader.load()
    if not torch.cuda.is_available() or afe.lib().afe_device_count() < 1:
        sys.exit("fft1024_bench: needs a CUDA device")
    stream = torch.cuda.Stream()
    arms = {k: [] for k in names}
    for _ in range(args.reps):
        for name in names:
            arms[name].append(time_arm(torch, afe, name, args.utts, args.steps, args.warmup, stream))
    summary = {}
    for name, runs in arms.items():
        v = [r["frames_per_s"] for r in runs]
        best = runs[int(np.argmax(v))]
        summary[name] = dict(best, frames_per_s=round(max(v)), frames_per_s_runs=[round(x) for x in v],
                             audio_hours_per_s=round(best["audio_hours_per_s"], 2),
                             spread=round((max(v) - min(v)) / max(v), 4), ms_per_step=min(r["ms_per_step"] for r in runs))
    base = summary["config3"]["frames_per_s"]
    for name in names:
        summary[name]["vs_config3"] = round(summary[name]["frames_per_s"] / base, 3)
    line = dict(
        tool="tools/fft1024_bench.py", card=card(),
        workload=f"{args.utts} synthetic 10 s utterances per arm at the arm's sample rate (seed 1234, the config-3 "
                 f"generator), device-resident, {args.steps} timed steps after {args.warmup} warm-up, {args.reps} "
                 f"alternating repetitions (best reported, spread = (max - min) / max)",
        unit="frames/s", arms=summary)
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
