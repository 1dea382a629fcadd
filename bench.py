#!/usr/bin/env python
"""bench.py — MFCC + delta + delta-delta feature frames/s on B200 (BASELINE.json metric).

A "step" = one pass of the hot path over one shard of synthetic PCM. `--config` picks the BASELINE.json configuration the
headline line is quoted on (default 3 = configs[2], the one the metric names); the other two travel in the same line as
"extra" blocks so that the driver's BENCH / SCALE records carry them:

  3  configs[2]: 10 000 utterances x 10 s of 16 kHz PCM per GPU, 40 mel, 13 MFCC + delta + delta-delta, per-utterance CMN
     (one launch of k_fused_mfcc per step; utterance-sharded, weak scaling, no data-path collective)
  4  configs[3]: 1000 audio-hours = 360 000 such utterances sharded over the GPUs, CORPUS-level CMVN: extract ->
     corpus record -> ONE NCCL all-reduce inside the Normalizer (afe_normalizer_allreduce) -> normalise. As an extra block
     (and at N = 1) every GPU takes the 45 000-utterance shard of the 8-GPU case.
  5  configs[4]: ONE 8 kHz stream of 28 800 000 samples (1 hour), 256-point FFT, 20 mel, fused deltas, without and with CMN
     (single GPU path: replicas at N > 1)

  value     whole-job frames/s with PCM and features resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e       same metric through the C-ABI call with HOST buffers (afe_batch_run_host: H2D PCM + kernels + D2H features), and
            its fraction of this box's measured copy ceiling (the same bytes moved with plain cudaMemcpyAsync, no kernels)
  roofline  the one kernel of the step (k_fused_mfcc): algorithmic bytes (2*S + 4*width per frame) / its event time,
            against MEASURED_PEAKS.json hbm_gbs
  parity    64 utterances of the TIMED output against the reference's own CPU classes (oracle/_ref), max abs / rel error
  cpu_baseline  the reference's CPU path on this box's host cores, bounded sample, with the FFT shim's cost per transform
  stream_object the drop-in ParamBase object (MfccCuda) on 10 s files: one handle, and several handles from host threads

`--impl reference` times that CPU path alone (no CUDA) and prints the same line with "impl": "reference".
`--dump-outputs DIR` writes the features of the last timed step (a fixed sample of utterances) to DIR/features.npy, so that
two builds can be compared output for output on identical inputs.
torch is used for device memory, streams, events and torch.distributed only; all compute is libafe_cuda.so.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "mfcc_delta_delta2_frames_per_s"
UNIT = "frames/s"
WIDTH = 39

# name -> geometry of the BASELINE configurations (SURVEY §8d)
CFG16 = dict(sr=16000, W=400, S=160, nb=40, hi=8000.0, n=160000)      # configs[2] and [3]: 10 s utterances
CFG8 = dict(sr=8000, W=200, S=80, nb=20, hi=4000.0, n=28_800_000)    # configs[4]: one 1-hour stream


def params_dict(g=CFG16, norm=1):
    return dict(window_size=g["W"], shift=g["S"], num_banks=g["nb"], sample_rate=float(g["sr"]), low_freq=64.0,
                high_freq=g["hi"], ceps_len=12, want_c0=1, lift_coef=22.0, norm=norm, dyn=2, delta_l1=3, delta_l2=3,
                norm_after_dyn=1, alpha=1.0)


def frames_of(n, g):
    return (n - (g["W"] - g["S"])) // g["S"]


def workload_config(config, n_utts, n_gpus):
    g = CFG16
    T = frames_of(g["n"], g)
    if config == 3:
        return {"workload": f"BASELINE configs[2]: synthetic 16 kHz PCM, {n_utts} utterances x 10 s per GPU, "
                            f"W=400/S=160, 512-pt FFT, 40 mel, 13 MFCC(12+c0)+delta+delta-delta (39-dim), per-utterance CMN",
                "utterances_per_gpu": n_utts, "samples_per_utterance": g["n"], "frames_per_gpu": n_utts * T,
                "sharding": f"utterance-sharded x{n_gpus}, no data-path collective",
                "l2_policy": f"inputs ({n_utts * g['n'] * 2 / 1e9:.2f} GB PCM + {n_utts * T * WIDTH * 4 / 1e9:.2f} GB "
                             "features per GPU) are larger than L2 (126 MB); no explicit flush"}
    if config == 4:
        return {"workload": f"BASELINE configs[3]: synthetic 1000 audio-hours (360 000 utterances x 10 s, 16 kHz) utterance-sharded, "
                            f"{n_utts} utterances per GPU x {n_gpus} GPU(s), 40 mel, 39-dim, CORPUS CMVN via one NCCL all-reduce",
                "utterances_per_gpu": n_utts, "samples_per_utterance": g["n"], "frames_per_gpu": n_utts * T,
                "sharding": f"utterance-sharded x{n_gpus}; one collective: ncclAllReduce x3 grouped on 157 doubles",
                "l2_policy": "inputs per GPU are larger than L2 (126 MB); no explicit flush"}
    g = CFG8
    return {"workload": "BASELINE configs[4]: ONE synthetic 8 kHz stream of 28 800 000 samples (1 hour), W=200/S=80, 256-pt FFT, "
                        "20 mel, 13 MFCC+delta+delta-delta fused",
            "utterances_per_gpu": 1, "samples_per_utterance": g["n"], "frames_per_gpu": frames_of(g["n"], g),
            "sharding": "one stream per GPU (replicas at N > 1)",
            "l2_policy": "57.6 MB PCM + 56.2 MB features fit in L2 (126 MB): a 256 MB buffer is written between timed iterations"}


def synth_host(n_utts, seed, g=CFG16):
    """SURVEY §8(d) generator on the host (used by the CPU arm)."""
    rng = np.random.default_rng(seed)
    n, sr = g["n"], g["sr"]
    t = np.arange(n) / sr
    out = np.empty((n_utts, n), np.int16)
    for u in range(n_utts):
        f = rng.uniform(100.0, 3800.0)
        x = 3000.0 * rng.standard_normal(n).astype(np.float32) + 8000.0 * np.sin(2 * np.pi * f * t)
        out[u] = np.clip(np.round(x), -32767, 32767).astype(np.int16)
    return out


def synth_device(torch, dev, n_utts, g, seed, extra=64):
    """The same generator on the device (plumbing): int16 [n_utts * n + extra]."""
    n, sr = g["n"], g["sr"]
    gen = torch.Generator(device=dev); gen.manual_seed(seed)
    pcm = torch.empty((n_utts * n + extra,), dtype=torch.int16, device=dev)
    pcm[n_utts * n:] = 0
    per = max(1, min(n_utts, (1 << 26) // n))            # <= 64 M samples of fp32 scratch at a time
    if n > (1 << 26):
        per = 1
    for u0 in range(0, n_utts, per):
        c = min(per, n_utts - u0)
        f = torch.empty((c, 1), device=dev).uniform_(100.0, 3800.0, generator=gen)
        for s0 in range(0, n, 1 << 24):                   # long streams in 16 M-sample pieces
            s1 = min(n, s0 + (1 << 24))
            t = torch.arange(s0, s1, device=dev, dtype=torch.float32) / sr
            x = 3000.0 * torch.randn((c, s1 - s0), device=dev, generator=gen) + 8000.0 * torch.sin(2 * np.pi * f * t)
            x = x.round_().clamp_(-32767, 32767).to(torch.int16)
            if c == 1:
                pcm[u0 * n + s0:u0 * n + s1] = x.reshape(-1)
            else:
                pcm[u0 * n:(u0 + c) * n].view(c, n)[:, s0:s1] = x
            del x
    return pcm


# ---------------------------------------------------------------------------------------------------------- CPU arm
def shim_us_per_transform(n2, rows=4096):
    """Cost of the FFT the CPU arm runs: oracle/fftw_shim.c (FFTW itself is not installed, BASELINE.md §3), one r2c row."""
    try:
        import oracle_lib as ol
        kind = "ref" if ol.available("ref") else "port"
        L = C.CDLL(ol._PATHS[kind])
        L.fftwf_alloc_real.restype = C.c_void_p; L.fftwf_alloc_real.argtypes = [C.c_size_t]
        L.fftwf_alloc_complex.restype = C.c_void_p; L.fftwf_alloc_complex.argtypes = [C.c_size_t]
        L.fftwf_plan_many_dft_r2c.restype = C.c_void_p
        L.fftwf_plan_many_dft_r2c.argtypes = [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int,
                                              C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_uint]
        L.fftwf_execute.argtypes = [C.c_void_p]
        L.fftwf_destroy_plan.argtypes = [C.c_void_p]
        L.fftwf_free.argtypes = [C.c_void_p]
        a, b = L.fftwf_alloc_real(rows * n2), L.fftwf_alloc_complex(rows * n2)
        C.memset(a, 0, rows * n2 * 4)
        nn = C.c_int(n2)
        plan = L.fftwf_plan_many_dft_r2c(1, C.byref(nn), rows, a, None, 1, n2, b, None, 1, n2, 0)   # mfcccpu.cpp:114
        L.fftwf_execute(plan)
        t0 = time.perf_counter()
        reps = 8
        for _ in range(reps):
            L.fftwf_execute(plan)
        us = (time.perf_counter() - t0) / (reps * rows) * 1e6
        L.fftwf_destroy_plan(plan); L.fftwf_free(a); L.fftwf_free(b)
        return us
    except Exception:
        return None


def cpu_stage_split(p, pcm):
    """One core, one utterance-sized MfccCpu per utterance: seconds in set_input + flush (segment + FFT), apply (mel, log, DCT,
    deltas, normalise) and get_output_data, as fractions."""
    import oracle_lib as ol
    lib = ol.RefLib("ref" if ol.available("ref") else "port")
    t_in = t_apply = t_out = 0.0
    for u in pcm:
        m = ol.RefMfcc(lib, len(u), p)
        m.set_window(lib.window(p["window_size"]))
        n = m.get_input_buffer_size()
        for pos in list(range(0, len(u), n)) + [None]:
            t0 = time.perf_counter()
            wc = m.flush() if pos is None else m.set_input(u[pos:pos + n])
            t1 = time.perf_counter()
            m.apply()
            t2 = time.perf_counter()
            if wc > 0:
                m.get_output_data(wc)
            t3 = time.perf_counter()
            t_in += t1 - t0; t_apply += t2 - t1; t_out += t3 - t2
        m.close()
    tot = t_in + t_apply + t_out
    return {"segment_fft": t_in / tot, "mel_log_dct_delta_norm": t_apply / tot, "get_output": t_out / tot}


def cpu_arm(n_utts, steps, warmup, threads, pcm=None, g=CFG16):
    """Times the reference's own CPU path (or the port when oracle/_ref is absent). Returns dict."""
    import oracle_lib as ol
    kind = "reference" if ol.available("ref") else "port"
    lib = ol.RefLib("ref" if kind == "reference" else "port")
    p = params_dict(g)
    if kind == "port":
        threads = 1
    if pcm is None:
        pcm = synth_host(n_utts, 1234, g)
    utts = [pcm[i] for i in range(n_utts)]
    frames = n_utts * frames_of(g["n"], g)
    times = []
    for i in range(warmup + steps):
        _, s = lib.extract(p, utts, sample_limit=0, n_threads=threads)   # Q5: MfccCpu sized to the utterance
        if i >= warmup:
            times.append(s)
    t = float(np.mean(times))
    return dict(kind=kind, cores=threads, value=frames / t, seconds_per_step=t, frames_per_step=frames,
                sample=f"{n_utts} utterances x 10 s of the same synthetic workload ({frames} frames) per step, "
                       f"fresh MfccCpu per utterance sized to it (Q3/Q5), FFT = oracle/fftw_shim.c (FFTW not installed)")


def cpu_arm_threads(ol):
    """Cores the CPU arm runs on, which its sample is sized for: every host core for the reference's build, one for the C port
    (single-threaded), which stands in when oracle/_ref was not built."""
    return (os.cpu_count() or 1) if ol.available("ref") else 1


def cpu_denominators(p, sample):
    return {"fft_shim_us_per_512pt": shim_us_per_transform(512), "fft_shim_us_per_256pt": shim_us_per_transform(256),
            "stage_split_1core": cpu_stage_split(p, sample)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib as ol
    threads = cpu_arm_threads(ol)
    lib = ol.RefLib("ref" if ol.available("ref") else "port")
    cal = synth_host(8, 99)
    _, s = lib.extract(params_dict(), [cal[i] for i in range(8)], sample_limit=0, n_threads=1)
    rate1 = 8 * 998 / s
    # ~3 s of wall time per step with all cores
    n_utts = int(max(threads * 4, min(4096, 3.0 * rate1 * threads / 998)))
    r = cpu_arm(n_utts, args.steps, max(1, min(args.warmup, 2)), threads)
    cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "value_1core": rate1}
    cpu.update(cpu_denominators(params_dict(), [cal[i] for i in range(4)]))
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(3, 10000, args.gpus),        # identical to the B200 arm's dict
            "cpu_baseline": cpu,
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "audio_hours_per_s": r["value"] * 160 / 16000 / 3600.0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------- plumbing
class ClockSampler:
    """nvidia-smi polled every 20 ms in the background; stop(t0, t1) keeps the samples taken inside the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc:
            self.proc.terminate()
        inside = [r for (t, r) in self.rows if t0 is None or (t0 <= t <= t1 + 0.03)]
        rows = inside if len(inside) >= 2 else [r for (_, r) in self.rows]
        sm, mx, power, reasons = [], 0, [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_in_timed_region": len(inside), "power_w_max": max(power) if power else None}


_FULL_AFFINITY = None


def bind_to_gpu_numa_node(torch, local):
    """Pin this rank to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is allocated: with 8 ranks
    per box the end-to-end path is bound by host memory / PCIe root-complex locality, not by the kernels."""
    global _FULL_AFFINITY
    _FULL_AFFINITY = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1} & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"bound": True, "cpus": len(cpus), "first_cpu": min(cpus)}
    except Exception as e:
        return {"bound": False, "why": str(e)[:120]}
    return {"bound": False, "why": "empty affinity mask"}


class Ctx:
    pass


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ---------------------------------------------------------------------------------------------------------- legs
def leg_config3(cx, args, pcm, out, offs, lens, n_utts):
    """Headline: one launch of k_fused_mfcc per step, per-utterance CMN inside the kernel."""
    torch, afe, stream = cx.torch, cx.afe, cx.stream
    g = CFG16
    frames = n_utts * frames_of(g["n"], g)
    b = afe.BatchMfcc(cx.ap16, cx.local, stats_scope=afe.STATS_REFERENCE_BLOCK, flags=cx.flags)
    b.set_stream(stream.cuda_stream)
    assert b.plan(offs, lens) == frames
    for _ in range(args.warmup):
        b.run_device(pcm.data_ptr(), out.data_ptr())
    cx.barrier()
    t_begin = time.perf_counter()
    launches = 0
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    mids = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev0[0].record(stream)
    for i in range(args.steps):
        b.run_device(pcm.data_ptr(), out.data_ptr())
        mids[i].record(stream)
        launches += b.kernel_launches                         # 1 per step (k_fused_mfcc)
        ev0[i + 1].record(stream)
    cx.barrier()
    t_end = time.perf_counter()
    total_ms = ev0[0].elapsed_time(ev0[-1])
    k1 = float(np.mean([ev0[i].elapsed_time(mids[i]) for i in range(args.steps)]))
    ms_per_step = cx.max_over_ranks(total_ms) / args.steps
    res = dict(frames=frames, ms_per_step=ms_per_step, value=cx.world * frames / (ms_per_step * 1e-3), k1_ms=k1,
               launches=launches, t_begin=t_begin, t_end=t_end, tiles=b.num_tiles, kernel=b.kernel_name)
    b.close()
    return res


DUMP_UTTS = 256     # 256 utterances x 998 frames x 39 x 4 B = 39.9 MB, under the 64 MB a dump may take


def dump_outputs(dirname, out, n_utts, T):
    """--dump-outputs: the rows the last timed step wrote for a fixed sample of whole utterances (seed 0, ascending utterance
    index) -> DIR/features.npy, float32 [k, T, 39]. The PCM is generated from fixed seeds, so the same arguments give the
    same inputs on every run."""
    import torch
    k = min(DUMP_UTTS, n_utts)
    pick = np.sort(np.random.default_rng(0).choice(n_utts, k, replace=False))
    feats = out.view(n_utts, T, WIDTH)[torch.from_numpy(pick).to(out.device)].cpu().numpy()
    assert feats.dtype == np.float32 and feats.nbytes <= 64 << 20
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "features.npy"), feats)


def parity_gate(cx, pcm, out, n_utts, g=CFG16, n_check=64):
    """BASELINE.md §3: 64 utterances of the TIMED output against the reference's own CPU classes (Q1-exact, single block)."""
    import oracle_lib as ol
    n, T = g["n"], frames_of(g["n"], g)
    k = min(n_check, n_utts)
    lib = ol.RefLib("ref" if ol.available("ref") else "port")
    sample = pcm[:k * n].cpu().numpy().reshape(k, n)
    want, _ = lib.extract(params_dict(g), [sample[i] for i in range(k)], sample_limit=1 << 22, n_threads=os.cpu_count() or 1)
    want = np.concatenate(want).astype(np.float64)
    got = out[:k * T].cpu().numpy().astype(np.float64)
    err = np.abs(got - want)
    rel = err / np.maximum(np.abs(want), 1.0)
    res = {"n_utts": k, "frames": int(k * T), "max_abs_static": float(err[:, :13].max()), "max_abs_delta": float(err[:, 13:].max()),
           "max_rel": float(rel.max()), "oracle": lib.kind, "tolerance": {"static": 5e-4, "delta": 2e-4, "rel": 2e-4}}
    res["ok"] = bool(res["max_abs_static"] <= 5e-4 and res["max_abs_delta"] <= 2e-4 and res["max_rel"] <= 2e-4)
    return res


def make_comm(cx):
    torch, afe, dist = cx.torch, cx.afe, cx.dist
    idbuf = torch.zeros(128, dtype=torch.uint8)
    if cx.rank == 0:
        raw = (C.c_char * 128)()
        afe._check(afe.lib().afe_nccl_get_unique_id(raw))
        idbuf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8).clone()
    if cx.world > 1:
        idd = idbuf.to(cx.dev); dist.broadcast(idd, 0); idbuf = idd.cpu()
    comm = C.c_void_p()
    afe._check(afe.lib().afe_nccl_comm_init(idbuf.numpy().tobytes(), cx.world, cx.rank, cx.local, C.byref(comm)))
    return comm


def leg_corpus(cx, args, pcm, out, offs, lens, n_utts, steps, verify=True):
    """Corpus CMVN (BASELINE configs[3]): extract -> corpus record -> NCCL all-reduce inside the Normalizer -> normalise,
    timed; then the exchange and the result are VERIFIED on every rank."""
    torch, afe, stream, dist = cx.torch, cx.afe, cx.stream, cx.dist
    g = CFG16
    T = frames_of(g["n"], g)
    frames = n_utts * T
    comm = make_comm(cx)
    # corpus statistics are not the reference's per-block semantics: no Q1 quirk here (it would write statics the statistics never saw)
    bc = afe.BatchMfcc(cx.ap16, cx.local, stats_scope=afe.STATS_CORPUS, flags=cx.flags & ~afe.BATCH_Q1_EXACT)
    bc.set_stream(stream.cuda_stream)
    bc.plan(offs, lens)
    launches = 0

    def cstep():
        nonlocal launches
        bc.extract_device(pcm.data_ptr(), out.data_ptr()); launches += bc.kernel_launches
        bc.corpus_stats(); launches += bc.kernel_launches
        bc.allreduce(comm.value)
        bc.normalize_device(out.data_ptr()); launches += bc.kernel_launches
    for _ in range(max(1, min(args.warmup, 3))):
        cstep()
    cx.barrier()
    launches = 0
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(stream)
    for _ in range(steps):
        cstep()
    c1.record(stream)
    cx.barrier()
    cms = cx.max_over_ranks(c0.elapsed_time(c1)) / steps
    peak = float(cx.peaks.get("hbm_gbs", 6650.0))
    alg = 2 * g["S"] + 12 * WIDTH
    res = {"value": cx.world * frames / (cms * 1e-3), "unit": UNIT, "ms_per_step": cms, "launches_per_step": launches // max(steps, 1),
           "collective": "ncclAllReduce x3 grouped (sum 79 | min 39 | max 39 doubles) via afe_normalizer_allreduce(afe_batch_normalizer)",
           "algorithmic_bytes_per_frame": alg,
           "roofline": {"bound": "hbm", "achieved": frames * alg / (cms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": frames * alg / (cms * 1e-3) / 1e9 / peak, "note": "whole sequence K1 + K2 + all-reduce + K3 per GPU"}}
    if verify:
        # (1) the exchange: local record -> our all-reduce; the same local record re-reduced with torch.distributed
        bc.extract_device(pcm.data_ptr(), out.data_ptr())
        bc.corpus_stats(); bc.synchronize()
        local = bc.corpus_record()
        bc.allreduce(comm.value); bc.synchronize()
        merged = bc.corpus_record()
        w = WIDTH
        ls = torch.tensor(local, device=cx.dev, dtype=torch.float64)
        s, mn, mx = ls[:2 * w + 1].clone(), ls[2 * w + 1:3 * w + 1].clone(), ls[3 * w + 1:].clone()
        if cx.world > 1:
            dist.all_reduce(s, op=dist.ReduceOp.SUM); dist.all_reduce(mn, op=dist.ReduceOp.MIN); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        ref = torch.cat([s, mn, mx]).cpu().numpy()
        count_ok = merged[2 * w] == cx.world * local[2 * w] == cx.world * n_utts * T   # corpus scope: every row of every utterance
        sum_rel = float(np.max(np.abs(merged[:2 * w] - ref[:2 * w]) / np.maximum(np.abs(ref[:2 * w]), 1e-300)))
        sum_bitwise = bool(np.array_equal(merged[:2 * w + 1], ref[:2 * w + 1]))
        minmax_exact = bool(np.array_equal(merged[2 * w + 1:], ref[2 * w + 1:]))
        # (2) the result: global column means of the normalised output over the rows the statistics cover
        bc.normalize_device(out.data_ptr()); bc.synchronize()
        col = torch.zeros(w, device=cx.dev, dtype=torch.float64)
        for r0 in range(0, n_utts * T, 1 << 22):             # fp64 column sums in pieces (no 2x copy of the features)
            col += out[r0:r0 + (1 << 22)].to(torch.float64).sum(0)
        if cx.world > 1:
            dist.all_reduce(col, op=dist.ReduceOp.SUM)
        mean_abs = float((col / merged[2 * w]).abs().max().item())
        ok = torch.tensor([int(count_ok and minmax_exact and sum_rel < 1e-13 and mean_abs < 1e-4)], device=cx.dev)
        if cx.world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        res["verified"] = {"ok_on_every_rank": bool(ok.item()), "count_equals_world_x_local": bool(count_ok), "sum_max_rel_vs_torch_allreduce": sum_rel,
                           "sum_bitwise_vs_torch_allreduce": sum_bitwise, "min_max_exact": minmax_exact,
                           "max_abs_global_column_mean_after_normalise": mean_abs, "ranks": cx.world}
    bc.close()
    afe.lib().afe_nccl_comm_destroy(comm)
    return res


def copy_ceiling(cx, h_pcm, h_out, d_pcm, d_out, reps=3):
    """What this box can move: the step's H2D and D2H bytes with plain cudaMemcpyAsync on two streams, concurrently, all ranks
    at once, no kernels. The end-to-end number cannot beat frames / this time."""
    torch = cx.torch
    s1, s2 = torch.cuda.Stream(device=cx.dev), torch.cuda.Stream(device=cx.dev)
    best = None
    for _ in range(reps + 1):
        cx.barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_pcm.copy_(h_pcm, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        s1.synchronize(); s2.synchronize()
        dt = cx.max_over_ranks(time.perf_counter() - t0)
        best = dt if best is None else min(best, dt)
    return best


def leg_e2e(cx, args, pcm, out, offs, lens, n_utts):
    torch, afe = cx.torch, cx.afe
    g = CFG16
    n, T = g["n"], frames_of(g["n"], g)
    frames = n_utts * T
    h_pcm = torch.empty((n_utts * n + 64,), dtype=torch.int16).pin_memory()
    h_pcm.copy_(pcm)
    h_out = torch.empty((frames, WIDTH), dtype=torch.float32).pin_memory()
    be = afe.BatchMfcc(cx.ap16, cx.local, stats_scope=afe.STATS_REFERENCE_BLOCK, flags=cx.flags)
    be.plan(offs, lens)
    lib = afe.lib()
    e2e_steps = max(2, min(args.steps, 5))
    afe._check(lib.afe_batch_run_host(be._h, C.c_void_p(h_pcm.data_ptr()), C.c_void_p(h_out.data_ptr())))
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        afe._check(lib.afe_batch_run_host(be._h, C.c_void_p(h_pcm.data_ptr()), C.c_void_p(h_out.data_ptr())))
    torch.cuda.synchronize()
    et = cx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e = {"value": cx.world * frames / et, "unit": UNIT, "h2d_bytes_per_step": int(n_utts * n * 2),
           "d2h_bytes_per_step": int(frames * WIDTH * 4), "ms_per_step": et * 1e3, "steps": e2e_steps,
           "api": "afe_batch_run_host (pinned host buffers)", "host_affinity": cx.affinity}
    # the host result must be the device result (whole shard)
    be.run_device(pcm.data_ptr(), out.data_ptr()); be.synchronize(); torch.cuda.synchronize()
    e2e["matches_device_path"] = bool(torch.equal(h_out.to(cx.dev), out))
    be.close()
    ceil_s = copy_ceiling(cx, h_pcm, h_out, pcm, out)
    e2e["copy_ceiling"] = {"ms": ceil_s * 1e3, "frames_per_s": cx.world * frames / ceil_s,
                           "aggregate_gb_s": cx.world * (n_utts * n * 2 + frames * WIDTH * 4) / ceil_s / 1e9,
                           "how": "same H2D + D2H bytes, plain cudaMemcpyAsync on two streams, all ranks concurrently, no kernels"}
    e2e["frac_of_copy_ceiling"] = e2e["value"] / e2e["copy_ceiling"]["frames_per_s"]
    del h_pcm, h_out
    return e2e


def leg_stream_object(cx, pcm, n_files=64, threads=(1, 4)):
    """The drop-in object: MfccCuda (ParamBase verbs: set_input -> apply -> get_output_data, flush -> apply -> get_output_data)
    on 10 s files from HOST buffers, one object per host thread, objects reset between files (afe_mfcc_reset)."""
    afe = cx.afe
    g = CFG16
    n, T = g["n"], frames_of(g["n"], g)
    host = pcm[:n_files * n].cpu().numpy().reshape(n_files, n)
    ap = afe.make_params(input_buffer_size=10_000_000, **{k: v for k, v in params_dict().items() if k != "alpha"})
    win = afe.make_window(g["W"])
    out = {}

    def worker(m, files, sink):
        for u in files:
            wc = m.set_input(u); m.apply(); a = m.get_output_data(wc)
            wc = m.flush(); m.apply(); b = m.get_output_data(wc)
            sink.append((a, b))
            m.reset()
    check = None
    for nt in threads:
        objs = [afe.MfccCuda(ap, cx.local) for _ in range(nt)]
        for m in objs:
            m.set_window(win)
        sinks = [[] for _ in range(nt)]
        worker(objs[0], host[:2], [])                       # warm-up
        ts = [threading.Thread(target=worker, args=(objs[i], host[i::nt], sinks[i])) for i in range(nt)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        dt = time.perf_counter() - t0
        out[f"{nt}_handles"] = {"frames_per_s": n_files * T / dt, "ms_per_file": dt / n_files * 1e3 * nt}
        if check is None:
            check = np.concatenate(sinks[0][0])
        fused = objs[0].uses_fused_kernel
        for m in objs:
            m.close()
    # the same sequence from C++ host threads through a ParamBase* (host/afe_stream_bench.cpp): no interpreter in the loop
    cpp = {}
    exe = os.path.join(ROOT, "asr-featext-opencl_b200", "afe_stream_bench")
    if os.path.exists(exe):
        for nt in (1, 4, 8, 16):
            try:
                r = subprocess.run([exe, "--files", "512", "--threads", str(nt), "--dev", str(cx.local)], stdout=subprocess.PIPE,
                                   stderr=subprocess.PIPE, text=True, timeout=120)
                cpp[f"{nt}_threads"] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-200:]}
            except Exception as e:
                cpp[f"{nt}_threads"] = {"error": str(e)[:200]}
    online = online_blocks(cx, host[0])
    best = max([v["frames_per_s"] for v in out.values()] + [v.get("frames_per_s", 0.0) for v in cpp.values()])
    return {"value": best, "unit": UNIT, "python_threads": out, "cpp_threads_parambase_ptr": cpp, "online_200ms_blocks": online, "files": n_files,
            "uses_fused_kernel": bool(fused),
            "api": "MfccCuda through the reference's verbs (set_input / set_alpha / apply / get_output_data / flush) per 10 s file, host "
                   "buffers in and out; one object per host thread",
            "first_file_rows": int(check.shape[0])}


def online_blocks(cx, u, block=3200):
    """The same object as an ONLINE front end: a 10 s file arrives in 200 ms blocks (set_input -> apply -> get_output_data per
    block, one launch of the fused kernel each); latency of a block from host buffer to host rows, and the rows against the
    reference's CPU object fed the same blocks (per-block CMN statistics, Q2)."""
    afe = cx.afe
    g = CFG16
    p = params_dict()
    ap = afe.make_params(input_buffer_size=block, **{k: v for k, v in p.items() if k != "alpha"})
    m = afe.MfccCuda(ap, cx.local)
    m.set_window(afe.make_window(g["W"]))
    limit = block
    block = m.get_input_buffer_size()                         # whole frames: est(limit) * S + W - S, as the reference driver feeds it
    lat, rows = [], []
    for rep in range(3):                                      # the last pass is reported
        lat, rows = [], []
        for pos in range(0, len(u), block):
            t0 = time.perf_counter()
            wc = m.set_input(u[pos:pos + block]); m.apply()
            r = m.get_output_data(wc) if wc > 0 else None
            lat.append(time.perf_counter() - t0)
            if r is not None:
                rows.append(r)
        wc = m.flush(); m.apply()
        if wc > 0:
            rows.append(m.get_output_data(wc))
        m.reset()
    m.close()
    got = np.concatenate(rows)
    res = {"block_samples": block, "blocks": len(lat), "us_per_block_median": float(np.median(lat) * 1e6),
           "us_per_block_max": float(np.max(lat) * 1e6), "real_time_factor": float(np.sum(lat) / (len(u) / g["sr"])),
           "rows": int(got.shape[0])}
    try:
        import oracle_lib as ol
        lib = ol.RefLib("ref" if ol.available("ref") else "port")
        want = lib.extract(p, [u], sample_limit=limit)[0][0]
        res["max_abs_vs_reference_same_blocks"] = float(np.abs(got - want).max()) if got.shape == want.shape else None
        res["rows_reference"] = int(want.shape[0])
    except Exception as e:  # noqa: BLE001
        res["reference_error"] = str(e)[:200]
    return res


def leg_config5(cx, args, steps):
    """One 1-hour 8 kHz stream: deltas fused, without and with CMN. The working set fits in L2, so a 256 MB buffer is written
    between timed iterations."""
    torch, afe, stream = cx.torch, cx.afe, cx.stream
    g = CFG8
    n, T = g["n"], frames_of(g["n"], g)
    pcm = synth_device(torch, cx.dev, 1, g, 4321 + cx.rank)
    out = torch.empty((T, WIDTH), dtype=torch.float32, device=cx.dev)
    flush = torch.empty(64 << 20, dtype=torch.float32, device=cx.dev)
    offs, lens = np.zeros(1, np.int64), np.full(1, n, np.int64)
    peak = float(cx.peaks.get("hbm_gbs", 6650.0))
    res = {}
    for name, norm, fl in (("no_norm", 0, 0), ("cmn", 1, 0), ("cmn_k2_k3_kernels", 1, afe.BATCH_UNFUSED_NORM)):
        p = params_dict(g, norm)
        ap = afe.make_params(input_buffer_size=1 << 22, **{k: v for k, v in p.items() if k != "alpha"})
        b = afe.BatchMfcc(ap, cx.local, flags=afe.BATCH_Q1_EXACT | fl)
        b.set_stream(stream.cuda_stream)
        assert b.plan(offs, lens) == T
        for _ in range(3):
            b.run_device(pcm.data_ptr(), out.data_ptr())
        ms = []
        for _ in range(steps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            b.run_device(pcm.data_ptr(), out.data_ptr())
            e1.record(stream)
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        t = cx.max_over_ranks(float(np.median(ms)))
        alg = T * (2 * g["S"] + 4 * WIDTH)
        res[name] = {"ms": t, "frames_per_s": cx.world * T / (t * 1e-3), "kernel_launches": b.kernel_launches, "tiles": b.num_tiles,
                     "roofline_frac": alg / (t * 1e-3) / 1e9 / peak}
        if name == "cmn" and cx.rank == 0:
            # bounded parity gate: the first 100 000 frames of the stream against the reference's CPU classes are checked by
            # tests/test_gpu_parity.py::test_config5_full_size_one_hour_stream at full size; here: column means ~ 0
            res[name]["max_abs_column_mean"] = float(out[:T - 6].to(torch.float64).mean(0).abs().max().item())
        b.close()
    res["cmn_over_no_norm"] = res["cmn"]["ms"] / res["no_norm"]["ms"]
    del pcm, out, flush
    return res


# ---------------------------------------------------------------------------------------------------------- main arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    import afe_loader
    afe = afe_loader.load()

    cx = Ctx()
    cx.torch, cx.dist, cx.afe = torch, dist, afe
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(cx.local)
    cx.dev = torch.device("cuda", cx.local)
    cx.affinity = bind_to_gpu_numa_node(torch, cx.local) if cx.world > 1 and not args.no_numa_bind else {"bound": False, "why": "single rank"}
    if cx.world > 1:
        dist.init_process_group("nccl", device_id=cx.dev)
    cx.peaks = load_peaks()

    def barrier():
        if cx.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device=cx.dev, dtype=torch.float64)
        if cx.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    cx.barrier, cx.max_over_ranks = barrier, max_over_ranks
    cx.flags = (afe.BATCH_Q1_EXACT | (afe.BATCH_NO_TMA if args.no_tma else 0) | (afe.BATCH_NO_CLUSTER if args.no_cluster else 0)
                | (afe.BATCH_MMA_PHASE2 if args.mma else 0))
    cx.ap16 = afe.make_params(input_buffer_size=1 << 22, **{k: v for k, v in params_dict().items() if k != "alpha"})
    # a dedicated (non-default) stream: the library launches on it and the CUDA events are recorded on it
    cx.stream = torch.cuda.Stream(device=cx.dev)
    torch.cuda.set_stream(cx.stream)

    g = CFG16
    n, T = g["n"], frames_of(g["n"], g)
    config = args.config
    sampler = ClockSampler(cx.local)
    if cx.rank == 0:
        sampler.start()

    extra, line = {}, None
    if config in (3, 4):
        if config == 3:
            n_utts = args.utts
        else:
            n_utts = args.utts if args.utts != 10000 else (360000 // cx.world if cx.world >= 2 else 45000)
        pcm = synth_device(torch, cx.dev, n_utts, g, 1234 + cx.rank)
        out = torch.empty((n_utts * T, WIDTH), dtype=torch.float32, device=cx.dev)
        offs = np.arange(n_utts, dtype=np.int64) * n
        lens = np.full(n_utts, n, np.int64)
        r3 = leg_config3(cx, args, pcm, out, offs, lens, n_utts)
        if args.dump_outputs and cx.rank == 0:
            dump_outputs(args.dump_outputs, out, n_utts, T)      # before the corpus leg reuses `out`
        parity = parity_gate(cx, pcm, out, n_utts) if cx.rank == 0 and not args.no_cpu else None
        clocks = sampler.stop(r3["t_begin"], r3["t_end"]) if cx.rank == 0 else None
        try:
            # the headline of --config 4 times exactly --steps steps; as a side block of --config 3, 2 to 10
            corpus_steps = args.steps if config == 4 else max(2, min(args.steps, 10))
            corpus = leg_corpus(cx, args, pcm, out, offs, lens, n_utts, steps=corpus_steps)
        except Exception as e:  # NCCL missing etc.: the headline number does not depend on it
            corpus = {"unavailable": str(e)[:300]}
        e2e = None if args.no_e2e else leg_e2e(cx, args, pcm, out, offs, lens, n_utts)
        stream_obj = None
        if not args.no_extras and cx.rank == 0:
            try:
                stream_obj = leg_stream_object(cx, pcm)
            except Exception as e:
                stream_obj = {"unavailable": str(e)[:300]}
        cpu = None
        if cx.rank == 0 and not args.no_cpu:
            if _FULL_AFFINITY:
                os.sched_setaffinity(0, _FULL_AFFINITY)   # the CPU baseline uses every host core, not one NUMA node
            import oracle_lib as ol
            threads = cpu_arm_threads(ol)
            sample = pcm[:64 * n].cpu().numpy().reshape(64, n)
            lib1 = ol.RefLib("ref" if ol.available("ref") else "port")
            _, s1 = lib1.extract(params_dict(), [sample[i] for i in range(16)], sample_limit=0, n_threads=1)
            rate1 = 16 * T / s1
            n_cpu = int(max(threads * 2, min(4096, 2.0 * rate1 * threads / T)))
            n_cpu = min(n_cpu, n_utts)
            cs = pcm[:n_cpu * n].cpu().numpy().reshape(n_cpu, n)
            r = cpu_arm(n_cpu, 2, 1, threads, pcm=cs)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                   "value_1core": rate1}
            cpu.update(cpu_denominators(params_dict(), [sample[i] for i in range(4)]))
        del pcm, out
        torch.cuda.empty_cache()
        if not args.no_extras:
            try:
                extra["config5"] = dict(leg_config5(cx, args, steps=max(5, min(args.steps, 20))), config=workload_config(5, 1, cx.world))
            except Exception as e:
                extra["config5"] = {"unavailable": str(e)[:300]}
            if config == 3:
                try:
                    n4 = 45000
                    pcm4 = synth_device(torch, cx.dev, n4, g, 777 + cx.rank)
                    out4 = torch.empty((n4 * T, WIDTH), dtype=torch.float32, device=cx.dev)
                    offs4, lens4 = np.arange(n4, dtype=np.int64) * n, np.full(n4, n, np.int64)
                    extra["config4"] = dict(leg_corpus(cx, args, pcm4, out4, offs4, lens4, n4, steps=max(2, min(args.steps, 5))),
                                            config=workload_config(4, n4, cx.world),
                                            note="every GPU takes the 45 000-utterance shard of the 8-GPU case (weak scaling); "
                                                 "`--config 4` runs 360 000 / N utterances per GPU")
                    del pcm4, out4
                except Exception as e:
                    extra["config4"] = {"unavailable": str(e)[:300]}
        if cx.rank == 0:
            peak = float(cx.peaks.get("hbm_gbs", 6650.0))
            frames = r3["frames"]
            if config == 3:
                k1 = r3["k1_ms"]
                alg_bytes = frames * (2 * g["S"] + 4 * WIDTH)
                achieved = alg_bytes / (k1 * 1e-3) / 1e9
                roof = {"bound": "hbm", "kernel": r3["kernel"], "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": None, "peak_source": "measured" if cx.peaks else "fallback",
                        "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": k1, "kernel_share_of_step": k1 / r3["ms_per_step"],
                        "note": "fp32-issue bound (FFT butterflies), not HBM bound; see DESIGN.md"}
                prof = os.path.join(ROOT, "profiles", "traffic.json")
                if os.path.exists(prof):
                    try:
                        per_frame = json.load(open(prof)).get("k_fused_mfcc_dram_bytes_per_frame")
                        roof["traffic"] = per_frame * frames if per_frame else None   # ncu dram read+write per frame x frames/launch
                        roof["traffic_source"] = "profiles/traffic.json (ncu --set full on a 2000-utterance launch, scaled per frame)"
                    except Exception:
                        pass
                value, ms_per_step, launches, scaling = r3["value"], r3["ms_per_step"], r3["launches"], "weak"
            else:
                # headline = the corpus-CMVN sequence (configs[3]); strong scaling: the corpus is fixed, the shard shrinks with N
                roof = dict(corpus.get("roofline", {}), kernel="k_fused_mfcc + k_reduce_partials(_level1) + ncclAllReduce + k_finalize_stats + k_normalize_tiles",
                            peak_source="measured" if cx.peaks else "fallback", traffic=None)
                value, ms_per_step = corpus.get("value"), corpus.get("ms_per_step")
                launches, scaling = corpus.get("launches_per_step", 0) * args.steps, "strong" if cx.world >= 2 else "weak"
                extra["config3_on_this_shard"] = {"value": r3["value"], "ms_per_step": r3["ms_per_step"]}
            line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": cx.world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": workload_config(config, n_utts, cx.world),
                    "audio_hours_per_s": value * g["S"] / g["sr"] / 3600.0 if value else None, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e,
                    "gpu_launches": launches, "clocks": clocks, "parity": parity, "corpus_cmvn": corpus, "stream_object": stream_obj,
                    "extra": extra, "kernels_per_step": [r3["kernel"]], "tiles_per_gpu": r3["tiles"],
                    "flags": {"tma": not args.no_tma, "devtools": bool(afe.lib().afe_build_flags() & 1), "abi": afe.lib().afe_abi_version()}}
    else:
        r5 = leg_config5(cx, args, steps=args.steps)
        clocks = sampler.stop() if cx.rank == 0 else None
        if cx.rank == 0:
            g8 = CFG8
            T8 = frames_of(g8["n"], g8)
            peak = float(cx.peaks.get("hbm_gbs", 6650.0))
            alg = T8 * (2 * g8["S"] + 4 * WIDTH)
            ms = r5["no_norm"]["ms"]
            roof = {"bound": "hbm", "kernel": "k_fused_mfcc<256,13,8,3,false>", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": "measured" if cx.peaks else "fallback",
                    "note": "0.15 ms of work: launch- and tail-latency dominated (720 tiles on 296 CTA slots)"}
            line = {"metric": METRIC, "value": r5["no_norm"]["frames_per_s"], "unit": UNIT, "n_gpus": cx.world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": workload_config(5, 1, cx.world),
                    "audio_hours_per_s": r5["no_norm"]["frames_per_s"] * g8["S"] / g8["sr"] / 3600.0, "roofline": roof,
                    "cpu_baseline": None, "e2e": None, "gpu_launches": r5["no_norm"]["kernel_launches"] * args.steps, "clocks": clocks,
                    "extra": {"config5": r5}, "flags": {"devtools": bool(afe.lib().afe_build_flags() & 1)}}
    if cx.rank == 0:
        print(json.dumps(line), flush=True)
    if cx.world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[3, 4, 5], help="BASELINE configuration of the headline line (1-based: "
                    "3 = configs[2], the metric's; 4 = 1000 audio-hours corpus CMVN; 5 = one 1-hour 8 kHz stream)")
    ap.add_argument("--utts", type=int, default=10000, help="utterances per GPU (BASELINE config 3: 10000)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin ranks to their GPU's NUMA node (A/B, N > 1)")
    ap.add_argument("--no-cluster", action="store_true", help="ticket-scheme normalisation instead of clusters + DSMEM (A/B)")
    ap.add_argument("--no-tma", action="store_true")
    ap.add_argument("--mma", action="store_true", help="mel + log + DCT on the tensor cores (AFE_BATCH_MMA_PHASE2) instead of CUDA cores (A/B)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-4 / config-5 / stream-object extra blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the features of the last timed step (256 utterances, fixed "
                    "sample) to DIR/features.npy (--config 3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != 3):
        ap.error("--dump-outputs writes the features of the --config 3 headline of the b200 implementation")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_b200(args)


if __name__ == "__main__":
    main()
