#!/usr/bin/env python
"""Benchmark of the spectral hot path (BASELINE.json metric: audio-seconds / second).

Workload (config.workload): BASELINE.json configs[1] -- GRID-shaped batch, 1,000 x 3 s 16 kHz
utterances + white noise at 0 dB SNR per GPU: SNR factor + fused mix/STFT/mel/dB + top_db floor
into 15 AV-aligned (80, 20) slices for mixed / speech / noise and the mixed PCM.  One "step" is
one pass over that batch.  Multi-GPU: every rank owns its own 1,000 utterances (weak scaling,
sharded by utterance, no data-path collective); rank 0 prints ONE JSON line.

  value     whole-job audio-s/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the host-facing API: pinned host buffers, H2D + D2H in the timed region
  roofline  dominant kernel (avse_forward4_kernel): algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the float64 CPU restatement of the reference path (oracle/), timed on host cores

--dump-outputs DIR writes what the timed path returned in its last step (mixed / speech / noise log-mel slices, mixed PCM,
and the inverse section's reconstructed PCM from those outputs) for a seeded sample of utterances.  The inputs depend only on the arguments,
so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as it found it (it may be read-only)

SR, FPS, SLICE_MS = 16000, 25.0, 200
UTT_SECONDS = 3.0
L = int(SR * UTT_SECONDS)          # 48000
N_VIDEO_SLICES = 15                # 75 mouth-crop frames / 5
BYTES_PER_SAMPLE_PAIR = 18         # SURVEY 8(d): read 4+4, write 4 (mixed PCM) + 3 * 80*4/160 (three log-mels)
INV_BYTES_PER_FRAME = 1600         # SURVEY 8(d): read mel 320 + mixture PCM 640, write PCM 640


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1000, help="utterances per GPU per step")
    ap.add_argument("--seconds", type=float, default=3.0, help="utterance duration (BASELINE configs[4] long form: 60)")
    ap.add_argument("--snr-sweep", action="store_true", help="per-utterance SNR cycling through -10, -5, 0, 5, 10 dB (configs[4])")
    ap.add_argument("--cpu-sample", type=int, default=0, help="utterances in the CPU baseline sample (0: auto)")
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of the CPU baseline (0: every host thread)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="chunks per step in the host pipeline")
    ap.add_argument("--e2e-streams", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-inverse", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the HBM-bound neighbours of the path (sample-set gather, video normaliser, MSE)")
    ap.add_argument("--sustain-s", type=float, default=2.0,
                    help="also run the step back to back for at least this many seconds and report the steady-state figure (0: skip)")
    ap.add_argument("--corpus", type=int, default=0,
                    help="BASELINE configs[2]: a corpus of this many utterances sharded contiguously by utterance over the ranks "
                         "(engine.shard_range, strong scaling); a step is one pass over the rank's whole shard in launches of --batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the last timed step (and their inverse) as DIR/<name>.npy, float32, "
                         "for a fixed seeded sample of utterances of at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle restatement of preprocess_audio_pair (dp:119-139), Pool over utterances (dp:194)
# ------------------------------------------------------------------------------------------------
def _cpu_one(seed):
    import numpy as np
    from oracle import avse_oracle as O
    s = O.AudioSignal(O.synth_speech(L, SR, seed).astype(np.float32), SR)
    n = O.AudioSignal(O.synth_noise(L, seed).astype(np.float32), SR)
    t0 = time.perf_counter()
    O.preprocess_audio_pair_signals(s, n, SLICE_MS, N_VIDEO_SLICES, FPS, snr_db=0)
    return time.perf_counter() - t0


SNR_SWEEP = (-10.0, -5.0, 0.0, 5.0, 10.0)
SWEEP = False


def set_workload(seconds, sweep):
    """Utterance duration / SNR policy of this run (module globals: the forked CPU workers inherit them)."""
    global UTT_SECONDS, L, N_VIDEO_SLICES, SWEEP
    UTT_SECONDS = float(seconds)
    N_VIDEO_SLICES = int(UTT_SECONDS * FPS / 5)           # dp:24-25: 5 video frames per 200 ms slice
    L = 3200 * N_VIDEO_SLICES                             # dp:36-37
    SWEEP = bool(sweep)


def _cpu_prepare(n):
    import numpy as np
    from oracle import avse_oracle as O
    return [(O.synth_speech(L, SR, i).astype(np.float32), O.synth_noise(L, i).astype(np.float32),
             SNR_SWEEP[i % 5] if SWEEP else 0.0) for i in range(n)]


def _cpu_work(pair):
    from oracle import avse_oracle as O
    s = O.AudioSignal(pair[0], SR)
    n = O.AudioSignal(pair[1], SR)
    out = O.preprocess_audio_pair_signals(s, n, SLICE_MS, N_VIDEO_SLICES, FPS, snr_db=pair[2])
    return out[0].shape[0]


def _cpu_fwd_keep(pair):
    from oracle import avse_oracle as O
    out = O.preprocess_audio_pair_signals(O.AudioSignal(pair[0], SR), O.AudioSignal(pair[1], SR), SLICE_MS, N_VIDEO_SLICES, FPS,
                                          snr_db=pair[2])
    return out[3].get_data(), out[1]


def _cpu_inv_work(item):
    from oracle import avse_oracle as O
    return O.reconstruct_speech_signal(O.AudioSignal(item[0], SR), item[1], FPS).get_number_of_samples()


_CPU_LIMIT = None


def _cpu_init():
    # one BLAS/OpenMP thread per worker: the pool itself is the parallelism (dp:194), avoid oversubscription
    global _CPU_LIMIT
    try:
        from threadpoolctl import threadpool_limits
        _CPU_LIMIT = threadpool_limits(1)
    except Exception:
        pass


_CPU_PAIRS = {}


def host_cores():
    """Host threads this process may use (affinity-aware)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_throughput(n_utts, procs):
    """audio-s/s of the oracle over n_utts 3 s pairs with `procs` worker processes (inputs prepared untimed)."""
    import multiprocessing as mp
    if n_utts not in _CPU_PAIRS:
        _CPU_PAIRS[n_utts] = _cpu_prepare(n_utts)
    pairs = _CPU_PAIRS[n_utts]
    if procs <= 1:
        t0 = time.perf_counter()
        for p in pairs:
            _cpu_work(p)
        dt = time.perf_counter() - t0
    else:
        ctx = mp.get_context("fork")
        with ctx.Pool(procs, initializer=_cpu_init) as pool:
            pool.map(_cpu_work, pairs[:procs])  # warm the workers (imports, FFT plans)
            t0 = time.perf_counter()
            pool.map(_cpu_work, pairs, chunksize=max(1, n_utts // (4 * procs)))
            dt = time.perf_counter() - t0
    return n_utts * UTT_SECONDS / dt, dt


def cpu_inverse_throughput(n_utts, procs):
    """audio-s/s of the oracle's reconstruct_speech_signal (dp:60-74) over n_utts utterances (inputs prepared untimed)."""
    import multiprocessing as mp
    if n_utts not in _CPU_PAIRS:
        _CPU_PAIRS[n_utts] = _cpu_prepare(n_utts)
    ctx = mp.get_context("fork")
    with ctx.Pool(procs, initializer=_cpu_init) as pool:
        items = pool.map(_cpu_fwd_keep, _CPU_PAIRS[n_utts])
        t0 = time.perf_counter()
        pool.map(_cpu_inv_work, items, chunksize=max(1, n_utts // (4 * procs)))
        dt = time.perf_counter() - t0
    return n_utts * UTT_SECONDS / dt, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = args.cpu_procs or host_cores()   # every host thread available (the reference itself hard-codes Pool(16), dp:194)
    n = args.cpu_sample or args.batch   # one step = the GPU arm's per-GPU batch (1,000 x 3 s: ~20-25 core-seconds)
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt = cpu_throughput(n, procs)
        if i >= args.warmup:
            vals.append((v, dt))
    total_audio = n * UTT_SECONDS * len(vals)
    total_t = sum(dt for _, dt in vals)
    value = total_audio / total_t
    line = {
        "impl": "reference", "metric": "audio-sec/sec", "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / len(vals), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.batch, args.gpus),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": procs, "kind": "port",
                         "sample": "%d x 3 s pairs per step, oracle/avse_oracle.py preprocess_audio_pair_signals (float64 numpy), "
                                   "multiprocessing Pool(%d) = all host threads (the reference hard-codes Pool(16), dp:194)" % (n, procs)},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "inverse": None if args.no_inverse else {"value": cpu_inverse_throughput(min(n, 256), procs)[0], "unit": "audio-s/s",
                                                  "what": "oracle reconstruct_speech_signal (dp:60-74), same pool"},
        "note": "reference's librosa/mediaio are not installable here; this is the float64 numpy restatement (oracle/) of dp:119-139",
    }
    print(json.dumps(line), flush=True)


def workload_config(batch, gpus):
    tag = "BASELINE configs[1]" if (UTT_SECONDS == 3.0 and not SWEEP) else ("BASELINE configs[4] (long form)" if UTT_SECONDS >= 30 else "custom")
    return {
        "workload": "%s: %d x %g s 16 kHz utterances + white noise @ %s per GPU; mix + 3x log-mel (n_fft 640, hop 160, 80 mel) + top_db floor + %d AV-aligned (80,20) slices + mixed PCM" % (
            tag, batch, UTT_SECONDS, "SNR sweep -10..+10 dB" if SWEEP else "0 dB", N_VIDEO_SLICES),
        "utterances_per_gpu": batch, "seconds_per_utterance": UTT_SECONDS, "sharding": "by utterance, no collective",
        "n_gpus": gpus,
        "l2": "per-step working set %.0f MB (inputs %.0f MB + outputs %.0f MB) > 126 MB L2; no explicit flush" % (
            batch * L * 18 / 1e6, batch * L * 8 / 1e6, batch * L * 10 / 1e6),
    }


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        # NVML polled from a thread (~1 ms period): the timed region is tens of ms, too short for `nvidia-smi -lms`
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            self.nvml = None
        if self.nvml is not None:
            self.samples = []
            self.running = True
            def poll():
                nv = self.nvml
                while self.running:
                    try:
                        sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                        mx = nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM)
                        pw = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                        self.samples.append((sm, mx, pw, rs))
                    except Exception:
                        pass
                    time.sleep(0.001)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if getattr(self, "nvml", None) is not None:
            self.running = False
            self.thread.join(timeout=2)
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                    "hw_power_brake": 0x80}
            reasons = set()
            for _, _, _, rs in self.samples:
                for nm, b in bits.items():
                    if rs & b:
                        reasons.add(nm)
            sm = [s[0] for s in self.samples]
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(s[1] for s in self.samples) if sm else None,
                    "power_w_max": max(s[2] for s in self.samples) if sm else None, "samples": len(sm), "reasons": sorted(reasons),
                    "source": "NVML polled during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def synth_batch(torch, B, device, seed):
    """Harmonic 'voiced' speech (f0 120 +- 30 Hz, 29 harmonics ~1/k, slow envelope, peak ~0.3) + white noise sigma 0.05 (SURVEY 8(d))."""
    g = torch.Generator(device=device).manual_seed(1234 + seed)
    t = torch.arange(L, device=device, dtype=torch.float32) / SR
    f0 = 120.0 + 30.0 * (2.0 * torch.rand((B, 1), generator=g, device=device) - 1.0)
    x = torch.zeros((B, L), device=device)
    for k in range(1, 30):
        ph = 2.0 * torch.pi * torch.rand((B, 1), generator=g, device=device)
        x += torch.sin(2.0 * torch.pi * k * f0 * t + ph) / k
    env = torch.sin(torch.pi * 1.5 * t + torch.rand((B, 1), generator=g, device=device)) ** 2
    x = x * env + 1e-3 * torch.randn((B, L), generator=g, device=device)
    x = 0.3 * x / x.abs().amax(dim=1, keepdim=True)
    n = 0.05 * torch.randn((B, L), generator=g, device=device)
    return x.contiguous(), n.contiguous()


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs closest to its GPU (NVML's ideal affinity) so that the pinned host buffers of the
    end-to-end pipeline are allocated on the GPU's own NUMA node; matters when several ranks share one host."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


def copy_ceiling(torch, dist, world, device, h_in, h_out, n_chunks, steps, barrier):
    """Host-link ceiling of the e2e step: the SAME pinned buffers and byte counts moved by bare cudaMemcpyAsync -- H2D on one
    stream, D2H on another, chunked like the pipeline, no kernels -- on all ranks at once (max over ranks).  What the
    pipeline can reach at best on this host at this number of GPUs."""
    d_in = [torch.empty(t.shape, dtype=t.dtype, device=device) for t in h_in]
    d_out = [torch.empty(t.shape, dtype=t.dtype, device=device) for t in h_out]
    s_up, s_down = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
    B = h_in[0].shape[0]
    ch = max(1, B // n_chunks)

    def one_step():
        for lo in range(0, B, ch):
            with torch.cuda.stream(s_up):
                for h, d in zip(h_in, d_in):
                    d[lo:lo + ch].copy_(h[lo:lo + ch], non_blocking=True)
            with torch.cuda.stream(s_down):
                for h, d in zip(h_out, d_out):
                    h[lo:lo + ch].copy_(d[lo:lo + ch], non_blocking=True)

    def timed(fn, streams):
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in streams]
        for (a, _), st in zip(ev, streams):
            a.record(st)
        for _ in range(steps):
            fn()
        for (_, b), st in zip(ev, streams):
            b.record(st)
        barrier()
        ms = max(a.elapsed_time(b) for a, b in ev) / steps
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    one_step()
    both = timed(one_step, [s_up, s_down])

    def up_only():
        with torch.cuda.stream(s_up):
            for h, d in zip(h_in, d_in):
                d.copy_(h, non_blocking=True)

    def down_only():
        with torch.cuda.stream(s_down):
            for h, d in zip(h_out, d_out):
                h.copy_(d, non_blocking=True)

    up = timed(up_only, [s_up])
    down = timed(down_only, [s_down])
    nb_in = sum(t.numel() * t.element_size() for t in h_in)
    nb_out = sum(t.numel() * t.element_size() for t in h_out)
    return {"ms_per_step": both, "h2d_alone_gbs": nb_in / up / 1e6, "d2h_alone_gbs": nb_out / down / 1e6,
            "bidirectional_gbs": (nb_in + nb_out) / both / 1e6, "ranks": world,
            "what": "bare pinned cudaMemcpyAsync of the step's buffers, H2D and D2H streams concurrently, all ranks at once, max over ranks"}


def corpus_batch(torch, n, device, base_seed):
    """n utterances of the synthetic corpus (synth_batch in blocks of 500 to bound the generator's temporaries)."""
    speech = torch.empty((n, L), device=device)
    noise = torch.empty((n, L), device=device)
    for lo in range(0, n, 500):
        m = min(500, n - lo)
        s, z = synth_batch(torch, m, device, seed=base_seed + lo)
        speech[lo:lo + m] = s
        noise[lo:lo + m] = z
    return speech, noise


DUMP_BYTES = 64 * 10 ** 6
DUMP_KEYS = ("mixed", "speech", "noise", "mixed_pcm")


def dump_rows(n, bytes_per_row):
    """--dump-outputs: a fixed, seeded sample of utterance indices in [0, n), ascending, whose outputs fit DUMP_BYTES."""
    import numpy as np
    k = max(1, min(n, DUMP_BYTES // bytes_per_row))
    return np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def dump_outputs(directory, outs, launch, rows, keys=DUMP_KEYS):
    """Write utterances `rows` of the per-launch output dicts `outs` (utterance i is row i % launch of outs[i // launch])
    as directory/<key>.npy in float32."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for k in keys:
        a = np.concatenate([outs[i // launch][k][i % launch:i % launch + 1].cpu().numpy() for i in rows])
        np.save(os.path.join(directory, k + ".npy"), a.astype(np.float32))


def run_corpus(args, torch, dist, eng, eng_mod, device, rank, world):
    """BASELINE configs[2]: N utterances sharded contiguously by utterance over the ranks (engine.shard_range), no collective on
    the data path.  One step = one pass over the rank's whole shard (resident in HBM), in launches of at most --batch utterances.
    Strong scaling: the corpus is fixed, the shard shrinks with the number of GPUs."""
    lo, hi = eng_mod.shard_range(args.corpus, rank, world)
    n = hi - lo
    speech, noise = corpus_batch(torch, n, device, base_seed=lo)
    launch = min(n, max(1, args.batch if args.batch != 1000 else 12500))
    drv = eng_mod.CorpusDriver(eng, rank=rank, world_size=world, launch=launch)       # the product-level sharding driver
    assert drv.shard(args.corpus) == (lo, hi)
    outs = [dict() for _ in range(0, n, launch)]

    def step():
        drv.preprocess(speech, noise, N_VIDEO_SLICES, out=outs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    barrier()
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    rows = None
    if args.dump_outputs and rank == 0:
        rows = dump_rows(n, 4 * (3 * N_VIDEO_SLICES * 80 * 20 + L))
        dump_outputs(args.dump_outputs, outs, launch, rows)
    t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    n_max = -(-args.corpus // world)
    line = {
        "metric": "audio-sec/sec", "value": args.corpus * UTT_SECONDS / (ms * 1e-3), "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[2]: %d-utterance synthetic corpus (3 s, 16 kHz, white noise @ 0 dB) sharded contiguously by "
                               "utterance over %d B200 (engine.shard_range): mix + 3x log-mel + top_db floor + 15 AV-aligned slices + mixed PCM" % (args.corpus, world),
                   "corpus_utterances": args.corpus, "utterances_per_gpu": n_max, "utterances_per_launch": launch,
                   "sharding": "contiguous by utterance, no collective", "n_gpus": world,
                   "l2": "per-launch working set %.1f GB >> 126 MB L2; no explicit flush" % (launch * L * 18 / 1e9)},
        "roofline": {"bound": "hbm", "kernel": "step (snr_factor + avse_forward4_kernel + floor)", "achieved": n_max * L * BYTES_PER_SAMPLE_PAIR / (ms * 1e-3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": n_max * L * BYTES_PER_SAMPLE_PAIR / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                     "note": "whole step of the largest shard (per-kernel figures: the default workload's line)"},
        "gpu_launches": 3 * len(outs) * args.steps, "clocks": clocks, "cpu_baseline": None, "e2e": None,
    }
    if rows is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "rows": rows.tolist()}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def set_host_memory_policy(policy):
    """policy "interleave": spread this process's future host allocations (the pinned staging buffers) round-robin over all NUMA
    nodes (set_mempolicy(MPOL_INTERLEAVE)); "local": the default first-touch policy.  Returns the node count seen, or None."""
    if policy != "interleave":
        return None
    try:
        import ctypes
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        if len(nodes) < 2:
            return len(nodes)
        mask = ctypes.c_ulong(sum(1 << n for n in nodes))
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 3, ctypes.byref(mask), ctypes.c_ulong(max(nodes) + 2))      # x86_64 set_mempolicy, MPOL_INTERLEAVE
        return len(nodes) if rc == 0 else None
    except Exception:
        return None


def main():
    args = parse_args()
    set_workload(args.seconds, args.snr_sweep)
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists for the product path)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    eng_mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    eng = eng_mod.SpectralEngine(SR, FPS, SLICE_MS, device=device)
    B = args.batch
    if args.corpus:
        return run_corpus(args, torch, dist, eng, eng_mod, device, rank, world)

    speech, noise = synth_batch(torch, B, device, seed=rank)
    T = eng.n_frames(L)
    out = {}
    snr = torch.tensor([SNR_SWEEP[i % 5] for i in range(B)], dtype=torch.float32, device=device) if SWEEP else None

    ev_k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev_k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]

    def step(i=None):
        factor, max_key = eng.snr_factor(speech, noise, snr_db=snr, max_key=out.get("max_key"))
        if i is not None:
            ev_k0[i].record()
        res = eng.forward_raw(speech, noise, L=L, factor=factor, n_slices=N_VIDEO_SLICES, max_key=max_key, out=out)
        if i is not None:
            ev_k1[i].record()
        eng.floor3_(res["speech"], res["noise"], res["mixed"], max_key)
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    rows = None
    if args.dump_outputs and rank == 0:
        # row budget includes the reconstructed PCM of the inverse section (shorter than L)
        rows = dump_rows(B, 4 * (3 * N_VIDEO_SLICES * 80 * 20 + 2 * L))
        dump_outputs(args.dump_outputs, [out], B, rows)
    ms_total = e0.elapsed_time(e1)
    k_ms = sum(a.elapsed_time(b) for a, b in zip(ev_k0, ev_k1)) / args.steps
    tmax = torch.tensor([ms_total, k_ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total, k_ms_max = float(tmax[0]), float(tmax[1])
    ms_per_step = ms_total / args.steps
    value = world * B * UTT_SECONDS / (ms_per_step * 1e-3)

    # ---------------- roofline of the dominant kernel ----------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650 GB/s"
    alg_bytes = B * L * BYTES_PER_SAMPLE_PAIR
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "forward_kernel_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "avse_forward4_kernel<float, false, false>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_per_step, "peak_source": peak_src,
                "note": "fused FFT kernel bound by FP32 issue + the shared-memory data pipe, not by HBM; see DESIGN.md section 5 and profiles/"}

    line = {
        "metric": "audio-sec/sec", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(B, world), "roofline": roofline,
        "gpu_launches": 3 * args.steps, "clocks": clocks, "host_cpus_bound_to_gpu_numa_node": numa,
    }
    if rows is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "rows": rows.tolist()}

    # ---------------- steady state: the same step back to back for >= --sustain-s seconds ----------------
    if args.sustain_s > 0:
        # blocks of steps, each bracketed by CUDA events, until the events add up to the requested time (the host stays ahead:
        # a block is queued while the previous one still runs only at the block boundary, one ~20 us bubble per >= 0.25 s block)
        blk = max(args.steps, int(0.25 / (ms_per_step * 1e-3)) + 1)
        sampler2 = ClockSampler(local_rank)
        barrier()
        if rank == 0:
            sampler2.start()
        sus_total, n_s = 0.0, 0
        while sus_total < args.sustain_s * 1e3:
            s0 = torch.cuda.Event(enable_timing=True)
            s1 = torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(blk):
                step()
            s1.record()
            s1.synchronize()
            ts = torch.tensor([s0.elapsed_time(s1)], device=device, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)      # every rank sees the same total and leaves the loop together
            sus_total += float(ts[0])
            n_s += blk
        barrier()
        clocks2 = sampler2.stop() if rank == 0 else None
        sus_ms = sus_total / n_s
        line["sustained"] = {"value": world * B * UTT_SECONDS / (sus_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": sus_ms, "steps": n_s,
                             "seconds": sus_total * 1e-3, "clocks": clocks2,
                             "note": "same step() as the headline, back to back in blocks of %d; the headline's %d timed steps last only %.0f ms" % (
                                 blk, args.steps, ms_total)}

    # ---------------- inverse path (config 4), reported beside the headline ----------------
    if not args.no_inverse and hasattr(eng._lib, "avse_inverse"):
        res = step()
        mixed_pcm = res["mixed_pcm"]
        mel = res["speech"]
        for _ in range(3):
            eng.reconstruct(mixed_pcm, mel)
        barrier()
        i0 = torch.cuda.Event(enable_timing=True)
        i1 = torch.cuda.Event(enable_timing=True)
        i0.record()
        for _ in range(args.steps):
            eng.reconstruct(mixed_pcm, mel)
        i1.record()
        barrier()
        if rows is not None:
            # one more call on the same inputs, after the timed region: holding each timed call's output alive would change
            # what the allocator does inside it
            dump_outputs(args.dump_outputs, [{"recon": eng.reconstruct(mixed_pcm, mel)}], B, rows, keys=("recon",))
        inv_ms = i0.elapsed_time(i1) / args.steps
        tinv = torch.tensor([inv_ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tinv, op=dist.ReduceOp.MAX)
        inv_ms = float(tinv[0])
        t_use = min(20 * N_VIDEO_SLICES, T)
        inv_bytes = B * t_use * INV_BYTES_PER_FRAME
        line["inverse"] = {"workload": "BASELINE configs[3]: %d enhanced mel-spectrograms (%d,80,20) + mixture PCM -> waveforms per GPU" % (B, N_VIDEO_SLICES),
                           "value": world * B * UTT_SECONDS / (inv_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": inv_ms,
                           "roofline": {"bound": "hbm", "kernel": "avse_inverse8_kernel<false, float>", "achieved": inv_bytes / (inv_ms * 1e-3) / 1e9,
                                        "peak": peak, "unit": "GB/s", "frac": inv_bytes / (inv_ms * 1e-3) / 1e9 / peak}}

    # ---------------- SURVEY 8(f) neighbours of the path: HBM-bound kernels, each against the copy roofline ----------------
    if not args.no_aux and rank == 0:
        def timed(fn, n=10):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a0 = torch.cuda.Event(enable_timing=True)
            a1 = torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n):
                fn()
            a1.record()
            torch.cuda.synchronize()
            return a0.elapsed_time(a1) / n
        res = step()
        rows = B * N_VIDEO_SLICES
        perm = torch.randperm(rows, device=device)
        ms = timed(lambda: eng.make_sample_set(res["mixed"], res["speech"], permutation=perm, check=False))
        gb = 2 * 2 * rows * 6400 / 1e9                       # two arrays, every row read once and written once
        aux = {"make_sample_set": {"kernel": "avse_gather_rows_kernel", "what": "se:241-262: concat + one shared permutation of %d (80,20) slices x 2 arrays" % rows,
                                   "ms": ms, "achieved_gbs": gb / (ms * 1e-3), "frac_of_hbm_peak": gb / (ms * 1e-3) / peak,
                                   "note": "SpectralEngine.make_sample_set incl. its output allocations; asynchronous (check=False)"}}
        nv = 2000
        video = torch.rand((nv, 128, 128, 5), device=device) * 255.0
        vn_holder = {}
        ms = timed(lambda: vn_holder.__setitem__("vn", eng_mod.VideoNormalizer(eng, video)))
        gb = video.numel() * 4 / 1e9
        aux["video_stats"] = {"kernel": "avse_video_stats_kernel<true>", "what": "dp:201-205: per-pixel mean / std over %d x (128,128,5) crops" % nv,
                              "ms": ms, "achieved_gbs": gb / (ms * 1e-3), "frac_of_hbm_peak": gb / (ms * 1e-3) / peak}
        ms = timed(lambda: vn_holder["vn"].normalize(video))
        aux["video_normalize"] = {"kernel": "avse_video_normalize_kernel<true>", "what": "dp:207-212 in place (read + write)",
                                  "ms": ms, "achieved_gbs": 2 * gb / (ms * 1e-3), "frac_of_hbm_peak": 2 * gb / (ms * 1e-3) / peak}
        ms = timed(lambda: eng_mod.mse(eng, res["mixed"], res["speech"]))
        gb = 2 * res["mixed"].numel() * 4 / 1e9
        aux["mse"] = {"kernel": "avse_mse_kernel", "what": "network.py:214-220 loss over the step's slices", "ms": ms,
                      "achieved_gbs": gb / (ms * 1e-3), "frac_of_hbm_peak": gb / (ms * 1e-3) / peak}
        del video, vn_holder
        line["aux"] = aux

    # ---------------- end to end through the host-facing API ----------------
    if not args.no_e2e:
        h_s = torch.empty((B, L), dtype=torch.float32, pin_memory=True)
        h_n = torch.empty((B, L), dtype=torch.float32, pin_memory=True)
        h_s.copy_(speech)
        h_n.copy_(noise)
        shape = (B, N_VIDEO_SLICES, 80, 20)
        h_out = [torch.empty(shape, dtype=torch.float32, pin_memory=True) for _ in range(3)]
        h_pcm = torch.empty((B, L), dtype=torch.float32, pin_memory=True)
        # the package's host-facing pipeline: chunks round-robin over 3 streams, H2D / kernels / D2H of neighbouring chunks
        # (and of consecutive steps) overlap; every copy is inside the timed region
        NCH = args.e2e_chunks if B % args.e2e_chunks == 0 else 1
        pipe = eng_mod.HostPipeline(eng, L, N_VIDEO_SLICES, chunk=B // NCH, n_streams=args.e2e_streams)
        main = torch.cuda.current_stream(device)

        def e2e_step():
            pipe.submit(h_s, h_n, h_out[0], h_out[1], h_out[2], h_pcm)

        pipe.begin_after(main)
        for _ in range(2):
            e2e_step()
        pipe.join(main)
        barrier()
        steps_e = max(3, min(args.steps, 10))
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        pipe.begin_after(main)
        for _ in range(steps_e):
            e2e_step()
        pipe.join(main)
        t1.record()
        barrier()
        e_ms = t0.elapsed_time(t1) / steps_e
        te = torch.tensor([e_ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e_ms = float(te[0])
        d2h = 3 * B * N_VIDEO_SLICES * 80 * 20 * 4 + B * L * 4
        ceiling = copy_ceiling(torch, dist, world, device, [h_s, h_n], h_out + [h_pcm], NCH, steps_e, barrier)
        line["e2e"] = {"value": world * B * UTT_SECONDS / (e_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": e_ms,
                       "h2d_bytes_per_step": 2 * B * L * 4, "d2h_bytes_per_step": d2h,
                       "ceiling": ceiling, "frac_of_ceiling": ceiling["ms_per_step"] / e_ms,
                       "api": "engine.HostPipeline.submit (SNR factor + fused forward + floor over the C ABI) on pinned host buffers; %d chunks per step round-robin over %d streams so H2D, kernels and D2H overlap within and across steps; all copies inside the timed region" % (NCH, args.e2e_streams),
                       "gpu_launches": 3 * NCH * steps_e,
                       "bound": "PCIe: D2H %.0f MB + H2D %.0f MB per step" % (d2h / 1e6, 2 * B * L * 4 / 1e6)}

        # the same pipeline fed with raw int16 WAV samples (the reference's on-disk format, dp:122-123): half the H2D bytes
        del pipe
        scale = 32767.0 / max(float(speech.abs().max()), float(noise.abs().max()))
        h_s16 = torch.empty((B, L), dtype=torch.int16, pin_memory=True)
        h_n16 = torch.empty((B, L), dtype=torch.int16, pin_memory=True)
        h_s16.copy_((speech * scale).round().to(torch.int16))
        h_n16.copy_((noise * scale).round().to(torch.int16))
        pipe16 = eng_mod.HostPipeline(eng, L, N_VIDEO_SLICES, chunk=B // NCH, n_streams=args.e2e_streams, sample_dtype=torch.int16)
        pipe16.begin_after(main)
        for _ in range(2):
            pipe16.submit(h_s16, h_n16, h_out[0], h_out[1], h_out[2], h_pcm)
        pipe16.join(main)
        barrier()
        t0.record()
        pipe16.begin_after(main)
        for _ in range(steps_e):
            pipe16.submit(h_s16, h_n16, h_out[0], h_out[1], h_out[2], h_pcm)
        pipe16.join(main)
        t1.record()
        barrier()
        e16 = t0.elapsed_time(t1) / steps_e
        te = torch.tensor([e16], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e16 = float(te[0])
        line["e2e_int16_input"] = {"value": world * B * UTT_SECONDS / (e16 * 1e-3), "unit": "audio-s/s", "ms_per_step": e16,
                                   "h2d_bytes_per_step": 2 * B * L * 2, "d2h_bytes_per_step": d2h,
                                   "note": "same pipeline, host inputs as int16 WAV samples decoded inside the kernels"}

    # ---------------- CPU baseline beside it (rank 0, N == 1 only) ----------------
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))     # the CPU baseline gets every host thread again
        except Exception:
            pass
        procs = args.cpu_procs or host_cores()
        n = args.cpu_sample or B     # the whole per-GPU batch once: ~20-25 core-seconds of float64 numpy
        v, dt = cpu_throughput(n, procs)
        line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": procs, "kind": "port",
                                "sample": "%d x 3 s pairs (%.1f s wall), oracle/avse_oracle.py float64 restatement of dp:119-139, "
                                          "Pool(%d) = all host threads (reference: Pool(16), dp:194)" % (n, dt, procs)}
    elif rank == 0:
        line["cpu_baseline"] = None

    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
