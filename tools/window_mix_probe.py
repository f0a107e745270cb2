#!/usr/bin/env python
"""Timing probe of training windows: mix_pools with speech_start and the video gather (avse_gather_video).

Per step: 1 000 rows of 3 s windows (16 kHz, 15 video slices) cut at random slice starts from a pool of 1 000 speech clips of
20 s (1.28 GB of float32 samples, ten times the L2), paired with 200 noise clips of 1-10 s at random offsets and SNRs.
Workloads, alternated in one process (CUDA events, medians and spread over rounds):
  windowed  -- mix_pools(..., speech_start=...) on the 20 s pool;
  whole     -- the same pairing without starts: every row's statistics run over its whole 20 s clip (the old behaviour);
  clips3s   -- the same pairing on a pool of 3 s clips without starts (the workload a pre-cut corpus gives);
  gather_u8 / gather_f32 -- avse_gather_video of the rows' 15 000 video slices (128 x 128 x 5) from a uint8 / float32 pool of
               1 000 x 100 slices (8.2 / 32.8 GB), normalised, in GB/s of pool reads + float32 writes;
  torch_u8  -- what it replaces: pool[idx].float() then VideoNormalizer.normalize;
  copy      -- a 4 GB device-to-device copy, the HBM copy roofline the gathers are compared against.
Reads the card's name and power limit in the same run.  Prints one JSON line.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5, help="steps per round and workload")
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import numpy as np
    import torch

    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    sr, nvs, B, Ns, Nn, clip_s = 16000, 15, 1000, 1000, 200, 20
    sps = 3200
    L = sps * nvs
    eng = mod.SpectralEngine(sr, 25.0, 200, device="cuda:0")
    dev = eng.device
    g = torch.Generator(device="cpu")
    g.manual_seed(0)
    Ls = clip_s * sr
    # speech: harmonic series with a slow envelope and a per-clip pitch, built on the device
    t = torch.arange(Ls, dtype=torch.float64, device=dev) / sr
    f0 = (100.0 + 60.0 * torch.rand(Ns, 1, generator=g, dtype=torch.float64)).to(dev)
    speech = torch.empty((Ns, Ls), dtype=torch.float32, device=dev)
    for k in range(0, Ns, 100):
        speech[k:k + 100] = (0.3 * torch.sin(2 * np.pi * f0[k:k + 100] * t) * torch.sin(np.pi * 0.37 * t) ** 2).to(torch.float32)
    speech_len = torch.full((Ns,), Ls, dtype=torch.int32, device=dev)
    speech3 = speech[:, :L].contiguous()
    speech3_len = torch.full((Ns,), L, dtype=torch.int32, device=dev)
    nlen_h = torch.randint(sr, 10 * sr + 1, (Nn,), generator=g)
    noise = (0.05 * torch.randn(Nn, (int(nlen_h.max()) + 3) // 4 * 4, generator=g)).to(dev)
    noise_len = nlen_h.to(torch.int32).to(dev)

    m = mod.DynamicMixer(eng, speech, speech_len, noise, noise_len, nvs, seed=0, clip_slices=torch.full((Ns,), clip_s * 5))
    si, ni, off, snr, start = m.draw(B)

    def windowed(out):
        return eng.mix_pools(speech, speech_len, noise, noise_len, si, ni, nvs, noise_offset=off, snr_db=snr, out=out, check=False,
                             speech_start=start)

    def whole(out):
        return eng.mix_pools(speech, speech_len, noise, noise_len, si, ni, nvs, noise_offset=off, snr_db=snr, out=out, check=False)

    def clips3s(out):
        return eng.mix_pools(speech3, speech3_len, noise, noise_len, si, ni, nvs, noise_offset=off, snr_db=snr, out=out, check=False)

    # video: 100 slices of 128 x 128 x 5 per clip; the 15 slices of every row's window
    H, W, F, S = 128, 128, 5, clip_s * 5
    vid8 = torch.randint(0, 256, (Ns, S, H, W, F), dtype=torch.uint8, device=dev)
    stats_src = vid8[:8].reshape(-1, H, W, F).float()
    norm = mod.VideoNormalizer(eng, stats_src)
    del stats_src
    k = start.long() // sps
    nb = torch.full((B,), nvs, dtype=torch.int64, device=dev)
    N = B * nvs
    idx = mod.video_slice_index(si, k, nb, nvs, S, torch.randperm(N, device=dev))
    row = H * W * F
    flat8 = vid8.view(-1, H, W, F)

    def gather_u8(out):
        return eng.gather_video(vid8, idx, normalizer=norm, check=False)

    def torch_u8(out):
        return norm.normalize(flat8[idx].float())

    cp_src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    cp_dst = torch.empty_like(cp_src)

    def copy(out):
        cp_dst.copy_(cp_src)

    work = {"windowed": windowed, "whole": whole, "clips3s": clips3s, "gather_u8": gather_u8, "torch_u8": torch_u8, "copy": copy}
    outs = {k: {} for k in work}
    for kk, fn in work.items():
        for _ in range(2):
            fn(outs[kk])
    torch.cuda.synchronize()
    # the windowed rows are the 3 s pool's rows shifted: check a few against copies made from the same windows
    ref_rows = [0, 1, 499, 999]
    cut = torch.stack([speech[int(si[b]), int(start[b]):int(start[b]) + L] for b in ref_rows])
    a = windowed(outs["windowed"])
    c = eng.mix_pools(cut, torch.full((len(ref_rows),), L, dtype=torch.int32, device=dev), noise, noise_len, torch.arange(len(ref_rows), device=dev),
                      ni[ref_rows], nvs, noise_offset=off[ref_rows], snr_db=snr[ref_rows])
    diff_db = max(float((x[ref_rows] - y).abs().max()) for x, y in zip(a[:3], c[:3]))
    gv = gather_u8(None)
    tv = torch_u8(None)
    torch.cuda.synchronize()
    gather_equal = bool(torch.equal(gv, tv))
    del gv, tv

    times = {kk: [] for kk in work}

    def timed(kk, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn(outs[kk])
        e1.record()
        e1.synchronize()
        times[kk].append(e0.elapsed_time(e1) / args.steps)

    for _ in range(args.rounds):
        for kk, fn in work.items():
            timed(kk, fn)
    # the float32 pool (32.8 GB) replaces the uint8 one for its own rounds
    del vid8, flat8
    torch.cuda.empty_cache()
    vid32 = torch.empty((Ns, S, H, W, F), dtype=torch.float32, device=dev)
    for c0 in range(0, Ns, 50):
        vid32[c0:c0 + 50].random_(0, 256)

    def gather_f32(out):
        return eng.gather_video(vid32, idx, normalizer=norm, check=False)

    times["gather_f32"], outs["gather_f32"] = [], {}
    for _ in range(2):
        gather_f32(None)
    for _ in range(args.rounds):
        timed("gather_f32", gather_f32)

    med = {kk: statistics.median(v) for kk, v in times.items()}
    res = {"card": card(), "gpu": torch.cuda.get_device_name(0), "rows": B, "seconds_per_row": L / sr, "clip_seconds": clip_s,
           "rounds": args.rounds, "steps": args.steps, "windowed_vs_copied_max_db": diff_db, "gather_equals_torch": gather_equal}
    for kk, v in times.items():
        res[kk + "_ms"] = {"median": round(med[kk], 4), "min": round(min(v), 4), "max": round(max(v), 4)}
    res["copy_GBps"] = round(2 * cp_src.numel() * 4 / (med["copy"] * 1e-3) / 1e9, 1)
    for kk, pix in (("gather_u8", 1), ("torch_u8", 1), ("gather_f32", 4)):
        res[kk + "_GBps"] = round(N * row * (pix + 4) / (med[kk] * 1e-3) / 1e9, 1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
