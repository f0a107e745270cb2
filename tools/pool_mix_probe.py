#!/usr/bin/env python
"""Timing probe of pooled-pair mixing (SpectralEngine.mix_pools / avse_mix_pooled) against the copy path it replaces.

Per step: 1 000 rows of 3 s (16 kHz, 15 video slices) drawn from a pool of 1 000 speech clips of 3 s and 200 noise clips of
1-10 s, random noise offsets and SNRs in [-10, 10] dB.  Three workloads, alternated in one process (CUDA events, medians and
spread over rounds):
  (a) pooled  -- mix_pools on the pairing;
  (b) copy    -- the same pairing materialised with torch (speech row gather, rolled + tiled noise) and run through
                 preprocess_pairs(..., noise_lengths=...);
  (c) tiled   -- the existing tiled workload: preprocess_pairs(speech [1000, L], noise [1000, L], noise_lengths=min(Ln, L)),
                 what the drop-in preprocess_data runs.
--only-tiled times (c) alone; with --tree pointing at another checkout (and AVSE_B200_LIB at its library) it measures that
build's (c) for a before / after comparison.  Prints one JSON line.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import sys

sys.dont_write_bytecode = True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="steps per round and workload")
    ap.add_argument("--only-tiled", action="store_true")
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree))
    import numpy as np
    import torch

    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    sr, nvs, B = 16000, 15, 1000
    L = 3200 * nvs
    eng = mod.SpectralEngine(sr, 25.0, 200, device="cuda:0")
    dev = eng.device
    g = torch.Generator(device="cpu")
    g.manual_seed(0)
    t = torch.arange(L, dtype=torch.float64) / sr
    # speech: 1 000 clips of 3 s (harmonic series with a slow envelope, per-clip pitch); noise: 200 clips of 1-10 s
    f0 = 100.0 + 60.0 * torch.rand(1000, 1, generator=g, dtype=torch.float64)
    speech = (0.3 * torch.sin(2 * np.pi * f0 * t) * torch.sin(np.pi * 1.5 * t) ** 2).to(torch.float32).to(dev)
    speech_len = torch.full((1000,), L, dtype=torch.int32, device=dev)
    nlen_h = torch.randint(sr, 10 * sr + 1, (200,), generator=g)
    nstride = (int(nlen_h.max()) + 3) // 4 * 4
    noise = (0.05 * torch.randn(200, nstride, generator=g)).to(dev)
    noise_len = nlen_h.to(torch.int32).to(dev)

    si = torch.randperm(1000, generator=g)[:B]
    ni = torch.randint(0, 200, (B,), generator=g)
    off = (torch.rand(B, generator=g, dtype=torch.float64) * nlen_h[ni].double()).long().clamp_max(nlen_h[ni] - 1).to(torch.int32)
    snr = (-10.0 + 20.0 * torch.rand(B, generator=g)).to(torch.float32)
    si_d, ni_d, off_d, snr_d = si.to(dev), ni.to(dev), off.to(dev), snr.to(dev)
    ln_d = noise_len[ni_d].long()

    # (c) the tiled workload: the noise rows carry their own clip (first min(Ln, L) samples), tiled inside the kernels
    Zc = torch.zeros((B, L), dtype=torch.float32, device=dev)
    m = min(L, nstride)
    Zc[:, :m] = noise[ni_d, :m]
    nl_c = torch.clamp(ln_d, max=L).to(torch.int32)
    Sc = speech[si_d].contiguous()
    lens_c = speech_len[si_d]

    def pooled(out):
        return eng.mix_pools(speech, speech_len, noise, noise_len, si_d, ni_d, nvs, noise_offset=off_d, snr_db=snr_d, out=out, check=False)

    def copy(out):
        S = speech[si_d]
        idx = (off_d.long().unsqueeze(1) + torch.arange(L, device=dev).unsqueeze(0)) % ln_d.unsqueeze(1)
        N = noise.view(-1)[ni_d.unsqueeze(1) * nstride + idx]
        return eng.preprocess_pairs(S, N, nvs, lengths=lens_c, snr_db=snr_d, out=out, noise_lengths=lens_c)

    def tiled(out):
        return eng.preprocess_pairs(Sc, Zc, nvs, lengths=lens_c, snr_db=snr_d, out=out, noise_lengths=nl_c)

    work = {"tiled": tiled} if args.only_tiled else {"pooled": pooled, "copy": copy, "tiled": tiled}
    outs = {k: {} for k in work}
    for k, fn in work.items():          # warm-up (and allocation of the re-used outputs)
        for _ in range(3):
            fn(outs[k])
    torch.cuda.synchronize()
    if not args.only_tiled:              # the pooled call computes what the copy path computes (its factors to ~1 ulp)
        a, b = pooled(outs["pooled"]), copy(outs["copy"])
        torch.cuda.synchronize()
        diff_db = max(float((x - y).abs().max()) for x, y in zip(a[:3], b[:3]))
    times = {k: [] for k in work}
    for _ in range(args.rounds):
        for k, fn in work.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn(outs[k])
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / args.steps)
    res = {"gpu": torch.cuda.get_device_name(0), "rows": B, "seconds_per_row": L / sr, "rounds": args.rounds, "steps": args.steps,
           "tree": os.path.abspath(args.tree), "lib": os.environ.get("AVSE_B200_LIB", "in-tree")}
    for k, v in times.items():
        res[k + "_ms"] = {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
    if not args.only_tiled:
        res["pooled_vs_copy_max_db"] = diff_db
    print(json.dumps(res))


if __name__ == "__main__":
    main()
