"""Timing of the differentiable reconstruction at config-4 size: 1 000 utterances x 3 s (mel slices [1000, 15, 80, 20], mixture
[1000, 48000]; the working set is larger than the 126 MB L2).

Times, with CUDA events around each iteration (after warm-up; median over --iters):
  * avse_inverse_backward alone;
  * forward + backward through autograd (SpectralEngine.reconstruct_differentiable, then y.backward(g));
  * the same computation in plain torch float32 autograd on the same GPU: torch.stft for the mixture's phase, a dense pinv(F)
    matmul, torch.istft, then y.backward(g).
The backward's algorithmic traffic is 1 920 B per reconstructed frame (read: gradient 640 B, mixture 640 B, dB 320 B; write 320 B).
Errors of both gradients against the float64 VJP of tests/inverse_vjp.py are reported on sampled rows, as max |err| / peak |oracle| per row.
Prints the card's name and power limit from the same run, and one JSON line (also written to --out when given).

    python tools/inverse_backward_bench.py [--B 1000] [--iters 30] [--warmup 5] [--rows 3] [--out result.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import avse_oracle as O  # noqa: E402
from tests import inverse_vjp as V  # noqa: E402

HBM_DENOM_GBS = 6547.0      # the project's achievable-HBM denominator (BASELINE.md)
BYTES_PER_FRAME = 1920


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    except (OSError, subprocess.TimeoutExpired):
        line = ""
    return name, line


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=1000)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rows", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inverse_backward_bench needs a CUDA device")
    eng_mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    eng = eng_mod.SpectralEngine(16000, 25.0, 200, device="cuda:0")
    B, n, L = args.B, 15, 48000
    T_use = min(20 * n, eng.n_frames(L))
    out_len = 160 * (T_use - 1)
    gen = torch.Generator(device="cuda").manual_seed(0)
    base = torch.from_numpy((O.synth_speech(L, 16000, 1) + O.synth_noise(L, 1)).astype(np.float32)).cuda()
    shifts = torch.randint(0, L, (B,), generator=gen, device="cuda")
    idx = (torch.arange(L, device="cuda")[None, :] + shifts[:, None]) % L
    pcm = (base[idx] * torch.rand(B, 1, generator=gen, device="cuda") * 2).contiguous()
    mel = (-40.0 + 12.0 * torch.randn(B, n, 80, 20, generator=gen, device="cuda")).contiguous()
    g = (torch.randn(B, out_len, generator=gen, device="cuda") / (B * out_len)).contiguous()     # d mean(.) / dy scale

    # 1) backward kernel alone
    bwd = lambda: eng._inverse_launch(pcm, mel, None, eng_mod.LAYOUT_SLICES, grad_pcm=g)
    t_bwd = timed(bwd, args.iters, args.warmup)

    # 2) forward + backward through autograd
    leaf = mel.clone().requires_grad_(True)

    def fused():
        leaf.grad = None
        eng.reconstruct_differentiable(pcm, leaf).backward(g)
    t_fused = timed(fused, args.iters, args.warmup)
    g_fused = leaf.grad.detach().clone()

    # 3) plain torch float32 autograd
    fb = torch.from_numpy(np.linalg.pinv(eng.filterbank()).astype(np.float32)).cuda()      # [321, 80]
    win = torch.hann_window(640, device="cuda")
    leaf_t = mel.clone().requires_grad_(True)

    def torch_path():
        leaf_t.grad = None
        D = torch.stft(pcm, 640, 160, window=win, center=True, pad_mode="reflect", return_complex=True)[:, :, :T_use]
        mag = D.abs()
        phase = torch.where(mag > 0, D / torch.where(mag > 0, mag, torch.ones_like(mag)), torch.ones_like(D))
        spec = leaf_t.permute(0, 2, 1, 3).reshape(B, 80, n * 20)[:, :, :T_use]
        lin = torch.matmul(fb, torch.pow(10.0, spec / 20.0))
        y = torch.istft(lin * phase, 640, 160, window=win, center=True, length=out_len)
        y.backward(g)
    t_torch = timed(torch_path, args.iters, args.warmup)
    g_torch = leaf_t.grad.detach().clone()

    # errors against the float64 oracle on sampled rows
    rows = np.linspace(0, B - 1, args.rows).astype(int)
    err_fused, err_torch = [], []
    for r in rows:
        want = V.reconstruct_speech_signal_vjp(O.AudioSignal(pcm[r].double().cpu().numpy(), 16000), mel[r].double().cpu().numpy(),
                                               25.0, g[r].double().cpu().numpy())
        peak = np.max(np.abs(want))
        err_fused.append(float(np.max(np.abs(g_fused[r].double().cpu().numpy() - want)) / peak))
        err_torch.append(float(np.max(np.abs(g_torch[r].double().cpu().numpy() - want)) / peak))

    frames = B * T_use
    gbs = BYTES_PER_FRAME * frames / (t_bwd[0] * 1e-3) / 1e9
    name, smi = card()
    res = dict(
        tool="inverse_backward_bench", card=name, nvidia_smi=smi, B=B, seconds_per_utt=L / 16000, frames=frames,
        backward_ms=t_bwd[0], backward_ms_min_max=t_bwd[1:], fused_fwd_bwd_ms=t_fused[0], fused_ms_min_max=t_fused[1:],
        torch_fp32_autograd_ms=t_torch[0], torch_ms_min_max=t_torch[1:], speedup_vs_torch=t_torch[0] / t_fused[0],
        backward_bytes=BYTES_PER_FRAME * frames, backward_GBs=gbs, backward_frac_of_6547GBs=gbs / HBM_DENOM_GBS,
        err_fused_vs_oracle=err_fused, err_torch_vs_oracle=err_torch, rows=rows.tolist(), iters=args.iters, warmup=args.warmup)
    print("card: %s (%s)" % (name, smi))
    print("backward kernel      %.3f ms   %.0f GB/s = %.1f %% of %.0f GB/s" % (t_bwd[0], gbs, 100 * gbs / HBM_DENOM_GBS, HBM_DENOM_GBS))
    print("fused fwd + bwd      %.3f ms" % t_fused[0])
    print("torch fp32 autograd  %.3f ms   (fused is %.1fx faster)" % (t_torch[0], t_torch[0] / t_fused[0]))
    print("max err / peak vs oracle: fused %s, torch %s" % (["%.2e" % e for e in err_fused], ["%.2e" % e for e in err_torch]))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
