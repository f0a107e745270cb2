"""Oracle checks AT the BASELINE configurations, on bench.py's own synthetic inputs (VERDICT r1 weak #9 / next #8): the launches the
numbers are quoted on are not only invariant-checked -- individual utterances of them (first, last, and the neighbours of the
persistent kernel's tile boundaries) are compared with the float64 oracle at the north_star tolerances.

  config 2: 1 000 x 3 s in ONE launch (bench.synth_batch, seed 0: exactly what `python bench.py` times), forward + inverse
  config 3: one 12 500-utterance launch = the per-GPU shard of the 100 k corpus on 8 GPUs
  config 5: 64 x 60 s long-form batch with the -10 ... +10 dB sweep
"""
import importlib

import numpy as np
import pytest
import torch

import bench
from oracle import avse_oracle as O

pytestmark = pytest.mark.gpu

SR, FPS = 16000, 25.0
TOL_DB, TOL_PCM = 1e-3, 1e-4


@pytest.fixture(scope="module")
def eng():
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


def _check(eng, speech, noise, outs, idx, nvs, snr_db=None, inverse=None):
    mixed, sp, nz, pcm = outs
    worst = 0.0
    for u in idx:
        s = O.AudioSignal(speech[u].double().cpu().numpy(), SR)
        n = O.AudioSignal(noise[u].double().cpu().numpy(), SR)
        snr = 0.0 if snr_db is None else float(snr_db[u])
        r_mixed, r_speech, r_noise, r_sig = O.preprocess_audio_pair_signals(s, n, 200, nvs, FPS, snr_db=snr)
        for name, got, ref in (("mixed", mixed, r_mixed), ("speech", sp, r_speech), ("noise", nz, r_noise)):
            err = float(np.max(np.abs(got[u].cpu().numpy() - ref)))
            worst = max(worst, err)
            assert err <= TOL_DB, (u, name, err)
        full = float(np.max(np.abs(r_sig.get_data())))
        assert float(np.max(np.abs(pcm[u].cpu().numpy() - r_sig.get_data()))) <= TOL_PCM * full, u
        if inverse is not None:
            sig = O.AudioSignal(pcm[u].double().cpu().numpy(), SR)
            want = O.reconstruct_speech_signal(sig, sp[u].double().cpu().numpy(), FPS).get_data()
            assert float(np.max(np.abs(inverse[u].cpu().numpy() - want))) <= TOL_PCM * full, (u, "inverse")
    return worst


def _tile_boundary_utterances(B, groups_per_utt, n_warps):
    """Utterances in which a persistent warp's contiguous tile range ends and the next one begins (avse_common.h WarpSplit:
    total / n_warps tiles per warp, the remainder one apiece to the first warps)."""
    total = B * groups_per_utt
    base, extras = divmod(total, n_warps)
    picks = set()
    for gw in (1, n_warps // 2, n_warps - 1):
        u = (gw * base + min(gw, extras)) // groups_per_utt
        picks.update(x for x in (u - 1, u, u + 1) if 0 <= x < B)
    return picks


def test_config2_bench_batch_matches_oracle(eng):
    bench.set_workload(3.0, False)
    speech, noise = bench.synth_batch(torch, 1000, torch.device("cuda", 0), seed=0)
    outs = eng.preprocess_pairs(speech, noise, 15)
    rec = eng.reconstruct(outs[3], outs[1])
    idx = sorted({0, 1, 499, 998, 999} | _tile_boundary_utterances(1000, 76, 148 * 8))[:12]
    worst = _check(eng, speech, noise, outs, idx, 15, inverse=rec)
    print("config 2: %d utterances of the benchmarked launch, worst log-mel error %.2e dB" % (len(idx), worst))


def test_config3_shard_launch_matches_oracle(eng):
    bench.set_workload(3.0, False)
    B = 12500
    speech, noise = bench.corpus_batch(torch, B, torch.device("cuda", 0), base_seed=0)
    outs = eng.preprocess_pairs(speech, noise, 15)
    idx = sorted({0, 6249, B - 1} | _tile_boundary_utterances(B, 76, 148 * 8))[:8]
    worst = _check(eng, speech, noise, outs, idx, 15)
    # and the launch equals the same utterances processed as a small batch (sharding changes nothing, SURVEY 8(e))
    sub = eng.preprocess_pairs(speech[B - 7:].contiguous(), noise[B - 7:].contiguous(), 15)
    for a, b in zip(outs, sub):
        assert torch.equal(a[B - 7:], b)
    print("config 3 shard (12 500 utterances): worst log-mel error %.2e dB" % worst)


def test_config5_long_form_batch_matches_oracle(eng):
    bench.set_workload(60.0, True)
    try:
        B = 64
        speech, noise = bench.synth_batch(torch, B, torch.device("cuda", 0), seed=0)
        snr = torch.tensor([bench.SNR_SWEEP[i % 5] for i in range(B)], dtype=torch.float32, device="cuda")
        info = {}
        outs = eng.preprocess_pairs(speech, noise, 300, snr_db=snr, info=info)
        rec = eng.reconstruct(outs[3], outs[1])
        worst = _check(eng, speech, noise, outs, [0, 31, 63], 300, snr_db=snr.cpu().numpy(), inverse=rec)
        # the statistics pass (P = 8 CTAs per utterance here): factor and equaliser within float32 rounding of numpy's float64
        fac, eq = info["factor"].cpu().numpy(), info["keys"].equalizer.cpu().numpy()
        for u in (0, 31, 63):
            s, z = speech[u].double().cpu().numpy(), noise[u].double().cpu().numpy()
            wf = np.sqrt(np.var(s) / np.var(z)) * 10.0 ** (-float(snr[u]) / 20.0)
            wg = np.sqrt(np.sum(s * s) / np.sum(z * z))
            assert abs(fac[u] - wf) <= 2e-7 * wf and abs(eq[u] - wg) <= 2e-7 * wg, (u, fac[u], wf, eq[u], wg)
        print("config 5 (64 x 60 s, SNR sweep): worst log-mel error %.2e dB" % worst)
    finally:
        bench.set_workload(3.0, False)


def test_corpus_driver_shards_equal_the_whole(eng):
    """engine.CorpusDriver (the product-level multi-GPU driver): two ranks' shards, each processed in launches of 40 utterances,
    concatenate to exactly what one launch over the whole corpus gives (no collective on the data path, SURVEY 8(e))."""
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    bench.set_workload(3.0, False)
    n = 101
    speech, noise = bench.synth_batch(torch, n, torch.device("cuda", 0), seed=3)
    snr = torch.linspace(-10, 10, n, device="cuda")
    whole = eng.preprocess_pairs(speech, noise, 15, snr_db=snr)
    parts = []
    for rank in range(2):
        drv = mod.CorpusDriver(eng, rank=rank, world_size=2, launch=40)
        lo, hi = drv.shard(n)
        res = drv.preprocess(speech[lo:hi], noise[lo:hi], 15, snr_db=snr[lo:hi])
        assert len(res) == -(-(hi - lo) // 40) and drv.launches == 3 * len(res)
        parts.append([torch.cat([r[k] for r in res]) for k in range(4)])
    for k in range(4):
        assert torch.equal(torch.cat([parts[0][k], parts[1][k]]), whole[k])
