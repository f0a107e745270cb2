"""GPU parity at BASELINE config 5: long-form 60 s utterances with an SNR sweep -10 ... +10 dB (fused mix + mel),
and the inverse path on the same long utterances.  Every utterance is checked against its own float64 oracle
(per-utterance variance / top_db max, dp:94, dp:130); tolerances are BASELINE.json's."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS, SLICE_MS

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
SNRS = [-10.0, -5.0, 0.0, 5.0, 10.0]
L60 = 60 * SR            # 960 000 samples, T = 6 001 frames, 300 slices (SURVEY Appendix B)


@pytest.fixture(scope="module")
def eng():
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    return mod.SpectralEngine(SR, FPS, SLICE_MS, device="cuda:0")


def _pair(seed, n):
    s = O.synth_speech(n, SR, seed).astype(np.float32)
    z = O.synth_noise(n, seed).astype(np.float32)
    return s, z


@pytest.fixture(scope="module")
def batch(eng):
    # utterance 4 is shorter than 60 s: zero padded to the slice multiple (dp:39-40), variance over its own length
    lens = [L60, L60, L60, L60, L60 - 123457]
    S = np.zeros((5, L60), np.float32)
    Z = np.zeros((5, L60), np.float32)
    for i, n in enumerate(lens):
        s, z = _pair(500 + i, n)
        S[i, :n], Z[i, :n] = s, z
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    info = {}
    out = eng.preprocess_pairs(d(S), d(Z), 300, lengths=d(np.array(lens, np.int32)), snr_db=d(np.array(SNRS, np.float32)), info=info)
    torch.cuda.synchronize()
    # (factor, equaliser) of the statistics pass, here at P = 8 (a cluster of 8 CTAs per utterance)
    return S, Z, lens, out, (info["factor"].cpu().numpy(), info["keys"].equalizer.cpu().numpy())


def _oracle(S, Z, lens, i):
    sp = O.AudioSignal(S[i, :lens[i]].astype(np.float64), SR)
    nz = O.AudioSignal(Z[i, :lens[i]].astype(np.float64), SR)
    return O.preprocess_audio_pair_signals(sp, nz, SLICE_MS, 300, FPS, snr_db=SNRS[i])


@pytest.mark.parametrize("i", range(5))
def test_long_form_snr_sweep_matches_oracle(batch, i):
    S, Z, lens, (mixed, speech, noise, pcm), gains = batch
    r_mixed, r_speech, r_noise, r_sig = _oracle(S, Z, lens, i)
    assert tuple(mixed.shape) == (5, 300, 80, 20)
    for name, got, ref in (("mixed", mixed, r_mixed), ("speech", speech, r_speech), ("noise", noise, r_noise)):
        err = np.max(np.abs(got[i].cpu().numpy() - ref))
        assert err <= TOL_DB, (name, SNRS[i], err)
    ref_pcm = r_sig.get_data()
    assert ref_pcm.shape == (L60,)
    assert np.max(np.abs(pcm[i].cpu().numpy() - ref_pcm)) <= TOL_PCM * np.max(np.abs(ref_pcm))
    # the mixture really sits at the requested SNR (population variances over the utterance's own length)
    n = lens[i]
    p = pcm[i, :n].double().cpu().numpy()
    s = S[i, :n].astype(np.float64)
    snr = 10.0 * np.log10(np.var(s) / np.var(p - s))
    assert abs(snr - SNRS[i]) < 1e-3
    # the statistics themselves: within float32 rounding of numpy's float64 values (a partition error of one sample is ~10 ulps)
    fac, eq = gains
    z = Z[i, :n].astype(np.float64)
    wf = np.sqrt(np.var(s) / np.var(z)) * 10.0 ** (-SNRS[i] / 20.0)
    wg = np.sqrt(np.sum(s * s) / np.sum(z * z))
    assert abs(fac[i] - wf) <= 2e-7 * wf and abs(eq[i] - wg) <= 2e-7 * wg, (i, fac[i], wf, eq[i], wg)


def test_long_form_inverse_matches_oracle(eng, batch):
    S, Z, lens, (mixed, speech, noise, pcm), gains = batch
    rec = eng.reconstruct(pcm, speech)
    assert tuple(rec.shape) == (5, 160 * (6000 - 1))          # hop * (T_use - 1), Appendix B: 959 840
    for i in (0, 4):
        sig = O.AudioSignal(pcm[i].double().cpu().numpy(), SR)
        want = O.reconstruct_speech_signal(sig, speech[i].double().cpu().numpy(), FPS).get_data()
        scale = float(pcm[i].abs().max())
        err = np.max(np.abs(rec[i].cpu().numpy() - want))
        assert err <= TOL_PCM * scale, (i, err / scale)


def test_sharded_halves_equal_the_whole(eng, batch):
    # SURVEY 8(e): utterances are independent units -- processing a contiguous shard alone gives bit-identical results
    S, Z, lens, (mixed, speech, noise, pcm), gains = batch
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    for rank in range(2):
        lo, hi = mod.shard_range(5, rank, 2)
        m2, s2, n2, p2 = eng.preprocess_pairs(d(S[lo:hi]), d(Z[lo:hi]), 300, lengths=d(np.array(lens[lo:hi], np.int32)),
                                              snr_db=d(np.array(SNRS[lo:hi], np.float32)))
        assert torch.equal(m2, mixed[lo:hi]) and torch.equal(s2, speech[lo:hi]) and torch.equal(n2, noise[lo:hi])
        assert torch.equal(p2, pcm[lo:hi])
