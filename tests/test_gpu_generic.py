"""GPU parity of the generic-geometry kernels (avse_create_ex, SURVEY 8(f) row 3): every n_fft the reference derives from
(sample rate, video frame rate) -- dp:44-45 -- against the float64 oracle, forward and inverse, at BASELINE.json's
tolerances.  Includes the reference's own odd-n_fft quirk (30 fps -> 533; librosa.istft then infers 532, dp:114)."""
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import FRAME_RATES, frame_rate_fps

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (sample rate, fps): n_fft 320 (16x20), 666 (18x37), 533 (13x41, odd), 1764 (42x42), 320 @ 8 kHz, 1920 (40x48), then the
# frame rates real videos carry (tests.cases.FRAME_RATES: prime, odd, rank-deficient and the largest sizes)
CONFIGS = [(16000, 50.0), (16000, 24.0), (16000, 30.0), (44100, 25.0), (8000, 25.0), (48000, 25.0)] + \
    [(g["sr"], frame_rate_fps(g)) for g in FRAME_RATES]


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


def _d(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _case(sr, n, seed):
    s = O.synth_speech(n, sr, seed).astype(np.float32)
    z = O.synth_noise(n, seed).astype(np.float32)
    return s, z


@pytest.mark.parametrize("sr,fps", CONFIGS, ids=["%d_%g" % c for c in CONFIGS])
def test_generic_pair_and_inverse_match_oracle(mod, sr, fps):
    eng = mod.SpectralEngine(sr, fps, 200, device="cuda:0")      # fmax 8000 like the reference (dp:88), also at 8 kHz
    assert not eng.specialised
    nvs = 6
    n_s = [int(1.25 * sr), int(0.9 * sr), int(1.2 * sr) + 17]
    snrs = [0.0, -10.0, 5.0]
    W = max(n_s)
    S = np.zeros((3, W), np.float32)
    Z = np.zeros((3, W), np.float32)
    for i, n in enumerate(n_s):
        s, z = _case(sr, n, 300 + i)
        S[i, :n], Z[i, :n] = s, z
    lens = _d(np.array(n_s, np.int32))
    mixed, speech, noise, pcm = eng.preprocess_pairs(_d(S), _d(Z), nvs, lengths=lens, snr_db=_d(np.array(snrs, np.float32)))
    rec = eng.reconstruct(pcm, speech)
    for i, n in enumerate(n_s):
        sp = O.AudioSignal(S[i, :n].astype(np.float64), sr)
        nz = O.AudioSignal(Z[i, :n].astype(np.float64), sr)
        r_mixed, r_speech, r_noise, r_sig = O.preprocess_audio_pair_signals(sp, nz, 200, nvs, fps, snr_db=snrs[i])
        assert tuple(mixed[i].shape) == r_mixed.shape == (r_mixed.shape[0], 80, eng.spss)
        for name, got, ref in (("mixed", mixed, r_mixed), ("speech", speech, r_speech), ("noise", noise, r_noise)):
            err = np.max(np.abs(got[i].cpu().numpy() - ref))
            assert err <= TOL_DB, (sr, fps, i, name, err)
        rp = r_sig.get_data()
        scale = np.max(np.abs(rp))
        assert np.max(np.abs(pcm[i].cpu().numpy() - rp)) <= TOL_PCM * scale
        # inverse on the GPU's own float32 outputs (so both sides start from identical inputs)
        sig = O.AudioSignal(pcm[i].double().cpu().numpy(), sr)
        want = O.reconstruct_speech_signal(sig, speech[i].double().cpu().numpy(), fps).get_data()
        got = rec[i].cpu().numpy()
        assert got.shape == want.shape, (got.shape, want.shape)
        assert np.max(np.abs(got - want)) <= TOL_PCM * scale, (sr, fps, i, np.max(np.abs(got - want)) / scale)


def test_generic_spectrogram_phase_and_mirror_functions(mod):
    dp = importlib.import_module("audio-visual-speech-enhancement_b200.data_processor")
    sr, n_fft, hop = 16000, 320, 80
    x = (O.synth_speech(12000, sr, 5) + O.synth_noise(12000, 5)).astype(np.float32)
    mag, phase = dp.signal_to_spectrogram(dp.AudioSignal(x.copy(), sr), n_fft, hop)
    r_mag, r_phase = O.signal_to_spectrogram(O.AudioSignal(x.astype(np.float64), sr), n_fft, hop)
    assert mag.shape == r_mag.shape == (80, 151) and phase.shape == r_phase.shape == (161, 151)
    assert np.max(np.abs(mag - r_mag)) <= TOL_DB
    D = O.stft(x.astype(np.float64), n_fft, hop)
    strong = np.abs(D) > 1e-3 * np.max(np.abs(D))
    assert np.max(np.abs(phase - r_phase)[strong]) < 1e-3
    got = dp.reconstruct_signal_from_spectrogram(r_mag, r_phase, sr, n_fft, hop).get_data()
    want = O.reconstruct_signal_from_spectrogram(r_mag, r_phase, sr, n_fft, hop).get_data()
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= TOL_PCM * np.max(np.abs(x))
    # preprocess_audio_signal at 50 fps: (n, 80, 40) slices, padded in place (dp:39-40)
    a = dp.AudioSignal(x[:11000].copy(), sr)
    sl = dp.preprocess_audio_signal(a, 200, 4, 50.0)
    ref = O.preprocess_audio_signal(O.AudioSignal(x[:11000].astype(np.float64), sr), 200, 4, 50.0)
    assert sl.shape == ref.shape == (4, 80, 40) and a.get_number_of_samples() == 12800
    assert np.max(np.abs(sl - ref)) <= TOL_DB


def test_generic_kernels_agree_with_the_specialised_ones_at_640():
    # the same library, forced onto the generic kernels at n_fft 640 (AVSE_FORCE_GENERIC=1), in a fresh process
    code = r'''
import importlib, sys, numpy as np, torch
sys.path.insert(0, %r)
from tests.cases import GOLDEN_CASES, make_inputs, oracle_pair, fitted_noise
mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
eng = mod.SpectralEngine(16000, 25.0, 200, device="cuda:0")
assert not eng.specialised
for case in GOLDEN_CASES:
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    out = eng.preprocess_pairs(d(s[None]), d(nf[None]), case["nvs"], lengths=d(np.array([len(s)], np.int32)),
                               snr_db=d(np.array([case["snr"]], np.float32)))
    ref = oracle_pair(case)
    for k, g in zip(("mixed", "speech", "noise"), out[:3]):
        assert np.max(np.abs(g[0].cpu().numpy() - ref[k])) <= 1e-3, (case["name"], k)
    rec = eng.reconstruct(out[3], out[1])[0].cpu().numpy()
    scale = np.max(np.abs(ref["mixed_pcm"]))
    assert np.max(np.abs(rec - ref["recon"])) <= 1e-4 * scale, case["name"]
print("generic-at-640 ok")
''' % ROOT
    env = dict(os.environ, AVSE_FORCE_GENERIC="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "generic-at-640 ok" in r.stdout, r.stdout + r.stderr


def test_generic_int16_in_and_out(mod):
    eng = mod.SpectralEngine(16000, 50.0, 200, device="cuda:0")
    rng = np.random.RandomState(3)
    s16 = (rng.randn(2, 19200) * 3000).astype(np.int16)
    n16 = (rng.randn(2, 19200) * 900).astype(np.int16)
    a = eng.preprocess_pairs(_d(s16), _d(n16), 6)
    b = eng.preprocess_pairs(_d(s16.astype(np.float32)), _d(n16.astype(np.float32)), 6)
    for x, y in zip(a, b):
        assert torch.equal(x, y)                       # int16 -> float is exact
    f32 = eng.reconstruct(a[3], a[0] + 6.0)
    i16 = eng.reconstruct(a[3], a[0] + 6.0, out_dtype=torch.int16)
    assert torch.equal(i16, torch.clamp(f32, -32768.0, 32767.0).to(torch.int32).to(torch.int16))


def test_generic_kernels_tile_short_noise_in_kernel(mod):
    """dp:125-128 on the generic path (50 fps: n_fft 320): the noise row holds only the file's own samples (rest poisoned) and the
    kernels address noise[i mod Ln]; result == the explicit host-side tiling."""
    sr, fps, nvs = 16000, 50.0, 6
    eng = mod.SpectralEngine(sr, fps, 200, device="cuda:0")
    assert not eng.specialised
    n_s, n_n = [19200, 15000, 19200], [4000, 333, 25000]
    W = max(n_s)
    S = np.zeros((3, W), np.float32)
    Zp = np.full((3, W), np.nan, np.float32)
    Zf = np.zeros((3, W), np.float32)
    for i in range(3):
        s, _ = _case(sr, n_s[i], 500 + i)
        z = O.synth_noise(n_n[i], 500 + i).astype(np.float32)
        S[i, :n_s[i]] = s
        m = min(n_n[i], n_s[i])
        Zp[i, :m] = z[:m]
        Zf[i, :n_s[i]] = z[np.arange(n_s[i]) % n_n[i]] if n_n[i] < n_s[i] else z[:n_s[i]]
    lens = _d(np.array(n_s, np.int32))
    nl = _d(np.array([min(a, b) for a, b in zip(n_n, n_s)], np.int32))
    got = eng.preprocess_pairs(_d(S), _d(Zp), nvs, lengths=lens, noise_lengths=nl)
    ref = eng.preprocess_pairs(_d(S), _d(Zf), nvs, lengths=lens)
    for a, b in zip(got, ref):
        assert torch.isfinite(a).all() and torch.allclose(a, b, rtol=0, atol=2e-5)
