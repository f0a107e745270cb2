"""Pins the float64 oracle (oracle/avse_oracle.py) with independent cross-checks.

The reference ships no golden vectors (SURVEY.md section 4) and librosa/mediaio are
not installable here, so the oracle is pinned against torch.stft / torch.istft,
torchaudio's Slaney filterbank and algebraic identities instead.
"""
import numpy as np
import pytest
import torch

from oracle import avse_oracle as O

SR, NFFT, HOP = 16000, 640, 160


def _sig(n, seed=0):
    return O.synth_speech(n, SR, seed) + O.synth_noise(n, seed)


def test_stft_matches_torch():
    y = _sig(48000, 1)
    D = O.stft(y, NFFT, HOP)
    assert D.shape == (321, 301)
    ref = torch.stft(torch.from_numpy(y), NFFT, HOP, window=torch.hann_window(NFFT, periodic=True, dtype=torch.float64),
                     center=True, pad_mode="reflect", return_complex=True).numpy()
    assert np.max(np.abs(D - ref)) < 1e-11


def test_istft_roundtrip_and_torch():
    y = _sig(48000, 2)
    D = O.stft(y, NFFT, HOP)
    yr = O.istft(D, HOP)
    assert yr.shape == (48000,)
    assert np.max(np.abs(yr - y)) < 1e-12
    ref = torch.istft(torch.from_numpy(D), NFFT, HOP, window=torch.hann_window(NFFT, periodic=True, dtype=torch.float64),
                      center=True).numpy()
    assert np.max(np.abs(yr - ref)) < 1e-12


def test_istft_length_and_wss_edges():
    # dp:68-70 feeds 300 of 301 frames -> hop*(T-1) = 47840 samples (SURVEY Appendix B)
    D = O.stft(_sig(48000, 3), NFFT, HOP)[:, :300]
    assert O.istft(D, HOP).shape == (47840,)
    wss = O.window_sumsquare(300, NFFT, HOP)[NFFT // 2:-(NFFT // 2)]
    assert abs(wss[0] - 1.25) < 1e-12 and abs(wss[HOP] - 1.5) < 1e-12 and abs(wss[-1] - wss[1]) < 1e-9
    assert np.allclose(wss[HOP:-HOP], 1.5)


def test_mel_filterbank_matches_torchaudio():
    torchaudio = pytest.importorskip("torchaudio")
    fb = O.mel_filterbank(SR, NFFT, 80, 0.0, 8000.0)
    ref = torchaudio.functional.melscale_fbanks(321, 0.0, 8000.0, 80, SR, norm="slaney", mel_scale="slaney").numpy().T
    assert fb.shape == (80, 321)
    assert np.max(np.abs(fb - ref)) < 2e-7  # torchaudio builds it in float32


def test_mel_filterbank_structure():
    fb = O.mel_filterbank(SR, NFFT, 80, 0.0, 8000.0)
    assert np.count_nonzero(fb) == 625
    assert np.count_nonzero(fb, axis=0).max() <= 2
    assert np.all(fb[:, 0] == 0) and np.all(fb[:, 320] == 0)
    G = fb @ fb.T
    off = G - np.diag(np.diag(G)) - np.diag(np.diag(G, 1), 1) - np.diag(np.diag(G, -1), -1)
    assert np.max(np.abs(off)) == 0.0
    P = np.linalg.pinv(fb)
    assert np.max(np.abs(fb @ P - np.eye(80))) < 1e-10
    assert np.max(np.abs(P - fb.T @ np.linalg.inv(G))) < 1e-10


def test_amplitude_db_roundtrip_and_floor():
    S = np.abs(np.random.RandomState(0).randn(80, 50)) * 10.0
    S[3, 4] = 0.0
    db = O.amplitude_to_db(S)
    assert db.max() - db.min() <= 80.0 + 1e-12
    keep = db > db.max() - 80.0
    assert np.allclose(O.db_to_amplitude(db)[keep], S[keep], rtol=1e-12)


def test_magphase_zero_convention():
    D = np.array([[0.0 + 0.0j, 3.0 + 4.0j]])
    mag, ph = O.magphase(D)
    assert ph[0, 0] == 1.0 + 0.0j and abs(ph[0, 1] - (0.6 + 0.8j)) < 1e-15 and mag[0, 1] == 5.0


def test_pair_shapes_and_snr():
    n = 48000
    s = O.AudioSignal(np.round(O.synth_speech(n, SR, 5) * 32767).astype(np.int16), SR)
    nz = O.AudioSignal(np.round(O.synth_noise(17000, 5) * 32767).astype(np.int16), SR)  # shorter: exercises dp:125-128
    mixed, speech, noise, mixed_sig = O.preprocess_audio_pair_signals(s, nz, 200, 15, 25.0)
    assert mixed.shape == speech.shape == noise.shape == (15, 80, 20)
    assert mixed_sig.get_number_of_samples() == 48000
    # 0 dB SNR: speech and scaled noise have equal variance
    sp = O.AudioSignal(np.round(O.synth_speech(n, SR, 5) * 32767).astype(np.int16), SR)
    nn = O.fit_noise_to_speech(O.AudioSignal(np.round(O.synth_noise(17000, 5) * 32767).astype(np.int16), SR), sp)
    f = O.AudioMixer.snr_factor(sp, nn, 0)
    assert abs(np.var(nn.get_data() * f) / np.var(sp.get_data().astype(float)) - 1.0) < 1e-12


def test_slices_reassemble():
    a = O.AudioSignal(_sig(50000, 7), SR)
    sl = O.preprocess_audio_signal(a, 200, 15, 25.0)
    assert a.get_number_of_samples() == 48000  # truncated in place (dp:42)
    full, _ = O.signal_to_spectrogram(a, NFFT, HOP)
    assert full.shape == (80, 301)
    assert np.array_equal(np.concatenate(list(sl), axis=1), full[:, :300])


def test_reconstruct_roundtrip_quality():
    a = O.AudioSignal(_sig(48000, 8), SR)
    sl = O.preprocess_audio_signal(a, 200, 15, 25.0)
    rec = O.reconstruct_speech_signal(a, sl, 25.0)
    assert rec.get_number_of_samples() == 47840
    x = a.get_data()[:47840]
    err = rec.get_data() - x
    assert np.sqrt(np.mean(err ** 2)) / np.sqrt(np.mean(x ** 2)) < 0.5  # mel round trip is lossy but close


def test_against_transformers_librosa_compatible_front_end():
    """Third independent pin of the a5 row (dp:77-96): transformers.audio_utils re-implements librosa's mel filterbank,
    STFT framing (periodic Hann, centre + reflect padding) and amplitude_to_db (reference 1, amin 1e-5, top_db 80)."""
    au = pytest.importorskip("transformers.audio_utils")
    fb_t = au.mel_filter_bank(321, 80, 0.0, 8000.0, SR, norm="slaney", mel_scale="slaney")        # (321, 80), float64
    assert np.max(np.abs(fb_t.T - O.mel_filterbank(SR, 640, 80, 0.0, 8000.0))) < 1e-14
    x = (O.synth_speech(48000, SR, 3) + O.synth_noise(48000, 3)).astype(np.float64)
    win = au.window_function(640, "hann", periodic=True)
    mag = au.spectrogram(x, win, 640, 160, fft_length=640, power=1.0, center=True, pad_mode="reflect", dtype=np.float64)
    D = O.stft(x, 640, 160)
    assert mag.shape == (321, 301) and np.max(np.abs(mag - np.abs(D))) < 1e-5 * np.max(np.abs(D))   # their FFT runs in complex64
    logmel = au.spectrogram(x, win, 640, 160, fft_length=640, power=1.0, center=True, pad_mode="reflect", mel_filters=fb_t,
                            mel_floor=0.0, log_mel="dB", reference=1.0, min_value=1e-5, db_range=80.0, dtype=np.float64)
    ref, _ = O.signal_to_spectrogram(O.AudioSignal(x, SR), 640, 160)
    assert logmel.shape == ref.shape == (80, 301)
    assert np.max(np.abs(logmel - ref)) < 1e-5                                                      # dB
    rng = np.random.RandomState(0)
    a = np.abs(rng.randn(80, 50)) * 10.0 ** rng.uniform(-9, 1, (80, 50))                            # spans the amin clamp and the 80 dB floor
    assert np.max(np.abs(au.amplitude_to_db(a, 1.0, 1e-5, 80.0) - O.amplitude_to_db(a))) < 1e-12


# ---- fourth independent pin (VERDICT r1 missing #3): scipy.signal's STFT / ISTFT and window machinery ----
def test_stft_and_istft_match_scipy_signal():
    """scipy.signal.stft / istft are a separate code base from torch's: same frames once librosa's centring (reflect pad by
    n_fft // 2) is applied by hand, scipy's 1 / sum(window) "spectrum" scaling undone; istft agrees away from the edges, where
    scipy normalises by the same window sum-square."""
    from scipy import signal
    y = _sig(48000, 11)
    win = signal.get_window("hann", NFFT, fftbins=True)                   # periodic Hann (librosa.stft's default window)
    assert np.max(np.abs(win - O.hann_periodic(NFFT))) < 1e-15
    yp = np.pad(y, NFFT // 2, mode="reflect")
    f, t, Z = signal.stft(yp, fs=SR, window=win, nperseg=NFFT, noverlap=NFFT - HOP, nfft=NFFT, boundary=None, padded=False,
                          return_onesided=True)
    D = O.stft(y, NFFT, HOP)
    assert Z.shape == D.shape == (321, 301)
    assert np.max(np.abs(Z * win.sum() - D)) < 1e-10
    # ISTFT: scipy on the same coefficients, trimmed like librosa's center=True
    _, yr = signal.istft(Z, fs=SR, window=win, nperseg=NFFT, noverlap=NFFT - HOP, nfft=NFFT, input_onesided=True, boundary=None)
    yo = O.istft(D, HOP)
    yr = yr[NFFT // 2:NFFT // 2 + len(yo)]
    assert np.max(np.abs(yr[NFFT:-NFFT] - yo[NFFT:-NFFT])) < 1e-11
    assert signal.check_COLA(win, NFFT, NFFT - HOP) and signal.check_NOLA(win, NFFT, NFFT - HOP)
    # window sum-square of the interior: sum_t w^2[n - t hop] = 1.5 for the periodic Hann at hop = N / 4 (librosa.istft's divisor)
    assert abs(sum(win[HOP * q] ** 2 for q in range(4)) - 1.5) < 1e-12


def test_snr_factor_is_invariant_to_the_variance_convention():
    """mediaio's AudioMixer.snr_factor is recalled, not citable (SURVEY A.2).  Whatever variance estimator it uses -- population
    (ddof 0) or sample (ddof 1) -- cancels in var(s) / var(n) because dp:128 truncates the noise to the speech length; the only
    convention that matters is mean removal, which np.var, the documented call, performs.  This pins the stand-in's value to the
    call site rather than to a recollection of the library."""
    rng = np.random.RandomState(4)
    s = rng.randn(20000) * 1000 + 40.0
    n = rng.randn(20000) * 30 - 7.0
    f = O.AudioMixer.snr_factor(O.AudioSignal(s, SR), O.AudioSignal(n, SR), 5.0)
    for ddof in (0, 1):
        assert abs(f - np.sqrt(np.var(s, ddof=ddof) / np.var(n, ddof=ddof)) * 10 ** (-5.0 / 20)) < 1e-12 * f
    # the mixture then has the requested SNR by construction: 10 log10(var(s) / var(f n)) == snr_db
    assert abs(10 * np.log10(np.var(s) / np.var(f * n)) - 5.0) < 1e-9


def test_band_edge_keywords_of_the_spectrogram_functions():
    """fmin / fmax default to the reference's 0 / 8000 (bit-identical), and otherwise select O.mel_filterbank(sr, n_fft, 80, fmin,
    fmax) in both directions: amplitude_to_db(fb |stft|) forward, istft((pinv(fb) 10^(mel/20)) phase) back."""
    x = _sig(8000, 5)
    sig = O.AudioSignal(x, SR)
    mag, phase = O.signal_to_spectrogram(sig, NFFT, HOP)
    mag0, phase0 = O.signal_to_spectrogram(sig, NFFT, HOP, fmin=0.0, fmax=8000.0)
    assert np.array_equal(mag, mag0) and np.array_equal(phase, phase0)
    back = O.reconstruct_signal_from_spectrogram(mag, phase, SR, NFFT, HOP).get_data()
    assert np.array_equal(back, O.reconstruct_signal_from_spectrogram(mag, phase, SR, NFFT, HOP, fmin=0.0, fmax=8000.0).get_data())
    fb = O.mel_filterbank(SR, NFFT, 80, 300.0, 3500.0)
    D = O.stft(x, NFFT, HOP)
    mag2, phase2 = O.signal_to_spectrogram(sig, NFFT, HOP, fmin=300.0, fmax=3500.0)
    assert np.array_equal(phase2, phase)
    assert np.max(np.abs(mag2 - O.amplitude_to_db(fb @ np.abs(D)))) < 1e-12
    assert np.max(np.abs(mag2 - mag)) > 1.0
    want = O.istft((np.linalg.pinv(fb) @ O.db_to_amplitude(mag2)) * phase2, HOP)
    got = O.reconstruct_signal_from_spectrogram(mag2, phase2, SR, NFFT, HOP, fmin=300.0, fmax=3500.0).get_data()
    assert np.max(np.abs(got - want)) < 1e-12 * np.max(np.abs(want))
