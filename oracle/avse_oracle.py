"""CPU oracle for the spectral front/back end of audio-visual-speech-enhancement.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` may be imported by the
product package (``audio-visual-speech-enhancement_b200/``).  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs use it, and there only as the checker / the timed CPU baseline.

PARITY UNPINNED: the reference's arithmetic lives in two third-party packages
that are neither vendored under /root/reference nor installable here (no
network): ``librosa`` (version unpinned, API implies >= 0.5) and ``mediaio``
(github.com/avivga/mediaio, unpinned).  The reference ships no tests, golden
vectors or fixtures for this path.  This file therefore *restates* the published
algorithms of those calls in float64 numpy, function for function with the
reference call sites (cited as ``dp:LINE`` = /root/reference/data_processor.py),
and is pinned instead by independent cross-checks in tests/test_oracle.py
(torch.stft / torch.istft / torchaudio Slaney filterbank / transformers.audio_utils'
librosa-compatible filterbank, amplitude_to_db and log-mel pipeline / algebraic identities).

Everything is float64 unless stated otherwise.
"""
from __future__ import annotations

import numpy as np

# ----------------------------------------------------------------------------
# mediaio stand-ins (call sites: dp:116, dp:122-133; SURVEY Appendix A.2)
# ----------------------------------------------------------------------------


class AudioSignal(object):
    """Minimal restatement of mediaio.audio_io.AudioSignal (only what dp: uses)."""

    def __init__(self, data, sample_rate):
        self._data = np.asarray(data).copy()
        self._sample_rate = int(sample_rate)

    @staticmethod
    def from_wav_file(path):  # dp:122-123
        from scipy.io import wavfile
        sr, data = wavfile.read(path)
        return AudioSignal(data, sr)

    def save_to_wav_file(self, path, sample_type=np.int16):  # se:176-177
        from scipy.io import wavfile
        info = np.iinfo(sample_type)
        data = np.clip(self._data, info.min, info.max).astype(sample_type)
        wavfile.write(path, self._sample_rate, data)

    def get_data(self, channel_index=None):  # dp:78
        if channel_index is None or self._data.ndim == 1:
            return self._data
        return self._data[:, channel_index]

    def get_number_of_samples(self):  # dp:39, dp:125
        return self._data.shape[0]

    def get_sample_rate(self):  # dp:36
        return self._sample_rate

    def pad_with_zeros(self, new_length):  # dp:40
        if self.get_number_of_samples() > new_length:
            raise Exception("cannot pad for shorter signal length")
        pad = [(0, new_length - self.get_number_of_samples())] + [(0, 0)] * (self._data.ndim - 1)
        self._data = np.pad(self._data, pad, mode="constant")

    def truncate(self, new_length):  # dp:42, dp:128
        if self.get_number_of_samples() < new_length:
            raise Exception("cannot truncate for longer signal length")
        self._data = self._data[:new_length]

    def amplify_by_factor(self, factor):  # dp:131
        self._data = self._data.astype(np.float64) * factor

    @staticmethod
    def concat(signals):  # dp:126
        return AudioSignal(np.concatenate([s.get_data() for s in signals]), signals[0].get_sample_rate())


class AudioMixer(object):
    @staticmethod
    def snr_factor(signal, noise, snr_db):  # dp:130
        s = signal.get_data().astype(np.float64)
        n = noise.get_data().astype(np.float64)
        if s.size != n.size:
            raise Exception("signal and noise must have the same length")
        return float(np.sqrt(np.var(s) / np.var(n)) * (10.0 ** (-snr_db / 20.0)))

    @staticmethod
    def mix(audio_signals, mixing_weights=None):  # dp:133
        if mixing_weights is None:
            mixing_weights = [1.0 / len(audio_signals)] * len(audio_signals)
        mixed = np.zeros(audio_signals[0].get_data().shape, dtype=np.float64)
        for sig, w in zip(audio_signals, mixing_weights):
            mixed += float(w) * sig.get_data().astype(np.float64)
        return AudioSignal(mixed, audio_signals[0].get_sample_rate())


# ----------------------------------------------------------------------------
# librosa restatements (SURVEY Appendix A.1)
# ----------------------------------------------------------------------------


def hann_periodic(n):
    """scipy.signal.get_window('hann', n, fftbins=True)."""
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n) / n)


def stft(y, n_fft, hop_length):
    """librosa.core.stft(y, n_fft, hop_length) with defaults (dp:79):
    win_length=n_fft, periodic Hann, center=True, pad_mode='reflect'.
    Returns complex128 (1 + n_fft//2, T)."""
    y = np.asarray(y, dtype=np.float64)
    win = hann_periodic(n_fft)
    yp = np.pad(y, n_fft // 2, mode="reflect")
    n_frames = 1 + (len(yp) - n_fft) // hop_length
    idx = np.arange(n_fft)[None, :] + hop_length * np.arange(n_frames)[:, None]
    frames = yp[idx] * win[None, :]
    return np.fft.rfft(frames, n=n_fft, axis=1).T.copy()


def magphase(D):
    """librosa.core.magphase (dp:80): mag = |D|, phase = exp(1j*angle(D)) (1+0j where D == 0)."""
    mag = np.abs(D)
    zeros = mag == 0
    safe = mag + zeros
    phase = D / safe + zeros
    return mag, phase


def hz_to_mel(f):
    f = np.asarray(f, dtype=np.float64)
    f_sp = 200.0 / 3
    mels = f / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, 1e-300) / min_log_hz) / logstep, mels)


def mel_to_hz(m):
    m = np.asarray(m, dtype=np.float64)
    f_sp = 200.0 / 3
    freqs = f_sp * m
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), freqs)


def mel_filterbank(sr, n_fft, n_mels=80, fmin=0.0, fmax=8000.0):
    """librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax) (dp:83-89, dp:104-110):
    Slaney scale, triangular, Slaney area norm.  Shape (n_mels, 1 + n_fft//2)."""
    n_bins = 1 + n_fft // 2
    fftfreqs = np.linspace(0.0, float(sr) / 2, n_bins)
    mel_f = mel_to_hz(np.linspace(hz_to_mel(fmin), hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    weights = np.zeros((n_mels, n_bins))
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, None]
    return weights


def amplitude_to_db(S, ref=1.0, amin=1e-5, top_db=80.0):
    """librosa.amplitude_to_db defaults (dp:94): power_to_db(S**2, ref**2, amin**2, top_db)."""
    power = np.square(np.abs(S))
    log_spec = 10.0 * np.log10(np.maximum(amin ** 2, power))
    log_spec -= 10.0 * np.log10(np.maximum(amin ** 2, ref ** 2))
    if top_db is not None:
        log_spec = np.maximum(log_spec, log_spec.max() - top_db)
    return log_spec


def db_to_amplitude(S_db, ref=1.0):
    """librosa.db_to_amplitude (dp:101): db_to_power(S_db, ref**2) ** 0.5."""
    return (ref ** 2 * np.power(10.0, 0.1 * np.asarray(S_db, dtype=np.float64))) ** 0.5


def window_sumsquare(n_frames, n_fft, hop_length):
    n = n_fft + hop_length * (n_frames - 1)
    x = np.zeros(n)
    w2 = hann_periodic(n_fft) ** 2
    for i in range(n_frames):
        x[i * hop_length:i * hop_length + n_fft] += w2
    return x


def istft(M, hop_length):
    """librosa.istft(M, hop_length) defaults (dp:114): n_fft = 2*(rows-1), periodic Hann,
    overlap-add, divide by window sum-square where > tiny(float32), center trim."""
    n_fft = 2 * (M.shape[0] - 1)
    n_frames = M.shape[1]
    win = hann_periodic(n_fft)
    y = np.zeros(n_fft + hop_length * (n_frames - 1))
    frames = np.fft.irfft(M.T, n=n_fft, axis=1) * win[None, :]
    for i in range(n_frames):
        y[i * hop_length:i * hop_length + n_fft] += frames[i]
    wss = window_sumsquare(n_frames, n_fft, hop_length)
    nz = wss > np.finfo(np.float32).tiny
    y[nz] /= wss[nz]
    return y[n_fft // 2:-(n_fft // 2)]


# ----------------------------------------------------------------------------
# data_processor.py restatement (dp:35-139)
# ----------------------------------------------------------------------------


def signal_to_spectrogram(audio_signal, n_fft, hop_length, mel=True, db=True, fmin=0.0, fmax=8000.0):  # dp:77-96
    """fmin / fmax: the filterbank's band edges (the reference hard-codes 0 / 8000)."""
    signal = audio_signal.get_data(channel_index=0)
    D = stft(signal, n_fft=n_fft, hop_length=hop_length)
    magnitude, phase = magphase(D)
    if mel:
        fb = mel_filterbank(audio_signal.get_sample_rate(), n_fft, n_mels=80, fmin=fmin, fmax=fmax)
        magnitude = np.dot(fb, magnitude)
    if db:
        magnitude = amplitude_to_db(magnitude)
    return magnitude, phase


def reconstruct_signal_from_spectrogram(magnitude, phase, sample_rate, n_fft, hop_length, mel=True, db=True, fmin=0.0,
                                        fmax=8000.0):  # dp:99-116
    if db:
        magnitude = db_to_amplitude(magnitude)
    if mel:
        fb = mel_filterbank(sample_rate, n_fft, n_mels=80, fmin=fmin, fmax=fmax)
        magnitude = np.dot(np.linalg.pinv(fb), magnitude)
    signal = istft(magnitude * phase, hop_length=hop_length)
    return AudioSignal(signal, sample_rate)


def preprocess_audio_signal(audio_signal, slice_duration_ms, n_video_slices, video_frame_rate):  # dp:35-57
    samples_per_slice = int((float(slice_duration_ms) / 1000) * audio_signal.get_sample_rate())
    signal_length = samples_per_slice * n_video_slices
    if audio_signal.get_number_of_samples() < signal_length:
        audio_signal.pad_with_zeros(signal_length)
    else:
        audio_signal.truncate(signal_length)
    n_fft = int(float(audio_signal.get_sample_rate()) / video_frame_rate)
    hop_length = int(n_fft / 4)
    mel_spectrogram, phase = signal_to_spectrogram(audio_signal, n_fft, hop_length, mel=True, db=True)
    spss = int(samples_per_slice / hop_length)
    n_slices = int(mel_spectrogram.shape[1] / spss)
    slices = [mel_spectrogram[:, (i * spss):((i + 1) * spss)] for i in range(n_slices)]
    return np.stack(slices)


def reconstruct_speech_signal(mixed_signal, speech_spectrograms, video_frame_rate):  # dp:60-74
    n_fft = int(float(mixed_signal.get_sample_rate()) / video_frame_rate)
    hop_length = int(n_fft / 4)
    _, original_phase = signal_to_spectrogram(mixed_signal, n_fft, hop_length, mel=True, db=True)
    speech_spectrogram = np.concatenate(list(speech_spectrograms), axis=1)
    spectrogram_length = min(speech_spectrogram.shape[1], original_phase.shape[1])
    speech_spectrogram = speech_spectrogram[:, :spectrogram_length]
    original_phase = original_phase[:, :spectrogram_length]
    return reconstruct_signal_from_spectrogram(
        speech_spectrogram, original_phase, mixed_signal.get_sample_rate(), n_fft, hop_length, mel=True, db=True
    )


def fit_noise_to_speech(noise_signal, speech_signal):  # dp:125-128
    while noise_signal.get_number_of_samples() < speech_signal.get_number_of_samples():
        noise_signal = AudioSignal.concat([noise_signal, noise_signal])
    noise_signal.truncate(speech_signal.get_number_of_samples())
    return noise_signal


def preprocess_audio_pair_signals(speech_signal, noise_signal, slice_duration_ms, n_video_slices,
                                  video_frame_rate, snr_db=0):
    """dp:119-139 with the two WAV reads (dp:122-123) replaced by in-memory AudioSignal objects.
    snr_db generalises the hard-coded 0 of dp:130."""
    noise_signal = fit_noise_to_speech(noise_signal, speech_signal)
    factor = AudioMixer.snr_factor(speech_signal, noise_signal, snr_db=snr_db)
    noise_signal.amplify_by_factor(factor)
    mixed_signal = AudioMixer.mix([speech_signal, noise_signal], mixing_weights=[1, 1])
    mixed_spectrograms = preprocess_audio_signal(mixed_signal, slice_duration_ms, n_video_slices, video_frame_rate)
    speech_spectrograms = preprocess_audio_signal(speech_signal, slice_duration_ms, n_video_slices, video_frame_rate)
    noise_spectrograms = preprocess_audio_signal(noise_signal, slice_duration_ms, n_video_slices, video_frame_rate)
    return mixed_spectrograms, speech_spectrograms, noise_spectrograms, mixed_signal


def preprocess_audio_pair(speech_file_path, noise_file_path, slice_duration_ms, n_video_slices, video_frame_rate):  # dp:119-139
    speech_signal = AudioSignal.from_wav_file(speech_file_path)
    noise_signal = AudioSignal.from_wav_file(noise_file_path)
    return preprocess_audio_pair_signals(speech_signal, noise_signal, slice_duration_ms, n_video_slices, video_frame_rate)


def make_sample_set(mixed_list, speech_list, video_list, permutation):
    """se:241-262 (next row f1): concatenate slices over samples and apply ONE shared permutation.
    The reference draws the permutation with np.random.permutation; here it is an argument."""
    mixed = np.concatenate(mixed_list, axis=0)
    speech = np.concatenate(speech_list, axis=0)
    video = np.concatenate(video_list, axis=0) if video_list is not None else None
    perm = np.asarray(permutation)
    return (video[perm] if video is not None else None), mixed[perm], speech[perm]


# ----------------------------------------------------------------------------
# deterministic synthetic inputs shared by tests, smoke() and bench.py
# ----------------------------------------------------------------------------


def synth_speech(n_samples, sr=16000, seed=0, scale=0.3):
    """Voiced-like harmonic series with a slow envelope (SURVEY 8(d)); float64, |x| <~ scale."""
    rng = np.random.RandomState(1234 + seed)
    t = np.arange(n_samples) / float(sr)
    f0 = 120.0 + 30.0 * (2.0 * rng.rand() - 1.0)
    x = np.zeros(n_samples)
    for k in range(1, 30):
        x += np.sin(2.0 * np.pi * k * f0 * t + 2.0 * np.pi * rng.rand()) / k
    env = np.sin(np.pi * 1.5 * t + rng.rand()) ** 2
    x = x * env
    x += 1e-3 * rng.randn(n_samples)
    return scale * x / np.max(np.abs(x))


def synth_noise(n_samples, seed=0, sigma=0.05):
    rng = np.random.RandomState(9000000 + seed)
    return sigma * rng.randn(n_samples)
