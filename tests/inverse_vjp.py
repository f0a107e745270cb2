"""Float64 vector-Jacobian products of the reference's mixture-phase reconstruction (dp:60-74, dp:99-116) with respect to
its dB input, built on the oracle's restatements (oracle/avse_oracle.py).  TEST INFRASTRUCTURE: the checker of
avse_inverse_backward, itself pinned against torch.autograd by tests/test_inverse_vjp.py."""
import numpy as np

from oracle import avse_oracle as O


def reconstruct_signal_from_spectrogram_vjp(dB, phase, sr, n_fft, hop, grad, fmin=0.0, fmax=8000.0):
    """Vector-Jacobian product of reconstruct_signal_from_spectrogram(mel=True, db=True) (dp:99-116) with respect to its dB
    input: dB (80, T) and phase (1 + n_fft//2, T) as the forward takes them, grad = dL/dy of the returned signal
    (length hop (T - 1)).  Returns dL/d dB, (80, T).  The phase is a constant here (gradients with respect to it, or to
    the mixture it came from, are not part of this product).

    The steps: the overlap-add's adjoint frames the (window-sum-square normalised, untrimmed) gradient, the irfft's adjoint
    is a forward rfft with the Hermitian weights c_k / n (c = 2 inside, 1 at DC and Nyquist, where the C2R transform only
    reads the real part), the phase multiply's adjoint is Re(conj(phase) .), pinv(F)'s is its transpose and
    db_to_amplitude's is ln(10) / 20 * a."""
    dB = np.asarray(dB, dtype=np.float64)
    phase = np.asarray(phase, dtype=np.complex128)
    T = dB.shape[1]
    bins = phase.shape[0]
    n_inv = 2 * (bins - 1)
    g = np.asarray(grad, dtype=np.float64)
    assert phase.shape[1] == T and g.shape == (hop * (T - 1),)
    e = np.zeros(n_inv + hop * (T - 1))
    e[n_inv // 2:n_inv // 2 + len(g)] = g
    wss = O.window_sumsquare(T, n_inv, hop)
    nz = wss > np.finfo(np.float32).tiny
    e[nz] /= wss[nz]
    idx = np.arange(n_inv)[None, :] + hop * np.arange(T)[:, None]
    H = np.fft.rfft(e[idx] * O.hann_periodic(n_inv)[None, :], n=n_inv, axis=1).T      # (bins, T)
    c = np.full(bins, 2.0)
    c[0] = 1.0
    c[n_inv // 2] = 1.0
    d = (c / n_inv)[:, None] * (phase.real * H.real + phase.imag * H.imag)
    d[0] = phase.real[0] * H.real[0] / n_inv
    d[n_inv // 2] = phase.real[n_inv // 2] * H.real[n_inv // 2] / n_inv
    fb = O.mel_filterbank(sr, n_fft, n_mels=dB.shape[0], fmin=fmin, fmax=fmax)
    q = np.linalg.pinv(fb).T @ d
    return (np.log(10.0) / 20.0) * O.db_to_amplitude(dB) * q


def reconstruct_speech_signal_vjp(mixed_signal, speech_spectrograms, video_frame_rate, grad):
    """Vector-Jacobian product of reconstruct_speech_signal (dp:60-74) with respect to the dB slices (n, 80, spss), the
    mixture being data.  grad: dL/dy of the returned signal.  Frames beyond min(n spss, T) get exactly 0."""
    n_fft = int(float(mixed_signal.get_sample_rate()) / video_frame_rate)
    hop_length = int(n_fft / 4)
    _, original_phase = O.signal_to_spectrogram(mixed_signal, n_fft, hop_length, mel=True, db=True)
    slices = np.asarray(speech_spectrograms, dtype=np.float64)
    n, n_mels, spss = slices.shape
    spec = np.concatenate(list(slices), axis=1)
    T_use = min(spec.shape[1], original_phase.shape[1])
    g_spec = np.zeros_like(spec)
    g_spec[:, :T_use] = reconstruct_signal_from_spectrogram_vjp(spec[:, :T_use], original_phase[:, :T_use],
                                                                mixed_signal.get_sample_rate(), n_fft, hop_length, grad)
    return g_spec.reshape(n_mels, n, spss).transpose(1, 0, 2).copy()
