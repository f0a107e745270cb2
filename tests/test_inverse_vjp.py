"""The float64 vector-Jacobian products of the mixture-phase reconstruction (tests/inverse_vjp.py) against torch.autograd
through an independent float64 restatement of the forward (pinv matmul, irfft, window, overlap-add by index_add, window
sum-square, centre trim), and Euler's identity sum(dL/d dB) = ln(10)/20 <y, g> that holds because y is linear in 10^(dB/20)."""
import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests import inverse_vjp as V
from tests.cases import FRAME_RATES, GOLDEN_CASES, SR, FPS, frame_rate_fps, oracle_pair

LN10_20 = np.log(10.0) / 20.0


def _torch_recon(dB, phase, sr, n_fft, hop):
    """dp:99-116 in float64 torch, differentiable in dB (80, T); phase (bins, T) complex constant."""
    bins, T = phase.shape
    n_inv = 2 * (bins - 1)
    fb = torch.from_numpy(np.linalg.pinv(O.mel_filterbank(sr, n_fft, n_mels=dB.shape[0])))
    lin = fb @ torch.pow(10.0, dB / 20.0)
    X = lin * torch.from_numpy(phase)
    win = torch.from_numpy(O.hann_periodic(n_inv))
    frames = torch.fft.irfft(X.T, n=n_inv, dim=1) * win[None, :]
    idx = (torch.arange(n_inv)[None, :] + hop * torch.arange(T)[:, None]).reshape(-1)
    y = torch.zeros(n_inv + hop * (T - 1), dtype=torch.float64).index_add(0, idx, frames.reshape(-1))
    wss = torch.from_numpy(O.window_sumsquare(T, n_inv, hop))
    nz = wss > np.finfo(np.float32).tiny
    y = torch.where(nz, y / torch.where(nz, wss, torch.ones_like(wss)), y)
    return y[n_inv // 2:n_inv // 2 + hop * (T - 1)]


def _autograd(dB, phase, sr, n_fft, hop, g):
    x = torch.from_numpy(np.array(dB, np.float64)).requires_grad_(True)
    y = _torch_recon(x, phase, sr, n_fft, hop)
    y.backward(torch.from_numpy(g))
    return x.grad.numpy(), y.detach().numpy()


def _check(got, want):
    peak = np.max(np.abs(want))
    assert peak > 0 and np.max(np.abs(got - want)) <= 1e-10 * peak, np.max(np.abs(got - want)) / peak


def _mixture(pcm, valid=None):
    x = np.asarray(pcm, np.float64).copy()
    if valid is not None:
        x[valid:] = 0.0
    return x


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
@pytest.mark.parametrize("extra_slices", [-1, 0, 1])
def test_slices_vjp_matches_autograd(case, extra_slices):
    """Mel frames <, = and > the mixture's T: the slices VJP equals autograd on the frames used and is 0 beyond."""
    o = oracle_pair(case)
    pcm = o["mixed_pcm"]
    T = 1 + len(pcm) // 160
    n = max(1, T // 20 + extra_slices)
    rng = np.random.RandomState(7)
    slices = np.concatenate([o["speech"]] * 2)[:n] if n > len(o["speech"]) else o["speech"][:n]
    T_use = min(20 * n, T)
    g = rng.randn(160 * (T_use - 1))
    got = V.reconstruct_speech_signal_vjp(O.AudioSignal(pcm, SR), slices, FPS, g)
    _, phase = O.magphase(O.stft(pcm, 640, 160))
    spec = np.concatenate(list(slices), axis=1)
    want, _ = _autograd(spec[:, :T_use], phase[:, :T_use], SR, 640, 160, g)
    got_spec = np.concatenate(list(got), axis=1)
    _check(got_spec[:, :T_use], want)
    assert np.all(got_spec[:, T_use:] == 0.0)
    assert got.shape == slices.shape


@pytest.mark.parametrize("valid", [16000, 9001, 4000])
def test_silence_and_zero_padding(valid):
    """Digital silence (zero-padded tail, silent frames with phase 1 + 0j) in the mixture."""
    pcm = _mixture(O.synth_speech(16000, SR, 3), valid)
    pcm[2000:5000] = 0.0
    T = 1 + len(pcm) // 160
    _, phase = O.magphase(O.stft(pcm, 640, 160))
    assert np.any(np.abs(O.stft(pcm, 640, 160)) == 0)
    rng = np.random.RandomState(1)
    dB = -30.0 + 10.0 * rng.randn(80, T)
    g = rng.randn(160 * (T - 1))
    got = V.reconstruct_signal_from_spectrogram_vjp(dB, phase, SR, 640, 160, g)
    want, y = _autograd(dB, phase, SR, 640, 160, g)
    _check(got, want)
    np.testing.assert_allclose(np.sum(got), LN10_20 * np.dot(y, g), rtol=1e-12)


@pytest.mark.parametrize("geo", FRAME_RATES, ids=[g["name"] for g in FRAME_RATES])
def test_frame_rate_geometries(geo):
    """Every generic geometry, odd n_fft included (the inverse then runs at n_inv = n_fft - 1)."""
    sr = geo["sr"]
    n_fft, hop = geo["geo"][0], geo["geo"][1]
    L = 6 * n_fft + 17
    pcm = O.synth_speech(L, sr, 5)
    D = O.stft(pcm, n_fft, hop)
    _, phase = O.magphase(D)
    T = D.shape[1]
    rng = np.random.RandomState(2)
    dB = -20.0 + 8.0 * rng.randn(80, T)
    n_inv = 2 * (phase.shape[0] - 1)
    assert n_inv == geo["geo"][5]
    g = rng.randn(hop * (T - 1))
    got = V.reconstruct_signal_from_spectrogram_vjp(dB, phase, sr, n_fft, hop, g)
    want, y = _autograd(dB, phase, sr, n_fft, hop, g)
    _check(got, want)
    np.testing.assert_allclose(np.sum(got), LN10_20 * np.dot(y, g), rtol=1e-10)
    assert frame_rate_fps(geo) > 0


def test_euler_identity_on_golden_slices():
    o = oracle_pair(GOLDEN_CASES[0])
    rng = np.random.RandomState(3)
    y = o["recon"]
    g = rng.randn(len(y))
    got = V.reconstruct_speech_signal_vjp(O.AudioSignal(o["mixed_pcm"], SR), o["speech"], FPS, g)
    np.testing.assert_allclose(np.sum(got), LN10_20 * np.dot(y, g), rtol=1e-12)
