"""GPU tests of the differentiable reconstruction (SpectralEngine.reconstruct_differentiable / reconstruct_spec_differentiable,
avse_inverse_backward) against the float64 VJP of tests/inverse_vjp.py, its invariants and its autograd plumbing.  The accuracy gate is 1e-4 of
the per-utterance peak |oracle gradient|."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests import inverse_vjp as V
from tests.cases import FRAME_RATES, GOLDEN_CASES, SR, FPS, oracle_pair

pytestmark = pytest.mark.gpu

TOL = 1e-4
LN10_20 = np.log(10.0) / 20.0


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _grad(eng, pcm, mel, g, lengths=None, spec=False):
    m = _dev(mel).requires_grad_(True)
    fn = eng.reconstruct_spec_differentiable if spec else eng.reconstruct_differentiable
    y = fn(_dev(pcm), m, lengths=lengths)
    y.backward(_dev(g))
    return m.grad.cpu().numpy(), y.detach().cpu().numpy()


def _want_spec(mel_spec, pcm, g, sr=SR, n_fft=640, hop=160, valid=None, fmin=0.0, fmax=8000.0):
    x = np.asarray(pcm, np.float64).copy()
    if valid is not None:
        x[valid:] = 0.0
    _, phase = O.magphase(O.stft(x, n_fft, hop))
    T_use = min(mel_spec.shape[1], phase.shape[1])
    out = np.zeros(mel_spec.shape)
    out[:, :T_use] = V.reconstruct_signal_from_spectrogram_vjp(np.asarray(mel_spec[:, :T_use], np.float64), phase[:, :T_use], sr,
                                                               n_fft, hop, np.asarray(g, np.float64), fmin=fmin, fmax=fmax)
    return out


def _check(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    peak = np.max(np.abs(want))
    assert peak > 0
    err = np.max(np.abs(got - want)) / peak
    assert err <= TOL, err


def _spec_case(seed, T_mel, L, scale=1.0, sr=SR):
    rng = np.random.RandomState(seed)
    pcm = ((O.synth_speech(L, sr, seed) + O.synth_noise(L, seed)) * scale).astype(np.float32)
    mel = (-40.0 + 12.0 * rng.randn(80, T_mel)).astype(np.float32)
    return pcm, mel, rng


def _slices_to_spec(s):
    return np.concatenate(list(s), axis=1)


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
@pytest.mark.parametrize("extra", [-1, 0, 1])
def test_golden_slices(eng, case, extra):
    """Golden mixtures (float and int16 scale), n slices <, = and > the mixture's frames."""
    o = oracle_pair(case)
    pcm = o["mixed_pcm"].astype(np.float32)
    sl = o["speech"].astype(np.float32)
    n = len(sl) + extra
    sl = np.concatenate([sl, sl])[:n]
    T_use = min(20 * n, 1 + len(pcm) // 160)
    g = np.random.RandomState(5).randn(1, 160 * (T_use - 1)).astype(np.float32)
    got, y = _grad(eng, pcm[None], sl[None], g)
    _check(_slices_to_spec(got[0]), _want_spec(_slices_to_spec(sl), pcm, g[0]))
    ref = eng.reconstruct(_dev(pcm[None]), _dev(sl[None])).cpu().numpy()
    assert np.array_equal(y, ref)                       # forward bit-identical to reconstruct


def test_lengths_and_spec_layout(eng):
    L = 16000
    pcm0, mel0, rng = _spec_case(3, 101, L)
    pcm1, mel1, _ = _spec_case(4, 101, L)
    pcm = np.stack([pcm0, pcm1])
    valid = np.array([L, 9001], np.int32)
    pcm[1, 9001:] = 7.0                                 # past `lengths`: never read
    mel = np.stack([mel0, mel1])
    g = rng.randn(2, 160 * 100).astype(np.float32)
    got, y = _grad(eng, pcm, mel, g, lengths=_dev(valid), spec=True)
    _check(got[0], _want_spec(mel0, pcm0, g[0]))
    _check(got[1], _want_spec(mel1, pcm[1], g[1], valid=9001))
    ref = eng.reconstruct_spec(_dev(pcm), _dev(mel), lengths=_dev(valid)).cpu().numpy()
    assert np.array_equal(y, ref)


@pytest.mark.parametrize("kind", ["dc", "hum", "tone", "silence"])
def test_offsets_hum_and_silence(eng, kind):
    """The mixtures the forward's DC / hum / level tests use: a DC offset, 50 Hz mains hum, a dominant tone, digital silence."""
    L = 24000
    pcm, mel, rng = _spec_case(9, 151, L)
    t = np.arange(L) / SR
    if kind == "dc":
        pcm = (pcm + 0.8).astype(np.float32)
    elif kind == "hum":
        pcm = (pcm + 2.0 * np.sin(2 * np.pi * 50 * t)).astype(np.float32)
    elif kind == "tone":
        pcm = (pcm + 30.0 * np.sin(2 * np.pi * 1000 * t)).astype(np.float32)
    else:
        pcm[5000:12000] = 0.0
    g = (1e-8 * rng.randn(1, 160 * 150)).astype(np.float32)
    got, _ = _grad(eng, pcm[None], mel[None], g, spec=True)
    _check(got[0], _want_spec(mel, pcm, g[0]))


@pytest.mark.parametrize("geo", FRAME_RATES, ids=[g["name"] for g in FRAME_RATES])
def test_generic_frame_rates(mod, geo):
    e = mod.SpectralEngine(geo["sr"], geo["fps"], 200, device="cuda:0", n_fft=geo["n_fft"])
    assert not e.specialised
    n_fft, hop = e.n_fft, e.hop
    L = 7 * n_fft + 5
    T = e.n_frames(L)
    pcm, mel, rng = _spec_case(12, T + 2, L, sr=geo["sr"])
    g = rng.randn(1, hop * (T - 1)).astype(np.float32)
    got, _ = _grad(e, pcm[None], mel[None], g, spec=True)
    _check(got[0], _want_spec(mel, pcm, g[0], sr=geo["sr"], n_fft=n_fft, hop=hop))
    assert np.all(got[0][:, T:] == 0.0)


def test_generic_refused_filterbank(mod):
    e = mod.SpectralEngine(SR, FPS, 200, fmin=80.0, fmax=3000.0, device="cuda:0")
    assert not e.specialised
    pcm, mel, rng = _spec_case(13, 60, 12000)
    sl = mel[:, :60].reshape(80, 3, 20).transpose(1, 0, 2).copy()
    T_use = 60
    g = rng.randn(1, 160 * (T_use - 1)).astype(np.float32)
    got, _ = _grad(e, pcm[None], sl[None], g)
    _check(_slices_to_spec(got[0]), _want_spec(mel[:, :60], pcm, g[0], fmin=80.0, fmax=3000.0))


def test_invariants(eng):
    pcm, mel, rng = _spec_case(21, 301, 48000)
    g = (1e-3 * rng.randn(1, 160 * 300)).astype(np.float32)
    g[0, 20000:26000] = 0.0
    got, y = _grad(eng, pcm[None], mel[None], g, spec=True)
    # Euler: y is linear in 10^(dB/20)
    lhs = np.sum(got.astype(np.float64))
    rhs = LN10_20 * np.dot(y[0].astype(np.float64), g[0].astype(np.float64))
    assert abs(lhs - rhs) <= 1e-5 * np.sum(np.abs(got.astype(np.float64))), (lhs, rhs)
    # power-of-two scaling of the gradient is exact
    for k in (-30, 7):
        got2, _ = _grad(eng, pcm[None], mel[None], (g * np.float32(2.0 ** k)).astype(np.float32), spec=True)
        assert np.array_equal(got2, got * np.float32(2.0 ** k))
    # frames whose window sees only zero gradient: frames 127 ... 160 (window [160 t - 320, 160 t + 320))
    assert np.all(got[0][:, 127:161] == 0.0)
    assert np.all(got[0][:, 126] != 0.0)


def test_reproducible_and_batch_independent(eng):
    B, L = 1000, 48000
    rng = np.random.RandomState(33)
    base = (O.synth_speech(L, SR, 1) + O.synth_noise(L, 1)).astype(np.float32)
    pcm = (base[None] * rng.uniform(0.1, 2.0, (B, 1))).astype(np.float32)
    for i in range(0, B, 7):
        pcm[i] = np.roll(pcm[i], i * 13)
    sl = (-40.0 + 12.0 * rng.randn(B, 15, 80, 20)).astype(np.float32)
    g = (1e-8 * rng.randn(B, 160 * 299)).astype(np.float32)      # T_use = min(300, 301) frames
    a, _ = _grad(eng, pcm, sl, g)
    b, _ = _grad(eng, pcm, sl, g)
    assert np.array_equal(a, b)
    for i in (0, 1, 499, 998, 999):
        one, _ = _grad(eng, pcm[i:i + 1], sl[i:i + 1], g[i:i + 1])
        assert np.array_equal(one[0], a[i])
    i = 17
    _check(_slices_to_spec(a[i]), _want_spec(_slices_to_spec(sl[i]), pcm[i], g[i]))


def _abi_args(mod, mel, pcm, layout, n_frames=0, ld_t=0, n_slices=0):
    a = mod.InverseArgs()
    a.mel_db, a.layout, a.n_slices, a.n_frames, a.ld_t = mel.data_ptr(), layout, n_slices, n_frames, ld_t
    a.mel_stride = mel.stride(0)
    a.mixed_pcm, a.pcm_stride, a.len_pcm = pcm.data_ptr(), pcm.stride(0), 0
    a.B, a.L = pcm.shape[0], pcm.shape[1]
    a.out_format = 0
    return a


def test_guard_bands_and_argument_errors(mod, eng):
    B, L = 3, 16000
    pcm = torch.from_numpy(np.stack([_spec_case(40 + i, 101, L)[0] for i in range(B)])).cuda()
    # SLICES rows with a guard band between utterances
    row = 5 * 80 * 20
    mel = torch.full((B, row + 64), float("nan"), device="cuda")
    mel[:, :row] = torch.randn(B, row, device="cuda") * 10 - 40
    gmel = torch.full_like(mel, float("nan"))
    g = torch.randn(B, 160 * 99, device="cuda")
    a = _abi_args(mod, mel, pcm, 0, n_slices=5)
    stream = torch.cuda.current_stream().cuda_stream
    assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a), g.data_ptr(), g.stride(0), gmel.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(gmel[:, :row]).all() and torch.isnan(gmel[:, row:]).all()
    # SPEC columns [n_frames, ld_t) untouched
    spec = torch.full((B, 80, 110), float("nan"), device="cuda")
    spec[:, :, :101] = torch.randn(B, 80, 101, device="cuda") * 10 - 40
    gspec = torch.full_like(spec, float("nan"))
    a = _abi_args(mod, spec, pcm, 1, n_frames=101, ld_t=110)
    a.mel_stride = 80 * 110
    g = torch.randn(B, 160 * 100, device="cuda")                 # T_use = 101 frames
    assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a), g.data_ptr(), g.stride(0), gspec.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(gspec[:, :, :101]).all() and torch.isnan(gspec[:, :, 101:]).all()
    # explicit phase or int16 output: AVSE_E_ARG
    ph = torch.zeros(B, 101, 321, 2, device="cuda")
    a.phase, a.phase_stride, a.phase_frames = ph.data_ptr(), 101 * 321, 101
    assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a), g.data_ptr(), g.stride(0), gspec.data_ptr(), stream) == -1
    a.phase, a.phase_stride, a.phase_frames = 0, 0, 0
    a.out_format = 1
    assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a), g.data_ptr(), g.stride(0), gspec.data_ptr(), stream) == -1


def test_autograd_plumbing(eng):
    pcm, mel, rng = _spec_case(50, 5 * 20, 16000)
    sl = mel.reshape(80, 5, 20).transpose(1, 0, 2).copy()
    # loss = y.sum(): a stride-0 expanded gradient
    m = _dev(sl[None]).requires_grad_(True)
    eng.reconstruct_differentiable(_dev(pcm[None]), m).sum().backward()
    want = _want_spec(_slices_to_spec(sl), pcm, np.ones(160 * 99))
    _check(_slices_to_spec(m.grad[0].cpu().numpy()), want)
    # a float64 leaf gets a float64 gradient
    m64 = _dev(sl[None].astype(np.float64)).requires_grad_(True)
    eng.reconstruct_differentiable(_dev(pcm[None]), m64).sum().backward()
    assert m64.grad.dtype == torch.float64
    assert torch.equal(m64.grad.float(), m.grad)
    # the mixture is data
    p = _dev(pcm[None]).requires_grad_(True)
    with pytest.raises(ValueError):
        eng.reconstruct_differentiable(p, _dev(sl[None]).requires_grad_(True))


def test_training_loop_lowers_waveform_loss(eng):
    """A few Adam steps on dB slices toward a target waveform (the reconstruction of other slices) lower an L1 loss."""
    o = oracle_pair(GOLDEN_CASES[0])
    pcm = _dev(o["mixed_pcm"].astype(np.float32)[None])
    target = eng.reconstruct(pcm, _dev(o["speech"].astype(np.float32)[None]))
    start = _dev((o["mixed"].astype(np.float32))[None]).requires_grad_(True)
    opt = torch.optim.Adam([start], lr=0.5)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = (eng.reconstruct_differentiable(pcm, start) - target).abs().mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < 0.9 * losses[0], losses
