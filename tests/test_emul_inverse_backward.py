"""CPU-side check of the inverse's backward kernel (csrc/avse_inverse_grad_stages.cuh, the loop of avse_inverse_grad_kernel)
against the float64 VJP of tests/inverse_vjp.py: tests/emul/avse_emul_grad.cpp runs the kernel's stage functions in the kernel's order, one warp
as a loop over lanes.  The gate is 1e-4 of the peak |oracle gradient| of the utterance."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests import inverse_vjp as V
from tests.cases import GOLDEN_CASES, SR, oracle_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio-visual-speech-enhancement_b200", "csrc")
TOL = 1e-4


@pytest.fixture(scope="module")
def emul_grad(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_grad") / "libavse_emul_grad.so")
    srcs = [os.path.join(ROOT, "tests", "emul", "avse_emul_grad.cpp"), os.path.join(CSRC, "avse_tables.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so] + srcs)
    lib = ctypes.CDLL(so)
    vp, i32, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    lib.emul_inverse_backward.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp, i32, f64, f64]
    lib.emul_inverse_backward.restype = i32
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _run(lib, mel, pcm, g, valid=None, layout=1, n_frames=None):
    """mel: SPEC [80, ld_t] (first n_frames columns used) or SLICES [n, 80, 20].  Returns grad_mel (NaN where not stored)."""
    mel = np.ascontiguousarray(mel, np.float32)
    pcm = np.ascontiguousarray(pcm, np.float32)
    g = np.ascontiguousarray(g, np.float32)
    out = np.full(mel.shape, np.nan, np.float32)
    if layout == 1:
        ld_t = mel.shape[1]
        n_frames = ld_t if n_frames is None else n_frames
        n_slices = 0
    else:
        ld_t, n_frames, n_slices = 0, 0, mel.shape[0]
    L = len(pcm)
    t = lib.emul_inverse_backward(_p(mel), layout, n_slices, n_frames, ld_t, _p(pcm), L, L if valid is None else valid, _p(g),
                                  _p(out), SR, 0.0, 8000.0)
    assert t >= 2
    return out


def _want(mel_spec, pcm, g, valid=None):
    """Oracle dL/d dB (80, T_mel) of the mixture-phase reconstruction, zeros beyond T_use."""
    x = np.asarray(pcm, np.float64).copy()
    if valid is not None:
        x[valid:] = 0.0
    _, phase = O.magphase(O.stft(x, 640, 160))
    T_use = min(mel_spec.shape[1], phase.shape[1])
    out = np.zeros(mel_spec.shape)
    out[:, :T_use] = V.reconstruct_signal_from_spectrogram_vjp(np.asarray(mel_spec[:, :T_use], np.float64), phase[:, :T_use], SR,
                                                               640, 160, np.asarray(g, np.float64))
    return out


def _check(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    peak = np.max(np.abs(want))
    assert peak > 0
    err = np.max(np.abs(got - want)) / peak
    assert err <= TOL, err


def _spec_case(seed, T_mel, L, scale=1.0):
    rng = np.random.RandomState(seed)
    pcm = (O.synth_speech(L, SR, seed) + O.synth_noise(L, seed)).astype(np.float32) * np.float32(scale)
    mel = (-40.0 + 12.0 * rng.randn(80, T_mel)).astype(np.float32)
    T_use = min(T_mel, 1 + L // 160)
    g = rng.randn(160 * (T_use - 1)).astype(np.float32)
    return mel, pcm, g


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
def test_golden_slices(emul_grad, case):
    o = oracle_pair(case)
    pcm = o["mixed_pcm"].astype(np.float32)
    slices = o["speech"].astype(np.float32)
    T_use = min(20 * len(slices), 1 + len(pcm) // 160)
    g = np.random.RandomState(11).randn(160 * (T_use - 1)).astype(np.float32)
    got = _run(emul_grad, slices, pcm, g, layout=0)
    spec = np.concatenate(list(slices), axis=1)
    want = _want(spec, pcm, g)
    _check(np.concatenate(list(got), axis=1), want)


@pytest.mark.parametrize("r", list(range(8)) + [31])
def test_frame_counts_mod_chunk(emul_grad, r):
    """T_use = 64 + r frames: every remainder of the 32-frame chunk the kernel's warps take, the first ones included."""
    T_mel = 64 + r
    mel, pcm, g = _spec_case(20 + r, T_mel, 160 * (T_mel + 3))
    _check(_run(emul_grad, mel, pcm, g), _want(mel, pcm, g))


@pytest.mark.parametrize("extra", [-5, 0, 7])
def test_mel_frames_against_mixture_frames(emul_grad, extra):
    """Mel frames <, = and > the mixture's T: frames past T_use get exact zeros."""
    L = 16000
    T = 1 + L // 160
    mel, pcm, g = _spec_case(31, T + extra, L)
    got = _run(emul_grad, mel, pcm, g)
    _check(got, _want(mel, pcm, g))
    assert np.all(got[:, T:] == 0.0)


@pytest.mark.parametrize("valid", [12000, 7777, 400])
def test_ragged_lengths(emul_grad, valid):
    mel, pcm, g = _spec_case(41, 101, 16000)
    _check(_run(emul_grad, mel, pcm, g, valid=valid), _want(mel, pcm, g, valid=valid))


def test_silent_mixture_frames(emul_grad):
    """Digital silence inside the mixture: phase 1 + 0j there, not the gradient channel's leakage."""
    mel, pcm, g = _spec_case(51, 101, 16000)
    pcm[3000:7000] = 0.0
    _check(_run(emul_grad, mel, pcm, g), _want(mel, pcm, g))


def test_zero_gradient_regions_are_exact_zeros(emul_grad):
    mel, pcm, g = _spec_case(61, 101, 16000)
    g[4000:9000] = 0.0
    got = _run(emul_grad, mel, pcm, g)
    _check(got, _want(mel, pcm, g))
    # frame t's window covers y[160 t - 320, 160 t + 320): frames 27 ... 54 see only zeros
    assert np.all(got[:, 27:55] == 0.0)
    assert np.all(got[:, 26] != 0.0) and np.all(got[:, 55] != 0.0)


@pytest.mark.parametrize("scale", [1e-9, 1e-6, 1e-3, 1.0, 1e3])
def test_gradient_scales(emul_grad, scale):
    """A loss gradient far under (mean over a large batch) or over the mixture: the per-frame power-of-two scaling keeps
    the packed FFT's leakage at the float32 level of each channel."""
    mel, pcm, g = _spec_case(71, 101, 16000)
    g = (g * scale).astype(np.float32)
    _check(_run(emul_grad, mel, pcm, g), _want(mel, pcm, g))


def test_gradient_step_60db(emul_grad):
    mel, pcm, g = _spec_case(81, 101, 16000)
    g[8000:] *= np.float32(1e-3)
    want = _want(mel, pcm, g)
    got = _run(emul_grad, mel, pcm, g)
    _check(got, want)
    quiet = want[:, 60:]            # the quiet part alone, against its own peak
    err = np.max(np.abs(got[:, 60:] - quiet)) / np.max(np.abs(quiet))
    assert err <= TOL, err


def test_power_of_two_scaling_is_exact(emul_grad):
    mel, pcm, g = _spec_case(91, 101, 16000)
    a = _run(emul_grad, mel, pcm, g)
    b = _run(emul_grad, mel, pcm, (g * np.float32(2.0 ** -20)).astype(np.float32))
    assert np.array_equal(a * np.float32(2.0 ** -20), b)


def test_spec_nan_beyond_n_frames(emul_grad):
    """SPEC [80, ld_t] holding n_frames < ld_t columns, NaN past them: the NaNs are neither read nor overwritten."""
    mel, pcm, g = _spec_case(95, 90, 16000)
    ld = np.full((80, 96), np.nan, np.float32)
    ld[:, :90] = mel
    got = _run(emul_grad, ld, pcm, g, n_frames=90)
    _check(got[:, :90], _want(mel, pcm, g))
    assert np.all(np.isnan(got[:, 90:]))
