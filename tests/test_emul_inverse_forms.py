"""CPU-side check of the two less-travelled call forms of the I8 inverse kernel (csrc/avse_inv8_stages.cuh, the loop of
avse_inverse8_kernel) against the float64 oracle:

  * explicit phase (the EXT instantiation: reconstruct_with_phase, the mirror's reconstruct_signal_from_spectrogram, dp:99-116):
    no pass 1 / pass 2, the post stage multiplies F^T c by the caller's phase of frames (t, t+1) of each packed FFT;
  * SPEC-layout mel [80][ld_t] (reconstruct_spec): only the load address of the coefficient stage differs from SLICES.

tests/emul/avse_emul_inv.cpp::emul_inverse8_ex runs the kernel's stage functions in the kernel's order, one warp as a loop over
lanes, with the warp's shared memory persistent across groups and chunks (a chunk that starts inside an utterance begins with a
warm-up group, like a warp range of the kernel)."""
import ctypes
import os

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests.cases import GOLDEN_CASES, SR
from tests.test_emul_forward import emul, _p, GOLD, TOL_PCM  # noqa: F401  (session fixture that builds the emulation library)


def _run(emul, mel, pcm=None, valid=None, phase=None, chunks=1, layout=1, n_frames=None, n_slices=0):
    """mel: SPEC [80, ld_t] (layout 1, first n_frames columns used) or SLICES [n, 80, 20] (layout 0).  pcm: mixture (its own phase)
    or phase: explicit [phase_frames, 321] complex64.  Returns the float32 PCM; every sample must be stored by the kernel's code."""
    fn = emul.emul_inverse8_ex
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                   ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double]
    mel = np.ascontiguousarray(mel, np.float32)
    if layout == 1:
        ld_t = mel.shape[1]
        n_frames = ld_t if n_frames is None else n_frames
        t_mel = n_frames
    else:
        ld_t, n_frames, n_slices = 0, 0, mel.shape[0]
        t_mel = 20 * n_slices
    if phase is not None:
        phase = np.ascontiguousarray(phase, np.complex64)
        T = phase.shape[0]
        L = valid = 0
    else:
        pcm = np.ascontiguousarray(pcm, np.float32)
        L = len(pcm)
        valid = L if valid is None else valid
        T = 1 + L // 160
    T_use = min(t_mel, T)
    out = np.full(160 * (T_use - 1), np.nan, np.float32)
    n = fn(_p(mel), layout, n_slices, n_frames, ld_t, _p(pcm), L, valid, _p(phase), 0 if phase is None else phase.shape[0], _p(out), len(out),
           chunks, SR, 0.0, 8000.0)
    assert n == len(out)
    return out


def _want_ext(mel_spec, phase):
    """dp:99-116 on the frames both arrays have (the oracle itself needs equal frame counts)."""
    T_use = min(mel_spec.shape[1], phase.shape[0])
    return O.reconstruct_signal_from_spectrogram(mel_spec[:, :T_use].astype(np.float64), phase[:T_use].T.astype(np.complex128),
                                                 SR, 640, 160).get_data()


def _want_mixture(mel_spec, pcm):
    """dp:60-74 restated with an (80, T) mel: the mixture's own phase, both cut to the shorter."""
    _, phase = O.magphase(O.stft(np.asarray(pcm, np.float64), 640, 160))
    return _want_ext(mel_spec, phase.T)


def _check(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    err = np.max(np.abs(got - want)) / np.max(np.abs(want))
    assert err <= TOL_PCM, err


def _random_phase(rng, T, zero_frac=0.0):
    ph = np.exp(2j * np.pi * rng.rand(T, 321)).astype(np.complex64)
    if zero_frac:
        ph[rng.rand(T, 321) < zero_frac] = 0.0
    return ph


def _slices_to_spec(mel):
    return np.ascontiguousarray(np.concatenate(list(mel), axis=1))


@pytest.mark.parametrize("chunks", [1, 2, 3])
@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
def test_explicit_mixture_phase_of_the_golden_cases(emul, case, chunks):
    """The reference's own route (dp:60-74 calls dp:99-116): the phase of O.magphase(O.stft(mixture)) handed over explicitly."""
    gold = np.load(os.path.join(GOLD, case["name"] + ".npz"))
    spec = _slices_to_spec(gold["speech"])
    _, phase = O.magphase(O.stft(gold["mixed_pcm"].astype(np.float64), 640, 160))
    phase = np.ascontiguousarray(phase.T, np.complex64)
    got = _run(emul, spec, phase=phase, chunks=chunks)
    _check(got, _want_ext(spec, phase))
    # same frames through the mixture-phase form: the same signal up to the phase's float32 rounding
    assert np.max(np.abs(got - _run(emul, spec, pcm=gold["mixed_pcm"], chunks=chunks))) <= TOL_PCM * np.max(np.abs(got))


@pytest.mark.parametrize("T_use", [42, 43, 44, 45, 46, 47, 48, 49, 17, 2])
@pytest.mark.parametrize("chunks", [1, 2, 3])
def test_explicit_random_phase_every_length_mod_8(emul, T_use, chunks):
    """Phases that are not a mixture's: the packed frames (t, t+1) of each FFT carry unrelated phases, so swapping them or
    taking the wrong frame shows.  T_use = 0 ... 7 (mod 8): partial last groups; chunks 2, 3: warm-up groups."""
    rng = np.random.RandomState(T_use * 10 + chunks)
    spec = (rng.rand(80, T_use) * 40.0 - 60.0).astype(np.float32)
    phase = _random_phase(rng, T_use)
    _check(_run(emul, spec, phase=phase, chunks=chunks), _want_ext(spec, phase))


@pytest.mark.parametrize("chunks", [1, 3])
def test_explicit_phase_with_zero_entries(emul, chunks):
    """Phase entries 0 + 0j (allowed by dp:114: magnitude * phase) make their bins contribute nothing -- no 1 + 0j substitution,
    which is magphase's rule for the mixture form only.  Whole zero frames, a zero packed partner, and scattered zero bins."""
    rng = np.random.RandomState(11)
    T = 61
    spec = (rng.rand(80, T) * 40.0 - 60.0).astype(np.float32)
    phase = _random_phase(rng, T, zero_frac=0.3)
    phase[8] = 0.0               # first frame of a packed pair
    phase[19] = 0.0              # second frame of a packed pair
    phase[30:34] = 0.0           # both frames of two FFTs
    phase[:, 0] = 0.0
    _check(_run(emul, spec, phase=phase, chunks=chunks), _want_ext(spec, phase))


@pytest.mark.parametrize("phase_frames", [37, 45, 53])
@pytest.mark.parametrize("chunks", [1, 2])
def test_explicit_phase_frames_fewer_equal_more_than_mel(emul, phase_frames, chunks):
    """T_use = min(mel frames, phase frames): frames of the longer array beyond it are never read (they hold NaN here)."""
    rng = np.random.RandomState(phase_frames)
    T_mel = 45
    spec = (rng.rand(80, T_mel) * 40.0 - 60.0).astype(np.float32)
    phase = _random_phase(rng, phase_frames)
    T_use = min(T_mel, phase_frames)
    poisoned_spec, poisoned_phase = spec.copy(), phase.copy()
    poisoned_spec[:, T_use:] = np.nan
    poisoned_phase[T_use:] = np.nan
    got = _run(emul, poisoned_spec, phase=poisoned_phase, chunks=chunks)
    assert got.shape == (160 * (T_use - 1),)
    _check(got, _want_ext(spec[:, :T_use], phase[:T_use]))


@pytest.mark.parametrize("n_frames,pad", [(60, 4), (60, 13), (47, 1), (100, 7)])
@pytest.mark.parametrize("explicit", [False, True])
def test_spec_layout_reads_n_frames_columns_at_stride_ld_t(emul, n_frames, pad, explicit):
    """SPEC [80][ld_t] with ld_t > n_frames: the columns in between hold NaN and must not be read; against the oracle, and
    bit-identical to SLICES on the same frames (identical arithmetic, only the load address differs)."""
    rng = np.random.RandomState(n_frames + pad)
    spec = (rng.rand(80, n_frames) * 40.0 - 60.0).astype(np.float32)
    wide = np.full((80, n_frames + pad), np.nan, np.float32)
    wide[:, :n_frames] = spec
    L = 160 * (n_frames + 3) + 37              # the mixture has more frames than the mel: n_frames limits
    pcm = (0.2 * rng.randn(L)).astype(np.float32)
    phase = _random_phase(rng, n_frames + 2) if explicit else None
    kw = dict(phase=phase) if explicit else dict(pcm=pcm)
    for chunks in (1, 3):
        got = _run(emul, wide, n_frames=n_frames, chunks=chunks, **kw)
        _check(got, _want_ext(spec, phase) if explicit else _want_mixture(spec, pcm))
        if n_frames % 20 == 0:
            slices = np.ascontiguousarray(spec.reshape(80, n_frames // 20, 20).transpose(1, 0, 2))
            assert np.array_equal(got, _run(emul, slices, layout=0, chunks=chunks, **kw))


@pytest.mark.parametrize("n_frames", [41, 50, 57])
def test_spec_layout_with_the_mixture_limiting(emul, n_frames):
    """Form (c) with more mel frames than the mixture has (T = 1 + L/160 limits), and a zero-padded mixture (valid < L)."""
    rng = np.random.RandomState(n_frames)
    L = 160 * 49 + 11                          # T = 50
    pcm = np.zeros(L, np.float32)
    valid = 6000
    pcm[:valid] = (0.2 * rng.randn(valid)).astype(np.float32)
    spec = (rng.rand(80, n_frames + 5) * 40.0 - 60.0).astype(np.float32)
    for chunks in (1, 2):
        got = _run(emul, spec, pcm=pcm, valid=valid, n_frames=n_frames, chunks=chunks)
        _check(got, _want_mixture(spec[:, :n_frames], pcm))
