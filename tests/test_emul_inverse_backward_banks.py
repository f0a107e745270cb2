"""CPU check of the inverse's backward stage code (tests/emul/avse_emul_grad.cpp) on every caller-chosen filterbank of the stratified
sample of test_emul_filterbanks.py.  The backward reads the bank's banded F (mel_w / mel_lo) and the Thomas factors of F F^T, and
those tables change with every (sample_rate, fmin, fmax) build_tables accepts; test_emul_inverse_backward.py runs the reference bank
only.  The oracle is the float64 VJP of tests/inverse_vjp.py built with the bank's own filterbank; the gate is 1e-4 of the peak
|oracle gradient|.  Banks build_tables refuses are refused by the emulator as by avse_create (the generic kernels serve them)."""
import ctypes

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests import inverse_vjp as V
from tests.test_emul_filterbanks import REFUSED, SPECIALISED, STRATA
from tests.test_emul_inverse_backward import emul_grad, _p, TOL  # noqa: F401  (module fixture that builds the emulation library)


def _ids(banks):
    return ["%d_%d_%d" % b for b in banks]


def _cond(b):
    fb = O.mel_filterbank(b[0], 640, 80, float(b[1]), float(b[2]))
    return float(np.linalg.cond(fb @ fb.T))


# the five worst-conditioned accepted banks, and the first accepted bank of each rate other than 16 kHz
HARD = sorted(SPECIALISED, key=_cond)[-5:]
for _sr in (11025, 22050, 24000):
    HARD += [b for b in SPECIALISED if b[0] == _sr and b not in HARD][:1]
assert len({b[0] for b in HARD}) == 4

ERR = {}            # (bank, case) -> error: filled by the tests below, summarised by test_report_worst_per_stratum


def _stratum(bank):
    return next(k for k, v in STRATA.items() if bank in v)


def _run(lib, bank, mel, pcm, g, layout):
    """mel: SPEC [80, T_mel] (layout 1) or SLICES [n, 80, 20] (layout 0).  Returns (rc, grad_mel)."""
    mel = np.ascontiguousarray(mel, np.float32)
    pcm = np.ascontiguousarray(pcm, np.float32)
    g = np.ascontiguousarray(g, np.float32)
    out = np.full(mel.shape, np.nan, np.float32)
    if layout == 1:
        n_slices, n_frames, ld_t = 0, mel.shape[1], mel.shape[1]
    else:
        n_slices, n_frames, ld_t = mel.shape[0], 0, 0
    L = len(pcm)
    rc = lib.emul_inverse_backward(_p(mel), layout, n_slices, n_frames, ld_t, _p(pcm), L, L, _p(g), _p(out), bank[0],
                                   float(bank[1]), float(bank[2]))
    return rc, out


def _want(bank, mel_spec, pcm, g):
    """Oracle dL/d dB (80, T_mel) with the bank's filterbank, zeros beyond T_use."""
    _, phase = O.magphase(O.stft(np.asarray(pcm, np.float64), 640, 160))
    T_use = min(mel_spec.shape[1], phase.shape[1])
    out = np.zeros(mel_spec.shape)
    out[:, :T_use] = V.reconstruct_signal_from_spectrogram_vjp(np.asarray(mel_spec[:, :T_use], np.float64), phase[:, :T_use], bank[0],
                                                               640, 160, np.asarray(g, np.float64), fmin=float(bank[1]),
                                                               fmax=float(bank[2]))
    return out


def _err(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    peak = np.max(np.abs(want))
    assert peak > 0
    return float(np.max(np.abs(got - want)) / peak)


def _case(bank, seed, T_mel, L, scale=1.0, g_scale=1.0):
    sr, fmin, fmax = bank
    rng = np.random.RandomState(seed + fmin * 7 + fmax + sr)
    pcm = ((O.synth_speech(L, sr, seed) + O.synth_noise(L, seed + 1)) * scale).astype(np.float32)
    mel = (-40.0 + 12.0 * rng.randn(80, T_mel)).astype(np.float32)
    T_use = min(T_mel, 1 + L // 160)
    g = (g_scale * rng.randn(160 * (T_use - 1))).astype(np.float32)
    return mel, pcm, g


def _spec_err(lib, bank, mel, pcm, g):
    rc, got = _run(lib, bank, mel, pcm, g, 1)
    assert rc == min(mel.shape[1], 1 + len(pcm) // 160)
    return _err(got, _want(bank, mel, pcm, g))


def _spec_75(lib, bank):
    """SPEC, 75 frames (two chunks, the second 11 frames short), T_use = 75 of the mixture's 76."""
    mel, pcm, g = _case(bank, 1, 75, 12000)
    return _spec_err(lib, bank, mel, pcm, g)


def _slices_4(lib, bank):
    """SLICES, 4 slices = 80 frames against the mixture's 76: frames 76 ... 79 get exact zeros."""
    mel, pcm, g = _case(bank, 2, 80, 12000)
    sl = mel.reshape(80, 4, 20).transpose(1, 0, 2).copy()
    rc, got = _run(lib, bank, sl, pcm, g, 0)
    assert rc == 76
    spec = np.concatenate(list(got), axis=1)
    assert np.all(spec[:, 76:] == 0.0)
    return _err(spec, _want(bank, mel, pcm, g))


def _hard(lib, bank, kind):
    if kind == "grad_1e-8":
        mel, pcm, g = _case(bank, 3, 101, 16000, g_scale=1e-8)
    elif kind == "int16_scale":
        mel, pcm, g = _case(bank, 4, 101, 16000, scale=32768.0)
    else:                                   # digital silence inside the mixture: phase 1 + 0j there
        mel, pcm, g = _case(bank, 5, 101, 16000)
        pcm[3000:7000] = 0.0
    return _spec_err(lib, bank, mel, pcm, g)


CASES = {"spec_75": _spec_75, "slices_4": _slices_4}
HARD_KINDS = ["grad_1e-8", "int16_scale", "silence"]


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("bank", SPECIALISED, ids=_ids(SPECIALISED))
def test_accepted_bank_against_the_vjp(emul_grad, bank, case):
    err = ERR[bank, case] = CASES[case](emul_grad, bank)
    assert err <= TOL, err


@pytest.mark.parametrize("kind", HARD_KINDS)
@pytest.mark.parametrize("bank", HARD, ids=_ids(HARD))
def test_hard_banks_at_extreme_levels(emul_grad, bank, kind):
    """The worst-conditioned banks and the 11.025 / 22.05 / 24 kHz banks with a loss gradient 1e-8 under the mixture, an int16-scale
    mixture and digital silence inside the mixture."""
    err = ERR[bank, kind] = _hard(emul_grad, bank, kind)
    assert err <= TOL, err


@pytest.mark.parametrize("bank", REFUSED, ids=_ids(REFUSED))
def test_refused_bank_is_refused(emul_grad, bank):
    mel, pcm, g = _case(bank, 6, 30, 4800)
    assert _run(emul_grad, bank, mel, pcm, g, 1)[0] == -2


def test_report_worst_per_stratum(emul_grad):
    """Worst error per stratum and case (run with -s to see it), over every accepted bank; cases the tests above did not run here
    are run now."""
    todo = [(b, c, lambda b=b, c=c: CASES[c](emul_grad, b)) for b in SPECIALISED for c in CASES]
    todo += [(b, k, lambda b=b, k=k: _hard(emul_grad, b, k)) for b in HARD for k in HARD_KINDS]
    worst = {}
    for bank, case, fn in todo:
        if (bank, case) not in ERR:
            ERR[bank, case] = fn()
        key = (_stratum(bank), case)
        if ERR[bank, case] > worst.get(key, (-1.0,))[0]:
            worst[key] = (ERR[bank, case], bank)
    for (stratum, case), (err, bank) in sorted(worst.items()):
        print("WORST %s %s %.3g at %s (cond %.3g)" % (stratum, case, err, "%d_%d_%d" % bank, _cond(bank)))
    assert max(e for e, _ in worst.values()) <= TOL
