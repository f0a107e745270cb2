"""GPU counterpart of tests/test_emul_offsets.py: DC offsets, hum and tones through the public entry points, every row against
its own float64 oracle, and the statistics pass's (factor, equalizer) against numpy.  The gate is 1e-3 dB on the log-mels and
1e-4 of full scale on PCM; rows outside the envelope of the float32 packed FFT (DESIGN section 4.4) are held to the bounds
measured on the CPU emulator of the same stage code."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS, fitted_noise

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
LOOSE_NOISE_DC_DB = 2e-3      # noise DC 5 ... 100 x its std (CPU emulator: worst 1.5e-3 dB)
LOOSE_SPEECH_DC_DB = 2e-3     # speech DC 1 x its std (CPU emulator: worst 1.4e-3 dB)
LOOSE_TONE_DB = 2.5e-3        # hum / tones 1 ... 1000 x the speech std (CPU emulator: worst 1.8e-3 dB)


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _oracle(s, z, snr, nvs, fps=FPS, off=0):
    """dp:119-139 on (s, z rolled by off): (mixed, speech, noise) slices and the mixture PCM."""
    zr = np.roll(z.astype(np.float64), -off)
    r = O.preprocess_audio_pair_signals(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(zr, SR), 200, nvs, fps, snr_db=snr)
    return r[0], r[1], r[2], r[3].get_data()


def _check_row(got, ref, tol, what):
    """got / ref: (mixed, speech, noise, pcm) of one row; returns the worst (log-mel dB, PCM / full scale)."""
    db = max(float(np.max(np.abs(g - r))) for g, r in zip(got[:3], ref[:3]))
    pcm = float(np.max(np.abs(got[3] - ref[3])) / np.max(np.abs(ref[3])))
    assert db <= tol and pcm <= TOL_PCM, (what, db, pcm)
    return db, pcm


def _gains_ref(s, n, snr):
    s, n = s.astype(np.float64), n.astype(np.float64)
    return (np.sqrt(np.var(s) / np.var(n)) * 10.0 ** (-snr / 20.0), np.sqrt(np.sum(s * s) / np.sum(n * n)))


def _rows():
    """(name, speech, noise, snr, log-mel bound) rows with DC offsets, int16-valued or float, ragged lengths."""
    rows = []
    snrs = (-10.0, 0.0, 10.0)
    for i, dc in enumerate((0.1, 1.0, 3.0, 5.0, 10.0, 30.0, 100.0)):
        n = 16000 - 997 * i
        s0, n0 = O.synth_speech(n, SR, 400 + i), O.synth_noise(n, 400 + i)
        rows.append(("noise_dc%g" % dc, s0, n0 + dc * n0.std(), snrs[i % 3], TOL_DB if dc <= 3.0 else LOOSE_NOISE_DC_DB))
    for i, dc in enumerate((3, 30, 200, 900)):
        n = 16000 - 1500 * i
        s0, n0 = O.synth_speech(n, SR, 420 + i), O.synth_noise(n, 420 + i)
        rows.append(("i16_noise_dc%d" % dc, np.round(s0 / s0.std() * 1000.0), np.round(n0 / n0.std() * 30.0 + dc), snrs[i % 3], TOL_DB))
    s0, n0 = O.synth_speech(15000, SR, 430), O.synth_noise(15000, 430)
    rows.append(("i16_both_dc", np.round(s0 / s0.std() * 1000.0 + 300.0), np.round(n0 / n0.std() * 30.0 + 200.0), 0.0, TOL_DB))
    rows.append(("speech_dc0.1", s0 + 0.1 * s0.std(), n0, -10.0, TOL_DB))
    return rows


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_preprocess_pairs_with_dc_offsets(eng, i16):
    """A ragged batch with per-row SNR; the factor within float32 rounding of numpy's float64 value and DbKeys.equalizer =
    sqrt(E[s^2] / E[n^2]) over the row's own samples."""
    rows = _rows()
    B, W = len(rows), 16000
    dt = np.int16 if i16 else np.float32
    S = np.zeros((B, W), dt)
    Z = np.zeros((B, W), dt)
    lens = np.zeros(B, np.int32)
    data = []
    for i, (name, s, z, snr, tol) in enumerate(rows):
        if i16 and not name.startswith("i16"):      # float-scale rows at int16 scale
            s, z = s * 10000.0, z * 10000.0
        if i16:
            s, z = np.round(s), np.round(z)
        s, z = s.astype(dt), z.astype(dt)
        data.append((s, z))
        S[i, :len(s)], Z[i, :len(s)], lens[i] = s, z, len(s)
    snr = np.array([r[3] for r in rows], np.float32)
    info = {}
    got = eng.preprocess_pairs(_dev(S), _dev(Z), 5, lengths=_dev(lens), snr_db=_dev(snr), info=info)
    got = [t.cpu().numpy() for t in got]
    fac, eq = info["factor"].cpu().numpy(), info["keys"].equalizer.cpu().numpy()
    worst = {}
    for i, (name, _, _, _, tol) in enumerate(rows):
        s, z = data[i]
        wf, wg = _gains_ref(s, z, float(snr[i]))
        assert abs(fac[i] - wf) <= 2e-7 * wf and abs(eq[i] - wg) <= 2e-7 * wg, (name, fac[i], wf, eq[i], wg)
        worst[name] = _check_row([g[i] for g in got], _oracle(s, z, float(snr[i]), 5), tol, name)
    print("preprocess_pairs %s worst (dB, PCM): %s" % ("i16" if i16 else "f32", worst))


def test_tiled_noise_with_dc(eng):
    """noise_lengths: noise files shorter than their speech, tiled in the kernels; the equaliser over the weighted period."""
    B, L = 4, 16000
    n_noise = [5000, 1121, 333, 16000]
    S = np.stack([O.synth_speech(L, SR, 440 + i) for i in range(B)]).astype(np.float32)
    Z = np.full((B, L), np.nan, np.float32)
    raw = []
    for i, m in enumerate(n_noise):
        n0 = O.synth_noise(m, 440 + i)
        z = (n0 + (1.0, 3.0)[i % 2] * n0.std()).astype(np.float32)
        raw.append(z)
        Z[i, :m] = z
    snr = np.array([-10.0, 0.0, 10.0, 3.0], np.float32)
    info = {}
    got = eng.preprocess_pairs(_dev(S), _dev(Z), 5, snr_db=_dev(snr), noise_lengths=_dev(np.array(n_noise, np.int32)), info=info)
    got = [t.cpu().numpy() for t in got]
    eq = info["keys"].equalizer.cpu().numpy()
    for i in range(B):
        _, wg = _gains_ref(S[i], fitted_noise(S[i], raw[i]), 0.0)
        assert abs(eq[i] - wg) <= 2e-7 * wg, i
        _check_row([g[i] for g in got], _oracle(S[i], raw[i], float(snr[i]), 5), TOL_DB, i)


def test_mix_pools_with_noise_dc(eng):
    """Pooled pairs with a noise DC of 3 x its std read from offsets 0, 1 and Ln - 1; float32 and int16 pools."""
    Ls, Lns = [16000, 12000], [5000, 20000]
    for i16 in (False, True):
        dt = np.int16 if i16 else np.float32
        scale = 1000.0 if i16 else 1.0
        sp = np.zeros((2, 16000), dt)
        npool = np.zeros((2, 20000), dt)
        sclips, nclips = [], []
        for j in range(2):
            s = O.synth_speech(Ls[j], SR, 450 + j) * scale
            n0 = O.synth_noise(Lns[j], 450 + j)
            z = (n0 / n0.std() * 0.05 + 0.15) * scale
            s, z = (np.round(s), np.round(z)) if i16 else (s, z)
            sp[j, :Ls[j]], npool[j, :Lns[j]] = s.astype(dt), z.astype(dt)
            sclips.append(sp[j, :Ls[j]])
            nclips.append(npool[j, :Lns[j]])
        si = np.array([0, 0, 0, 1, 1, 1], np.int64)
        ni = np.array([0, 0, 0, 1, 1, 0], np.int64)
        off = np.array([0, 1, 4999, 0, 19999, 1], np.int32)
        snr = np.array([-10.0, 0.0, 10.0, -5.0, 5.0, 0.0], np.float32)
        info = {}
        got = eng.mix_pools(_dev(sp), _dev(np.array(Ls, np.int32)), _dev(npool), _dev(np.array(Lns, np.int32)), _dev(si), _dev(ni), 5,
                            noise_offset=_dev(off), snr_db=_dev(snr), info=info)
        got = [t.cpu().numpy() for t in got]
        eq = info["keys"].equalizer.cpu().numpy()
        for b in range(len(si)):
            s, z = sclips[si[b]], nclips[ni[b]]
            _, wg = _gains_ref(s, fitted_noise(s, np.roll(z, -off[b])), 0.0)
            assert abs(eq[b] - wg) <= 2e-7 * wg, (i16, b)
            _check_row([g[b] for g in got], _oracle(s, z, float(snr[b]), 5, off=int(off[b])), TOL_DB, (i16, b))


def test_spectrogram_and_stft_with_dc_and_hum(eng):
    """spectrogram(..., stft=True) of single signals with a DC offset or a hum inside the envelope (0.3 x the std) and, held to
    the measured bounds, a strong hum and a DC of 1 x the std; the complex STFT within 2e-6 of its peak in every case."""
    L = 20000
    t = np.arange(L) / SR
    x0 = O.synth_speech(L, SR, 460)
    cases = [(x0 + 0.3 * x0.std(), TOL_DB), (x0 + 0.3 * x0.std() * np.sin(2 * np.pi * 50 * t), TOL_DB),
             (x0 + 100.0 * x0.std() * np.sin(2 * np.pi * 60 * t), LOOSE_TONE_DB), (x0 + 1.0 * x0.std(), LOOSE_SPEECH_DC_DB)]
    X = np.stack([c[0] for c in cases]).astype(np.float32)
    db, D = eng.spectrogram(_dev(X), stft=True)
    for i, (_, tol) in enumerate(cases):
        ref_db, _ = O.signal_to_spectrogram(O.AudioSignal(X[i].astype(np.float64), SR), 640, 160)
        assert np.max(np.abs(db[i].cpu().numpy() - ref_db)) <= tol, i
        ref_D = O.stft(X[i].astype(np.float64), 640, 160)
        assert np.max(np.abs(D[i].cpu().numpy().T - ref_D)) <= 2e-6 * np.max(np.abs(ref_D)), i


def test_reconstruct_on_mixtures_with_dc_and_hum(eng):
    """reconstruct (dp:60-74) of mixtures carrying a DC offset, a hum or a tone, with the clean speech's mel."""
    L = 16000
    t = np.arange(L) / SR
    mixes, mels = [], []
    for i, (kind, level) in enumerate((("dc", 1.0), ("dc", 10.0), ("dc", 100.0), (50.0, 10.0), (60.0, 100.0), (1012.5, 100.0))):
        s0, n0 = O.synth_speech(L, SR, 470 + i), O.synth_noise(L, 470 + i)
        extra = level * s0.std() * (1.0 if kind == "dc" else np.sin(2 * np.pi * kind * t))
        mixes.append((s0 + n0 + extra).astype(np.float32))
        mels.append(O.preprocess_audio_signal(O.AudioSignal(s0.copy(), SR), 200, 5, FPS).astype(np.float32))
    rec = eng.reconstruct(_dev(np.stack(mixes)), _dev(np.stack(mels))).cpu().numpy()
    for i in range(len(mixes)):
        want = O.reconstruct_speech_signal(O.AudioSignal(mixes[i].astype(np.float64), SR), mels[i].astype(np.float64), FPS).get_data()
        assert np.max(np.abs(rec[i] - want)) <= TOL_PCM * np.max(np.abs(want)), i


def test_generic_geometry_control(mod):
    """320 @ 50 fps runs the generic kernels, which compute in float64 and ignore the equaliser: a noise DC of 100 x its std
    stays within the gate there (a control for the float32 limit of the specialised kernels)."""
    e = mod.SpectralEngine(SR, 50.0, 200, device="cuda:0")
    assert not e.specialised
    L = 16000
    s0, n0 = O.synth_speech(L, SR, 480), O.synth_noise(L, 480)
    S = np.stack([s0, s0 + 0.3 * s0.std()]).astype(np.float32)
    Z = np.stack([n0 + 100.0 * n0.std(), n0 + 10.0 * n0.std()]).astype(np.float32)
    snr = np.array([0.0, -10.0], np.float32)
    info = {}
    got = [t.cpu().numpy() for t in e.preprocess_pairs(_dev(S), _dev(Z), 5, snr_db=_dev(snr), info=info)]
    eq = info["keys"].equalizer.cpu().numpy()
    for i in range(2):
        _, wg = _gains_ref(S[i], Z[i], 0.0)
        assert abs(eq[i] - wg) <= 2e-7 * wg, i
        _check_row([g[i] for g in got], _oracle(S[i], Z[i], float(snr[i]), 5, fps=50.0), TOL_DB, i)
