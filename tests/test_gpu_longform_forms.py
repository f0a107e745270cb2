"""Every entry point at 60 s against the float64 oracle: the int16 and PAD / TILED instantiations of the F4 forward kernel,
mix_pools, HostPipeline, the F2 single-signal kernel (spectrogram, preprocess_signals), the SLICES / SPEC / EXT inverse forms and
the int16 store, the backward's 32-frame work items (188 per utterance), and a generic-geometry context.  A ragged batch of rows of
L60, L60 - 1 and L60 - 123457 samples with poison (NaN / int16 30000) past every row's length; output rows are views of wider
buffers whose guard bands must come back untouched.  The gates are the suite's: 1e-3 dB on log-mels, 1e-4 of the peak on PCM,
+-1 LSB on int16 output, 1e-4 of the peak gradient."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests import inverse_vjp as V
from tests.cases import FRAME_RATES, FPS
from tests.longform_cases import L60, POOL_NOISE, POOL_ROWS, SR, build_pools, pool_row_noise

pytestmark = pytest.mark.gpu

TOL_DB, TOL_PCM, TOL_GRAD = 1e-3, 1e-4, 1e-4
NVS = 300
LENS = [L60, L60 - 1, L60 - 123457]
GUARD = 16
SENTINEL = -12345.0
LN10_20 = np.log(10.0) / 20.0
GENERIC = next(g for g in FRAME_RATES if g["name"] == "22k05_29.97")


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _rows(lens, width, seed, i16=False, sr=SR):
    """Speech / noise rows (float32, or int16 WAV scale) with poison past each row's length; the clean rows as a list."""
    dt, poison = (np.int16, 30000) if i16 else (np.float32, np.nan)
    S = np.full((len(lens), width), poison, dt)
    Z = np.full((len(lens), width), poison, dt)
    rows = []
    for i, n in enumerate(lens):
        s, z = O.synth_speech(n, sr, seed + i), O.synth_noise(n, seed + i)
        if i16:
            s, z = np.round(s * 20000.0), np.round(z * 20000.0)
        S[i, :n], Z[i, :n] = s.astype(dt), z.astype(dt)
        rows.append((S[i, :n].copy(), Z[i, :n].copy()))
    return S, Z, rows


def _guarded(shape, dtype=torch.float32):
    """A [B, ...] output view whose rows are followed by GUARD sentinel elements; returns (view, the whole buffer)."""
    B, per = shape[0], int(np.prod(shape[1:]))
    buf = torch.full((B, per + GUARD), SENTINEL, dtype=dtype, device="cuda")
    return buf[:, :per].view(shape), buf


def _guards_intact(buf):
    assert torch.all(buf[:, -GUARD:] == SENTINEL)


def _pair_oracle(s, z, snr, fps=FPS, sr=SR, nvs=NVS):
    r = O.preprocess_audio_pair_signals(O.AudioSignal(np.asarray(s, np.float64), sr), O.AudioSignal(np.asarray(z, np.float64), sr), 200,
                                        nvs, fps, snr_db=snr)
    return r[0], r[1], r[2], r[3].get_data()


def _pair_err(got, b, ref):
    db = max(float(np.max(np.abs(got[k][b] - ref[k]))) for k in range(3))
    pcm = float(np.max(np.abs(got[3][b] - ref[3])) / np.max(np.abs(ref[3])))
    assert db <= TOL_DB and pcm <= TOL_PCM, (b, db, pcm)
    return db, pcm


def _pair_out(eng, B, L, n):
    out, bufs = {}, []
    for k in ("mixed", "speech", "noise"):
        out[k], buf = _guarded((B, n, eng.n_mels, eng.spss))
        bufs.append(buf)
    out["mixed_pcm"], buf = _guarded((B, L))
    bufs.append(buf)
    return out, bufs


def test_preprocess_pairs_int16_ragged(eng):
    """The int16 PAD instantiation of F4 (raw WAV samples, per-row lengths) with guard bands after every output row."""
    S, Z, rows = _rows(LENS, L60, 600, i16=True)
    snr = np.array([-10.0, 0.0, 7.5], np.float32)
    out, bufs = _pair_out(eng, len(LENS), L60, NVS)
    got = eng.preprocess_pairs(_dev(S), _dev(Z), NVS, lengths=_dev(np.array(LENS, np.int32)), snr_db=_dev(snr), out=out)
    for buf in bufs:
        _guards_intact(buf)
    got = [t.cpu().numpy() for t in got]
    worst = [max(e) for e in zip(*[_pair_err(got, b, _pair_oracle(s, z, float(snr[b]))) for b, (s, z) in enumerate(rows)])]
    print("preprocess_pairs int16 PAD at 60 s: worst %.2e dB, %.2e of the PCM peak" % tuple(worst))


def test_preprocess_pairs_tiled_noise(eng):
    """TILED: a 27 371-sample noise under every row (period boundaries inside about 35 of a row's groups, a large q in the
    interior shift)."""
    Pn = 27371
    S, _, rows = _rows(LENS, L60, 610)
    Z = np.full((len(LENS), L60), np.nan, np.float32)
    raw = []
    for i in range(len(LENS)):
        z = O.synth_noise(Pn, 620 + i).astype(np.float32)
        Z[i, :Pn] = z
        raw.append(z)
    snr = np.array([5.0, -5.0, 0.0], np.float32)
    got = eng.preprocess_pairs(_dev(S), _dev(Z), NVS, lengths=_dev(np.array(LENS, np.int32)), snr_db=_dev(snr),
                               noise_lengths=_dev(np.full(len(LENS), Pn, np.int32)))
    got = [t.cpu().numpy() for t in got]
    worst = [max(e) for e in zip(*[_pair_err(got, b, _pair_oracle(rows[b][0], raw[b], float(snr[b]))) for b in range(len(LENS))])]
    print("preprocess_pairs TILED at 60 s: worst %.2e dB, %.2e of the PCM peak" % tuple(worst))


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_mix_pools_at_60s(mod, eng, i16):
    """The cluster pools of test_gpu_snr_clusters.py mixed at 60 s (the 40 s clip zero padded): a wrapping window, the periodic
    regime at off = 1 and a wrapping window of a 10 s clip."""
    sp, slen, nz, nlen, sclips, nclips = build_pools(mod, i16, True, 8)
    pick = [0, 3, 8]
    rows = [POOL_ROWS[k] for k in pick]
    snr = np.array([-10.0, 0.0, 10.0], np.float32)
    got = eng.mix_pools(sp, slen, nz, nlen, torch.tensor([r[0] for r in rows]), torch.tensor([r[1] for r in rows]), NVS,
                        noise_offset=torch.tensor([r[2] for r in rows], dtype=torch.int32), snr_db=_dev(snr))
    got = [t.cpu().numpy() for t in got]
    errs = []
    for b, (si, ni, off) in enumerate(rows):
        s, z = sclips[si], nclips[ni]
        errs.append(_pair_err(got, b, _pair_oracle(s, pool_row_noise(z, POOL_NOISE[ni], off, len(s)), float(snr[b]))))
    print("mix_pools %s at 60 s: worst %.2e dB, %.2e of the PCM peak" % (("i16" if i16 else "f32",) + tuple(max(e) for e in zip(*errs))))


def test_host_pipeline_equals_preprocess_pairs(mod, eng):
    """HostPipeline at 60 s, two utterances per chunk, tiled noises: bit-identical to preprocess_pairs on the same rows."""
    B = 3
    S, _, _ = _rows([L60] * B, L60, 630)
    nl = np.array([27371, 960000, 4099], np.int32)
    Z = np.full((B, L60), np.nan, np.float32)
    for i in range(B):
        Z[i, :nl[i]] = O.synth_noise(int(nl[i]), 640 + i)
    snr = np.array([-3.0, 0.0, 3.0], np.float32)
    pipe = mod.HostPipeline(eng, L60, NVS, chunk=2, n_streams=2)
    n = eng.n_slices(L60)
    h = {k: torch.empty((B, n, 80, 20)).pin_memory() for k in ("mixed", "speech", "noise")}
    h_pcm = torch.empty((B, L60)).pin_memory()
    assert pipe.submit(torch.from_numpy(S).pin_memory(), torch.from_numpy(Z).pin_memory(), h["mixed"], h["speech"], h["noise"], h_pcm,
                       snr_db=torch.from_numpy(snr).pin_memory(), noise_lengths=torch.from_numpy(nl).pin_memory()) == 2
    pipe.synchronize()
    want = eng.preprocess_pairs(_dev(S), _dev(Z), NVS, snr_db=_dev(snr), noise_lengths=_dev(nl))
    for got, w in zip((h["mixed"], h["speech"], h["noise"], h_pcm), want):
        assert torch.equal(got, w.cpu())


def test_spectrogram_and_preprocess_signals_ragged(eng):
    """The F2 single-signal kernel: floored dB and the complex STFT (within 2e-6 of its peak), and the dB slices, rows zero
    padded past their lengths."""
    X, _, rows = _rows(LENS, L60, 650)
    ln = _dev(np.array(LENS, np.int32))
    db, D = eng.spectrogram(_dev(X), lengths=ln, stft=True)
    sl = eng.preprocess_signals(_dev(X), NVS, lengths=ln).cpu().numpy()
    db, D = db.cpu().numpy(), D.cpu().numpy()
    w_db = w_st = w_sl = 0.0
    for i, (x, _) in enumerate(rows):
        xp = np.zeros(L60)
        xp[:len(x)] = x
        ref_db, _ = O.signal_to_spectrogram(O.AudioSignal(xp, SR), 640, 160)
        w_db = max(w_db, float(np.max(np.abs(db[i] - ref_db))))
        ref_D = O.stft(xp, 640, 160)
        w_st = max(w_st, float(np.max(np.abs(D[i].T - ref_D)) / np.max(np.abs(ref_D))))
        ref_sl = O.preprocess_audio_signal(O.AudioSignal(x.astype(np.float64), SR), 200, NVS, FPS)
        w_sl = max(w_sl, float(np.max(np.abs(sl[i] - ref_sl))))
        assert w_db <= TOL_DB and w_st <= 2e-6 and w_sl <= TOL_DB, (i, w_db, w_st, w_sl)
    print("spectrogram / STFT / preprocess_signals at 60 s: worst %.2e dB, %.2e of the STFT peak, %.2e dB" % (w_db, w_st, w_sl))


def _mixtures(eng, seed, sr=SR, fps=FPS, lens=LENS):
    """Mixture PCM rows (ragged, poison past each length) and clean-speech dB slices from the oracle."""
    width = max(lens)
    P, _, rows = _rows(lens, width, seed, sr=sr)
    for i, (x, _) in enumerate(rows):
        P[i, :len(x)] += (O.synth_noise(len(x), seed + 50 + i) * 0.5).astype(np.float32)
    n = eng.n_slices(eng.samples_per_slice * (width // eng.samples_per_slice))
    mels = np.stack([O.preprocess_audio_signal(O.AudioSignal(O.synth_speech(width, sr, seed + 90 + i), sr), 200, n, fps)
                     for i in range(len(lens))]).astype(np.float32)
    return P, mels


def _clean(P, lens):
    out = []
    for i, n in enumerate(lens):
        x = np.zeros(P.shape[1])
        x[:n] = P[i, :n]
        out.append(x)
    return out


def test_inverse_forms(eng):
    """reconstruct (float32 and the int16 store, guard bands after every row), reconstruct_spec (SPEC layout) and
    reconstruct_with_phase (EXT: the oracle's own phase of each mixture) on the ragged 60 s rows."""
    P, mels = _mixtures(eng, 660)
    B = len(LENS)
    ln = _dev(np.array(LENS, np.int32))
    T_use = min(20 * mels.shape[1], eng.n_frames(L60))
    out_len = 160 * (T_use - 1)
    out32, buf32 = _guarded((B, out_len))
    rec = eng.reconstruct(_dev(P), _dev(mels), lengths=ln, out=out32).cpu().numpy()
    loud = _dev(mels + 90.0)
    out16, buf16 = _guarded((B, out_len), torch.int16)
    rec16 = eng.reconstruct(_dev(P), loud, lengths=ln, out=out16, out_dtype=torch.int16).cpu().numpy().astype(np.int32)
    _guards_intact(buf32)
    _guards_intact(buf16)
    spec = np.concatenate([mels[:, k] for k in range(mels.shape[1])], axis=2)       # [B, 80, 20 n]
    rec_spec = eng.reconstruct_spec(_dev(P), _dev(spec), lengths=ln).cpu().numpy()
    phases = []
    worst = {"slices": 0.0, "int16": 0, "spec": 0.0, "ext": 0.0}
    for i, x in enumerate(_clean(P, LENS)):
        sig = O.AudioSignal(x, SR)
        want = O.reconstruct_speech_signal(sig, mels[i].astype(np.float64), FPS).get_data()
        scale = float(np.max(np.abs(x)))
        worst["slices"] = max(worst["slices"], float(np.max(np.abs(rec[i] - want))) / scale)
        worst["spec"] = max(worst["spec"], float(np.max(np.abs(rec_spec[i] - want))) / scale)
        want16 = O.reconstruct_speech_signal(sig, mels[i].astype(np.float64) + 90.0, FPS).get_data()
        ref16 = np.clip(want16, -32768, 32767).astype(np.int16).astype(np.int32)
        worst["int16"] = max(worst["int16"], int(np.max(np.abs(rec16[i] - ref16))))
        _, ph = O.magphase(O.stft(x, 640, 160))
        phases.append(ph.T.astype(np.complex64))
        assert worst["slices"] <= TOL_PCM and worst["spec"] <= TOL_PCM and worst["int16"] <= 1, (i, worst)
    got = eng.reconstruct_with_phase(_dev(spec), _dev(np.stack(phases))).cpu().numpy()
    for i, x in enumerate(_clean(P, LENS)):
        want = O.reconstruct_signal_from_spectrogram(spec[i].astype(np.float64)[:, :T_use], phases[i].T.astype(np.complex128)[:, :T_use],
                                                     SR, 640, 160).get_data()
        worst["ext"] = max(worst["ext"], float(np.max(np.abs(got[i] - want)) / np.max(np.abs(want))))
        assert worst["ext"] <= TOL_PCM, (i, worst)
    print("inverse forms at 60 s: worst %s" % worst)


def test_reconstruct_differentiable(eng):
    """The backward's 32-frame work items at 60 s (188 per utterance) against tests/inverse_vjp.py on every row, and the
    oracle-free identity sum dL/d dB = ln10 / 20 <y, g> (y is linear in 10^(dB / 20))."""
    P, mels = _mixtures(eng, 670)
    ln = _dev(np.array(LENS, np.int32))
    m = _dev(mels).requires_grad_(True)
    y = eng.reconstruct_differentiable(_dev(P), m, lengths=ln)
    g = np.random.RandomState(671).randn(*y.shape).astype(np.float32)
    y.backward(_dev(g))
    got, yv = m.grad.cpu().numpy(), y.detach().cpu().numpy()
    worst = 0.0
    for i, x in enumerate(_clean(P, LENS)):
        want = V.reconstruct_speech_signal_vjp(O.AudioSignal(x, SR), mels[i].astype(np.float64), FPS, g[i].astype(np.float64))
        err = float(np.max(np.abs(got[i] - want)) / np.max(np.abs(want)))
        worst = max(worst, err)
        assert err <= TOL_GRAD, (i, err)
        lhs = float(np.sum(got[i].astype(np.float64)))
        rhs = LN10_20 * float(np.dot(yv[i].astype(np.float64), g[i].astype(np.float64)))
        assert abs(lhs - rhs) <= 1e-5 * float(np.sum(np.abs(got[i].astype(np.float64)))), (i, lhs, rhs)
    print("reconstruct_differentiable at 60 s: worst gradient error %.2e of the peak" % worst)


def test_generic_geometry_at_60s(mod):
    """22.05 kHz at 29.97 fps (n_fft 735, hop 183): the generic forward pair, the three inverse forms and the backward at 60 s."""
    e = mod.SpectralEngine(GENERIC["sr"], GENERIC["fps"], 200, device="cuda:0")
    assert not e.specialised
    sr, fps = GENERIC["sr"], GENERIC["fps"]
    L = e.samples_per_slice * NVS
    lens = [L, L - 1, L - 123457]
    S, Z, rows = _rows(lens, L, 680, sr=sr)
    snr = np.array([-10.0, 0.0, 10.0], np.float32)
    got = e.preprocess_pairs(_dev(S), _dev(Z), NVS, lengths=_dev(np.array(lens, np.int32)), snr_db=_dev(snr))
    got = [t.cpu().numpy() for t in got]
    fw = [max(v) for v in zip(*[_pair_err(got, b, _pair_oracle(s, z, float(snr[b]), fps=fps, sr=sr)) for b, (s, z) in enumerate(rows)])]
    n_fft, hop = e.n_fft, e.hop
    pcm = _dev(np.nan_to_num(got[3]))
    sl = _dev(got[1])
    ln = _dev(np.array(lens, np.int32))
    rec = e.reconstruct(pcm, sl, lengths=ln).cpu().numpy()
    spec = np.concatenate([got[1][:, k] for k in range(got[1].shape[1])], axis=2)
    rec_spec = e.reconstruct_spec(pcm, _dev(spec), lengths=ln).cpu().numpy()
    m = sl.clone().requires_grad_(True)
    y = e.reconstruct_differentiable(pcm, m, lengths=ln)
    g = np.random.RandomState(681).randn(*y.shape).astype(np.float32)
    y.backward(_dev(g))
    grad = m.grad.cpu().numpy()
    T_use = min(e.spss * got[1].shape[1], e.n_frames(L))
    phases = []
    worst = {"slices": 0.0, "spec": 0.0, "ext": 0.0, "grad": 0.0}
    for i, n in enumerate(lens):
        x = np.zeros(L)
        x[:n] = got[3][i, :n]
        sig = O.AudioSignal(x, sr)
        want = O.reconstruct_speech_signal(sig, got[1][i].astype(np.float64), fps).get_data()
        scale = float(np.max(np.abs(x)))
        worst["slices"] = max(worst["slices"], float(np.max(np.abs(rec[i] - want))) / scale)
        worst["spec"] = max(worst["spec"], float(np.max(np.abs(rec_spec[i] - want))) / scale)
        wg = V.reconstruct_speech_signal_vjp(sig, got[1][i].astype(np.float64), fps, g[i].astype(np.float64))
        worst["grad"] = max(worst["grad"], float(np.max(np.abs(grad[i] - wg)) / np.max(np.abs(wg))))
        _, ph = O.magphase(O.stft(x, n_fft, hop))
        phases.append(ph.T[:T_use].astype(np.complex64))
    ext = e.reconstruct_with_phase(_dev(spec[:, :, :T_use]), _dev(np.stack(phases))).cpu().numpy()
    for i in range(len(lens)):
        want = O.reconstruct_signal_from_spectrogram(spec[i, :, :T_use].astype(np.float64), phases[i].T.astype(np.complex128), sr,
                                                     n_fft, hop).get_data()
        worst["ext"] = max(worst["ext"], float(np.max(np.abs(ext[i] - want)) / np.max(np.abs(want))))
    print("generic 22.05 kHz / 29.97 fps at 60 s: forward %.2e dB, %.2e of the PCM peak; inverse %s" % (fw[0], fw[1], worst))
    assert worst["slices"] <= TOL_PCM and worst["spec"] <= TOL_PCM and worst["ext"] <= TOL_PCM and worst["grad"] <= TOL_GRAD, worst
