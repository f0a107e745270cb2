"""GPU parity of every entry point on caller-chosen mel filterbanks (SpectralEngine(..., fmin, fmax)).

At the 640 / 160 / 80 / 20 geometry the specialised kernels serve a bank build_tables accepts -- the F4 or the fused-scan F2 forward
kernel where the tables allow it, the F2 band-gather kernel otherwise, and the I8 inverse -- and the generic kernels serve a bank it
refuses (no I8 walk, or F F^T too ill-conditioned for the float32 solve).  One bank per accepted flag combination, the refused
banks the I8 inverse used to get wrong, and one 24 kHz bank reached through the engine's own geometry.  The oracle is the float64
composition of O.stft / O.mel_filterbank(sr, 640, 80, fmin, fmax) / O.amplitude_to_db and, back, istft((pinv(fb) 10^(mel/20)) phase).
Tolerances are BASELINE.json's: 1e-3 dB on log-mel, 1e-4 of the peak on PCM."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.test_gpu_inverse_forms import _inverse

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4

# (sample rate, video fps, slice ms, fmin, fmax, specialised)
BANKS = [
    (16000, 25.0, 200, 0.0, 8000.0, True),       # reference: F4 + fused scan + I8
    (16000, 25.0, 200, 0.0, 7900.0, True),       # no scan tables: F2 band gather + I8
    (16000, 25.0, 200, 50.0, 7000.0, True),
    (16000, 25.0, 200, 1000.0, 8000.0, True),    # F2 band gather + I8
    (16000, 25.0, 200, 80.0, 3000.0, False),     # no I8 walk
    (16000, 25.0, 200, 980.0, 6200.0, False),    # no I8 walk (scan tables valid)
    (16000, 25.0, 200, 550.0, 4600.0, False),    # cond(F F^T) ~ 2e15
    (16000, 25.0, 200, 300.0, 3500.0, False),    # cond(F F^T) ~ 1e17, no I8 walk
    (24000, 37.5, 133.34, 50.0, 8000.0, False),  # n_fft 640, 20 frames per slice; no I8 walk
]
IDS = ["%d_%g_%g" % (b[0], b[3], b[4]) for b in BANKS]


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


_ENGINES = {}


@pytest.fixture(params=BANKS, ids=IDS)
def bank(request, mod):
    b = request.param
    if b not in _ENGINES:
        _ENGINES[b] = mod.SpectralEngine(b[0], b[1], b[2], fmin=b[3], fmax=b[4], device="cuda:0")
    return _ENGINES[b], b


def _d(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _fb(b):
    return O.mel_filterbank(b[0], 640, 80, b[3], b[4])


def _spec(x, b):
    """signal_to_spectrogram (dp:77-96) with the bank's filterbank: floored dB (80, T) and the phase (321, T)."""
    return O.signal_to_spectrogram(O.AudioSignal(np.asarray(x, np.float64), b[0]), 640, 160, fmin=b[3], fmax=b[4])


def _signal(n, sr, seed):
    """Broadband 'speech': synthetic speech has little energy above ~5 kHz, and a band where the noise is > 60 dB above the speech
    is beyond the packed FFT's float32 cross-talk on any bank."""
    return (O.synth_speech(n, sr, seed) + 0.3 * O.synth_noise(n, seed + 1)).astype(np.float32)


def _pair_oracle(s, z, L, snr, b):
    """preprocess_audio_pair (dp:119-139) with the bank's filterbank: slices (mixed, speech, noise) and the mixture PCM."""
    sp = O.AudioSignal(s.astype(np.float64), b[0])
    nz = O.fit_noise_to_speech(O.AudioSignal(z.astype(np.float64), b[0]), sp)
    nz.amplify_by_factor(O.AudioMixer.snr_factor(sp, nz, snr))
    mixed = sp.get_data() + nz.get_data()
    out = []
    for x in (mixed, sp.get_data(), nz.get_data()):
        x = np.concatenate([x, np.zeros(max(0, L - len(x)))])[:L]
        mel = _spec(x, b)[0]
        n = mel.shape[1] // 20
        out.append(np.stack([mel[:, 20 * i:20 * i + 20] for i in range(n)]))
    return out, np.concatenate([mixed, np.zeros(max(0, L - len(mixed)))])[:L]


def _worst(b, entry, err):
    print("WORST %s %s %.3g" % ("%d_%g_%g" % (b[0], b[3], b[4]), entry, err))


def test_dispatch_and_filterbank(bank):
    eng, b = bank
    assert eng.specialised == b[5]
    assert (eng.n_fft, eng.hop, eng.n_mels, eng.spss) == (640, 160, 80, 20)
    assert np.max(np.abs(eng.filterbank() - _fb(b))) < 1e-13


def test_preprocess_pairs_ragged_with_guard_bands(bank):
    """Three utterances of different lengths, per-row SNR; the outputs written into rows with a sentinel guard band after each and
    a spare row: log-mel slices within 1e-3 dB, the mixture within 1e-4 of its peak, every guard word untouched."""
    eng, b = bank
    sr = b[0]
    nvs = 5
    L = eng.samples_per_slice * nvs
    lens = np.array([L, int(0.7 * L) + 3, int(0.45 * L) + 1], np.int32)
    B = len(lens)
    S = np.zeros((B, L), np.float32)
    Z = np.zeros((B, L), np.float32)
    for i, n in enumerate(lens):
        S[i, :n] = _signal(n, sr, 10 + i)
        Z[i, :n] = O.synth_noise(n, 20 + i) * (0.3, 3.0, 0.05)[i]
    snr = np.array([-5.0, 0.0, 7.5], np.float32)
    n = min(nvs, eng.n_frames(L) // 20)
    SENT, gap = -12345.0, 48
    row = n * 80 * 20 + gap
    bufs = {k: torch.full((B + 1, row), SENT, device="cuda") for k in ("speech", "noise", "mixed")}
    pcm_buf = torch.full((B + 1, L + gap), SENT, device="cuda")
    out = {k: torch.as_strided(v, (B, n, 80, 20), (row, 1600, 20, 1)) for k, v in bufs.items()}
    out["mixed_pcm"] = pcm_buf[:B, :L]
    got = eng.preprocess_pairs(_d(S), _d(Z), nvs, lengths=_d(lens), snr_db=_d(snr), out=out)
    torch.cuda.synchronize()
    for v in list(bufs.values()):
        assert torch.all(v[:B, n * 1600:] == SENT) and torch.all(v[B] == SENT)
    assert torch.all(pcm_buf[:B, L:] == SENT) and torch.all(pcm_buf[B] == SENT)
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in got)
    worst = worst_pcm = 0.0
    for i in range(B):
        want, want_pcm = _pair_oracle(S[i, :lens[i]], Z[i, :lens[i]], L, float(snr[i]), b)
        for g, w, name in zip((mixed[i], speech[i], noise[i]), want, ("mixed", "speech", "noise")):
            assert g.shape == w.shape, name
            err = float(np.max(np.abs(g - w)))
            worst = max(worst, err)
            assert err <= TOL_DB, (i, name, err)
        err = float(np.max(np.abs(pcm[i] - want_pcm)) / np.max(np.abs(want_pcm)))
        worst_pcm = max(worst_pcm, err)
        assert err <= TOL_PCM, (i, err)
    _worst(b, "preprocess_pairs_db", worst)
    _worst(b, "preprocess_pairs_pcm", worst_pcm)


def test_spectrogram_stft_magphase_floor_gather(bank):
    """spectrogram(..., stft=True) of ragged signals (zeros past each length), magphase of its STFT, and the SPEC -> slices
    floor_gather of the un-floored forward output."""
    eng, b = bank
    sr = b[0]
    L = 4 * eng.samples_per_slice + 77
    lens = np.array([L, L - 1000, L // 2], np.int32)
    B = len(lens)
    X = np.zeros((B, L), np.float32)
    for i, n in enumerate(lens):
        X[i, :n] = _signal(n, sr, 40 + i)
    spec, st = eng.spectrogram(_d(X), lengths=_d(lens), stft=True)
    mag, phase = eng.magphase(st)
    res = eng.forward_raw(_d(X), None, len_speech=_d(lens), layout=1, want=("speech",), mixed_pcm=False)
    n = res["T"] // 20
    sl = eng.floor_gather(res["speech"], res["max_key"], 0, n).cpu().numpy()
    spec, st, mag, phase = (t.cpu().numpy() for t in (spec, st, mag, phase))
    worst = [0.0, 0.0, 0.0]
    for i in range(B):
        x = X[i].astype(np.float64)
        want, _ = _spec(x, b)
        assert spec[i].shape == want.shape
        worst[0] = max(worst[0], float(np.max(np.abs(spec[i] - want))))
        D = O.stft(x, 640, 160)
        worst[1] = max(worst[1], float(np.max(np.abs(st[i].T - D)) / np.max(np.abs(D))))
        m, p = O.magphase(st[i].T.astype(np.complex128))
        assert np.max(np.abs(mag[i] - m)) <= 1e-6 * np.max(m)
        assert np.max(np.abs(phase[i] - p)) <= 2e-6
        ws = np.stack([want[:, 20 * j:20 * j + 20] for j in range(n)])
        worst[2] = max(worst[2], float(np.max(np.abs(sl[i] - ws))))
    assert worst[0] <= TOL_DB and worst[1] <= 2e-6 and worst[2] <= TOL_DB, worst
    _worst(b, "spectrogram_db", worst[0])
    _worst(b, "stft", worst[1])
    _worst(b, "floor_gather_db", worst[2])


def test_mix_pools_with_wrapping_offsets(bank):
    eng, b = bank
    sr = b[0]
    nvs = 4
    sp = [_signal(n, sr, 60 + k) for k, n in enumerate((13000, 9001, 16000))]
    nz = [(O.synth_noise(n, 70 + k) * (0.2, 3.0)[k % 2]).astype(np.float32) for k, n in enumerate((5000, 20000, 1121))]
    stride = max(len(c) for c in sp + nz) + 4
    spP = np.full((len(sp), stride), np.nan, np.float32)
    nzP = np.full((len(nz), stride), np.nan, np.float32)
    for k, c in enumerate(sp):
        spP[k, :len(c)] = c
    for k, c in enumerate(nz):
        nzP[k, :len(c)] = c
    si = np.array([0, 1, 2, 0, 2], np.int64)
    ni = np.array([0, 1, 2, 1, 0], np.int64)
    off = np.array([0, 19999, 560, 12345, 4999], np.int32)
    snr = np.array([-10.0, -2.5, 0.0, 4.0, 10.0], np.float32)
    got = eng.mix_pools(_d(spP), [len(c) for c in sp], _d(nzP), [len(c) for c in nz], _d(si), _d(ni), nvs, noise_offset=_d(off),
                        snr_db=_d(snr))
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in got)
    L = eng.samples_per_slice * nvs
    worst = worst_pcm = 0.0
    for r in range(len(si)):
        z = np.roll(nz[ni[r]], -int(off[r]))
        want, want_pcm = _pair_oracle(sp[si[r]], z, L, float(snr[r]), b)
        for g, w in zip((mixed[r], speech[r], noise[r]), want):
            assert g.shape == w.shape
            worst = max(worst, float(np.max(np.abs(g - w))))
        worst_pcm = max(worst_pcm, float(np.max(np.abs(pcm[r] - want_pcm)) / np.max(np.abs(want_pcm))))
    assert worst <= TOL_DB and worst_pcm <= TOL_PCM, (worst, worst_pcm)
    _worst(b, "mix_pools_db", worst)


def _inverse_oracle(mel, phase, b):
    """dp:99-116 with the bank's filterbank; mel (80, T) dB, phase (321, T)."""
    return O.reconstruct_signal_from_spectrogram(mel.astype(np.float64), phase, b[0], 640, 160, fmin=b[3], fmax=b[4]).get_data()


def _rel(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    return float(np.max(np.abs(got - want)) / np.max(np.abs(want)))


def test_inverse_forms_against_the_pinv_oracle(bank):
    """reconstruct (SLICES + mixture phase, ragged lengths), reconstruct_with_phase (explicit phase) and reconstruct_spec (SPEC +
    mixture phase), float32 and int16 out, every output row followed by a guard band and a spare row that must keep the sentinel."""
    eng, b = bank
    sr = b[0]
    rng = np.random.RandomState(int(b[3] + b[4]))
    B, n_sl = 3, 6
    T = 20 * n_sl
    L = 160 * (T + 2) + 37
    lens = np.array([L, L - 3000, L // 2 + 11], np.int32)
    pcm = np.zeros((B, L), np.float32)
    for i, n in enumerate(lens):
        pcm[i, :n] = _signal(n, sr, 80 + i)
    mel = (rng.rand(B, 80, T) * 40.0 - 60.0).astype(np.float32)
    slices = np.ascontiguousarray(mel.reshape(B, 80, n_sl, 20).transpose(0, 2, 1, 3))
    phase = np.exp(2j * np.pi * rng.rand(B, T, 321)).astype(np.complex64)
    out_len = 160 * (T - 1)
    d_pcm, d_mel, d_sl, d_lens, d_ph = _d(pcm), _d(mel), _d(slices), _d(lens), _d(phase)
    SENT, gap = -12345.0, 40

    def guarded(dtype, fill):
        return torch.full((B + 1, out_len + gap), fill, dtype=dtype, device="cuda")

    def intact(buf, fill):
        return bool(torch.all(buf[:B, out_len:] == fill)) and bool(torch.all(buf[B] == fill))

    buf = guarded(torch.float32, SENT)
    rec = eng.reconstruct(d_pcm, d_sl, lengths=d_lens, out=buf[:B, :out_len])
    assert intact(buf, SENT)
    buf16 = guarded(torch.int16, 12321)
    rec16 = eng.reconstruct(d_pcm, d_sl + 90.0, lengths=d_lens, out=buf16[:B, :out_len], out_dtype=torch.int16)
    assert intact(buf16, 12321)
    loud = eng.reconstruct(d_pcm, d_sl + 90.0, lengths=d_lens)
    assert torch.equal(rec16, torch.clamp(loud, -32768.0, 32767.0).to(torch.int32).to(torch.int16))

    bufe = guarded(torch.float32, SENT)
    ext = _inverse(eng, d_mel, bufe[:B], phase=d_ph)
    assert intact(bufe, SENT) and torch.equal(ext, eng.reconstruct_with_phase(d_mel, d_ph))
    bufe16 = guarded(torch.int16, 12321)
    ext16 = _inverse(eng, d_mel + 90.0, bufe16[:B], phase=d_ph)
    assert intact(bufe16, 12321)
    ext_loud = eng.reconstruct_with_phase(d_mel + 90.0, d_ph)
    assert torch.equal(ext16, torch.clamp(ext_loud, -32768.0, 32767.0).to(torch.int32).to(torch.int16))

    bufs = guarded(torch.float32, SENT)
    spec = _inverse(eng, d_mel, bufs[:B], pcm=d_pcm, lengths=d_lens)
    assert intact(bufs, SENT) and torch.equal(spec, eng.reconstruct_spec(d_pcm, d_mel, lengths=d_lens))

    # int16 out is checked above as the clipped, truncated float32 result; the loud float32 results go to the oracle here (a
    # 1-LSB bound would not hold: pinv of the ill-conditioned banks scales the output far past int16 range)
    rec, loud, spec, ext, ext_loud = (t.cpu().numpy() for t in (rec, loud, spec, ext, ext_loud))
    worst = {"reconstruct": 0.0, "reconstruct_spec": 0.0, "reconstruct_with_phase": 0.0}
    for i in range(B):
        x = pcm[i].astype(np.float64)
        _, mix_phase = O.magphase(O.stft(x, 640, 160))
        ph = phase[i].T.astype(np.complex128)
        for key, got, m, p in (("reconstruct", rec, mel, mix_phase[:, :T]), ("reconstruct", loud, mel + 90.0, mix_phase[:, :T]),
                               ("reconstruct_spec", spec, mel, mix_phase[:, :T]), ("reconstruct_with_phase", ext, mel, ph),
                               ("reconstruct_with_phase", ext_loud, mel + 90.0, ph)):
            worst[key] = max(worst[key], _rel(got[i], _inverse_oracle(m[i], p, b)))
    assert max(worst.values()) <= TOL_PCM, worst
    for k, v in worst.items():
        _worst(b, k, v)
