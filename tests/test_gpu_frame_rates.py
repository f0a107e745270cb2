"""GPU parity of the generic-geometry kernels at the frame rates real videos carry (tests.cases.FRAME_RATES).

A video reader reports its frame rate as a float such as 30000/1001, and the reference derives its STFT geometry from it
(n_fft = int(sr / fps), hop = int(n_fft / 4), spss = int(samples_per_slice / hop), dp:44-45, dp:49).  With common audio rates
that gives prime sizes (1471, 1601: the forward factor pair is (1, n_fft), a full n_fft-point DFT in the second stage), odd sizes
whose inverse runs at librosa.istft's inferred n_fft - 1 (735 -> 734 = 2 x 367, 1067 -> 1066 = 26 x 41), rank-deficient banks
(266: rank 68; n_fft 160: 8 empty bands, rank 55), the largest shared-memory footprint (4000, and 4096, the ceiling
build_generic accepts), and geometries with spss * hop < samples_per_slice, where int(T / spss) slices (dp:50) exceed
n_video_slices.  Every output is compared with the float64 oracle on the same inputs; tolerances are BASELINE.json's: 1e-3 dB on
log-mel, 1e-4 of the peak on PCM, 1 LSB of the clipped and truncated oracle on int16 PCM."""
import importlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import FRAME_RATES
from tests.test_gpu_inverse_forms import _inverse

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
PKG = "audio-visual-speech-enhancement_b200"
IDS = [g["name"] for g in FRAME_RATES]
BY_NAME = {g["name"]: g for g in FRAME_RATES}
_ENGINES = {}


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module(PKG + ".engine")


@pytest.fixture(params=FRAME_RATES, ids=IDS)
def geo(request, mod):
    g = request.param
    if g["name"] not in _ENGINES:
        _ENGINES[g["name"]] = mod.SpectralEngine(g["sr"], g["fps"], 200, device="cuda:0", n_fft=g["n_fft"])
    return _ENGINES[g["name"]], g


def _d(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _worst(g, entry, err):
    print("WORST %s %s %.3g" % (g["name"], entry, err))


def _spec(x, eng):
    """signal_to_spectrogram (dp:77-96) at the engine's geometry: floored dB (80, T) and the phase (bins, T)."""
    return O.signal_to_spectrogram(O.AudioSignal(np.asarray(x, np.float64), eng.sample_rate), eng.n_fft, eng.hop)


def _slices(mel, spss):
    """dp:49-51: int(T / spss) slices of spss frames."""
    return np.stack([mel[:, spss * i:spss * (i + 1)] for i in range(mel.shape[1] // spss)])


def _pair_oracle(s, z, L, snr, eng):
    """preprocess_audio_pair (dp:119-139): slices (mixed, speech, noise) and the mixture PCM padded / truncated to L.  z is the
    noise file (tiled to the speech length, dp:125-128).  An empty speech mixes two empty arrays: numpy's factor is nan, the
    result is silence, so the factor is taken as 0 there."""
    sp = O.AudioSignal(s.astype(np.float64), eng.sample_rate)
    nz = O.fit_noise_to_speech(O.AudioSignal(z.astype(np.float64), eng.sample_rate), sp)
    nz.amplify_by_factor(O.AudioMixer.snr_factor(sp, nz, snr) if len(s) else 0.0)
    mixed = sp.get_data() + nz.get_data()
    fit = lambda x: np.concatenate([x, np.zeros(max(0, L - len(x)))])[:L]
    return [_slices(_spec(fit(x), eng)[0], eng.spss) for x in (mixed, sp.get_data(), nz.get_data())], fit(mixed)


def _pcm_err(got, want):
    peak = np.max(np.abs(want))
    if peak == 0.0:
        assert np.all(got == 0.0)
        return 0.0
    return float(np.max(np.abs(got - want)) / peak)


def test_engine_geometry_and_filterbank(geo):
    eng, g = geo
    n_fft, hop, spss = g["geo"][:3]
    assert not eng.specialised
    assert (eng.n_fft, eng.hop, eng.spss, eng.n_bins, eng.n_mels) == (n_fft, hop, spss, 1 + n_fft // 2, 80)
    assert np.max(np.abs(eng.filterbank() - O.mel_filterbank(g["sr"], n_fft, 80, 0.0, 8000.0))) < 1e-13


# ---------------------------------------------------------------------------------------------------------------------------------
# preprocess_pairs: ragged batch, per-row SNR, float32 and int16, noise tiled in the kernels, strided outputs with guard bands
# ---------------------------------------------------------------------------------------------------------------------------------
def _ragged_batch(eng, i16):
    """Five rows: longer than L (truncated), 0.6 L, just above n_fft / 2, empty, L - hop - 1.  Each noise file is shorter than,
    as long as or longer than its speech; the row holds only the samples the kernels may read, the rest is poisoned (NaN, or
    30000 for int16).  Returns (S, Z, speech lengths, noise files, noise_lengths, snr, L, nvs)."""
    sr, n_fft, hop = eng.sample_rate, eng.n_fft, eng.hop
    nvs = 4
    L = eng.samples_per_slice * nvs
    W = L + 2 * hop + 5
    lens = [W, int(0.6 * L) + 3, n_fft // 2 + 3, 0, L - hop - 1]
    n_lens = [W + 100, int(0.25 * L) + 7, n_fft // 2 + 3, 500, 3 * hop + 11]
    scale = 12000.0 if i16 else 1.0
    dt = np.int16 if i16 else np.float32
    S = np.zeros((len(lens), W), dt)
    Z = np.full((len(lens), W), 30000 if i16 else np.nan, dt)
    files = []
    for i, (n, m) in enumerate(zip(lens, n_lens)):
        s = (O.synth_speech(n, sr, 10 + i) + 0.3 * O.synth_noise(n, 30 + i)) * scale if n else np.zeros(0)
        z = O.synth_noise(m, 20 + i) * scale * (0.5, 3.0, 0.05, 1.0, 0.2)[i]
        s, z = (np.round(s).astype(dt), np.round(z).astype(dt)) if i16 else (s.astype(dt), z.astype(dt))
        S[i, :n] = s
        Z[i, :min(n, m)] = z[:min(n, m)]
        files.append(z)
    nlens = np.array([min(n, m) for n, m in zip(lens, n_lens)], np.int32)
    snr = np.array([-10.0, 0.0, 10.0, 0.0, -10.0], np.float32)
    return S, Z, np.array(lens, np.int32), files, nlens, snr, L, nvs


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_preprocess_pairs_ragged_tiled_with_guard_bands(geo, i16):
    eng, g = geo
    S, Z, lens, files, nlens, snr, L, nvs = _ragged_batch(eng, i16)
    B = len(lens)
    n = eng.n_slices(L)
    per = n * 80 * eng.spss
    gap = 48
    bufs = {k: torch.full((B + 1, per + gap), float("nan"), device="cuda") for k in ("speech", "noise", "mixed")}
    pcm_buf = torch.full((B + 1, L + gap), float("nan"), device="cuda")
    out = {k: torch.as_strided(v, (B, n, 80, eng.spss), (per + gap, 80 * eng.spss, eng.spss, 1)) for k, v in bufs.items()}
    out["mixed_pcm"] = pcm_buf[:B, :L]
    got = eng.preprocess_pairs(_d(S), _d(Z), nvs, lengths=_d(lens), snr_db=_d(snr), out=out, noise_lengths=_d(nlens))
    torch.cuda.synchronize()
    for v in list(bufs.values()) + [pcm_buf]:
        assert bool(torch.isnan(v[:B, v.shape[1] - gap:]).all()) and bool(torch.isnan(v[B]).all())
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in got)
    worst = worst_pcm = 0.0
    for i in range(B):
        want, want_pcm = _pair_oracle(S[i, :lens[i]], files[i], L, float(snr[i]), eng)
        for gt, w, name in zip((mixed[i], speech[i], noise[i]), want, ("mixed", "speech", "noise")):
            assert gt.shape == w.shape == (n, 80, eng.spss), name
            err = float(np.max(np.abs(gt - w)))
            worst = max(worst, err)
            assert err <= TOL_DB, (i, name, err)
        err = _pcm_err(pcm[i], want_pcm)
        worst_pcm = max(worst_pcm, err)
        assert err <= TOL_PCM, (i, err)
    _worst(g, "preprocess_pairs_%s_db" % ("i16" if i16 else "f32"), worst)
    _worst(g, "preprocess_pairs_%s_pcm" % ("i16" if i16 else "f32"), worst_pcm)


def test_each_utterance_alone_is_bit_identical_to_the_batch(geo):
    """The generic kernels run one CTA per (frame, utterance): an utterance's results cannot depend on its neighbours."""
    eng, g = geo
    S, Z, lens, _, nlens, snr, L, nvs = _ragged_batch(eng, False)
    dS, dZ, dl, dn, ds = _d(S), _d(Z), _d(lens), _d(nlens), _d(snr)
    whole = eng.preprocess_pairs(dS, dZ, nvs, lengths=dl, snr_db=ds, noise_lengths=dn)
    rec = eng.reconstruct(whole[3], whole[1] + 60.0, lengths=dl, out_dtype=torch.int16)
    rec_f = eng.reconstruct(whole[3], whole[1], lengths=dl)
    for i in range(S.shape[0]):
        r = slice(i, i + 1)
        part = eng.preprocess_pairs(dS[r], dZ[r], nvs, lengths=dl[r], snr_db=ds[r], noise_lengths=dn[r])
        for a, b in zip(part, whole):
            assert torch.equal(a[0], b[i]), i
        assert torch.equal(eng.reconstruct(whole[3][r], whole[1][r] + 60.0, lengths=dl[r], out_dtype=torch.int16)[0], rec[i]), i
        assert torch.equal(eng.reconstruct(whole[3][r], whole[1][r], lengths=dl[r])[0], rec_f[i]), i


# ---------------------------------------------------------------------------------------------------------------------------------
# spectrogram(..., stft=True), magphase, floor_gather
# ---------------------------------------------------------------------------------------------------------------------------------
def test_spectrogram_stft_magphase_floor_gather(geo):
    eng, g = geo
    sr, n_fft, hop, spss = eng.sample_rate, eng.n_fft, eng.hop, eng.spss
    L = 4 * eng.samples_per_slice + 77
    lens = np.array([L, L - 5 * hop - 3, n_fft // 2 + 3], np.int32)
    B = len(lens)
    X = np.zeros((B, L), np.float32)
    for i, n in enumerate(lens):
        X[i, :n] = O.synth_speech(n, sr, 40 + i) + 0.3 * O.synth_noise(n, 50 + i)
    spec, st = eng.spectrogram(_d(X), lengths=_d(lens), stft=True)
    mag, phase = eng.magphase(st)
    res = eng.forward_raw(_d(X), None, len_speech=_d(lens), layout=1, want=("speech",), mixed_pcm=False)
    n = res["T"] // spss
    assert n == eng.n_slices(L)
    sl = eng.floor_gather(res["speech"], res["max_key"], 0, n).cpu().numpy()
    spec, st, mag, phase = (t.cpu().numpy() for t in (spec, st, mag, phase))
    worst = [0.0, 0.0, 0.0]
    for i in range(B):
        x = X[i].astype(np.float64)
        want, _ = _spec(x, eng)
        assert spec[i].shape == want.shape
        worst[0] = max(worst[0], float(np.max(np.abs(spec[i] - want))))
        D = O.stft(x, n_fft, hop)
        assert st[i].T.shape == D.shape
        worst[1] = max(worst[1], float(np.max(np.abs(st[i].T - D)) / np.max(np.abs(D))))
        m, p = O.magphase(st[i].T.astype(np.complex128))
        assert np.max(np.abs(mag[i] - m)) <= 1e-6 * np.max(m)
        assert np.max(np.abs(phase[i] - p)) <= 2e-6
        worst[2] = max(worst[2], float(np.max(np.abs(sl[i] - _slices(want, spss)))))
    assert worst[0] <= TOL_DB and worst[1] <= 2e-6 and worst[2] <= TOL_DB, worst
    _worst(g, "spectrogram_db", worst[0])
    _worst(g, "stft", worst[1])
    _worst(g, "floor_gather_db", worst[2])


# ---------------------------------------------------------------------------------------------------------------------------------
# mix_pools: offsets 0, 1, Ln - 1 and a wrap inside the window, against the oracle on np.roll(z, -off)
# ---------------------------------------------------------------------------------------------------------------------------------
def test_mix_pools_offsets_and_wraps(geo):
    eng, g = geo
    sr, n_fft, hop = eng.sample_rate, eng.n_fft, eng.hop
    nvs = 4
    L = eng.samples_per_slice * nvs
    sp = [(O.synth_speech(n, sr, 60 + k) + 0.3 * O.synth_noise(n, 65 + k)).astype(np.float32)
          for k, n in enumerate((int(0.8 * L), L + 2 * hop, n_fft // 2 + 5))]
    nz = [(O.synth_noise(n, 70 + k) * (0.2, 3.0, 1.0)[k]).astype(np.float32) for k, n in enumerate((int(0.3 * L) + 1, int(1.5 * L), 2 * n_fft + 3))]
    stride = (max(len(c) for c in sp + nz) + 3) // 4 * 4 + 4
    spP = np.full((len(sp), stride), np.nan, np.float32)
    nzP = np.full((len(nz), stride), np.nan, np.float32)
    for k, c in enumerate(sp):
        spP[k, :len(c)] = c
    for k, c in enumerate(nz):
        nzP[k, :len(c)] = c
    Ln = [len(c) for c in nz]
    si = np.array([0, 1, 0, 1, 2, 0, 1], np.int64)
    ni = np.array([0, 1, 1, 0, 2, 2, 1], np.int64)
    off = np.array([0, 1, Ln[1] - 1, Ln[0] // 2, Ln[2] - 1, 1, Ln[1] - L // 3], np.int32)     # the last wraps inside the window
    snr = np.array([-10.0, -5.0, 0.0, 3.0, 10.0, 0.0, 7.0], np.float32)
    got = eng.mix_pools(_d(spP), [len(c) for c in sp], _d(nzP), Ln, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr))
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in got)
    assert mixed.shape == (len(si), eng.n_slices(L), 80, eng.spss)
    worst = worst_pcm = 0.0
    for r in range(len(si)):
        want, want_pcm = _pair_oracle(sp[si[r]], np.roll(nz[ni[r]], -int(off[r])), L, float(snr[r]), eng)
        for gt, w in zip((mixed[r], speech[r], noise[r]), want):
            assert gt.shape == w.shape
            worst = max(worst, float(np.max(np.abs(gt - w))))
        worst_pcm = max(worst_pcm, _pcm_err(pcm[r], want_pcm))
    assert worst <= TOL_DB and worst_pcm <= TOL_PCM, (worst, worst_pcm)
    _worst(g, "mix_pools_db", worst)
    _worst(g, "mix_pools_pcm", worst_pcm)


# ---------------------------------------------------------------------------------------------------------------------------------
# the three inverse forms, float32 and int16 out, guard bands
# ---------------------------------------------------------------------------------------------------------------------------------
def test_inverse_forms_float32_and_int16(geo):
    """reconstruct (SLICES + mixture phase, ragged lengths), reconstruct_spec (SPEC + mixture phase) and reconstruct_with_phase
    (explicit phase) in float32 against the oracle, and in int16 -- at a level where the loudest samples clip -- within 1 LSB of
    the clipped, truncated oracle; every output row is followed by a guard band and a spare row that must keep the sentinel."""
    eng, g = geo
    sr, n_fft, hop, spss, bins = eng.sample_rate, eng.n_fft, eng.hop, eng.spss, eng.n_bins
    rng = np.random.RandomState(g["sr"] + g["geo"][0])
    B, n_sl = 3, 3
    T = spss * n_sl
    L = hop * (T + 2) + 37
    lens = np.array([L, L - 7 * hop, L // 2 + 11], np.int32)
    pcm = np.zeros((B, L), np.float32)
    for i, n in enumerate(lens):
        pcm[i, :n] = O.synth_speech(n, sr, 80 + i) + 0.3 * O.synth_noise(n, 90 + i)
    mel = (rng.rand(B, 80, T) * 40.0 - 60.0).astype(np.float32)
    phase = np.exp(2j * np.pi * rng.rand(B, T, bins)).astype(np.complex64)
    mix_phase = []
    for i in range(B):
        x = pcm[i].astype(np.float64)
        x[lens[i]:] = 0.0
        mix_phase.append(O.magphase(O.stft(x, n_fft, hop))[1][:, :T])
    want = {}
    for i in range(B):
        for form, ph in (("mixture", mix_phase[i]), ("explicit", phase[i].T.astype(np.complex128))):
            want[form, i] = O.reconstruct_signal_from_spectrogram(mel[i].astype(np.float64), ph, sr, n_fft, hop).get_data()
    # the int16 runs add the same gain in dB to every row: the loudest oracle sample lands at 1.5x full scale
    peak = max(np.max(np.abs(w)) for w in want.values())
    gain_db = float(20.0 * np.log10(1.5 * 32767.0 / peak))
    out_len = hop * (T - 1)
    slices = lambda m: np.ascontiguousarray(m.reshape(B, 80, n_sl, spss).transpose(0, 2, 1, 3))
    d_pcm, d_lens, d_ph = _d(pcm), _d(lens), _d(phase)
    SENT, gap = -12345.0, 40

    def guarded(dtype, fill):
        return torch.full((B + 1, out_len + gap), fill, dtype=dtype, device="cuda")

    def intact(buf, fill):
        return bool(torch.all(buf[:B, out_len:] == fill)) and bool(torch.all(buf[B] == fill))

    res = {}
    for i16 in (False, True):
        m = mel + (gain_db if i16 else 0.0)
        dt, fill = (torch.int16, 12321) if i16 else (torch.float32, SENT)
        buf = guarded(dt, fill)
        res["reconstruct", i16] = eng.reconstruct(d_pcm, _d(slices(m)), lengths=d_lens, out=buf[:B, :out_len], out_dtype=dt)
        assert intact(buf, fill)
        buf = guarded(dt, fill)
        res["reconstruct_spec", i16] = _inverse(eng, _d(m), buf[:B], pcm=d_pcm, lengths=d_lens)
        assert intact(buf, fill)
        buf = guarded(dt, fill)
        res["reconstruct_with_phase", i16] = _inverse(eng, _d(m), buf[:B], phase=d_ph)
        assert intact(buf, fill)
    assert torch.equal(res["reconstruct_spec", False], eng.reconstruct_spec(d_pcm, _d(mel), lengths=d_lens))
    assert torch.equal(res["reconstruct_with_phase", False], eng.reconstruct_with_phase(_d(mel), d_ph))
    gain = 10.0 ** (gain_db / 20.0)
    clipped = 0
    for name, form in (("reconstruct", "mixture"), ("reconstruct_spec", "mixture"), ("reconstruct_with_phase", "explicit")):
        f32, i16 = res[name, False].cpu().numpy(), res[name, True].cpu().numpy().astype(np.int32)
        worst = worst_lsb = 0
        for i in range(B):
            w = want[form, i]
            assert f32[i].shape == w.shape and np.isfinite(f32[i]).all()
            worst = max(worst, float(np.max(np.abs(f32[i] - w)) / np.max(np.abs(w))))
            w16 = np.clip(gain * w, -32768, 32767).astype(np.int16).astype(np.int32)
            clipped += int(np.sum(np.abs(gain * w) > 32767.0))
            worst_lsb = max(worst_lsb, int(np.max(np.abs(i16[i] - w16))))
        assert worst <= TOL_PCM and worst_lsb <= 1, (name, worst, worst_lsb)
        _worst(g, name, worst)
        _worst(g, name + "_int16_lsb", worst_lsb)
    assert clipped > 0


# ---------------------------------------------------------------------------------------------------------------------------------
# the mirror above the slice-count threshold: preprocess_audio_pair returns int(T / spss) slices, Sample keeps min(video, audio)
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,nvs", [("16k_23.976", 66), ("48k_12", 15)])
def test_mirror_slice_count_above_the_threshold(name, nvs, tmp_path):
    from scipy.io import wavfile
    dp = importlib.import_module(PKG + ".data_processor")
    g = BY_NAME[name]
    sr, fps = g["sr"], g["fps"]
    sps = int(0.2 * sr)
    L = sps * nvs
    s16 = np.round((O.synth_speech(L - 1234, sr, 7) + 0.2 * O.synth_noise(L - 1234, 8)) * 15000).astype(np.int16)
    z16 = np.round(O.synth_noise(3 * sps + 17, 9) * 8000).astype(np.int16)
    ref = O.preprocess_audio_pair_signals(O.AudioSignal(s16.astype(np.float64), sr), O.AudioSignal(z16.astype(np.float64), sr), 200, nvs,
                                          fps)
    n_audio = ref[0].shape[0]
    assert n_audio == nvs + 1                  # int(T / spss) (dp:50) exceeds n_video_slices here

    def check(got, n):
        for gt, w, what in zip(got[:3], ref[:3], ("mixed", "speech", "noise")):
            assert gt.shape == (n, 80, g["geo"][2]), what
            err = float(np.max(np.abs(gt - w[:n])))
            assert err <= TOL_DB, (what, err)
        return err

    got = dp.preprocess_audio_pair_signals(dp.AudioSignal(s16.copy(), sr), dp.AudioSignal(z16.copy(), sr), 200, nvs, fps)
    check(got, n_audio)
    assert _pcm_err(got[3].get_data(), ref[3].get_data()) <= TOL_PCM

    sp_path, nz_path = str(tmp_path / "speech.wav"), str(tmp_path / "noise.wav")
    wavfile.write(sp_path, sr, s16)
    wavfile.write(nz_path, sr, z16)
    Entry = namedtuple("Entry", ["speaker_id", "audio_path", "video_path"])
    video = np.random.RandomState(1).rand(nvs, 4, 4, 5).astype(np.float32)
    samples = dp.preprocess_data([Entry("s1", sp_path, "v.mp4")], [nz_path], video_preprocessor=lambda path, ms: (video, fps))
    assert len(samples) == 1
    smp = samples[0]
    assert smp.video_samples.shape[0] == nvs          # dp:164: min(video, audio)
    check((smp.mixed_spectrograms, smp.speech_spectrograms, smp.noise_spectrograms), nvs)
