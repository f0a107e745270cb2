"""SURVEY 8 rows a9 / a10: the mirror module is a drop-in for `import data_processor` in the reference's own entry points.

The reference's speech_enhancer.py `preprocess(args)` (se:17-28) and `predict(args)` (se:61-88) are restated call for call
by tests.dropin_support.CallSequenceDriver (se:25-28 / se:66-83), with stand-ins for the out-of-scope third-party imports
(mediaio.video_io, facedetection, the Keras network), and run on a synthetic dataset tree:

* `test_speech_enhancer_call_sequence_runs_on_the_mirror` (CPU): the product has no CPU path, so the engine behind the
  mirror is an oracle-backed test double: what this test pins is the module surface (names, positional signatures, return
  types, pickling, in-place mutation).
* `test_dropin_call_sequence_on_gpu` (-m gpu): the same call sequence on the REAL CUDA path, checked against the float64
  oracle.
"""
import importlib
import json
import os
import pickle

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests import dropin_support as D

TOL_DB, TOL_PCM = 1e-3, 1e-4
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _oracle_sample(sample):
    """float64 oracle of preprocess_sample's audio half (dp:160-174) for the files a Sample names."""
    sp = O.AudioSignal.from_wav_file(sample.speech_file_path)
    nz = O.AudioSignal.from_wav_file(sample.noise_file_path)
    with open(sample.video_file_path, "rb") as fd:
        frames = np.load(fd)
    n_video_slices = frames.shape[0] // 5
    mixed, speech, noise, sig = O.preprocess_audio_pair_signals(sp, nz, 200, n_video_slices, D.FPS, snr_db=0)
    n = min(n_video_slices, mixed.shape[0])
    video = np.stack([np.moveaxis(frames[5 * i:5 * i + 5], 0, 2) for i in range(n_video_slices)]).astype(np.float32)
    return dict(mixed=mixed[:n], speech=speech[:n], noise=noise[:n], pcm=sig.get_data(), video=video[:n], n=n)


def _check_samples(samples, tol_db, tol_pcm):
    assert sorted(os.path.basename(s.video_file_path) for s in samples) == ["clip%d.mpg" % i for i in range(len(D.CLIPS))]
    for s in samples:
        ref = _oracle_sample(s)
        assert s.speaker_id == "s1" and s.video_frame_rate == D.FPS
        assert s.mixed_spectrograms.shape == s.speech_spectrograms.shape == s.noise_spectrograms.shape == (ref["n"], 80, 20)
        assert s.video_samples.shape == (ref["n"], 128, 128, 5) and np.array_equal(s.video_samples, ref["video"])
        for got, want in ((s.mixed_spectrograms, ref["mixed"]), (s.speech_spectrograms, ref["speech"]), (s.noise_spectrograms, ref["noise"])):
            assert np.max(np.abs(got - want)) <= tol_db
        pcm = s.mixed_signal.get_data()
        assert pcm.shape == ref["pcm"].shape
        assert np.max(np.abs(pcm - ref["pcm"])) <= tol_pcm * np.max(np.abs(ref["pcm"]))


def _check_enhanced_wav(path, sample_before_predict, predicted, tol_lsb):
    """enhanced.wav == save_to_wav_file(reconstruct_speech_signal(mixed_signal, predicted, fps)) (dp:60-74, se:176-177)."""
    from scipy.io import wavfile
    sr, got = wavfile.read(path)
    mixed_sig = O.AudioSignal(np.asarray(sample_before_predict.mixed_signal.get_data(), dtype=np.float64), D.SR)
    ref = O.reconstruct_speech_signal(mixed_sig, np.asarray(predicted, dtype=np.float64), D.FPS).get_data()
    want = np.clip(ref, -32768, 32767).astype(np.int16)
    assert sr == D.SR and got.dtype == np.int16 and got.shape == want.shape
    assert np.max(np.abs(got.astype(np.int32) - want.astype(np.int32))) <= tol_lsb


def _run_call_sequence(dp, paths, tol_db, tol_pcm, tol_lsb, tol_video):
    """preprocess then predict of the reference's speech_enhancer.py against module `dp`: int16 WAVs on disk -> pickled
    Samples -> enhanced WAVs."""
    saved = D.install_stubs()
    try:
        drv = D.CallSequenceDriver(dp)
        blob = os.path.join(paths["base"], "d.pkl")
        drv.preprocess(paths, blob)
        with open(blob, "rb") as fd:
            samples = pickle.load(fd)
        _check_samples(samples, tol_db, tol_pcm)
        # what `train` leaves behind for predict (se:45-56): the normaliser built with the reference constructor and pickled
        video = np.concatenate([s.video_samples for s in samples], axis=0)
        norm_path = os.path.join(paths["base"], "normalization.pkl")
        with open(norm_path, "wb") as fd:
            pickle.dump(dp.VideoNormalizer(video), fd)
        outs = drv.predict(blob, norm_path, paths["base"])
        assert len(outs) == len(samples)
        for sample, predicted, wav in outs:
            _check_enhanced_wav(wav, sample, predicted, tol_lsb)
        # VideoNormalizer == numpy statistics (dp:201-212); normalised in place by predict (se:73)
        mean, std = np.mean(video, axis=(0, 3)), np.std(video, axis=(0, 3))
        first = [s for s in samples if s.video_file_path == outs[0][0].video_file_path][0]
        assert np.allclose(outs[0][0].video_samples, (first.video_samples - mean[None, :, :, None]) / std[None, :, :, None], atol=tol_video)
    finally:
        D.restore_modules(saved)


def test_speech_enhancer_call_sequence_runs_on_the_mirror(tmp_path, monkeypatch):
    dp = importlib.import_module(D.PKG + ".data_processor")
    eng_mod = importlib.import_module(D.PKG + ".engine")
    doubles = {}

    def get_engine(sample_rate=16000, video_frame_rate=25.0, slice_duration_ms=200, device=None):
        key = (sample_rate, video_frame_rate, slice_duration_ms)
        if key not in doubles:
            doubles[key] = D.OracleEngineDouble(sample_rate, video_frame_rate, slice_duration_ms)
        return doubles[key]

    monkeypatch.setattr(dp, "get_engine", get_engine)                      # no GPU here: oracle-backed engine double
    monkeypatch.setattr(eng_mod, "VideoNormalizer", D.NumpyVideoNormalizerDouble)
    paths = D.build_dataset(str(tmp_path))
    _run_call_sequence(dp, paths, tol_db=1e-4, tol_pcm=1e-6, tol_lsb=1, tol_video=2e-5)


def test_reference_call_forms_bind(tmp_path, monkeypatch):
    """The exact call forms the reference uses (dp:135-137, dp:160-162, dp:189, se:25, se:45, se:81) bind against the mirror's
    signatures: same positional order, same defaults."""
    import inspect
    dp = importlib.import_module(D.PKG + ".data_processor")
    sig = {n: inspect.signature(getattr(dp, n)) for n in (
        "preprocess_video_sample", "preprocess_audio_signal", "reconstruct_speech_signal", "signal_to_spectrogram",
        "reconstruct_signal_from_spectrogram", "preprocess_audio_pair", "preprocess_sample", "try_preprocess_sample", "preprocess_data")}
    sig["preprocess_data"].bind("entries", "noise_paths")                                   # se:25
    sig["preprocess_sample"].bind("entry", "noise")                                         # dp:182 via *sample_paths
    sig["try_preprocess_sample"].bind(("entry", "noise"))                                   # dp:195
    sig["preprocess_audio_pair"].bind("s.wav", "n.wav", 200, 15, 25.0)                      # dp:160-162
    sig["preprocess_audio_signal"].bind("sig", 200, 15, 25.0)                               # dp:135-137
    sig["signal_to_spectrogram"].bind("sig", 640, 160, mel=True, db=True)                   # dp:47, dp:64
    sig["reconstruct_signal_from_spectrogram"].bind("mag", "ph", 16000, 640, 160, mel=True, db=True)   # dp:72-74
    sig["reconstruct_speech_signal"].bind("mixed", "spec", 25.0)                            # se:81-83
    sig["preprocess_video_sample"].bind("v.mpg", 200)                                       # dp:159
    assert list(inspect.signature(dp.VideoNormalizer.__init__).parameters) == ["self", "video_samples"]   # se:45
    assert list(inspect.signature(dp.VideoNormalizer.normalize).parameters) == ["self", "video_samples"]  # se:46, se:73
    # the reference module's public names all exist on the mirror
    with open(os.path.join(GOLD, "reference_data_processor_names.json")) as fd:
        names = json.load(fd)["names"]
    assert len(names) == 11
    for name in names:
        assert hasattr(dp, name), name
    assert dp.Sample._fields == ("speaker_id", "video_file_path", "speech_file_path", "noise_file_path", "video_samples",
                                 "mixed_spectrograms", "speech_spectrograms", "noise_spectrograms", "mixed_signal", "video_frame_rate")


@pytest.mark.gpu
def test_dropin_call_sequence_on_gpu(tmp_path):
    """The real CUDA path under the reference's entry points: int16 WAVs on disk -> pickled Samples -> enhanced WAVs."""
    dp = importlib.import_module(D.PKG + ".data_processor")
    paths = D.build_dataset(str(tmp_path))
    _run_call_sequence(dp, paths, TOL_DB, TOL_PCM, tol_lsb=4, tol_video=2e-4)      # 1e-4 of int16 full scale = 3.3 LSB


@pytest.mark.gpu
def test_batch_driver_isolates_failures_per_sample(tmp_path):
    """dp:180-186: one bad sample (missing WAV, silent noise file, unreadable video) is dropped, the rest of its bucket
    survives -- also when the failure only shows up in the arithmetic (zero-variance noise -> non-finite SNR factor)."""
    from scipy.io import wavfile
    dp = importlib.import_module(D.PKG + ".data_processor")
    rng = np.random.RandomState(0)
    entries, noises = [], []
    for i in range(5):
        sp, nz = tmp_path / ("s%d.wav" % i), tmp_path / ("n%d.wav" % i)
        wavfile.write(str(sp), D.SR, (rng.randn(16000) * 3000).astype(np.int16))
        wavfile.write(str(nz), D.SR, (rng.randn(9000) * 1000).astype(np.int16))
        entries.append(D.AudioVisualEntry("spk", str(sp), "v%d" % i))
        noises.append(str(nz))
    wavfile.write(noises[1], D.SR, np.zeros(9000, np.int16))                  # silent noise: var == 0 -> inf factor
    entries[3] = D.AudioVisualEntry("spk", str(tmp_path / "missing.wav"), "v3")

    def video(path, slice_ms):
        if path == "v4":
            raise IOError("cannot decode")
        return np.zeros((5, 128, 128, 5), np.float32), D.FPS

    samples = dp.preprocess_data(entries, noises, video)
    assert [s.video_file_path for s in samples] == ["v0", "v2"]
    for s in samples:
        assert np.isfinite(s.mixed_spectrograms).all() and s.mixed_spectrograms.shape == (5, 80, 20)


@pytest.mark.gpu
def test_mel_converter_facade_and_magphase():
    """BASELINE.json's north_star names `MelConverter`; the reference snapshot has free functions instead (SURVEY section 0).  The
    façade routes to the same CUDA path; signal_to_spectrogram's phase is librosa.magphase (dp:80: 1 + 0j where D == 0), computed
    by avse_magphase."""
    dp = importlib.import_module(D.PKG + ".data_processor")
    compat = importlib.import_module(D.PKG + ".mediaio_compat")
    mc = dp.MelConverter(D.SR, D.FPS, 200)
    s = O.synth_speech(16000, D.SR, 21).astype(np.float32)
    s[6000:9000] = 0.0                                               # digital silence: exact zero frames -> phase 1 + 0j
    n = O.synth_noise(16000, 21).astype(np.float32)
    ref_db, ref_phase = O.signal_to_spectrogram(O.AudioSignal(s.astype(np.float64), D.SR), 640, 160)
    got_db = mc.signal_to_mel_spectrogram(compat.AudioSignal(s, D.SR))
    assert got_db.shape == ref_db.shape == (80, 101) and np.max(np.abs(got_db - ref_db)) <= TOL_DB
    mag, phase = dp.signal_to_spectrogram(compat.AudioSignal(s, D.SR), 640, 160)
    assert phase.shape == ref_phase.shape == (321, 101) and phase.dtype == np.complex64
    Dref = O.stft(s.astype(np.float64), 640, 160)
    zero = np.abs(Dref) == 0
    assert zero.any() and np.all(phase[zero] == 1.0 + 0.0j)
    strong = np.abs(Dref) > 1e-3 * np.abs(Dref).max()
    assert np.max(np.abs(phase[strong] - ref_phase[strong])) <= 2e-3
    assert np.max(np.abs(np.abs(phase[~zero]) - 1.0)) <= 1e-5
    slices = mc.signal_to_slices(compat.AudioSignal(s, D.SR), 5)
    want = O.preprocess_audio_signal(O.AudioSignal(s.astype(np.float64), D.SR), 200, 5, D.FPS)
    assert slices.shape == (5, 80, 20) and np.max(np.abs(slices - want)) <= TOL_DB
    mixed, speech, noise, sig = mc.mix_pair(compat.AudioSignal(s, D.SR), compat.AudioSignal(n, D.SR), 5, snr_db=5)
    r = O.preprocess_audio_pair_signals(O.AudioSignal(s.astype(np.float64), D.SR), O.AudioSignal(n.astype(np.float64), D.SR), 200, 5, D.FPS, snr_db=5)
    for a, b in zip((mixed, speech, noise), r[:3]):
        assert np.max(np.abs(a - b)) <= TOL_DB
    rec = mc.reconstruct_signal_from_mel_spectrogram(sig, speech)
    want = O.reconstruct_speech_signal(O.AudioSignal(sig.get_data().astype(np.float64), D.SR), speech.astype(np.float64), D.FPS).get_data()
    assert np.max(np.abs(rec.get_data() - want)) <= TOL_PCM * np.max(np.abs(sig.get_data()))
