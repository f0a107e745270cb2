"""Test scaffolding for the drop-in tests (tests/test_dropin_speech_enhancer.py): a synthetic GRID-like dataset tree on
disk, stand-ins for the third-party / out-of-scope modules that the mirror's video front end imports (mediaio.video_io,
facedetection) and for the reference's Keras network, the reference's speech_enhancer.py call sequence restated, and --
for the CPU-only run -- an engine double backed by the float64 oracle.
TEST INFRASTRUCTURE: nothing here is imported by the product."""
import os
import pickle
import sys
import types
from collections import namedtuple

import numpy as np

from oracle import avse_oracle as O

SR, FPS = 16000, 25.0
PKG = "audio-visual-speech-enhancement_b200"

# (name, speech samples, noise samples, video frames): ragged on purpose -- a noise shorter than the speech (in-kernel tiling,
# dp:125-128), a video shorter than the audio (n_slices = min(video, audio), dp:164), speech shorter than the video (dp:40)
CLIPS = [
    ("clip0", 48000, 60000, 75),
    ("clip1", 47000, 11000, 75),
    ("clip2", 50000, 48000, 70),
    ("clip3", 30000, 33000, 75),
]


def build_dataset(root):
    """<root>/data/<speaker>/{audio,video}/clipN.{wav,mpg} + <root>/noise/*.wav + <root>/base.  Returns a dict of paths."""
    from scipy.io import wavfile
    data, noise, base = os.path.join(root, "data"), os.path.join(root, "noise"), os.path.join(root, "base")
    for d in (os.path.join(data, "s1", "audio"), os.path.join(data, "s1", "video"), noise, base):
        os.makedirs(d)
    for i, (name, n_s, n_n, n_frames) in enumerate(CLIPS):
        s = np.round(O.synth_speech(n_s, SR, 300 + i) * 20000).astype(np.int16)
        n = np.round(O.synth_noise(n_n, 300 + i) * 32767 * (0.2 + 0.3 * i)).astype(np.int16)    # unrelated raw levels
        wavfile.write(os.path.join(data, "s1", "audio", name + ".wav"), SR, s)
        wavfile.write(os.path.join(noise, "noise%d.wav" % i), SR, n)
        frames = np.random.RandomState(i).randint(0, 256, size=(n_frames, 128, 128)).astype(np.uint8)
        with open(os.path.join(data, "s1", "video", name + ".mpg"), "wb") as fd:
            np.save(fd, frames)
    return dict(data=data, noise=noise, base=base)


# ---------------------------------------------------------------------------------------------
# stand-ins for out-of-scope third-party modules
# ---------------------------------------------------------------------------------------------
class _VideoFileReader(object):
    """mediaio.video_io.VideoFileReader surface used by dp:17-26 over the .npy payload written by build_dataset."""

    def __init__(self, path):
        self._path = path

    def __enter__(self):
        with open(self._path, "rb") as fd:
            self._frames = np.load(fd)
        return self

    def __exit__(self, *exc):
        return False

    def read_all_frames(self, convert_to_gray_scale=False):
        return self._frames

    def get_frame_count(self):
        return int(self._frames.shape[0])

    def get_frame_rate(self):
        return FPS


class _FaceDetector(object):
    def crop_mouth(self, frame, bounding_box_shape):
        assert frame.shape == (bounding_box_shape[1], bounding_box_shape[0])
        return frame


class FakeNetwork(object):
    """network.SpeechEnhancementNetwork surface used by se:64, se:75-78: a deterministic stand-in for the Keras model."""
    predictions = {}

    @staticmethod
    def load(model_cache_path):
        return FakeNetwork()

    def evaluate(self, mixed_spectrograms, video_samples, speech_spectrograms):
        return float(np.mean((np.asarray(mixed_spectrograms) - np.asarray(speech_spectrograms)) ** 2))

    def predict(self, mixed_spectrograms, video_samples):
        out = (np.asarray(mixed_spectrograms, dtype=np.float32) * 0.9 - 3.0).astype(np.float32)
        FakeNetwork.predictions[out.shape + (float(out.sum()),)] = out
        FakeNetwork.last = out
        return out


def install_stubs():
    """sys.modules entries for the third-party modules the mirror's preprocess_video_sample imports (dp:7, dp:9)."""
    mediaio = types.ModuleType("mediaio")
    video_io = types.ModuleType("mediaio.video_io")
    video_io.VideoFileReader = _VideoFileReader
    mediaio.video_io = video_io
    facedetection = types.ModuleType("facedetection")
    fd_mod = types.ModuleType("facedetection.face_detection")
    fd_mod.FaceDetector = _FaceDetector
    facedetection.face_detection = fd_mod
    mods = {"mediaio": mediaio, "mediaio.video_io": video_io, "facedetection": facedetection, "facedetection.face_detection": fd_mod}
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    return saved


def restore_modules(saved):
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v


# ---------------------------------------------------------------------------------------------
# the call sequence of se:17-28 / se:61-88, restated
# ---------------------------------------------------------------------------------------------
AudioVisualEntry = namedtuple("AudioVisualEntry", ["speaker_id", "audio_path", "video_path"])


class CallSequenceDriver(object):
    """What speech_enhancer.preprocess / predict ask of data_processor, call for call (se:25, se:27-28, se:66-67, se:73,
    se:81-83, se:176-177), with the asset layout reduced to two paths."""

    def __init__(self, dp_module):
        self.dp = dp_module

    def preprocess(self, paths, blob_path):
        import glob
        audio = sorted(glob.glob(os.path.join(paths["data"], "s1", "audio", "*.wav")))
        entries = [AudioVisualEntry("s1", a, glob.glob(os.path.splitext(a.replace("audio", "video"))[0] + ".*")[0]) for a in audio]
        noises = sorted(os.path.join(paths["noise"], f) for f in os.listdir(paths["noise"]))
        samples = self.dp.preprocess_data(entries, noises)                                   # se:25
        with open(blob_path, "wb") as fd:
            pickle.dump(samples, fd)                                                         # se:27-28

    def predict(self, blob_path, normalizer_path, out_dir):
        network = FakeNetwork.load(None)
        with open(normalizer_path, "rb") as fd:
            video_normalizer = pickle.load(fd)                                               # se:66-67
        with open(blob_path, "rb") as fd:
            samples = pickle.load(fd)
        outs = []
        for sample in samples:
            video_normalizer.normalize(sample.video_samples)                                 # se:73
            network.evaluate(sample.mixed_spectrograms, sample.video_samples, sample.speech_spectrograms)
            predicted = network.predict(sample.mixed_spectrograms, sample.video_samples)
            signal = self.dp.reconstruct_speech_signal(sample.mixed_signal, predicted, sample.video_frame_rate)   # se:81-83
            path = os.path.join(out_dir, os.path.splitext(os.path.basename(sample.video_file_path))[0] + "_enhanced.wav")
            signal.save_to_wav_file(path)                                                    # se:176-177
            outs.append((sample, predicted, path))
        return outs


# ---------------------------------------------------------------------------------------------
# CPU-only engine double (oracle-backed) so that the call sequence can be driven through the mirror where there is no
# GPU.  It implements exactly the engine surface data_processor.py touches.
# ---------------------------------------------------------------------------------------------
class OracleEngineDouble(object):
    import torch as _torch

    def __init__(self, sample_rate=16000, video_frame_rate=25.0, slice_duration_ms=200):
        self.sample_rate, self.video_frame_rate = int(sample_rate), float(video_frame_rate)
        self.samples_per_slice = int((float(slice_duration_ms) / 1000) * sample_rate)
        self.n_fft = int(float(sample_rate) / video_frame_rate)
        self.hop = int(self.n_fft / 4)
        self.spss = int(self.samples_per_slice / self.hop)
        self.n_mels, self.n_bins = 80, self.n_fft // 2 + 1
        self.device = self._torch.device("cpu")

    def n_frames(self, L):
        return 1 + L // self.hop

    def preprocess_pairs(self, speech, noise, n_video_slices, lengths=None, snr_db=None, out=None, noise_lengths=None, info=None):
        torch = self._torch
        B = speech.shape[0]
        res = [[], [], [], []]
        factors = []
        for u in range(B):
            n_s = int(lengths[u]) if lengths is not None else speech.shape[1]
            n_n = int(noise_lengths[u]) if noise_lengths is not None else n_s
            sp = O.AudioSignal(speech[u, :n_s].numpy().copy(), self.sample_rate)
            nz = O.AudioSignal(noise[u, :n_n].numpy().copy(), self.sample_rate)
            snr = float(snr_db[u]) if snr_db is not None else 0.0
            fitted = O.fit_noise_to_speech(O.AudioSignal(nz.get_data().copy(), self.sample_rate), sp)
            factors.append(O.AudioMixer.snr_factor(sp, fitted, snr))
            mixed, spc, nzc, sig = O.preprocess_audio_pair_signals(sp, nz, 1000.0 * self.samples_per_slice / self.sample_rate,
                                                                   int(n_video_slices), self.video_frame_rate, snr_db=snr)
            for lst, v in zip(res, (mixed, spc, nzc, sig.get_data())):
                lst.append(torch.from_numpy(np.asarray(v, dtype=np.float32)))
        if info is not None:
            info["factor"] = torch.tensor(factors, dtype=torch.float32)
        return tuple(torch.stack(r) for r in res)

    def reconstruct(self, mixed_pcm, mel_slices, lengths=None, out=None, work=None, out_dtype=None):
        torch = self._torch
        outs = []
        mixed_pcm = mixed_pcm.unsqueeze(0) if mixed_pcm.dim() == 1 else mixed_pcm
        mel_slices = mel_slices.unsqueeze(0) if mel_slices.dim() == 3 else mel_slices
        for u in range(mixed_pcm.shape[0]):
            sig = O.reconstruct_speech_signal(O.AudioSignal(mixed_pcm[u].numpy().astype(np.float64), self.sample_rate),
                                              mel_slices[u].numpy().astype(np.float64), self.video_frame_rate)
            outs.append(torch.from_numpy(sig.get_data().astype(np.float32)))
        return torch.stack(outs)

    def make_sample_set(self, mixed, speech, n_slices=None, permutation=None, generator=None, extra=None):
        m = mixed.reshape((-1,) + tuple(mixed.shape[2:]))
        s = speech.reshape((-1,) + tuple(speech.shape[2:]))
        return m[permutation], s[permutation], permutation


class NumpyVideoNormalizerDouble(object):
    """engine.VideoNormalizer surface used by data_processor.VideoNormalizer, in numpy (CPU-only test double)."""

    def __init__(self, engine, video_samples):
        import torch
        if video_samples is not None:
            v = np.asarray(video_samples, dtype=np.float32)
            self.mean_image = torch.from_numpy(np.mean(v, axis=(0, 3)))
            self.std_image = torch.from_numpy(np.std(v, axis=(0, 3)))

    @classmethod
    def from_images(cls, engine, mean_image, std_image):
        import torch
        self = cls(engine, None)
        self.mean_image, self.std_image = torch.from_numpy(np.asarray(mean_image)), torch.from_numpy(np.asarray(std_image))
        return self

    def normalize(self, video_samples):
        video_samples -= self.mean_image.numpy()[None, :, :, None]
        video_samples /= self.std_image.numpy()[None, :, :, None]
        return video_samples
