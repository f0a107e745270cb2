"""Seeded synthetic cases shared by the golden generator, the emulation tests and the GPU parity tests."""
import numpy as np

from oracle import avse_oracle as O

SR, FPS, SLICE_MS = 16000, 25.0, 200

GOLDEN_CASES = [
    dict(name="pair_1s_snr0", n_s=16000, n_n=16000, nvs=5, snr=0.0, seed=101, scale=1.0),
    dict(name="pair_1s_snrm10_shortnoise", n_s=17000, n_n=5000, nvs=5, snr=-10.0, seed=102, scale=1.0),
    dict(name="pair_1s_zeropad_int16scale", n_s=12000, n_n=12000, nvs=5, snr=5.0, seed=103, scale=32767.0),
    dict(name="pair_3s_snr0", n_s=48000, n_n=48000, nvs=15, snr=0.0, seed=104, scale=1.0),
]


# Generic-kernel geometries at the frame rates real videos carry, as a video reader reports them (a float such as 30000/1001).
# n_fft: explicit SpectralEngine(..., n_fft=...) (fps is then only nominal); None: int(sr / fps) (dp:44).
# geo: (n_fft, hop, spss, n1, n2, n_inv, i1, i2) -- forward factor pair n_fft = n1 n2, librosa.istft's inferred size
# n_inv = 2 (bins - 1) = i1 i2 (avse_generic.h).
FRAME_RATES = [
    dict(name="44k1_29.97", sr=44100, fps=30000 / 1001, n_fft=None, geo=(1471, 367, 24, 1, 1471, 1470, 35, 42)),      # prime: n1 = 1
    dict(name="48k_29.97", sr=48000, fps=30000 / 1001, n_fft=None, geo=(1601, 400, 24, 1, 1601, 1600, 40, 40)),       # prime: n1 = 1
    dict(name="22k05_29.97", sr=22050, fps=30000 / 1001, n_fft=None, geo=(735, 183, 24, 21, 35, 734, 2, 367)),
    dict(name="16k_23.976", sr=16000, fps=24000 / 1001, n_fft=None, geo=(667, 166, 19, 23, 29, 666, 18, 37)),
    dict(name="16k_59.94", sr=16000, fps=60000 / 1001, n_fft=None, geo=(266, 66, 48, 14, 19, 266, 14, 19)),          # bank rank 68
    dict(name="16k_nfft160", sr=16000, fps=25.0, n_fft=160, geo=(160, 40, 80, 10, 16, 160, 10, 16)),                # 8 empty bands
    dict(name="48k_12", sr=48000, fps=12.0, n_fft=None, geo=(4000, 1000, 9, 50, 80, 4000, 50, 80)),
    dict(name="48k_nfft4096", sr=48000, fps=25.0, n_fft=4096, geo=(4096, 1024, 9, 64, 64, 4096, 64, 64)),            # largest n_fft
    dict(name="32k_29.97", sr=32000, fps=30000 / 1001, n_fft=None, geo=(1067, 266, 24, 11, 97, 1066, 26, 41)),
]


def frame_rate_fps(g):
    """A frame rate from which dp:44 derives the entry's n_fft (sr / n_fft for the explicit-n_fft entries)."""
    return g["fps"] if g["n_fft"] is None else g["sr"] / g["n_fft"]


def make_inputs(case):
    """float32 speech / noise exactly as the GPU path receives them."""
    s = (O.synth_speech(case["n_s"], SR, case["seed"]) * case["scale"]).astype(np.float32)
    n = (O.synth_noise(case["n_n"], case["seed"]) * case["scale"]).astype(np.float32)
    return s, n


def oracle_pair(case, s=None, n=None):
    """float64 oracle of preprocess_audio_pair (dp:119-139) + reconstruct_speech_signal (dp:60-74) on those inputs."""
    if s is None:
        s, n = make_inputs(case)
    sp = O.AudioSignal(s.astype(np.float64), SR)
    nz = O.AudioSignal(n.astype(np.float64), SR)
    mixed, speech, noise, mixed_sig = O.preprocess_audio_pair_signals(sp, nz, SLICE_MS, case["nvs"], FPS, snr_db=case["snr"])
    recon = O.reconstruct_speech_signal(O.AudioSignal(mixed_sig.get_data().copy(), SR), speech, FPS)
    return dict(mixed=mixed, speech=speech, noise=noise, mixed_pcm=mixed_sig.get_data(), recon=recon.get_data())


def fitted_noise(s, n):
    """dp:125-128 on the host: periodic tiling of the noise up to the speech length."""
    if len(n) < len(s):
        n = n[np.arange(len(s)) % len(n)]
    return np.ascontiguousarray(n[:len(s)])
