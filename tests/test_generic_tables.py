"""CPU check of the generic-geometry host tables (csrc/avse_generic_tables.cpp) against the oracle and numpy:
librosa.filters.mel for any n_fft, np.linalg.pinv (one-sided Jacobi SVD), periodic Hann, twiddles, factor pairs."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests.cases import FRAME_RATES, frame_rate_fps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio-visual-speech-enhancement_b200", "csrc")


@pytest.fixture(scope="module")
def lib():
    out_dir = os.path.join(ROOT, "build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libavse_emul_generic.so")
    srcs = [os.path.join(ROOT, "tests", "emul", "avse_emul_generic.cpp"), os.path.join(CSRC, "avse_generic_tables.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so] + srcs)
    lb = ctypes.CDLL(so)
    lb.emul_generic_tables.argtypes = [ctypes.c_int] * 5 + [ctypes.c_double] * 2 + [ctypes.c_void_p] * 6
    return lb


def _tables(lib, sr, n_fft, n_mels=80, fmin=0.0, fmax=8000.0):
    hop = int(n_fft / 4)
    spss = max(1, int(int(0.2 * sr) / hop))
    bins = 1 + n_fft // 2
    geo = np.zeros(10, np.int32)
    fb = np.zeros((n_mels, bins), np.float64)
    pinv = np.zeros((bins, n_mels), np.float32)
    band = np.zeros((n_mels, 2), np.int32)
    win = np.zeros(n_fft, np.float32)
    tw = np.zeros((n_fft, 2), np.float64)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = lib.emul_generic_tables(sr, n_fft, hop, n_mels, spss, fmin, fmax, p(geo), p(fb), p(pinv), p(band), p(win), p(tw))
    assert rc == 0
    return geo, fb, pinv, band, win, tw


# n_fft of each FRAME_RATES entry as the reference derives it from the reader's float frame rate (dp:44) -> its geo row
FRAME_RATE_GEO = {(g["sr"], g["n_fft"] or int(float(g["sr"]) / g["fps"])): g["geo"] for g in FRAME_RATES}


@pytest.mark.parametrize("sr,n_fft", [(16000, 640), (16000, 320), (16000, 666), (16000, 533), (44100, 1764), (48000, 1920), (8000, 320),
                                      (16000, 1021)] + list(FRAME_RATE_GEO))
def test_generic_tables_match_oracle_and_numpy(lib, sr, n_fft):
    fmax = min(8000.0, sr / 2.0)
    geo, fb, pinv, band, win, tw = _tables(lib, sr, n_fft, fmax=fmax)
    bins = 1 + n_fft // 2
    assert list(geo[:5]) == [n_fft, n_fft // 4, bins, 80, max(1, int(0.2 * sr) // (n_fft // 4))]
    assert geo[5] * geo[6] == n_fft and geo[5] <= geo[6] and geo[7] == 2 * (bins - 1) and geo[8] * geo[9] == geo[7]
    if (sr, n_fft) in FRAME_RATE_GEO:
        want = FRAME_RATE_GEO[(sr, n_fft)]
        assert (geo[0], geo[1], geo[4]) == want[:3] and tuple(geo[5:10]) == want[3:], (list(geo), want)
    ref = O.mel_filterbank(sr, n_fft, 80, 0.0, fmax)
    assert np.max(np.abs(fb - ref)) < 1e-13
    # banded form covers exactly the non-zeros
    for m in range(80):
        nz = np.nonzero(fb[m])[0]
        if len(nz):
            assert band[m, 0] == nz[0] and band[m, 1] == nz[-1] - nz[0] + 1
        else:
            assert band[m, 1] == 0
    want = np.linalg.pinv(ref)
    scale = np.max(np.abs(want))
    assert np.max(np.abs(pinv - want)) <= 2e-6 * scale          # float32 rounding of a float64 result
    n = np.arange(n_fft)
    assert np.max(np.abs(win - (0.5 - 0.5 * np.cos(2 * np.pi * n / n_fft)))) < 1e-7
    a = -2.0 * np.pi * n / n_fft            # real arithmetic: numpy's complex division would add its own rounding
    assert np.max(np.abs(tw[:, 0] + 1j * tw[:, 1] - (np.cos(a) + 1j * np.sin(a)))) < 1e-15


def test_rank_deficient_filterbank_gives_numpy_pinv(lib):
    # 80 mel bands on 41 bins (n_fft 80): many empty / dependent filters; np.linalg.pinv drops the null space
    geo, fb, pinv, band, win, tw = _tables(lib, 16000, 80)
    ref = O.mel_filterbank(16000, 80, 80, 0.0, 8000.0)
    assert np.max(np.abs(fb - ref)) < 1e-13
    want = np.linalg.pinv(ref)
    assert np.max(np.abs(pinv - want)) <= 1e-5 * np.max(np.abs(want))
    assert (band[:, 1] == 0).any()


def test_bad_configurations_are_refused(lib):
    z = ctypes.c_void_p()
    geo = np.zeros(10, np.int32)
    p = geo.ctypes.data_as(ctypes.c_void_p)
    assert lib.emul_generic_tables(16000, 8192, 2048, 80, 1, 0.0, 8000.0, p, z, z, z, z, z) == 1     # n_fft too large
    assert lib.emul_generic_tables(16000, 640, 0, 80, 20, 0.0, 8000.0, p, z, z, z, z, z) == 1        # hop 0
    assert lib.emul_generic_tables(16000, 640, 160, 80, 20, 9000.0, 8000.0, p, z, z, z, z, z) == 1   # fmin > fmax


def _reference_counts(sr, fps, n_fft, nvs):
    """dp:36-50 integer arithmetic: (samples_per_slice, n_fft, hop, spss, frames T, int(T / spss)).  T is the oracle's
    1 + (len(np.pad(y, n_fft // 2, 'reflect')) - n_fft) // hop (O.stft); n_fft None: int(sr / fps) (dp:44)."""
    sps = int((200.0 / 1000) * sr)
    n_fft = int(float(sr) / fps) if n_fft is None else n_fft
    hop = int(n_fft / 4)
    spss = int(sps / hop)
    L = sps * nvs
    T = 1 + (L + 2 * (n_fft // 2) - n_fft) // hop
    return sps, n_fft, hop, spss, T, int(T / spss)


@pytest.mark.parametrize("g", FRAME_RATES, ids=[g["name"] for g in FRAME_RATES])
def test_geometry_and_slice_count_match_the_reference(g):
    """engine.geometry and engine.slice_count against the reference's arithmetic for n_video_slices 1 ... 400.  The slice count
    is int(T / spss) (dp:50), which exceeds n_video_slices once spss * hop < samples_per_slice; min(video, audio) (dp:164)
    is applied later.  O.stft's own frame count is checked on zero signals at every nvs up to 12, at 400 and around the
    first nvs where the count exceeds nvs (a full sweep through O.stft would take minutes at 48 kHz)."""
    eng = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    sr, fps, n_fft = g["sr"], g["fps"], g["n_fft"]
    sps, nf, hop, spss, _, _ = _reference_counts(sr, fps, n_fft, 1)
    assert (nf, hop, spss) == g["geo"][:3]
    assert eng.geometry(sr, frame_rate_fps(g), 200) == (sps, nf, hop, spss)
    if n_fft is None:
        assert eng.geometry(sr, fps, 200) == (sps, nf, hop, spss)
    first = None
    for nvs in range(1, 401):
        _, _, _, _, T, n = _reference_counts(sr, fps, n_fft, nvs)
        L = sps * nvs
        assert eng.frame_count(L, nf, hop) == T, nvs
        assert eng.slice_count(L, nf, hop, spss) == n, nvs
        if n != nvs and first is None:
            first = nvs
    assert first is None or spss * hop < sps
    checked = set(range(1, 13)) | {400} | ({first - 1, first, first + 1} if first else set())
    for nvs in sorted(checked):
        T = O.stft(np.zeros(sps * nvs), nf, hop).shape[1]
        assert T == _reference_counts(sr, fps, n_fft, nvs)[4], nvs
