"""CPU checks of windowed pooled rows (avse_mix_pooled with speech_start) and of the host side of windowed training batches.

Row semantics: with a start a on a clip of Ls samples, row b is the reference's preprocess_audio_pair (dp:119-139) run on
the window s = clip[a : a + Lw], Lw = min(L, Ls - a), and the noise np.roll(z, -off): statistics over the window, reflect
padding mirrored inside it, PCM zero padded to L.  The emulator (tests/emul/avse_emul_windows.cpp) resolves every row through
pool_row, the same __host__ __device__ function the statistics pass and the forward kernels call, then runs the kernels'
stage code warp by warp.
"""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio-visual-speech-enhancement_b200", "csrc")
TOL_DB = 1e-3
TOL_PCM = 1e-4
SPS = 3200                      # samples per 200 ms slice at 16 kHz
NVS = 5                         # slices per row: L = 16 000
L = SPS * NVS


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def emul():
    out_dir = os.path.join(ROOT, "build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libavse_emul_windows.so")
    srcs = [os.path.join(ROOT, "tests", "emul", "avse_emul_windows.cpp"), os.path.join(CSRC, "avse_tables.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so] + srcs)
    lib = ctypes.CDLL(so)
    vp, i32, i64, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_double
    lib.emul_window_row.argtypes = [vp, i32, vp, i64, i64, vp, vp, i64, i64, i64, i64, i32, vp, i32, f64, i32,
                                    vp, vp, vp, vp, vp, vp, vp, i32]
    lib.emul_window_row.restype = i32
    return lib


@pytest.fixture(scope="module")
def eng_mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


def _pool(clips, dtype, pad):
    """A pool [n, stride]: each clip, then NaN (float32) -- a read past a clip's length poisons the result."""
    stride = max(len(c) for c in clips) + pad
    pool = np.full((len(clips), stride), np.nan if dtype == np.float32 else 0, dtype)
    for k, c in enumerate(clips):
        pool[k, :len(c)] = c
    return pool, np.array([len(c) for c in clips], np.int32)


def _run(emul, spool, slen, npool, nlen, si, ni, off, start, snr=0.0, f2=False):
    fmt = 0 if spool.dtype == np.float32 else 1
    ns = NVS
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    sums = np.zeros(4, np.float64)
    gains = np.zeros(2, np.float32)
    st = None if start is None else np.array([start], np.int32)
    rc = emul.emul_window_row(_p(spool), fmt, _p(slen), spool.shape[0], spool.shape[1], _p(npool), _p(nlen), npool.shape[0],
                              npool.shape[1], si, ni, off, _p(st), L, snr, ns, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm), _p(mx),
                              _p(sums), _p(gains), 1 if f2 else 0)
    assert rc in (0, 1), rc
    floored = [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)]
    return rc, floored, pcm, sums, gains


def _oracle(clip, a, z, off, snr):
    Lw = min(L, len(clip) - a)
    s = clip[a:a + Lw].astype(np.float64)
    zr = np.roll(z.astype(np.float64), -off)
    return O.preprocess_audio_pair_signals(O.AudioSignal(s, SR), O.AudioSignal(zr, SR), 200, NVS, FPS, snr_db=snr)


def _check(got, pcm, ref):
    for k, r in zip(range(3), (ref[1], ref[2], ref[0])):          # emulator (speech, noise, mixed), reference (mixed, speech, noise)
        assert np.all(np.isfinite(got[k])), k
        assert np.max(np.abs(got[k] - r)) <= TOL_DB, (k, np.max(np.abs(got[k] - r)))
    want = ref[3].get_data()
    assert np.max(np.abs(pcm - want)) <= TOL_PCM * np.max(np.abs(want))


LS_LONG = 5 * L + 777           # a clip several windows long, its length not on a slice boundary
# (name, clip length, start): starts off and on slice boundaries, windows cut short by the clip's end (Lw < L), the last sample
WINDOW_CASES = [
    ("a0", LS_LONG, 0),
    ("a1", LS_LONG, 1),
    ("a3", LS_LONG, 3),
    ("a159", LS_LONG, 159),
    ("a_sps", LS_LONG, SPS),
    ("a_sps_k_full", LS_LONG, SPS * 20),
    ("a_sps_k_short", LS_LONG, SPS * 24),          # Lw = 4 * SPS + 777 < L
    ("a_sps_k_tiny", LS_LONG, SPS * 25),           # Lw = 777
    ("a_Ls-3", LS_LONG, LS_LONG - 3),              # a three-sample window
    ("short_clip_a0", L - 3001, 0),                # Ls < L
    ("short_clip_a_sps", L - 3001, SPS),
    ("long_60s_a_sps_k", 60 * SR, SPS * 200),      # a 60 s clip under a 1 s window
    ("long_60s_last_full", 60 * SR, 60 * SR - L),
]


# (kernel, pool format): the 2-frame kernel serves float32 pools only (int16 needs the F4 tables)
KERNEL_FORMATS = [(False, "f32"), (True, "f32"), (False, "i16")]


@pytest.mark.parametrize("f2,fmt", KERNEL_FORMATS, ids=["f4-f32", "f2-f32", "f4-i16"])
@pytest.mark.parametrize("case", WINDOW_CASES, ids=[c[0] for c in WINDOW_CASES])
def test_windowed_row_matches_oracle(emul, case, f2, fmt):
    name, Ls, a = case
    seed = 700 + WINDOW_CASES.index(case)
    clip = O.synth_speech(Ls, SR, seed)
    z = O.synth_noise(7001, seed) * 2.0
    if fmt == "i16":
        clip = np.round(clip * 20000.0).astype(np.int16)
        z = np.round(z * 20000.0).astype(np.int16)
        spool, slen = _pool([clip[:100], clip], np.int16, 5)
        npool, nlen = _pool([z], np.int16, 3)
    else:
        clip = clip.astype(np.float32)
        z = z.astype(np.float32)
        spool, slen = _pool([clip[:100], clip], np.float32, 5)
        npool, nlen = _pool([z], np.float32, 3)
        # NaN before the window and after it: the kernels read neither clip[a - 1] nor clip[a + Lw]
        Lw = min(L, Ls - a)
        if a > 0:
            spool[1, a - 1] = np.nan
        if a + Lw < Ls:
            spool[1, a + Lw] = np.nan
    off = 1234
    snr = float(np.linspace(-8, 8, len(WINDOW_CASES))[WINDOW_CASES.index(case)])
    rc, got, pcm, sums, _ = _run(emul, spool, slen, npool, nlen, 1, 0, off, a, snr, f2)
    assert rc == 1
    _check(got, pcm, _oracle(clip, a, z, off, snr))


def test_last_sample_start_is_valid(emul):
    """a = Ls - 1 is a valid one-sample window; its noise window has zero variance, so the factor is NaN like numpy's."""
    clip = O.synth_speech(LS_LONG, SR, 3).astype(np.float32)
    z = O.synth_noise(7001, 3).astype(np.float32)
    spool, slen = _pool([clip], np.float32, 5)
    npool, nlen = _pool([z], np.float32, 3)
    rc, _, _, sums, gains = _run(emul, spool, slen, npool, nlen, 0, 0, 100, LS_LONG - 1)
    assert rc == 1 and np.isnan(gains[0])
    assert sums[0] == np.float64(clip[-1]) and sums[2] == np.float64(z[100])


def test_nan_around_window_is_never_read(emul):
    """The whole clip outside the window is NaN: any read of it (statistics, reflect padding, interior loads) poisons a slice."""
    Ls, a = 4 * L, 3 * SPS + 1
    Lw = min(L, Ls - a)
    clip = np.full(Ls, np.nan, np.float32)
    clip[a:a + Lw] = O.synth_speech(Lw, SR, 5)
    z = (O.synth_noise(20000, 5) * 3.0).astype(np.float32)
    spool, slen = _pool([clip], np.float32, 0)
    npool, nlen = _pool([z], np.float32, 1)
    for f2 in (False, True):
        rc, got, pcm, sums, _ = _run(emul, spool, slen, npool, nlen, 0, 0, 777, a, -3.0, f2)
        assert rc == 1 and np.all(np.isfinite(sums)) and np.all(np.isfinite(pcm))
        _check(got, pcm, _oracle(np.nan_to_num(clip), a, z, 777, -3.0))


@pytest.mark.parametrize("fmt", ["f32", "i16"])
@pytest.mark.parametrize("Ls,a,Ln,off", [(5 * L + 3, 0, 7001, 0), (5 * L + 3, 3, 7001, 7000), (5 * L + 3, 5 * L, 7001, 5),
                                          (5 * L + 3, 2 * SPS, 40000, 39000), (L - 1, SPS, 999, 500), (60 * SR, 295 * SPS, 3 * L, 2 * L), (60 * SR, 299 * SPS, 3 * L, 2 * L)])
def test_windowed_statistics_sums(emul, fmt, Ls, a, Ln, off):
    """The statistics pass's sums of a windowed row are numpy's sums of the window and its rolled noise."""
    rng = np.random.RandomState(Ls + a + Ln)
    dt = np.float32 if fmt == "f32" else np.int16
    clip = (rng.randn(Ls) * (0.3 if fmt == "f32" else 5000)).astype(dt)
    z = (rng.randn(Ln) * (0.1 if fmt == "f32" else 3000) + (0.01 if fmt == "f32" else 40)).astype(dt)
    spool, slen = _pool([clip], dt, 4)
    npool, nlen = _pool([z], dt, 4)
    rc, _, _, sums, gains = _run(emul, spool, slen, npool, nlen, 0, 0, off, a, 0.0, False)
    assert rc == 1
    Lw = min(L, Ls - a)
    s = clip[a:a + Lw].astype(np.float64)
    n = z.astype(np.float64)[(off + np.arange(Lw)) % Ln]
    for got, want in zip(sums, (s.sum(), (s * s).sum(), n.sum(), (n * n).sum())):
        assert abs(got - want) <= 1e-9 * max(1.0, abs(want), np.abs(s).sum() + np.abs(n).sum()), (got, want)
    f = np.sqrt(s.var() / n.var())
    assert abs(float(gains[0]) - f) <= 1e-6 * f


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "f2"])
@pytest.mark.parametrize("a", [-1, "Ls", "Ls+5"])
def test_invalid_start_is_the_empty_pair(emul, a, f2):
    """A start outside {0} u (0, Ls): nothing is read (the pools are all NaN here), every slice at the amin floor, PCM zeros."""
    Ls = 9000
    a = {"Ls": Ls, "Ls+5": Ls + 5}.get(a, a)
    spool = np.full((1, Ls + 16), np.nan, np.float32)
    npool = np.full((1, 5000), np.nan, np.float32)
    slen, nlen = np.array([Ls], np.int32), np.array([5000], np.int32)
    rc, got, pcm, sums, gains = _run(emul, spool, slen, npool, nlen, 0, 0, 0, a, 0.0, f2)
    assert rc == 0
    for o in got:
        assert np.all(o == np.float32(-100.0))
    assert np.all(pcm == 0.0) and np.all(sums == 0.0) and np.all(gains == 0.0)


def test_start_zero_on_empty_clip_is_valid(emul):
    """a == 0 on an empty speech clip stays what it is without windows: a valid empty pair (factor 0)."""
    spool = np.zeros((1, 8), np.float32)
    npool = (np.random.RandomState(1).randn(1, 5000)).astype(np.float32)
    slen, nlen = np.array([0], np.int32), np.array([5000], np.int32)
    rc, got, pcm, sums, gains = _run(emul, spool, slen, npool, nlen, 0, 0, 10, 0, 0.0, False)
    assert rc == 1 and gains[0] == 0.0
    for o in got:
        assert np.all(o == np.float32(-100.0))
    rc_bad, *_ = _run(emul, spool, slen, npool, nlen, 0, 0, 10, 1, 0.0, False)
    assert rc_bad == 0


def test_start_none_is_the_whole_clip(emul):
    """Without starts a row is the whole clip from sample 0: statistics over all Ls samples, even past L."""
    clip = O.synth_speech(2 * L, SR, 9).astype(np.float32)
    z = (O.synth_noise(3000, 9) * 2).astype(np.float32)
    spool, slen = _pool([clip], np.float32, 0)
    npool, nlen = _pool([z], np.float32, 0)
    rc, _, _, sums, _ = _run(emul, spool, slen, npool, nlen, 0, 0, 0, None, 0.0, False)
    assert rc == 1 and abs(sums[1] - float((clip.astype(np.float64) ** 2).sum())) <= 1e-9 * sums[1]


# ---- host side: DynamicMixer's window draw and sample_set's video index ----

class _Eng(object):
    """The engine attributes DynamicMixer reads, on the CPU (draw and video indexing need no device)."""
    device = torch.device("cpu")
    samples_per_slice = SPS


def _mixer(eng_mod, clip_slices, seed, ns=7):
    sp = torch.zeros((ns, 8))
    return eng_mod.DynamicMixer(_Eng(), sp, torch.full((ns,), 8, dtype=torch.int32), torch.zeros((3, 8)),
                                torch.tensor([8, 5, 3], dtype=torch.int32), n_video_slices=NVS, seed=seed, clip_slices=clip_slices)


CLIP_SLICES = [30, 5, 2, 0, 300, 6, 17]


def test_window_draw_keeps_the_pairing_sequence(eng_mod):
    """The (speech, noise, offset, SNR) draws of a seed are the same with and without windows, epoch after epoch."""
    plain, windowed = _mixer(eng_mod, None, 21), _mixer(eng_mod, CLIP_SLICES, 21)
    for _ in range(4):
        p, w = plain.draw(50), windowed.draw(50)
        assert len(p) == 4 and len(w) == 5
        for x, y in zip(p, w[:4]):
            assert torch.equal(x, y)


def test_window_starts_are_slice_aligned_and_in_range(eng_mod):
    m = _mixer(eng_mod, CLIP_SLICES, 3)
    cs = torch.tensor(CLIP_SLICES)
    seen = set()
    for _ in range(100):
        si, _, _, _, start = m.draw(70)
        assert start.dtype == torch.int32
        assert bool((start % SPS == 0).all())
        k = start.long() // SPS
        kmax = (cs[si] - NVS).clamp(min=0)
        assert bool((k >= 0).all()) and bool((k <= kmax).all())
        assert bool((k[cs[si] <= NVS] == 0).all())                  # a clip no longer than the window starts at 0
        seen |= set(k[si == 4].tolist())
    assert len(seen) > 250 and min(seen) == 0 and max(seen) == 295  # the 300-slice clip: 296 starts, every one drawn about 3 times


def test_window_draw_is_deterministic_per_seed(eng_mod):
    def epochs(seed):
        m = _mixer(eng_mod, CLIP_SLICES, seed)
        return [m.draw(40) for _ in range(3)]

    a, b, c = epochs(8), epochs(8), epochs(9)
    for ea, eb in zip(a, b):
        for x, y in zip(ea, eb):
            assert torch.equal(x, y)
    assert not torch.equal(a[0][4], c[0][4])


def test_mixer_refuses_bad_clip_slices(eng_mod):
    with pytest.raises(ValueError):
        _mixer(eng_mod, CLIP_SLICES[:-1], 0)
    with pytest.raises(ValueError):
        _mixer(eng_mod, [-1] + CLIP_SLICES[1:], 0)


def test_video_index_follows_make_sample_set_order(eng_mod):
    """Concatenated row r of a sample set is (sample b, slice j) in sample-major, slice-minor order, then permuted: its video
    slice is clip speech_index[b]'s slice k_b + j -- the same rows the oracle's make_sample_set picks from per-sample lists."""
    rng = np.random.RandomState(4)
    B, n, s_max, ns = 9, 5, 40, 6
    si = torch.tensor(rng.randint(0, ns, B), dtype=torch.int64)
    k = torch.tensor(rng.randint(0, 30, B), dtype=torch.int64)
    nb = torch.tensor([5, 0, 3, 5, 1, 5, 2, 0, 4], dtype=torch.int64)
    N = int(nb.sum())
    perm = torch.tensor(rng.permutation(N), dtype=torch.int64)
    got = eng_mod.video_slice_index(si, k, nb, n, s_max, perm)
    per_sample = [np.array([int(si[b]) * s_max + int(k[b]) + j for j in range(int(nb[b]))], np.int64).reshape(-1, 1) for b in range(B)]
    want, _, _ = O.make_sample_set(per_sample, per_sample, per_sample, perm.numpy())
    assert got.dtype == torch.int64 and got.tolist() == want.reshape(-1).tolist()
