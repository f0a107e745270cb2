"""CPU checks of pooled-pair mixing (avse_mix_pooled): the forward stage code with a noise phase and separate speech / noise
rows, the statistics helper of the two noise regimes, and the host-side pairing draw of DynamicMixer.

Row semantics: speech s = the first Ls samples of its clip, noise n[i] = z[(off + i) mod Ln] for i < Ls, i.e. the reference's
preprocess_audio_pair (dp:119-139) run on (s, np.roll(z, -off)).  The emulator (tests/emul/avse_emul_pool.cpp) runs the SAME
__host__ __device__ stage code as the kernels, warp by warp.
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


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def emul():
    out_dir = os.path.join(ROOT, "build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libavse_emul_pool.so")
    srcs = [os.path.join(ROOT, "tests", "emul", "avse_emul_pool.cpp"), os.path.join(CSRC, "avse_tables.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so] + srcs)
    lib = ctypes.CDLL(so)
    vp, i32, f32, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double
    lib.emul_forward_pool.argtypes = [vp, i32, vp, i32, i32, i32, f32, f32, i32, vp, vp, vp, vp, vp, i32, f64, f64, i32]
    lib.emul_noise_sums.argtypes = [vp, i32, i32, i32, vp]
    return lib


@pytest.fixture(scope="module")
def eng_mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


def _clip_row(x, stride):
    """A pool row: the clip, then NaN -- anything read past the clip's length poisons the result."""
    row = np.full(stride, np.nan, np.float32)
    row[:len(x)] = x
    return row


def _run_pool(emul, s, z, off, nvs, snr, f2):
    L = 3200 * nvs
    ns = min(nvs, (1 + L // 160) // 20)
    zr = np.roll(z.astype(np.float64), -off) if len(z) else z.astype(np.float64)
    nfit = O.fit_noise_to_speech(O.AudioSignal(zr, SR), O.AudioSignal(s.astype(np.float64), SR)).get_data()
    fac = np.float32(O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nfit, SR), snr))
    gain = np.float32(float(fac) / 10.0 ** (-snr / 20.0))
    srow, zrow = _clip_row(s, len(s) + 37), _clip_row(z, len(z) + 41)
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    rc = emul.emul_forward_pool(_p(srow), len(s), _p(zrow), len(z), off, L, fac, gain, ns, _p(outs[0]), _p(outs[1]), _p(outs[2]),
                                _p(pcm), _p(mx), SR, 0.0, 8000.0, 1 if f2 else 0)
    assert rc == 1 or (f2 and rc in (0, 1))
    floored = [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)]
    ref = O.preprocess_audio_pair_signals(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(zr, SR), 200, nvs, FPS, snr_db=snr)
    return floored, pcm, ref


# (Ls, Ln, off) at nvs = 5 (L = 16 000).  F4 group g covers noise samples [640 g - 320, 640 g + 800): with a = 2 880 (g = 5)
# a wrap at i = Ln - off = a + 500 lies inside an interior group, one at a or a + 1 120 on a group edge.
POOL_CASES = [
    ("short_noise_off0", 16000, 5000, 0),
    ("short_noise_off1", 16000, 5000, 1),
    ("short_noise_off159", 16000, 5000, 159),
    ("short_noise_offLn-1", 16000, 5000, 4999),
    ("long_noise_off0", 16000, 20000, 0),
    ("long_noise_nowrap", 16000, 20000, 3000),
    ("long_noise_wrap", 16000, 20000, 19000),
    ("long_noise_offLn-1", 16000, 20000, 19999),
    ("wrap_inside_group", 16000, 12000, 12000 - 3380),
    ("wrap_at_group_start", 16000, 12000, 12000 - 2880),
    ("wrap_at_group_end", 16000, 12000, 12000 - 4000),
    ("noise_eq_speech_wrap", 16000, 16000, 7777),
    ("speech_shorter_than_L", 12000, 7000, 6000),
    ("speech_shorter_long_noise", 12000, 30000, 25000),
    ("speech_longer_than_L", 17000, 5000, 4321),
    ("speech_longer_long_noise", 17000, 40000, 33000),
]


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "f2"])
@pytest.mark.parametrize("case", POOL_CASES, ids=[c[0] for c in POOL_CASES])
def test_pooled_row_matches_oracle_on_rolled_noise(emul, case, f2):
    name, Ls, Ln, off = case
    seed = 300 + POOL_CASES.index(case)
    s = O.synth_speech(Ls, SR, seed).astype(np.float32)
    z = (O.synth_noise(Ln, seed) * (3.0 if Ln % 2 else 0.3)).astype(np.float32)
    snr = float(np.linspace(-10, 10, len(POOL_CASES))[POOL_CASES.index(case)])
    got, pcm, ref = _run_pool(emul, s, z, off, 5, snr, f2)
    for k, r in zip(range(3), (ref[1], ref[2], ref[0])):         # emulator (speech, noise, mixed), reference (mixed, speech, noise)
        assert np.all(np.isfinite(got[k])), k
        assert np.max(np.abs(got[k] - r)) <= TOL_DB, (k, np.max(np.abs(got[k] - r)))
    want = ref[3].get_data()
    assert np.max(np.abs(pcm - want)) <= TOL_PCM * np.max(np.abs(want))


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "f2"])
@pytest.mark.parametrize("off", [-1, 5000, 5001])
def test_invalid_phase_is_the_empty_pair(emul, off, f2):
    """off outside [0, Ln): nothing is read (both rows are all NaN here), every slice sits at the amin floor, PCM zeros."""
    L, ns = 16000, 5
    srow = np.full(16000, np.nan, np.float32)
    zrow = np.full(5000, np.nan, np.float32)
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.ones(L, np.float32)
    mx = np.zeros(3, np.float32)
    emul.emul_forward_pool(_p(srow), 16000, _p(zrow), 5000, off, L, 0.0, 0.0, ns, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm), _p(mx),
                           SR, 0.0, 8000.0, 1 if f2 else 0)
    for o in outs:
        assert np.all(o == np.float32(-100.0))
    assert np.all(pcm == 0.0)


SUM_SWEEP = [(1, 1, 0), (1, 7, 0), (3, 3, 0), (3, 3, 2), (5, 12, 4), (7, 7, 6), (160, 1000, 159), (1000, 1000, 999), (999, 1000, 1),
             (48000, 3000, 45000), (48000, 3000, 45001), (48000, 3000, 47999), (48000, 3000, 0), (4000, 3000, 1000), (4000, 3000, 1001),
             (2049, 48000, 2048), (640, 48000, 333), (12000, 16000, 8620), (16000, 16000, 7777), (5, 0, 3), (1, 0, 0)]


@pytest.mark.parametrize("Ln,Ls,off", SUM_SWEEP)
def test_noise_span_weights_reproduce_direct_sums(emul, Ln, Ls, off):
    """noise_span / noise_weight (the statistics pass's regimes: window ranges for Ln >= Ls, weighted period for Ln < Ls) give
    the sums of the materialised noise n[i] = z[(off + i) mod Ln], i < Ls."""
    z = np.random.RandomState(Ln * 7 + Ls + off).randn(Ln).astype(np.float32)
    out = np.zeros(2, np.float64)
    periodic = emul.emul_noise_sums(_p(z), Ln, Ls, off, _p(out))
    assert periodic == (1 if Ln < Ls else 0)
    n = z.astype(np.float64)[(off + np.arange(Ls)) % Ln]
    assert abs(out[0] - n.sum()) <= 1e-9 * max(1.0, np.abs(n).sum())
    assert abs(out[1] - (n * n).sum()) <= 1e-9 * max(1.0, (n * n).sum())


def test_draw_pairings_ranges_and_balance(eng_mod):
    g = torch.Generator()
    g.manual_seed(5)
    nl = torch.tensor([1, 7, 16000, 48000, 3], dtype=torch.int32)
    B, Ns = 1003, 10
    si, ni, off, snr = eng_mod.draw_pairings(g, B, Ns, nl, snr_db=(-10.0, 10.0))
    assert si.dtype == torch.int64 and ni.dtype == torch.int64 and off.dtype == torch.int32 and snr.dtype == torch.float32
    assert all(t.shape == (B,) for t in (si, ni, off, snr))
    counts = torch.bincount(si, minlength=Ns)
    assert int(counts.min()) == B // Ns and int(counts.max()) == -(-B // Ns)
    assert int(ni.min()) >= 0 and int(ni.max()) < nl.numel()
    assert len(set(ni.tolist())) == nl.numel()
    assert bool((off >= 0).all()) and bool((off.long() < nl.long()[ni]).all())
    assert int(off[ni == 0].abs().max()) == 0                       # a 1-sample clip has the single phase 0
    assert bool((snr >= -10.0).all()) and bool((snr < 10.0).all()) and float(snr.std()) > 3.0
    _, _, _, snr2 = eng_mod.draw_pairings(g, 500, Ns, nl, snr_db=[-5.0, 0.0, 5.0])
    assert set(snr2.tolist()) == {-5.0, 0.0, 5.0}
    _, _, _, snr3 = eng_mod.draw_pairings(g, 8, Ns, nl, snr_db=2.5)
    assert bool((snr3 == 2.5).all())


def test_draw_pairings_is_deterministic_per_seed(eng_mod):
    nl = torch.tensor([5000, 20000, 777], dtype=torch.int32)

    def epochs(seed):
        g = torch.Generator()
        g.manual_seed(seed)
        return [eng_mod.draw_pairings(g, 300, 40, nl) for _ in range(3)]

    a, b, c = epochs(11), epochs(11), epochs(12)
    for ea, eb in zip(a, b):
        for x, y in zip(ea, eb):
            assert torch.equal(x, y)
    assert not torch.equal(a[0][0], a[1][0])                         # a fresh permutation every epoch
    assert not all(torch.equal(x, y) for x, y in zip(a[0], c[0]))
    with pytest.raises(ValueError):
        eng_mod.draw_pairings(torch.Generator(), 4, 2, torch.tensor([10, 0], dtype=torch.int32))


def test_pack_clips_layout(eng_mod):
    clips = [np.arange(5, dtype=np.float32), np.zeros(0, np.float32), O.AudioSignal(np.ones(9), SR), torch.full((3,), 2.0)]
    pool, lens = eng_mod.pack_clips(clips, "cpu")
    assert pool.dtype == torch.float32 and pool.shape == (4, 12) and lens.dtype == torch.int32
    assert lens.tolist() == [5, 0, 9, 3]
    assert pool[0, :5].tolist() == [0, 1, 2, 3, 4] and float(pool[0, 5:].abs().sum()) == 0.0
    assert float(pool[2, :9].sum()) == 9.0 and float(pool[3, :3].sum()) == 6.0
    p16, _ = eng_mod.pack_clips([np.array([1, -2, 3], np.int16)], "cpu", dtype=torch.int16)
    assert p16.dtype == torch.int16 and p16.shape == (1, 4) and p16[0].tolist() == [1, -2, 3, 0]
    with pytest.raises(ValueError):
        eng_mod.pack_clips(clips, "cpu", allow_empty=False)
