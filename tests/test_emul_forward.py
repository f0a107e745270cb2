"""CPU-side check of the kernel's warp-stage code (csrc/avse_fwd_stages.cuh, avse_dft.cuh, avse_tables.cpp).

tests/emul/avse_emul.cpp compiles the SAME __host__ __device__ stage functions with g++ and runs a
warp as a loop over lanes, so index maps / twiddles / tables / float32 arithmetic are validated
against the float64 oracle and the golden vectors without a GPU.  (The emulation is test
infrastructure; the product has no CPU path.)
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests.cases import GOLDEN_CASES, SR, make_inputs, oracle_pair, fitted_noise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio-visual-speech-enhancement_b200", "csrc")
GOLD = os.path.join(ROOT, "tests", "golden")
TOL_DB = 1e-3      # BASELINE.json north_star: <= 1e-3 dB on log-mel
TOL_PCM = 1e-4     # <= 1e-4 of full scale on PCM


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="session")
def emul():
    out_dir = os.path.join(ROOT, "build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libavse_emul.so")
    srcs = [os.path.join(ROOT, "tests", "emul", "avse_emul.cpp"), os.path.join(ROOT, "tests", "emul", "avse_emul_inv.cpp"),
            os.path.join(CSRC, "avse_tables.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so] + srcs)
    lib = ctypes.CDLL(so)
    lib.emul_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                 ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_double]
    ex = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_int,
          ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
          ctypes.c_int, ctypes.c_double, ctypes.c_double]
    lib.emul_forward4_ex.argtypes = ex
    lib.emul_forward_mode_ex.argtypes = ex + [ctypes.c_int]
    lib.emul_filterbank.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_void_p]
    lib.emul_tables_info.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return lib


def test_fft640_codelets(emul):
    rng = np.random.RandomState(0)
    for _ in range(3):
        re = rng.randn(640).astype(np.float32)
        im = rng.randn(640).astype(np.float32)
        ore = np.zeros(640, np.float32)
        oim = np.zeros(640, np.float32)
        assert emul.emul_fft640(_p(re), _p(im), _p(ore), _p(oim)) == 0
        ref = np.fft.fft(re.astype(np.float64) + 1j * im.astype(np.float64))
        assert np.max(np.abs((ore + 1j * oim) - ref)) < 4e-7 * np.max(np.abs(ref))


def test_filterbank_and_tridiagonal_tables(emul):
    fb = np.zeros((80, 321))
    assert emul.emul_filterbank(SR, 0.0, 8000.0, _p(fb)) == 0
    ref = O.mel_filterbank(SR, 640, 80, 0.0, 8000.0)
    assert np.max(np.abs(fb - ref)) < 1e-14
    lo = np.zeros(80, np.int32)
    width = np.zeros(80, np.int32)
    tri = np.zeros(240, np.float32)
    assert emul.emul_tables_info(SR, 0.0, 8000.0, _p(lo), _p(width), _p(tri)) == 0
    assert width.max() <= 24 and width.min() >= 2 and width.sum() == 625
    # Thomas factors solve (F F^T) y = a like np.linalg.pinv (dp:112)
    w, ipiv, sup = tri[:80].astype(np.float64), tri[80:160].astype(np.float64), tri[160:].astype(np.float64)
    a = np.abs(np.random.RandomState(1).randn(80))
    d = a.copy()
    for i in range(1, 80):
        d[i] -= w[i] * d[i - 1]
    y = np.zeros(80)
    y[79] = d[79] * ipiv[79]
    for i in range(78, -1, -1):
        y[i] = (d[i] - sup[i] * y[i + 1]) * ipiv[i]
    lin = ref.T @ y
    assert np.max(np.abs(lin - np.linalg.pinv(ref) @ a)) < 1e-5 * np.max(np.abs(lin))
    # unsupported configuration is refused, not silently mis-computed
    assert emul.emul_filterbank(SR, 0.0, 100.0, _p(fb)) == -2


def _run_emul(emul, case):
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    L = 3200 * case["nvs"]
    fac = O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nf.astype(np.float64), SR), case["snr"])
    ns = min(case["nvs"], (1 + L // 160) // 20)
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    rc = emul.emul_forward(_p(s), _p(nf), L, len(s), len(s), fac, 0, ns, 0, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm), _p(mx),
                           SR, 0.0, 8000.0)
    assert rc == 0
    floored = [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)]
    return dict(speech=floored[0], noise=floored[1], mixed=floored[2], mixed_pcm=pcm)


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
def test_stage_code_matches_oracle_and_golden(emul, case):
    got = _run_emul(emul, case)
    ref = oracle_pair(case)
    gold = np.load(os.path.join(GOLD, case["name"] + ".npz"))
    for k in ("mixed", "speech", "noise"):
        assert np.max(np.abs(got[k] - ref[k])) <= TOL_DB, k
        assert np.max(np.abs(got[k] - gold[k])) <= TOL_DB + 2e-5, k
    scale = np.max(np.abs(ref["mixed_pcm"]))
    assert np.max(np.abs(got["mixed_pcm"] - ref["mixed_pcm"])) <= TOL_PCM * scale


def test_single_signal_spec_layout(emul):
    # signal_to_spectrogram on one signal of arbitrary length (dp:77-96), SPEC layout [80][ld_t]
    n = 5000
    x = O.synth_speech(n, SR, 7).astype(np.float32)
    T = 1 + n // 160
    ld = (T + 3) // 4 * 4
    out = np.zeros((80, ld), np.float32)
    mx = np.zeros(3, np.float32)
    rc = emul.emul_forward(_p(x), None, n, n, n, 0.0, 1, 0, ld, _p(out), None, None, None, _p(mx), SR, 0.0, 8000.0)
    assert rc == 0
    ref, _ = O.signal_to_spectrogram(O.AudioSignal(x.astype(np.float64), SR), 640, 160)
    got = np.maximum(out[:, :T], mx[0] - 80.0)
    assert ref.shape == got.shape
    assert np.max(np.abs(got - ref)) <= TOL_DB


def _run_mode(emul, s, nf, L, fac, ns, mode, fmin=0.0, fmax=8000.0):
    emul.emul_forward_mode.argtypes = emul.emul_forward.argtypes + [ctypes.c_int]
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    rc = emul.emul_forward_mode(_p(s), _p(nf), L, len(s), len(s), fac, 0, ns, 0, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm), _p(mx),
                                SR, fmin, fmax, mode)
    assert rc >= 0
    return rc, [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)]


def test_scan_and_generic_paths_agree_with_oracle(emul):
    """The fused post+mel scan (default for the reference filterbank) and the generic banded gather must both
    match the oracle; a non-reference filterbank (fmin 50, fmax 7000) exercises whichever path its tables allow."""
    case = GOLDEN_CASES[0]
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    L = 3200 * case["nvs"]
    fac = O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nf.astype(np.float64), SR), case["snr"])
    ref = oracle_pair(case)
    used_scan, got = _run_mode(emul, s, nf, L, fac, 5, 0)
    assert used_scan == 1
    used_scan, got_gen = _run_mode(emul, s, nf, L, fac, 5, 1)
    assert used_scan == 0
    for g in (got, got_gen):
        for k, o in zip(("speech", "noise", "mixed"), g):
            assert np.max(np.abs(o - ref[k])) <= TOL_DB, k
    # other filterbank: oracle with the same fmin/fmax
    fb = O.mel_filterbank(SR, 640, 80, 50.0, 7000.0)
    mix = s.astype(np.float64) + fac * nf.astype(np.float64)
    D = O.stft(mix[:L], 640, 160)
    want = O.amplitude_to_db(fb @ np.abs(D))
    for mode in (0, 1):
        _, g = _run_mode(emul, s, nf, L, fac, 5, mode, 50.0, 7000.0)
        got_full = np.concatenate(list(g[2]), axis=1)
        assert np.max(np.abs(got_full - want[:, :100])) <= TOL_DB, mode


# ---- F4 kernel (avse_fwd4_stages.cuh): four frames per warp, dense emission ----
def _run_emul4(emul, s, nf, L, fac, ns, valid=None, fmin=0.0, fmax=8000.0, gain=0.0, period=0, f2=False):
    """gain: the level-equaliser part of `fac` applied to the noise at load (0: all of `fac`, like a NULL
    avse_forward_args::equalizer); period: noise[i] = nf[i mod period] (dp:125-128); f2: the 2-frame kernel's stages."""
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    v = len(s) if valid is None else valid
    if f2:
        rc = emul.emul_forward_mode_ex(_p(s), _p(nf), L, v, v, fac, gain, period, 0, ns, 0, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm),
                                       _p(mx), SR, fmin, fmax, 0)
    else:
        rc = emul.emul_forward4_ex(_p(s), _p(nf), L, v, v, fac, gain, period, 0, ns, 0, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm),
                                   _p(mx), SR, fmin, fmax)
    assert rc == 1
    floored = [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)]
    return dict(speech=floored[0], noise=floored[1], mixed=floored[2], mixed_pcm=pcm, max=mx)


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
def test_f4_stage_code_matches_oracle_and_golden(emul, case):
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    L = 3200 * case["nvs"]
    fac = O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nf.astype(np.float64), SR), case["snr"])
    ns = min(case["nvs"], (1 + L // 160) // 20)
    got = _run_emul4(emul, s, nf, L, fac, ns)
    ref = oracle_pair(case)
    gold = np.load(os.path.join(GOLD, case["name"] + ".npz"))
    for k in ("mixed", "speech", "noise"):
        assert np.max(np.abs(got[k] - ref[k])) <= TOL_DB, k
        assert np.max(np.abs(got[k] - gold[k])) <= TOL_DB + 2e-5, k
    scale = np.max(np.abs(ref["mixed_pcm"]))
    assert np.max(np.abs(got["mixed_pcm"] - ref["mixed_pcm"])) <= TOL_PCM * scale


def test_f4_agrees_with_two_frame_kernel_and_other_filterbank(emul):
    case = GOLDEN_CASES[0]
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    L = 3200 * case["nvs"]
    fac = O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nf.astype(np.float64), SR), case["snr"])
    got4 = _run_emul4(emul, s, nf, L, fac, 5)
    _, got2 = _run_mode(emul, s, nf, L, fac, 5, 0)
    for k, o in zip(("speech", "noise", "mixed"), got2):
        assert np.max(np.abs(got4[k] - o)) <= 2e-4, k      # same arithmetic up to summation order of the band sums
    fb = O.mel_filterbank(SR, 640, 80, 50.0, 7000.0)
    mix = s.astype(np.float64) + fac * nf.astype(np.float64)
    want = O.amplitude_to_db(fb @ np.abs(O.stft(mix[:L], 640, 160)))
    g = _run_emul4(emul, s, nf, L, fac, 5, fmin=50.0, fmax=7000.0)
    assert np.max(np.abs(np.concatenate(list(g["mixed"]), axis=1) - want[:, :100])) <= TOL_DB


@pytest.mark.parametrize("n_valid,nvs", [(16000, 5), (10000, 5), (7013, 3), (3200, 1), (330, 1)])
def test_f4_ragged_and_zero_padded_lengths(emul, n_valid, nvs):
    """pad_with_zeros (dp:40) / short utterances: every group takes the edge path or mixes edge and interior groups."""
    rng = np.random.RandomState(n_valid)
    L = 3200 * nvs
    s = np.zeros(L, np.float32)
    nf = np.zeros(L, np.float32)
    nv = min(n_valid, L)
    s[:nv] = O.synth_speech(nv, SR, 3).astype(np.float32)
    nf[:nv] = (0.05 * rng.randn(nv)).astype(np.float32)
    fac = 0.7
    ns = min(nvs, (1 + L // 160) // 20)
    got = _run_emul4(emul, s, nf, L, fac, ns, valid=nv)
    for k, x in (("speech", s.astype(np.float64)), ("noise", fac * nf.astype(np.float64)), ("mixed", s.astype(np.float64) + fac * nf.astype(np.float64))):
        ref, _ = O.signal_to_spectrogram(O.AudioSignal(x, SR), 640, 160)
        want = np.stack([ref[:, 20 * i:20 * i + 20] for i in range(ns)])
        assert np.max(np.abs(got[k] - want)) <= TOL_DB, k
        assert abs(got["max"][("speech", "noise", "mixed").index(k)] - ref.max()) <= TOL_DB


def test_f4_stage_code_fuzz_against_oracle(emul):
    """Property test (hypothesis): random valid lengths (edge / interior group mixes, zero padding), slice counts, input
    scales (unit ... int16) and SNR factors -- the F4 stage code stays within the 1e-3 dB gate of the float64 oracle and
    reproduces the mixture PCM; the running max equals the oracle's max over ALL frames (dp:94)."""
    hyp = pytest.importorskip("hypothesis")
    st = hyp.strategies

    @hyp.settings(max_examples=25, deadline=None, derandomize=True, suppress_health_check=list(hyp.HealthCheck))
    @hyp.given(nvs=st.integers(1, 4), frac=st.floats(0.11, 1.0), log_scale=st.floats(-2.0, 4.5), log_nscale=st.floats(-4.0, 4.5),
               snr=st.floats(-10.0, 10.0), seed=st.integers(0, 10 ** 6))
    def check(nvs, frac, log_scale, log_nscale, snr, seed):
        # speech and noise levels are drawn INDEPENDENTLY (a float WAV next to an int16 one ...): the level equaliser
        # g goes to the kernel stages as `gain`, the full factor as `factor`; zero-mean noise: sqrt(sum s^2 / sum n^2) is
        # within rounding of the ratio of standard deviations used here
        L = 3200 * nvs
        nv = max(330, min(L, int(frac * L)))
        rng = np.random.RandomState(seed)
        scale = 10.0 ** log_scale
        s = np.zeros(L, np.float32)
        nf = np.zeros(L, np.float32)
        s[:nv] = (O.synth_speech(nv, SR, seed) * scale).astype(np.float32)
        nf[:nv] = (10.0 ** log_nscale * rng.randn(nv)).astype(np.float32)
        gain = np.float32(np.sqrt(np.var(s[:nv].astype(np.float64)) / np.var(nf[:nv].astype(np.float64))))
        fac = np.float32(float(gain) * 10.0 ** (-snr / 20.0))
        ns = min(nvs, (1 + L // 160) // 20)
        got = _run_emul4(emul, s, nf, L, fac, ns, valid=nv, gain=gain)
        f = float(fac)
        mix = s.astype(np.float64) + f * nf.astype(np.float64)
        assert np.max(np.abs(got["mixed_pcm"] - mix)) <= TOL_PCM * max(np.max(np.abs(mix)), 1e-30)
        for k, x in (("speech", s.astype(np.float64)), ("noise", f * nf.astype(np.float64)), ("mixed", mix)):
            ref, _ = O.signal_to_spectrogram(O.AudioSignal(x, SR), 640, 160)
            want = np.stack([ref[:, 20 * i:20 * i + 20] for i in range(ns)])
            assert np.max(np.abs(got[k] - want)) <= TOL_DB, (k, nvs, nv, scale, log_nscale, snr)
            assert abs(got["max"][("speech", "noise", "mixed").index(k)] - ref.max()) <= TOL_DB

    check()


# ---- level mismatch between the two files (VERDICT r1 "what's weak" #1): speech and noise at unrelated raw levels ----
LEVELS = [(1.0, 1.0), (1.0, 10.0), (1.0, 100.0), (1.0, 32767.0), (100.0, 1.0), (32767.0, 1.0), (1e-4, 1.0), (1.0, 1e-4), (3000.0, 30000.0)]


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "f2"])
@pytest.mark.parametrize("snr", [-10.0, 0.0, 10.0])
def test_level_mismatch_holds_the_gate(emul, snr, f2):
    """dp:130-133 exists precisely for files recorded at different levels.  With the noise equalised to the speech power
    before the packed FFT (gain = sqrt(sum s^2 / sum n^2), the statistics pass's equaliser) and only the rest applied by linearity, the three log-mels
    stay within 1e-3 dB of the float64 oracle and the mixture PCM within 1e-4 of full scale for raw level ratios from
    1e-4 to 3e4 (float WAV vs int16 WAV) at -10 / 0 / +10 dB."""
    L = 16000
    for ss, nsx in LEVELS:
        s = (O.synth_speech(L, SR, 5) * ss).astype(np.float32)
        n = (O.synth_noise(L, 5) * nsx).astype(np.float32)
        if max(ss, nsx) > 1000.0:
            s, n = np.round(s), np.round(n) if nsx > 1000.0 else n    # int16-valued samples at int16 scale
        sp, nz = O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(n.astype(np.float64), SR)
        fac = np.float32(O.AudioMixer.snr_factor(sp, nz, snr))
        gain = np.float32(O.AudioMixer.snr_factor(sp, nz, 0.0))
        mixed, speech, noise, msig = O.preprocess_audio_pair_signals(sp, nz, 200, 5, 25.0, snr_db=snr)
        got = _run_emul4(emul, s, n, L, fac, 5, gain=gain, f2=f2)
        for k, ref in (("speech", speech), ("noise", noise), ("mixed", mixed)):
            assert np.max(np.abs(got[k] - ref)) <= TOL_DB, (k, ss, nsx, snr)
        full = np.max(np.abs(msig.get_data()))
        assert np.max(np.abs(got["mixed_pcm"] - msig.get_data())) <= TOL_PCM * full, (ss, nsx, snr)


def test_unequalised_packing_would_fail(emul):
    """The failure the equaliser removes, kept as a regression guard for the test itself: with the whole factor applied
    only after the unpack (gain = 1) a 100x level gap breaks the speech log-mel by more than 10x the gate."""
    L = 16000
    s = O.synth_speech(L, SR, 5).astype(np.float32)
    n = (O.synth_noise(L, 5) * 100.0).astype(np.float32)
    sp, nz = O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(n.astype(np.float64), SR)
    fac = np.float32(O.AudioMixer.snr_factor(sp, nz, 0.0))
    _, speech, _, _ = O.preprocess_audio_pair_signals(sp, nz, 200, 5, 25.0, snr_db=0.0)
    bad = _run_emul4(emul, s, n, L, fac, 5, gain=1.0)
    good = _run_emul4(emul, s, n, L, fac, 5, gain=fac)
    assert np.max(np.abs(bad["speech"] - speech)) > 10 * TOL_DB
    assert np.max(np.abs(good["speech"] - speech)) <= TOL_DB


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "f2"])
@pytest.mark.parametrize("n_noise", [5000, 1121, 640, 333, 15999, 16000, 40000])
def test_in_kernel_noise_tiling(emul, n_noise, f2):
    """dp:125-128: a noise file shorter than the speech is doubled until it covers it and truncated == noise[i mod Ln].
    The stage code addresses the stored period itself (interior groups that do not straddle a period boundary keep
    the fast loads, the others take the edge loader) and must equal the oracle run on the materialised tiling."""
    L = 16000
    s = O.synth_speech(L, SR, 11).astype(np.float32)
    n = O.synth_noise(n_noise, 11).astype(np.float32)
    sp, nz = O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(n.astype(np.float64), SR)
    mixed, speech, noise, msig = O.preprocess_audio_pair_signals(sp, nz, 200, 5, 25.0, snr_db=3.0)
    nfit = fitted_noise(s, n)
    fac = np.float32(O.AudioMixer.snr_factor(O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(nfit.astype(np.float64), SR), 3.0))
    gain = np.float32(float(fac) / 10.0 ** (-3.0 / 20.0))
    row = np.zeros(L, np.float32)                       # only the first min(Ln, L) samples of the row exist
    m = min(n_noise, L)
    row[:m] = n[:m]
    row[m:] = np.nan                                    # anything read past the period would poison the result
    got = _run_emul4(emul, s, row, L, fac, 5, gain=gain, period=n_noise, f2=f2)
    for k, ref in (("speech", speech), ("noise", noise), ("mixed", mixed)):
        assert np.max(np.abs(got[k] - ref)) <= TOL_DB, k
    assert np.max(np.abs(got["mixed_pcm"] - msig.get_data())) <= TOL_PCM * np.max(np.abs(msig.get_data()))


@pytest.mark.parametrize("L", [2560, 2561, 2719, 3333, 4001, 6400, 16000, 16100])
def test_f4_reflect_only_edge_groups_at_awkward_lengths(emul, L):
    """Full-length utterances (no zero padding) take the interior pass 1 with mirrored load indices in their first and last groups
    (AVSE_F4_REFLECT_FAST; L >= 4 n_fft): lengths that are not multiples of the hop, last groups holding 1, 2, 3 or 4 frames, and
    the shortest length the path accepts -- log-mel, running max and mixture PCM against the oracle."""
    rng = np.random.RandomState(L)
    s = O.synth_speech(L, SR, L % 7).astype(np.float32)
    nf = (0.05 * rng.randn(L)).astype(np.float32)
    fac = 0.9
    T = 1 + L // 160
    ns = max(1, T // 20)
    got = _run_emul4(emul, s, nf, L, fac, ns)
    for k, x in (("speech", s.astype(np.float64)), ("noise", fac * nf.astype(np.float64)), ("mixed", s.astype(np.float64) + fac * nf.astype(np.float64))):
        ref, _ = O.signal_to_spectrogram(O.AudioSignal(x, SR), 640, 160)
        assert ref.shape[1] == T
        if T >= 20:
            want = np.stack([ref[:, 20 * i:20 * i + 20] for i in range(ns)])
            assert np.max(np.abs(got[k] - want)) <= TOL_DB, k
        assert abs(got["max"][("speech", "noise", "mixed").index(k)] - ref.max()) <= TOL_DB, k
    want_pcm = s.astype(np.float64) + fac * nf.astype(np.float64)
    assert np.max(np.abs(got["mixed_pcm"] - want_pcm)) <= TOL_PCM * np.max(np.abs(want_pcm))
