"""GPU parity of the explicit-phase and SPEC-layout forms of avse_inverse against the float64 oracle.

avse_inverse serves three call forms: (a) dB slices + mixture PCM (reconstruct; covered in test_gpu_inverse.py), (b) an explicit
phase (reconstruct_with_phase, the mirror's reconstruct_signal_from_spectrogram, dp:99-116: the EXT instantiation of the I8
kernel, or the generic kernels' caller-phase branch) and (c) a SPEC-layout mel [B][80][ld_t] + mixture PCM (reconstruct_spec).
This file covers (b) and (c) on the specialised I8 kernel and on the generic-geometry kernels."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS
from tests.test_gpu_generic import CONFIGS

pytestmark = pytest.mark.gpu

TOL_PCM = 1e-4   # of full scale (BASELINE.json north_star)
PKG = "audio-visual-speech-enhancement_b200"


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module(PKG + ".engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


@pytest.fixture(scope="module")
def dp():
    return importlib.import_module(PKG + ".data_processor")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _inverse(eng, mel, out, phase=None, pcm=None, lengths=None, n_frames=None):
    """avse_inverse through the C ABI with a SPEC-layout mel [B, 80, ld_t] (first n_frames columns used) and either an explicit
    phase [B, T_ph, bins] complex64 or the mixture pcm [B, L]; out [B, >= out_len] float32 or int16 (rows may be strided).
    Returns the out_len = hop (T_use - 1) columns of `out`."""
    native = importlib.import_module(PKG + "._native")
    B, _, ld_t = mel.shape
    n_frames = ld_t if n_frames is None else n_frames
    T = phase.shape[1] if phase is not None else eng.n_frames(pcm.shape[1])
    T_use = min(n_frames, T)
    per = ctypes.c_longlong(0)
    work = None
    if eng._needs_inverse_scratch():
        native.check(eng._lib.avse_inverse_work_elems_ctx(eng._ctx, T_use, ctypes.byref(per)), "avse_inverse_work_elems_ctx")
        work = torch.empty((B, per.value), dtype=torch.float32, device=mel.device)
    a = native.InverseArgs()
    a.mel_db, a.layout, a.n_slices, a.n_frames, a.ld_t = mel.data_ptr(), 1, 0, n_frames, ld_t
    a.mel_stride = mel.stride(0)
    if phase is not None:
        assert phase.dtype == torch.complex64 and phase.stride(2) == 1 and phase.stride(1) == phase.shape[2]
        a.phase, a.phase_stride, a.phase_frames = torch.view_as_real(phase).data_ptr(), phase.stride(0), phase.shape[1]
    else:
        a.mixed_pcm, a.pcm_stride, a.len_pcm = pcm.data_ptr(), pcm.stride(0), 0 if lengths is None else lengths.data_ptr()
        a.L = pcm.shape[1]
    a.B = B
    a.out_pcm, a.out_stride = out.data_ptr(), out.stride(0)
    a.out_format = 1 if out.dtype == torch.int16 else 0
    a.work, a.work_stride = 0 if work is None else work.data_ptr(), per.value
    with torch.cuda.device(eng.device):
        native.check(eng._lib.avse_inverse(eng._ctx, ctypes.byref(a), eng._stream()), "avse_inverse")
    return out[:, :eng.hop * (T_use - 1)]


def _want_ext(mel, phase, sr=SR, n_fft=640, hop=160):
    """dp:99-116 in float64 on the frames both arrays have: mel (80, T) dB, phase (T_ph, bins) frame-major."""
    T_use = min(mel.shape[1], phase.shape[0])
    return O.reconstruct_signal_from_spectrogram(mel[:, :T_use].astype(np.float64), phase[:T_use].T.astype(np.complex128), sr, n_fft,
                                                 hop).get_data()


def _mixture_phase(pcm, n_fft=640, hop=160):
    _, ph = O.magphase(O.stft(np.asarray(pcm, np.float64), n_fft, hop))
    return np.ascontiguousarray(ph.T)


def _phase(rng, kind, T, bins=321, n_fft=640, hop=160, sr=SR):
    """Phase sources: the phase of a synthetic mixture, random unit-modulus phases, or random ones with 30 % of entries 0 + 0j."""
    if kind == "mixture":
        n = hop * (T - 1) + 1                      # T frames also for an odd n_fft: 1 + (n + 2 (n_fft // 2) - n_fft) // hop
        x = O.synth_speech(n, sr, int(rng.randint(1000))) + O.synth_noise(n, int(rng.randint(1000)))
        ph = _mixture_phase(x, n_fft, hop)
        assert ph.shape == (T, bins)
        return ph.astype(np.complex64)
    ph = np.exp(2j * np.pi * rng.rand(T, bins)).astype(np.complex64)
    if kind == "zero":
        ph[rng.rand(T, bins) < 0.3] = 0.0
        ph[T // 2] = 0.0
    return ph


def _err(got, want):
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.isfinite(got).all()
    return float(np.max(np.abs(got - want)) / np.max(np.abs(want)))


def _mel(rng, B, T, lo=-60.0, hi=-20.0):
    return (rng.rand(B, 80, T) * (hi - lo) + lo).astype(np.float32)


KINDS = ("mixture", "random", "zero")


# ---------------------------------------------------------------------------------------------------------------------------------
# specialised geometry (640 / 160): the EXT instantiation of the I8 kernel and its SPEC loads
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("frames", ["equal", "more_mel", "more_phase"])
@pytest.mark.parametrize("T", [40, 41, 42, 43, 44, 45, 46, 47, 301])
def test_explicit_phase_batch_matches_oracle(eng, T, frames):
    """12 utterances per launch (mixture / random / partly zero phases): the launch's groups are cut into one range per warp, so
    ranges start inside utterances (warm-up groups).  T = 0 ... 7 (mod 8) and a 3 s utterance; mel and phase frame counts equal
    or either one longer (T_use = the shorter)."""
    rng = np.random.RandomState(T)
    B = 12
    T_mel = T + 3 if frames == "more_mel" else T
    T_ph = T + 5 if frames == "more_phase" else T
    mel = _mel(rng, B, T_mel)
    phase = np.stack([_phase(rng, KINDS[i % 3], T_ph) for i in range(B)])
    got = eng.reconstruct_with_phase(_dev(mel), _dev(phase)).cpu().numpy()
    assert got.shape == (B, 160 * (T - 1))
    for i in range(B):
        err = _err(got[i], _want_ext(mel[i], phase[i]))
        assert err <= TOL_PCM, (i, KINDS[i % 3], err)


def test_explicit_phase_is_independent_of_the_work_partition(eng):
    """Bit-identical results whatever the batch size (i.e. wherever the warp ranges start), float32 and int16 out."""
    rng = np.random.RandomState(21)
    B, T = 13, 157
    mel = _dev(_mel(rng, B, T))
    phase = _dev(np.stack([_phase(rng, KINDS[i % 3], T) for i in range(B)]))
    whole = eng.reconstruct_with_phase(mel, phase)
    assert torch.equal(_inverse(eng, mel, torch.empty_like(whole), phase=phase), whole)
    loud = mel + 90.0
    whole16 = _inverse(eng, loud, torch.empty(whole.shape, dtype=torch.int16, device="cuda"), phase=phase)
    for lo, hi in ((0, 1), (5, 9), (B - 1, B)):
        part = eng.reconstruct_with_phase(mel[lo:hi].contiguous(), phase[lo:hi].contiguous())
        assert torch.equal(part, whole[lo:hi]), (lo, hi)
        part16 = _inverse(eng, loud[lo:hi].contiguous(), torch.empty(part.shape, dtype=torch.int16, device="cuda"), phase=phase[lo:hi].contiguous())
        assert torch.equal(part16, whole16[lo:hi]), (lo, hi)


def test_explicit_phase_int16_out(eng):
    """avse_inverse8_kernel<true, short>: the float32 result clipped to [-32768, 32767] and truncated toward zero, exactly; at int16
    scale (+90 dB, and +110 dB where the output clips) within 1 LSB of the clipped and truncated oracle."""
    rng = np.random.RandomState(22)
    B, T = 6, 93
    mel = _mel(rng, B, T)
    mel[:3] += 90.0
    mel[3:] += 110.0
    phase = np.stack([_phase(rng, KINDS[i % 3], T) for i in range(B)])
    d_mel, d_phase = _dev(mel), _dev(phase)
    f32 = eng.reconstruct_with_phase(d_mel, d_phase)
    i16 = _inverse(eng, d_mel, torch.empty(f32.shape, dtype=torch.int16, device="cuda"), phase=d_phase)
    assert torch.equal(i16, torch.clamp(f32, -32768.0, 32767.0).to(torch.int32).to(torch.int16))
    got = i16.cpu().numpy().astype(np.int32)
    clipped = 0
    for i in range(B):
        want = _want_ext(mel[i], phase[i])
        clipped += int(np.sum(np.abs(want) > 32767.0))
        want16 = np.clip(want, -32768, 32767).astype(np.int16).astype(np.int32)
        assert np.max(np.abs(got[i] - want16)) <= 1, i
    assert clipped > 0        # the +110 dB utterances do reach the clip


@pytest.mark.parametrize("T_mel", [280, 300, 320])
def test_spec_layout_with_mixture_phase(eng, T_mel):
    """reconstruct_spec (form c): mel frames fewer than, equal to and more than the mixture's 1 + L/160 = 300; ragged lengths
    (samples past a row's length are garbage the kernel must treat as zeros); against dp:60-74 restated with an (80, T) mel, and
    bit-identical to reconstruct on the same frames in SLICES layout."""
    rng = np.random.RandomState(T_mel)
    B, L = 4, 47900
    lens = np.array([L, 30001, L, 12345], np.int32)
    pcm = (0.1 * rng.randn(B, L)).astype(np.float32)
    mel = _mel(rng, B, T_mel)
    d_pcm, d_mel, d_lens = _dev(pcm), _dev(mel), _dev(lens)
    got = eng.reconstruct_spec(d_pcm, d_mel, lengths=d_lens)
    T_use = min(T_mel, 300)
    assert got.shape == (B, 160 * (T_use - 1))
    slices = d_mel.view(B, 80, T_mel // 20, 20).permute(0, 2, 1, 3).contiguous()
    assert torch.equal(got, eng.reconstruct(d_pcm, slices, lengths=d_lens))
    got = got.cpu().numpy()
    for i in range(B):
        x = pcm[i].copy()
        x[lens[i]:] = 0.0
        err = _err(got[i], _want_ext(mel[i], _mixture_phase(x)))
        assert err <= TOL_PCM, (i, err)


def test_poisoned_unread_inputs_and_guard_bands(eng):
    """Only in-bounds memory is poisoned: phase frames at or past T_use and the SPEC columns between n_frames and ld_t hold NaN.
    The output must be finite and equal to the clean run, and every output row's guard band and a spare trailing utterance
    keep their sentinel -- EXT float32, EXT int16 and SPEC + mixture."""
    rng = np.random.RandomState(23)
    B, T, pad, gap = 5, 123, 7, 64
    out_len = 160 * (T - 1)
    mel = _dev(_mel(rng, B, T))
    phase = _dev(np.stack([_phase(rng, KINDS[i % 3], T) for i in range(B)]))
    wide = torch.full((B, 80, T + pad), float("nan"), device="cuda")
    wide[:, :, :T] = mel
    long_phase = torch.full((B, T + 9, 321), complex(float("nan"), float("nan")), dtype=torch.complex64, device="cuda")
    long_phase[:, :T] = phase
    L = 160 * (T + 4)
    pcm = _dev((0.1 * rng.randn(B, L)).astype(np.float32))

    SENT = -12345.0
    buf = torch.full((B + 1, out_len + gap), SENT, device="cuda")
    got = _inverse(eng, wide, buf[:B], phase=long_phase, n_frames=T)
    assert got.data_ptr() == buf.data_ptr()
    assert torch.all(buf[:B, out_len:] == SENT) and torch.all(buf[B] == SENT)
    assert torch.isfinite(got).all() and torch.equal(got, eng.reconstruct_with_phase(mel, phase))

    buf16 = torch.full((B + 1, out_len + gap), 12321, dtype=torch.int16, device="cuda")
    got16 = _inverse(eng, wide + 90.0, buf16[:B], phase=long_phase, n_frames=T)
    assert torch.all(buf16[:B, out_len:] == 12321) and torch.all(buf16[B] == 12321)
    clean16 = _inverse(eng, mel + 90.0, torch.empty((B, out_len), dtype=torch.int16, device="cuda"), phase=phase)
    assert torch.equal(got16, clean16)

    buf.fill_(SENT)
    got = _inverse(eng, wide, buf[:B], pcm=pcm, n_frames=T)
    assert torch.all(buf[:B, out_len:] == SENT) and torch.all(buf[B] == SENT)
    assert torch.isfinite(got).all() and torch.equal(got, eng.reconstruct_spec(pcm, mel))


def test_reference_chain_on_the_device(dp):
    """What the reference itself runs: dp:60-74 is signal_to_spectrogram(mixed) -> reconstruct_signal_from_spectrogram(mel, phase).
    The mirror's two routes -- the F2 kernel + avse_magphase followed by the EXT inverse, and the I8 kernel recomputing the phase --
    must agree with each other and with the oracle, also across a stretch of digital silence (phase 1 + 0j in both)."""
    x = (O.synth_speech(32000, SR, 7) + O.synth_noise(32000, 7)).astype(np.float32)
    x[9000:15000] = 0.0
    mel, phase = dp.signal_to_spectrogram(dp.AudioSignal(x.copy(), SR), 640, 160)
    assert mel.shape == (80, 201) and phase.shape == (321, 201)
    n = mel.shape[1] // 20
    slices = np.stack([mel[:, 20 * i:20 * (i + 1)] for i in range(n)])
    silent = np.arange(201)[(np.arange(201) * 160 - 320 >= 9000) & (np.arange(201) * 160 + 320 <= 15000)]
    assert len(silent) > 20 and np.all(phase[:, silent[1:-1]] == 1.0)     # (the outermost ones may share a packed FFT with sound)
    route_b = dp.reconstruct_signal_from_spectrogram(mel[:, :20 * n], phase[:, :20 * n], SR, 640, 160).get_data()
    route_a = dp.reconstruct_speech_signal(dp.AudioSignal(x.copy(), SR), slices, FPS).get_data()
    want = O.reconstruct_speech_signal(O.AudioSignal(x.astype(np.float64), SR), slices.astype(np.float64), FPS).get_data()
    full = np.max(np.abs(x))
    assert route_a.shape == route_b.shape == want.shape == (160 * (20 * n - 1),)
    assert np.max(np.abs(route_a - route_b)) <= TOL_PCM * full
    assert np.max(np.abs(route_a - want)) <= TOL_PCM * full
    assert np.max(np.abs(route_b - want)) <= TOL_PCM * full


# ---------------------------------------------------------------------------------------------------------------------------------
# generic geometries: the caller-phase branch and the SPEC loads of avse_generic_inverse_frame_kernel
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sr,fps", CONFIGS, ids=["%d_%g" % c for c in CONFIGS])
def test_generic_explicit_phase_spec_and_int16(mod, sr, fps):
    eng = mod.SpectralEngine(sr, fps, 200, device="cuda:0")
    assert not eng.specialised
    n_fft, hop, bins = eng.n_fft, eng.hop, eng.n_bins
    rng = np.random.RandomState(sr + int(fps))
    B = 3
    # explicit phase, float32: two launches with different frame counts, phase frames longer than the mel in the second
    for T, T_ph in ((37, 37), (52, 58)):
        mel = _mel(rng, B, T)
        phase = np.stack([_phase(rng, KINDS[i], T_ph, bins, n_fft, hop, sr) for i in range(B)])
        got = eng.reconstruct_with_phase(_dev(mel), _dev(phase)).cpu().numpy()
        assert got.shape == (B, hop * (T - 1))      # at n_fft 533 the oracle's istft infers 532: still hop (T - 1)
        for i in range(B):
            err = _err(got[i], _want_ext(mel[i], phase[i], sr, n_fft, hop))
            assert err <= TOL_PCM, (T, i, err)
    # explicit phase, int16 out == the float32 result clipped and truncated
    loud = _dev(mel + 100.0)
    d_phase = _dev(phase)
    f32 = eng.reconstruct_with_phase(loud, d_phase)
    i16 = _inverse(eng, loud, torch.empty(f32.shape, dtype=torch.int16, device="cuda"), phase=d_phase)
    assert torch.equal(i16, torch.clamp(f32, -32768.0, 32767.0).to(torch.int32).to(torch.int16))
    # SPEC + mixture phase, ragged lengths; mel frames fewer than the mixture's
    L = int(1.1 * sr)
    lens = np.array([L, L - 3 * hop - 5, L // 2 + 7], np.int32)
    pcm = (0.1 * rng.randn(B, L)).astype(np.float32)
    T_mel = eng.n_frames(L) - 2
    mel = _mel(rng, B, T_mel)
    got = eng.reconstruct_spec(_dev(pcm), _dev(mel), lengths=_dev(lens)).cpu().numpy()
    assert got.shape == (B, hop * (T_mel - 1))
    for i in range(B):
        x = pcm[i].copy()
        x[lens[i]:] = 0.0
        err = _err(got[i], _want_ext(mel[i], _mixture_phase(x, n_fft, hop), sr, n_fft, hop))
        assert err <= TOL_PCM, ("spec", i, err)
