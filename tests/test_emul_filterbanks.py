"""CPU check of the specialised context's tables and kernel stage code on filterbanks other than the reference's 0 / 8000 Hz.

SpectralEngine(..., fmin, fmax) / avse_create(sr, fmin, fmax) serve a caller-chosen Slaney bank on the specialised 640 / 160 / 80 / 20
geometry when build_tables (csrc/avse_tables.cpp) accepts it, and on the generic kernels otherwise.  build_tables sets three flags:
scan4_ok (F4 forward kernel), scan_ok (fused-scan F2 forward kernel; otherwise the F2 band-gather kernel) and post_ok (the I8
inverse's post-stage walk tables), and it refuses a bank the I8 inverse cannot serve: post_ok == false, or cond(F F^T) above
GRAM_COND_MAX (the float32 tridiagonal solve would drift from np.linalg.pinv, dp:112).

  * table invariants over a dense grid of banks at four sample rates (numpy only);
  * the I8 inverse (both phase forms), the F2 scan / gather and the F4 forward stage code against the float64 oracle on a
    stratified sample of banks (every flag combination, cond(F F^T) from 6 to 1e19);
  * for the banks refused, the generic path's pinv table against np.linalg.pinv."""
import ctypes

import numpy as np
import pytest

from oracle import avse_oracle as O
from tests.test_emul_forward import emul, _p, TOL_DB, TOL_PCM  # noqa: F401  (session fixture that builds the emulation library)
from tests.test_generic_tables import lib  # noqa: F401  (module fixture: the generic-table hooks)

GRAM_COND_MAX = 1e5          # csrc/avse_tables.h
SCAN4_BINS = 328

# Stratified sample (sr, fmin, fmax), drawn from a 20 Hz x 100 Hz grid at the four rates and spread over cond(F F^T) within each
# stratum; test_sample_strata pins what each stratum claims, so the sample keeps its meaning if the tables change.
STRATA = {
    # accepted, (scan4, scan, post) = (1, 1, 1): F4 forward, fused-scan F2 forward, I8 inverse
    "specialised_111": [(11025, 0, 1500), (11025, 80, 2680), (11025, 0, 3100), (11025, 440, 3240), (11025, 260, 3560),
                        (16000, 20, 4020), (16000, 180, 4180), (11025, 300, 4300), (11025, 540, 4640), (16000, 300, 4800),
                        (11025, 120, 1820), (11025, 340, 5140), (11025, 200, 5500), (16000, 1000, 6300), (16000, 620, 5920),
                        (16000, 200, 5900), (16000, 200, 6200), (16000, 20, 6320), (16000, 780, 7280), (16000, 680, 6980),
                        (16000, 20, 7120), (16000, 420, 7520), (16000, 320, 7420), (16000, 460, 7860), (22050, 180, 7980),
                        (16000, 720, 5520), (24000, 0, 7600), (24000, 0, 7700), (24000, 0, 7800), (24000, 0, 7900),
                        (16000, 0, 8000), (16000, 50, 7000)],
    # accepted, (0, 0, 1): the F2 band-gather forward kernel, I8 inverse
    "specialised_001": [(11025, 1480, 3780), (11025, 1360, 4060), (11025, 1380, 4380), (11025, 1280, 4380), (16000, 1480, 5580),
                        (11025, 1000, 3800), (16000, 1380, 5380), (11025, 900, 3800), (11025, 1280, 5080), (11025, 700, 3100),
                        (11025, 1280, 5280), (16000, 1160, 5560), (16000, 1440, 6440), (16000, 1180, 5180), (11025, 820, 4420),
                        (16000, 1500, 7000), (16000, 1100, 5700), (16000, 1500, 7500), (16000, 1060, 5860), (16000, 1300, 7200),
                        (11025, 840, 4840), (16000, 1240, 7140), (16000, 1140, 7140), (16000, 1120, 6920), (16000, 1060, 6760),
                        (16000, 980, 6080), (16000, 1000, 7400), (16000, 1240, 5540), (22050, 1440, 7640), (22050, 1480, 7280),
                        (16000, 0, 7900), (16000, 1000, 8000)],
    # walk tables valid, cond(F F^T) > GRAM_COND_MAX: refused
    "ill_conditioned": [(22050, 1380, 7480), (16000, 620, 5120), (22050, 60, 6260), (22050, 1240, 7640), (22050, 1180, 7880),
                        (22050, 1240, 7840), (22050, 1240, 7940), (11025, 720, 3020), (22050, 200, 7100), (16000, 520, 4620),
                        (16000, 1000, 5400), (22050, 1180, 7780), (16000, 1300, 4900), (16000, 1200, 5000), (16000, 1180, 4880),
                        (16000, 900, 5600), (16000, 20, 2820), (16000, 880, 5380), (16000, 1400, 4800), (16000, 300, 3700),
                        (16000, 1080, 4980), (16000, 1000, 5300), (22050, 1280, 7380), (16000, 900, 5500), (16000, 960, 5060),
                        (16000, 800, 5400), (16000, 1200, 4900), (22050, 1460, 6660), (16000, 400, 4000),
                        (16000, 550, 4600), (16000, 600, 4800)],
    # post_ok == false (no walk): refused, whatever cond(F F^T)
    "no_walk": [(11025, 300, 2000), (16000, 940, 5440), (22050, 1300, 7300), (22050, 1300, 7100), (22050, 1360, 7160),
                (24000, 1420, 7420), (22050, 1240, 7240), (24000, 1420, 7320), (24000, 1420, 7220), (24000, 1320, 7720),
                (11025, 20, 1520), (16000, 1260, 5060), (22050, 1360, 7860), (22050, 1220, 7920), (11025, 940, 3240),
                (16000, 920, 5120), (11025, 980, 3180), (22050, 1480, 6480), (22050, 1240, 7040), (22050, 1440, 6540),
                (22050, 1260, 7060), (22050, 960, 7960), (16000, 820, 4520), (22050, 100, 5800), (16000, 920, 4220),
                (11025, 1120, 3120), (24000, 340, 6940), (24000, 200, 7100), (16000, 1140, 4040), (16000, 760, 4660),
                (24000, 1360, 6260), (22050, 1040, 7540), (24000, 1240, 7140), (16000, 920, 3720), (22050, 760, 7460),
                (24000, 860, 7960), (22050, 640, 7040), (22050, 260, 6460), (16000, 1080, 4680), (16000, 880, 4580),
                (16000, 80, 3000), (16000, 980, 6200), (24000, 50, 8000), (16000, 300, 3500)],
}
SPECIALISED = STRATA["specialised_111"] + STRATA["specialised_001"]
REFUSED = STRATA["ill_conditioned"] + STRATA["no_walk"]


def _ids(banks):
    return ["%d_%d_%d" % b for b in banks]


def _flags(emul, sr, fmin, fmax):
    """(accepted, (scan4_ok, scan_ok, post_ok), C++ 1-norm cond(F F^T))."""
    fn = emul.emul_table_flags
    fn.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]
    out = np.zeros(3, np.int32)
    cond = ctypes.c_double(0.0)
    rc = fn(sr, float(fmin), float(fmax), _p(out), ctypes.byref(cond))
    assert rc in (0, -2)
    return rc == 0, tuple(int(v) for v in out), cond.value


def _inverse_tables(emul, sr, fmin, fmax):
    fn = emul.emul_inverse_tables
    fn.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double] + [ctypes.c_void_p] * 4
    post_w = np.zeros((SCAN4_BINS, 2), np.float32)
    post_mask = np.zeros((8, 4), np.uint32)
    tri = np.zeros((3, 80), np.float32)
    spike = np.zeros((4, 116), np.float32)
    assert fn(sr, float(fmin), float(fmax), _p(post_w), _p(post_mask), _p(tri), _p(spike)) == 0
    return post_w, post_mask, tri, spike


def _walk_matrix(post_w, post_mask):
    """F^T as the I8 post stage walks it: chunk p = bins 41 p ... 41 p + 40 starts on the pair (y[b], y[b + 1]) with b = its first
    band and moves up one band before bin i where bit i of its mask is set.  Returns the dense [80, 321] weights, or None when the
    walk leaves bands 0 ... 79."""
    W = np.zeros((80, SCAN4_BINS), np.float64)
    i = np.arange(41)
    for p in range(8):
        lo, hi, first = (int(v) for v in post_mask[p, :3])
        bits = np.where(i < 32, (lo >> np.minimum(i, 31)) & 1, (hi >> np.maximum(i - 32, 0)) & 1)
        bits[0] = 0                                        # the walk starts on `first`
        b = first + np.cumsum(bits)
        if b.min() < 0 or b.max() > 78:
            return None
        k = 41 * p + i
        W[b, k] += post_w[k, 0]
        W[b + 1, k] += post_w[k, 1]
    return W[:, :321]


def _thomas(tri, y):
    """The Thomas solve of mel_to_coef / the I4 kernel with the float32 factors (w, 1/pivot, sup), in float64; y [80, n]."""
    w, ipiv, sup = (tri[j].astype(np.float64) for j in range(3))
    d = y.copy()
    for i in range(1, 80):
        d[i] -= w[i] * d[i - 1]
    d[79] *= ipiv[79]
    for i in range(78, -1, -1):
        d[i] = (d[i] - sup[i] * d[i + 1]) * ipiv[i]
    return d


def _spike(spike, y):
    """The I8 kernel's partitioned solve (i8_coef_local / i8_coef_finish) with the float32 tables, in float64; y [80, n]."""
    tb = spike.astype(np.float64)
    Q = 20
    parts = []
    for p in range(4):
        lw, lipiv, lsup = tb[p, :Q], tb[p, Q:2 * Q], tb[p, 2 * Q:3 * Q]
        d = y[Q * p:Q * p + Q].copy()
        for i in range(1, Q):
            d[i] -= lw[i] * d[i - 1]
        d[Q - 1] *= lipiv[Q - 1]
        for i in range(Q - 2, -1, -1):
            d[i] = (d[i] - lsup[i] * d[i + 1]) * lipiv[i]
        parts.append(d)
    xch = np.stack([v for d in parts for v in (d[0], d[Q - 1])])              # [8, n]: (top, bottom) of each block
    out = []
    for p in range(4):
        rb, rt = tb[p, 5 * Q:5 * Q + 8], tb[p, 5 * Q + 8:5 * Q + 16]
        bprev, tnext = rb @ xch, rt @ xch
        out.append(parts[p] - tb[p, 3 * Q:4 * Q, None] * bprev[None] - tb[p, 4 * Q:5 * Q, None] * tnext[None])
    return np.concatenate(out)


# ---------------------------------------------------------------------------------------------------------------------------------
# table invariants, dense grid
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sr", [16000, 22050, 24000, 11025])
def test_table_invariants_on_a_dense_grid(emul, sr):
    """Every bank the specialised context accepts: the filterbank is librosa's (O.mel_filterbank), the walk tables reproduce every
    column of F^T exactly (float32 weights), cond(F F^T) <= GRAM_COND_MAX, and both the Thomas and the SPIKE factors give
    F^T (F F^T)^-1 y = pinv(F) y to float32 precision.  A bank whose tables are complete but that has no walk is refused."""
    fb_out = np.zeros((80, 321))
    y = np.random.RandomState(sr).rand(80, 8) + 0.01              # amplitudes: positive
    top = min(8000, sr // 2)
    n_accepted = n_refused = 0
    worst = 0.0
    for fmin in range(0, 1501, 50):
        for fmax in range(fmin + 500, top + 1, 250):
            ok, (scan4, scan, post), cond = _flags(emul, sr, fmin, fmax)
            if not ok:
                if cond > 0.0:                                     # tables complete: refused for the walk or the conditioning
                    assert post == 0 or cond > GRAM_COND_MAX, (fmin, fmax)
                    n_refused += 1
                continue
            n_accepted += 1
            assert post == 1 and cond <= GRAM_COND_MAX and (scan == 1 or scan4 == 0), (fmin, fmax)
            assert emul.emul_filterbank(sr, float(fmin), float(fmax), _p(fb_out)) == 0
            fb = O.mel_filterbank(sr, 640, 80, float(fmin), float(fmax))
            assert np.max(np.abs(fb_out - fb)) < 1e-13, (fmin, fmax)
            G = fb @ fb.T
            c2 = np.linalg.cond(G)
            assert c2 <= cond * (1 + 1e-6) and cond <= 80.0 * c2, (fmin, fmax, c2, cond)    # kappa_2 <= kappa_1 <= n kappa_2
            post_w, post_mask, tri, spike = _inverse_tables(emul, sr, fmin, fmax)
            W = _walk_matrix(post_w, post_mask)
            assert W is not None and np.array_equal(W, fb_out.astype(np.float32)), (fmin, fmax)   # (fb_out: edge residues ~1e-16 snapped to 0)
            want = fb.T @ np.linalg.solve(G, y)
            scale = np.max(np.abs(want))
            for x in (_thomas(tri, y), _spike(spike, y)):
                err = np.max(np.abs(fb.T @ x - want)) / scale
                worst = max(worst, err)
                assert err <= 1e-5, (fmin, fmax, err)
    assert n_accepted >= {24000: 1, 22050: 20}.get(sr, 50) and n_refused > 0, (n_accepted, n_refused)   # 24 kHz: most banks have no walk


def test_the_reference_bank_and_its_dispatch_are_unchanged(emul):
    assert _flags(emul, 16000, 0, 8000)[:2] == (True, (1, 1, 1))


# ---------------------------------------------------------------------------------------------------------------------------------
# kernel stage code, stratified sample
# ---------------------------------------------------------------------------------------------------------------------------------
def test_sample_strata(emul):
    """What each stratum claims of its banks: flags, conditioning (numpy's 2-norm cond(F F^T)) and the verdict."""
    for name, banks in STRATA.items():
        for b in banks:
            ok, flags, cond = _flags(emul, *b)
            fb = O.mel_filterbank(b[0], 640, 80, float(b[1]), float(b[2]))
            c2 = np.linalg.cond(fb @ fb.T)
            if name == "specialised_111":
                assert ok and flags == (1, 1, 1) and c2 <= GRAM_COND_MAX, b
            elif name == "specialised_001":
                assert ok and flags == (0, 0, 1) and c2 <= GRAM_COND_MAX, b
            elif name == "ill_conditioned":
                assert not ok and flags[2] == 1 and cond > GRAM_COND_MAX, b
            else:
                assert not ok and flags[2] == 0 and cond > 0.0, b
    # the sample spans the conditioning on both sides of the threshold, and well-conditioned banks without a walk
    conds = [np.linalg.cond(O.mel_filterbank(b[0], 640, 80, float(b[1]), float(b[2])) @
                            O.mel_filterbank(b[0], 640, 80, float(b[1]), float(b[2])).T) for b in REFUSED]
    assert min(conds) < 100.0 and max(conds) > 1e15
    assert sum(c < 1e3 for c, b in zip(conds, REFUSED) if b in STRATA["no_walk"]) >= 10


def _run_i8(emul, sr, fmin, fmax, mel, pcm=None, phase=None, chunks=1):
    fn = emul.emul_inverse8_ex
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                   ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double]
    T = mel.shape[1]
    out = np.full(160 * (T - 1), np.nan, np.float32)
    L = 0 if pcm is None else len(pcm)
    n = fn(_p(mel), 1, 0, T, T, _p(pcm), L, L, _p(phase), 0 if phase is None else phase.shape[0], _p(out), len(out), chunks, sr,
           float(fmin), float(fmax))
    return n, out


def _err(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    return float(np.max(np.abs(got - want)) / np.max(np.abs(want)))


def _pinv_oracle(fb, mel, phase):
    """dp:99-116 with the bank's own filterbank: istft((pinv(F) 10^(mel/20)) phase, 160); phase [bins, T]."""
    return O.istft((np.linalg.pinv(fb) @ O.db_to_amplitude(mel.astype(np.float64))) * phase, 160)


@pytest.mark.parametrize("bank", SPECIALISED + REFUSED, ids=_ids(SPECIALISED + REFUSED))
def test_inverse_matches_the_pinv_oracle(emul, lib, bank):  # noqa: F811
    """Accepted banks: the I8 stage code, mixture-phase form and explicit-phase form (two chunks: a warm-up group), within 1e-4 of
    the peak of the float64 pinv oracle.  Refused banks: the emulator (like avse_create) refuses them, and the generic path's
    pinv table (Jacobi SVD in float64, rounded to float32) is np.linalg.pinv and reconstructs within the same gate."""
    sr, fmin, fmax = bank
    fb = O.mel_filterbank(sr, 640, 80, float(fmin), float(fmax))
    rng = np.random.RandomState(fmin * 7 + fmax + sr)
    T = 26
    mel = (rng.rand(80, T) * 40.0 - 60.0).astype(np.float32)
    phase = np.exp(2j * np.pi * rng.rand(T, 321)).astype(np.complex64)
    pcm = (O.synth_speech(160 * (T - 1), 16000, fmin) + O.synth_noise(160 * (T - 1), fmax)).astype(np.float32)
    _, mix_phase = O.magphase(O.stft(pcm.astype(np.float64), 640, 160))
    ok = _flags(emul, *bank)[0]
    if ok:
        n, got = _run_i8(emul, sr, fmin, fmax, mel, phase=phase, chunks=2)
        assert n == len(got)
        err_ext = _err(got, _pinv_oracle(fb, mel, phase.T.astype(np.complex128)))
        n, got = _run_i8(emul, sr, fmin, fmax, mel, pcm=pcm)
        assert n == len(got)
        err_mix = _err(got, _pinv_oracle(fb, mel, mix_phase))
        assert max(err_ext, err_mix) <= TOL_PCM, (err_ext, err_mix)
        return
    assert _run_i8(emul, sr, fmin, fmax, mel, phase=phase)[0] == -2
    geo = np.zeros(10, np.int32)
    pinv = np.zeros((321, 80), np.float32)
    z = ctypes.c_void_p()
    assert lib.emul_generic_tables(sr, 640, 160, 80, 20, float(fmin), float(fmax), _p(geo), z, _p(pinv), z, z, z) == 0
    want = np.linalg.pinv(fb)
    assert np.max(np.abs(pinv - want)) <= 2e-6 * np.max(np.abs(want))
    for ph in (phase.T.astype(np.complex128), mix_phase):
        got = O.istft((pinv.astype(np.float64) @ O.db_to_amplitude(mel.astype(np.float64))) * ph, 160)
        assert _err(got, _pinv_oracle(fb, mel, ph)) <= TOL_PCM


def _run_forward(emul, bank, s, nf, fac, gain, kernel):
    """kernel: "f2" (the library's pick: fused scan where scan_ok, band gather otherwise), "gather" (forced), "f4"."""
    sr, fmin, fmax = bank
    L = len(s)
    ns = (1 + L // 160) // 20
    outs = [np.zeros((ns, 80, 20), np.float32) for _ in range(3)]
    pcm = np.zeros(L, np.float32)
    mx = np.zeros(3, np.float32)
    args = (_p(s), _p(nf), L, L, L, fac, gain, 0, 0, ns, 0, _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(pcm), _p(mx), sr, float(fmin),
            float(fmax))
    if kernel == "f4":
        rc = emul.emul_forward4_ex(*args)
        assert rc == 1
    else:
        rc = emul.emul_forward_mode_ex(*args, 0 if kernel == "f2" else 1)
        assert rc == (1 if kernel == "f2" and _flags(emul, *bank)[1][1] else 0)
    return [np.maximum(o, m - 80.0) for o, m in zip(outs, mx)], pcm


@pytest.mark.parametrize("bank", SPECIALISED, ids=_ids(SPECIALISED))
def test_forward_matches_the_oracle(emul, bank):
    """The F2 stage code (fused scan where scan_ok, the band gather otherwise, and the gather forced on every bank) and the F4
    stage code (where scan4_ok): speech, noise and mixture log-mel within 1e-3 dB of amplitude_to_db(fb |stft|), and the mixture."""
    sr, fmin, fmax = bank
    L = 6400
    # broadband speech: with the noise far above the speech in a band (synthetic speech has little energy above ~5 kHz) the
    # packed FFT's float32 cross-talk alone exceeds the gate, whatever the tables
    s = (O.synth_speech(L, sr, fmin) + 0.5 * O.synth_noise(L, fmin + 1)).astype(np.float32)
    nf = O.synth_noise(L, fmax).astype(np.float32)
    gain = np.float32(np.sqrt(np.var(s.astype(np.float64)) / np.var(nf.astype(np.float64))))   # the level equaliser (snr_factor)
    fac = np.float32(0.8 * gain)
    fb = O.mel_filterbank(sr, 640, 80, float(fmin), float(fmax))
    f = float(fac)
    mix = s.astype(np.float64) + f * nf.astype(np.float64)
    want = [O.amplitude_to_db(fb @ np.abs(O.stft(x, 640, 160)))[:, :40] for x in (s.astype(np.float64), f * nf.astype(np.float64), mix)]
    kernels = ["f2", "gather"] + (["f4"] if _flags(emul, *bank)[1][0] else [])
    for kernel in kernels:
        got, pcm = _run_forward(emul, bank, s, nf, fac, gain, kernel)
        for name, g, w in zip(("speech", "noise", "mixed"), got, want):
            err = np.max(np.abs(np.concatenate(list(g), axis=1) - w))
            assert err <= TOL_DB, (kernel, name, err)
        assert np.max(np.abs(pcm - mix)) <= TOL_PCM * np.max(np.abs(mix)), kernel
