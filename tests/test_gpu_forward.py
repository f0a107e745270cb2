"""GPU parity tests of the forward path: CUDA kernels (through the C ABI) vs the float64 oracle and golden vectors.

Tolerances are BASELINE.json's: <= 1e-3 dB on log-mel, <= 1e-4 of full scale on PCM.
"""
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import GOLDEN_CASES, SR, FPS, make_inputs, oracle_pair, fitted_noise

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL_DB = 1e-3
TOL_PCM = 1e-4


@pytest.fixture(scope="module")
def eng():
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


@pytest.fixture(scope="module")
def dp():
    return importlib.import_module("audio-visual-speech-enhancement_b200.data_processor")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _run_pair(eng, case):
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    lens = _dev(np.array([len(s)], np.int32))
    snr = _dev(np.array([case["snr"]], np.float32))
    mixed, speech, noise, pcm = eng.preprocess_pairs(_dev(s[None]), _dev(nf[None]), case["nvs"], lengths=lens, snr_db=snr)
    torch.cuda.synchronize()
    return dict(mixed=mixed[0].cpu().numpy(), speech=speech[0].cpu().numpy(), noise=noise[0].cpu().numpy(),
                mixed_pcm=pcm[0].cpu().numpy())


def test_library_is_loaded_and_filterbank_matches(eng):
    fb = eng.filterbank()
    assert np.max(np.abs(fb - O.mel_filterbank(SR, 640, 80, 0.0, 8000.0))) < 1e-14


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c["name"] for c in GOLDEN_CASES])
def test_pair_matches_oracle_and_golden(eng, case):
    got = _run_pair(eng, case)
    ref = oracle_pair(case)
    gold = np.load(os.path.join(GOLD, case["name"] + ".npz"))
    for k in ("mixed", "speech", "noise"):
        assert got[k].shape == ref[k].shape
        assert np.max(np.abs(got[k] - ref[k])) <= TOL_DB, (k, np.max(np.abs(got[k] - ref[k])))
        assert np.max(np.abs(got[k] - gold[k])) <= TOL_DB + 2e-5, k
    scale = np.max(np.abs(ref["mixed_pcm"]))
    assert np.max(np.abs(got["mixed_pcm"] - ref["mixed_pcm"])) <= TOL_PCM * scale


def test_snr_factor_matches_mediaio_semantics(eng):
    rng = np.random.RandomState(3)
    B, L = 7, 20000
    s = (rng.randn(B, L) * 1000 + 37.0).astype(np.float32)   # DC offset: variance must be mean-removed
    n = (rng.randn(B, L) * 30 - 5.0).astype(np.float32)
    lens = np.array([20000, 19999, 12345, 321, 5000, 20000, 7], np.int32)
    snr = np.array([0, -10, 10, 5, -5, 2.5, 0], np.float32)
    f, _ = eng.snr_factor(_dev(s), _dev(n), lengths=_dev(lens), snr_db=_dev(snr))
    f = f.cpu().numpy()
    for u in range(B):
        ref = np.sqrt(np.var(s[u, :lens[u]].astype(np.float64)) / np.var(n[u, :lens[u]].astype(np.float64))) * 10 ** (-snr[u] / 20.0)
        assert abs(f[u] - ref) <= 2e-7 * ref


def test_batch_of_mixed_lengths_and_snrs(eng):
    # ragged batch: every utterance must match its own single-utterance oracle (per-utterance max / variance)
    cases = [dict(name="b%d" % i, n_s=[16000, 9000, 16000, 20000, 700][i], n_n=16000, nvs=5, snr=[0.0, -10.0, 10.0, 5.0, -5.0][i],
                  seed=200 + i, scale=[1.0, 1.0, 32767.0, 0.01, 1.0][i]) for i in range(5)]
    W = 20000
    S = np.zeros((5, W), np.float32)
    N = np.zeros((5, W), np.float32)
    lens = np.zeros(5, np.int32)
    for i, c in enumerate(cases):
        s, n = make_inputs(c)
        S[i, :len(s)] = s
        N[i, :len(s)] = fitted_noise(s, n)
        lens[i] = len(s)
    snr = np.array([c["snr"] for c in cases], np.float32)
    mixed, speech, noise, pcm = eng.preprocess_pairs(_dev(S), _dev(N), 5, lengths=_dev(lens), snr_db=_dev(snr))
    for i, c in enumerate(cases):
        ref = oracle_pair(c)
        for k, got in (("mixed", mixed), ("speech", speech), ("noise", noise)):
            err = np.max(np.abs(got[i].cpu().numpy() - ref[k]))
            assert err <= TOL_DB, (i, k, err)
        scale = np.max(np.abs(ref["mixed_pcm"]))
        assert np.max(np.abs(pcm[i].cpu().numpy() - ref["mixed_pcm"])) <= TOL_PCM * scale


def test_video_alignment_truncates_slices(eng):
    # dp:164: n_slices = min(video, audio).  The floor still uses the max over ALL frames of the signal (dp:94).
    case = GOLDEN_CASES[3]
    s, n = make_inputs(case)
    nf = fitted_noise(s, n)
    ref = oracle_pair(case)
    res = eng.forward_raw(_dev(s[None]), _dev(nf[None]), L=48000, factor=eng.snr_factor(_dev(s[None]), _dev(nf[None]))[0],
                          n_slices=11)
    sp = eng.floor_(res["speech"], res["max_key"], 0)[0].cpu().numpy()
    assert sp.shape == (11, 80, 20)
    assert np.max(np.abs(sp - ref["speech"][:11])) <= TOL_DB


def test_spectrogram_layout_gather_and_stft(eng):
    x = (O.synth_speech(30000, SR, 9) + O.synth_noise(30000, 9)).astype(np.float32)
    db, D = eng.spectrogram(_dev(x), stft=True)
    ref_db, _ = O.signal_to_spectrogram(O.AudioSignal(x.astype(np.float64), SR), 640, 160)
    ref_D = O.stft(x.astype(np.float64), 640, 160)
    assert db.shape == (1, 80, 188)
    assert np.max(np.abs(db[0].cpu().numpy() - ref_db)) <= TOL_DB
    got_D = D[0].cpu().numpy().T
    assert np.max(np.abs(got_D - ref_D)) <= 2e-6 * np.max(np.abs(ref_D))
    # SPEC -> slices through the segment-gather kernel == dp:49-57
    res = eng.forward_raw(_dev(x), None, layout=1, want=("speech",), mixed_pcm=False)
    sl = eng.floor_gather(res["speech"], res["max_key"], 0, 9)[0].cpu().numpy()
    a = O.AudioSignal(x.astype(np.float64), SR)
    full, _ = O.signal_to_spectrogram(a, 640, 160)
    want = np.stack([full[:, 20 * i:20 * (i + 1)] for i in range(9)])
    assert np.max(np.abs(sl - want)) <= TOL_DB


def test_linearity_and_scale_invariants_full_size(eng):
    # size-independent properties at BASELINE config-2 scale (1000 x 3 s) without a CPU oracle pass:
    # (1) scaling the inputs by c shifts every un-floored dB value by 20 log10(c); (2) speech-only == pair's speech
    B, L = 1000, 48000
    g = torch.Generator(device="cuda").manual_seed(1)
    s = torch.randn((B, L), generator=g, device="cuda") * 0.1
    n = torch.randn((B, L), generator=g, device="cuda") * 0.05
    f, mk = eng.snr_factor(s, n)
    r1 = eng.forward_raw(s, n, factor=f, max_key=mk)
    f2, mk2 = eng.snr_factor(s * 4.0, n * 4.0)
    r2 = eng.forward_raw(s * 4.0, n * 4.0, factor=f2, max_key=mk2)
    assert torch.max(torch.abs(f - f2)).item() < 1e-5
    shift = 20.0 * np.log10(4.0)
    for k in ("speech", "noise", "mixed"):
        d = (r2[k] - r1[k] - shift).abs().max().item()
        assert d <= 2e-3, (k, d)   # two independent float32 evaluations: 2 x the 1e-3 dB gate
    assert (r2["mixed_pcm"] - 4.0 * r1["mixed_pcm"]).abs().max().item() <= 1e-5
    # every utterance's running max equals the max of what was written plus the dropped tail frame
    mx = eng.max_db(mk)
    assert torch.all(mx[:, 2] >= r1["mixed"].amax(dim=(1, 2, 3)) - 1e-6)
    # floor: idempotent and exactly max - 80
    sp = r1["speech"].clone()
    eng.floor_(sp, mk, 0)
    sp2 = sp.clone()
    eng.floor_(sp2, mk, 0)
    assert torch.equal(sp, sp2)
    assert torch.all(sp.amin(dim=(1, 2, 3)) >= mx[:, 0] - 80.0)


def test_floor_skip_uses_the_stored_minimum(eng):
    # min keys = min over the STORED un-floored values; the floor pass that skips on them equals the unconditional floor,
    # both for utterances that need no clipping (white noise) and for ones that do (digital silence -> -100 dB).
    B, L = 6, 16000
    g = torch.Generator(device="cuda").manual_seed(7)
    s = torch.randn((B, L), generator=g, device="cuda") * 0.1
    n = torch.randn((B, L), generator=g, device="cuda") * 0.05
    s[1, 4000:9000] = 0.0
    n[1, 4000:9000] = 0.0       # silence in both: every signal of utterance 1 hits amin
    s[4, 2000:6000] = 0.0       # silence in the speech only
    f, keys = eng.snr_factor(s, n)
    r = eng.forward_raw(s, n, factor=f, n_slices=4, max_key=keys)   # 4 of 5 slices stored
    mn, mx = eng.min_db(keys), eng.max_db(keys)
    for j, k in enumerate(("speech", "noise", "mixed")):
        assert torch.equal(mn[:, j], r[k].amin(dim=(1, 2, 3))), k
        want = torch.maximum(r[k], (mx[:, j] - 80.0).view(B, 1, 1, 1))
        got = r[k].clone()
        eng.floor_(got, keys, j)            # with min keys (skips where possible)
        assert torch.equal(got, want), k
        got2 = r[k].clone()
        eng.floor_(got2, keys.max, j)       # bare max keys: unconditional pass
        assert torch.equal(got2, want), k
    need = (mn < mx - 80.0).cpu().numpy()
    assert need[1].all() and need[4, 0] and not need[0].any() and not need[4, 1]
    sp, nz, mi = r["speech"].clone(), r["noise"].clone(), r["mixed"].clone()
    eng.floor3_(sp, nz, mi, keys)
    assert torch.equal(sp, torch.maximum(r["speech"], (mx[:, 0] - 80.0).view(B, 1, 1, 1)))
    assert torch.equal(mi, torch.maximum(r["mixed"], (mx[:, 2] - 80.0).view(B, 1, 1, 1)))


def test_data_processor_signatures(dp):
    case = GOLDEN_CASES[0]
    s, n = make_inputs(case)
    ref = oracle_pair(case)
    sp = dp.AudioSignal((s * 1.0), SR)
    nz = dp.AudioSignal((n * 1.0), SR)
    mixed, speech, noise, mixed_signal = dp.preprocess_audio_pair_signals(sp, nz, 200, case["nvs"], FPS, snr_db=case["snr"])
    assert mixed.shape == (5, 80, 20) and mixed_signal.get_number_of_samples() == 16000
    assert np.max(np.abs(mixed - ref["mixed"])) <= TOL_DB
    a = dp.AudioSignal(s[:15000], SR)
    sl = dp.preprocess_audio_signal(a, 200, 5, FPS)
    assert a.get_number_of_samples() == 16000  # padded in place (dp:40)
    oa = O.AudioSignal(s[:15000].astype(np.float64), SR)
    assert np.max(np.abs(sl - O.preprocess_audio_signal(oa, 200, 5, FPS))) <= TOL_DB
    mag, phase = dp.signal_to_spectrogram(dp.AudioSignal(s, SR), 640, 160)
    rmag, rphase = O.signal_to_spectrogram(O.AudioSignal(s.astype(np.float64), SR), 640, 160)
    assert mag.shape == (80, 101) and phase.shape == (321, 101)
    assert np.max(np.abs(mag - rmag)) <= TOL_DB


def test_host_pipeline_equals_device_batch(eng):
    # engine.HostPipeline (pinned host in/out, chunked over streams, ragged last chunk, two batches back to back)
    # must reproduce preprocess_pairs on the same data bit for bit
    mod = importlib.import_module("audio-visual-speech-enhancement_b200.engine")
    B, L, nvs = 11, 16000, 5
    g = torch.Generator().manual_seed(3)
    hs = (torch.randn((B, L), generator=g) * 0.1).pin_memory()
    hn = (torch.randn((B, L), generator=g) * 0.05).pin_memory()
    snr = torch.tensor([-10.0, -5.0, 0.0, 5.0, 10.0, 0.0, 3.0, -3.0, 1.0, 2.0, 7.0]).pin_memory()
    pipe = mod.HostPipeline(eng, L, nvs, chunk=4, n_streams=2)
    outs = [[torch.zeros((B, 5, 80, 20)).pin_memory() for _ in range(3)] + [torch.zeros((B, L)).pin_memory()] for _ in range(2)]
    pipe.begin_after(torch.cuda.current_stream())
    assert pipe.submit(hs, hn, *outs[0], snr_db=snr) == 3
    pipe.submit(hn, hs, *outs[1])            # second batch right behind the first (roles swapped, 0 dB)
    pipe.synchronize()
    ref0 = eng.preprocess_pairs(hs.cuda(), hn.cuda(), nvs, snr_db=snr.cuda())
    ref1 = eng.preprocess_pairs(hn.cuda(), hs.cuda(), nvs)
    for got, ref in ((outs[0], ref0), (outs[1], ref1)):
        for a, b in zip(got, ref):
            assert torch.equal(a, b.cpu())


def test_gpu_fuzz_ragged_batch_against_oracle(eng):
    """40 utterances with random lengths (tile ranges of different warps start and end anywhere: edge groups, prefetch and
    software-pipelined loads across utterance boundaries), scales from 1e-2 to int16 range and SNRs in [-10, 10] dB: every
    one must match its own float64 oracle; then the inverse on the GPU's own outputs."""
    rng = np.random.RandomState(2024)
    B, nvs = 40, 10
    Lmax = 3200 * nvs
    lens = rng.randint(400, Lmax + 1, size=B).astype(np.int32)
    lens[:3] = [Lmax, 321 + 9, Lmax - 1]
    scales = 10.0 ** rng.uniform(-2.0, 4.4, size=B)
    nscales = 10.0 ** rng.uniform(-3.0, 5.8, size=B)      # noise level drawn independently of the speech level
    snrs = rng.uniform(-10.0, 10.0, size=B).astype(np.float32)
    S = np.zeros((B, Lmax), np.float32)
    Z = np.zeros((B, Lmax), np.float32)
    for i in range(B):
        n = int(lens[i])
        S[i, :n] = (O.synth_speech(n, SR, 700 + i) * scales[i]).astype(np.float32)
        Z[i, :n] = (O.synth_noise(n, 700 + i) * nscales[i]).astype(np.float32)
    mixed, speech, noise, pcm = eng.preprocess_pairs(_dev(S), _dev(Z), nvs, lengths=_dev(lens), snr_db=_dev(snrs))
    rec = eng.reconstruct(pcm, speech, lengths=None)
    worst = 0.0
    for i in range(B):
        n = int(lens[i])
        sp = O.AudioSignal(S[i, :n].astype(np.float64), SR)
        nz = O.AudioSignal(Z[i, :n].astype(np.float64), SR)
        r_mixed, r_speech, r_noise, r_sig = O.preprocess_audio_pair_signals(sp, nz, 200, nvs, FPS, snr_db=float(snrs[i]))
        for name, got, ref in (("mixed", mixed, r_mixed), ("speech", speech, r_speech), ("noise", noise, r_noise)):
            err = np.max(np.abs(got[i].cpu().numpy() - ref))
            worst = max(worst, err)
            assert err <= TOL_DB, (i, name, n, scales[i], snrs[i], err)
        rp = r_sig.get_data()
        scale = np.max(np.abs(rp))
        assert np.max(np.abs(pcm[i].cpu().numpy() - rp)) <= TOL_PCM * scale, i
        if i % 4 == 0:
            sig = O.AudioSignal(pcm[i].double().cpu().numpy(), SR)
            want = O.reconstruct_speech_signal(sig, speech[i].double().cpu().numpy(), FPS).get_data()
            assert np.max(np.abs(rec[i].cpu().numpy() - want)) <= TOL_PCM * scale, (i, "recon")
    assert worst > 0.0


LEVELS = [(1.0, 1.0), (1.0, 10.0), (1.0, 100.0), (1.0, 32767.0), (100.0, 1.0), (32767.0, 1.0), (1e-4, 1.0), (1.0, 1e-4), (3000.0, 30000.0)]


@pytest.mark.parametrize("f2", [False, True], ids=["f4", "stft-f2"])
def test_level_mismatch_between_speech_and_noise_files(eng, f2):
    """VERDICT r1 weak #1 / ADVICE high: speech and noise recorded at unrelated raw levels (float WAV vs int16 WAV, 1e-4 ... 3e4
    ratios) at -10 / 0 / +10 dB.  The noise is equalised to the speech's raw power before the packed FFT
    (avse_forward_args::equalizer = sqrt(sum s^2 / sum n^2)) and only the rest of the factor is applied by linearity, so all three log-mels hold 1e-3 dB and the mixture PCM 1e-4 of full scale.
    f2: the 2-frame kernel (taken when a complex STFT output is requested)."""
    L, nvs = 16000, 5
    cases = [(ss, nsx, snr) for ss, nsx in LEVELS for snr in (-10.0, 0.0, 10.0)]
    B = len(cases)
    S = np.zeros((B, L), np.float32)
    Z = np.zeros((B, L), np.float32)
    for i, (ss, nsx, snr) in enumerate(cases):
        S[i] = (O.synth_speech(L, SR, 5 + i) * ss).astype(np.float32)
        Z[i] = (O.synth_noise(L, 5 + i) * nsx).astype(np.float32)
    snrs = np.array([c[2] for c in cases], np.float32)
    if f2:
        f, keys = eng.snr_factor(_dev(S), _dev(Z), snr_db=_dev(snrs))
        r = eng.forward_raw(_dev(S), _dev(Z), factor=f, max_key=keys, stft=True)
        eng.floor3_(r["speech"], r["noise"], r["mixed"], keys)
        mixed, speech, noise, pcm = r["mixed"], r["speech"], r["noise"], r["mixed_pcm"]
    else:
        mixed, speech, noise, pcm = eng.preprocess_pairs(_dev(S), _dev(Z), nvs, snr_db=_dev(snrs))
    worst = 0.0
    for i, (ss, nsx, snr) in enumerate(cases):
        sp, nz = O.AudioSignal(S[i].astype(np.float64), SR), O.AudioSignal(Z[i].astype(np.float64), SR)
        r_mixed, r_speech, r_noise, r_sig = O.preprocess_audio_pair_signals(sp, nz, 200, nvs, FPS, snr_db=snr)
        for name, got, ref in (("mixed", mixed, r_mixed), ("speech", speech, r_speech), ("noise", noise, r_noise)):
            err = np.max(np.abs(got[i].cpu().numpy() - ref))
            worst = max(worst, err)
            assert err <= TOL_DB, (name, ss, nsx, snr, err)
        full = np.max(np.abs(r_sig.get_data()))
        assert np.max(np.abs(pcm[i].cpu().numpy() - r_sig.get_data())) <= TOL_PCM * full, (ss, nsx, snr)
    print("level-mismatch sweep: worst log-mel error %.2e dB" % worst)


def test_unequalised_packing_is_what_the_equaliser_fixes(eng):
    """Regression guard for the test above: the same launch WITHOUT the equaliser (bare max_key tensor -> the whole factor is
    applied at load, which equals equalisation only at 0 dB) still passes at 0 dB, but a deliberately wrong equaliser of 1.0
    (the round-1 behaviour: raw noise packed next to the speech) breaks the speech log-mel at a 100x level gap."""
    L, nvs = 16000, 5
    s = O.synth_speech(L, SR, 5).astype(np.float32)
    z = (O.synth_noise(L, 5) * 100.0).astype(np.float32)
    sp, nz = O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(z.astype(np.float64), SR)
    _, r_speech, _, _ = O.preprocess_audio_pair_signals(sp, nz, 200, nvs, FPS, snr_db=0.0)
    f, keys = eng.snr_factor(_dev(s[None]), _dev(z[None]))
    good = eng.forward_raw(_dev(s[None]), _dev(z[None]), factor=f, max_key=keys)
    eng.floor_(good["speech"], keys, 0)
    assert np.max(np.abs(good["speech"][0].cpu().numpy() - r_speech)) <= TOL_DB
    f, keys = eng.snr_factor(_dev(s[None]), _dev(z[None]))
    keys.equalizer.fill_(1.0)
    bad = eng.forward_raw(_dev(s[None]), _dev(z[None]), factor=f, max_key=keys)
    eng.floor_(bad["speech"], keys, 0)
    assert np.max(np.abs(bad["speech"][0].cpu().numpy() - r_speech)) > 5 * TOL_DB


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_in_kernel_noise_tiling(eng, i16):
    """dp:125-128 inside the kernels: noise files shorter than their speech are addressed as noise[i mod Ln] by the SNR pass and
    the forward loaders (no tiled copy is materialised; the rest of each noise row is poisoned), longer ones are truncated.
    Every utterance must match its own oracle, and the batch must be bit-identical to the explicit-copy path."""
    nvs, L = 10, 32000
    n_noise = [5000, 1121, 640, 333, 31999, 32000, 50000, 16000, 7, 2049]
    n_speech = [32000, 32000, 30000, 32000, 32000, 32000, 32000, 20000, 32000, 25000]
    B = len(n_noise)
    scale = 20000.0 if i16 else 1.0
    dt = np.int16 if i16 else np.float32
    S = np.zeros((B, L), dt)
    Zp = np.full((B, L), 30000 if i16 else np.nan, dt)     # period-only rows: anything read past Ln poisons the result
    Zf = np.zeros((B, L), dt)                               # explicit tiling (the round-1 host-side fit)
    raw = []
    for i in range(B):
        s = O.synth_speech(n_speech[i], SR, 40 + i) * scale
        n = O.synth_noise(n_noise[i], 40 + i) * scale * (3.0 if i % 2 else 0.2)
        s, n = (np.round(s).astype(dt), np.round(n).astype(dt)) if i16 else (s.astype(dt), n.astype(dt))
        raw.append((s, n))
        S[i, :len(s)] = s
        m = min(len(n), len(s))
        Zp[i, :m] = n[:m]
        Zf[i, :len(s)] = fitted_noise(s, n)
    lens = _dev(np.array(n_speech, np.int32))
    nlens = _dev(np.array([min(a, b) for a, b in zip(n_noise, n_speech)], np.int32))
    snr = _dev(np.linspace(-10, 10, B).astype(np.float32))
    got = eng.preprocess_pairs(_dev(S), _dev(Zp), nvs, lengths=lens, snr_db=snr, noise_lengths=nlens)
    ref = eng.preprocess_pairs(_dev(S), _dev(Zf), nvs, lengths=lens, snr_db=snr)
    for a, b, name in zip(got, ref, ("mixed", "speech", "noise", "pcm")):
        assert torch.isfinite(a).all(), name
        # same arithmetic on the same values; only the float64 summation order of the variance differs (period sums)
        assert torch.allclose(a, b, rtol=0, atol=2e-5 if name != "pcm" else 1e-6 * scale), name
    for i in range(B):
        if n_noise[i] == 7:
            continue        # a 7-sample period is a line spectrum with > 80 dB valleys: float32 FFT territory, checked above vs the copy path
        s, n = raw[i]
        sp, nz = O.AudioSignal(s.astype(np.float64), SR), O.AudioSignal(n.astype(np.float64), SR)
        r = O.preprocess_audio_pair_signals(sp, nz, 200, nvs, FPS, snr_db=float(snr[i]))
        for k in range(3):
            assert np.max(np.abs(got[k][i].cpu().numpy() - r[k])) <= TOL_DB, (i, k)
        full = np.max(np.abs(r[3].get_data()))
        assert np.max(np.abs(got[3][i].cpu().numpy() - r[3].get_data())) <= TOL_PCM * full, i


def test_empty_and_tiny_utterances(eng):
    """lengths[u] == 0 (empty WAV): the reference mixes two empty arrays and zero-pads (dp:39-40) -> every log-mel is the
    amin floor (-100 dB) and the mixture is silence; nothing is NaN.  Lengths beyond the row are clamped, not read."""
    B, L, nvs = 4, 16000, 5
    g = torch.Generator(device="cuda").manual_seed(5)
    s = torch.randn((B, L), generator=g, device="cuda") * 0.1
    z = torch.randn((B, L), generator=g, device="cuda") * 0.05
    lens = torch.tensor([0, 1, 16000, 10 ** 9], dtype=torch.int32, device="cuda")
    info = {}
    mixed, speech, noise, pcm = eng.preprocess_pairs(s, z, nvs, lengths=lens, info=info)
    f = info["factor"].cpu().numpy()
    assert f[0] == 0.0 and np.isfinite(f[2:]).all()
    for t in (speech, mixed, noise):
        assert float((t[0] + 100.0).abs().max()) <= 1e-4
    assert torch.all(pcm[0] == 0)
    ref = eng.preprocess_pairs(s[2:4].contiguous(), z[2:4].contiguous(), nvs)
    for a, b in zip((mixed, speech, noise, pcm), ref):
        assert torch.equal(a[2:4], b)                                    # the over-long length behaves like the full row


def test_batch_beyond_65535_utterances(eng):
    """ADVICE r1 / VERDICT missing #5: nothing on the pair path is capped at a grid.y of 65 535 any more (the floor kernels carry
    the utterance on grid.x).  70 000 one-slice utterances in ONE launch; spot-checked against sub-batches."""
    B, nvs, L = 70000, 1, 3200
    g = torch.Generator(device="cuda").manual_seed(9)
    s = torch.randn((B, L), generator=g, device="cuda") * 0.1
    s[:, 1600:] *= 1e-6                                   # quiet second half: every utterance needs the top_db clip
    z = torch.randn((B, L), generator=g, device="cuda") * 0.02
    mixed, speech, noise, pcm = eng.preprocess_pairs(s, z, nvs)
    assert torch.isfinite(speech).all()
    for lo in (0, 65530, 69990):
        ref = eng.preprocess_pairs(s[lo:lo + 10].contiguous(), z[lo:lo + 10].contiguous(), nvs)
        for a, b in zip((mixed, speech, noise, pcm), ref):
            assert torch.equal(a[lo:lo + 10], b)
    # the floor really ran for the late utterances: min == max - 80 where the quiet half was clipped
    sp = speech[69999]
    assert float(sp.max() - sp.min()) <= 80.0 + 1e-4
    rec = eng.reconstruct(pcm[65530:65540], speech[65530:65540])
    assert torch.isfinite(rec).all()


def test_noise_tiling_on_the_two_frame_kernel(eng):
    """The 2-frame kernel (taken when a complex STFT output is requested) reads a periodically tiled noise through its edge
    loader: same log-mels as the F4 kernel's TILED instantiation on the same batch."""
    L, nvs = 16000, 5
    S = np.stack([O.synth_speech(L, SR, 60 + i).astype(np.float32) for i in range(3)])
    n_noise = [5000, 640, 16000]
    Z = np.full((3, L), np.nan, np.float32)
    for i, n in enumerate(n_noise):
        Z[i, :n] = O.synth_noise(n, 60 + i).astype(np.float32)
    nl = _dev(np.array(n_noise, np.int32))
    f, keys = eng.snr_factor(_dev(S), _dev(Z), noise_lengths=nl)
    r2 = eng.forward_raw(_dev(S), _dev(Z), factor=f, max_key=keys, stft=True, noise_lengths=nl)
    eng.floor3_(r2["speech"], r2["noise"], r2["mixed"], keys)
    ref = eng.preprocess_pairs(_dev(S), _dev(Z), nvs, noise_lengths=nl)
    for k, b in zip(("mixed", "speech", "noise", "mixed_pcm"), ref):
        # two kernels with different summation orders, each within 1e-3 dB of the oracle: <= 2e-3 dB between them
        assert torch.isfinite(r2[k]).all() and torch.allclose(r2[k], b, rtol=0, atol=2e-3 if k != "mixed_pcm" else 1e-6), k
    D = r2["stft"][0].cpu().numpy().T
    want = O.stft(S[0].astype(np.float64), 640, 160)
    assert np.max(np.abs(D - want)) <= 2e-5 * np.max(np.abs(want))


@pytest.mark.parametrize("L", [3200, 3333, 4001, 6400, 16100])
def test_reflect_only_edge_groups_at_awkward_lengths(eng, L):
    """Full-length utterances (no `lengths`): the first and last groups take the interior pass 1 on mirrored load indices
    (AVSE_F4_REFLECT_FAST / AVSE_I8_REFLECT_FAST).  Lengths that are not multiples of the hop, last groups of 1 ... 4 (forward)
    and 1 ... 8 (inverse) frames: forward and inverse against the oracle, float and int16 input, and the same rows bit-identical
    when the utterances carry explicit lengths == L."""
    B = 3
    rng = np.random.RandomState(L)
    S = np.stack([O.synth_speech(L, SR, 10 + i) for i in range(B)]).astype(np.float32)
    N = (0.05 * rng.randn(B, L)).astype(np.float32)
    nvs = max(1, (1 + L // 160) // 20)
    mixed, speech, noise, pcm = eng.preprocess_pairs(_dev(S), _dev(N), nvs)
    again = eng.preprocess_pairs(_dev(S), _dev(N), nvs, lengths=_dev(np.full(B, L, np.int32)))
    for a, b in zip((mixed, speech, noise, pcm), again):
        assert torch.equal(a, b)
    rec = eng.reconstruct(pcm, speech)
    for i in range(B):
        r_mixed, r_speech, r_noise, r_sig = O.preprocess_audio_pair_signals(O.AudioSignal(S[i].astype(np.float64), SR),
                                                                            O.AudioSignal(N[i].astype(np.float64), SR), 200, nvs, FPS)
        for name, got, ref in (("mixed", mixed, r_mixed), ("speech", speech, r_speech), ("noise", noise, r_noise)):
            assert np.max(np.abs(got[i].cpu().numpy() - ref)) <= TOL_DB, (i, name)
        full = np.max(np.abs(r_sig.get_data()))
        assert np.max(np.abs(pcm[i].cpu().numpy() - r_sig.get_data())) <= TOL_PCM * full
        want = O.reconstruct_speech_signal(O.AudioSignal(pcm[i].double().cpu().numpy(), SR), speech[i].double().cpu().numpy(), FPS).get_data()
        assert np.max(np.abs(rec[i].cpu().numpy()[:len(want)] - want)) <= TOL_PCM * full, (i, "inverse")
    # int16 input through the same groups
    S16 = np.round(S * 20000.0).astype(np.int16)
    N16 = np.round(N * 20000.0).astype(np.int16)
    m16, s16, n16, p16 = eng.preprocess_pairs(_dev(S16), _dev(N16), nvs)
    mf, sf, nf_, pf = eng.preprocess_pairs(_dev(S16.astype(np.float32)), _dev(N16.astype(np.float32)), nvs)
    for a, b in zip((m16, s16, n16, p16), (mf, sf, nf_, pf)):
        assert torch.equal(a, b)
