"""GPU tests of pooled-pair mixing (SpectralEngine.mix_pools / avse_mix_pooled, DynamicMixer).

Row b mixes speech clip speech_index[b] with noise clip noise_index[b] read from sample noise_offset[b] on, wrapped around
its length: the reference's preprocess_audio_pair (dp:119-139) on (s, np.roll(z, -off)).  Tolerances are BASELINE.json's:
<= 1e-3 dB on log-mel, <= 1e-4 of full scale on PCM.
"""
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS, FRAME_RATES, frame_rate_fps

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
SPEECH_LENS = [32000, 20000, 35000, 25000, 31999, 12001]
NOISE_LENS = [5000, 1121, 640, 40000, 32000, 7, 50000, 2049]


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


def _d(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _clips(i16, sr=SR, speech_lens=SPEECH_LENS, noise_lens=NOISE_LENS, seed=0):
    scale = 20000.0 if i16 else 1.0
    dt = np.int16 if i16 else np.float32
    sp, nz = [], []
    for k, n in enumerate(speech_lens):
        x = O.synth_speech(n, sr, seed + 50 + k) * scale
        sp.append(np.round(x).astype(dt) if i16 else x.astype(dt))
    for k, n in enumerate(noise_lens):
        x = O.synth_noise(n, seed + 70 + k) * scale * (3.0 if k % 2 else 0.2)
        nz.append(np.round(x).astype(dt) if i16 else x.astype(dt))
    return sp, nz


def _pool(clips, poison):
    """[N, stride] pool (stride a multiple of 4), everything past each clip's length = `poison`."""
    stride = (max(len(c) for c in clips) + 3) // 4 * 4 + 4
    P = np.full((len(clips), stride), poison, clips[0].dtype)
    for k, c in enumerate(clips):
        P[k, :len(c)] = c
    return _d(P), _d(np.array([len(c) for c in clips], np.int32))


def _poison(i16):
    return 30000 if i16 else np.nan


def _pairing(rng, B, noise_lens, n_speech):
    si = rng.randint(0, n_speech, B).astype(np.int64)
    ni = rng.randint(0, len(noise_lens), B).astype(np.int64)
    off = np.array([rng.randint(0, noise_lens[k]) for k in ni], np.int32)
    for b in range(min(B, 6)):           # pinned phases: 0, Ln - 1 and a wrap near the middle of the speech
        off[b] = (0, noise_lens[ni[b]] - 1, noise_lens[ni[b]] // 2)[b % 3]
    snr = np.linspace(-10, 10, B).astype(np.float32)
    return si, ni, off, snr


def _oracle_row(s, z, off, nvs, snr, sr=SR, fps=FPS):
    zr = np.roll(z.astype(np.float64), -int(off))
    return O.preprocess_audio_pair_signals(O.AudioSignal(s.astype(np.float64), sr), O.AudioSignal(zr, sr), 200, nvs, fps, snr_db=float(snr))


def _check_rows(out, sp, nz, si, ni, off, snr, nvs, rows, sr=SR, fps=FPS):
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in out)
    for b in rows:
        if len(nz[ni[b]]) < 16:
            continue        # a period of a few samples is a line spectrum with > 80 dB valleys: float32 FFT territory (see test 2)
        r = _oracle_row(sp[si[b]], nz[ni[b]], off[b], nvs, snr[b], sr, fps)
        for got, ref, name in ((mixed[b], r[0], "mixed"), (speech[b], r[1], "speech"), (noise[b], r[2], "noise")):
            assert got.shape == ref.shape, name
            err = np.max(np.abs(got - ref))
            assert err <= TOL_DB, (b, name, err)
        full = np.max(np.abs(r[3].get_data()))
        assert np.max(np.abs(pcm[b] - r[3].get_data())) <= TOL_PCM * full, b


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_pooled_rows_match_oracle_and_ignore_pool_padding(eng, i16):
    """Tests 1 and 3: every row against its own float64 oracle; pools poisoned past every clip (NaN / 30000) give finite
    outputs bit-identical to zero-padded pools."""
    sp, nz = _clips(i16)
    rng = np.random.RandomState(7)
    B, nvs = 30, 10
    si, ni, off, snr = _pairing(rng, B, NOISE_LENS, len(sp))
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    info = {}
    got = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), info=info)
    torch.cuda.synchronize()
    for t in got:
        assert torch.isfinite(t).all()
    assert bool(info["valid"].all())
    _check_rows(got, sp, nz, si, ni, off, snr, nvs, range(B))
    sp0, _ = _pool(sp, 0)
    nz0, _ = _pool(nz, 0)
    clean = eng.mix_pools(sp0, sl, nz0, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr))
    for a, b in zip(got, clean):
        assert torch.equal(a, b)


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_same_arithmetic_as_the_copy_path(eng, mod, i16):
    """Test 2: each pairing materialised (speech row copy, rolled + tiled noise) through forward_raw + floor3_ with the pooled
    call's own factor and equaliser: bit-identical slices and PCM; the factors agree to 1 float32 ulp (the float64 sums are
    reordered).  With every offset 0, the pooled call is bit-identical to preprocess_pairs(..., noise_lengths=...)."""
    sp, nz = _clips(i16, seed=3)
    rng = np.random.RandomState(11)
    B, nvs = 24, 10
    L = 3200 * nvs
    si, ni, off, snr = _pairing(rng, B, NOISE_LENS, len(sp))
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    info = {}
    got = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), info=info)
    W = max(SPEECH_LENS) + 4
    dt = np.int16 if i16 else np.float32
    S = np.zeros((B, W), dt)
    N = np.zeros((B, W), dt)
    for b in range(B):
        s, z = sp[si[b]], nz[ni[b]]
        S[b, :len(s)] = s
        N[b, :len(s)] = z[(off[b] + np.arange(len(s))) % len(z)]
    lens = _d(np.array([len(sp[k]) for k in si], np.int32))
    f_copy, _ = eng.snr_factor(_d(S), _d(N), lengths=lens, snr_db=_d(snr))
    f_pool = info["factor"]
    assert torch.all(torch.abs(f_pool - f_copy) <= torch.abs(f_copy) * np.finfo(np.float32).eps)
    keys = mod.DbKeys(B, eng.device)
    keys.equalizer = info["keys"].equalizer.clone()
    eng._lib.avse_reset_max(eng._ctx, keys.max.data_ptr(), keys.min.data_ptr(), 3 * B, eng._stream())
    n = got[0].shape[1]
    r = eng.forward_raw(_d(S), _d(N), L=L, len_speech=lens, len_noise=lens, factor=f_pool.clone(), n_slices=n, max_key=keys,
                        noise_lengths=lens)
    eng.floor3_(r["speech"], r["noise"], r["mixed"], keys)
    for a, b in zip(got, (r["mixed"], r["speech"], r["noise"], r["mixed_pcm"])):
        assert torch.equal(a, b)
    # every offset 0: the reference's own rule, bit-identical to the in-kernel tiling of preprocess_pairs
    zero = np.zeros(B, np.int32)
    Z = np.zeros((B, W), dt)
    for b in range(B):
        z = nz[ni[b]]
        m = min(len(z), W)
        Z[b, :m] = z[:m]
    nlens = _d(np.array([min(len(nz[k]), W) for k in ni], np.int32))
    p0 = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(zero), snr_db=_d(snr))
    c0 = eng.preprocess_pairs(_d(S), _d(Z), nvs, lengths=lens, snr_db=_d(snr), noise_lengths=nlens)
    for a, b in zip(p0, c0):
        assert torch.equal(a, b)


def test_invalid_rows_flag_and_empty_pair(eng):
    """Test 4: out-of-range speech / noise index, negative offset, offset >= Ln, an empty noise clip under a non-empty speech:
    the flag is raised, the row is the empty pair, every other row is bit-identical to a launch without the bad rows."""
    sp, nz = _clips(False, seed=5)
    nz = nz + [np.zeros(0, np.float32)]                   # pool clip 8: empty
    lens_n = [len(z) for z in nz]
    spP, sl = _pool(sp, np.nan)
    nzP = np.full((len(nz), max(lens_n) + 4), np.nan, np.float32)
    for k, z in enumerate(nz):
        nzP[k, :len(z)] = z
    nzP, nl = _d(nzP), _d(np.array(lens_n, np.int32))
    rng = np.random.RandomState(13)
    B, nvs = 12, 5
    si, ni, off, snr = _pairing(rng, B, NOISE_LENS, len(sp))
    good = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr))
    bad = [(len(sp), 0, 0), (-1, 0, 0), (0, len(nz), 0), (0, -3, 0), (1, 0, -1), (1, 0, NOISE_LENS[0]), (2, len(nz) - 1, 0)]
    for (s_i, n_i, o) in bad:
        si2 = np.insert(si, 5, s_i)
        ni2 = np.insert(ni, 5, n_i)
        off2 = np.insert(off, 5, o)
        snr2 = np.insert(snr, 5, 3.0)
        with pytest.raises(IndexError):
            eng.mix_pools(spP, sl, nzP, nl, _d(si2), _d(ni2), nvs, noise_offset=_d(off2), snr_db=_d(snr2))
        info = {}
        out = eng.mix_pools(spP, sl, nzP, nl, _d(si2), _d(ni2), nvs, noise_offset=_d(off2), snr_db=_d(snr2), info=info, check=False)
        torch.cuda.synchronize()
        assert float(info["factor"][5]) == 0.0 and not bool(info["valid"][5])
        assert bool(info["valid"][:5].all()) and bool(info["valid"][6:].all())
        for k in range(3):
            assert bool((out[k][5] == -100.0).all())
            assert torch.equal(out[k][:5], good[k][:5]) and torch.equal(out[k][6:], good[k][5:])
        assert bool((out[3][5] == 0.0).all())
        assert torch.equal(out[3][:5], good[3][:5]) and torch.equal(out[3][6:], good[3][5:])


def test_partition_independence(eng):
    """Test 5: one launch of B rows == two launches of B / 2, bit for bit."""
    sp, nz = _clips(False, seed=9)
    spP, sl = _pool(sp, np.nan)
    nzP, nl = _pool(nz, np.nan)
    rng = np.random.RandomState(17)
    B, nvs = 64, 10
    si, ni, off, snr = (_d(x) for x in _pairing(rng, B, NOISE_LENS, len(sp)))
    whole = eng.mix_pools(spP, sl, nzP, nl, si, ni, nvs, noise_offset=off, snr_db=snr)
    h = B // 2
    a = eng.mix_pools(spP, sl, nzP, nl, si[:h], ni[:h], nvs, noise_offset=off[:h], snr_db=snr[:h])
    b = eng.mix_pools(spP, sl, nzP, nl, si[h:], ni[h:], nvs, noise_offset=off[h:], snr_db=snr[h:])
    for w, x, y in zip(whole, a, b):
        assert torch.equal(w, torch.cat([x, y]))


def test_scale_70k_rows_from_small_pools(eng):
    """Test 6: 70 000 rows drawn from 8 speech x 5 noise clips in one launch, oracle spot checks."""
    sl_ = [16000, 12000, 17000, 15999, 9000, 16000, 14000, 16500]
    nl_ = [5000, 30000, 16000, 2049, 64000]
    sp, nz = _clips(False, speech_lens=sl_, noise_lens=nl_, seed=21)
    spP, sl = _pool(sp, np.nan)
    nzP, nl = _pool(nz, np.nan)
    rng = np.random.RandomState(23)
    B, nvs = 70000, 5
    si, ni, off, snr = _pairing(rng, B, nl_, len(sp))
    info = {}
    out = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), info=info)
    torch.cuda.synchronize()
    assert bool(info["valid"].all())
    for t in out:
        assert bool(torch.isfinite(t).all())
    rows = [0, 1, 2, 12345, 40000, 69999]
    _check_rows([t[rows] for t in out], sp, nz, si[rows], ni[rows], off[rows], snr[rows], nvs, range(len(rows)))


OTHER_CONTEXTS = [("f2", 16000, 25.0), ("n320", 16000, 50.0), ("n533", 16000, 30.0), ("n1764", 44100, 25.0)] + \
    [(g["name"], g["sr"], frame_rate_fps(g)) for g in FRAME_RATES]


@pytest.mark.parametrize("name,sr,fps", OTHER_CONTEXTS, ids=[c[0] for c in OTHER_CONTEXTS])
def test_other_contexts_match_oracle(mod, name, sr, fps):
    """Test 7: the 2-frame kernel (AVSE_FORCE_F2=1) and the generic-geometry kernels serve pooled pairs too."""
    prev = os.environ.get("AVSE_FORCE_F2")
    if name == "f2":
        os.environ["AVSE_FORCE_F2"] = "1"
    try:
        e = mod.SpectralEngine(sr, fps, 200, device="cuda:0")
    finally:
        if prev is None:
            os.environ.pop("AVSE_FORCE_F2", None)
        else:
            os.environ["AVSE_FORCE_F2"] = prev
    assert e.specialised == (name == "f2")
    k = sr / 16000.0
    sl_ = [int(20000 * k), int(14000 * k) + 3, int(22000 * k)]
    nl_ = [int(5000 * k), int(30000 * k), int(19000 * k) + 1]
    sp, nz = _clips(False, sr=sr, speech_lens=sl_, noise_lens=nl_, seed=31)
    spP, sl = _pool(sp, np.nan)
    nzP, nl = _pool(nz, np.nan)
    rng = np.random.RandomState(29)
    B, nvs = 8, 6
    si, ni, off, snr = _pairing(rng, B, nl_, len(sp))
    off[6] = 1                       # rows 0-5 pin offsets 0, Ln - 1 and Ln // 2
    out = e.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr))
    torch.cuda.synchronize()
    _check_rows(out, sp, nz, si, ni, off, snr, nvs, range(B), sr, fps)


def test_dynamic_mixer_epochs(eng, mod):
    """Test 8: the same seed gives bit-identical epochs, another seed other pairings; rows whose factor is not finite (a
    silent noise clip) are marked not valid and drop out of the make_sample_set chain."""
    sp, nz = _clips(False, seed=41)
    nz = nz[:4] + [np.zeros(3000, np.float32)]              # a silent clip: var 0 -> inf factor, like numpy
    spP, sl = mod.pack_clips(sp, eng.device)
    nzP, nl = mod.pack_clips(nz, eng.device, allow_empty=False)
    nvs = 10
    clip_slices = torch.tensor([min(nvs, len(s) // 3200 + 1) for s in sp], device=eng.device)

    def run(seed):
        m = mod.DynamicMixer(eng, spP, sl, nzP, nl, nvs, snr_db=(-10.0, 10.0), seed=seed)
        res = []
        for _ in range(2):
            pairing = m.draw(40)
            mixed, speech, noise, pcm, valid = m.mix(pairing)
            res.append((pairing, mixed.clone(), speech.clone(), pcm.clone(), valid.clone()))
        return res

    def same(x, y):         # bit for bit, NaN where NaN (the rows that drew the silent clip)
        return torch.equal(torch.isnan(x), torch.isnan(y)) and torch.equal(torch.nan_to_num(x, nan=0.0), torch.nan_to_num(y, nan=0.0))

    a, b, c = run(1), run(1), run(2)
    for ea, eb in zip(a, b):
        for x, y in zip(ea[0], eb[0]):
            assert torch.equal(x, y)
        for x, y in zip(ea[1:], eb[1:]):
            assert same(x, y) if x.is_floating_point() else torch.equal(x, y)
    assert not torch.equal(a[0][0][1], c[0][0][1]) or not torch.equal(a[0][0][2], c[0][0][2])
    pairing, mixed, speech, pcm, valid = a[0]
    assert bool((valid == (pairing[1] != 4)).all())       # exactly the rows that drew the silent clip are not valid
    n = torch.where(valid, clip_slices[pairing[0]], torch.zeros_like(clip_slices[pairing[0]]))
    X_mixed, X_speech, perm = eng.make_sample_set(mixed, speech, n_slices=n)
    assert X_mixed.shape[0] == int(n.sum()) and bool(torch.isfinite(X_mixed).all()) and bool(torch.isfinite(X_speech).all())
