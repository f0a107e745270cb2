"""GPU tests of training windows: mix_pools(..., speech_start=...) / avse_mix_pooled with speech_start, the video gather
(SpectralEngine.gather_video / avse_gather_video) and DynamicMixer's windowed draw and sample_set.

Row b with start a is the reference's preprocess_audio_pair (dp:119-139) on the window clip[a : a + min(L, Ls - a)] and the
noise np.roll(z, -off).  Tolerances are BASELINE.json's: <= 1e-3 dB on log-mel, <= 1e-4 of full scale on PCM.
"""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_PCM = 1e-4
SR = 16000
SPS = 3200


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, 25.0, 200, device="cuda:0")


def _d(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _clips(i16, lens, seed, sr=SR, noise=False):
    scale = 20000.0 if i16 else 1.0
    out = []
    for k, n in enumerate(lens):
        x = (O.synth_noise(n, seed + k) * (3.0 if k % 2 else 0.5) if noise else O.synth_speech(n, sr, seed + k)) * scale
        out.append(np.round(x).astype(np.int16) if i16 else x.astype(np.float32))
    return out


def _pool(clips, poison):
    stride = (max(len(c) for c in clips) + 3) // 4 * 4 + 4
    P = np.full((len(clips), stride), poison, clips[0].dtype)
    for k, c in enumerate(clips):
        P[k, :len(c)] = c
    return _d(P), _d(np.array([len(c) for c in clips], np.int32))


def _poison(i16):
    return 30000 if i16 else np.nan


def _check_rows(out, sp, nz, si, ni, off, start, snr, nvs, rows, sr=SR, fps=25.0):
    mixed, speech, noise, pcm = (t.cpu().numpy() for t in out)
    L = int(sr * 0.2) * nvs
    for b in rows:
        clip, a = sp[si[b]], int(start[b])
        s = clip[a:a + min(L, len(clip) - a)].astype(np.float64)
        zr = np.roll(nz[ni[b]].astype(np.float64), -int(off[b]))
        r = O.preprocess_audio_pair_signals(O.AudioSignal(s, sr), O.AudioSignal(zr, sr), 200, nvs, fps, snr_db=float(snr[b]))
        for got, ref, name in ((mixed[b], r[0], "mixed"), (speech[b], r[1], "speech"), (noise[b], r[2], "noise")):
            assert got.shape == ref.shape, name
            err = np.max(np.abs(got - ref))
            assert err <= TOL_DB, (b, name, err)
        full = np.max(np.abs(r[3].get_data()))
        assert np.max(np.abs(pcm[b] - r[3].get_data())) <= TOL_PCM * full, b


def _draw(rng, B, sp, nz, nvs, sps, aligned=True):
    si = rng.randint(0, len(sp), B).astype(np.int64)
    ni = rng.randint(0, len(nz), B).astype(np.int64)
    off = np.array([rng.randint(0, len(nz[k])) for k in ni], np.int32)
    if aligned:
        start = np.array([sps * rng.randint(0, max(0, len(sp[k]) // sps - nvs) + 1) for k in si], np.int32)
    else:
        start = np.array([rng.randint(0, len(sp[k])) for k in si], np.int32)
    snr = np.linspace(-10, 10, B).astype(np.float32)
    return si, ni, off, start, snr


GEOMETRIES = [("16k_25", 25.0), ("16k_29.97", 30000 / 1001)]


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
@pytest.mark.parametrize("name,fps", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_windows_of_60s_clips_match_oracle(mod, eng, name, fps, i16):
    """3 s windows at random slice starts of 60 s clips (and of shorter ones: windows cut by the clip's end), per row
    against the float64 oracle; 16 kHz / 30000/1001 fps runs the generic kernels (n_fft 533)."""
    e = eng if fps == 25.0 else mod.SpectralEngine(SR, fps, 200, device="cuda:0")
    assert e.specialised == (fps == 25.0)
    sp = _clips(i16, [60 * SR, 60 * SR + 1111, 20 * SR + 7, 2 * SR + 5], 400)
    nz = _clips(i16, [50000, 7001, 3 * 60 * SR], 500, noise=True)
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    rng = np.random.RandomState(3)
    B, nvs = 14, 15
    si, ni, off, start, snr = _draw(rng, B, sp, nz, nvs, SPS)
    si[:2], start[:2] = 2, (20 * SR // SPS - 2) * SPS           # windows shorter than L at the end of the 20 s clip
    info = {}
    out = e.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), speech_start=_d(start), info=info)
    torch.cuda.synchronize()
    assert bool(info["valid"].all())
    for t in out:
        assert bool(torch.isfinite(t).all())
    _check_rows(out, sp, nz, si, ni, off, start, snr, nvs, range(B), fps=fps)


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_windows_equal_copied_windows(eng, i16):
    """The same windows copied into a pool of their own (pack_clips of clip[a : a + L]) and mixed without starts: slices and
    PCM bit-identical wherever the factors agree; the factors within 1 float32 ulp (the statistics sums run from another
    alignment, so in another order)."""
    sp = _clips(i16, [60 * SR, 31 * SR + 3], 600)
    nz = _clips(i16, [40000, 9001], 700, noise=True)
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    rng = np.random.RandomState(5)
    B, nvs = 48, 15
    L = SPS * nvs
    si, ni, off, start, snr = _draw(rng, B, sp, nz, nvs, SPS)
    start[:4] = [1, 3, 4097, 59 * SR + 1]                       # a few starts off the slice grid, the last one cut short
    si[:4] = 0
    info = {}
    got = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), speech_start=_d(start), info=info)
    copies = [sp[si[b]][start[b]:start[b] + L] for b in range(B)]
    cpP, cl = _pool(copies, _poison(i16))
    info_c = {}
    ref = eng.mix_pools(cpP, cl, nzP, nl, _d(np.arange(B)), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), info=info_c)
    torch.cuda.synchronize()
    f, fc = info["factor"], info_c["factor"]
    eps = np.finfo(np.float32).eps
    assert bool(torch.all(torch.abs(f - fc) <= torch.abs(fc) * eps))
    same = (f == fc) & (info["keys"].equalizer == info_c["keys"].equalizer)
    assert int(same.sum()) >= B // 2
    for a, b in zip(got, ref):
        assert torch.equal(a[same], b[same])


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_zero_starts_on_short_clips_equal_no_starts(eng, i16):
    """speech_start of all zeros on clips no longer than L is the whole-clip row, bit for bit."""
    nvs = 10
    L = SPS * nvs
    sp = _clips(i16, [L, L - 1, 12001, 3], 800)
    nz = _clips(i16, [5000, 40000], 900, noise=True)
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    rng = np.random.RandomState(7)
    B = 16
    si, ni, off, _, snr = _draw(rng, B, sp, nz, nvs, SPS)
    a = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr))
    b = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), speech_start=_d(np.zeros(B, np.int32)))
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_misaligned_starts_match_oracle(eng, i16):
    """Odd sample starts: the statistics pass falls back from vector loads on a misaligned window, the loaders read it
    sample by sample."""
    sp = _clips(i16, [20 * SR + 1, 7 * SR + 2], 1000)
    nz = _clips(i16, [30001, 6000], 1100, noise=True)
    spP, sl = _pool(sp, _poison(i16))
    nzP, nl = _pool(nz, _poison(i16))
    rng = np.random.RandomState(9)
    B, nvs = 10, 5
    si, ni, off, start, snr = _draw(rng, B, sp, nz, nvs, SPS, aligned=False)
    start[:5] = [1, 2, 3, 5, 3201]
    start |= 1                                                  # every start odd, inside its clip
    start = np.where(start >= np.array([len(sp[k]) for k in si]), start - 2, start).astype(np.int32)
    out = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), speech_start=_d(start))
    torch.cuda.synchronize()
    _check_rows(out, sp, nz, si, ni, off, start, snr, nvs, range(B))


def test_22k05_windows_match_oracle(mod):
    """22.05 kHz / 25 fps: 4410 samples per slice, not a multiple of 4, so slice-boundary starts are misaligned too."""
    sr = 22050
    e = mod.SpectralEngine(sr, 25.0, 200, device="cuda:0")
    sps = e.samples_per_slice
    assert sps == 4410
    sp = _clips(False, [30 * sr + 3, 5 * sr], 1200, sr=sr)
    nz = _clips(False, [50000, 9000], 1300, noise=True)
    spP, sl = _pool(sp, np.nan)
    nzP, nl = _pool(nz, np.nan)
    rng = np.random.RandomState(11)
    B, nvs = 8, 6
    si, ni, off, start, snr = _draw(rng, B, sp, nz, nvs, sps)
    start[0], si[0] = sps, 0
    start[1], si[1] = 3 * sps, 0
    out = e.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), snr_db=_d(snr), speech_start=_d(start))
    torch.cuda.synchronize()
    _check_rows(out, sp, nz, si, ni, off, start, snr, nvs, range(B), sr=sr)


def test_bad_start_raises_or_gives_the_empty_pair(eng):
    sp = _clips(False, [20000, 9000], 1400)
    nz = _clips(False, [5000], 1500, noise=True)
    spP, sl = _pool(sp, np.nan)
    nzP, nl = _pool(nz, np.nan)
    B, nvs = 6, 5
    si, ni = np.array([0, 1, 0, 1, 0, 1]), np.zeros(B, np.int64)
    off = np.full(B, 17, np.int32)
    good_start = np.array([0, 0, 3200, 6400, 16000, 100], np.int32)
    good = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), speech_start=_d(good_start))
    for bad in (-1, 9000, 9005):
        start = good_start.copy()
        start[3] = bad
        with pytest.raises(IndexError):
            eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), speech_start=_d(start))
        info = {}
        out = eng.mix_pools(spP, sl, nzP, nl, _d(si), _d(ni), nvs, noise_offset=_d(off), speech_start=_d(start), info=info, check=False)
        torch.cuda.synchronize()
        assert not bool(info["valid"][3]) and bool(info["valid"][[0, 1, 2, 4, 5]].all())
        assert float(info["factor"][3]) == 0.0
        for k in range(3):
            assert bool((out[k][3] == -100.0).all())
        assert bool((out[3][3] == 0.0).all())
        keep = [0, 1, 2, 4, 5]
        for x, y in zip(out, good):
            assert torch.equal(x[keep], y[keep])


# ---- video ----

def _video_pool(mod, dtype, seed, counts=(7, 3, 12, 1), hwf=(16, 12, 5)):
    rng = np.random.RandomState(seed)
    clips = []
    for c in counts:
        x = rng.randint(0, 256, (c,) + hwf)
        clips.append(x.astype(np.uint8) if dtype == torch.uint8 else (x + rng.rand(*x.shape)).astype(np.float32))
    return mod.pack_video(clips, "cuda:0", dtype=dtype)


@pytest.mark.parametrize("dtype", [torch.uint8, torch.float32], ids=["u8", "f32"])
def test_gather_video_matches_normalize(eng, mod, dtype):
    pool, counts = _video_pool(mod, dtype, 1)
    flat = pool.view(-1, *pool.shape[2:])
    norm = mod.VideoNormalizer(eng, flat.float())
    rows = _d(np.random.RandomState(2).randint(0, flat.shape[0], 333).astype(np.int64))
    got = eng.gather_video(pool, rows, normalizer=norm)
    want = norm.normalize(flat.float()[rows].contiguous())
    assert got.dtype == torch.float32 and got.shape == want.shape
    assert torch.equal(got, want)
    plain = eng.gather_video(pool, rows)
    assert torch.equal(plain, flat.float()[rows])


def test_gather_video_bad_index_and_sizes(eng, mod):
    pool, counts = _video_pool(mod, torch.uint8, 3)
    n_pool = pool.shape[0] * pool.shape[1]
    with pytest.raises(IndexError):
        eng.gather_video(pool, _d(np.array([0, n_pool], np.int64)))
    with pytest.raises(IndexError):
        eng.gather_video(pool, _d(np.array([-1], np.int64)))
    empty = eng.gather_video(pool, _d(np.zeros(0, np.int64)))
    assert empty.shape == (0,) + tuple(pool.shape[2:])
    small, _ = mod.pack_video([np.arange(3 * 2 * 2 * 5).reshape(3, 2, 2, 5) % 256], "cuda:0")   # 20 pixels per slice
    rows = torch.arange(70001, device="cuda:0", dtype=torch.int64) % 3
    big = eng.gather_video(small, rows)
    torch.cuda.synchronize()
    assert big.shape[0] == 70001 and torch.equal(big, small[0].float()[rows])


def _tone_clip(n_slices, sps, bank, sr, seed):
    """Speech whose slice k is a tone at the centre of mel band 10 + k (the band's heaviest filterbank bin)."""
    n_fft = 2 * (bank.shape[1] - 1)
    x = np.zeros(n_slices * sps)
    t = np.arange(sps) / sr
    for k in range(n_slices):
        f = np.argmax(bank[10 + k]) * sr / n_fft
        x[k * sps:(k + 1) * sps] = 0.3 * np.sin(2 * np.pi * f * t + seed + k)
    return x.astype(np.float32)


def test_sample_set_pairs_video_and_audio(eng, mod):
    """End to end: video slice k of every clip holds the value k + 1, speech slice k a tone in mel band 10 + k.  Every row of
    sample_set pairs video value v with a speech slice whose loudest band is 9 + v, whatever the index construction."""
    bank = eng.filterbank()
    slices = [30, 9, 17, 5, 3]                                  # clip 4 is shorter than the window: k = 0, fewer slices
    sp = [_tone_clip(c, SPS, bank, SR, k) for k, c in enumerate(slices)]
    video = [np.broadcast_to((np.arange(c) + 1).reshape(c, 1, 1, 1), (c, 8, 6, 5)).astype(np.uint8) for c in slices]
    spP, sl = mod.pack_clips(sp, eng.device)
    nzP, nl = mod.pack_clips(_clips(False, [7000, 20000], 1600, noise=True), eng.device, allow_empty=False)
    vpool = mod.pack_video(video, eng.device)
    nvs = 5
    m = mod.DynamicMixer(eng, spP, sl, nzP, nl, nvs, snr_db=30.0, seed=4, clip_slices=slices, video_pool=vpool)
    total = 0
    for _ in range(3):
        pairing = m.draw(40)
        assert len(pairing) == 5
        mixed, speech, noise, pcm, valid = m.mix(pairing)
        X_video, X_mixed, X_speech, perm = m.sample_set(pairing, mixed, speech, valid)
        torch.cuda.synchronize()
        assert X_video.shape[0] == X_speech.shape[0] == X_mixed.shape[0] == perm.numel()
        v = X_video.cpu().numpy()
        assert np.all(v == v[:, :1, :1, :1])                    # a slice is one constant
        k = v[:, 0, 0, 0].astype(np.int64) - 1
        band = np.argmax(np.median(X_speech.cpu().numpy(), axis=2), axis=1)
        assert np.array_equal(band, 10 + k)
        total += len(k)
        si = pairing[0].cpu().numpy()
        want = sum(min(slices[s], nvs) for s in si)
        assert X_video.shape[0] == want
    assert total > 0


def test_sample_set_is_deterministic_and_normalised(eng, mod):
    """Two mixers with the same seed (and permutation generators with the same seed) give bit-identical sample sets; the
    normalised video equals normalize() of the decoded rows."""
    slices = [40, 12, 25]
    sp = _clips(False, [c * SPS + 11 for c in slices], 1700)
    spP, sl = mod.pack_clips(sp, eng.device)
    nzP, nl = mod.pack_clips(_clips(False, [9000, 30000], 1800, noise=True), eng.device, allow_empty=False)
    rng = np.random.RandomState(5)
    video = [rng.randint(0, 256, (c, 8, 8, 5)).astype(np.uint8) for c in slices]
    vpool = mod.pack_video(video, eng.device)
    norm = mod.VideoNormalizer(eng, vpool[0].view(-1, 8, 8, 5).float())

    def run():
        m = mod.DynamicMixer(eng, spP, sl, nzP, nl, 15, seed=77, clip_slices=slices, video_pool=vpool)
        g = torch.Generator(device=eng.device)
        g.manual_seed(5)
        res = []
        for _ in range(2):
            p = m.draw(9)
            mixed, speech, noise, pcm, valid = m.mix(p)
            res.append(tuple(t.clone() for t in m.sample_set(p, mixed, speech, valid, normalizer=norm, generator=g)) + (p,))
        return res

    a, b = run(), run()
    for ra, rb in zip(a, b):
        for x, y in zip(ra[:4], rb[:4]):
            assert torch.equal(x, y)
    X_video, _, _, perm, p = a[0]
    si, k = p[0], p[4].long() // SPS
    nb = (torch.tensor(slices, device=eng.device)[si] - k).clamp(0, 15)
    idx = mod.video_slice_index(si, k, nb, 15, vpool[0].shape[1], perm)
    want = norm.normalize(vpool[0].view(-1, 8, 8, 5).float()[idx].contiguous())
    assert torch.equal(X_video, want)
