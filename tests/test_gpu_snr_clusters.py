"""The SNR statistics pass (avse_snr_factor_kernel<S, CLUSTER>, csrc/avse_kernels.cu) at every cluster size it launches.

A long utterance is split over P = 1, 2, 4 or 8 CTAs of a thread-block cluster (snr_factor_launch, mirrored by
tests.longform_cases.cluster_size): each CTA sums its share of every range the pair reads and rank 0 gathers the partials over
distributed shared memory.  One sample dropped or counted twice moves a 60 s row's variance by about 1e-6 -- invisible at 1e-3 dB
or 1e-4 of the peak, about 10 float32 ulps of the factor.  So every row carries spikes of 30 (speech) / 12 (noise) times its std
on both sides of every CTA boundary, at the start of the scalar tail, at the last sample and, in noise rows, at the wrap point
and the periodic weight step, each computed from the pass's own per4 / perp arithmetic for the row's P and alignment: such an
error then moves the factor by ~1e-3 relative.  The gate is test_gpu_offsets.py's: factor and equaliser within 2e-7 relative of
numpy's float64 sqrt(var_s / var_n) 10^(-snr/20) and sqrt(sum s^2 / sum n^2) over exactly the samples the reference reads
(dp:125-130).  Samples past every row's length are poison (NaN / int16 -32768)."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import FRAME_RATES, FPS
from tests.longform_cases import (POOL_NOISE, POOL_ROWS, POOL_SPEECH, SECONDS_FOR_P, SPIKE_N, SPIKE_S, SR, aligned, base_row,
                                  build_pools, check_gains, cluster_size, gains_ref, num_sms, periodic_spikes, pool_row_noise,
                                  range_spikes, spike)

pytestmark = pytest.mark.gpu

PS = [1, 2, 4, 8]
TOL_DB, TOL_PCM = 1e-3, 1e-4
GENERIC = next(g for g in FRAME_RATES if g["name"] == "22k05_29.97")


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


@pytest.fixture(scope="module")
def sms():
    return num_sms()


def _report(what, ulps):
    """Prints the worst (factor, equaliser) error of a batch in float32 ulps (run with -s)."""
    print("%s: worst factor / equaliser error %.2f / %.2f ulp" % (what, max(u[0] for u in ulps), max(u[1] for u in ulps)))


def _form_lengths(L, P):
    """Full length; n mod 4 = 3, 2, 1; a short row inside the long batch; n < 4 P (CTAs without a share); 5; empty."""
    return [L, L - 1, L - 2, L - 3, 2 * L // 3 + 1, 1001, max(4 * P - 1, 3), 5, 0]


def _tiled_rows(L, P):
    """(n, Pn): Pn < P, Pn odd and not a multiple of 4, Pn just below n, Pn = n."""
    return [(L, max(P - 1, 3)), (L, 27371), (L - 1, 4099), (L - 3, L - 4), (L - 2, L - 2), (2 * L // 3 + 1, 12347)]


def _alloc(B, L, dt, layout):
    """[B, L] device view: contiguous, an odd row stride (a view of a wider buffer) or a storage offset of one sample."""
    if layout == "contiguous":
        return torch.empty((B, L), dtype=dt, device="cuda")
    if layout == "odd_stride":
        return torch.empty((B, L + 1), dtype=dt, device="cuda")[:, :L]
    return torch.empty(B * L + 1, dtype=dt, device="cuda")[1:].view(B, L)


def _identity_batch(rows, L, P, i16, layout="contiguous", seed=0):
    """Device views (S, Z) with the rows (n, Pn or None) spiked at the statistics pass's partition points, and their host copies.
    Identity rows read speech and noise with one joint alignment test per row."""
    B = len(rows)
    dt = torch.int16 if i16 else torch.float32
    esize = 2 if i16 else 4
    S, Z = _alloc(B, L, dt, layout), _alloc(B, L, dt, layout)
    poison = -32768 if i16 else np.nan
    hS = np.full((B, L), poison, np.float64)
    hZ = np.full((B, L), poison, np.float64)
    for u, (n, Pn) in enumerate(rows):
        ps, pz = S.data_ptr() + u * S.stride(0) * esize, Z.data_ptr() + u * Z.stride(0) * esize
        vec = aligned(ps, esize) and aligned(pz, esize)
        s, ssd = base_row(n, seed + 10 * u, i16)
        spike(s, range_spikes(n, vec, P), SPIKE_S * ssd)
        m = n if Pn is None else Pn
        z, zsd = base_row(m, seed + 10 * u + 5, i16, noise=True)
        spike(z, range_spikes(n, vec, P) if Pn is None or Pn >= n else periodic_spikes(Pn, n, 0, P), SPIKE_N * zsd)
        hS[u, :n], hZ[u, :m] = s, z
    np_dt = np.int16 if i16 else np.float32
    hS, hZ = hS.astype(np_dt), hZ.astype(np_dt)
    S.copy_(torch.from_numpy(hS))
    Z.copy_(torch.from_numpy(hZ))
    return S, Z, hS, hZ


def _check_identity(factor, eq, rows, hS, hZ, snr, what):
    ulps = []
    for u, (n, Pn) in enumerate(rows):
        m = n if Pn is None else min(Pn, n)
        nseq = hZ[u, :m][np.arange(n) % m] if n else hZ[u, :0]
        wf, wg = gains_ref(hS[u, :n], nseq, snr[u])
        ulps.append(check_gains(float(factor[u]), float(eq[u]), wf, wg, (what, u, n, Pn)))
    _report(what, ulps)


def _snr(B):
    return np.array([(-10.0, -3.5, 0.0, 4.25, 10.0)[u % 5] for u in range(B)], np.float32)


def test_parametrisation_reaches_every_cluster_size(sms):
    """P is not observable from outside: every row form's (B, L) must give P = 1, 2, 4 and 8 under the launcher's rule."""
    forms = {"forms": 9, "unaligned": 9, "tiled": 6}
    for name, B in forms.items():
        got = {P: cluster_size(B, SECONDS_FOR_P[P] * SR, sms) for P in PS}
        assert got == {P: P for P in PS}, (name, sms, got)
    assert cluster_size(len(POOL_ROWS), (max(POOL_SPEECH) + 3) // 4 * 4, sms) == 8
    assert cluster_size(len(POOL_ROWS), max(POOL_SPEECH) | 1, sms) == 8
    assert cluster_size(9, 60 * GENERIC["sr"], sms) == 8
    print("%d SMs: forms / unaligned / tiled rows at P = 1, 2, 4, 8; pools and the generic context at P = 8" % sms)


@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_row_forms(eng, sms, P, i16):
    """Full-length, ragged (n mod 4 = 1, 2, 3), short, n < 4 P, tiny and empty rows in one batch."""
    L = SECONDS_FOR_P[P] * SR
    lens = _form_lengths(L, P)
    rows = [(n, None) for n in lens]
    assert cluster_size(len(rows), L, sms) == P
    S, Z, hS, hZ = _identity_batch(rows, L, P, i16, seed=100 + P)
    snr = _snr(len(rows))
    factor, keys = eng.snr_factor(S, Z, lengths=torch.tensor(lens, dtype=torch.int32), snr_db=torch.from_numpy(snr))
    f, e = factor.cpu().numpy(), keys.equalizer.cpu().numpy()
    assert f[-1] == 0.0 and e[-1] == 0.0          # the empty row
    _check_identity(f, e, rows, hS, hZ, snr, ("forms", P, i16))


@pytest.mark.parametrize("layout", ["odd_stride", "offset1"])
@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_unaligned_rows(eng, sms, P, i16, layout):
    """Rows that are not 4-sample aligned take the all-scalar path on the last CTA: an odd row stride (every other row is
    unaligned) and a storage offset of one sample (every row is)."""
    L = SECONDS_FOR_P[P] * SR
    lens = _form_lengths(L, P)
    rows = [(n, None) for n in lens]
    assert cluster_size(len(rows), L, sms) == P
    S, Z, hS, hZ = _identity_batch(rows, L, P, i16, layout=layout, seed=200 + P)
    esize = 2 if i16 else 4
    n_unaligned = sum(not aligned(S.data_ptr() + u * S.stride(0) * esize, esize) for u in range(len(rows)))
    assert n_unaligned >= (len(rows) if layout == "offset1" else len(rows) // 2)
    snr = _snr(len(rows))
    factor, keys = eng.snr_factor(S, Z, lengths=torch.tensor(lens, dtype=torch.int32), snr_db=torch.from_numpy(snr))
    _check_identity(factor.cpu().numpy(), keys.equalizer.cpu().numpy(), rows, hS, hZ, snr, ("unaligned", layout, P, i16))


@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_tiled_noise(eng, sms, P, i16):
    """noise_lengths (dp:125-128 tiling in the kernel): the periodic regime's weighted pass over parts of ceil(Pn / P)."""
    L = SECONDS_FOR_P[P] * SR
    rows = _tiled_rows(L, P)
    assert cluster_size(len(rows), L, sms) == P
    S, Z, hS, hZ = _identity_batch(rows, L, P, i16, seed=300 + P)
    snr = _snr(len(rows))
    factor, keys = eng.snr_factor(S, Z, lengths=torch.tensor([r[0] for r in rows], dtype=torch.int32), snr_db=torch.from_numpy(snr),
                                  noise_lengths=torch.tensor([r[1] for r in rows], dtype=torch.int32))
    _check_identity(factor.cpu().numpy(), keys.equalizer.cpu().numpy(), rows, hS, hZ, snr, ("tiled", P, i16))


@pytest.mark.parametrize("layout,i16", [("offset1", False), ("odd_stride", True)], ids=["f32_offset1", "i16_odd_stride"])
def test_unaligned_rows_through_preprocess_pairs(eng, sms, layout, i16):
    """The same unaligned views through preprocess_pairs at P = 2.  The forward kernels read samples with scalar loads (the
    only vector loads of inputs are the statistics pass's Sample4, behind its alignment test), so no alignment is required:
    the factor is gated as above and the outputs against the float64 oracle."""
    P = 2
    L = SECONDS_FOR_P[P] * SR
    lens = [L, L - 3, 1001]
    rows = [(n, None) for n in lens]
    assert cluster_size(len(rows), L, sms) == P
    S, Z, hS, hZ = _identity_batch(rows, L, P, i16, layout=layout, seed=400)
    snr = _snr(len(rows))
    info = {}
    got = eng.preprocess_pairs(S, Z, L // 3200, lengths=torch.tensor(lens, dtype=torch.int32), snr_db=torch.from_numpy(snr), info=info)
    _check_identity(info["factor"].cpu().numpy(), info["keys"].equalizer.cpu().numpy(), rows, hS, hZ, snr, ("preprocess_pairs", layout, i16))
    got = [t.cpu().numpy() for t in got]
    for u in (0, 1):
        n = lens[u]
        s, z = hS[u, :n].astype(np.float64), hZ[u, :n].astype(np.float64)
        r = O.preprocess_audio_pair_signals(O.AudioSignal(s, SR), O.AudioSignal(z, SR), 200, L // 3200, FPS, snr_db=float(snr[u]))
        db = max(float(np.max(np.abs(got[k][u] - r[k]))) for k in range(3))
        ref_pcm = r[3].get_data()
        pcm = float(np.max(np.abs(got[3][u] - ref_pcm)) / np.max(np.abs(ref_pcm)))
        assert db <= TOL_DB and pcm <= TOL_PCM, (u, db, pcm)


@pytest.mark.parametrize("odd_stride", [False, True], ids=["pack_clips", "odd_stride"])
@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_mix_pools_under_a_cluster(mod, eng, sms, i16, odd_stride):
    """mix_pools with a 40 s speech clip in the pool: every row runs at P = 8.  Window and periodic regimes, wrapping windows,
    odd offsets, offsets 0, 1 and Ln - 1, Ln = n and n - 1, a 31-sample clip; with an odd pool stride odd clips start unaligned.
    The log-mels and PCM of every row against the oracle at 3 s (the statistics are over the whole clip, dp:130)."""
    P = 8
    sp, slen, nz, nlen, sclips, nclips = build_pools(mod, i16, odd_stride, P)
    assert cluster_size(len(POOL_ROWS), sp.stride(0), sms) == P
    si = torch.tensor([r[0] for r in POOL_ROWS])
    ni = torch.tensor([r[1] for r in POOL_ROWS])
    off = torch.tensor([r[2] for r in POOL_ROWS], dtype=torch.int32)
    snr = _snr(len(POOL_ROWS))
    info = {}
    got = eng.mix_pools(sp, slen, nz, nlen, si, ni, 15, noise_offset=off, snr_db=torch.from_numpy(snr), info=info)
    f, e = info["factor"].cpu().numpy(), info["keys"].equalizer.cpu().numpy()
    got = [t.cpu().numpy() for t in got]
    ulps = []
    for b, (s_k, n_k, o) in enumerate(POOL_ROWS):
        s = sclips[s_k].astype(np.float64)
        z = nclips[n_k].astype(np.float64)
        nseq = pool_row_noise(z, POOL_NOISE[n_k], o, len(s))
        wf, wg = gains_ref(s, nseq, snr[b])
        ulps.append(check_gains(float(f[b]), float(e[b]), wf, wg, ("pool", b)))
        r = O.preprocess_audio_pair_signals(O.AudioSignal(s, SR), O.AudioSignal(np.roll(z, -o), SR), 200, 15, FPS, snr_db=float(snr[b]))
        db = max(float(np.max(np.abs(got[k][b] - r[k]))) for k in range(3))
        ref_pcm = r[3].get_data()
        pcm = float(np.max(np.abs(got[3][b] - ref_pcm)) / np.max(np.abs(ref_pcm)))
        assert db <= TOL_DB and pcm <= TOL_PCM, (b, db, pcm)
    _report(("mix_pools", odd_stride, i16), ulps)


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_mix_pools_invalid_row_under_a_cluster(mod, eng, i16):
    """An offset equal to its clip's length (outside [0, Ln)) makes its row invalid: factor and equaliser 0, the flag raised, and
    every other row bit-identical to the batch with a valid row in its place."""
    sp, slen, nz, nlen, _, _ = build_pools(mod, i16, False, 8)
    rows = list(POOL_ROWS)
    bad = 4
    si = torch.tensor([r[0] for r in rows])
    ni = torch.tensor([r[1] for r in rows])
    off_ok = torch.tensor([r[2] for r in rows], dtype=torch.int32)
    off_bad = off_ok.clone()
    off_bad[bad] = POOL_NOISE[rows[bad][1]]
    snr = torch.from_numpy(_snr(len(rows)))
    out_ok, out_bad, info_ok, info_bad = {}, {}, {}, {}
    ok = eng.mix_pools(sp, slen, nz, nlen, si, ni, 15, noise_offset=off_ok, snr_db=snr, out=out_ok, info=info_ok)
    got = eng.mix_pools(sp, slen, nz, nlen, si, ni, 15, noise_offset=off_bad, snr_db=snr, out=out_bad, info=info_bad, check=False)
    assert int(out_bad["bad_row_flag"].item()) == 1 and int(out_ok["bad_row_flag"].item()) == 0
    assert float(info_bad["factor"][bad]) == 0.0 and float(info_bad["keys"].equalizer[bad]) == 0.0
    assert not bool(info_bad["valid"][bad])
    keep = [b for b in range(len(rows)) if b != bad]
    assert torch.equal(info_bad["factor"][keep], info_ok["factor"][keep])
    assert torch.equal(info_bad["keys"].equalizer[keep], info_ok["keys"].equalizer[keep])
    for a, b in zip(got, ok):
        assert torch.equal(a[keep], b[keep])
    assert torch.all(got[3][bad] == 0.0)
    with pytest.raises(IndexError):
        eng.mix_pools(sp, slen, nz, nlen, si, ni, 15, noise_offset=off_bad, snr_db=snr)


@pytest.mark.parametrize("i16", [False, True], ids=["f32", "i16"])
def test_generic_context_at_60s(mod, sms, i16):
    """A generic-geometry context (22.05 kHz at 29.97 fps) runs the same statistics kernel with its own L: 60 s rows, P = 8."""
    e = mod.SpectralEngine(GENERIC["sr"], GENERIC["fps"], 200, device="cuda:0")
    assert not e.specialised
    L = 60 * GENERIC["sr"]
    P = 8
    lens = _form_lengths(L, P)
    rows = [(n, None) for n in lens]
    assert cluster_size(len(rows), L, sms) == P
    S, Z, hS, hZ = _identity_batch(rows, L, P, i16, seed=500)
    snr = _snr(len(rows))
    factor, keys = e.snr_factor(S, Z, lengths=torch.tensor(lens, dtype=torch.int32), snr_db=torch.from_numpy(snr))
    _check_identity(factor.cpu().numpy(), keys.equalizer.cpu().numpy(), rows, hS, hZ, snr, ("generic", i16))

