"""Shared inputs of the long-form tests (tests/test_gpu_snr_clusters.py, tests/test_gpu_longform_forms.py): the statistics pass's
cluster-size rule, the sample positions where its work changes hands, spiked rows and the clip pools that run under a cluster."""
import numpy as np
import torch

SR = 16000
L60 = 60 * SR                     # 960 000 samples: T = 6 001 frames, 300 slices
SECONDS_FOR_P = {1: 5, 2: 10, 4: 20, 8: 60}     # row lengths that give P = 1 / 2 / 4 / 8 for a small batch (cluster_size)
SPIKE_S, SPIKE_N = 30.0, 12.0     # spike heights in row stds: different for speech and noise, so that a dropped or repeated
                                  # spike moves var_s / var_n (and sum s^2 / sum n^2) instead of cancelling in the ratio
TOL_GAIN = 2e-7                   # factor and equaliser: float32 rounding of the float64 statistics


def cluster_size(B, L, num_sms):
    """The statistics pass's cluster size, mirrored from snr_factor_launch (csrc/avse_kernels.cu): P doubles while P < 8,
    B P < 4 num_sms and L / (2 P) >= 65 536 (L: the row width, or the speech pool's stride for mix_pools).  A change to that
    rule has to be made here too."""
    P = 1
    while P < 8 and B * P < 4 * num_sms and L // (2 * P) >= 65536:
        P *= 2
    return P


def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def aligned(ptr, esize):
    """The alignment test of the statistics pass: a range is read with 4-sample vector loads when its start is 4-sample aligned."""
    return ptr % (4 * esize) == 0


def range_cuts(length, vec, P):
    """Where range_sums (csrc/avse_kernels.cu) hands a range [0, length) from one CTA to the next: the CTA boundaries 4 k per4
    (per4 = ceil(n4 / P) groups of four, n4 = 0 for an unaligned range), the start of the scalar tail 4 n4 and the end."""
    n4 = length // 4 if vec else 0
    per4 = -(-n4 // P)
    return {4 * k * per4 for k in range(1, P)} | {4 * n4, length}


def range_spikes(length, vec, P):
    """Both sides of every cut of range_cuts, the first and the last sample, inside [0, length)."""
    pos = {0, length - 1}
    for c in range_cuts(length, vec, P):
        pos |= {c - 1, c}
    return {p for p in pos if 0 <= p < length}


def periodic_spikes(Pn, n, off, P):
    """The periodic regime (a noise period Pn shorter than the speech, n = q Pn + rem): the weighted pass splits the period in
    parts of perp = ceil(Pn / P) samples; the wrap point (Pn - 1, 0) and the weight step ((off + rem - 1) mod Pn, (off + rem)
    mod Pn) sit inside it."""
    perp = -(-Pn // P)
    rem = n % Pn
    pos = {0, Pn - 1, (off + rem - 1) % Pn, (off + rem) % Pn}
    for k in range(1, P):
        pos |= {k * perp - 1, k * perp}
    return {p for p in pos if 0 <= p < Pn}


def window_spikes(Ln, n, off, ptr_z, esize, P):
    """The window regime (Ln >= n): positions in the stored noise clip of the two ranges [off, off + len0) and [0, len1),
    each partitioned on its own base with its own alignment test."""
    len0 = min(Ln - off, n)
    len1 = n - len0
    pos = {off + p for p in range_spikes(len0, aligned(ptr_z + off * esize, esize), P)}
    if len1 > 0:
        pos |= range_spikes(len1, aligned(ptr_z, esize), P)
    return pos


def spike(x, pos, height):
    """x[p] = +-height at the positions (alternating signs), in place."""
    for k, p in enumerate(sorted(pos)):
        x[p] = height if k % 2 == 0 else -height


def base_row(n, seed, i16, noise=False):
    """A random row with a small DC: std 0.1 (speech) / 0.05 (noise), or about 800 / 600 in int16 units."""
    rng = np.random.RandomState(seed)
    if i16:
        sd = 600.0 if noise else 800.0
        return np.round(rng.randn(n) * sd + (-17.0 if noise else 23.0)), sd
    sd = 0.05 if noise else 0.1
    return rng.randn(n) * sd + (-0.003 if noise else 0.01), sd


def gains_ref(s, nseq, snr):
    """numpy float64 (factor, equaliser) over exactly the samples the reference reads (dp:125-130)."""
    if len(s) == 0:
        return 0.0, 0.0
    s, n = np.asarray(s, np.float64), np.asarray(nseq, np.float64)
    f = np.sqrt(np.var(s) / np.var(n)) * 10.0 ** (-float(np.float32(snr)) / 20.0)
    return f, np.sqrt(np.sum(s * s) / np.sum(n * n))


def check_gains(fac, eq, wf, wg, what):
    """The gate; returns the errors in float32 ulps of the reference (factor, equaliser)."""
    if wf == 0.0:
        assert fac == 0.0 and eq == 0.0, (what, fac, eq)
        return 0.0, 0.0
    assert abs(fac - wf) <= TOL_GAIN * wf and abs(eq - wg) <= TOL_GAIN * wg, (what, float(fac), wf, float(eq), wg)
    return abs(fac - wf) / np.spacing(np.float32(wf)), abs(eq - wg) / np.spacing(np.float32(wg))


# ---------------------------------------------------------------------------------------------------------------- clip pools
# A speech pool with a 40 s clip: mix_pools sizes the statistics clusters from the speech pool's stride, so every row -- 3 s and
# 2 ms clips included -- runs at P = 8.  Rows cover the window regime with a wrap (len1 > 0), odd offsets (z + off misaligned),
# the periodic regime at offsets 0, 1 and Ln - 1, Pn = n and Pn = n - 1.
POOL_SPEECH = [640003, 48001, 160002, 31]
POOL_NOISE = [700001, 27371, 48001, 48000]
POOL_ROWS = [        # (speech clip, noise clip, offset)
    (0, 0, 99999),   # window, wraps: len0 = 600 002, len1 = 40 001; odd offset
    (0, 0, 0),       # window, no wrap
    (0, 1, 0),       # periodic, off 0
    (0, 1, 1),       # periodic, off 1
    (0, 1, 27370),   # periodic, off Ln - 1
    (1, 0, 700000),  # window, off Ln - 1: len0 = 1
    (1, 2, 1),       # Ln = n, off 1: len1 = 1
    (1, 3, 12345),   # Ln = n - 1: periodic, q = 1, rem = 1
    (2, 0, 654321),  # window, wraps: len0 = 45 680, len1 = 114 322
    (3, 1, 5),       # 31 samples (< 4 P): CTAs without a share
    (2, 1, 1),       # periodic
]


def pool_row_noise(z, Ln, off, n):
    """n[i] = z[(off + i) mod Ln], i < n (avse_common.h pool_row / noise_span)."""
    return z[(off + np.arange(n)) % Ln]


def build_pools(mod, i16, odd_stride, P, device="cuda"):
    """Spiked speech / noise pools on the device: pack_clips' layout (stride rounded up to 4 samples), or a hand-built pool with
    an odd stride, so that odd clips start unaligned.  Everything past a clip is poison (NaN / 30000).  Returns
    (speech_pool, speech_lengths, noise_pool, noise_lengths, speech clips, noise clips) with the clips as stored (host)."""
    dt = torch.int16 if i16 else torch.float32
    esize = 2 if i16 else 4
    sclips, nclips, ssd, nsd = [], [], [], []
    for k, n in enumerate(POOL_SPEECH):
        x, sd = base_row(n, 700 + k, i16)
        sclips.append(x)
        ssd.append(sd)
    for k, n in enumerate(POOL_NOISE):
        x, sd = base_row(n, 720 + k, i16, noise=True)
        nclips.append(x)
        nsd.append(sd)
    poison = 30000.0 if i16 else np.nan
    if odd_stride:
        ws = max(POOL_SPEECH) | 1
        wn = max(POOL_NOISE) + 2
        wn |= 1
        sp = torch.empty((len(sclips), ws), dtype=dt, device=device)
        nz = torch.empty((len(nclips), wn), dtype=dt, device=device)
        slen = torch.tensor(POOL_SPEECH, dtype=torch.int32, device=device)
        nlen = torch.tensor(POOL_NOISE, dtype=torch.int32, device=device)
    else:
        sp, slen = mod.pack_clips([c.astype(np.float32) for c in sclips], device, dtype=dt)
        nz, nlen = mod.pack_clips([c.astype(np.float32) for c in nclips], device, dtype=dt, allow_empty=False)
    ps, pn = sp.data_ptr(), nz.data_ptr()
    rs, rn = sp.stride(0), nz.stride(0)
    for (si, ni, off) in POOL_ROWS:
        ls, Ln = POOL_SPEECH[si], POOL_NOISE[ni]
        spike(sclips[si], range_spikes(ls, aligned(ps + si * rs * esize, esize), P), SPIKE_S * ssd[si])
        if Ln < ls:
            pos = periodic_spikes(Ln, ls, off, P)
        else:
            pos = window_spikes(Ln, ls, off, pn + ni * rn * esize, esize, P)
        spike(nclips[ni], pos, SPIKE_N * nsd[ni])
    np_dt = np.int16 if i16 else np.float32
    hs = np.full(tuple(sp.shape), poison, np_dt)
    hn = np.full(tuple(nz.shape), poison, np_dt)
    sclips = [c.astype(np_dt) for c in sclips]
    nclips = [c.astype(np_dt) for c in nclips]
    for k, c in enumerate(sclips):
        hs[k, :len(c)] = c
    for k, c in enumerate(nclips):
        hn[k, :len(c)] = c
    sp.copy_(torch.from_numpy(hs))
    nz.copy_(torch.from_numpy(hn))
    return sp, slen, nz, nlen, sclips, nclips
