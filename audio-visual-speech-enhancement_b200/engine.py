"""Batched, device-resident host mirror of the reference's spectral path.

`SpectralEngine` owns one `avse_ctx` (constant tables on one GPU) and exposes the batched
equivalents of /root/reference/data_processor.py:35-139 on torch CUDA tensors.  All arithmetic
runs in libavse_b200.so (hand-written CUDA, sm_100a) through the C ABI; torch only supplies
device memory and the current stream.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np
import torch

from . import _native
from ._native import ForwardArgs, InverseArgs, PoolMixArgs, check

N_FFT, HOP, N_BINS, N_MELS, SPSS = 640, 160, 321, 80, 20
LAYOUT_SLICES, LAYOUT_SPEC = 0, 1
SAMPLE_F32, SAMPLE_I16 = 0, 1
PIXEL_U8, PIXEL_F32 = 0, 1


import functools


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _on_device(fn):
    """Run an engine method with the engine's GPU as the current device: the launchers refuse a context whose device is
    not current, and torch allocates on the current device."""
    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapped


def _row_array(x, B, dtype, device, name):
    """A per-row side array (lengths: int32, SNRs: float32) as the kernels read it: a contiguous [B] tensor of `dtype` on
    `device`.  Takes a tensor of any dtype, device or stride, a numpy array or a list; None stays None.  An int64 tensor
    handed to the kernel as it is would be read as int32 pairs (row 1 of `[16000, 9001]` would see the high word of 16000,
    0), so every entry point that forwards such an array converts it here.  Raises ValueError unless it holds B values."""
    if x is None:
        return None
    t = x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x))
    if t.shape != (B,):
        raise ValueError("%s: expected one value per row, shape (%d,), got %s" % (name, B, tuple(t.shape)))
    return t.to(device=device, dtype=dtype).contiguous()


def _rs(t):
    """Row stride in elements; a size-1 leading dimension may carry an arbitrary (even 0) stride."""
    if t is None:
        return 0
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t[0].numel())


class DbKeys(object):
    """Per-utterance side data that the statistics pass (avse_snr_factor) hands to the forward pass, device resident:
    the running dB extrema of (speech, noise, mixed) as order-preserving int32 keys -- `max` [B, 3] over all frames
    (librosa's top_db reference, dp:94), `min` [B, 3] over the stored values (lets the floor pass skip utterances that
    need no clipping) -- and `equalizer` [B] = sqrt(sum s^2 / sum n^2), the ratio of the raw powers of speech and noise that
    conditions the packed FFT of the forward kernels (avse_forward_args::equalizer; None until snr_factor has filled it)."""
    __slots__ = ("buf", "max", "min", "equalizer", "_eq_buf")

    def __init__(self, B, device):
        self.buf = torch.empty((2, B, 3), dtype=torch.int32, device=device)
        self.max = self.buf[0]
        self.min = self.buf[1]
        self._eq_buf = torch.empty((B,), dtype=torch.float32, device=device)
        self.equalizer = None


def _keys(k):
    """(max_key tensor, min_key tensor or None) of a DbKeys or of a bare [B, 3] max-key tensor."""
    if isinstance(k, DbKeys):
        return k.max, k.min
    return k, None


def geometry(sample_rate, video_frame_rate, slice_duration_ms=200):
    """dp:36, dp:44-45, dp:49 integer geometry."""
    samples_per_slice = int((float(slice_duration_ms) / 1000) * sample_rate)
    n_fft = int(float(sample_rate) / video_frame_rate)
    hop = int(n_fft / 4)
    spss = int(samples_per_slice / hop) if hop else 0
    return samples_per_slice, n_fft, hop, spss


def frame_count(L, n_fft, hop):
    """librosa.stft(center=True) frame count of a length-L signal: 1 + (L + 2 (n_fft // 2) - n_fft) // hop."""
    return 1 + (int(L) + 2 * (n_fft // 2) - n_fft) // hop


def slice_count(L, n_fft, hop, spss):
    """Slices of a length-L signal, int(T / spss) (dp:50).  This is the count preprocess_audio_pair returns; the
    min(video, audio) cut of dp:164 comes later, in data_processor.assemble_sample.  It exceeds n_video_slices
    (L = samples_per_slice * n_video_slices) when spss * hop < samples_per_slice, e.g. from 65 slices on at 16 kHz /
    24000/1001 fps."""
    return frame_count(L, n_fft, hop) // spss


class SpectralEngine(object):
    """One GPU's worth of the spectral front/back end."""

    def __init__(self, sample_rate=16000, video_frame_rate=25.0, slice_duration_ms=200, fmin=0.0, fmax=8000.0, device=None,
                 n_fft=None, hop=None):
        """Geometry from (sample_rate, video_frame_rate, slice_duration_ms) as the reference derives it (dp:36, dp:44-45,
        dp:49); n_fft / hop may be given explicitly instead (signal_to_spectrogram's own arguments, dp:77)."""
        if not torch.cuda.is_available():
            raise RuntimeError("SpectralEngine needs a CUDA device: this framework has no CPU path")
        sps, n_fft_d, hop_d, spss = geometry(sample_rate, video_frame_rate, slice_duration_ms)
        if n_fft is None:
            n_fft, hop = n_fft_d, hop_d
        else:
            n_fft = int(n_fft)
            hop = int(n_fft / 4) if hop is None else int(hop)
            spss = int(sps / hop) if hop else 0
        if hop < 1 or spss < 1:
            raise ValueError("degenerate geometry: n_fft=%d hop=%d frames per slice=%d" % (n_fft, hop, spss))
        self.sample_rate = int(sample_rate)
        self.video_frame_rate = float(video_frame_rate)
        self.slice_duration_ms = slice_duration_ms
        self.samples_per_slice = sps
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("SpectralEngine needs a CUDA device: this framework has no CPU path")
        if self.device.index is None:        # a bare "cuda" means the current device, not GPU 0
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = _native.load()
        h = ctypes.c_void_p()
        # (640, 160, 80, 20) -- the reference's 16 kHz / 25 fps -- gets the specialised kernels; any other geometry the
        # reference can derive (dp:44-45) runs the generic fallback kernels behind the same entry points
        check(self._lib.avse_create_ex(self.sample_rate, n_fft, hop, N_MELS, spss, float(fmin), float(fmax), self.device.index,
                                       ctypes.byref(h)), "avse_create_ex")
        self._ctx = h
        geo = (ctypes.c_int * 6)()
        check(self._lib.avse_get_geometry(self._ctx, ctypes.byref(geo)), "avse_get_geometry")
        self.n_fft, self.hop, self.n_bins, self.n_mels, self.spss = (int(v) for v in geo[:5])
        self.specialised = geo[5] == 0      # False: the generic fallback kernels serve this geometry

    def __del__(self):
        try:
            if getattr(self, "_ctx", None):
                self._lib.avse_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def filterbank(self):
        """librosa.filters.mel(sr, 640, 80, fmin, fmax) as built by the library (float64 (80, 321))."""
        fb = np.zeros((self.n_mels, self.n_bins), dtype=np.float64)
        check(self._lib.avse_get_filterbank(self._ctx, fb.ctypes.data), "avse_get_filterbank")
        return fb

    def _as_batch(self, x, keep_int16=False):
        """[B, n] contiguous-row view; float32, or raw int16 WAV samples when the kernel decodes them itself."""
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dtype != torch.float32 and not (keep_int16 and x.dtype == torch.int16):
            x = x.to(torch.float32)
        if x.stride(-1) != 1:
            x = x.contiguous()
        return x

    def _needs_inverse_scratch(self):
        """The specialised I8 inverse kernel keeps the pinv coefficients on chip; only generic-geometry contexts and the
        round-1 4-frame kernel (AVSE_INV4=1, A/B runs) need the `work` scratch of avse_inverse_work_elems."""
        return (not self.specialised) or os.environ.get("AVSE_INV4") == "1"

    def n_frames(self, L):
        """librosa.stft(center=True) frame count: 1 + (L + 2 (n_fft // 2) - n_fft) // hop (== 1 + L // hop for even n_fft)."""
        return frame_count(L, self.n_fft, self.hop)

    def n_slices(self, L):
        """Slices a length-L row yields, int(T / spss) (dp:50; see slice_count)."""
        return slice_count(L, self.n_fft, self.hop, self.spss)

    # ------------------------------------------------------------------ a3: SNR factor
    @_on_device
    def snr_factor(self, speech, noise, lengths=None, snr_db=None, max_key=None, noise_lengths=None):
        """AudioMixer.snr_factor (dp:130) for a batch; returns (factor[B], DbKeys) with the keys reset and the level
        equaliser filled in.  noise_lengths [B] int32: own length of each noise file; a noise shorter than its speech is
        tiled periodically inside the kernel (dp:125-128) instead of being materialised."""
        i16 = speech.dtype == torch.int16 and noise.dtype == torch.int16
        speech, noise = self._as_batch(speech, i16), self._as_batch(noise, i16)
        B, L = speech.shape
        assert noise.shape[0] == B and _rs(noise) == _rs(speech)
        assert noise_lengths is not None or noise.shape[1] >= L, "a noise batch narrower than the speech needs noise_lengths"
        lengths = _row_array(lengths, B, torch.int32, self.device, "lengths")
        noise_lengths = _row_array(noise_lengths, B, torch.int32, self.device, "noise_lengths")
        snr_db = _row_array(snr_db, B, torch.float32, self.device, "snr_db")
        factor = torch.empty(B, dtype=torch.float32, device=self.device)
        if max_key is None:
            max_key = DbKeys(B, self.device)
        kmax, kmin = _keys(max_key)
        eq = None
        if isinstance(max_key, DbKeys):
            eq = max_key.equalizer = max_key._eq_buf
        check(self._lib.avse_snr_factor(self._ctx, _ptr(speech), _ptr(noise), SAMPLE_I16 if i16 else SAMPLE_F32, _rs(speech), _ptr(lengths),
                                        _ptr(noise_lengths), B, L, _ptr(snr_db), _ptr(factor), _ptr(eq), _ptr(kmax), _ptr(kmin),
                                        self._stream()), "avse_snr_factor")
        return factor, max_key

    # ------------------------------------------------------------------ a1/a4/a5: forward
    @_on_device
    def forward_raw(self, speech, noise=None, L=None, len_speech=None, len_noise=None, factor=None, layout=LAYOUT_SLICES,
                    n_slices=None, want=("speech", "noise", "mixed"), mixed_pcm=True, max_key=None, stft=False, out=None,
                    noise_lengths=None):
        """Launch avse_forward.  Returns dict with un-floored outputs + max_key (see include/avse_b200.h).
        When `max_key` is the DbKeys that snr_factor returned, its level equaliser rides along (numerical conditioning of
        the packed FFT; the result is s + factor * n either way)."""
        # raw int16 samples go to the kernel as they are (decode fused into its loads) for pair batches
        i16 = noise is not None and speech.dtype == torch.int16 and noise.dtype == torch.int16 and not stft
        speech = self._as_batch(speech, i16)
        B = speech.shape[0]
        if L is None:
            L = speech.shape[1]
        if noise is not None:
            noise = self._as_batch(noise, i16)
            assert _rs(noise) == _rs(speech) and noise.shape[0] == B
        len_speech = _row_array(len_speech, B, torch.int32, self.device, "len_speech")
        len_noise = _row_array(len_noise, B, torch.int32, self.device, "len_noise")
        noise_lengths = _row_array(noise_lengths, B, torch.int32, self.device, "noise_lengths")
        T = self.n_frames(L)
        if n_slices is None:
            n_slices = self.n_slices(L)
        res = {} if out is None else out
        ld_t = (T + 3) // 4 * 4
        shape = (B, n_slices, self.n_mels, self.spss) if layout == LAYOUT_SLICES else (B, self.n_mels, ld_t)
        for name in ("speech", "noise", "mixed"):
            if name in want and (name == "speech" or noise is not None):
                if name not in res:
                    res[name] = torch.empty(shape, dtype=torch.float32, device=self.device)
            else:
                res.setdefault(name, None)
        if mixed_pcm and noise is not None:
            if "mixed_pcm" not in res:
                res["mixed_pcm"] = torch.empty((B, L), dtype=torch.float32, device=self.device)
        else:
            res.setdefault("mixed_pcm", None)
        if max_key is None:
            max_key = DbKeys(B, self.device)
            check(self._lib.avse_reset_max(self._ctx, _ptr(max_key.max), _ptr(max_key.min), 3 * B, self._stream()), "avse_reset_max")
        kmax, kmin = _keys(max_key)
        res["max_key"] = max_key
        res["stft"] = torch.empty((B, T, self.n_bins), dtype=torch.complex64, device=self.device) if stft else None
        ref = res["speech"]
        a = ForwardArgs()
        a.speech, a.noise, a.in_stride = _ptr(speech), _ptr(noise), _rs(speech)
        a.len_speech, a.len_noise, a.factor = _ptr(len_speech), _ptr(len_noise), _ptr(factor)
        a.B, a.L = B, L
        a.layout, a.n_slices, a.ld_t = layout, n_slices, ld_t
        a.out_speech, a.out_noise, a.out_mixed = _ptr(res["speech"]), _ptr(res["noise"]), _ptr(res["mixed"])
        a.out_stride = _rs(ref)
        a.mixed_pcm = _ptr(res["mixed_pcm"])
        a.pcm_stride = _rs(res["mixed_pcm"])
        a.max_key = _ptr(kmax)
        a.min_key = _ptr(kmin)
        a.sample_format = SAMPLE_I16 if i16 else SAMPLE_F32
        a.stft_speech = _ptr(res["stft"])
        a.equalizer = _ptr(max_key.equalizer) if (isinstance(max_key, DbKeys) and factor is not None and noise is not None) else 0
        a.noise_period = _ptr(noise_lengths) if noise is not None else 0
        check(self._lib.avse_forward(self._ctx, ctypes.byref(a), self._stream()), "avse_forward")
        res["T"], res["ld_t"], res["n_slices"], res["layout"] = T, ld_t, n_slices, layout
        return res

    @_on_device
    def floor_(self, data, max_key, which):
        """amplitude_to_db's top_db floor (dp:94), in place, per utterance."""
        B = data.shape[0]
        n = data[0].numel()
        kmax, kmin = _keys(max_key)
        check(self._lib.avse_floor_inplace(self._ctx, _ptr(data), _rs(data), n, B, _ptr(kmax), _ptr(kmin), which, self._stream()),
              "avse_floor_inplace")
        return data

    @_on_device
    def floor3_(self, speech, noise, mixed, max_key):
        """The top_db floor for the three outputs of a pair batch in one launch."""
        B = speech.shape[0]
        n = speech[0].numel()
        assert _rs(speech) == _rs(noise) == _rs(mixed)
        kmax, kmin = _keys(max_key)
        check(self._lib.avse_floor_inplace3(self._ctx, _ptr(speech), _ptr(noise), _ptr(mixed), _rs(speech), n, B, _ptr(kmax), _ptr(kmin),
                                            self._stream()), "avse_floor_inplace3")

    @_on_device
    def floor_gather(self, spec, max_key, which, n_slices):
        """dp:49-57: SPEC [B,80,ld_t] (un-floored) -> floored slices [B,n_slices,80,20]."""
        B, _, ld_t = spec.shape
        out = torch.empty((B, n_slices, self.n_mels, self.spss), dtype=torch.float32, device=self.device)
        check(self._lib.avse_floor_gather(self._ctx, _ptr(spec), _rs(spec), ld_t, _ptr(out), _rs(out), n_slices, B,
                                          _ptr(_keys(max_key)[0]), which, self._stream()), "avse_floor_gather")
        return out

    @_on_device
    def max_db(self, max_key):
        """Decoded running maxima [B, 3] in dB."""
        max_key = _keys(max_key)[0]
        out = torch.empty(max_key.shape, dtype=torch.float32, device=self.device)
        check(self._lib.avse_max_db(self._ctx, _ptr(max_key), max_key.numel(), _ptr(out), self._stream()), "avse_max_db")
        return out

    @_on_device
    def min_db(self, keys):
        """Decoded running minima [B, 3] of the stored dB values (same key encoding as the maxima)."""
        kmin = _keys(keys)[1]
        out = torch.empty(kmin.shape, dtype=torch.float32, device=self.device)
        check(self._lib.avse_max_db(self._ctx, _ptr(kmin), kmin.numel(), _ptr(out), self._stream()), "avse_max_db")
        return out

    # ------------------------------------------------------------------ batched reference-level operations
    @_on_device
    def preprocess_pairs(self, speech, noise, n_video_slices, lengths=None, snr_db=None, out=None, noise_lengths=None, info=None):
        """Batched preprocess_audio_pair (dp:119-139) on device tensors.

        speech, noise: [B, >=max(lengths)] float32 or int16, same row stride.  noise_lengths [B] int32 (optional): own
        length of each noise file -- a noise shorter than its speech is tiled periodically inside the kernels
        (dp:125-128); without it the noise rows must already cover the speech length (see fit_noise).
        Returns (mixed_slices, speech_slices, noise_slices, mixed_pcm) with shapes [B, n, 80, spss] x3 and [B, L];
        n = int(T / spss) (dp:50, see slice_count), L = samples_per_slice * n_video_slices.  Batches of any size: nothing
        here is capped at 65 535.
        """
        i16 = speech.dtype == torch.int16 and noise.dtype == torch.int16
        speech, noise = self._as_batch(speech, i16), self._as_batch(noise, i16)
        L = self.samples_per_slice * int(n_video_slices)
        n = self.n_slices(L)
        B = speech.shape[0]        # the side arrays feed two launches: convert them once
        lengths = _row_array(lengths, B, torch.int32, self.device, "lengths")
        snr_db = _row_array(snr_db, B, torch.float32, self.device, "snr_db")
        noise_lengths = _row_array(noise_lengths, B, torch.int32, self.device, "noise_lengths")
        if lengths is None and speech.shape[1] != L:
            lengths = torch.full((speech.shape[0],), speech.shape[1], dtype=torch.int32, device=self.device)
        # info: optional dict that receives the SNR factors and the dB keys
        # dp:130: the variances are over the ORIGINAL speech length (the whole row), before the pad / truncate to L
        factor, max_key = self.snr_factor(speech, noise, lengths=lengths, snr_db=snr_db, noise_lengths=noise_lengths)
        res = self.forward_raw(speech, noise, L=L, len_speech=lengths, len_noise=lengths, factor=factor, layout=LAYOUT_SLICES,
                               n_slices=n, max_key=max_key, out=out, noise_lengths=noise_lengths)
        self.floor3_(res["speech"], res["noise"], res["mixed"], max_key)
        if info is not None:        # side data for callers that need it: the SNR factors (dp:130) and the dB extrema
            info["factor"], info["keys"] = factor, max_key
        return res["mixed"], res["speech"], res["noise"], res["mixed_pcm"]

    @_on_device
    def mix_pools(self, speech_pool, speech_lengths, noise_pool, noise_lengths, speech_index, noise_index, n_video_slices,
                  noise_offset=None, snr_db=None, out=None, info=None, check=True, speech_start=None):
        """preprocess_audio_pair (dp:119-139) of pairings drawn from two device-resident clip pools (avse_mix_pooled).

        speech_pool [Ns, >= max clip] / noise_pool [Nn, >= max clip]: float32, or int16 for both (raw WAV samples, decoded in
        the kernels); speech_lengths [Ns] / noise_lengths [Nn] int32 clip lengths (see pack_clips).  Row b mixes speech clip
        speech_index[b] with noise clip noise_index[b] read from sample noise_offset[b] on and wrapped around its length:
        n[i] = z[(off + i) mod Ln] (off = 0, the default, is the reference's tile-or-truncate rule, dp:125-128), at snr_db[b]
        (default 0 dB, dp:130).  No pairing is materialised.
        Returns (mixed, speech, noise, mixed_pcm) shaped like preprocess_pairs: [B, n, 80, spss] x3 and [B, L],
        n = int(T / spss) (dp:50, see slice_count).
        speech_start [B] (optional): row b mixes the window s = clip[a : a + Lw] of its speech clip instead of the whole clip,
        a = speech_start[b], Lw = min(L, Ls - a): the SNR statistics run over the window, the reflect padding mirrors inside it,
        and n[i] = z[(off + i) mod Ln] for i < Lw.  Starts on slice boundaries (a = samples_per_slice * k) keep audio slice j
        aligned with video slice k + j of the clip; any sample start is accepted.  A start is valid when a == 0 or 0 < a < Ls.
        A row with an index out of range, an offset outside [0, Ln) or an invalid start is invalid: it is processed as an empty
        pair (every slice at -100 dB, PCM zeros).  check=True reads the device flag back (one synchronisation) and raises IndexError; check=False
        stays asynchronous.  out: dict whose tensors are re-used from call to call (like preprocess_pairs / HostPipeline).
        info: optional dict that receives `factor` [B], the dB `keys` (DbKeys) and `valid` [B] bool = row valid and factor
        finite (a silent noise window gives inf / nan like numpy)."""
        i16 = speech_pool.dtype == torch.int16 and noise_pool.dtype == torch.int16
        sp, nz = self._as_batch(speech_pool, i16), self._as_batch(noise_pool, i16)
        dev = self.device
        slen = torch.as_tensor(speech_lengths, device=dev).to(torch.int32).contiguous()
        nlen = torch.as_tensor(noise_lengths, device=dev).to(torch.int32).contiguous()
        assert slen.numel() == sp.shape[0] and nlen.numel() == nz.shape[0], "one length per pool clip"
        si = torch.as_tensor(speech_index, device=dev).to(torch.int64).contiguous()
        ni = torch.as_tensor(noise_index, device=dev).to(torch.int64).contiguous()
        B = si.numel()
        assert ni.numel() == B and B > 0
        off = None if noise_offset is None else torch.as_tensor(noise_offset, device=dev).to(torch.int32).contiguous()
        snr = None if snr_db is None else torch.as_tensor(snr_db, device=dev).to(torch.float32).contiguous()
        start = None if speech_start is None else torch.as_tensor(speech_start, device=dev).to(torch.int32).contiguous()
        assert off is None or off.numel() == B
        assert snr is None or snr.numel() == B
        assert start is None or start.numel() == B
        L = self.samples_per_slice * int(n_video_slices)
        n = self.n_slices(L)
        res = {} if out is None else out

        def buf(name, shape, dtype):
            t = res.get(name)
            if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
                t = res[name] = torch.empty(shape, dtype=dtype, device=dev)
            return t

        shape = (B, n, self.n_mels, self.spss)
        mixed, speech, noise = (buf(k, shape, torch.float32) for k in ("mixed", "speech", "noise"))
        pcm = buf("mixed_pcm", (B, L), torch.float32)
        factor = buf("factor", (B,), torch.float32)
        keys = res.get("keys")
        if not isinstance(keys, DbKeys) or keys.max.shape[0] != B:
            keys = res["keys"] = DbKeys(B, dev)
        keys.equalizer = keys._eq_buf
        bad = buf("bad_row_flag", (1,), torch.int32)
        bad.zero_()
        a = PoolMixArgs()
        a.speech_pool, a.speech_len, a.speech_stride, a.n_speech = _ptr(sp), _ptr(slen), _rs(sp), sp.shape[0]
        a.noise_pool, a.noise_len, a.noise_stride, a.n_noise = _ptr(nz), _ptr(nlen), _rs(nz), nz.shape[0]
        a.sample_format = SAMPLE_I16 if i16 else SAMPLE_F32
        a.speech_index, a.noise_index, a.noise_offset, a.snr_db = _ptr(si), _ptr(ni), _ptr(off), _ptr(snr)
        a.B, a.L, a.n_slices = B, L, n
        a.out_speech, a.out_noise, a.out_mixed, a.out_stride = _ptr(speech), _ptr(noise), _ptr(mixed), _rs(mixed)
        a.mixed_pcm, a.pcm_stride = _ptr(pcm), _rs(pcm)
        a.factor_out, a.equalizer_out = _ptr(factor), _ptr(keys.equalizer)
        a.max_key, a.min_key, a.bad_row_flag = _ptr(keys.max), _ptr(keys.min), _ptr(bad)
        a.speech_start = _ptr(start)
        _native.check(self._lib.avse_mix_pooled(self._ctx, ctypes.byref(a), self._stream()), "avse_mix_pooled")   # (`check` is the flag here)
        if info is not None:
            ok = (si >= 0) & (si < sp.shape[0]) & (ni >= 0) & (ni < nz.shape[0])
            ln = nlen[ni.clamp(0, nz.shape[0] - 1)].clamp(0, _rs(nz))
            o = torch.zeros_like(ln) if off is None else off
            ok &= (o >= 0) & (o < ln)
            if start is not None:
                ls = slen[si.clamp(0, sp.shape[0] - 1)].clamp(0, _rs(sp))
                ok &= (start == 0) | ((start > 0) & (start < ls))
            info["factor"], info["keys"], info["valid"] = factor, keys, ok & torch.isfinite(factor)
        if check and int(bad.item()):
            raise IndexError("mix_pools: a row has an index outside its pool, a noise offset outside [0, noise length) or a speech "
                             "start outside [0, speech length)")
        return mixed, speech, noise, pcm

    @_on_device
    def spectrogram(self, signals, lengths=None, stft=False):
        """Batched signal_to_spectrogram(mel=True, db=True) (dp:77-96): floored dB [B, 80, T] (+ complex STFT)."""
        signals = self._as_batch(signals)
        res = self.forward_raw(signals, None, len_speech=lengths, layout=LAYOUT_SPEC, want=("speech",), mixed_pcm=False, stft=stft)
        self.floor_spec_(res["speech"], res["max_key"], 0, res["T"])
        out = res["speech"][:, :, :res["T"]]
        return (out, res["stft"]) if stft else out

    @_on_device
    def magphase(self, stft):
        """librosa.core.magphase (dp:80) of a complex STFT [B, T, bins] (as `spectrogram(..., stft=True)` returns it):
        (|D| float32 [B, bins, T], D/|D| complex64 [B, bins, T] with 1 + 0j where D == 0), in the reference's (freq, time) orientation."""
        st = torch.view_as_real(stft.contiguous())
        B, T, bins = stft.shape
        mag = torch.empty((B, bins, T), dtype=torch.float32, device=self.device)
        phase = torch.empty((B, bins, T), dtype=torch.complex64, device=self.device)
        check(self._lib.avse_magphase(self._ctx, st.data_ptr(), B, T, bins, _ptr(mag), torch.view_as_real(phase).data_ptr(), self._stream()),
              "avse_magphase")
        return mag, phase

    def floor_spec_(self, spec, max_key, which, T):
        # pad columns (>= T) are untouched garbage; floor the whole padded rows (harmless)
        return self.floor_(spec, max_key, which)

    @_on_device
    def preprocess_signals(self, signals, n_video_slices, lengths=None):
        """Batched preprocess_audio_signal (dp:35-57): [B, n, 80, spss] floored dB slices, n = int(T / spss) (dp:50)."""
        signals = self._as_batch(signals)
        L = self.samples_per_slice * int(n_video_slices)
        if lengths is None and signals.shape[1] < L:
            lengths = torch.full((signals.shape[0],), signals.shape[1], dtype=torch.int32, device=self.device)
        n = self.n_slices(L)
        res = self.forward_raw(signals, None, L=L, len_speech=lengths, layout=LAYOUT_SLICES, n_slices=n, want=("speech",), mixed_pcm=False)
        return self.floor_(res["speech"], res["max_key"], 0)

    @_on_device
    def reconstruct(self, mixed_pcm, mel_slices, lengths=None, out=None, work=None, out_dtype=torch.float32):
        """Batched reconstruct_speech_signal (dp:60-74): mixture PCM [B, L] + dB slices [B, n, 80, 20] -> PCM [B, 160*(min(20n, T)-1)].
        out_dtype=torch.int16 fuses AudioSignal.save_to_wav_file's clip + cast (se:176-177) into the last store."""
        mixed_pcm = self._as_batch(mixed_pcm)
        mel = mel_slices if mel_slices.dtype == torch.float32 else mel_slices.to(torch.float32)
        if mel.dim() == 3:
            mel = mel.unsqueeze(0)
        mel = mel.contiguous()
        B, L = mixed_pcm.shape
        lengths = _row_array(lengths, B, torch.int32, self.device, "lengths")
        n = mel.shape[1]
        T_use = min(self.spss * n, self.n_frames(L))
        out_len = self.hop * (T_use - 1)
        if out is None:
            out = torch.empty((B, out_len), dtype=out_dtype, device=self.device)
        assert out.dtype in (torch.float32, torch.int16)
        per = ctypes.c_longlong(0)
        if self._needs_inverse_scratch():
            check(self._lib.avse_inverse_work_elems_ctx(self._ctx, T_use, ctypes.byref(per)), "avse_inverse_work_elems_ctx")
            if work is None or work.numel() < B * per.value:
                work = torch.empty((B, per.value), dtype=torch.float32, device=self.device)
        else:
            work = None
        a = InverseArgs()
        a.mel_db, a.layout, a.n_slices, a.n_frames, a.ld_t = _ptr(mel), LAYOUT_SLICES, n, 0, 0
        a.mel_stride = _rs(mel)
        a.mixed_pcm, a.pcm_stride, a.len_pcm = _ptr(mixed_pcm), _rs(mixed_pcm), _ptr(lengths)
        a.B, a.L = B, L
        a.out_pcm, a.out_stride = _ptr(out), _rs(out)
        a.out_format = SAMPLE_I16 if out.dtype == torch.int16 else SAMPLE_F32
        a.work, a.work_stride = _ptr(work), per.value
        check(self._lib.avse_inverse(self._ctx, ctypes.byref(a), self._stream()), "avse_inverse")
        return out

    @_on_device
    def reconstruct_with_phase(self, mel_db, phase):
        """reconstruct_signal_from_spectrogram(mel=True, db=True) (dp:99-116) with an explicit phase:
        mel_db [B, 80, T] dB, phase [B, T_ph, 321] complex64 (frame-major).  Returns PCM [B, 160*(min(T, T_ph)-1)]."""
        mel = mel_db.to(torch.float32).contiguous()
        ph = torch.view_as_real(phase.to(torch.complex64).contiguous())
        B, _, T_mel = mel.shape
        T_ph = phase.shape[1]
        T_use = min(T_mel, T_ph)
        out = torch.empty((B, self.hop * (T_use - 1)), dtype=torch.float32, device=self.device)
        per = ctypes.c_longlong(0)
        work = None
        if self._needs_inverse_scratch():
            check(self._lib.avse_inverse_work_elems_ctx(self._ctx, T_use, ctypes.byref(per)), "avse_inverse_work_elems_ctx")
            work = torch.empty((B, per.value), dtype=torch.float32, device=self.device)
        a = InverseArgs()
        a.mel_db, a.layout, a.n_slices, a.n_frames, a.ld_t = _ptr(mel), LAYOUT_SPEC, 0, T_mel, T_mel
        a.mel_stride = _rs(mel)
        a.mixed_pcm, a.pcm_stride, a.len_pcm = 0, 0, 0
        a.B, a.L = B, 0
        a.out_pcm, a.out_stride = _ptr(out), _rs(out)
        a.work, a.work_stride = _ptr(work), per.value
        a.phase, a.phase_stride, a.phase_frames = ph.data_ptr(), T_ph * self.n_bins, T_ph
        check(self._lib.avse_inverse(self._ctx, ctypes.byref(a), self._stream()), "avse_inverse")
        return out

    @_on_device
    def reconstruct_spec(self, mixed_pcm, mel_db, lengths=None):
        """Same with a SPEC-layout spectrogram [B, 80, T_mel] (dp:99-116 called directly with mel=True, db=True)."""
        mixed_pcm = self._as_batch(mixed_pcm)
        mel = mel_db if mel_db.dtype == torch.float32 else mel_db.to(torch.float32)
        if mel.dim() == 2:
            mel = mel.unsqueeze(0)
        mel = mel.contiguous()
        B, L = mixed_pcm.shape
        lengths = _row_array(lengths, B, torch.int32, self.device, "lengths")
        T_use = min(mel.shape[2], self.n_frames(L))
        out = torch.empty((B, self.hop * (T_use - 1)), dtype=torch.float32, device=self.device)
        per = ctypes.c_longlong(0)
        work = None
        if self._needs_inverse_scratch():
            check(self._lib.avse_inverse_work_elems_ctx(self._ctx, T_use, ctypes.byref(per)), "avse_inverse_work_elems_ctx")
            work = torch.empty((B, per.value), dtype=torch.float32, device=self.device)
        a = InverseArgs()
        a.mel_db, a.layout, a.n_slices, a.n_frames, a.ld_t = _ptr(mel), LAYOUT_SPEC, 0, mel.shape[2], mel.shape[2]
        a.mel_stride = _rs(mel)
        a.mixed_pcm, a.pcm_stride, a.len_pcm = _ptr(mixed_pcm), _rs(mixed_pcm), _ptr(lengths)
        a.B, a.L = B, L
        a.out_pcm, a.out_stride = _ptr(out), _rs(out)
        a.work, a.work_stride = _ptr(work), per.value
        check(self._lib.avse_inverse(self._ctx, ctypes.byref(a), self._stream()), "avse_inverse")
        return out

    def reconstruct_differentiable(self, mixed_pcm, mel_slices, lengths=None):
        """reconstruct (dp:60-74) as a differentiable op in the dB slices: the output is bit-identical to reconstruct's float32
        PCM, and backward runs avse_inverse_backward, so a loss on the waveform trains the slice predictor through the fixed
        reconstruction.  The mixture is data: a mixed_pcm that requires grad raises ValueError."""
        mel = mel_slices if mel_slices.dim() == 4 else mel_slices.unsqueeze(0)
        return _InverseFn.apply(mel, self, mixed_pcm, lengths, LAYOUT_SLICES)

    def reconstruct_spec_differentiable(self, mixed_pcm, mel_db, lengths=None):
        """reconstruct_spec as a differentiable op in mel_db [B, 80, T_mel] (see reconstruct_differentiable)."""
        mel = mel_db if mel_db.dim() == 3 else mel_db.unsqueeze(0)
        return _InverseFn.apply(mel, self, mixed_pcm, lengths, LAYOUT_SPEC)

    @_on_device
    def _inverse_launch(self, mixed_pcm, mel, lengths, layout, grad_pcm=None):
        """avse_inverse (grad_pcm None: returns the PCM) or avse_inverse_backward (returns dL/d mel, float32, mel's shape) for a
        contiguous float32 mel in SLICES [B, n, 80, spss] or SPEC [B, 80, T_mel] layout."""
        B, L = mixed_pcm.shape
        t_mel = self.spss * mel.shape[1] if layout == LAYOUT_SLICES else mel.shape[2]
        T_use = min(t_mel, self.n_frames(L))
        a = InverseArgs()
        a.mel_db, a.layout = _ptr(mel), layout
        if layout == LAYOUT_SLICES:
            a.n_slices, a.n_frames, a.ld_t = mel.shape[1], 0, 0
        else:
            a.n_slices, a.n_frames, a.ld_t = 0, t_mel, t_mel
        a.mel_stride = _rs(mel)
        a.mixed_pcm, a.pcm_stride, a.len_pcm = _ptr(mixed_pcm), _rs(mixed_pcm), _ptr(lengths)
        a.B, a.L = B, L
        a.out_format = SAMPLE_F32
        if grad_pcm is not None:
            grad_mel = torch.empty_like(mel)
            check(self._lib.avse_inverse_backward(self._ctx, ctypes.byref(a), _ptr(grad_pcm), _rs(grad_pcm), _ptr(grad_mel),
                                                  self._stream()), "avse_inverse_backward")
            return grad_mel
        out = torch.empty((B, self.hop * (T_use - 1)), dtype=torch.float32, device=self.device)
        per = ctypes.c_longlong(0)
        work = None
        if self._needs_inverse_scratch():
            check(self._lib.avse_inverse_work_elems_ctx(self._ctx, T_use, ctypes.byref(per)), "avse_inverse_work_elems_ctx")
            work = torch.empty((B, per.value), dtype=torch.float32, device=self.device)
        a.out_pcm, a.out_stride = _ptr(out), _rs(out)
        a.work, a.work_stride = _ptr(work), per.value
        check(self._lib.avse_inverse(self._ctx, ctypes.byref(a), self._stream()), "avse_inverse")
        return out


    # ------------------------------------------------------------------ next row f1: make_sample_set on the device
    @_on_device
    def make_sample_set(self, mixed_slices, speech_slices, n_slices=None, permutation=None, generator=None, extra=None, check=True):
        """speech_enhancer.py:241-262 without the pickle / numpy round trip: concatenate the slices of all samples
        (np.concatenate over `sample.mixed_spectrograms` / `.speech_spectrograms`) and apply ONE shared permutation.

        mixed_slices, speech_slices: [B, n_max, 80, 20] device tensors (outputs of preprocess_pairs); n_slices: per-sample
        slice counts [B] (dp:164 min(video, audio); None: n_max for all); permutation: int64 permutation of the
        sum(n_slices) concatenated rows (None: torch.randperm with `generator`); extra: optional third [B, n_max, ...]
        float32 array gathered with the same permutation (e.g. noise slices).
        check: validate a caller-supplied permutation (the kernel flags out-of-range indices; reading the flag back is the
        call's only host synchronisation -- pass False to stay asynchronous).
        Returns (mixed [N, 80, 20], speech [N, 80, 20], permutation) (+ extra rows when given)."""
        B, n_max = mixed_slices.shape[0], mixed_slices.shape[1]
        srcs = [mixed_slices, speech_slices] + ([extra] if extra is not None else [])
        for t in srcs:
            assert t.dtype == torch.float32 and t.is_contiguous() and t.shape[:2] == (B, n_max)
        row = mixed_slices[0, 0].numel()
        assert all(t[0, 0].numel() == row for t in srcs), "rows of all arrays must have the same size"
        rows = None                                  # None: every row is kept, concatenated row i is source row i
        N = B * n_max
        if n_slices is not None:
            ns = torch.as_tensor(n_slices, device=self.device, dtype=torch.int64)
            j = torch.arange(n_max, device=self.device, dtype=torch.int64)
            keep = j.unsqueeze(0) < ns.unsqueeze(1)                        # concatenation order: sample-major, slice-minor
            rows = (torch.arange(B, device=self.device, dtype=torch.int64).unsqueeze(1) * n_max + j.unsqueeze(0))[keep]
            N = rows.numel()
        user_perm = permutation is not None
        if permutation is None:
            permutation = torch.randperm(N, device=self.device, generator=generator)
        permutation = torch.as_tensor(permutation, device=self.device, dtype=torch.int64)
        if permutation.numel() != N:
            raise IndexError("permutation must hold %d indices in [0, %d)" % (N, N))
        if rows is None:
            index = permutation.contiguous()
            src_rows = B * n_max
        else:
            # out-of-range entries must reach the kernel's own check instead of faulting in this gather
            index = rows[permutation.clamp(0, max(N - 1, 0))].contiguous()
            if user_perm:
                index = torch.where((permutation < 0) | (permutation >= N), torch.full_like(index, -1), index)
            src_rows = B * n_max
        outs = [torch.empty((N,) + tuple(t.shape[2:]), dtype=torch.float32, device=self.device) for t in srcs]
        bad = torch.zeros(1, dtype=torch.int32, device=self.device)
        p = [_ptr(t) for t in srcs] + [0] * (3 - len(srcs))
        q = [_ptr(t) for t in outs] + [0] * (3 - len(outs))
        rc = self._lib.avse_gather_rows(self._ctx, p[0], p[1], p[2], src_rows, row, _ptr(index), N, q[0], q[1], q[2], _ptr(bad),
                                              self._stream())
        _native.check(rc, "avse_gather_rows")
        if user_perm and check and int(bad.item()):
            raise IndexError("permutation must hold %d indices in [0, %d)" % (N, N))
        return tuple(outs[:2]) + (permutation,) + tuple(outs[2:])

    @_on_device
    def gather_video(self, video_pool, index, normalizer=None, check=True):
        """Video rows of a training batch (avse_gather_video): out[i] = video_pool[index[i]] decoded to float32 and, with a
        VideoNormalizer, normalised per pixel exactly as its normalize() does (bit-identical to
        normalizer.normalize(video_pool.float()[index])).  video_pool: uint8 or float32 device tensor whose last three dimensions
        are one slice [H, W, F] (e.g. pack_video's [Ns, S_max, H, W, F], indexed as [Ns * S_max] slices); index: int64 slice
        indices.  An index outside the pool leaves its row unset and, with check=True, raises IndexError (one synchronisation).
        Returns [N, H, W, F] float32."""
        if video_pool.dtype not in (torch.uint8, torch.float32):
            raise ValueError("gather_video: the pool must be uint8 or float32, got %s" % video_pool.dtype)
        if video_pool.dim() < 3 or not video_pool.is_cuda or not video_pool.is_contiguous():
            raise ValueError("gather_video: expected a contiguous device pool [..., H, W, F]")
        H, W, F = (int(d) for d in video_pool.shape[-3:])
        n_pool = video_pool.numel() // max(1, H * W * F)
        if (H * W * F) % 4:
            raise ValueError("gather_video: H * W * F must be a multiple of 4")
        idx = torch.as_tensor(index, device=self.device).to(torch.int64).contiguous().view(-1)
        N = idx.numel()
        out = torch.empty((N, H, W, F), dtype=torch.float32, device=self.device)
        mean = stdv = None
        if normalizer is not None:
            assert tuple(normalizer.shape) == (H, W), "gather_video: the normaliser's image shape differs from the pool's"
            mean, stdv = normalizer.mean_image.contiguous(), normalizer.std_image.contiguous()
        bad = torch.zeros(1, dtype=torch.int32, device=self.device)
        fmt = PIXEL_U8 if video_pool.dtype == torch.uint8 else PIXEL_F32
        check_rc = self._lib.avse_gather_video(self._ctx, _ptr(video_pool), fmt, n_pool, H * W, F, _ptr(idx), N, _ptr(mean), _ptr(stdv),
                                               _ptr(out), _ptr(bad), self._stream())
        _native.check(check_rc, "avse_gather_video")
        if check and N and int(bad.item()):
            raise IndexError("gather_video: a slice index lies outside the pool's %d slices" % n_pool)
        return out


class _InverseFn(torch.autograd.Function):
    """The mixture-phase reconstruction with its vector-Jacobian product in the dB input (avse_inverse / avse_inverse_backward)."""

    @staticmethod
    def forward(ctx, mel, engine, mixed_pcm, lengths, layout):
        if mixed_pcm.requires_grad:
            raise ValueError("reconstruct_differentiable: mixed_pcm is data here (no gradient flows to the mixture or its phase); "
                             "pass mixed_pcm.detach()")
        pcm = engine._as_batch(mixed_pcm)
        # one int32 copy for both launches: the backward reads the lengths the forward read
        lengths = _row_array(lengths, pcm.shape[0], torch.int32, engine.device, "lengths")
        mel32 = (mel if mel.dtype == torch.float32 else mel.to(torch.float32)).contiguous()
        ctx.engine, ctx.layout, ctx.mel_dtype = engine, layout, mel.dtype
        ctx.save_for_backward(mel32, pcm, lengths)
        return engine._inverse_launch(pcm, mel32, lengths, layout)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        mel32, pcm, lengths = ctx.saved_tensors
        g = grad_out.to(torch.float32).contiguous()      # y.sum() hands over a stride-0 expanded tensor
        grad_mel = ctx.engine._inverse_launch(pcm, mel32, lengths, ctx.layout, grad_pcm=g)
        return grad_mel.to(ctx.mel_dtype), None, None, None, None


class VideoNormalizer(object):
    """data_processor.VideoNormalizer (dp:201-212) on the device: per-pixel mean / std over (slices, frames) of the
    mouth-crop tensor [N, H, W, F] and the in-place normalisation (SURVEY 8(f) row 4)."""

    def __init__(self, engine, video_samples):
        self.eng = engine
        self.device = engine.device
        if video_samples is None:
            return
        with torch.cuda.device(self.device):
            v = self._as_dev(engine, video_samples)
            N, H, W, F = v.shape
            self.shape = (H, W)
            self.mean_image = torch.empty((H, W), dtype=torch.float32, device=engine.device)
            self.std_image = torch.empty((H, W), dtype=torch.float32, device=engine.device)
            scratch = torch.empty(2 * H * W, dtype=torch.float64, device=engine.device)
            check(engine._lib.avse_video_stats(engine._ctx, _ptr(v), N, H * W, F, _ptr(scratch), _ptr(self.mean_image),
                                               _ptr(self.std_image), engine._stream()), "avse_video_stats")

    @classmethod
    def from_images(cls, engine, mean_image, std_image):
        """Normaliser from stored statistics (the unpickled state of data_processor.VideoNormalizer, se:66-67)."""
        self = cls(engine, None)
        self.mean_image = torch.as_tensor(np.ascontiguousarray(mean_image, dtype=np.float32)).to(engine.device)
        self.std_image = torch.as_tensor(np.ascontiguousarray(std_image, dtype=np.float32)).to(engine.device)
        self.shape = tuple(self.mean_image.shape)
        return self

    @staticmethod
    def _as_dev(engine, video_samples):
        v = video_samples if torch.is_tensor(video_samples) else torch.from_numpy(np.ascontiguousarray(video_samples, dtype=np.float32))
        v = v.to(engine.device, dtype=torch.float32).contiguous()
        assert v.dim() == 4, "video_samples: slices x height x width x frames_per_slice"
        return v

    @_on_device
    def normalize(self, video_samples):
        """In place like the reference: a CUDA float32 tensor is modified directly, a numpy array is overwritten."""
        on_dev = torch.is_tensor(video_samples) and video_samples.is_cuda and video_samples.dtype == torch.float32 and video_samples.is_contiguous()
        v = video_samples if on_dev else self._as_dev(self.eng, video_samples)
        N, H, W, F = v.shape
        assert (H, W) == self.shape
        check(self.eng._lib.avse_video_normalize(self.eng._ctx, _ptr(v), N, H * W, F, _ptr(self.mean_image), _ptr(self.std_image),
                                                 self.eng._stream()), "avse_video_normalize")
        if not on_dev:
            if torch.is_tensor(video_samples):
                video_samples.copy_(v)
            else:
                video_samples[...] = v.cpu().numpy()
        return video_samples


def mse(engine, a, b):
    """Mean squared error over every element (the loss of network.evaluate on log-mel slices, network.py:214-220)."""
    a = a.to(engine.device, dtype=torch.float32).contiguous()
    b = b.to(engine.device, dtype=torch.float32).contiguous()
    assert a.shape == b.shape
    with torch.cuda.device(engine.device):
        scratch = torch.empty(1, dtype=torch.float64, device=engine.device)
        out = torch.empty(1, dtype=torch.float32, device=engine.device)
        check(engine._lib.avse_mse(engine._ctx, _ptr(a), _ptr(b), a.numel(), _ptr(scratch), _ptr(out), engine._stream()), "avse_mse")
    return out


class HostPipeline(object):
    """preprocess_audio_pair (dp:119-139) for a HOST-resident batch: pinned host waveforms in, pinned host slices out.

    The reference's driver hands every (speech, noise) pair to a pool worker and gets numpy arrays back (dp:189-198).
    Here the batch is cut into chunks of `chunk` utterances that go round-robin through `n_streams` CUDA streams, each
    with its own device staging slot: host->device copy, SNR factor + fused forward + floor kernels, device->host copy.
    Copies of one chunk overlap the kernels and copies of its neighbours, consecutive submit() calls keep the ring
    going (no barrier between batches), and nothing synchronises with the host until synchronize()."""

    def __init__(self, engine, L, n_video_slices, chunk=125, n_streams=3, sample_dtype=torch.float32):
        assert sample_dtype in (torch.float32, torch.int16)   # int16: raw WAV samples, decoded inside the kernels
        self.eng = engine
        self.L = int(L)
        self.n_video_slices = int(n_video_slices)
        self.n_slices = engine.n_slices(self.L)
        self.chunk = int(chunk)
        dev = engine.device
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
        self.slots = []
        for _ in range(n_streams):
            self.slots.append({
                "s": torch.empty((self.chunk, self.L), dtype=sample_dtype, device=dev),
                "n": torch.empty((self.chunk, self.L), dtype=sample_dtype, device=dev),
                "snr": torch.zeros((self.chunk,), dtype=torch.float32, device=dev),
                "nlen": torch.zeros((self.chunk,), dtype=torch.int32, device=dev),
                "out": {},
            })
        self._next = 0
        self.launches = 0

    def begin_after(self, stream):
        """Order all pipeline streams after the work already queued on `stream` (e.g. a timing event)."""
        for st in self.streams:
            st.wait_stream(stream)

    def join(self, stream):
        """Make `stream` wait for everything submitted so far."""
        for st in self.streams:
            stream.wait_stream(st)

    def synchronize(self):
        for st in self.streams:
            st.synchronize()

    def submit(self, h_speech, h_noise, h_mixed, h_speech_out, h_noise_out, h_pcm, snr_db=None, noise_lengths=None):
        """Queue one batch.  h_speech / h_noise: pinned [B, L] of the pipeline's sample dtype; h_mixed / h_speech_out /
        h_noise_out: pinned [B, n_slices, 80, 20]; h_pcm: pinned [B, L]; snr_db: optional pinned [B] float32 (None: 0 dB,
        dp:130); noise_lengths: optional pinned [B] int32, the noise files' own lengths -- shorter noises are tiled inside the
        kernels (dp:125-128); without it the noise rows must already cover L.  Returns the number of chunks queued."""
        B = h_speech.shape[0]
        eng = self.eng
        n_chunks = 0
        for lo in range(0, B, self.chunk):
            hi = min(B, lo + self.chunk)
            k = self._next % len(self.streams)
            self._next += 1
            slot, st = self.slots[k], self.streams[k]
            m = hi - lo
            with torch.cuda.stream(st):
                d_s, d_n = slot["s"][:m], slot["n"][:m]
                d_s.copy_(h_speech[lo:hi], non_blocking=True)
                d_n.copy_(h_noise[lo:hi], non_blocking=True)
                snr = None
                if snr_db is not None:
                    snr = slot["snr"][:m]
                    snr.copy_(snr_db[lo:hi], non_blocking=True)
                nlen = None
                if noise_lengths is not None:
                    nlen = slot["nlen"][:m]
                    nlen.copy_(noise_lengths[lo:hi], non_blocking=True)
                out = slot["out"] if m == self.chunk else {}
                factor, keys = eng.snr_factor(d_s, d_n, snr_db=snr, max_key=out.get("max_key"), noise_lengths=nlen)
                r = eng.forward_raw(d_s, d_n, L=self.L, factor=factor, n_slices=self.n_slices, max_key=keys, out=out, noise_lengths=nlen)
                eng.floor3_(r["speech"], r["noise"], r["mixed"], keys)
                h_mixed[lo:hi].copy_(r["mixed"], non_blocking=True)
                h_speech_out[lo:hi].copy_(r["speech"], non_blocking=True)
                h_noise_out[lo:hi].copy_(r["noise"], non_blocking=True)
                h_pcm[lo:hi].copy_(r["mixed_pcm"], non_blocking=True)
            self.launches += 3
            n_chunks += 1
        return n_chunks


def shard_range(n_utterances, rank, world_size):
    """Contiguous utterance range [lo, hi) owned by `rank` (SURVEY 8(e)): utterances are independent units, ranks own
    disjoint ranges and no collective is needed on the data path.  Sizes differ by at most one."""
    base, rem = divmod(int(n_utterances), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class CorpusDriver(object):
    """Product-level multi-GPU driver (SURVEY 8(e), BASELINE configs[2]): ONE corpus, cut into contiguous utterance shards, one
    process per GPU.  Utterances are independent units (the variance of dp:130 and the top_db maximum of dp:94 are
    per-utterance), so there is NO collective on the data path: every rank runs `preprocess` on its own shard in launches of
    at most `launch` utterances.  The only communication is the optional `gather` of the results to one rank at the very end
    (torch.distributed: NCCL over NVLink for CUDA tensors, gloo in the CPU tests), outside the hot path.

    The reference's counterpart is `multiprocess.Pool(16).map` over samples (dp:194-195); `--gpus` is parsed and never read
    (se:283, se:289)."""

    def __init__(self, engine, rank=None, world_size=None, launch=12500):
        import torch.distributed as dist
        self.eng = engine
        ready = dist.is_available() and dist.is_initialized()
        self.rank = int(rank if rank is not None else (dist.get_rank() if ready else 0))
        self.world_size = int(world_size if world_size is not None else (dist.get_world_size() if ready else 1))
        self.launch = int(launch)
        self.launches = 0

    def shard(self, n_utterances):
        """[lo, hi) of this rank."""
        return shard_range(n_utterances, self.rank, self.world_size)

    def preprocess(self, speech, noise, n_video_slices, lengths=None, snr_db=None, noise_lengths=None, out=None):
        """preprocess_audio_pair (dp:119-139) over THIS rank's shard (device tensors [n, >= L]); returns a list with one
        (mixed, speech, noise, mixed_pcm) tuple per launch, or fills / re-uses `out` (a list of dicts from a previous call)."""
        n = speech.shape[0]
        results = []
        outs = out if out is not None else [dict() for _ in range(0, n, self.launch)]
        for j, a in enumerate(range(0, n, self.launch)):
            b = min(n, a + self.launch)
            cut = lambda t: None if t is None else t[a:b]
            results.append(self.eng.preprocess_pairs(speech[a:b], noise[a:b], n_video_slices, lengths=cut(lengths), snr_db=cut(snr_db),
                                                     noise_lengths=cut(noise_lengths), out=outs[j]))
            self.launches += 3
        self.out = outs
        return results

    def gather(self, shard_tensor, n_utterances, dst=0):
        """Optional final gather of a per-utterance result [n_shard, ...] to rank `dst` (None elsewhere); rows come back in
        corpus order.  Shards differ by at most one row, so they are padded to the largest and trimmed after the collective."""
        import torch.distributed as dist
        if self.world_size == 1:
            return shard_tensor
        sizes = [b - a for a, b in (shard_range(n_utterances, r, self.world_size) for r in range(self.world_size))]
        m = max(sizes)
        pad = shard_tensor
        if shard_tensor.shape[0] < m:
            pad = torch.cat([shard_tensor, shard_tensor.new_zeros((m - shard_tensor.shape[0],) + tuple(shard_tensor.shape[1:]))])
        pieces = [torch.empty_like(pad) for _ in range(self.world_size)] if self.rank == dst else None
        dist.gather(pad.contiguous(), pieces, dst=dst)
        if self.rank != dst:
            return None
        return torch.cat([p[:k] for p, k in zip(pieces, sizes)])


def pack_clips(clips, device=None, dtype=torch.float32, allow_empty=True):
    """A list of 1-D clips (numpy arrays, tensors or AudioSignal objects) -> (pool [N, stride], lengths [N] int32) on `device`,
    the layout SpectralEngine.mix_pools and DynamicMixer read: clip k in row k, zeros after its length, stride = the longest
    clip rounded up to a multiple of 4 samples (aligned vector loads).  dtype torch.int16 keeps raw WAV samples (decoded in
    the kernels).  allow_empty=False rejects an empty clip -- pack noise pools that way: a row that draws an empty noise clip
    is invalid (there is nothing to tile, dp:125-126)."""
    datas = [np.asarray(c.get_data() if hasattr(c, "get_data") else (c.cpu().numpy() if torch.is_tensor(c) else c)) for c in clips]
    if not datas:
        raise ValueError("pack_clips: no clips")
    for k, d in enumerate(datas):
        if d.ndim != 1:
            raise ValueError("pack_clips: clip %d is not 1-D (shape %s)" % (k, d.shape))
        if not allow_empty and d.size == 0:
            raise ValueError("pack_clips: clip %d is empty" % k)
    lengths = np.array([d.size for d in datas], dtype=np.int64)
    if lengths.max() > 0x7fffffff:
        raise ValueError("pack_clips: clips longer than 2^31 - 1 samples")
    stride = max(4, (int(lengths.max()) + 3) // 4 * 4)
    np_dtype = np.int16 if dtype == torch.int16 else np.float32
    host = np.zeros((len(datas), stride), dtype=np_dtype)
    for k, d in enumerate(datas):
        host[k, :d.size] = d
    return torch.from_numpy(host).to(device), torch.from_numpy(lengths.astype(np.int32)).to(device)


def pack_video(clips, device=None, dtype=torch.uint8):
    """A list of per-clip video slices [S_k, H, W, F] (numpy arrays or tensors) -> (pool [N, S_max, H, W, F], counts [N] int32)
    on `device`: clip k's slices in row k, zeros after its count.  dtype torch.uint8 keeps the decoder's pixels (a quarter of
    the float32 bytes; values must be integers in [0, 255]), torch.float32 stores them as they are.  SpectralEngine.gather_video
    and DynamicMixer.sample_set decode and normalise the slices they gather."""
    if dtype not in (torch.uint8, torch.float32):
        raise ValueError("pack_video: dtype must be torch.uint8 or torch.float32")
    datas = [c.detach().cpu().numpy() if torch.is_tensor(c) else np.asarray(c) for c in clips]
    if not datas:
        raise ValueError("pack_video: no clips")
    shape = None
    for k, d in enumerate(datas):
        if d.ndim != 4 or (shape is not None and d.shape[1:] != shape):
            raise ValueError("pack_video: clip %d has shape %s; expected [slices, H, W, F] like the others" % (k, d.shape))
        shape = d.shape[1:]
        if dtype == torch.uint8 and d.dtype != np.uint8 and d.size:
            if not (np.all(d >= 0) and np.all(d <= 255) and np.all(d == np.round(d))):
                raise ValueError("pack_video: clip %d holds values that are not uint8 pixels; pack it as float32" % k)
    counts = np.array([d.shape[0] for d in datas], dtype=np.int64)
    host = np.zeros((len(datas), max(1, int(counts.max()))) + tuple(shape), dtype=np.uint8 if dtype == torch.uint8 else np.float32)
    for k, d in enumerate(datas):
        host[k, :d.shape[0]] = d
    return torch.from_numpy(host).to(device), torch.from_numpy(counts.astype(np.int32)).to(device)


def draw_pairings(generator, B, n_speech, noise_lengths, snr_db=(-10.0, 10.0)):
    """The random pairing of one DynamicMixer epoch, drawn on the host from `generator` (a CPU torch.Generator: the same seed
    gives the same pairing on any machine).  Returns CPU tensors (speech_index int64, noise_index int64, noise_offset int32,
    snr_db float32), each [B]:
      speech_index -- a fresh permutation of range(n_speech), repeated and cut to B: every clip appears floor(B / n_speech)
                      or ceil(B / n_speech) times;
      noise_index  -- uniform over the noise pool (noise_lengths [Nn], all > 0);
      noise_offset -- uniform in [0, Ln) of the drawn noise clip;
      snr_db       -- uniform in [lo, hi) for a (lo, hi) tuple, a uniform choice among the values of a list, or a constant."""
    B, n_speech = int(B), int(n_speech)
    nl = torch.as_tensor(noise_lengths).to("cpu", torch.int64)
    if B <= 0 or n_speech <= 0 or nl.numel() == 0:
        raise ValueError("draw_pairings: need B > 0 and non-empty pools")
    if bool((nl <= 0).any()):
        raise ValueError("draw_pairings: empty noise clip in the pool")
    perm = torch.randperm(n_speech, generator=generator)
    speech_index = perm.repeat((B + n_speech - 1) // n_speech)[:B].contiguous()
    noise_index = torch.randint(0, nl.numel(), (B,), generator=generator, dtype=torch.int64)
    ln = nl[noise_index]
    u = torch.rand(B, generator=generator, dtype=torch.float64)
    noise_offset = torch.minimum((u * ln.to(torch.float64)).to(torch.int64), ln - 1).to(torch.int32)
    if isinstance(snr_db, tuple):
        lo, hi = float(snr_db[0]), float(snr_db[1])
        snr = (lo + (hi - lo) * torch.rand(B, generator=generator, dtype=torch.float64)).to(torch.float32)
    elif isinstance(snr_db, (list, np.ndarray)) or torch.is_tensor(snr_db):
        values = torch.as_tensor(np.asarray(snr_db, dtype=np.float32).reshape(-1))
        snr = values[torch.randint(0, values.numel(), (B,), generator=generator, dtype=torch.int64)]
    else:
        snr = torch.full((B,), float(snr_db), dtype=torch.float32)
    return speech_index, noise_index, noise_offset, snr.contiguous()


class DynamicMixer(object):
    """Fresh (speech, noise, noise offset, SNR) combinations every training epoch, mixed on the device from two clip pools
    without materialising any pairing (SpectralEngine.mix_pools).  The reference mixes each speech file with one noise file
    once, at 0 dB from noise sample 0, and re-reads those frozen mixtures every epoch (speech_enhancer.py:17-58).

    Every row is L = samples_per_slice * n_video_slices samples long.  Without clip_slices a row is the start of its speech
    clip (all clips of such a mixer should share one duration, as preprocess_data buckets).  With clip_slices [Ns] -- each
    speech clip's min(video, audio) slice count (dp:164) -- clips of any length share one mixer: every row is a window that
    starts on a random slice boundary k of its clip, k uniform in [0, max(0, clip_slices[s] - n_video_slices)], so every part
    of a long clip is trained on.  video_pool = pack_video(...)'s (pool, counts) lets sample_set gather the matching video
    slices on the device.

    Pairings come from the mixer's own torch.Generator (seeded with `seed`), window starts from a second one seeded from the
    same `seed`: the same seed and the same sequence of calls give bit-identical epochs, and the pairings of a seed are the
    same with and without windows.  In a multi-GPU job give every rank its own seed.

    One epoch::

        speech_pool, speech_len = pack_clips(speech_clips, eng.device)
        noise_pool, noise_len = pack_clips(noise_clips, eng.device, allow_empty=False)
        video = pack_video(video_clips, eng.device)                     # uint8 [Ns, S_max, H, W, F], counts [Ns]
        mixer = DynamicMixer(eng, speech_pool, speech_len, noise_pool, noise_len, n_video_slices=15, snr_db=(-10.0, 10.0),
                             seed=rank, clip_slices=clip_slices, video_pool=video)
        for epoch in range(n_epochs):
            pairing = mixer.draw(3 * len(speech_clips))                 # three noisy windows of every clip per epoch
            mixed, speech, noise, pcm, valid = mixer.mix(pairing)
            X_video, X_mixed, X_speech, perm = mixer.sample_set(pairing, mixed, speech, valid, normalizer=normalizer)
    """

    def __init__(self, engine, speech_pool, speech_lengths, noise_pool, noise_lengths, n_video_slices, snr_db=(-10.0, 10.0), seed=0,
                 clip_slices=None, video_pool=None):
        self.eng = engine
        self.device = engine.device
        self.speech_pool, self.noise_pool = speech_pool, noise_pool
        self.speech_lengths = torch.as_tensor(speech_lengths).to(self.device, torch.int32)
        self.noise_lengths = torch.as_tensor(noise_lengths).to(self.device, torch.int32)
        self._noise_lengths_host = self.noise_lengths.cpu()           # the offset draw needs them on the host (one copy, here)
        if bool((self._noise_lengths_host <= 0).any()):
            raise ValueError("DynamicMixer: the noise pool holds an empty clip (pack it with pack_clips(..., allow_empty=False))")
        self.n_video_slices = int(n_video_slices)
        self.snr_db = snr_db
        self.generator = torch.Generator()
        self.generator.manual_seed(int(seed))
        Ns = speech_pool.shape[0]
        self.clip_slices = None
        if clip_slices is not None:
            cs = torch.as_tensor(np.asarray(clip_slices) if not torch.is_tensor(clip_slices) else clip_slices).to("cpu", torch.int64)
            if cs.shape != (Ns,) or bool((cs < 0).any()):
                raise ValueError("DynamicMixer: clip_slices must hold one slice count >= 0 per speech clip (%d)" % Ns)
            self._clip_slices_host = cs
            self.clip_slices = cs.to(self.device)
            # window starts: a second generator, so the pairing sequence of a seed does not depend on whether windows are drawn
            self.start_generator = torch.Generator()
            self.start_generator.manual_seed((int(seed) * 0x9E3779B97F4A7C15 + 0x632BE59BD9B4E019) % (1 << 64))
        self.video_pool = self.video_counts = None
        if video_pool is not None:
            pool, counts = video_pool
            counts = torch.as_tensor(counts).to("cpu", torch.int64)
            if self.clip_slices is None:
                raise ValueError("DynamicMixer: video_pool needs clip_slices (the slices of each clip the audio may use)")
            if pool.dim() != 5 or pool.shape[0] != Ns or counts.shape != (Ns,):
                raise ValueError("DynamicMixer: video_pool must be pack_video's (pool [Ns, S_max, H, W, F], counts [Ns])")
            if bool((self._clip_slices_host > counts).any()):
                raise ValueError("DynamicMixer: clip_slices exceeds the video slices stored for a clip")
            self.video_pool = pool.to(self.device).contiguous()
            self.video_counts = counts.to(self.device)

    def draw(self, B):
        """(speech_index, noise_index, noise_offset, snr_db) device tensors of B fresh rows (see draw_pairings); with
        clip_slices, a fifth tensor speech_start [B] int32 = samples_per_slice * k, k uniform in
        [0, max(0, clip_slices[speech_index] - n_video_slices)]."""
        pairing = draw_pairings(self.generator, B, self.speech_pool.shape[0], self._noise_lengths_host, self.snr_db)
        if self.clip_slices is not None:
            kmax = (self._clip_slices_host[pairing[0]] - self.n_video_slices).clamp(min=0)
            u = torch.rand(int(B), generator=self.start_generator, dtype=torch.float64)
            k = torch.minimum((u * (kmax + 1).to(torch.float64)).to(torch.int64), kmax)
            pairing = pairing + ((k * self.eng.samples_per_slice).to(torch.int32),)
        return tuple(t.to(self.device) for t in pairing)

    def mix(self, pairing, out=None):
        """mix_pools of a drawn pairing (4-tuple, or 5-tuple with speech_start): (mixed, speech, noise, mixed_pcm, valid),
        valid [B] bool = row valid and factor finite (a silent noise window gives inf / nan).  Asynchronous: nothing is read
        back."""
        info = {}
        si, ni, off, snr = pairing[:4]
        start = pairing[4] if len(pairing) > 4 else None
        mixed, speech, noise, pcm = self.eng.mix_pools(self.speech_pool, self.speech_lengths, self.noise_pool, self.noise_lengths, si, ni,
                                                       self.n_video_slices, noise_offset=off, snr_db=snr, out=out, info=info, check=False,
                                                       speech_start=start)
        return mixed, speech, noise, pcm, info["valid"]

    def _rows(self, pairing, n, valid):
        """Per row: its first video slice k_b (speech_start / samples_per_slice) and kept slice count n_b."""
        si = pairing[0].to(self.device, torch.int64)
        k = torch.zeros_like(si)
        if len(pairing) > 4:
            k = pairing[4].to(self.device, torch.int64) // self.eng.samples_per_slice
        if self.clip_slices is not None:
            nb = (self.clip_slices[si] - k).clamp(0, n)
        else:
            nb = torch.full_like(si, n)
        nb = torch.where(torch.as_tensor(valid, device=self.device), nb, torch.zeros_like(nb))
        return si, k, nb

    def sample_set(self, pairing, mixed, speech, valid, normalizer=None, permutation=None, generator=None):
        """make_sample_set of one mixed batch together with its video: (video [N, H, W, F] float32, X_mixed, X_speech,
        permutation).  Row b keeps n_b = min(clip_slices[s_b] - k_b, n) slices (n = the batch's slice count, k_b = the window's
        first slice, 0 without windows; 0 slices for a row that is not valid).  Video row r is slice k_b + j of clip s_b where
        (b, j) is concatenated row permutation[r], so video and audio rows stay paired; with a VideoNormalizer it is normalised
        as normalizer.normalize would.  video is None when the mixer has no video_pool."""
        n = int(mixed.shape[1])
        si, k, nb = self._rows(pairing, n, valid)
        X_mixed, X_speech, perm = self.eng.make_sample_set(mixed, speech, n_slices=nb, permutation=permutation, generator=generator)
        video = None
        if self.video_pool is not None:
            index = video_slice_index(si, k, nb, n, int(self.video_pool.shape[1]), perm)
            video = self.eng.gather_video(self.video_pool, index, normalizer=normalizer, check=False)
        return video, X_mixed, X_speech, perm


def video_slice_index(speech_index, first_slice, n_slices, n, s_max, permutation):
    """Video slice indices (into a pack_video pool flattened to [Ns * s_max] slices) of the concatenated rows permutation[r],
    in make_sample_set's order (sample-major, slice-minor, rows j < n_slices[b] of each sample b of n): concatenated row (b, j)
    is clip speech_index[b], slice first_slice[b] + j.  All tensors on one device; returns int64 [N]."""
    dev = speech_index.device
    j = torch.arange(int(n), device=dev, dtype=torch.int64)
    keep = j.unsqueeze(0) < n_slices.to(dev, torch.int64).unsqueeze(1)
    src = (speech_index.to(torch.int64) * int(s_max) + first_slice.to(dev, torch.int64)).unsqueeze(1) + j.unsqueeze(0)
    return src[keep][torch.as_tensor(permutation, device=dev, dtype=torch.int64)].contiguous()


def fit_noise(noise, n_noise, n_speech_max):
    """dp:125-128 for a batch as an explicit copy: periodic tiling noise[i mod n_noise] up to the speech length.  The
    product path does not need it (pass `noise_lengths` to preprocess_pairs: the kernels address noise[i mod Ln]
    themselves); kept for callers that want the fitted noise as a tensor."""
    idx = torch.arange(n_speech_max, device=noise.device) % int(n_noise)
    return noise[..., :n_noise].index_select(-1, idx).contiguous()
