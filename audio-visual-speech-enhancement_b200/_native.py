"""ctypes binding of libavse_b200.so (the C ABI declared in include/avse_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or no CUDA device is present,
calls raise.  PyTorch is used only as plumbing (device buffers, streams)."""
from __future__ import annotations

import ctypes
import os

from .build import LIB_PATH, build_library

_c = ctypes
_lib = None


class ForwardArgs(_c.Structure):
    _fields_ = [
        ("speech", _c.c_void_p), ("noise", _c.c_void_p), ("in_stride", _c.c_longlong),
        ("len_speech", _c.c_void_p), ("len_noise", _c.c_void_p), ("factor", _c.c_void_p),
        ("B", _c.c_int), ("L", _c.c_int),
        ("layout", _c.c_int), ("n_slices", _c.c_int), ("ld_t", _c.c_int),
        ("out_speech", _c.c_void_p), ("out_noise", _c.c_void_p), ("out_mixed", _c.c_void_p),
        ("out_stride", _c.c_longlong),
        ("mixed_pcm", _c.c_void_p), ("pcm_stride", _c.c_longlong),
        ("max_key", _c.c_void_p),
        ("stft_speech", _c.c_void_p),
        ("min_key", _c.c_void_p),
        ("sample_format", _c.c_int),
        ("equalizer", _c.c_void_p),
        ("noise_period", _c.c_void_p),
    ]


class InverseArgs(_c.Structure):
    _fields_ = [
        ("mel_db", _c.c_void_p), ("layout", _c.c_int), ("n_slices", _c.c_int), ("n_frames", _c.c_int), ("ld_t", _c.c_int),
        ("mel_stride", _c.c_longlong),
        ("mixed_pcm", _c.c_void_p), ("pcm_stride", _c.c_longlong), ("len_pcm", _c.c_void_p),
        ("B", _c.c_int), ("L", _c.c_int),
        ("out_pcm", _c.c_void_p), ("out_stride", _c.c_longlong),
        ("work", _c.c_void_p), ("work_stride", _c.c_longlong),
        ("phase", _c.c_void_p), ("phase_stride", _c.c_longlong), ("phase_frames", _c.c_int),
        ("out_format", _c.c_int),
    ]


class PoolMixArgs(_c.Structure):
    _fields_ = [
        ("speech_pool", _c.c_void_p), ("speech_len", _c.c_void_p), ("speech_stride", _c.c_longlong), ("n_speech", _c.c_longlong),
        ("noise_pool", _c.c_void_p), ("noise_len", _c.c_void_p), ("noise_stride", _c.c_longlong), ("n_noise", _c.c_longlong),
        ("sample_format", _c.c_int),
        ("speech_index", _c.c_void_p), ("noise_index", _c.c_void_p), ("noise_offset", _c.c_void_p), ("snr_db", _c.c_void_p),
        ("B", _c.c_int), ("L", _c.c_int), ("n_slices", _c.c_int),
        ("out_speech", _c.c_void_p), ("out_noise", _c.c_void_p), ("out_mixed", _c.c_void_p), ("out_stride", _c.c_longlong),
        ("mixed_pcm", _c.c_void_p), ("pcm_stride", _c.c_longlong),
        ("factor_out", _c.c_void_p), ("equalizer_out", _c.c_void_p),
        ("max_key", _c.c_void_p), ("min_key", _c.c_void_p), ("bad_row_flag", _c.c_void_p),
        ("speech_start", _c.c_void_p),
    ]


EXPORTS = [
    "avse_create", "avse_destroy", "avse_last_error", "avse_version", "avse_get_filterbank",
    "avse_snr_factor", "avse_forward", "avse_floor_inplace", "avse_floor_gather", "avse_reset_max", "avse_max_db",
    "avse_inverse", "avse_inverse_work_elems", "avse_floor_inplace3", "avse_gather_rows",
    "avse_create_ex", "avse_get_geometry", "avse_inverse_work_elems_ctx",
    "avse_video_stats", "avse_video_normalize", "avse_mse", "avse_magphase", "avse_mix_pooled", "avse_inverse_backward",
    "avse_gather_video",
]


def load(build=True):
    """Load (building if needed) libavse_b200.so and declare prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("AVSE_B200_LIB")  # tuning experiments: a variant build of the same sources
    if not path:
        if build:
            build_library()
        path = LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError("libavse_b200.so is missing; run `python -m __graft_entry__` / build() first (no CPU fallback exists)")
    lib = _c.CDLL(path)
    vp, ll, i32, f64 = _c.c_void_p, _c.c_longlong, _c.c_int, _c.c_double
    lib.avse_create.argtypes = [i32, f64, f64, i32, _c.POINTER(vp)]
    lib.avse_create.restype = i32
    lib.avse_destroy.argtypes = [vp]
    lib.avse_destroy.restype = None
    lib.avse_last_error.restype = _c.c_char_p
    lib.avse_version.restype = _c.c_char_p
    lib.avse_get_filterbank.argtypes = [vp, vp]
    lib.avse_get_filterbank.restype = i32
    lib.avse_snr_factor.argtypes = [vp, vp, vp, i32, ll, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    lib.avse_snr_factor.restype = i32
    lib.avse_forward.argtypes = [vp, _c.POINTER(ForwardArgs), vp]
    lib.avse_forward.restype = i32
    lib.avse_floor_inplace.argtypes = [vp, vp, ll, ll, i32, vp, vp, i32, vp]
    lib.avse_floor_inplace.restype = i32
    lib.avse_floor_inplace3.argtypes = [vp, vp, vp, vp, ll, ll, i32, vp, vp, vp]
    lib.avse_floor_inplace3.restype = i32
    lib.avse_floor_gather.argtypes = [vp, vp, ll, i32, vp, ll, i32, i32, vp, i32, vp]
    lib.avse_floor_gather.restype = i32
    lib.avse_reset_max.argtypes = [vp, vp, vp, i32, vp]
    lib.avse_reset_max.restype = i32
    lib.avse_max_db.argtypes = [vp, vp, i32, vp, vp]
    lib.avse_max_db.restype = i32
    lib.avse_inverse.argtypes = [vp, _c.POINTER(InverseArgs), vp]
    lib.avse_inverse.restype = i32
    lib.avse_inverse_backward.argtypes = [vp, _c.POINTER(InverseArgs), vp, ll, vp, vp]
    lib.avse_inverse_backward.restype = i32
    lib.avse_inverse_work_elems.argtypes = [i32, _c.POINTER(ll)]
    lib.avse_inverse_work_elems.restype = i32
    lib.avse_create_ex.argtypes = [i32, i32, i32, i32, i32, f64, f64, i32, _c.POINTER(vp)]
    lib.avse_create_ex.restype = i32
    lib.avse_get_geometry.argtypes = [vp, _c.POINTER(i32 * 6)]
    lib.avse_get_geometry.restype = i32
    lib.avse_inverse_work_elems_ctx.argtypes = [vp, i32, _c.POINTER(ll)]
    lib.avse_inverse_work_elems_ctx.restype = i32
    lib.avse_video_stats.argtypes = [vp, vp, ll, i32, i32, vp, vp, vp, vp]
    lib.avse_video_stats.restype = i32
    lib.avse_video_normalize.argtypes = [vp, vp, ll, i32, i32, vp, vp, vp]
    lib.avse_video_normalize.restype = i32
    lib.avse_mse.argtypes = [vp, vp, vp, ll, vp, vp, vp]
    lib.avse_mse.restype = i32
    lib.avse_magphase.argtypes = [vp, vp, ll, i32, i32, vp, vp, vp]
    lib.avse_magphase.restype = i32
    lib.avse_gather_rows.argtypes = [vp, vp, vp, vp, ll, ll, vp, ll, vp, vp, vp, vp, vp]
    lib.avse_gather_rows.restype = i32
    lib.avse_mix_pooled.argtypes = [vp, _c.POINTER(PoolMixArgs), vp]
    lib.avse_mix_pooled.restype = i32
    lib.avse_gather_video.argtypes = [vp, vp, i32, ll, i32, i32, vp, ll, vp, vp, vp, vp, vp]
    lib.avse_gather_video.restype = i32
    _lib = lib
    return lib


class AvseError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = load().avse_last_error().decode("utf-8", "replace")
        raise AvseError("%s failed (%d): %s" % (what, rc, msg))
