"""ctypes binding of ``liblidfe.so`` (the C ABI declared in ``include/lidfe.h``).

There is no CPU fallback: if the shared library has not been built, importing the compute entry
points raises immediately with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LIDFE_LIB_PATH: development only (load a library built elsewhere, e.g. from another commit, to compare the two)
LIB_PATH = os.environ.get("LIDFE_LIB_PATH") or os.path.join(_HERE, "liblidfe.so")

# include/lidfe.h
E_NULL, E_CONFIG, E_SHORT, E_OFFSETS, E_ARG, E_MELBANK, E_NOMEM = -1, -2, -3, -4, -5, -6, -7
IN_F32, IN_I16 = 0, 1
CMVN_NONE, CMVN_PER_UTT, CMVN_APPLY_GLOBAL, CMVN_ACCUM_GLOBAL, POST_TOPDB = 0, 1, 2, 3, 4
FRAMING_KALDI, FRAMING_CENTER = 0, 1
LOG_NATURAL, LOG_DB10 = 0, 1
ABI_VERSION = 8
WINDOW_POVEY, WINDOW_HANNING, WINDOW_HAMMING, WINDOW_RECTANGULAR, WINDOW_BLACKMAN, WINDOW_HANN_PERIODIC = 0, 1, 2, 3, 4, 5

EXPORTS = (
    "lidfe_create", "lidfe_destroy", "lidfe_num_frames", "lidfe_out_dim", "lidfe_plan_create",
    "lidfe_plan_destroy", "lidfe_plan_total_frames", "lidfe_plan_num_tiles", "lidfe_plan_frames",
    "lidfe_featurize", "lidfe_cmvn_apply", "lidfe_wave_stages", "lidfe_wave_stages_i16", "lidfe_mask_apply", "lidfe_strerror",
    "lidfe_abi_version", "lidfe_launch_count", "lidfe_profile_begin", "lidfe_profile_end", "lidfe_profile_set_stride", "lidfe_mel_plan", "lidfe_mel_plan_expand",
    "lidfe_resampler_create", "lidfe_resampler_destroy", "lidfe_resample_out_len", "lidfe_resample",
    "lidfe_plan_create_async", "lidfe_plan_num_spans", "lidfe_featurize_raw", "lidfe_fp32_probe", "lidfe_pool_stats", "lidfe_pack_host", "lidfe_h2d_gather", "lidfe_wgemm_create", "lidfe_stft_mel_db",
    "lidfe_set_precision", "lidfe_add_noise",
)


class LidfeConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_int), ("frame_len", C.c_int), ("frame_shift", C.c_int),
                ("fft_len", C.c_int), ("n_mels", C.c_int), ("n_ceps", C.c_int), ("preemph", C.c_float),
                ("remove_dc", C.c_int), ("log_floor", C.c_float), ("in_dtype", C.c_int),
                ("in_scale", C.c_float), ("framing", C.c_int), ("pad", C.c_int), ("log_kind", C.c_int),
                ("top_db", C.c_float), ("dither", C.c_float), ("window_type", C.c_int),
                ("seed", C.c_ulonglong)]


class LidfeError(RuntimeError):
    def __init__(self, rc: int, msg: str):
        super().__init__("%s (rc=%d)" % (msg, rc))
        self.rc = rc


_lib = None


def load_library() -> C.CDLL:
    """dlopen liblidfe.so and declare every prototype.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "speech_lid_b200: %s is missing -- the sm_100a extension has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` in the repo root. "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, ll, i32, f32 = C.c_void_p, C.c_longlong, C.c_int, C.c_float
    pll = C.POINTER(C.c_longlong)
    lib.lidfe_create.argtypes = [C.POINTER(vp), C.POINTER(LidfeConfig), vp, vp, vp, vp]
    lib.lidfe_create.restype = i32
    lib.lidfe_destroy.argtypes = [vp]
    lib.lidfe_destroy.restype = i32
    lib.lidfe_num_frames.argtypes = [ll, C.POINTER(LidfeConfig)]
    lib.lidfe_num_frames.restype = ll
    lib.lidfe_out_dim.argtypes = [vp]
    lib.lidfe_out_dim.restype = i32
    lib.lidfe_plan_create.argtypes = [vp, C.POINTER(vp), i32, pll, pll, pll, pll]
    lib.lidfe_plan_create.restype = i32
    lib.lidfe_plan_create_async.argtypes = [vp, C.POINTER(vp), i32, pll, pll, pll, pll, vp]
    lib.lidfe_plan_create_async.restype = i32
    lib.lidfe_plan_destroy.argtypes = [vp]
    lib.lidfe_plan_destroy.restype = i32
    for name in ("lidfe_plan_total_frames", "lidfe_plan_num_tiles", "lidfe_plan_num_spans"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = ll
    lib.lidfe_plan_frames.argtypes = [vp, i32]
    lib.lidfe_plan_frames.restype = ll
    lib.lidfe_featurize.argtypes = [vp, vp, vp, vp, ll, vp, i32, i32, vp, vp, vp]
    lib.lidfe_featurize.restype = i32
    lib.lidfe_featurize_raw.argtypes = [vp, vp, vp, vp, ll, vp, i32, i32, vp, vp, vp]
    lib.lidfe_featurize_raw.restype = i32
    lib.lidfe_fp32_probe.argtypes = [f32, C.POINTER(C.c_double), vp]
    lib.lidfe_fp32_probe.restype = i32
    lib.lidfe_set_precision.argtypes = [vp, i32]
    lib.lidfe_set_precision.restype = i32
    lib.lidfe_pool_stats.argtypes = [vp, pll, pll]
    lib.lidfe_pool_stats.restype = i32
    lib.lidfe_pack_host.argtypes = [vp, C.POINTER(vp), pll, pll, i32, i32, ll, i32]
    lib.lidfe_pack_host.restype = i32
    lib.lidfe_h2d_gather.argtypes = [vp, C.POINTER(vp), pll, pll, i32, i32, vp]
    lib.lidfe_h2d_gather.restype = i32
    lib.lidfe_wgemm_create.argtypes = [C.POINTER(vp), i32, i32, vp, i32, i32]
    lib.lidfe_wgemm_create.restype = i32
    lib.lidfe_stft_mel_db.argtypes = [vp, vp, vp, i32, ll, i32, vp, vp, vp, i32, i32, f32, vp, vp, vp, i32, vp]
    lib.lidfe_stft_mel_db.restype = i32
    lib.lidfe_cmvn_apply.argtypes = [vp, vp, vp, ll, vp, i32, vp, vp]
    lib.lidfe_cmvn_apply.restype = i32
    lib.lidfe_mask_apply.argtypes = [vp, vp, vp, ll, vp, i32, vp]
    lib.lidfe_mask_apply.restype = i32
    lib.lidfe_wave_stages.argtypes = [vp, vp, vp, vp, i32, f32, vp, f32, vp]
    lib.lidfe_wave_stages.restype = i32
    lib.lidfe_profile_set_stride.argtypes = [vp, i32]
    lib.lidfe_profile_set_stride.restype = i32
    lib.lidfe_profile_begin.argtypes = [vp, i32]
    lib.lidfe_profile_begin.restype = i32
    lib.lidfe_profile_end.argtypes = [vp, C.POINTER(C.c_float), i32, C.POINTER(C.c_int)]
    lib.lidfe_profile_end.restype = i32
    pi = C.POINTER(C.c_int)
    lib.lidfe_mel_plan.argtypes = [i32, vp, pi, pi, pi, pi]
    lib.lidfe_mel_plan.restype = i32
    lib.lidfe_mel_plan_expand.argtypes = [i32, vp, vp]
    lib.lidfe_mel_plan_expand.restype = i32
    lib.lidfe_resampler_create.argtypes = [C.POINTER(vp), i32, i32, vp, i32, i32]
    lib.lidfe_resampler_create.restype = i32
    lib.lidfe_resampler_destroy.argtypes = [vp]
    lib.lidfe_resampler_destroy.restype = i32
    lib.lidfe_resample_out_len.argtypes = [vp, ll]
    lib.lidfe_resample_out_len.restype = ll
    lib.lidfe_resample.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, ll, vp]
    lib.lidfe_resample.restype = i32
    lib.lidfe_wave_stages_i16.argtypes = [vp, vp, vp, f32, vp, i32, f32, vp, f32, vp]
    lib.lidfe_wave_stages_i16.restype = i32
    lib.lidfe_add_noise.argtypes = [vp, vp, vp, i32, f32, vp, vp, ll, vp, vp, C.c_ulonglong, i32, vp]
    lib.lidfe_add_noise.restype = i32
    lib.lidfe_strerror.argtypes = [i32]
    lib.lidfe_strerror.restype = C.c_char_p
    lib.lidfe_abi_version.argtypes = []
    lib.lidfe_abi_version.restype = i32
    lib.lidfe_launch_count.argtypes = []
    lib.lidfe_launch_count.restype = ll
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Map a non-zero return code to an exception, mirroring the reference's error behaviour:
    a too-short utterance raises AssertionError like ``torchaudio.compliance.kaldi`` does
    (ta: compliance/kaldi.py:142); everything else is a RuntimeError."""
    if rc == 0:
        return
    msg = load_library().lidfe_strerror(rc).decode()
    if rc == E_SHORT:
        raise AssertionError(msg)
    raise LidfeError(rc, msg)
