"""ctypes binding of ``libwefax_b200.so`` (the C-ABI in ``include/wefax_b200.h``).

There is no CPU fallback: if the library is missing it must be built
(``python -m wefax_b200.build``), and creating a context without a CUDA device
raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WEFAX_B200_LIB") or os.path.join(HERE, "libwefax_b200.so")   # override: A/B builds

MAX_PEAKS = 100
TARGET_RATE = 11025

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = 0, 1, 2, 3, 4
REC_OK, REC_NO_GROUPS, REC_NO_LINES, REC_NAN = 0, 1, 2, 4
F_PCM_ON_DEVICE, F_OUT_ON_DEVICE, F_PCM_FLOAT32 = 1, 2, 4

#: every symbol include/wefax_b200.h declares
EXPORTED_SYMBOLS = (
    "wefax_ctx_create", "wefax_ctx_destroy", "wefax_last_error", "wefax_ctx_sync", "wefax_ctx_stream",
    "wefax_ctx_launch_count", "wefax_ctx_set_workspace_limit", "wefax_abi_version", "wefax_device_count",
    "wefax_line_constants_for", "wefax_resampled_length", "wefax_notch_coefficients",
    "wefax_fft_plan_describe", "wefax_decode_batch", "wefax_fft_c2c", "wefax_hilbert_envelope",
    "wefax_resample", "wefax_filtfilt", "wefax_digitalize", "wefax_sync_raster",
    "wefax_ctx_enable_timing", "wefax_ctx_timings", "wefax_tone_scan", "wefax_decode_fm",
    "wefax_segment_envelope", "wefax_segment_histogram", "wefax_segment_quantise", "wefax_segment_sync",
    "wefax_segment_raster", "wefax_sync_pulse_scan", "wefax_segment_select_init", "wefax_segment_histogram_dev",
    "wefax_segment_select_dev", "wefax_segment_quantise_dev", "wefax_decode_fm_slant",
)
ABI_VERSION = 5


class LineConstants(C.Structure):
    _fields_ = [("frame_len", C.c_double), ("n1", C.c_int), ("n0", C.c_int), ("template_len", C.c_int),
                ("mindistance", C.c_int), ("width", C.c_int), ("dev_min", C.c_double), ("dev_max", C.c_double)]


class BatchDesc(C.Structure):
    _fields_ = [("n_recordings", C.c_int), ("n_frames", C.c_longlong), ("channels", C.c_int),
                ("sample_rate", C.c_int), ("notch_freq", C.c_double), ("notch_q", C.c_double),
                ("flags", C.c_uint)]


class BatchOut(C.Structure):
    _fields_ = [("audio", C.c_void_p), ("demodulated", C.c_void_p), ("digitalized", C.c_void_p),
                ("peaks", C.c_void_p), ("n_peaks", C.c_void_p), ("phasing", C.c_void_p),
                ("n_phasing", C.c_void_p), ("start_frame", C.c_void_p), ("height", C.c_void_p),
                ("status", C.c_void_p), ("low_high", C.c_void_p), ("raster", C.c_void_p),
                ("raster_stride", C.c_longlong)]


class ToneSettings(C.Structure):
    _fields_ = [("start_distance", C.c_double), ("stop_distance", C.c_double), ("height", C.c_double),
                ("prominence", C.c_double), ("min_frequency", C.c_double), ("max_frequency", C.c_double),
                ("min_amount", C.c_int), ("max_amount", C.c_int)]


class SyncPulseSettings(C.Structure):
    _fields_ = [("height", C.c_double), ("prominence", C.c_double), ("min_frequency", C.c_double),
                ("max_frequency", C.c_double), ("notch_freq", C.c_double), ("notch_q", C.c_double)]


MAX_PULSES = 16
SEG_STATE_HIST, SEG_STATE_WORDS = 32, 32 + 4 * 2048


class FmParams(C.Structure):
    _fields_ = [("lpm", C.c_double), ("ioc", C.c_int), ("black_hz", C.c_double), ("white_hz", C.c_double),
                ("band_lo_hz", C.c_double), ("band_hi_hz", C.c_double), ("fir_taps", C.c_int),
                ("search_from", C.c_longlong), ("fold_lines", C.c_int), ("image_end", C.c_longlong)]


class FmOut(C.Structure):
    _fields_ = [("grey", C.c_void_p), ("image", C.c_void_p), ("image_capacity", C.c_longlong),
                ("rows", C.c_void_p), ("width", C.c_void_p), ("line_start", C.c_void_p)]


FM_SLANT_OFF, FM_SLANT_FIXED, FM_SLANT_AUTO = 0, 1, 2
FM_SLANT_OK, FM_SLANT_NOT_FOUND = 0, 1
FM_SLANT_MAX_PPM = 2000.0


class FmSlant(C.Structure):
    _fields_ = [("mode", C.c_int), ("ppm", C.c_double), ("max_ppm", C.c_double), ("min_contrast", C.c_double),
                ("min_lines", C.c_int)]


class FmSlantOut(C.Structure):
    _fields_ = [("line_length", C.c_double), ("ppm", C.c_double), ("first_line", C.c_double),
                ("lines_total", C.c_int32), ("lines_used", C.c_int32), ("residual_rms", C.c_double),
                ("status", C.c_int32)]


class NativeLibraryMissing(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} is not built; run `python -m wefax_b200.build` (needs nvcc). "
            "wefax_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i, ll, d = C.c_void_p, C.c_int, C.c_longlong, C.c_double
    lib.wefax_ctx_create.argtypes = [i, vp, C.POINTER(vp)]
    lib.wefax_ctx_create.restype = i
    lib.wefax_ctx_destroy.argtypes = [vp]
    lib.wefax_ctx_destroy.restype = None
    lib.wefax_last_error.argtypes = [vp]
    lib.wefax_last_error.restype = C.c_char_p
    lib.wefax_ctx_sync.argtypes = [vp]
    lib.wefax_ctx_sync.restype = i
    lib.wefax_ctx_stream.argtypes = [vp]
    lib.wefax_ctx_stream.restype = vp
    lib.wefax_ctx_launch_count.argtypes = [vp]
    lib.wefax_ctx_launch_count.restype = ll
    lib.wefax_ctx_set_workspace_limit.argtypes = [vp, ll]
    lib.wefax_ctx_set_workspace_limit.restype = i
    lib.wefax_ctx_enable_timing.argtypes = [vp, i]
    lib.wefax_ctx_enable_timing.restype = i
    lib.wefax_ctx_timings.argtypes = [vp, C.c_char_p, ll, i]
    lib.wefax_ctx_timings.restype = i
    lib.wefax_abi_version.argtypes = []
    lib.wefax_abi_version.restype = i
    lib.wefax_device_count.argtypes = []
    lib.wefax_device_count.restype = i
    lib.wefax_line_constants_for.argtypes = [d, i, C.POINTER(LineConstants)]
    lib.wefax_line_constants_for.restype = i
    lib.wefax_resampled_length.argtypes = [ll, i]
    lib.wefax_resampled_length.restype = ll
    lib.wefax_notch_coefficients.argtypes = [d, d, d, C.POINTER(d * 3), C.POINTER(d * 3)]
    lib.wefax_notch_coefficients.restype = i
    lib.wefax_fft_plan_describe.argtypes = [ll, C.POINTER(i), C.POINTER(i * 8), C.POINTER(ll)]
    lib.wefax_fft_plan_describe.restype = i
    lib.wefax_decode_batch.argtypes = [vp, C.POINTER(BatchDesc), vp, vp, C.POINTER(BatchOut)]
    lib.wefax_decode_batch.restype = i
    lib.wefax_fft_c2c.argtypes = [vp, ll, i, vp, vp, i]
    lib.wefax_fft_c2c.restype = i
    lib.wefax_hilbert_envelope.argtypes = [vp, ll, i, vp, vp]
    lib.wefax_hilbert_envelope.restype = i
    lib.wefax_resample.argtypes = [vp, ll, ll, i, vp, vp]
    lib.wefax_resample.restype = i
    lib.wefax_filtfilt.argtypes = [vp, ll, i, d, d, vp, vp]
    lib.wefax_filtfilt.restype = i
    lib.wefax_digitalize.argtypes = [vp, ll, i, vp, vp, vp, vp, vp]
    lib.wefax_digitalize.restype = i
    lib.wefax_sync_raster.argtypes = [vp, ll, i, vp, vp, C.POINTER(BatchOut)]
    lib.wefax_sync_raster.restype = i
    lib.wefax_tone_scan.argtypes = [vp, vp, ll, i, i, ll, C.c_uint, C.POINTER(ToneSettings), vp, vp, vp, vp]
    lib.wefax_tone_scan.restype = i
    lib.wefax_sync_pulse_scan.argtypes = [vp, vp, ll, i, i, ll, C.c_uint, C.POINTER(SyncPulseSettings), vp, vp, vp, vp, vp,
                                          vp, vp]
    lib.wefax_sync_pulse_scan.restype = i
    lib.wefax_decode_fm.argtypes = [vp, C.POINTER(BatchDesc), vp, C.POINTER(FmParams), C.POINTER(FmOut)]
    lib.wefax_decode_fm.restype = i
    lib.wefax_decode_fm_slant.argtypes = [vp, C.POINTER(BatchDesc), vp, C.POINTER(FmParams), C.POINTER(FmSlant),
                                          C.POINTER(FmOut), C.POINTER(FmSlantOut)]
    lib.wefax_decode_fm_slant.restype = i
    lib.wefax_segment_envelope.argtypes = [vp, C.POINTER(BatchDesc), vp, ll, ll, ll, ll]
    lib.wefax_segment_envelope.restype = i
    lib.wefax_segment_histogram.argtypes = [vp, i, C.POINTER(C.c_uint32 * 4), vp]
    lib.wefax_segment_histogram.restype = i
    lib.wefax_segment_quantise.argtypes = [vp, d, d, vp, vp]
    lib.wefax_segment_quantise.restype = i
    lib.wefax_segment_select_init.argtypes = [vp, vp, C.POINTER(C.c_uint32 * 4), d, d]
    lib.wefax_segment_select_init.restype = i
    lib.wefax_segment_histogram_dev.argtypes = [vp, i, vp]
    lib.wefax_segment_histogram_dev.restype = i
    lib.wefax_segment_select_dev.argtypes = [vp, i, vp]
    lib.wefax_segment_select_dev.restype = i
    lib.wefax_segment_quantise_dev.argtypes = [vp, vp, vp, vp]
    lib.wefax_segment_quantise_dev.restype = i
    lib.wefax_segment_sync.argtypes = [vp, d, C.POINTER(BatchOut)]
    lib.wefax_segment_sync.restype = i
    lib.wefax_segment_raster.argtypes = [vp, d, ll, i, i, i, vp]
    lib.wefax_segment_raster.restype = i
    _lib = lib
    return lib


def line_constants(lpm: float, sample_rate: int = TARGET_RATE) -> dict:
    lc = LineConstants()
    rc = load().wefax_line_constants_for(float(lpm), int(sample_rate), C.byref(lc))
    if rc != OK:
        raise ValueError(f"invalid lines per minute {lpm!r}")
    return {name: getattr(lc, name) for name, _ in LineConstants._fields_}


def resampled_length(n_frames: int, sample_rate: int) -> int:
    return int(load().wefax_resampled_length(int(n_frames), int(sample_rate)))


def notch_coefficients(freq: float, q: float, fs: float):
    b, a = (C.c_double * 3)(), (C.c_double * 3)()
    rc = load().wefax_notch_coefficients(float(freq), float(q), float(fs), C.byref(b), C.byref(a))
    if rc != OK:
        raise ValueError("w0 should be such that 0 < w0 < 1")
    return list(b), list(a)


def fft_plan_describe(n: int):
    npass, lens, blu = C.c_int(), (C.c_int * 8)(), C.c_longlong()
    rc = load().wefax_fft_plan_describe(int(n), C.byref(npass), C.byref(lens), C.byref(blu))
    if rc != OK:
        raise ValueError(f"no transform plan for n={n}")
    return list(lens)[: npass.value], int(blu.value)
