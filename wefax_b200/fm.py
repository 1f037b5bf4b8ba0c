"""EXTENSION (SURVEY.md §8(f) N4): FM-discriminator decode with exact line length and IOC pixel columns.

The reference never implemented what its README describes (README.md:85-101: black 1500 Hz, white
2300 Hz, start tone 300 / 675 Hz, phasing lines, stop tone 450 Hz); it slope-detects and rasters
``int(samples per line)`` columns.  This module is the decoder the README describes, on the GPU
(``csrc/fm.cu`` through ``wefax_decode_fm``): band-pass, analytic signal, instantaneous frequency,
phasing-pulse line start, ``round(pi * IOC)`` pixels per line.  It is off the reference-exact path
and has no reference parity; see ``oracle/fm_oracle.py`` and ``tests/test_gpu_fm.py``.

:func:`decode_fm` decodes one picture whose LPM and IOC the caller knows.  Its default span comes from the AM path's
tone test (:func:`image_span`), which finds only the first IOC 576 chart of a recording.  :func:`decode_fm_charts`
finds every chart of a recording in the FM grey stream itself (start tones at 300 / 675 Hz, stop tone at 450 Hz),
measures each chart's LPM from its phasing lines and decodes them all from one front end (``wefax_decode_fm_charts``);
:func:`decode_fm_charts_batch` does the same for a batch of equal-length recordings in one call.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
from dataclasses import dataclass

import numpy as np

from . import _native as N


@dataclass
class FmSlant:
    """What the slant correction used (``wefax_fm_slant_out``)."""
    line_length: float         # samples (at 11025 Hz) per image line
    ppm: float                 # sample-clock error: (60 / lpm * 11025 / line_length - 1) * 1e6
    first_line: float          # fractional sample of the first image line
    lines_total: int           # auto: lines tracked
    lines_used: int            # auto: lines whose pulse entered the fit
    residual_rms: float        # auto: rms distance (samples) of those pulses from the fitted line
    status: int                # N.FM_SLANT_OK, or N.FM_SLANT_NOT_FOUND (auto found too few pulses: uncorrected image)

    @property
    def found(self) -> bool:
        return self.status == N.FM_SLANT_OK


@dataclass
class FmLevels:
    """A chart's tuning offset, measured from its phasing lines (``wefax_fm_levels_out``)."""
    black_hz: float            # measured black level (NaN when the body set is empty)
    white_hz: float            # measured white level (NaN when the pulse set is empty)
    offset_hz: float           # (black_hz + white_hz) / 2 minus the centre of the grey scale (1900 Hz by default)
    black_samples: int         # samples the black level is the lower median of
    white_samples: int         # samples the white level is the lower median of
    status: int                # N.FM_LEVELS_OK (picture corrected by offset_hz), N.FM_LEVELS_NOT_FOUND (uncorrected)

    @property
    def found(self) -> bool:
        return self.status == N.FM_LEVELS_OK


@dataclass
class FmResult:
    image: np.ndarray          # (rows, width) uint8, 0 = black (1500 Hz), 255 = white (2300 Hz)
    line_start: int            # sample (at 11025 Hz) of the first image row
    width: int                 # round(pi * ioc)
    search_from: int
    image_end: int
    grey: np.ndarray | None = None     # per-sample grey before clipping (float32), when asked for
    slant: FmSlant | None = None       # with slant="auto" or a ppm value


@dataclass
class FmChart:
    """One chart of a recording (``wefax_fm_chart``); positions are samples at 11025 Hz."""
    tone_begin: int            # first sample of the start tone
    search_from: int           # sample after the start tone: the phasing search starts here
    image_end: int             # first sample of the stop tone, of the next start tone, or the end of the recording
    stop_found: bool
    ioc: int                   # 576 or 288 from the start tone (or the forced value)
    lpm: float                 # from the phasing lines (or the forced value)
    lpm_score: float           # the phasing score of that LPM (about 1 on a clean signal; 0 when the LPM is forced)
    status: int                # N.FM_CHART_OK, or N.FM_CHART_NO_LPM (no LPM scored N.FM_LPM_MIN_SCORE: no picture)
    width: int                 # round(pi * ioc)
    line_start: int            # sample of the first picture line (-1: no picture decoded)
    image: np.ndarray | None   # (rows, width) uint8; None when pictures were not asked for or status is not OK
    slant: FmSlant | None = None
    levels: FmLevels | None = None      # with levels="auto", when the chart has a picture


@dataclass
class FmCharts:
    charts: list               # FmChart of the first max_charts charts, in recording order
    n_found: int               # charts found (may exceed len(charts))
    grey: np.ndarray | None = None          # per-sample grey (float32), when asked for
    tone_scores: np.ndarray | None = None   # (windows, 4) float32: r_300, r_450, r_675, V per 0.2 s window


def image_span(start_flags, stop_flags, sample_rate_out: int = N.TARGET_RATE, packet_seconds: float = 1.0):
    """Where the picture lies according to the tone scan: from the end of the first run of start-tone
    packets (>= 3 in a row) to the beginning of the first later run of stop-tone packets (>= 3)."""
    n = len(start_flags)
    k, run = 0, 0
    begin = 0
    while k < n:
        run = run + 1 if start_flags[k] else 0
        if run >= 3:
            while k + 1 < n and start_flags[k + 1]:
                k += 1
            begin = k + 1
            break
        k += 1
    end, run = n, 0
    for j in range(begin, n):
        run = run + 1 if stop_flags[j] else 0
        if run >= 3:
            end = j - 2
            break
    per = int(round(sample_rate_out * packet_seconds))
    return begin * per, end * per


def slant_params(slant, max_slant_ppm: float = 300.0):
    """``N.FmSlant`` for ``slant`` = None (no correction: None is returned), ``"auto"`` (measure the clock error
    within +-``max_slant_ppm``) or a clock error in ppm; ValueError for anything else."""
    if slant is None:
        return None
    if isinstance(slant, str):
        if slant != "auto":
            raise ValueError(f"slant must be None, 'auto' or a ppm value, not {slant!r}")
        if isinstance(max_slant_ppm, bool) or not isinstance(max_slant_ppm, numbers.Real) or \
                not 0.0 < float(max_slant_ppm) <= N.FM_SLANT_MAX_PPM:
            raise ValueError(f"max_slant_ppm must be in (0, {N.FM_SLANT_MAX_PPM:g}], not {max_slant_ppm!r}")
        return N.FmSlant(N.FM_SLANT_AUTO, 0.0, float(max_slant_ppm), 0.3, 8)
    if isinstance(slant, bool) or not isinstance(slant, numbers.Real) or not abs(float(slant)) <= N.FM_SLANT_MAX_PPM:
        raise ValueError(f"slant must be None, 'auto' or a ppm value within +-{N.FM_SLANT_MAX_PPM:g}, not {slant!r}")
    return N.FmSlant(N.FM_SLANT_FIXED, float(slant), 0.0, 0.0, 0)


def decode_fm(decoder, pcm, sample_rate: int, lpm: float = 120, ioc: int = 576, search_from: int | None = None,
              image_end: int | None = None, fold_lines: int = 20, black_hz: float = 1500.0, white_hz: float = 2300.0,
              band=(1200.0, 2600.0), fir_taps: int = 63, want_grey: bool = False, slant=None,
              max_slant_ppm: float = 300.0) -> FmResult:
    """Decode one recording (int16 numpy, mono ``(n,)`` or stereo ``(n, 2)``).

    ``search_from`` / ``image_end`` (samples at 11025 Hz) default to what the start / stop tone scan
    finds (:func:`image_span`).  That scan is the AM path's packet test: it finds only the first IOC 576 chart of a
    recording (it misses the 675 Hz start tone); :func:`decode_fm_charts` finds every chart.  ``slant`` corrects the recording's sample-clock error: ``"auto"`` measures
    it from the white line pulses (within +-``max_slant_ppm``), a number is the error in ppm (what
    ``result.slant.ppm`` reported for an earlier decode); None decodes lines of exactly 60 / lpm s."""
    sp = slant_params(slant, max_slant_ppm)
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    n_in, ch = int(pcm.shape[0]), (1 if pcm.ndim == 1 else int(pcm.shape[1]))
    n_out = n_in if sample_rate == N.TARGET_RATE else N.resampled_length(n_in, sample_rate)
    if search_from is None or image_end is None:
        from .tones import scan_tones
        start, stop, _, _ = scan_tones(decoder, pcm, sample_rate)
        s0, s1 = image_span(start, stop)
        search_from = s0 if search_from is None else search_from
        image_end = min(s1, n_out) if image_end is None else image_end
    ls = 60.0 / lpm * N.TARGET_RATE
    if sp is not None:       # the image is sized for the shortest line the mode allows (as the library checks)
        ls = ls / (1.0 + (sp.max_ppm if sp.mode == N.FM_SLANT_AUTO else sp.ppm) * 1e-6)
    width = int(round(math.pi * ioc))
    rows_max = max(0, int(math.floor((image_end - search_from) / ls)))
    img = np.zeros(max(1, rows_max * width), dtype=np.uint8)
    grey = np.zeros(n_out, dtype=np.float32) if want_grey else None
    rows, w, start_s = C.c_int32(0), C.c_int32(0), C.c_int64(0)
    desc = N.BatchDesc(1, n_in, ch, int(sample_rate), 0.0, 0.0, 0)
    prm = N.FmParams(float(lpm), int(ioc), float(black_hz), float(white_hz), float(band[0]), float(band[1]),
                     int(fir_taps), int(search_from), int(fold_lines), int(image_end))
    out = N.FmOut(grey.ctypes.data if want_grey else None, img.ctypes.data, img.size,
                  C.addressof(rows), C.addressof(w), C.addressof(start_s))
    so = None
    if sp is None:
        decoder._check(decoder._lib.wefax_decode_fm(decoder._h, C.byref(desc), C.c_void_p(pcm.ctypes.data),
                                                    C.byref(prm), C.byref(out)))
    else:
        sout = N.FmSlantOut()
        decoder._check(decoder._lib.wefax_decode_fm_slant(decoder._h, C.byref(desc), C.c_void_p(pcm.ctypes.data),
                                                          C.byref(prm), C.byref(sp), C.byref(out), C.byref(sout)))
        so = FmSlant(**{name: getattr(sout, name) for name, _ in N.FmSlantOut._fields_})
    return FmResult(img[: rows.value * width].reshape(rows.value, width), int(start_s.value), width,
                    int(search_from), int(image_end), grey, so)


def chart_params(lpm=None, ioc=None, lpm_candidates=None, slant=None, max_slant_ppm: float = 300.0,
                 fold_lines: int = 20, black_hz: float = 1500.0, white_hz: float = 2300.0, band=(1200.0, 2600.0),
                 fir_taps: int = 63):
    """``N.FmChartParams`` for :func:`decode_fm_charts`; ValueError for arguments the library would refuse."""
    def real(v):
        return not isinstance(v, bool) and isinstance(v, numbers.Real) and math.isfinite(float(v))
    if lpm is not None and not (real(lpm) and float(lpm) > 0):
        raise ValueError(f"lpm must be None (detect) or a positive number, not {lpm!r}")
    if ioc is not None and not (isinstance(ioc, numbers.Integral) and not isinstance(ioc, bool) and ioc > 0):
        raise ValueError(f"ioc must be None (detect) or a positive integer, not {ioc!r}")
    cands = N.FM_STANDARD_LPMS if lpm_candidates is None else tuple(lpm_candidates)
    if not 1 <= len(cands) <= N.FM_MAX_LPM_CANDIDATES or not all(real(c) and 60 <= float(c) <= 240 for c in cands):
        raise ValueError(f"lpm_candidates: 1 to {N.FM_MAX_LPM_CANDIDATES} values within [60, 240], not {lpm_candidates!r}")
    if isinstance(fold_lines, bool) or not isinstance(fold_lines, numbers.Integral) or fold_lines < 1:
        raise ValueError(f"fold_lines must be a positive integer, not {fold_lines!r}")
    sp = slant_params(slant, max_slant_ppm) or N.FmSlant(N.FM_SLANT_OFF, 0.0, 0.0, 0.0, 0)
    prm = N.FmParams(float(lpm or 0.0), int(ioc or 0), float(black_hz), float(white_hz), float(band[0]),
                     float(band[1]), int(fir_taps), 0, int(fold_lines), 0)
    arr = (C.c_double * N.FM_MAX_LPM_CANDIDATES)(*[float(c) for c in cands])
    return N.FmChartParams(prm, sp, len(cands), arr)


def levels_params(levels=None, max_offset_hz: float = 200.0):
    """``N.FmLevels`` for ``levels`` = None (no correction) or ``"auto"`` (measure each chart's tuning offset from its
    phasing lines and correct it when it is within +-``max_offset_hz``); ValueError for anything else."""
    if levels is not None and levels != "auto":
        raise ValueError(f"levels must be None or 'auto', not {levels!r}")
    if isinstance(max_offset_hz, bool) or not isinstance(max_offset_hz, numbers.Real) or \
            not 0.0 < float(max_offset_hz) <= N.FM_LEVELS_MAX_OFFSET_HZ:
        raise ValueError(f"max_offset_hz must be in (0, {N.FM_LEVELS_MAX_OFFSET_HZ:g}], not {max_offset_hz!r}")
    return N.FmLevels(N.FM_LEVELS_OFF if levels is None else N.FM_LEVELS_AUTO, float(max_offset_hz))


def _max_charts(max_charts):
    if isinstance(max_charts, bool) or not isinstance(max_charts, numbers.Integral) or max_charts < 0:
        raise ValueError(f"max_charts must be a non-negative integer, not {max_charts!r}")
    return int(max_charts)


def _image_bound(prm, lpm, ioc, n_out: int) -> int:
    """Bytes that hold the pictures of any recording of n_out samples (at 11025 Hz): the charts' spans are disjoint,
    so ceil(n_out / shortest line) rows of the widest picture hold them all."""
    ls_min = 60.0 / (float(lpm) if lpm else max(prm.lpm_candidates[: prm.n_lpm_candidates])) * N.TARGET_RATE
    sp = prm.slant
    if sp.mode != N.FM_SLANT_OFF:
        ls_min = ls_min / (1.0 + (sp.max_ppm if sp.mode == N.FM_SLANT_AUTO else max(sp.ppm, 0.0)) * 1e-6)
    w_max = int(round(math.pi * (ioc if ioc else 576)))
    return int(math.ceil(n_out / ls_min)) * w_max


def _charts(out, lev, n_found: int, max_charts: int, img, prm) -> list:
    """FmChart of the native chart entries ``out`` and their levels ``lev`` (pictures cut from ``img``, None when
    pictures were not asked for)."""
    charts = []
    for c, lo in zip(out[: min(n_found, max_charts)], lev):
        decoded = img is not None and c.status == N.FM_CHART_OK
        picture = img[c.image_offset: c.image_offset + c.rows * c.width].reshape(c.rows, c.width) if decoded else None
        so = FmSlant(**{name: getattr(c.slant, name) for name, _ in N.FmSlantOut._fields_}) \
            if (decoded and prm.slant.mode != N.FM_SLANT_OFF) else None
        lv = FmLevels(**{name: getattr(lo, name) for name, _ in N.FmLevelsOut._fields_}) \
            if lo.status != N.FM_LEVELS_NOT_MEASURED else None
        charts.append(FmChart(int(c.tone_begin), int(c.search_from), int(c.image_end), bool(c.stop_found), int(c.ioc),
                              float(c.lpm), float(c.lpm_score), int(c.status), int(c.width), int(c.line_start),
                              picture, so, lv))
    return charts


def decode_fm_charts(decoder, pcm, sample_rate: int, lpm=None, ioc=None, lpm_candidates=None, slant=None,
                     max_slant_ppm: float = 300.0, max_charts: int = 64, fold_lines: int = 20,
                     black_hz: float = 1500.0, white_hz: float = 2300.0, band=(1200.0, 2600.0), fir_taps: int = 63,
                     want_images: bool = True, want_grey: bool = False, want_tone_scores: bool = False,
                     image_capacity: int | None = None, levels=None, max_offset_hz: float = 200.0) -> FmCharts:
    """Find and decode every chart of a recording (int16 numpy, mono ``(n,)`` or stereo ``(n, 2)``).

    Each chart starts at a start tone (300 Hz: IOC 576, 675 Hz: IOC 288) and ends at the stop tone, the next start
    tone or the end of the recording; its LPM is the candidate (default 60, 90, 100, 120, 180, 240) whose phasing
    fold shows the sharpest line pulse.  ``lpm`` / ``ioc`` force a value for every chart.  ``slant`` as for
    :func:`decode_fm`, for every chart.  Each chart's picture equals ``decode_fm`` with that chart's lpm, ioc,
    search_from and image_end.  ``want_images=False`` returns the chart list only; ``image_capacity`` overrides the
    size of the picture buffer (bytes; default: enough for any recording of this length).  ``levels="auto"`` measures
    each decoded chart's tuning offset from its phasing lines (``chart.levels``) and, when it is found within
    +-``max_offset_hz``, shifts the chart's grey levels by it (the grey stream and the tone scores stay uncorrected)."""
    prm = chart_params(lpm, ioc, lpm_candidates, slant, max_slant_ppm, fold_lines, black_hz, white_hz, band, fir_taps)
    lvp = levels_params(levels, max_offset_hz)
    max_charts = _max_charts(max_charts)
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    n_in, ch = int(pcm.shape[0]), (1 if pcm.ndim == 1 else int(pcm.shape[1]))
    n_out = n_in if sample_rate == N.TARGET_RATE else N.resampled_length(n_in, sample_rate)
    if image_capacity is None:
        image_capacity = _image_bound(prm, lpm, ioc, n_out) if want_images else 0
    img = np.zeros(max(1, image_capacity), dtype=np.uint8) if want_images else None
    grey = np.zeros(n_out, dtype=np.float32) if want_grey else None
    tones = np.zeros((n_out // N.FM_TONE_WINDOW, 4), dtype=np.float32) if want_tone_scores else None
    out = (N.FmChart * max(1, max_charts))()
    lev = (N.FmLevelsOut * max(1, max_charts))()
    n_found = C.c_int(0)
    desc = N.BatchDesc(1, n_in, ch, int(sample_rate), 0.0, 0.0, 0)
    decoder._check(decoder._lib.wefax_decode_fm_charts_levels(
        decoder._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm), C.byref(lvp), out, lev,
        int(max_charts), C.byref(n_found), img.ctypes.data if want_images else None, int(image_capacity),
        tones.ctypes.data if want_tone_scores else None, grey.ctypes.data if want_grey else None))
    return FmCharts(_charts(out, lev, n_found.value, max_charts, img, prm), int(n_found.value), grey, tones)


def decode_fm_charts_batch(decoder, pcm, sample_rate: int, lpm=None, ioc=None, lpm_candidates=None, slant=None,
                           max_slant_ppm: float = 300.0, max_charts: int = 64, fold_lines: int = 20,
                           black_hz: float = 1500.0, white_hz: float = 2300.0, band=(1200.0, 2600.0),
                           fir_taps: int = 63, want_images: bool = True, want_grey: bool = False,
                           want_tone_scores: bool = False, image_capacity: int | None = None, levels=None,
                           max_offset_hz: float = 200.0) -> list:
    """:func:`decode_fm_charts` of R recordings of equal length in one call (``wefax_decode_fm_charts_batch``): one
    FmCharts per recording, each what :func:`decode_fm_charts` returns for that recording alone.

    ``pcm``: int16 ``(R, n)`` mono or ``(R, n, 2)`` stereo, as numpy (host) or as a CUDA torch tensor (read in place on
    the device).  The outputs are numpy arrays on the host.  ``image_capacity`` is the byte size of the picture buffer
    of the whole batch (default: R times the bound of :func:`decode_fm_charts`).  ``levels`` / ``max_offset_hz`` as
    for :func:`decode_fm_charts`."""
    prm = chart_params(lpm, ioc, lpm_candidates, slant, max_slant_ppm, fold_lines, black_hz, white_hz, band, fir_taps)
    lvp = levels_params(levels, max_offset_hz)
    max_charts = _max_charts(max_charts)
    if isinstance(sample_rate, bool) or not isinstance(sample_rate, numbers.Integral) or sample_rate < 1:
        raise ValueError(f"sample_rate must be a positive integer, not {sample_rate!r}")
    flags, keep = 0, pcm
    if type(pcm).__module__.startswith("torch"):
        import torch
        if not pcm.is_cuda or pcm.dtype != torch.int16:
            raise ValueError(f"a torch pcm must be an int16 CUDA tensor, not {pcm.dtype} on {pcm.device}")
        keep = pcm.contiguous()
        ptr, shape, flags = keep.data_ptr(), tuple(keep.shape), N.F_PCM_ON_DEVICE
    else:
        keep = np.ascontiguousarray(pcm, dtype=np.int16)
        ptr, shape = keep.ctypes.data, keep.shape
    if not (len(shape) == 2 or (len(shape) == 3 and shape[2] == 2)) or shape[0] < 1 or shape[1] < 1:
        raise ValueError(f"pcm must be (R, n) or (R, n, 2) with R, n >= 1, not {shape}")
    R, n_in, ch = int(shape[0]), int(shape[1]), (1 if len(shape) == 2 else 2)
    n_out = n_in if sample_rate == N.TARGET_RATE else N.resampled_length(n_in, sample_rate)
    if image_capacity is None:
        image_capacity = R * _image_bound(prm, lpm, ioc, n_out) if want_images else 0
    img = np.zeros(max(1, image_capacity), dtype=np.uint8) if want_images else None
    grey = np.zeros((R, n_out), dtype=np.float32) if want_grey else None
    tones = np.zeros((R, n_out // N.FM_TONE_WINDOW, 4), dtype=np.float32) if want_tone_scores else None
    out = (N.FmChart * max(1, R * max_charts))()
    lev = (N.FmLevelsOut * max(1, R * max_charts))()
    n_found = (C.c_int * R)()
    desc = N.BatchDesc(R, n_in, ch, int(sample_rate), 0.0, 0.0, flags)
    decoder._check(decoder._lib.wefax_decode_fm_charts_levels(
        decoder._h, C.byref(desc), C.c_void_p(ptr), C.byref(prm), C.byref(lvp), out, lev, max_charts, n_found,
        img.ctypes.data if want_images else None, int(image_capacity),
        tones.ctypes.data if want_tone_scores else None, grey.ctypes.data if want_grey else None))
    res = []
    for r in range(R):
        entries = out[r * max_charts: (r + 1) * max_charts]
        levs = lev[r * max_charts: (r + 1) * max_charts]
        res.append(FmCharts(_charts(entries, levs, n_found[r], max_charts, img, prm), int(n_found[r]),
                            None if grey is None else grey[r], None if tones is None else tones[r]))
    return res


def _pcm16(data: np.ndarray) -> np.ndarray:
    """int16 samples of what wavio.read returns (uint8, int16, int32 or float PCM)."""
    if data.dtype == np.int16:
        return data
    if data.dtype == np.uint8:
        return ((data.astype(np.int16) - 128) << 8).astype(np.int16)
    if data.dtype == np.int32:
        return (data >> 16).astype(np.int16)
    return np.clip(np.round(data.astype(np.float64) * 32767.0), -32768, 32767).astype(np.int16)


def main(argv=None) -> int:
    import argparse

    ap = argparse.ArgumentParser(prog="python -m wefax_b200.fm",
                                 description="FM-discriminator WEFAX decode of a WAV recording into a greyscale PNG.")
    ap.add_argument("wav", help="input recording (WAV)")
    ap.add_argument("png", help="output picture (8-bit greyscale PNG); with --all, OUT-01.png, OUT-02.png, ...")
    ap.add_argument("--all", action="store_true",
                    help="find every chart of the recording by its start / stop tones and write one PNG per chart")
    ap.add_argument("--lpm", type=float, default=None,
                    help="lines per minute (default 120; with --all: measured per chart from its phasing lines)")
    ap.add_argument("--ioc", type=int, default=None,
                    help="index of cooperation: 576 or 288 (default 576; with --all: from each chart's start tone)")
    ap.add_argument("--slant", default=None, metavar="auto|PPM",
                    help="correct the sample-clock error: 'auto' measures it, a number gives it in ppm")
    ap.add_argument("--max-slant-ppm", type=float, default=300.0, help="largest error 'auto' searches (default 300)")
    ap.add_argument("--levels", choices=["auto"], default=None,
                    help="with --all: measure each chart's tuning offset from its phasing lines and correct its grey levels")
    ap.add_argument("--max-offset-hz", type=float, default=200.0,
                    help="largest tuning offset --levels auto corrects (default 200)")
    ap.add_argument("--device", type=int, default=0, help="CUDA device (default 0)")
    a = ap.parse_args(argv)
    slant = a.slant
    if slant is not None and slant != "auto":
        try:
            slant = float(slant)
        except ValueError:
            ap.error(f"--slant takes 'auto' or a number, not {a.slant!r}")
    if a.levels is not None and not a.all:
        ap.error("--levels needs --all")
    try:
        slant_params(slant, a.max_slant_ppm)
        levels_params(a.levels, a.max_offset_hz)
    except ValueError as e:
        ap.error(str(e))

    from . import pngio, wavio
    from .decoder import Decoder

    sample_rate, data = wavio.read(a.wav)
    if a.all:
        return _main_all(a, slant, _pcm16(data), sample_rate, ap)
    with Decoder(a.device) as dec:
        res = decode_fm(dec, _pcm16(data), sample_rate, lpm=120.0 if a.lpm is None else a.lpm,
                        ioc=576 if a.ioc is None else a.ioc, slant=slant, max_slant_ppm=a.max_slant_ppm)
    pngio.write_png_gray8(a.png, res.image)
    print(f"{a.png}: {res.image.shape[0]} x {res.image.shape[1]} pixels, first line at sample {res.line_start}")
    if res.slant is not None:
        s = res.slant
        if s.found:
            print(f"slant {s.ppm:+.3f} ppm (line length {s.line_length:.4f} samples; {s.lines_used} of "
                  f"{s.lines_total} line pulses fit, rms {s.residual_rms:.2f} samples); "
                  f"reuse with --slant {s.ppm:.3f}")
        else:
            print("slant: too few line pulses to measure it; the picture is not corrected")
    return 0


def _main_all(a, slant, pcm, sample_rate, ap) -> int:
    import os

    from . import pngio
    from .decoder import Decoder

    try:
        chart_params(a.lpm, a.ioc, slant=slant, max_slant_ppm=a.max_slant_ppm)
    except ValueError as e:
        ap.error(str(e))
    stem, ext = os.path.splitext(a.png)
    with Decoder(a.device) as dec:
        res = decode_fm_charts(dec, pcm, sample_rate, lpm=a.lpm, ioc=a.ioc, slant=slant, max_slant_ppm=a.max_slant_ppm,
                               levels=a.levels, max_offset_hz=a.max_offset_hz)
    if res.n_found > len(res.charts):
        print(f"{res.n_found} charts found, the first {len(res.charts)} decoded")
    for k, c in enumerate(res.charts, 1):
        t0, t1 = c.tone_begin / N.TARGET_RATE, c.image_end / N.TARGET_RATE
        where = f"chart {k}: {t0:8.1f} s - {t1:8.1f} s{'' if c.stop_found else ' (no stop tone)'}, IOC {c.ioc}"
        if c.status != N.FM_CHART_OK:
            print(f"{where}, no LPM found (best {c.lpm:g}, score {c.lpm_score:.2f}): not decoded")
            continue
        path = f"{stem}-{k:02d}{ext or '.png'}"
        pngio.write_png_gray8(path, c.image)
        line = f"{where}, LPM {c.lpm:g} (score {c.lpm_score:.2f}), {path}: {c.image.shape[0]} x {c.image.shape[1]}"
        if c.slant is not None:
            line += f", slant {c.slant.ppm:+.3f} ppm" if c.slant.found else ", slant not measured"
        if a.levels is not None:
            line += f", tuning offset {c.levels.offset_hz:+.1f} Hz" if (c.levels and c.levels.found) \
                else ", tuning offset not measured"
        print(line)
    if not res.n_found:
        print("no chart found (no start tone of 2 s or more)")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
