"""EXTENSION (SURVEY.md §8(f) N4): FM-discriminator decode with exact line length and IOC pixel columns.

The reference never implemented what its README describes (README.md:85-101: black 1500 Hz, white
2300 Hz, start tone 300 / 675 Hz, phasing lines, stop tone 450 Hz); it slope-detects and rasters
``int(samples per line)`` columns.  This module is the decoder the README describes, on the GPU
(``csrc/fm.cu`` through ``wefax_decode_fm``): band-pass, analytic signal, instantaneous frequency,
phasing-pulse line start, ``round(pi * IOC)`` pixels per line.  It is off the reference-exact path
and has no reference parity; see ``oracle/fm_oracle.py`` and ``tests/test_gpu_fm.py``.
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
class FmResult:
    image: np.ndarray          # (rows, width) uint8, 0 = black (1500 Hz), 255 = white (2300 Hz)
    line_start: int            # sample (at 11025 Hz) of the first image row
    width: int                 # round(pi * ioc)
    search_from: int
    image_end: int
    grey: np.ndarray | None = None     # per-sample grey before clipping (float32), when asked for
    slant: FmSlant | None = None       # with slant="auto" or a ppm value


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
    finds (:func:`image_span`).  ``slant`` corrects the recording's sample-clock error: ``"auto"`` measures
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
    ap.add_argument("png", help="output picture (8-bit greyscale PNG)")
    ap.add_argument("--lpm", type=float, default=120.0, help="lines per minute (default 120)")
    ap.add_argument("--ioc", type=int, default=576, help="index of cooperation: 576 or 288 (default 576)")
    ap.add_argument("--slant", default=None, metavar="auto|PPM",
                    help="correct the sample-clock error: 'auto' measures it, a number gives it in ppm")
    ap.add_argument("--max-slant-ppm", type=float, default=300.0, help="largest error 'auto' searches (default 300)")
    ap.add_argument("--device", type=int, default=0, help="CUDA device (default 0)")
    a = ap.parse_args(argv)
    slant = a.slant
    if slant is not None and slant != "auto":
        try:
            slant = float(slant)
        except ValueError:
            ap.error(f"--slant takes 'auto' or a number, not {a.slant!r}")
    try:
        slant_params(slant, a.max_slant_ppm)
    except ValueError as e:
        ap.error(str(e))

    from . import pngio, wavio
    from .decoder import Decoder

    sample_rate, data = wavio.read(a.wav)
    with Decoder(a.device) as dec:
        res = decode_fm(dec, _pcm16(data), sample_rate, lpm=a.lpm, ioc=a.ioc, slant=slant,
                        max_slant_ppm=a.max_slant_ppm)
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


if __name__ == "__main__":
    raise SystemExit(main())
