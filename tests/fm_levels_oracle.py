"""TEST INFRASTRUCTURE — float64 restatement of the FM chart decode's tuning-offset measurement (csrc/fm.cu
fm_levels_kernel, api.cu fm_tail; DESIGN.md §4.7d), next to oracle/fm_oracle.py, whose picture it corrects.

sets: the pulse and body samples of a chart's phasing lines; measure: the lower medians b (body) and w (pulse) of the
unclipped grey, delta = (b + w) / 2 - 0.5, the offset in Hz and the status; corrected_image: the picture of
grey - float32(delta), as the image kernel reads it.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import fm_oracle as F

OK, NOT_FOUND = 0, 1
SPAN_MIN, SPAN_MAX = 0.75, 1.25
DEFAULT_MAX_OFFSET_HZ = 200.0


def set_offsets(Ls: float):
    """(wb, e, pulse offsets, body offsets): wb = max(1, round(0.05 Ls)), e = ceil(wb / 4), pulse o in [e, wb - e),
    body o in [wb + e, floor(Ls) - e)."""
    wb = max(1, int(round(0.05 * Ls)))
    e = (wb + 3) // 4
    return wb, e, np.arange(e, wb - e), np.arange(wb + e, int(math.floor(Ls)) - e)


def set_indices(start: int, Ls: float, fold_lines: int, end: int, offsets: np.ndarray) -> np.ndarray:
    """Sample indices start + floor(l * Ls + o) (l * Ls rounded, then + o rounded, as fm_fold_kernel) of lines
    l < fold_lines, kept where 0 <= i < end, in line order."""
    if offsets.size == 0 or fold_lines <= 0:
        return np.zeros(0, dtype=np.int64)
    l = np.arange(fold_lines, dtype=np.float64)[:, None]
    idx = start + np.floor(l * Ls + offsets[None, :].astype(np.float64)).astype(np.int64)
    idx = idx.ravel()
    return idx[(idx >= 0) & (idx < end)]


def lower_median(v: np.ndarray):
    """Element floor((m - 1) / 2) of the ascending sort (NaN for an empty set)."""
    if v.size == 0:
        return float("nan")
    return np.partition(v, (v.size - 1) // 2)[(v.size - 1) // 2]


def sets(grey: np.ndarray, start: int, Ls: float, fold_lines: int = 20, image_end: int | None = None):
    """(pulse values, body values) of the grey at the chart's line start and line length; end = min(n, image_end)."""
    n = grey.shape[0]
    end = n if image_end is None else min(n, image_end)
    _, _, po, bo = set_offsets(Ls)
    return grey[set_indices(start, Ls, fold_lines, end, po)], grey[set_indices(start, Ls, fold_lines, end, bo)]


def measure(grey: np.ndarray, start: int, Ls: float, fold_lines: int = 20, image_end: int | None = None,
            black_hz: float = 1500.0, white_hz: float = 2300.0, max_offset_hz: float = DEFAULT_MAX_OFFSET_HZ) -> dict:
    """The levels of one chart.  grey: float32 (the decoder's) or float64 (the restatement's) grey stream."""
    pulse, body = sets(grey, start, Ls, fold_lines, image_end)
    b, w = lower_median(body), lower_median(pulse)
    span = white_hz - black_hz
    delta = (float(b) + float(w)) / 2.0 - 0.5
    offset = delta * span
    ok = body.size > 0 and pulse.size > 0 and SPAN_MIN <= float(w) - float(b) <= SPAN_MAX and abs(offset) <= max_offset_hz
    return dict(b=b, w=w, delta=delta, offset_hz=offset, black_hz=black_hz + float(b) * span,
                white_hz=black_hz + float(w) * span, black_samples=int(body.size), white_samples=int(pulse.size),
                status=OK if ok else NOT_FOUND)


def corrected_image(grey: np.ndarray, start: int, Ls: float, ioc: int, image_end: int | None, delta: float):
    """The picture of grey - float32(delta) (float32 subtraction, as the image kernel), else oracle/fm_oracle.image."""
    g = np.asarray(grey, dtype=np.float32) - np.float32(delta)
    return F.image(g, start, None, ioc, image_end, line_length=Ls)
