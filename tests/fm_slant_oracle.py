"""TEST INFRASTRUCTURE — float64 restatement of the FM decode's slant search (csrc/fm.cu slant kernels + the line fit
in csrc/api.cu; DESIGN.md §4.7a), on top of the FM restatement in oracle/fm_oracle.py.

Same integer geometry, candidate order and tie rules as the CUDA path; sums in float64 where the device sums in
float32, so the two agree to a fraction of a ppm rather than bit for bit (tests/test_gpu_fm_slant.py)."""
from __future__ import annotations

import numpy as np

from oracle import fm_oracle as F

TARGET_RATE = F.TARGET_RATE


def image(grey: np.ndarray, start: float, line_length: float, ioc: int, image_end: int | None = None) -> np.ndarray:
    """oracle/fm_oracle.py image() with lines of exactly `line_length` samples (not a round trip through lpm, which
    can move the line length by an ulp, and an ulp can decide the row count)."""
    return F.image(grey, start, None, ioc, image_end, line_length=line_length)


SLANT_OK, SLANT_NOT_FOUND = 0, 1
SLANT_COARSE_LINES = 1024


def _lround(x: float) -> int:
    """llround for the non-negative values used here (half away from zero, not Python's half to even)."""
    return int(np.floor(x + 0.5))


def slant_geometry(lpm: float, search_from: int, image_end: int, max_ppm: float) -> dict:
    """Integer geometry of the slant search (csrc/api.cu: slant_geometry)."""
    Ls = 60.0 / lpm * TARGET_RATE
    wb = max(1, _lround(0.05 * Ls))
    D = max(1, _lround(wb / 16.0))
    Bn = int(np.ceil(Ls / D))
    span = image_end - search_from
    L = max(0, int(np.floor(span / (Ls / (1.0 - max_ppm * 1e-6))))) if span > 0 else 0
    Lc = min(L, SLANT_COARSE_LINES)
    K = int(np.ceil(max_ppm * 1e-6 * Ls * Lc / D))
    return dict(Ls=Ls, wb=wb, D=D, Bn=Bn, L=L, Lc=Lc, J=(K + 1) // 2, wbb=max(1, _lround(wb / D)), R=5 * D)


def _coarse(gc: np.ndarray, frm: int, geo: dict):
    """Stage 1: profile Q[l][b] of D-sample bins, sheared folds S_k, circular boxcar, best (k, b)."""
    Ls, D, Bn, Lc, J, wbb = geo["Ls"], geo["D"], geo["Bn"], geo["Lc"], geo["J"], geo["wbb"]
    n = gc.shape[0]
    cs = np.concatenate([[0.0], np.cumsum(gc)])
    l = np.arange(Lc)
    lo = frm + np.floor(l * Ls).astype(np.int64)[:, None] + np.arange(Bn)[None, :] * D
    Q = (cs[np.clip(lo + D, 0, n)] - cs[np.clip(lo, 0, n)]) / D          # samples at or past n count as 0
    best = (-1.0, 0, 0)
    for c in range(2 * J + 1):                     # candidate order 0, -2, +2, -4, +4, ...: smallest |k| wins ties
        k = 0 if c == 0 else (c + 1) // 2 * 2 * (-1 if c % 2 else 1)
        shift = (2 * l * k + Lc) // (2 * Lc)       # round(l * k / Lc), halves up
        cols = (np.arange(Bn)[None, :] + shift[:, None]) % Bn
        S = np.take_along_axis(Q, cols, axis=1).sum(axis=0)
        pre = np.concatenate([[0.0], np.cumsum(np.concatenate([S, S[:wbb]]))])
        score = pre[wbb:wbb + Bn] - pre[:Bn]
        b = int(np.argmax(score))                  # smallest b on ties
        if score[b] > best[0]:
            best = (float(score[b]), k, b)
    return best[1], best[2]


def _track(gc: np.ndarray, cs: np.ndarray, a: float, s: float, lines: int, geo: dict, min_contrast: float):
    """Stage 2: per line, arg max of the width-wb boxcar within +-R of a + l*s; contrast against the guard bands."""
    wb, R = geo["wb"], geo["R"]
    n = gc.shape[0]
    ls, ys = [], []
    for li in range(lines):
        c = int(np.floor(a + li * s + 0.5))
        if c - R - wb < 0 or c + R + 2 * wb > n:
            continue
        x = np.arange(c - R, c + R + 1)
        box = cs[x + wb] - cs[x]
        j = int(np.argmax(box))
        xs = int(x[j])
        guard = (cs[xs] - cs[xs - wb]) + (cs[xs + 2 * wb] - cs[xs + wb])
        if box[j] / wb - guard / (2 * wb) >= min_contrast:
            ls.append(li)
            ys.append(xs)
    return np.asarray(ls, dtype=np.float64), np.asarray(ys, dtype=np.float64)


def _fit(l: np.ndarray, y: np.ndarray):
    ml, my = l.mean(), y.mean()
    s = np.sum((l - ml) * (y - my)) / np.sum((l - ml) ** 2)
    return my - s * ml, s


def _robust_fit(l: np.ndarray, y: np.ndarray, min_lines: int):
    """Least squares, then twice: drop |residual| > max(1, 3 * 1.4826 * MAD) and refit.  None: too few lines."""
    if l.shape[0] < max(2, min_lines):
        return None
    a, s = _fit(l, y)
    for _ in range(2):
        r = np.abs(y - (a + s * l))
        keep = r <= max(1.0, 3.0 * 1.4826 * float(np.median(r)))
        l, y = l[keep], y[keep]
        if l.shape[0] < max(2, min_lines):
            return None
        a, s = _fit(l, y)
    r = y - (a + s * l)
    return a, s, int(l.shape[0]), float(np.sqrt(np.mean(r * r)))


def slant(grey: np.ndarray, search_from: int, lpm: float, image_end: int, max_ppm: float = 300.0,
          min_contrast: float = 0.3, min_lines: int = 8) -> dict:
    """Sample-clock error from the white line pulses (the AUTO slant mode of csrc/fm.cu + api.cu), float64.

    Stage 1 shears the folded profile of the first Lc lines over every total drift within +-max_ppm (steps of
    2 bins of D samples) and keeps the best (drift, offset); stage 2 finds each line's pulse within +-5 D samples
    of that track; stage 3 fits a line through the pulse positions with two rounds of outlier rejection.  Stages
    2-3 run on the Lc lines, then once more on all L lines from the first fit.
    ppm = (Ls / line_length - 1) * 1e6: positive when the recording's lines are shorter than nominal."""
    geo = slant_geometry(lpm, search_from, image_end, max_ppm)
    Ls, L, Lc = geo["Ls"], geo["L"], geo["Lc"]
    out = dict(status=SLANT_NOT_FOUND, line_length=Ls, ppm=0.0, first_line=float(search_from),
               line_start=int(search_from), lines_total=L, lines_used=0, residual_rms=0.0)
    if L < max(2, min_lines):
        return out
    gc = np.clip(np.asarray(grey, dtype=np.float64), 0.0, 1.0)
    cs = np.concatenate([[0.0], np.cumsum(gc)])
    k, b = _coarse(gc, search_from, geo)
    a, s = search_from + b * geo["D"], Ls + k * geo["D"] / Lc
    fit = None
    for lines in (Lc, L):
        fit = _robust_fit(*_track(gc, cs, a, s, lines, geo, min_contrast), min_lines)
        if fit is None:
            return out
        a, s = fit[0], fit[1]
    ppm = (Ls / s - 1.0) * 1e6
    if not abs(ppm) <= max_ppm:
        return out
    first = a - np.floor((a - search_from) / s) * s
    out.update(status=SLANT_OK, line_length=s, ppm=ppm, first_line=first, line_start=_lround(first),
               lines_used=fit[2], residual_rms=fit[3])
    return out
