"""TEST INFRASTRUCTURE — float64 restatement of the FM chart finder (csrc/fm.cu fm_tone_kernel / fm_lpm_kernel, api.cu
find_charts; DESIGN.md §4.7b), next to oracle/fm_oracle.py, which restates the single-picture decode it feeds.

tone_scores: (r_300, r_450, r_675, V) of every whole window of 2205 samples; tone_classes: the host's class rule;
find_charts: the segmentation into charts; lpm_scores / best_lpm: each LPM candidate's phasing score and the choice.
"""
from __future__ import annotations

import numpy as np

TARGET_RATE = 11025
TONE_WINDOW = 2205                    # 0.2 s: 300, 450 and 675 Hz have 60, 90 and 135 whole periods in a window
TONE_FREQS = (300, 450, 675)
TONE_MIN_RATIO, TONE_MIN_VAR, TONE_MIN_RUN = 0.5, 0.01, 10
LPM_MIN_SCORE = 0.3
STANDARD_LPMS = (60.0, 90.0, 100.0, 120.0, 180.0, 240.0)
NONE, START_576, STOP, START_288 = 0, 1, 2, 3


def tone_scores(grey: np.ndarray) -> np.ndarray:
    """(n // T, 4): (r_300, r_450, r_675, V) of every whole window of T samples.  u = clip(grey, 0, 1), V = mean((u -
    mu)^2), r_f = 2 |sum_j (u_j - mu) exp(-2 pi i f j / 11025)|^2 / (T^2 V), 0 when V = 0."""
    T = TONE_WINDOW
    nw = grey.shape[0] // T
    u = np.clip(np.asarray(grey[: nw * T], dtype=np.float64), 0.0, 1.0).reshape(nw, T)
    d = u - u.mean(axis=1, keepdims=True)
    V = (d * d).mean(axis=1)
    j = np.arange(T)
    out = np.zeros((nw, 4))
    out[:, 3] = V
    for k, f in enumerate(TONE_FREQS):
        w = np.exp(-2j * np.pi * ((f * j) % TARGET_RATE) / TARGET_RATE)
        C = d @ w
        with np.errstate(invalid="ignore", divide="ignore"):
            out[:, k] = np.where(V > 0, 2.0 * np.abs(C) ** 2 / (T * T * np.where(V > 0, V, 1.0)), 0.0)
    return out


def tone_classes(scores: np.ndarray) -> np.ndarray:
    """START_576 / STOP / START_288 where r_300 / r_450 / r_675 is the largest (the first on ties), >= TONE_MIN_RATIO,
    and V >= TONE_MIN_VAR; NONE elsewhere."""
    k = np.argmax(scores[:, :3], axis=1)
    r = scores[np.arange(scores.shape[0]), k]
    ok = (r >= TONE_MIN_RATIO) & (scores[:, 3] >= TONE_MIN_VAR)
    return np.where(ok, np.array([START_576, STOP, START_288])[k], NONE)


def find_charts(classes, n: int) -> list:
    """Charts from window classes: runs of >= TONE_MIN_RUN windows of one class at their full length; a start run opens
    a chart, which the first later STOP run (stop_found), the next start run, or the end of the recording closes.  A
    STOP run with no chart open is ignored.  Each chart: dict(tone_begin, search_from, image_end, stop_found, ioc)."""
    T = TONE_WINDOW
    charts, k, nw = [], 0, len(classes)
    while k < nw:
        e = k + 1
        while e < nw and classes[e] == classes[k]:
            e += 1
        c = int(classes[k])
        if e - k >= TONE_MIN_RUN and c != NONE:
            if charts and charts[-1]["image_end"] is None:
                charts[-1].update(image_end=k * T, stop_found=c == STOP)
            if c != STOP:
                charts.append(dict(tone_begin=k * T, search_from=e * T, image_end=None, stop_found=False,
                                   ioc=576 if c == START_576 else 288))
        k = e
    if charts and charts[-1]["image_end"] is None:
        charts[-1]["image_end"] = n
    return charts


def lpm_scores(grey: np.ndarray, search_from: int, candidates=STANDARD_LPMS, fold_lines: int = 20) -> np.ndarray:
    """Phasing score of each LPM candidate: the phasing fold (phasing_scores' float32 sums) of fold_lines lines of
    60 / lpm * 11025 samples from search_from, best circular boxcar of wb = max(1, round(0.05 Ls)) over (wb * lines),
    minus the fold's mean over lines."""
    out = []
    frm = min(search_from, grey.shape[0] - 1)
    for lpm in candidates:
        Ls = 60.0 / lpm * TARGET_RATE
        Lc = int(np.ceil(Ls))
        wb = max(1, int(round(0.05 * Ls)))
        g = np.clip(grey, 0.0, 1.0).astype(np.float32)
        P = np.zeros(Lc, dtype=np.float32)
        o = np.arange(Lc)
        for l in range(fold_lines):
            idx = frm + np.floor(l * Ls + o).astype(np.int64)
            ok = idx < g.shape[0]
            P[ok] += g[idx[ok]]
        P64 = P.astype(np.float64)
        pre = np.concatenate([[0.0], np.cumsum(np.concatenate([P64, P64]))])
        box = pre[o + wb] - pre[o]
        out.append(box.max() / (wb * fold_lines) - P64.mean() / fold_lines)
    return np.array(out)


def best_lpm(scores, candidates=STANDARD_LPMS):
    """(lpm, score) of the highest score, the first listed on ties; lpm None below LPM_MIN_SCORE."""
    k = int(np.argmax(scores))
    return (candidates[k] if scores[k] >= LPM_MIN_SCORE else None), float(scores[k])
