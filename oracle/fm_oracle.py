"""TEST INFRASTRUCTURE — float64 restatement of the FM-discriminator extension (csrc/fm.cu).

SURVEY.md §8(f) N4.  This mode does NOT exist in the reference (wojlin/WEFAX only describes
it: README.md:85-101), so there is nothing of the reference to restate and PARITY IS UNPINNED
with respect to it.  What this file pins instead: the CUDA extension against a plain numpy
float64 computation of the same definition, and (tests/test_gpu_fm.py) both against the ground
truth of the synthetic generator.

Definition:  x = zero-phase FIR band-pass of the samples (taps applied forwards and backwards
with the edge treatment of the notch kernel: odd extension by 9, steady-state constants),
z = x + i*Hilbert(x) where the transform runs on x zero-padded to npad = 2 * next_smooth_length(
(n + 1) / 2) samples and the first n are kept, grey[i] = (arg(z[i] conj z[i-1]) * sr / 2pi - black) /
(white - black) with grey[0] repeating the first step, line start = search_from + argmax_o
boxcar_{5 % of a line}(sum over lines l of clip(grey[search_from + floor(l * Ls + o)]), l * Ls and the
sum each rounded to float64), rows = floor((image_end - line_start) / Ls) in float64, pixel = box
average of clip(grey) over its exact sample span.
"""
from __future__ import annotations

import numpy as np

TARGET_RATE = 11025


def next_smooth_length(m: int) -> int:
    """The smallest 2^a 3^b 5^c 7^d >= m that the library's transform can plan (csrc/fft_plan.cu:
    next_smooth_length): for every odd part 3^b 5^c 7^d < 2m, the least power-of-two multiple >= m.
    -1 when none can be planned.  The planning test is the library's own (host only, no device)."""
    from wefax_b200 import _native as N

    def can_plan(v: int) -> bool:
        try:
            return N.fft_plan_describe(v)[1] == 0
        except ValueError:
            return False

    cands = set()
    p7 = 1
    while p7 < 2 * m:
        p5 = p7
        while p5 < 2 * m:
            p3 = p5
            while p3 < 2 * m:
                v = p3
                while v < m:
                    v *= 2
                cands.add(v)
                p3 *= 3
            p5 *= 5
        p7 *= 7
    for v in sorted(cands):
        if can_plan(v):
            return v
    return -1


def transform_length(n: int) -> int:
    """npad: the even length the FM decode's Hilbert transform runs on (csrc/api.cu, wefax_decode_fm_slant)."""
    return 2 * next_smooth_length((n + 1) // 2)


def bandpass_taps(lo_hz: float, hi_hz: float, fs: float, taps: int) -> np.ndarray:
    """Hamming windowed-sinc band-pass, unit gain at the band centre, rounded to float32 as the
    device constants are (csrc/fm.cu: make_bandpass_fir)."""
    if taps % 2 == 0:
        taps -= 1
    i = np.arange(taps, dtype=np.float64)
    mid = (taps - 1) / 2.0
    t = i - mid
    fl, fh = lo_hz / fs, hi_hz / fs
    with np.errstate(invalid="ignore", divide="ignore"):
        ideal = (np.sin(2 * np.pi * fh * t) - np.sin(2 * np.pi * fl * t)) / (np.pi * t)
    ideal[t == 0] = 2.0 * (fh - fl)
    h = ideal * (0.54 - 0.46 * np.cos(2 * np.pi * i / (taps - 1)))
    fc = 0.5 * (fl + fh)
    gain = np.hypot(np.sum(h * np.cos(2 * np.pi * fc * t)), np.sum(h * np.sin(2 * np.pi * fc * t)))
    return (h / gain).astype(np.float32).astype(np.float64)


def fir_filtfilt(h: np.ndarray, x: np.ndarray, pad: int = 9) -> np.ndarray:
    """Causal FIR then anti-causal FIR, edges as csrc/stages.cu filtfilt_kernel (= scipy filtfilt with
    padlen 9 for an FIR): odd extension by `pad`, constant ext[0] to the left of the forward section,
    constant last forward value to the right of the backward section."""
    x = np.asarray(x, dtype=np.float64)
    n, K = x.shape[0], h.shape[0]
    ext = np.concatenate([2 * x[0] - x[pad:0:-1], x, 2 * x[-1] - x[-2:-pad - 2:-1]])
    yf = np.convolve(np.concatenate([np.full(K - 1, ext[0]), ext]), h, mode="valid")
    yb = np.convolve(np.concatenate([yf, np.full(K - 1, yf[-1])])[::-1], h, mode="valid")[::-1]
    return yb[pad:pad + n]


def hilbert_imag(x: np.ndarray) -> np.ndarray:
    n = x.shape[0]
    X = np.fft.fft(x)
    hmask = np.zeros(n)
    if n % 2 == 0:
        hmask[0] = hmask[n // 2] = 1
        hmask[1:n // 2] = 2
    else:
        hmask[0] = 1
        hmask[1:(n + 1) // 2] = 2
    return np.fft.ifft(X * hmask).imag


def analytic(pcm: np.ndarray, lo_hz=1200.0, hi_hz=2600.0, taps=63, padded: bool = True) -> np.ndarray:
    """z = x + i Hilbert(x) of the band-passed mono samples at 11025 Hz.  ``padded`` takes the transform
    at the decoder's zero-padded length (transform_length) and keeps the first n; False takes it at n."""
    x = fir_filtfilt(bandpass_taps(lo_hz, hi_hz, TARGET_RATE, taps), pcm)
    n = x.shape[0]
    if padded:
        y = hilbert_imag(np.concatenate([x, np.zeros(transform_length(n) - n)]))[:n]
    else:
        y = hilbert_imag(x)
    return x + 1j * y


def grey_stream(pcm: np.ndarray, lo_hz=1200.0, hi_hz=2600.0, taps=63, black_hz=1500.0, white_hz=2300.0,
                padded: bool = True):
    """Per-sample grey of mono samples at 11025 Hz (``padded`` as for analytic())."""
    return grey_of(analytic(pcm, lo_hz, hi_hz, taps, padded), black_hz, white_hz)


def grey_of(z: np.ndarray, black_hz=1500.0, white_hz=2300.0) -> np.ndarray:
    step = z[1:] * np.conj(z[:-1])
    d = np.angle(step)
    d = np.concatenate([d[:1], d])
    f = d * TARGET_RATE / (2 * np.pi)
    return (f - black_hz) / (white_hz - black_hz)


def _line_length(lpm, line_length):
    return 60.0 / lpm * TARGET_RATE if line_length is None else float(line_length)


def phasing_scores(grey: np.ndarray, search_from: int, lpm: float | None, fold_lines: int,
                   line_length: float | None = None) -> np.ndarray:
    """The phasing search's score for every offset o < ceil(Ls) (float32, as the device keeps it)."""
    Ls = _line_length(lpm, line_length)
    Lc = int(np.ceil(Ls))
    wb = max(1, int(round(0.05 * Ls)))
    g = np.clip(grey, 0.0, 1.0).astype(np.float32)
    P = np.zeros(Lc, dtype=np.float32)
    o = np.arange(Lc)
    for l in range(fold_lines):
        idx = search_from + np.floor(l * Ls + o).astype(np.int64)    # l * Ls rounded, then + o rounded
        ok = idx < g.shape[0]
        P[ok] += g[idx[ok]]
    pre = np.concatenate([[0.0], np.cumsum(np.concatenate([P, P]).astype(np.float64))])
    return (pre[o + wb] - pre[o]).astype(np.float32)


def line_start(grey: np.ndarray, search_from: int, lpm: float | None, fold_lines: int,
               line_length: float | None = None) -> int:
    """Phasing-pulse line start; lines of ``line_length`` samples when given, else of 60 / lpm s."""
    score = phasing_scores(grey, search_from, lpm, fold_lines, line_length)
    return search_from + int(np.argmax(score))          # first maximum = smallest offset on ties


def image(grey: np.ndarray, start: int, lpm: float | None, ioc: int, image_end: int | None = None,
          line_length: float | None = None) -> np.ndarray:
    """The picture from ``start``; lines of ``line_length`` samples when given, else of 60 / lpm s."""
    Ls = _line_length(lpm, line_length)
    W = int(round(np.pi * ioc))
    end = grey.shape[0] if image_end is None else image_end
    rows = max(0, int(np.floor((end - start) / Ls)))
    g = np.clip(np.asarray(grey, dtype=np.float64), 0.0, 1.0)     # float64 sums also for the decoder's float32 grey
    cs = np.concatenate([[0.0], np.cumsum(g)])           # integral of the piecewise-constant grey
    n = g.shape[0]

    def integral(t):
        t = np.clip(t, 0.0, float(n))
        i = np.minimum(np.floor(t).astype(np.int64), n - 1)
        return cs[i] + (t - i) * g[i]

    step = Ls / W
    r = np.arange(rows)[:, None]
    p = np.arange(W)[None, :]
    a = start + r * Ls + p * step
    avg = (integral(a + step) - integral(a)) / step
    return np.clip(np.rint(255.0 * avg), 0, 255).astype(np.uint8)


def decode(pcm: np.ndarray, lpm: float = 120, ioc: int = 576, search_from: int = 0, fold_lines: int = 20,
           image_end: int | None = None, **band) -> dict:
    g = grey_stream(pcm, **band)
    ls = line_start(g, search_from, lpm, fold_lines)
    return dict(grey=g, line_start=ls, image=image(g, ls, lpm, ioc, image_end))
