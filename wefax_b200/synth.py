"""Deterministic synthetic WEFAX recordings (int16 mono PCM).

Signal model (SURVEY.md §8d; transmission format from the reference's
README.md:85-101): grey g in [0,1] maps to an instantaneous frequency
f = 1500 + 800*g Hz (black 1500 Hz, white 2300 Hz), the phase is the running
sum of f, amplitude is 0.25 of full scale.  A transmission is

    5 s start tone (black/white alternating at 300 Hz for IOC576, 675 Hz for IOC288)
    n_phasing lines: 5 % white, 95 % black
    image lines:     5 % white, then seeded block-constant greys (no white part with line_pulse=False)
    5 s stop tone (450 Hz alternation)
    10 s black

Impairments for the "noisy" configs: AWGN, a constant carrier offset and a
sample-clock drift (time-warp t -> t*(1+ppm*1e-6)).

Everything here is host-side numpy: these are the inputs both the oracle and
the CUDA path eat.  Nothing here is on the decode path.
"""
from __future__ import annotations

import struct

import numpy as np

TARGET_RATE = 11025

#: (lpm, ioc) cycle used by the batch configs (BASELINE.json configs[3]).
BATCH_LPMS = (60, 90, 120, 240)
BATCH_IOCS = (576, 288)


def synth_recording(duration_s: float,
                    sample_rate: int = TARGET_RATE,
                    lpm: int = 120,
                    ioc: int = 576,
                    seed: int = 0,
                    n_phasing: int = 30,
                    noise_sigma: float = 0.0,
                    carrier_offset_hz: float = 0.0,
                    drift_ppm: float = 0.0,
                    block: int = 8,
                    amplitude: float = 0.25,
                    return_grey: bool = False,
                    line_pulse: bool = True):
    """One synthetic transmission, ``int(round(duration_s*sample_rate))`` int16 samples.

    ``line_pulse=False``: image lines carry no white pulse, only the phasing lines do (as on most real charts)."""
    n = int(round(duration_s * sample_rate))
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64) / sample_rate
    if drift_ppm:
        t = t * (1.0 + drift_ppm * 1e-6)

    line_t = 60.0 / lpm
    start_len, stop_len, black_len = 5.0, 5.0, 10.0
    tail = stop_len + black_len
    # keep the structure sensible for very short test clips
    if duration_s < start_len + tail + (n_phasing + 4) * line_t:
        scale = duration_s / (start_len + tail + (n_phasing + 4) * line_t)
        start_len *= scale
        stop_len *= scale
        black_len *= scale
        tail = stop_len + black_len
        n_phasing = max(2, int(n_phasing * scale))
    t_phase0 = start_len
    t_img0 = t_phase0 + n_phasing * line_t
    t_stop0 = duration_s - tail
    t_black0 = duration_s - black_len

    grey = np.zeros(n, dtype=np.float64)

    start_hz = 300.0 if ioc == 576 else 675.0
    m = t < t_phase0
    grey[m] = (np.floor(2.0 * start_hz * t[m]) % 2 == 0).astype(np.float64)

    m = (t >= t_phase0) & (t < t_img0)
    frac = ((t[m] - t_phase0) / line_t) % 1.0
    grey[m] = (frac < 0.05).astype(np.float64)

    m = (t >= t_img0) & (t < t_stop0)
    idx = np.nonzero(m)[0]
    if idx.size:
        frac = ((t[idx] - t_img0) / line_t) % 1.0
        nblk = idx.size // block + 1
        levels = rng.integers(0, 256, size=nblk).astype(np.float64) / 255.0
        content = np.repeat(levels, block)[: idx.size]
        grey[idx] = np.where(frac < 0.05, 1.0, content) if line_pulse else content

    m = (t >= t_stop0) & (t < t_black0)
    grey[m] = (np.floor(2.0 * 450.0 * (t[m] - t_stop0)) % 2 == 0).astype(np.float64)
    # t >= t_black0 stays black (0)

    f = 1500.0 + 800.0 * grey + carrier_offset_hz
    if drift_ppm:
        f = f * (1.0 + drift_ppm * 1e-6)
    phase = 2.0 * np.pi * np.cumsum(f) / sample_rate
    x = amplitude * np.sin(phase)
    if noise_sigma:
        x = x + rng.normal(0.0, noise_sigma, size=n)
    x = np.clip(np.round(x * 32767.0), -32768, 32767)
    if return_grey:      # the per-sample grey level that was transmitted (ground truth of the FM extension)
        return x.astype(np.int16), grey
    return x.astype(np.int16)


def batch_spec(k: int, noisy: bool = False) -> dict:
    """Parameters of recording ``k`` of the batch configs (SURVEY.md §8d C4/C5)."""
    spec = dict(lpm=BATCH_LPMS[k % 4], ioc=BATCH_IOCS[(k // 4) % 2],
                seed=(5000 if noisy else 1000) + k)
    if noisy:
        r = np.random.default_rng(7_000_000 + k)
        spec.update(noise_sigma=float(r.uniform(0.02, 0.1)),
                    carrier_offset_hz=float(r.uniform(-50.0, 50.0)),
                    drift_ppm=5.0)
    return spec


def write_wav(path: str, pcm: np.ndarray, sample_rate: int) -> None:
    """Minimal RIFF/WAVE PCM16 writer (mono ``(n,)`` or interleaved ``(n, ch)``)."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    ch = 1 if pcm.ndim == 1 else pcm.shape[1]
    data = pcm.tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE"
    hdr += b"fmt " + struct.pack("<IHHIIHH", 16, 1, ch, sample_rate,
                                 sample_rate * ch * 2, ch * 2, 16)
    hdr += b"data" + struct.pack("<I", len(data))
    with open(path, "wb") as fh:
        fh.write(hdr)
        fh.write(data)
