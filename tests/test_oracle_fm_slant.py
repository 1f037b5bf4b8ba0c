"""CPU tests of the FM slant correction: the float64 restatement (tests/fm_slant_oracle.py) against the ground
truth of the synthetic generator, and the host side of the Python layer (argument checks, struct layouts, the
command line).  The CUDA path is checked against both in tests/test_gpu_fm_slant.py."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import fm_oracle as F
from wefax_b200 import _native as N
from wefax_b200 import synth

import fm_slant_oracle as S

SR = 11025
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DRIFTS = (-150.0, -40.0, 5.0, 100.0)
LPMS = (60, 120, 240)
NOISES = (0.0, 0.05)


def truth_start(line_start: int, drift: float, lpm: float):
    """The synthetic transmission's line start nearest `line_start` and its true line length (samples)."""
    Lt = 60.0 / lpm * SR / (1.0 + drift * 1e-6)
    t0 = 5 * SR / (1.0 + drift * 1e-6)          # the phasing lines start 5 s into the transmitter's time
    return t0 + round((line_start - t0) / Lt) * Lt, Lt


def truth_error(image, line_start, truth, drift, lpm, ioc, image_end):
    ts, Lt = truth_start(line_start, drift, lpm)
    timg = S.image(truth, ts, Lt, ioc, image_end)
    rows = min(image.shape[0], timg.shape[0])
    return np.abs(image[:rows].astype(int) - timg[:rows].astype(int))


@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("lpm", LPMS)
@pytest.mark.parametrize("drift", DRIFTS)
def test_oracle_slant_recovers_the_drift(drift, lpm, noise):
    pcm, truth = synth.synth_recording(240.0, lpm=lpm, seed=11, block=64, drift_ppm=drift, noise_sigma=noise,
                                       return_grey=True)
    g = F.grey_stream(pcm)
    frm, end = 5 * SR, len(pcm) - 15 * SR
    r = S.slant(g, frm, lpm, end)
    assert r["status"] == S.SLANT_OK
    assert abs(r["ppm"] - drift) < 0.5, r
    assert frm <= r["first_line"] < frm + r["line_length"]
    assert r["lines_used"] >= 0.8 * r["lines_total"]
    err = truth_error(S.image(g, r["line_start"], r["line_length"], 576, end), r["line_start"],
                      truth, drift, lpm, 576, end)
    assert err.mean() < (6.0 if noise == 0 else 14.0), float(err.mean())
    assert (err <= 16).mean() > (0.93 if noise == 0 else 0.75), float((err <= 16).mean())
    if abs(drift) >= 100:       # the uncorrected picture fails the same bars
        ls0 = F.line_start(g, frm, lpm, 20)
        err0 = truth_error(F.image(g, ls0, lpm, 576, end), ls0, truth, drift, lpm, 576, end)
        assert err0.mean() > 30, float(err0.mean())


#: recordings whose image lines carry no pulse: the fit rests on the ~30 phasing lines
PHASING_ONLY = [(120, 100.0), (120, -40.0), (60, 60.0)]


@pytest.mark.parametrize("lpm,drift", PHASING_ONLY)
def test_oracle_slant_from_the_phasing_lines_only(lpm, drift):
    pcm = synth.synth_recording(300.0, lpm=lpm, seed=4, block=8, drift_ppm=drift, noise_sigma=0.05, line_pulse=False)
    r = S.slant(F.grey_stream(pcm), 5 * SR, lpm, len(pcm) - 15 * SR)
    assert r["status"] == S.SLANT_OK and abs(r["ppm"] - drift) < 2.5, r
    assert r["lines_used"] <= 31


def test_oracle_slant_finds_nothing_in_noise():
    rng = np.random.default_rng(3)
    pcm = np.clip(rng.normal(0, 8000, size=60 * SR), -32768, 32767).astype(np.int16)
    r = S.slant(F.grey_stream(pcm), 5 * SR, 120, 55 * SR)
    assert r["status"] == S.SLANT_NOT_FOUND


def test_slant_geometry():
    geo = S.slant_geometry(120, 5 * SR, 65 * SR, 300.0)
    assert (geo["wb"], geo["D"], geo["Bn"], geo["wbb"], geo["R"]) == (276, 17, 325, 16, 85)
    assert geo["L"] == 119 and geo["Lc"] == 119          # 60 s = 120 lines, less what +-300 ppm may cost
    assert S.slant_geometry(120, 0, 3600 * SR, 300.0)["Lc"] == S.SLANT_COARSE_LINES


def test_synth_line_pulse_only_removes_the_image_line_pulses():
    kw = dict(lpm=120, seed=2, block=16, return_grey=True)
    _, a = synth.synth_recording(40.0, **kw)
    _, b = synth.synth_recording(40.0, line_pulse=False, **kw)
    img = slice(int((5 + 30 * 0.5) * SR), int(25 * SR))          # image lines: after 30 phasing lines, before the stop tone
    assert np.array_equal(a[:img.start], b[:img.start]) and np.array_equal(a[img.stop:], b[img.stop:])
    frac = (np.arange(img.start, img.stop) / (0.5 * SR)) % 1.0
    pulse = frac < 0.049
    assert (a[img][pulse] == 1.0).all() and not (b[img][pulse] == 1.0).all()
    assert np.array_equal(a[img][frac > 0.051], b[img][frac > 0.051])


def test_slant_struct_layouts():
    # sizes and offsets the C compiler gives wefax_fm_slant / wefax_fm_slant_out (LP64)
    assert ctypes.sizeof(N.FmSlant) == 40
    assert [getattr(N.FmSlant, f).offset for f, _ in N.FmSlant._fields_] == [0, 8, 16, 24, 32]
    assert ctypes.sizeof(N.FmSlantOut) == 48
    assert [getattr(N.FmSlantOut, f).offset for f, _ in N.FmSlantOut._fields_] == [0, 8, 16, 24, 28, 32, 40]


class _NoNative:
    """A decoder whose native calls fail the test: argument checks must come first."""
    def __getattr__(self, name):
        raise AssertionError(f"native layer reached ({name})")


@pytest.mark.parametrize("kw", [dict(slant="AUTO"), dict(slant="fixed"), dict(slant=2500.0), dict(slant=-2000.5),
                                dict(slant=float("nan")), dict(slant=float("inf")), dict(slant=True),
                                dict(slant=[5.0]), dict(slant="auto", max_slant_ppm=0.0),
                                dict(slant="auto", max_slant_ppm=-10.0), dict(slant="auto", max_slant_ppm=2001.0),
                                dict(slant="auto", max_slant_ppm=float("nan"))])
def test_decode_fm_rejects_bad_slant_arguments(kw):
    from wefax_b200.fm import decode_fm
    pcm = np.zeros(SR, dtype=np.int16)
    with pytest.raises(ValueError):
        decode_fm(_NoNative(), pcm, SR, search_from=0, image_end=SR, **kw)


def test_slant_params_accepts_the_documented_forms():
    from wefax_b200.fm import slant_params
    assert slant_params(None) is None
    a = slant_params("auto", 150)
    assert (a.mode, a.max_ppm, a.min_contrast, a.min_lines) == (N.FM_SLANT_AUTO, 150.0, 0.3, 8)
    f = slant_params(-12)
    assert (f.mode, f.ppm) == (N.FM_SLANT_FIXED, -12.0)
    assert slant_params(np.float32(2000.0)).ppm == 2000.0


def test_fm_command_line_help():
    r = subprocess.run([sys.executable, "-m", "wefax_b200.fm", "--help"], cwd=ROOT, capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stderr
    assert "--slant" in r.stdout and "--lpm" in r.stdout and "--ioc" in r.stdout
    r = subprocess.run([sys.executable, "-m", "wefax_b200.fm", "in.wav", "out.png", "--slant", "sideways"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--slant" in r.stderr
