"""GPU tests of the FM slant correction (csrc/fm.cu slant kernels, api.cu wefax_decode_fm_slant, DESIGN.md §4.7a).

The measured clock error is checked against the generator's truth and against the float64 restatement
(tests/fm_slant_oracle.py) run on the same grey stream; the corrected picture against the transmitted grey levels
rendered at the true line length, with the bars of tests/test_gpu_fm.py."""
import ctypes as C

import numpy as np
import pytest

from wefax_b200 import _native as N
from wefax_b200 import synth

import fm_slant_oracle as S
from test_oracle_fm_slant import DRIFTS, LPMS, NOISES, PHASING_ONLY, truth_error

pytestmark = pytest.mark.gpu

SR = 11025


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def _span(pcm, sample_rate=SR):
    n = len(pcm) if sample_rate == SR else N.resampled_length(len(pcm), sample_rate)
    return 5 * SR, n - 15 * SR          # phasing starts 5 s in, the stop tone 15 s before the end


def test_slant_off_and_fixed_zero_are_the_plain_decode(dec):
    from wefax_b200.fm import decode_fm
    pcm = synth.synth_recording(240.0, lpm=120, seed=11, block=64, drift_ppm=100.0, noise_sigma=0.05)
    frm, end = _span(pcm)
    a = decode_fm(dec, pcm, SR, search_from=frm, image_end=end)
    b = decode_fm(dec, pcm, SR, search_from=frm, image_end=end, slant=0.0)
    assert a.slant is None
    assert a.line_start == b.line_start and a.image.shape == b.image.shape and np.array_equal(a.image, b.image)
    assert b.slant.found and b.slant.ppm == 0.0 and b.slant.line_length == 60.0 / 120 * SR
    assert b.slant.first_line == b.line_start


@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("lpm", LPMS)
@pytest.mark.parametrize("drift", DRIFTS)
def test_auto_slant_recovers_the_drift_and_the_picture(dec, drift, lpm, noise):
    from wefax_b200.fm import decode_fm
    pcm, truth = synth.synth_recording(240.0, lpm=lpm, seed=11, block=64, drift_ppm=drift, noise_sigma=noise,
                                       return_grey=True)
    frm, end = _span(pcm)
    res = decode_fm(dec, pcm, SR, lpm=lpm, search_from=frm, image_end=end, slant="auto", want_grey=True)
    s = res.slant
    assert s.found and abs(s.ppm - drift) < 0.5, s
    assert res.line_start == int(np.floor(s.first_line + 0.5)) and frm <= s.first_line < frm + s.line_length
    ref = S.slant(res.grey, frm, lpm, end)          # float64 stages on the same grey stream
    assert ref["status"] == S.SLANT_OK
    assert abs(s.ppm - ref["ppm"]) < 0.3 and abs(res.line_start - ref["line_start"]) <= 1, (s, ref)
    err = truth_error(res.image, res.line_start, truth, drift, lpm, 576, end)
    assert err.mean() < (6.0 if noise == 0 else 14.0), float(err.mean())
    assert (err <= 16).mean() > (0.93 if noise == 0 else 0.75), float((err <= 16).mean())
    if abs(drift) >= 100:       # without the correction the same recording fails those bars
        off = decode_fm(dec, pcm, SR, lpm=lpm, search_from=frm, image_end=end)
        err0 = truth_error(off.image, off.line_start, truth, drift, lpm, 576, end)
        assert err0.mean() > 30, float(err0.mean())


@pytest.mark.parametrize("lpm,drift", PHASING_ONLY)
def test_auto_slant_from_the_phasing_lines_only(dec, lpm, drift):
    from wefax_b200.fm import decode_fm
    pcm = synth.synth_recording(300.0, lpm=lpm, seed=4, block=8, drift_ppm=drift, noise_sigma=0.05, line_pulse=False)
    frm, end = _span(pcm)
    s = decode_fm(dec, pcm, SR, lpm=lpm, search_from=frm, image_end=end, slant="auto").slant
    assert s.found and abs(s.ppm - drift) < 2.5, s


@pytest.mark.parametrize("lpm,drift", [(120, 100.0), (120, -150.0), (60, 100.0)])
def test_fixed_slant_at_the_true_drift_matches_auto(dec, lpm, drift):
    """FIXED takes its line start from the phasing fold, AUTO from the fit: the starts agree within a sample and the
    pictures within +-16 levels (a one-sample shift moves the pixels on a grey step by more than one level)."""
    from wefax_b200.fm import decode_fm
    pcm = synth.synth_recording(240.0, lpm=lpm, seed=11, block=64, drift_ppm=drift)
    frm, end = _span(pcm)
    auto = decode_fm(dec, pcm, SR, lpm=lpm, search_from=frm, image_end=end, slant="auto")
    fixed = decode_fm(dec, pcm, SR, lpm=lpm, search_from=frm, image_end=end, slant=drift)
    assert fixed.slant.ppm == drift and fixed.slant.line_length == 60.0 / lpm * SR / (1 + drift * 1e-6)
    m = int(round((auto.line_start - fixed.line_start) / fixed.slant.line_length))
    assert abs(auto.line_start - fixed.line_start - m * fixed.slant.line_length) <= 1.0
    a, b = auto.image, fixed.image[m:]
    rows = min(a.shape[0], b.shape[0])
    d = np.abs(a[:rows].astype(int) - b[:rows].astype(int))
    assert (d <= 16).mean() >= 0.99 and d.mean() < 1.5, (float((d <= 16).mean()), float(d.mean()))


def test_auto_slant_of_a_48k_recording(dec):
    from wefax_b200.fm import decode_fm
    pcm = synth.synth_recording(240.0, sample_rate=48000, lpm=120, seed=5, block=64, drift_ppm=60.0)
    frm, end = _span(pcm, 48000)
    s = decode_fm(dec, pcm, 48000, search_from=frm, image_end=end, slant="auto").slant
    assert s.found and abs(s.ppm - 60.0) < 0.5, s


def _tone(f_hz, seconds):
    t = np.arange(int(seconds * SR)) / SR
    return np.round(8000 * np.sin(2 * np.pi * f_hz * t)).astype(np.int16)


@pytest.mark.parametrize("kind", ["noise", "tone"])
def test_auto_slant_without_pulses_is_not_found_and_uncorrected(dec, kind):
    from wefax_b200.fm import decode_fm
    rng = np.random.default_rng(9)
    pcm = (np.clip(rng.normal(0, 8000, size=120 * SR), -32768, 32767).astype(np.int16) if kind == "noise"
           else _tone(1900.0, 120))
    frm, end = 5 * SR, 115 * SR
    off = decode_fm(dec, pcm, SR, search_from=frm, image_end=end)
    auto = decode_fm(dec, pcm, SR, search_from=frm, image_end=end, slant="auto")
    assert auto.slant.status == N.FM_SLANT_NOT_FOUND and not auto.slant.found
    assert auto.slant.lines_used == 0 and auto.slant.ppm == 0.0
    assert auto.line_start == off.line_start and np.array_equal(auto.image, off.image)


def test_slant_rejects_bad_parameters(dec):
    from wefax_b200.fm import decode_fm
    pcm = synth.synth_recording(60.0, seed=1)
    for kw in (dict(slant="sideways"), dict(slant=2500.0), dict(slant="auto", max_slant_ppm=0.0),
               dict(slant="auto", max_slant_ppm=2500.0)):
        with pytest.raises(ValueError):
            decode_fm(dec, pcm, SR, search_from=0, image_end=len(pcm), **kw)
    # the library's own checks, past the Python layer
    desc = N.BatchDesc(1, len(pcm), 1, SR, 0.0, 0.0, 0)
    prm = N.FmParams(120.0, 576, 1500.0, 2300.0, 1200.0, 2600.0, 63, 0, 20, len(pcm))
    img = np.zeros(200 * 1810, dtype=np.uint8)
    rows, w, ls = C.c_int32(0), C.c_int32(0), C.c_int64(0)
    out = N.FmOut(None, img.ctypes.data, img.size, C.addressof(rows), C.addressof(w), C.addressof(ls))
    so = N.FmSlantOut()
    bad = [N.FmSlant(7, 0.0, 0.0, 0.0, 0), N.FmSlant(N.FM_SLANT_FIXED, 2000.5, 0.0, 0.0, 0),
           N.FmSlant(N.FM_SLANT_FIXED, float("nan"), 0.0, 0.0, 0), N.FmSlant(N.FM_SLANT_AUTO, 0.0, 0.0, 0.3, 8),
           N.FmSlant(N.FM_SLANT_AUTO, 0.0, 2000.5, 0.3, 8), N.FmSlant(N.FM_SLANT_AUTO, 0.0, 300.0, 1.5, 8),
           N.FmSlant(N.FM_SLANT_AUTO, 0.0, 300.0, 0.3, 1)]
    for sp in bad:
        rc = dec._lib.wefax_decode_fm_slant(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm),
                                            C.byref(sp), C.byref(out), C.byref(so))
        assert rc == N.ERR_INVALID, (sp.mode, sp.ppm, sp.max_ppm, sp.min_contrast, sp.min_lines)
    # an image sized for nominal lines is too small for the shortest line AUTO may find
    prm.image_end = int(119.9 * 5512.5)                 # 119 nominal lines, 120 at -2000 ppm
    small = np.zeros(119 * 1810, dtype=np.uint8)
    out_small = N.FmOut(None, small.ctypes.data, small.size, C.addressof(rows), C.addressof(w), C.addressof(ls))
    rc = dec._lib.wefax_decode_fm_slant(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm),
                                        C.byref(N.FmSlant(N.FM_SLANT_AUTO, 0.0, 2000.0, 0.3, 8)), C.byref(out_small),
                                        C.byref(so))
    assert rc == N.ERR_INVALID


@pytest.mark.slow
@pytest.mark.parametrize("k", range(8))
def test_auto_slant_on_the_noisy_batch_recordings(dec, k):
    from wefax_b200.fm import decode_fm
    spec = synth.batch_spec(k, noisy=True)
    pcm = synth.synth_recording(600.0, block=8, **spec)
    frm, end = _span(pcm)
    s = decode_fm(dec, pcm, SR, lpm=spec["lpm"], ioc=spec["ioc"], search_from=frm, image_end=end, slant="auto").slant
    assert s.found and abs(s.ppm - spec["drift_ppm"]) < 0.2, (spec, s)
