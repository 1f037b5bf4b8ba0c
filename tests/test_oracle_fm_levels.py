"""CPU tests of the tuning-offset measurement's float64 restatement (tests/fm_levels_oracle.py, DESIGN.md §4.7d).

The restatement runs on the float64 grey of oracle/fm_oracle.grey_stream (the transform at the recording's own length)
of synthetic transmissions, at the phasing line start of oracle/fm_oracle.line_start:
  * accuracy over offsets of -150 .. +150 Hz, noise sigma 0, 0.05 and 0.1, four seeds with (LPM, IOC) pairs from 60
    to 240 LPM and both IOCs, against bars set from the restatement's own worst case;
  * NOT_FOUND on noise only, a steady 1900 Hz tone, a transmission with a 400 Hz shift and an offset beyond
    max_offset_hz;
  * the sets' geometry: 240 LPM (wb = 138, e = 35), an image end or a recording end inside the fold lines, empty sets;
  * Python argument checks and the ctypes struct sizes, without a GPU.
"""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

import fm_levels_oracle as FL
from oracle import fm_oracle as F
from wefax_b200 import _native as N
from wefax_b200 import synth
from wefax_b200.fm import decode_fm_charts, decode_fm_charts_batch, main

SR = 11025
PAIRS = {1: (120, 576), 2: (240, 288), 3: (60, 576), 4: (90, 288)}     # seed -> (LPM, IOC)
OFFSETS = (-150.0, -50.0, 0.0, 45.0, 150.0)
FROM = 5 * SR                     # the phasing lines start 5 s into synth_recording

# |estimate - truth| bars in Hz, (|offset| <= 50, |offset| = 150), per noise sigma.  Worst cases of the restatement over
# this grid: 0.0014 / 0.0014 (sigma 0), 0.99 / 3.59 (0.05), 2.86 / 13.2 (0.1); the bars are 1.5 times the larger of
# these and of an independent run over seeds 1-4 (0.05: 1.34 / 4.28; 0.1: 2.71 / 13.4), rounded up.
BARS = {0.0: (0.01, 0.01), 0.05: (2.1, 6.5), 0.1: (4.3, 20.1)}


def _rec(seed, sigma, offset, lpm=None, ioc=None, **kw):
    lpm_, ioc_ = PAIRS[seed]
    lpm, ioc = lpm or lpm_, ioc or ioc_
    return synth.synth_recording(20.0 + 60.0 / lpm * 44, lpm=lpm, ioc=ioc, seed=seed, n_phasing=20, block=64,
                                 noise_sigma=sigma, carrier_offset_hz=offset, **kw)


def _measure(pcm, lpm, **kw):
    g = F.grey_stream(pcm.astype(np.float64), padded=False)
    s = F.line_start(g, FROM, lpm, 20)
    return FL.measure(g, s, 60.0 / lpm * SR, **kw), g, s


@pytest.mark.parametrize("sigma", sorted(BARS))
def test_offset_accuracy(sigma):
    for seed, (lpm, _) in PAIRS.items():
        for off in OFFSETS:
            m, _, _ = _measure(_rec(seed, sigma, off), lpm)
            assert m["status"] == FL.OK, (seed, off, m)
            err = abs(m["offset_hz"] - off)
            k = int(abs(off) > 50)
            assert err <= BARS[sigma][k], (seed, off, m["offset_hz"])
            # noise pulls both levels toward the band centre: the span shrinks, never grows past the transmitter's
            assert m["white_hz"] - m["black_hz"] <= 800.01
            if sigma == 0.1 and abs(off) == 150:
                assert abs(m["offset_hz"]) < abs(off) and abs(m["offset_hz"]) >= 0.85 * abs(off)


def test_a_clean_transmission_is_measured_exactly_at_its_levels():
    m, g, _ = _measure(_rec(1, 0.0, 45.0), 120)
    assert abs(m["black_hz"] - 1545.0) < 0.01 and abs(m["white_hz"] - 2345.0) < 0.01
    # 120 LPM: wb = 276, e = 69; pulse o in [69, 207), body o in [345, 5443) on each of the 20 lines
    assert (m["white_samples"], m["black_samples"]) == (20 * 138, 20 * 5098)


def _noise(n, seed):
    rng = np.random.default_rng(seed)
    return np.clip(np.round(rng.normal(0.0, 0.1, n) * 32767.0), -32768, 32767).astype(np.int16)


def test_not_found_on_noise_only():
    m, _, _ = _measure(_noise(40 * SR, 3), 120)
    assert m["black_samples"] > 0 and m["white_samples"] > 0
    assert m["status"] == FL.NOT_FOUND and abs(m["white_hz"] - m["black_hz"]) < 100


def test_not_found_on_a_steady_tone():
    t = np.arange(40 * SR) / SR
    pcm = np.round(8000 * np.sin(2 * np.pi * 1900.0 * t)).astype(np.int16)
    m, _, _ = _measure(pcm, 120)
    assert m["status"] == FL.NOT_FOUND and abs(m["white_hz"] - m["black_hz"]) < 1.0


def test_not_found_on_a_400_hz_shift():
    _, grey = synth.synth_recording(20.0 + 0.5 * 44, lpm=120, seed=5, n_phasing=20, block=64, return_grey=True)
    phase = 2.0 * np.pi * np.cumsum(1700.0 + 400.0 * grey) / SR
    pcm = np.clip(np.round(0.25 * np.sin(phase) * 32767.0), -32768, 32767).astype(np.int16)
    m, _, _ = _measure(pcm, 120)
    assert abs((m["white_hz"] - m["black_hz"]) - 400.0) < 1.0 and abs(m["offset_hz"]) < 1.0
    assert m["status"] == FL.NOT_FOUND


def test_not_found_beyond_max_offset_hz():
    m, _, _ = _measure(_rec(1, 0.0, 150.0), 120, max_offset_hz=100.0)
    assert abs(m["offset_hz"] - 150.0) < 0.01 and m["status"] == FL.NOT_FOUND
    m, _, _ = _measure(_rec(1, 0.0, 250.0), 120)           # the default bound is 200 Hz
    assert abs(m["offset_hz"] - 250.0) < 0.01 and m["status"] == FL.NOT_FOUND
    m, _, _ = _measure(_rec(1, 0.0, 250.0), 120, max_offset_hz=300.0)
    assert m["status"] == FL.OK


def _brute(start, Ls, lines, end, o_lo, o_hi):
    out = []
    for l in range(lines):
        for o in range(o_lo, o_hi):
            i = start + math.floor(l * Ls + o)
            if 0 <= i < end:
                out.append(i)
    return out


def test_sets_at_240_lpm():
    Ls = 60.0 / 240 * SR
    wb, e, po, bo = FL.set_offsets(Ls)
    assert (wb, e) == (138, 35)
    assert (po[0], po[-1] + 1, bo[0], bo[-1] + 1) == (35, 103, 173, 2721)
    for offs, lo, hi in ((po, 35, 103), (bo, 173, 2721)):
        got = FL.set_indices(1001, Ls, 20, 10 ** 9, offs)
        assert got.tolist() == _brute(1001, Ls, 20, 10 ** 9, lo, hi)
    m, _, _ = _measure(_rec(2, 0.0, 0.0), 240)
    assert (m["white_samples"], m["black_samples"]) == (20 * 68, 20 * 2548) and m["status"] == FL.OK


@pytest.mark.parametrize("Ls", [5512.5, 11025.0, 7350.0, 5512.5 / (1 + 123.4e-6)])
def test_an_image_end_inside_the_fold_lines(Ls):
    start = 777
    end = start + int(7.3 * Ls)           # 7 whole lines and part of the eighth
    _, _, po, bo = FL.set_offsets(Ls)
    for offs in (po, bo):
        got = FL.set_indices(start, Ls, 20, end, offs)
        assert got.tolist() == _brute(start, Ls, 20, end, int(offs[0]), int(offs[-1]) + 1)
        assert 7 * offs.size < got.size < 20 * offs.size
    # the recording itself ending there: the same sets through measure
    g = np.random.default_rng(1).random(end).astype(np.float32)
    a = FL.measure(g, start, Ls, image_end=None)
    b = FL.measure(np.concatenate([g, np.zeros(5000, np.float32)]), start, Ls, image_end=end)
    assert (a["black_samples"], a["white_samples"], a["b"], a["w"]) == (b["black_samples"], b["white_samples"], b["b"],
                                                                       b["w"])


def test_empty_sets():
    g = np.linspace(0.0, 1.0, 50000).astype(np.float32)
    m = FL.measure(g, 60000, 5512.5)                        # the line start past the end: both sets empty
    assert (m["black_samples"], m["white_samples"]) == (0, 0) and m["status"] == FL.NOT_FOUND
    assert math.isnan(m["b"]) and math.isnan(m["w"])
    m = FL.measure(g, 0, 10.0)                              # wb = 1, e = 1: no pulse offset
    assert m["white_samples"] == 0 and m["black_samples"] > 0 and m["status"] == FL.NOT_FOUND


def test_lower_median_is_an_element():
    v = np.array([3.0, 1.0, 2.0, 4.0], np.float32)
    assert FL.lower_median(v) == np.float32(2.0) and FL.lower_median(v[:3]) == np.float32(2.0)


# ---- Python arguments and the C structs, without a GPU -----------------------------------------------------------------

@pytest.mark.parametrize("bad", [dict(levels="on"), dict(levels=True), dict(levels="auto", max_offset_hz=0.0),
                                 dict(levels="auto", max_offset_hz=-5.0), dict(levels="auto", max_offset_hz=300.5),
                                 dict(levels="auto", max_offset_hz=float("nan")), dict(max_offset_hz=True),
                                 dict(levels="auto", max_offset_hz="100")])
def test_bad_levels_arguments(bad):
    with pytest.raises(ValueError):
        decode_fm_charts(None, np.zeros(4096, np.int16), SR, **bad)
    with pytest.raises(ValueError):
        decode_fm_charts_batch(None, np.zeros((2, 4096), np.int16), SR, **bad)


def test_cli_levels_needs_all(tmp_path, capsys):
    wav, png = str(tmp_path / "missing.wav"), str(tmp_path / "out.png")
    with pytest.raises(SystemExit) as e:
        main([wav, png, "--levels", "auto"])
    assert e.value.code == 2 and "--levels needs --all" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        main([wav, png, "--all", "--levels", "auto", "--max-offset-hz", "400"])
    assert e.value.code == 2


def test_struct_sizes_and_constants():
    assert C.sizeof(N.FmLevels) == 16 and C.sizeof(N.FmLevelsOut) == 48
    assert C.sizeof(N.FmChartParams) == 192 and C.sizeof(N.FmChart) == 128
    hdr = open(os.path.join(os.path.dirname(N.HERE), "include", "wefax_b200.h")).read()
    consts = dict(re.findall(r"#define WEFAX_FM_LEVELS_(\w+) ([\d.]+)", hdr))
    assert {k: float(v) for k, v in consts.items()} == {
        "OFF": N.FM_LEVELS_OFF, "AUTO": N.FM_LEVELS_AUTO, "OK": N.FM_LEVELS_OK, "NOT_FOUND": N.FM_LEVELS_NOT_FOUND,
        "NOT_MEASURED": N.FM_LEVELS_NOT_MEASURED, "MAX_OFFSET_HZ": N.FM_LEVELS_MAX_OFFSET_HZ}
    assert "wefax_decode_fm_charts_levels" in N.EXPORTED_SYMBOLS and N.ABI_VERSION == 5
