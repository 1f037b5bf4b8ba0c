"""CPU tests of the chart finder's float64 restatement (tests/fm_charts_oracle.py: tone_scores, find_charts, lpm_scores;
DESIGN.md §4.7b) and of the ctypes layout of wefax_decode_fm_charts.

On the generator's transmitted grey and on the float64 grey stream of short broadcasts, every chart is found with its
IOC and LPM, and its spans are within one tone window of the truth.  The segmentation rules are checked on hand-made
window classes, and noise alone or a steady carrier yields no chart.
"""
import ctypes as C

import numpy as np
import pytest

import fm_charts_oracle as FC
from oracle import fm_oracle as F
from wefax_b200 import _native as N
from wefax_b200 import synth

SR = 11025
T = FC.TONE_WINDOW
LPMS = (60, 90, 100, 120, 180, 240)


def _broadcast(ioc, noise_sigma=0.0, seed=5):
    charts = [dict(duration_s=20 + 60 / lpm * 40, lpm=lpm, ioc=ioc, block=64, n_phasing=20) for lpm in LPMS]
    return synth.synth_broadcast(charts, noise_sigma=noise_sigma, gap_s=3.0, seed=seed, return_grey=True)


def _check_charts(grey, truth):
    charts = FC.find_charts(FC.tone_classes(FC.tone_scores(grey)), len(grey))
    assert len(charts) == len(truth)
    for c, tr in zip(charts, truth):
        assert c["ioc"] == tr["ioc"]
        assert abs(c["tone_begin"] - tr["tone_begin"]) <= T
        assert abs(c["search_from"] - tr["search_from"]) <= T
        assert abs(c["image_end"] - tr["stop_begin"]) <= T and c["stop_found"]
        lpm, score = FC.best_lpm(FC.lpm_scores(grey, c["search_from"]))
        assert lpm == tr["lpm"] and score > 0.8, (tr, lpm, score)
    return charts


@pytest.mark.parametrize("ioc", [576, 288])
def test_every_chart_on_the_transmitted_grey(ioc):
    _, truth, grey = _broadcast(ioc)
    _check_charts(grey, truth)


@pytest.mark.parametrize("ioc,noise", [(576, 0.0), (288, 0.0), (576, 0.05), (288, 0.05)])
def test_every_chart_on_the_grey_stream(ioc, noise):
    pcm, truth, _ = _broadcast(ioc, noise, seed=6)
    _check_charts(F.grey_stream(pcm), truth)


def test_lpm_scores_of_related_and_unrelated_line_lengths():
    """Measured on the clean 576 broadcast: the true LPM scores 0.93-0.95; half or double 0.34-0.45; 1.5 times
    0.25-0.35; three or four times 0.09-0.30; LPM 100 against the others (no small ratio) 0.05-0.15."""
    pcm, truth, _ = _broadcast(576)
    grey = F.grey_stream(pcm)
    charts = FC.find_charts(FC.tone_classes(FC.tone_scores(grey)), len(grey))
    for c, tr in zip(charts, truth):
        s = FC.lpm_scores(grey, c["search_from"], LPMS)
        for lpm, v in zip(LPMS, s):
            ratio = max(lpm, tr["lpm"]) / min(lpm, tr["lpm"])
            if lpm == tr["lpm"]:
                assert v > 0.9
            elif ratio == 2:
                assert v <= 0.5
            elif ratio == 1.5:
                assert v <= 0.4
            elif ratio in (3, 4):
                assert v <= 0.35
            else:
                assert v <= 0.2, (tr["lpm"], lpm, v)


def test_sinusoid_and_square_wave_ratios():
    j = np.arange(4 * T)
    sine = 0.5 + 0.5 * np.sin(2 * np.pi * 300 * j / SR + 0.3)
    square = (np.floor(2 * 450 * j / SR) % 2 == 0).astype(float)
    s = FC.tone_scores(sine)
    assert np.allclose(s[:, 0], 1.0, atol=1e-9) and np.allclose(s[:, 1:3], 0.0, atol=1e-9)
    q = FC.tone_scores(square)
    assert np.allclose(q[:, 1], 8 / np.pi ** 2, atol=1e-3)
    assert (FC.tone_classes(s) == FC.START_576).all() and (FC.tone_classes(q) == FC.STOP).all()
    assert (FC.tone_scores(np.full(2 * T, 0.75)) == 0).all()      # V = 0 exactly: no ratio


def _classes(*runs):
    return np.concatenate([np.full(k, c) for c, k in runs])


def test_chart_without_a_stop_tone():
    cl = _classes((FC.START_576, 12), (FC.NONE, 50))
    n = len(cl) * T + 100
    assert FC.find_charts(cl, n) == [dict(tone_begin=0, search_from=12 * T, image_end=n, stop_found=False, ioc=576)]


def test_two_start_tones_back_to_back():
    cl = _classes((FC.NONE, 3), (FC.START_576, 12), (FC.START_288, 11), (FC.NONE, 30), (FC.STOP, 10), (FC.NONE, 4))
    got = FC.find_charts(cl, len(cl) * T)
    assert got == [dict(tone_begin=3 * T, search_from=15 * T, image_end=15 * T, stop_found=False, ioc=576),
                   dict(tone_begin=15 * T, search_from=26 * T, image_end=56 * T, stop_found=True, ioc=288)]


def test_short_start_tone_and_lone_stop_tone_are_ignored():
    cl = _classes((FC.STOP, 12), (FC.NONE, 5), (FC.START_288, 9), (FC.NONE, 20), (FC.START_576, 10), (FC.NONE, 7),
                  (FC.STOP, 9), (FC.NONE, 5))
    n = len(cl) * T
    assert FC.find_charts(cl, n) == [dict(tone_begin=46 * T, search_from=56 * T, image_end=n, stop_found=False,
                                         ioc=576)]
    assert FC.find_charts(_classes((FC.START_576, 9), (FC.NONE, 40), (FC.STOP, 12)), 61 * T) == []


def test_tone_run_at_the_very_end():
    cl = _classes((FC.NONE, 5), (FC.START_288, 10))
    n = len(cl) * T + 1000
    assert FC.find_charts(cl, n) == [dict(tone_begin=5 * T, search_from=15 * T, image_end=n, stop_found=False,
                                         ioc=288)]
    # a broadcast ending in its start tone: the chart is reported, its fold reads one sample (no LPM)
    assert FC.lpm_scores(np.ones(n), n).max() < 1e-3


def test_noise_and_a_steady_carrier_are_no_charts():
    rng = np.random.default_rng(3)
    noise = np.clip(np.round(rng.normal(0, 0.2, 30 * SR) * 32767), -32768, 32767)
    carrier = np.round(0.25 * 32767 * np.sin(2 * np.pi * 1900.0 * np.arange(30 * SR) / SR))
    for pcm in (noise, carrier, np.zeros(30 * SR)):
        grey = F.grey_stream(pcm)
        assert FC.find_charts(FC.tone_classes(FC.tone_scores(grey)), len(grey)) == []


def test_broadcast_truth_and_pieces():
    charts = [dict(duration_s=40.0, lpm=120, ioc=576, seed=3, block=64), dict(duration_s=30.0, lpm=240, ioc=288)]
    pcm, truth = synth.synth_broadcast(charts, gap_s=2.0, seed=1)
    first = synth.synth_recording(40.0, lpm=120, ioc=576, seed=3, block=64)
    assert np.array_equal(pcm[: len(first)], first)
    assert (pcm[len(first): len(first) + 2 * SR] == 0).all()
    assert len(pcm) == 72 * SR
    assert truth == [dict(tone_begin=0, search_from=5 * SR, stop_begin=25 * SR, lpm=120, ioc=576),
                     dict(tone_begin=42 * SR, search_from=47 * SR, stop_begin=57 * SR, lpm=240, ioc=288)]


def test_chart_structs_are_pinned():
    assert C.sizeof(N.FmChartParams) == 192
    assert C.sizeof(N.FmChart) == 128
    assert N.FmChart.slant.offset == 80 and N.FmChart.line_start.offset == 64
    assert N.FmChartParams.lpm_candidates.offset == 128
    assert "wefax_decode_fm_charts" in N.EXPORTED_SYMBOLS and N.ABI_VERSION == 5
