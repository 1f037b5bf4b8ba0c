"""CPU tests of the FM-extension oracle (oracle/fm_oracle.py; SURVEY.md §8(f) N4) and its host logic.
No reference parity exists for this mode; the oracle is pinned to scipy for its filter / Hilbert pieces
and to the ground truth of the synthetic generator for the whole definition."""
from fractions import Fraction

import numpy as np

from oracle import fm_oracle as F
from wefax_b200 import synth

SR = 11025


def test_fir_filtfilt_is_scipy_filtfilt_with_padlen_9():
    import scipy.signal
    rng = np.random.default_rng(2)
    x = rng.normal(size=4000) * 1000
    h = F.bandpass_taps(1200, 2600, SR, 63)
    ref = scipy.signal.filtfilt(h, [1.0], x, padlen=9)
    assert np.allclose(F.fir_filtfilt(h, x), ref, rtol=0, atol=1e-9 * np.abs(ref).max())
    assert np.allclose(F.hilbert_imag(x), scipy.signal.hilbert(x).imag, rtol=0, atol=1e-9 * np.abs(x).max())
    assert np.allclose(F.hilbert_imag(x[:-1]), scipy.signal.hilbert(x[:-1]).imag, rtol=0, atol=1e-9 * np.abs(x).max())


def test_bandpass_taps_pass_the_carrier_and_stop_the_rest():
    h = F.bandpass_taps(1200, 2600, SR, 63)
    assert h.shape == (63,) and np.allclose(h, h[::-1])
    f = np.fft.rfftfreq(8192, 1 / SR)
    H2 = np.abs(np.fft.rfft(h, 8192)) ** 2            # applied forwards and backwards
    band = (f > 1500) & (f < 2300)
    assert H2[band].min() > 0.9 and H2[band].max() < 1.1
    assert H2[(f < 700) | (f > 3100)].max() < 1e-4


def test_fm_oracle_recovers_the_transmitted_picture():
    pcm, truth = synth.synth_recording(60.0, seed=7, block=64, return_grey=True)
    d = F.decode(pcm, 120, 576, search_from=5 * SR, fold_lines=20, image_end=45 * SR)
    assert abs(d["line_start"] - 5 * SR) <= 2
    timg = F.image(truth, 5 * SR, 120, 576, 45 * SR)
    rows = min(timg.shape[0], d["image"].shape[0])
    err = np.abs(d["image"][:rows].astype(int) - timg[:rows].astype(int))
    assert err.mean() < 4.0 and (err <= 16).mean() > 0.95
    # a frequency offset shifts every grey level by offset / 800 Hz: the mean error shows it
    pcm_off = synth.synth_recording(60.0, seed=7, block=64, carrier_offset_hz=40.0)
    d2 = F.decode(pcm_off, 120, 576, search_from=5 * SR, fold_lines=20, image_end=45 * SR)
    rows = min(timg.shape[0], d2["image"].shape[0])
    shift = (d2["image"][30:rows].astype(int) - timg[30:rows].astype(int)).mean()
    assert 8 < shift < 16            # 40 / 800 * 255 = 12.75 levels, less what clips at white


def test_image_span_from_tone_flags():
    from wefax_b200.fm import image_span
    start = np.zeros(60, dtype=bool)
    stop = np.zeros(60, dtype=bool)
    start[:5] = True
    start[45:50] = True        # the stop tone also passes the start-tone test (SURVEY.md §8c)
    stop[45:50] = True
    assert image_span(start, stop) == (5 * SR, 45 * SR)
    assert image_span(np.zeros(10, dtype=bool), np.zeros(10, dtype=bool)) == (0, 10 * SR)


def _smooth7(v):
    for p in (2, 3, 5, 7):
        while v % p == 0:
            v //= p
    return v == 1


def test_next_smooth_length_is_the_librarys():
    """The restatement of csrc/fft_plan.cu next_smooth_length against a brute-force search with the library's own
    planning test: primes, numbers just above a 7-smooth one, powers of two and small m."""
    from wefax_b200 import _native as N

    def can_plan(v):
        try:
            return N.fft_plan_describe(v)[1] == 0
        except ValueError:
            return False

    def brute(m):
        v = m
        while not (_smooth7(v) and can_plan(v)):
            v += 1
        return v

    primes = [p for p in range(2, 6000) if all(p % q for q in range(2, int(p ** 0.5) + 1))]
    smooth = [v for v in range(2, 400_000) if _smooth7(v)]
    ms = list(range(1, 70)) + primes[::8] + [v + 1 for v in smooth[::6]] + [2 ** k for k in range(1, 19)]
    ms += [330750, 330751, 1_000_003, 2_205_000 + 1]        # 60 s and 400 s at 11025 Hz halved; a large prime
    assert len(ms) >= 300
    for m in ms:
        assert F.next_smooth_length(m) == brute(m), m


def test_padded_and_unpadded_grey_agree_when_nothing_is_padded():
    pcm, _ = synth.synth_recording(10.0, seed=3, block=64, return_grey=True)
    for n in (1000, 5000, 66150):                 # halves 500, 2500, 33075 = 3^3 5^2 7^2: npad == n
        assert F.transform_length(n) == n
        a, b = F.grey_stream(pcm[:n]), F.grey_stream(pcm[:n], padded=False)
        assert np.array_equal(a, b)
    # 11027: padded to 2 * 5600.  The transforms differ mostly at the ends, by several grey ranges at the last
    # samples, which is why the restatement must pad as the decoder does
    n = 11027
    assert F.transform_length(n) == 2 * F.next_smooth_length(5514) == 11200
    d = np.abs(F.grey_stream(pcm[:n]) - F.grey_stream(pcm[:n], padded=False))
    assert d[1000:-1000].max() < 1e-3 and d[-10:].max() > 1.0


def test_oracle_rows_use_the_exact_line_length():
    """rows = floor((end - start) / Ls) with the caller's Ls.  Here D / Ls rounds to exactly 65 although 65 * Ls is a
    fraction of an ulp above D: the 65th row ends at image_end and is part of the picture."""
    ls, ppm, D = 55125, 29.304888055303476, 358302
    Ls = 5512.5 / (1.0 + ppm * 1e-6)
    assert D / Ls == 65.0 and Fraction(65) * Fraction(Ls) > D
    g = np.linspace(0.0, 1.0, ls + D + 100)
    img = F.image(g, ls, None, 576, ls + D, line_length=Ls)
    assert img.shape == (65, 1810)
    assert np.array_equal(img, F.image(g, ls, 120, 576, ls + D, line_length=Ls))    # lpm is ignored
