"""GPU parity tests: the CUDA path, called through the C-ABI, against the oracle
(oracle/wefax_oracle.py) on the same inputs and against the golden vectors made
by the unmodified reference (tests/golden).

Tolerances (BASELINE.json north_star):
  * float stages (audio_data, demodulated_data): max|d| / max|ref| <= 1e-4
    (the CUDA path computes in fp32, the reference in float64);
  * detected line starts (peaks / phasing_signals / start_frame): bit-exact
    - always on identical digitalized input (stage test),
    - end to end wherever the fp32 envelope does not flip a grey level that the
      greedy picker is sensitive to (all committed golden cases);
  * output pixels: >= 99.9 % within +-1 grey level end to end, bit-exact on
    identical digitalized input.
"""
import hashlib

import numpy as np
import pytest

from conftest import golden_full_names, load_digests, load_golden_full
from oracle import wefax_oracle as O
from wefax_b200 import synth

pytestmark = pytest.mark.gpu

FLOAT_TOL = 1e-4
PIXEL_FRACTION = 0.999
N_SAME_START_MEASURED = 30   # test_noisy_batch_at_scale: recordings whose start_frame equals the float64 oracle's


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def rel_err(a, ref):
    return float(np.abs(np.asarray(a, dtype=np.float64) - ref).max() / np.abs(ref).max())


def frac_within_one(a, ref):
    d = np.abs(np.asarray(a, dtype=np.int64) - np.asarray(ref, dtype=np.int64))
    return float((d <= 1).mean()), int(d.max(initial=0))


def frac_identical(a, ref):
    return float((np.asarray(a, dtype=np.int64) == np.asarray(ref, dtype=np.int64)).mean())


# Fraction of grey levels that must be BIT-IDENTICAL to the float64 oracle (the fp32 envelope differs from the
# float64 one by ~5e-7 of its peak, so a level flips only where 255*(m-low)/delta sits within ~1e-4 of a rounding
# boundary).  Measured on B200 over every end-to-end case of this file: >= 0.9990 (see MEASURED below); the bound
# asserted leaves a little room for other data.
IDENTICAL_FRACTION = 0.998


def record_measurement(name, value):
    """Measured parity figures go to gpurun_out/parity_measurements.jsonl (scratch; the ones quoted in DESIGN.md
    are copied to profiles/)."""
    import json
    import os
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "parity_measurements.jsonl"), "a") as fh:
            fh.write(json.dumps({"name": name, "value": value}) + "\n")
    except OSError:
        pass


# --------------------------------------------------------------------------- FFT engine
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 8, 11, 13, 16, 60, 105, 256, 1001, 4096, 8192,
                               11025, 2 * 3 * 5 * 7 * 11 * 13, 49 * 225, 65536, 330750, 275625,
                               1000 * 6615 // 5, 2 ** 20, 3 ** 12, 13 ** 5])
def test_fft_matches_numpy(dec, n):
    rng = np.random.default_rng(n)
    batch = 3 if n < 100000 else 1
    x = (rng.normal(size=(batch, n)) + 1j * rng.normal(size=(batch, n))).astype(np.complex64)
    ref = np.fft.fft(x.astype(np.complex128), axis=-1)
    y = dec.fft(x)
    assert np.abs(y - ref).max() / np.abs(ref).max() < 2e-6
    xb = dec.fft(y, inverse=True)
    assert np.abs(xb - x).max() / np.abs(x).max() < 4e-6


@pytest.mark.slow
@pytest.mark.parametrize("n", [6_615_000, 13_230_000])
def test_fft_large(dec, n):
    rng = np.random.default_rng(1)
    x = (rng.normal(size=n) + 1j * rng.normal(size=n)).astype(np.complex64)
    ref = np.fft.fft(x.astype(np.complex128))
    y = dec.fft(x)
    assert np.abs(y - ref).max() / np.abs(ref).max() < 4e-6


# --------------------------------------------------------------------------- single stages
@pytest.mark.parametrize("n", [10, 11, 64, 2047, 2048, 2049, 4095, 11025, 100003, 330750])
def test_filtfilt_stage(dec, n):
    rng = np.random.default_rng(n)
    x = np.round(rng.normal(size=(2, n)) * 6000).astype(np.float32)
    b, a = O.notch_coefficients(2600, 1, 11025)
    ref = np.stack([O.filtfilt(b, a, r.astype(np.float64)) for r in x])
    y = dec.filtfilt(x)
    assert rel_err(y, ref) < 2e-6


def test_filtfilt_other_notch_settings(dec):
    rng = np.random.default_rng(5)
    x = np.round(rng.normal(size=5000) * 6000).astype(np.float32)
    for f0, q in ((2600, 2), (1900, 0.7), (3000, 2.5)):
        b, a = O.notch_coefficients(f0, q, 11025)
        assert rel_err(dec.filtfilt(x, f0, q), O.filtfilt(b, a, x.astype(np.float64))) < 5e-6


def test_filtfilt_high_quality_factors_take_the_recursive_form(dec, tmp_path, monkeypatch):
    """config.json may hold any notch_filter_quality_factor (wefax.py:64): responses too long for the FIR kernels
    (Q = 3 needs 76 taps, Q = 30 needs 773) run scipy's recursion itself, in float64, block-parallel."""
    rng = np.random.default_rng(6)
    for n in (5000, 123457):
        x = np.round(rng.normal(size=n) * 6000).astype(np.float32)
        for f0, q in ((2600, 3), (2600, 30), (1900, 8), (2600, 100)):
            b, a = O.notch_coefficients(f0, q, 11025)
            assert rel_err(dec.filtfilt(x, f0, q), O.filtfilt(b, a, x.astype(np.float64))) < 5e-6, (n, f0, q)
    # the whole decode with the reference's config format carrying Q = 30
    import json
    from wefax_b200.wefax import Demodulator
    pcm = synth.synth_recording(30.0, lpm=120, seed=41, noise_sigma=0.03)
    (tmp_path / "config").mkdir()
    (tmp_path / "config" / "config.json").write_text(json.dumps(
        {"notch_filter_settings": {"notch_filter_frequency": 2600, "notch_filter_quality_factor": 30}}))
    wav = str(tmp_path / "q30.wav")
    synth.write_wav(wav, pcm, 11025)
    monkeypatch.chdir(tmp_path)
    d = Demodulator(wav, lines_per_minute=120, tcp_stream=False, quiet=True)
    try:
        d.process()
    except (ValueError, IndexError):
        pass
    o = O.decode(pcm, 11025, 120, notch_freq=2600, notch_q=30)
    assert rel_err(d.audio_data, o["audio_data"]) < FLOAT_TOL
    assert rel_err(d.demodulated_data, o["demodulated_data"]) < FLOAT_TOL


def test_filtfilt_rejects_short_input(dec):
    with pytest.raises(ValueError, match="greater than padlen"):
        dec.filtfilt(np.zeros(9, dtype=np.float32))


@pytest.mark.parametrize("n", [2, 3, 16, 1000, 11025, 100003, 99991, 330750, 2 ** 17 + 1])
def test_hilbert_envelope_stage(dec, n):
    """abs(hilbert(x)); 100003, 99991 and 2**17+1 have large prime factors (Bluestein)."""
    rng = np.random.default_rng(n)
    t = np.arange(n)
    x = (4000 * np.sin(2 * np.pi * 0.17 * t + 3 * np.sin(2 * np.pi * 0.001 * t)) +
         rng.normal(size=n) * 300).astype(np.float32)
    ref = np.abs(O.hilbert(x.astype(np.float64)))
    y = dec.hilbert_envelope(np.stack([x, x[::-1].copy()]))
    assert rel_err(y[0], ref) < 1e-5
    assert rel_err(y[1], np.abs(O.hilbert(x[::-1].astype(np.float64)))) < 1e-5


@pytest.mark.parametrize("n,num", [(48000, 11025), (48001, 11025), (44100, 11025), (8000, 11025), (8001, 11026),
                                   (12000, 12000), (100003, 22973), (480000, 110250), (22050, 11025), (22051, 11025),
                                   # even -> even with plannable halves: real-input fast path (rfft_gather / irfft_scatter)
                                   (48000, 22050), (22050, 48000), (96000, 11026 * 2), (4_800_000, 1_102_500), (640, 146)])
def test_resample_stage(dec, n, num):
    rng = np.random.default_rng(n + num)
    x = np.round(rng.normal(size=(2, n)) * 5000).astype(np.float32)
    ref = np.stack([O.resample(r.astype(np.float64), num) for r in x])
    y = dec.resample(x, num)
    assert y.shape == ref.shape
    assert rel_err(y, ref) < 1e-5


@pytest.mark.parametrize("n", [5, 6, 100, 1023, 4096, 11025, 330750, 1_000_003])
def test_digitalize_stage_bit_exact(dec, n):
    """median-5, percentiles and rounding on an identical float32 envelope: integers bit-exact."""
    rng = np.random.default_rng(n)
    env = (np.abs(rng.normal(size=(2, n))) * 3000 + 50 * rng.random(size=(2, n))).astype(np.float32)
    env[1, : n // 3] = env[1, 0]          # long runs of duplicates
    dem, dig, lh, st = dec.digitalize(env)
    for r in range(2):
        m = O.medfilt5(env[r].astype(np.float64))
        assert np.array_equal(dem[r].astype(np.float64), m)
        d, low, high = O.digitalize(m)
        assert lh[r, 0] == low and lh[r, 1] == high
        assert st[r] == 0
        assert np.array_equal(dig[r].astype(np.int64), d)


@pytest.mark.parametrize("mode", ["bracket", "radix"])
@pytest.mark.parametrize("kind", ["noise", "ramp", "duplicates", "two_level", "periodic"])
def test_percentile_paths_agree_with_numpy(dec, mode, kind, monkeypatch):
    """Both selection strategies (sample-bracketed single pass with exact fallback, and the
    3-level radix select) must return numpy's percentiles exactly, also on data that defeats
    the systematic sample (monotone ramps, a period equal to the sampling stride)."""
    monkeypatch.setenv("WEFAX_PCT_MODE", mode)
    n = 1_300_007
    rng = np.random.default_rng(7)
    if kind == "noise":
        env = np.abs(rng.normal(size=n)) * 2000
    elif kind == "ramp":
        env = np.linspace(1.0, 9000.0, n)
    elif kind == "duplicates":
        env = rng.integers(0, 40, size=n).astype(np.float64) * 100.0
    elif kind == "two_level":
        env = np.where(rng.random(n) < 0.004, 50.0, 3000.0) + rng.random(n)
    else:
        env = 1000.0 + 900.0 * np.sin(2 * np.pi * np.arange(n) / 127.0) + rng.random(n)
    env = env.astype(np.float32)
    dem, dig, lh, st = dec.digitalize(env[None])
    m = O.medfilt5(env.astype(np.float64))
    d, low, high = O.digitalize(m)
    assert lh[0, 0] == low and lh[0, 1] == high, (mode, kind)
    assert st[0] == 0 and np.array_equal(dig[0].astype(np.int64), d)


def test_digitalize_constant_envelope_flags_nan(dec):
    env = np.full((1, 5000), 7.0, dtype=np.float32)
    _, _, lh, st = dec.digitalize(env)
    assert st[0] == 4 and lh[0, 0] == lh[0, 1]


def _oracle_sync_image(dig, lpm):
    consts = O.line_constants(lpm)
    peaks = O.pattern_search(dig, consts)
    try:
        ph = O.find_phasing(peaks, consts)
    except ValueError as e:
        return peaks, None, None, ("ValueError", str(e))
    sf = ph[-1] if ph else 0
    try:
        img = O.convert_to_image(dig[sf:], consts["width"])
    except IndexError as e:
        return peaks, ph, None, ("IndexError", str(e))
    return peaks, ph, img, None


@pytest.mark.parametrize("name", sorted(load_digests()["cases"]))
def test_sync_and_raster_bit_exact_on_oracle_digitalized(dec, name):
    """Line starts and pixels on the oracle's own digitalized data: bit-exact."""
    c = load_digests()["cases"][name]
    pcm = synth.synth_recording(**c["synth"])
    o = O.decode(pcm, c["synth"].get("sample_rate", 11025), c["lpm"])
    dig = o["digitalized_data"]
    res = dec.sync_raster(dig.astype(np.uint8), c["lpm"])
    assert res.peaks[0] == o["peaks"]
    if o["error"] is None:
        assert res.status[0] == 0
        assert res.phasing_signals[0] == list(o["phasing_signals"])
        assert int(res.start_frame[0]) == o["start_frame"]
        assert np.array_equal(res.image(0), o["output_image"])
    else:
        assert type(res.error(0)).__name__ == o["error"][0] and str(res.error(0)) == o["error"][1]


@pytest.mark.parametrize("lpm", [60, 90, 100, 120, 180, 240, 75, 360])
def test_sync_and_raster_random_digitalized(dec, lpm):
    """Random grey levels with dips every ~line: exercises replacement / opening / grouping."""
    rng = np.random.default_rng(lpm)
    consts = O.line_constants(lpm)
    n = consts["width"] * 130 + 77
    dig = rng.integers(60, 256, size=(3, n)).astype(np.uint8)
    for r in range(3):
        period = consts["width"] + (0.5 if r == 0 else (3 if r == 1 else -7))
        for k in range(int(n / period)):
            s = int(k * period + 100 * r)
            dig[r, s: s + consts["template_len"]] = rng.integers(0, 8 + 40 * r)
    dig[2, : 20 * consts["width"]] = 200      # a long flat start: ties and late first peak
    res = dec.sync_raster(dig, lpm)
    for r in range(3):
        peaks, ph, img, err = _oracle_sync_image(dig[r].astype(np.int64), lpm)
        assert res.peaks[r] == peaks
        if err is None:
            assert res.status[r] == 0 and res.phasing_signals[r] == list(ph)
            assert np.array_equal(res.image(r), img)
        else:
            assert type(res.error(r)).__name__ == err[0]


def test_sync_short_and_degenerate_inputs(dec):
    for n, lpm in ((30, 120), (59, 120), (60, 120), (5000, 120), (5512, 120), (5513, 120), (11100, 120)):
        rng = np.random.default_rng(n)
        dig = rng.integers(0, 256, size=n).astype(np.uint8)
        res = dec.sync_raster(dig, lpm)
        peaks, ph, img, err = _oracle_sync_image(dig.astype(np.int64), lpm)
        assert res.peaks[0] == peaks, n
        if err is None:
            assert res.status[0] == 0 and np.array_equal(res.image(0), img)
        else:
            assert type(res.error(0)).__name__ == err[0], n


# --------------------------------------------------------------------------- whole path vs golden
def _check_end_to_end(res, i, ref, n_ref_image=None):
    """Common end-to-end assertions against a reference-decoder result dict."""
    assert rel_err(res.audio[i], ref["audio_data"]) < FLOAT_TOL
    assert rel_err(res.demodulated[i], ref["demodulated_data"]) < FLOAT_TOL
    frac, worst = frac_within_one(res.digitalized[i], ref["digitalized_data"])
    assert frac >= PIXEL_FRACTION and worst <= 2, (frac, worst)
    same = frac_identical(res.digitalized[i], ref["digitalized_data"])
    record_measurement("grey_levels_identical_to_float64", same)
    assert same >= IDENTICAL_FRACTION, same


@pytest.mark.parametrize("name", golden_full_names())
def test_decode_matches_reference_golden(dec, name):
    g = load_golden_full(name)
    res = dec.decode(g["pcm"], g["sample_rate_in"], g["lpm"],
                     want=("audio", "demodulated", "digitalized", "raster"))
    _check_end_to_end(res, 0, g)
    if g["error"] is None:
        assert res.error(0) is None
        assert res.phasing_signals[0] == [int(v) for v in g["phasing_signals"]]
        assert int(res.start_frame[0]) == g["start_frame"]
        img = res.image(0)
        assert img.shape == g["output_image"].shape
        frac, worst = frac_within_one(img, g["output_image"])
        assert frac >= PIXEL_FRACTION, (frac, worst)
    else:
        err = res.error(0)
        assert [type(err).__name__, str(err)] == list(g["error"])


@pytest.mark.parametrize("name", sorted(load_digests()["cases"]))
def test_decode_matches_oracle_and_digest(dec, name):
    c = load_digests()["cases"][name]
    pcm = synth.synth_recording(**c["synth"])
    assert hashlib.sha256(pcm.tobytes()).hexdigest() == c["pcm_sha256"]
    sr = c["synth"].get("sample_rate", 11025)
    o = O.decode(pcm, sr, c["lpm"])
    res = dec.decode(pcm, sr, c["lpm"], want=("audio", "demodulated", "digitalized", "raster"))
    assert res.n_out == c["n_out"]
    _check_end_to_end(res, 0, o)
    # the float samples stored from the real reference
    idx = np.linspace(0, c["n_out"] - 1, 4096).astype(np.int64)
    assert np.abs(res.audio[0][idx] - np.asarray(c["audio_sample"])).max() / c["audio_absmax"] < FLOAT_TOL
    assert np.abs(res.demodulated[0][idx] - np.asarray(c["demod_sample"])).max() / c["demod_absmax"] < FLOAT_TOL
    if c["error"] is None:
        assert res.error(0) is None
        assert res.phasing_signals[0] == c["phasing_signals"]
        assert int(res.start_frame[0]) == c["start_frame"]
        img = res.image(0)
        assert list(img.shape) == c["image_shape"]
        frac, worst = frac_within_one(img, o["output_image"])
        assert frac >= PIXEL_FRACTION, (frac, worst)


def test_decode_batch_mixed_lpm(dec):
    """A batch of equal-length recordings with different LPM (configs[3] in miniature)."""
    specs = [synth.batch_spec(k, noisy=(k % 2 == 1)) for k in range(8)]
    pcm = np.stack([synth.synth_recording(36.0, **s) for s in specs])
    lpms = [s["lpm"] for s in specs]
    res = dec.decode(pcm, 11025, lpms, want=("audio", "demodulated", "digitalized", "raster"))
    for i, s in enumerate(specs):
        o = O.decode(pcm[i], 11025, s["lpm"])
        _check_end_to_end(res, i, o)
        if o["error"] is None:
            assert res.error(i) is None
            # line starts on the CUDA path's own digitalized data: bit-exact against the oracle picker
            consts = O.line_constants(s["lpm"])
            assert res.peaks[i] == O.pattern_search(res.digitalized[i].astype(np.int64), consts)
            if res.phasing_signals[i] == list(o["phasing_signals"]):
                frac, worst = frac_within_one(res.image(i), o["output_image"])
                assert frac >= PIXEL_FRACTION, (i, frac, worst)
        else:
            assert type(res.error(i)).__name__ == o["error"][0]


def test_decode_device_resident(dec):
    """Inputs and large outputs resident in HBM (torch tensors): same results as host buffers."""
    import torch
    pcm = np.stack([synth.synth_recording(20.0, seed=21 + k, noise_sigma=0.03) for k in range(3)])
    host = dec.decode(pcm, 11025, 120, want=("audio", "demodulated", "digitalized", "raster"))
    dev = dec.decode(torch.from_numpy(pcm).cuda(), 11025, 120,
                     want=("audio", "demodulated", "digitalized", "raster"), device_outputs=True)
    torch.cuda.synchronize()
    assert np.array_equal(dev.digitalized.cpu().numpy(), host.digitalized)
    assert np.array_equal(dev.audio.cpu().numpy(), host.audio)
    assert np.array_equal(dev.start_frame, host.start_frame)
    for i in range(3):
        h, w = int(host.height[i]), host.width[i]
        assert np.array_equal(dev.raster_flat[i, : h * w].cpu().numpy(), host.raster_flat[i][: h * w])


def test_decode_waves_equal_single_wave(dec):
    """A tiny workspace limit forces several waves; results must not change."""
    from wefax_b200.decoder import Decoder
    pcm = np.stack([synth.synth_recording(12.0, seed=40 + k, lpm=240, noise_sigma=0.02) for k in range(5)])
    ref = dec.decode(pcm, 11025, 240)
    small = Decoder(0, workspace_limit=8 << 20)
    try:
        res = small.decode(pcm, 11025, 240)
    finally:
        small.close()
    assert np.array_equal(res.digitalized, ref.digitalized)
    assert np.array_equal(res.start_frame, ref.start_frame) and np.array_equal(res.height, ref.height)
    for i in range(5):
        assert np.array_equal(res.image(i), ref.image(i))


@pytest.mark.parametrize("lanes,lane_wave", [(1, 1), (2, 1), (3, 2), (4, 3)])
def test_decode_lanes_equal_one_wave(dec, monkeypatch, lanes, lane_wave):
    """Depth-first lanes (child contexts on their own streams and host threads, a few recordings at a time)
    produce bit for bit what the whole batch produces in one wave: host and device buffers, mixed LPM."""
    import torch
    from wefax_b200.decoder import Decoder
    specs = [synth.batch_spec(k, noisy=(k % 3 == 0)) for k in range(11)]
    pcm = np.stack([synth.synth_recording(24.0, **s) for s in specs])
    lpms = [s["lpm"] for s in specs]
    want = ("audio", "demodulated", "digitalized", "raster")
    ref = dec.decode(pcm, 11025, lpms, want=want)
    monkeypatch.setenv("WEFAX_DEPTH_FIRST", "1")
    monkeypatch.setenv("WEFAX_LANES", str(lanes))
    monkeypatch.setenv("WEFAX_LANE_WAVE", str(lane_wave))
    laned = Decoder(0)
    try:
        res = laned.decode(pcm, 11025, lpms, want=want)
        dev = laned.decode(torch.from_numpy(pcm).cuda(), 11025, lpms, want=want, device_outputs=True)
        torch.cuda.synchronize()
    finally:
        laned.close()
    assert np.array_equal(res.status, ref.status) and np.array_equal(res.start_frame, ref.start_frame)
    assert res.peaks == ref.peaks and res.phasing_signals == ref.phasing_signals
    assert np.array_equal(res.low_high, ref.low_high)
    for name in ("audio", "demodulated", "digitalized"):
        assert np.array_equal(getattr(res, name), getattr(ref, name)), name
        assert np.array_equal(getattr(dev, name).cpu().numpy(), getattr(ref, name)), name
    for i in range(len(specs)):
        assert np.array_equal(res.image(i), ref.image(i)), i
        h, w = int(ref.height[i]), ref.width[i]
        assert np.array_equal(dev.raster_flat[i, : h * w].cpu().numpy(), ref.raster_flat[i][: h * w]), i


# --------------------------------------------------------------------------- the drop-in class
def test_demodulator_drop_in(dec, tmp_path):
    import json
    from PIL import Image
    from wefax_b200.wefax import Demodulator
    g = load_golden_full("synth_12s_240")
    wav = str(tmp_path / "rec.wav")
    synth.write_wav(wav, g["pcm"], g["sample_rate_in"])
    d = Demodulator(wav, lines_per_minute=240, tcp_stream=True, quiet=True)
    assert d.file_info()["sample_rate"] == 11025
    d.process()
    assert d.sample_rate == 11025 and d.start_frame == g["start_frame"]
    assert d.phasing_signals == [int(v) for v in g["phasing_signals"]]
    assert isinstance(d.output_image, Image.Image) and d.output_image.mode == "L"
    assert d.output_image.size == (g["output_image"].shape[1], g["output_image"].shape[0])
    frac, _ = frac_within_one(np.asarray(d.output_image), g["output_image"])
    assert frac >= PIXEL_FRACTION
    assert rel_err(d.audio_data, g["audio_data"]) < FLOAT_TOL
    assert rel_err(d.demodulated_data, g["demodulated_data"]) < FLOAT_TOL
    titles = [m.get("progress_title", m.get("message_content")) for m in d.websocket_stack]
    ref_titles = json.loads(str(g["progress_titles"]))
    assert [t for i, t in enumerate(titles) if i == 0 or titles[i - 1] != t] == \
           [t for i, t in enumerate(ref_titles) if i == 0 or ref_titles[i - 1] != t]
    assert titles == ref_titles
    assert d.websocket_stack[-1] == {"data_type": "message", "message_content": "convert_end"}
    out = str(tmp_path / "out.png")
    d.save_output_image(out)
    assert np.array_equal(np.asarray(Image.open(out)), np.asarray(d.output_image))


def test_demodulator_reference_errors(dec, tmp_path):
    """The shipped 1-s fixtures make the reference raise ValueError from max([]) (wefax.py:294)."""
    from wefax_b200.wefax import Demodulator
    g = load_golden_full("fixture_start_tone")
    wav = str(tmp_path / "start_tone.wav")
    synth.write_wav(wav, g["pcm"], g["sample_rate_in"])
    d = Demodulator(wav, lines_per_minute=120, tcp_stream=True, quiet=True)
    with pytest.raises(ValueError, match=r"max\(\) iterable argument is empty"):
        d.process()
    assert rel_err(d.audio_data, g["audio_data"]) < FLOAT_TOL
    assert d.digitalized_data.shape[0] == 11025 and d.sample_rate == 11025


def test_demodulator_stereo(dec, tmp_path):
    from wefax_b200.wefax import Demodulator
    g = load_golden_full("synth_stereo_8s_240")
    wav = str(tmp_path / "st.wav")
    synth.write_wav(wav, g["pcm"], g["sample_rate_in"])
    d = Demodulator(wav, lines_per_minute=240, tcp_stream=False, quiet=True)
    assert d.file_info()["channels"] == 2
    d.process()
    assert d.start_frame == g["start_frame"]
    assert rel_err(d.audio_data, g["audio_data"]) < FLOAT_TOL
    frac, _ = frac_within_one(np.asarray(d.output_image), g["output_image"])
    assert frac >= PIXEL_FRACTION
    # with the stream on: the same message sequence as the reference, "merging channels" included
    # (wefax.py:364-370: one message per 1000 frames and one for the last frame)
    import json
    s = Demodulator(wav, lines_per_minute=240, tcp_stream=True, quiet=True)
    s.process()
    titles = [m.get("progress_title", m.get("message_content")) for m in s.websocket_stack]
    assert titles == json.loads(str(g["progress_titles"]))
    parts = g["pcm"].shape[0]
    merging = [m["percentage"] for m in s.websocket_stack if m.get("progress_title") == "merging channels"]
    expect = [(q + 1) / parts * 100 for q in range(parts) if q % 1000 == 0 or q == parts - 1]
    assert merging == expect


# --------------------------------------------------------------------------- full size (BASELINE.json configs[1])
@pytest.mark.slow
def _reference_ingest(data):
    """What wefax.py:348-373 hands to filtfilt for scipy's ``data``: mono as stored, stereo merged frame by frame
    with np.divide(np.add(L, R), 2) in the stored dtype (integer sums wrap)."""
    if data.ndim == 1:
        return np.asarray(data, dtype=np.float64)
    with np.errstate(over="ignore"):
        return np.asarray(np.divide(np.add(data[:, 0], data[:, 1]), 2), dtype=np.float64)


@pytest.mark.parametrize("fmt", ["pcm24", "pcm32", "float32", "float64", "pcm32_stereo", "float32_stereo", "pcm24_stereo"])
def test_demodulator_other_wav_sample_formats(dec, tmp_path, fmt):
    """wefax.py:349 accepts whatever scipy.io.wavfile.read returns: 24 / 32-bit PCM (int32), IEEE float.  The
    drop-in converts them on the host with the reference's arithmetic and feeds float32 to the same kernels."""
    from scipy.io import wavfile
    from test_host import write_wav_pcm24
    from wefax_b200.wefax import Demodulator
    base = synth.synth_recording(30.0, lpm=120, seed=77, noise_sigma=0.04).astype(np.int64)
    other = np.roll(base, 5000) // 3
    wav = str(tmp_path / f"{fmt}.wav")
    stereo = fmt.endswith("_stereo")
    kind = fmt.replace("_stereo", "")
    cols = np.stack([base, other], axis=1) if stereo else base[:, None]
    if kind == "pcm24":
        write_wav_pcm24(wav, (cols * 200).astype(np.int32), 11025)
    elif kind == "pcm32":
        # the second channel is large enough for the stereo sum to wrap around int32
        big = cols.astype(np.int64) * 60000
        wavfile.write(wav, 11025, np.clip(big, -2 ** 31, 2 ** 31 - 1).astype(np.int32).squeeze())
    elif kind == "float32":
        wavfile.write(wav, 11025, (cols / 32768.0).astype(np.float32).squeeze())
    else:
        wavfile.write(wav, 11025, (cols / 32768.0).astype(np.float64).squeeze())
    _, data = wavfile.read(wav)
    x = _reference_ingest(data)
    o = O.decode(x, 11025, 120)
    d = Demodulator(wav, lines_per_minute=120, tcp_stream=False, quiet=True)
    assert d.file_info()["channels"] == (2 if stereo else 1)
    try:
        d.process()
        err = None
    except (ValueError, IndexError) as exc:
        err = [type(exc).__name__, str(exc)]
    assert (err is None) == (o["error"] is None), (err, o["error"])
    assert rel_err(d.audio_data, o["audio_data"]) < FLOAT_TOL
    assert rel_err(d.demodulated_data, o["demodulated_data"]) < FLOAT_TOL
    frac, worst = frac_within_one(d.digitalized_data, o["digitalized_data"])
    assert frac >= PIXEL_FRACTION and worst <= 2, (frac, worst)
    if err is None and list(d.phasing_signals) == list(o["phasing_signals"]):
        frac, _ = frac_within_one(np.asarray(d.output_image), o["output_image"])
        assert frac >= PIXEL_FRACTION


def test_demodulator_concurrent_conversions(dec, tmp_path):
    """main.py:53,294-309 keeps several conversions in flight, one request thread each.  Every thread gets its
    own native context (no process-wide lock): results equal the sequential ones."""
    import threading
    from wefax_b200.wefax import Demodulator
    wavs = []
    for k, lpm in enumerate((120, 240, 120, 60)):
        p = str(tmp_path / f"c{k}.wav")
        synth.write_wav(p, synth.synth_recording(40.0 + k, lpm=lpm, seed=900 + k, noise_sigma=0.03), 11025)
        wavs.append((p, lpm))
    sequential = []
    for p, lpm in wavs:
        d = Demodulator(p, lines_per_minute=lpm, tcp_stream=False, quiet=True)
        d.process()
        sequential.append(d)
    results, errors = [None] * len(wavs), []
    barrier = threading.Barrier(len(wavs))

    def work(i):
        try:
            p, lpm = wavs[i]
            d = Demodulator(p, lines_per_minute=lpm, tcp_stream=True, quiet=True)
            barrier.wait()
            for _ in range(3):
                d.process()
            results[i] = d
        except Exception as exc:   # surfaces in the main thread
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(wavs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for a, b in zip(results, sequential):
        assert a.start_frame == b.start_frame and a.phasing_signals == b.phasing_signals
        assert np.array_equal(a.digitalized_data, b.digitalized_data)
        assert np.array_equal(np.asarray(a.output_image), np.asarray(b.output_image))
        assert a.websocket_stack[-1] == {"data_type": "message", "message_content": "convert_end"}


def test_full_size_60min_stage_properties(dec):
    """The 60-min / 39.69 M-sample recording the benchmark runs.  Every stage is checked
    against the oracle's stage applied to the CUDA path's own upstream output, which is
    size-independent and bit-exact for the integer stages; the fp32 stages are compared with
    the float64 oracle on a 2 M-sample window around the middle and at both ends."""
    lpm = 120
    pcm = synth.synth_recording(3600.0, lpm=lpm, seed=0)
    n = pcm.shape[0]
    res = dec.decode(pcm, 11025, lpm, want=("audio", "demodulated", "digitalized", "raster"))
    assert res.error(0) is None and res.n_out == n == 39_690_000
    audio, dem, dig = res.audio[0], res.demodulated[0], res.digitalized[0]
    # zero-phase notch: FIR of finite support -> windows are independent of the rest
    b, a = O.notch_coefficients(2600, 1, 11025)
    for lo in (0, n // 2 - 1_000_000, n - 2_000_000):
        hi = lo + 2_000_000
        pad_lo, pad_hi = max(lo - 200, 0), min(hi + 200, n)
        ref = O.filtfilt(b, a, pcm[pad_lo:pad_hi].astype(np.float64))[lo - pad_lo: lo - pad_lo + (hi - lo)]
        keep = slice(100 if lo else 0, (hi - lo) - (100 if hi < n else 0))
        assert np.abs(audio[lo:hi][keep] - ref[keep]).max() / np.abs(ref).max() < FLOAT_TOL
    # median-5 of an envelope cannot exceed the analytic-signal magnitude bound, and the envelope of
    # this constant-amplitude FM signal stays near 0.25 FS * notch gain: sanity of the global transform
    assert np.isfinite(dem).all() and dem.min() >= 0
    # percentiles + rounding: exactly numpy on the CUDA path's own median-filtered envelope
    d, low, high = O.digitalize(dem.astype(np.float64))
    assert res.low_high[0, 0] == low and res.low_high[0, 1] == high
    assert np.array_equal(dig, d.astype(np.uint8))
    # order-statistic property of the two percentiles on the full data
    assert (dem < low).sum() <= 0.005 * (n - 1) + 1 <= (dem <= low).sum() + 1
    assert (dem > high).sum() <= 0.005 * (n - 1) + 1 <= (dem >= high).sum() + 1
    # phasing search and raster: exactly the oracle on the CUDA path's own grey levels
    consts = O.line_constants(lpm)
    peaks = O.pattern_search(dig[: 200 * consts["width"]].astype(np.int64), consts)
    assert res.peaks[0] == peaks and len(peaks) == 100
    ph = O.find_phasing(peaks, consts)
    assert res.phasing_signals[0] == list(ph)
    sf = ph[-1] if ph else 0
    assert int(res.start_frame[0]) == sf
    img = res.image(0)
    assert img.shape == (4 * ((n - sf) // consts["width"]), consts["width"])
    for r0 in (0, img.shape[0] // 8 - 101, img.shape[0] // 4 - 300):       # top, middle and bottom bands
        rows = slice(max(r0, 0), min(r0 + 300, img.shape[0] // 4))
        band = dig[sf + rows.start * consts["width"]: sf + rows.stop * consts["width"]].astype(np.int64)
        full_ref = O.convert_to_image(band, consts["width"])
        inner = slice(8 if rows.start else 0, full_ref.shape[0] - (8 if rows.stop < img.shape[0] // 4 else 0))
        assert np.array_equal(img[4 * rows.start: 4 * rows.stop][inner], full_ref[inner])


def test_demodulator_with_a_polling_consumer(dec, tmp_path):
    """What main.py does around the decoder (main.py:63-83, 270-291): one thread runs process()
    and save_output_image(), another pops websocket_stack until it sees convert_end."""
    import threading
    from wefax_b200.wefax import Demodulator
    g = load_golden_full("synth_12s_240")
    wav = str(tmp_path / "upload.wav")
    synth.write_wav(wav, g["pcm"], g["sample_rate_in"])
    d = Demodulator(wav, lines_per_minute=120, tcp_stream=True, quiet=True)     # /load_file
    seen, done = [], threading.Event()

    def poll():
        while not done.is_set():
            if d.websocket_stack:
                msg = d.websocket_stack.pop(0)
                seen.append(msg)
                if msg.get("message_content") == "convert_end":
                    done.set()

    t = threading.Thread(target=poll, daemon=True)
    t.start()
    d.update_lines_per_minute(int("240"))                                          # /convert_file
    d.process()
    d.save_output_image(str(tmp_path / "upload.png"))
    assert done.wait(timeout=30)
    t.join(timeout=5)
    titles = [m.get("progress_title") for m in seen if m["data_type"] == "progress_bar"]
    assert titles[0] == "demodulating signal" and "converting signal to image" in titles
    assert all(0 <= m["percentage"] <= 100 for m in seen if m["data_type"] == "progress_bar")
    assert (tmp_path / "upload.png").stat().st_size > 1000


# --------------------------------------------------------------------------- edge shapes
@pytest.mark.parametrize("n", [10, 11, 58, 59, 60, 100, 2000, 5511, 5512, 5513, 5600])
def test_decode_tiny_recordings_match_oracle(dec, n):
    """Shorter than a line / than the sync template: same outputs and the same exception as the oracle."""
    rng = np.random.default_rng(n)
    pcm = np.round(4000 * np.sin(2 * np.pi * 1900 * np.arange(n) / 11025) + rng.normal(size=n) * 500).astype(np.int16)
    o = O.decode(pcm, 11025, 120)
    res = dec.decode(pcm, 11025, 120, want=("audio", "demodulated", "digitalized", "raster"))
    assert rel_err(res.audio[0], o["audio_data"]) < FLOAT_TOL
    assert rel_err(res.demodulated[0], o["demodulated_data"]) < FLOAT_TOL
    frac, worst = frac_within_one(res.digitalized[0], o["digitalized_data"])
    assert frac >= 0.99 and worst <= 2
    err = res.error(0)
    if o["error"] is None:
        assert err is None and res.image(0).shape == o["output_image"].shape
    else:
        assert err is not None and type(err).__name__ == o["error"][0]


def test_decode_rejects_what_the_reference_rejects(dec):
    with pytest.raises(ValueError, match="greater than padlen"):
        dec.decode(np.zeros(9, dtype=np.int16), 11025, 120)
    with pytest.raises(TypeError):
        dec.decode(np.zeros(100, dtype=np.float64), 11025, 120)
    with pytest.raises(Exception):
        dec.decode(np.zeros(5000, dtype=np.int16), 11025, 0)


def test_decode_batch_odd_length_and_stereo(dec):
    """Odd n takes the full-length complex transform (and LDG tile loads for batch elements that
    are not 16-byte aligned); stereo goes through the wrapping merge."""
    n = 33075                                   # 3 s, odd
    mono = np.stack([synth.synth_recording(3.0, lpm=240, seed=70 + k, noise_sigma=0.03) for k in range(3)])
    res = dec.decode(mono, 11025, 240, want=("audio", "demodulated", "digitalized", "raster"))
    for i in range(3):
        o = O.decode(mono[i], 11025, 240)
        _check_end_to_end(res, i, o)
        assert (res.error(i) is None) == (o["error"] is None)
    left = mono.astype(np.int32) * 3
    stereo = np.stack([left, np.roll(left, 5, axis=1)], axis=2).astype(np.int16)      # sums wrap
    res = dec.decode(stereo, 11025, 240, want=("audio", "demodulated", "digitalized", "raster"))
    for i in range(3):
        o = O.decode(stereo[i], 11025, 240)
        _check_end_to_end(res, i, o)


@pytest.mark.slow
def test_noisy_batch_at_scale(dec):
    """BASELINE.json configs[4] in miniature: 32 noisy recordings (AWGN 0.02-0.1 FS, +-50 Hz carrier
    offset, 5 ppm clock drift), LPM 60/90/120/240.  Phasing search, grouping and raster are checked
    bit for bit against the oracle applied to the CUDA path's own grey levels for every recording;
    the fp32 stages and the end-to-end image against the float64 oracle."""
    specs = [synth.batch_spec(k, noisy=True) for k in range(32)]
    pcm = np.stack([synth.synth_recording(45.0, **s) for s in specs])
    lpms = [s["lpm"] for s in specs]
    res = dec.decode(pcm, 11025, lpms, want=("audio", "demodulated", "digitalized", "raster"))
    n_same_start = 0
    for i, s in enumerate(specs):
        consts = O.line_constants(s["lpm"])
        dig = res.digitalized[i].astype(np.int64)
        peaks, ph, img, err = _oracle_sync_image(dig, s["lpm"])
        assert res.peaks[i] == peaks, i
        if err is None:
            assert res.error(i) is None and res.phasing_signals[i] == list(ph)
            assert np.array_equal(res.image(i), img), i
        else:
            assert type(res.error(i)).__name__ == err[0]
        o = O.decode(pcm[i], 11025, s["lpm"])
        _check_end_to_end(res, i, o)
        if err is None and o["error"] is None and int(res.start_frame[i]) == o["start_frame"]:
            n_same_start += 1
            frac, worst = frac_within_one(res.image(i), o["output_image"])
            assert frac >= PIXEL_FRACTION, (i, frac, worst)
    # the fp32 envelope may flip single grey levels, which the greedy picker can amplify into a
    # different start line on noise; on this set every recording that the reference decodes keeps the
    # reference's start line (measured on B200: N_SAME_START_MEASURED; asserted exactly, so a change is noticed)
    record_measurement("noisy_batch_same_start_of_32", n_same_start)
    assert n_same_start >= N_SAME_START_MEASURED, n_same_start


# --------------------------------------------------------------------------- every specialised kernel instantiation
_FAST_R = sorted({a * b for a in (12, 14, 15, 16) for b in (12, 14, 15, 16)} | {105})
_MID_L = (392, 300, 210, 150, 140)


def _two_pass_cases():
    from wefax_b200 import _native as N
    cases = []
    for R in _FAST_R:
        for L in _MID_L:
            if R * L >= (1 << 16) and N.fft_plan_describe(R * L) == ([R, L], 0):
                cases.append((R, L))
    return cases


@pytest.mark.parametrize("R,L", _two_pass_cases())
def test_hilbert_and_fft_on_every_specialised_kernel(dec, R, L):
    """Half-length plans [R, L] with R on fft_fast_strided_kernel<R1, R2> (both store functors) and L on
    hilbert_mid_warp_kernel<R1, R2>: envelope against numpy's analytic signal, complex DFT against numpy's FFT."""
    m = R * L
    rng = np.random.default_rng(m)
    x = (rng.normal(size=(2, 2 * m)) * 3000).astype(np.float32)
    env = dec.hilbert_envelope(x)
    ref = np.stack([np.abs(O.hilbert(r.astype(np.float64))) for r in x])
    assert rel_err(env, ref) < 1e-5
    c = (rng.normal(size=m) + 1j * rng.normal(size=m)).astype(np.complex64)
    y = dec.fft(c)
    refc = np.fft.fft(c.astype(np.complex128))
    assert np.abs(y - refc).max() / np.abs(refc).max() < 2e-6
    assert np.abs(dec.fft(y, inverse=True) - c).max() / np.abs(c).max() < 4e-6


@pytest.mark.slow
@pytest.mark.parametrize("m,plan", [(5_927_040, [105, 144, 392]), (2_315_250, [105, 105, 210]),
                                    (1_653_750, [105, 105, 150]), (1_543_500, [105, 105, 140])])
def test_hilbert_on_three_pass_plans_of_the_remaining_kernels(dec, m, plan):
    """15x7 and 12x12 strided passes (plain store in the middle pass, envelope store in the last inverse pass)
    and the 210 / 150 / 140-point fused middle kernels."""
    from wefax_b200 import _native as N
    assert N.fft_plan_describe(m)[0] == plan
    rng = np.random.default_rng(m)
    x = (rng.normal(size=2 * m) * 3000).astype(np.float32)
    env = dec.hilbert_envelope(x[None, :])[0]
    ref = np.abs(O.hilbert(x.astype(np.float64)))
    assert rel_err(env, ref) < 1e-5
