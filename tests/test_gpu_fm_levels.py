"""GPU tests of the chart decode's tuning-offset correction (wefax_decode_fm_charts_levels, DESIGN.md §4.7d).

  * on the decoder's own grey stream, at each chart's line start and line length (also AUTO slant charts): the black and
    white levels are numpy's lower medians of the same float32 values, the sample counts and the status are the
    restatement's (tests/fm_levels_oracle.py), and the picture is the restatement's picture of grey - float32(delta)
    with the per-pixel bars of tests/test_gpu_fm_stages.py;
  * a broadcast with a different offset per chart at sigma = 0.05: each offset within the CPU bar, each picture as close
    to the transmitted grey as the same chart sent on tune, and with OFF the bias of offset / 800 * 255 levels;
  * OFF through the new entry point is wefax_decode_fm_charts_batch bit for bit, every chart NOT_MEASURED;
  * AUTO: batch equals single bit for bit, levels included (batches of 1, 2 and 5, several waves, device PCM and
    outputs, AUTO slant, max_charts below the charts found, no picture buffer);
  * AUTO costs one launch per wave; a bad mode or max_offset_hz is rejected.
"""
import ctypes as C

import numpy as np
import pytest

import fm_levels_oracle as FL
from oracle import fm_oracle as F
from wefax_b200 import _native as N
from wefax_b200 import synth
from wefax_b200.fm import chart_params, decode_fm_charts, decode_fm_charts_batch, levels_params

pytestmark = pytest.mark.gpu

SR = 11025
N_MIXED = 85 * SR
PIX_IDENTICAL = 0.9999
CPU_BAR_HZ = (2.1, 6.5)          # sigma = 0.05, |offset| <= 50 Hz / up to 150 Hz (tests/test_oracle_fm_levels.py)
# picture error against the transmitted grey, AUTO minus the same chart sent on tune (levels).  B200: 1.03 at -120 Hz,
# where black (1380 Hz) lies in the transition band of the band-pass's 1200 Hz edge and is noisier than on tune
MAE_EXCESS = 1.5
WAVE_LIMITS = (40 * N_MIXED, 1 << 20)   # workspace limits: waves of 2, 2 and 1 recordings; waves of one


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def _spec(lpm, ioc, offset=0.0, block=64):
    return dict(duration_s=20.0 + 60.0 / lpm * 44, lpm=lpm, ioc=ioc, block=block, n_phasing=20,
                carrier_offset_hz=offset)


def _fit(pcm, n):
    return np.concatenate([pcm, np.zeros((max(0, n - len(pcm)),) + pcm.shape[1:], np.int16)])[:n]


def _noise(n, seed, sigma=0.05):
    rng = np.random.default_rng(seed)
    return np.clip(np.round(rng.normal(0.0, sigma, n) * 32767.0), -32768, 32767).astype(np.int16)


@pytest.fixture(scope="module")
def mixed():
    """five recordings of N_MIXED samples, mistuned: one, one, two and one charts, a noise-only one in the middle"""
    recs = [synth.synth_broadcast([_spec(120, 576, 30.0)], seed=50)[0],
            synth.synth_broadcast([_spec(60, 288, -40.0)], drift_ppm=60.0, seed=51)[0],
            _noise(N_MIXED, 52),
            synth.synth_broadcast([_spec(240, 288, 100.0), _spec(90, 576, -20.0)], gap_s=2.0, seed=53)[0],
            synth.synth_broadcast([_spec(180, 576, 0.0)], noise_sigma=0.03, seed=54)[0]]
    return np.stack([_fit(r, N_MIXED) for r in recs])


OFFSETS = (-120.0, 0.0, 45.0, 150.0)
PIECES = ((120, 576), (240, 288), (60, 576), (90, 288))


def _broadcast(offs, sigma=0.05):
    """(pcm, truth, grey) of the four PIECES with the carrier offsets offs"""
    return synth.synth_broadcast([_spec(l, i, o) for (l, i), o in zip(PIECES, offs)], noise_sigma=sigma, gap_s=3.0,
                                 seed=70, return_grey=True)


@pytest.fixture(scope="module")
def offsets_broadcast():
    """the four charts with OFFSETS at sigma = 0.05, and the same broadcast (same noise) sent on tune"""
    return _broadcast(OFFSETS), _broadcast((0.0,) * len(OFFSETS))


def _line_length(c):
    return c.slant.line_length if c.slant is not None else 60.0 / c.lpm * SR


def _same_levels(a, b):
    if a is None or b is None:
        return a is None and b is None
    x = np.array([a.black_hz, a.white_hz, a.offset_hz, a.black_samples, a.white_samples, a.status], np.float64)
    y = np.array([b.black_hz, b.white_hz, b.offset_hz, b.black_samples, b.white_samples, b.status], np.float64)
    return np.array_equal(x, y, equal_nan=True)


def _same(batch, single):
    assert batch.n_found == single.n_found and len(batch.charts) == len(single.charts)
    for a, b in zip(batch.charts, single.charts):
        assert (a.tone_begin, a.search_from, a.image_end, a.ioc, a.lpm, a.status, a.line_start) == \
            (b.tone_begin, b.search_from, b.image_end, b.ioc, b.lpm, b.status, b.line_start)
        assert a.slant == b.slant and _same_levels(a.levels, b.levels)
        assert (a.image is None) == (b.image is None)
        if a.image is not None:
            assert a.image.shape == b.image.shape and np.array_equal(a.image, b.image)
    for x, y in ((batch.grey, single.grey), (batch.tone_scores, single.tone_scores)):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x, y)


def _check(dec, pcm, sr=SR, batch_dec=None, **kw):
    res = decode_fm_charts_batch(batch_dec or dec, pcm, sr, want_grey=True, want_tone_scores=True, levels="auto", **kw)
    for r, one in enumerate(res):
        _same(one, decode_fm_charts(dec, pcm[r], sr, want_grey=True, want_tone_scores=True, levels="auto", **kw))
    return res


def _check_against_the_restatement(res, record=None):
    """Every decoded chart of one FmCharts (want_grey=True, levels="auto") against fm_levels_oracle on its grey."""
    checked = 0
    for c in res.charts:
        if c.image is None:
            assert c.levels is None
            continue
        Ls = _line_length(c)
        m = FL.measure(res.grey, c.line_start, Ls, 20, c.image_end)
        lv = c.levels
        assert (lv.black_samples, lv.white_samples, lv.status) == (m["black_samples"], m["white_samples"], m["status"])
        assert lv.black_hz == m["black_hz"] and lv.white_hz == m["white_hz"] and lv.offset_hz == m["offset_hz"]
        ref = FL.corrected_image(res.grey, c.line_start, Ls, c.ioc, c.image_end,
                                 m["delta"] if m["status"] == FL.OK else 0.0)
        assert c.image.shape == ref.shape
        if ref.size:
            d = np.abs(c.image.astype(int) - ref.astype(int))
            same = float((d == 0).mean())
            assert d.max() <= 1 and same >= PIX_IDENTICAL, (int(d.max()), same)
            if record:
                record(f"pixels_identical_{checked}", same)
        checked += 1
    return checked


@pytest.mark.parametrize("slant", [None, "auto"])
def test_levels_and_picture_on_the_decoders_grey(dec, offsets_broadcast, slant, record_property):
    (pcm, _, _), _ = offsets_broadcast
    res = decode_fm_charts(dec, pcm, SR, slant=slant, levels="auto", want_grey=True)
    assert len(res.charts) == len(OFFSETS)
    if slant == "auto":      # (a chart whose fit is found takes the fitted line start and line length)
        assert any(c.slant.found for c in res.charts)
    assert _check_against_the_restatement(res, record_property) == len(OFFSETS)


def test_mixed_batch_against_the_restatement(dec, mixed):
    for r in decode_fm_charts_batch(dec, mixed, SR, levels="auto", slant="auto", want_grey=True):
        _check_against_the_restatement(r)


def _truth_image(grey_truth, c):
    return F.image(grey_truth, c.line_start, None, c.ioc, c.image_end, line_length=_line_length(c))


def test_per_chart_offsets(dec, offsets_broadcast, record_property):
    (pcm, _, grey_t), (pcm0, _, grey_t0) = offsets_broadcast
    auto = decode_fm_charts(dec, pcm, SR, levels="auto")
    tuned = decode_fm_charts(dec, pcm0, SR, levels="auto")
    assert len(auto.charts) == len(tuned.charts) == len(OFFSETS)
    for k, (a, t, delta) in enumerate(zip(auto.charts, tuned.charts, OFFSETS)):
        assert a.levels.found, a.levels
        err = abs(a.levels.offset_hz - delta)
        assert err <= CPU_BAR_HZ[int(abs(delta) > 50)], (delta, a.levels.offset_hz)
        record_property(f"offset_err_hz_{k}", err)
        ta, tt = _truth_image(grey_t, a), _truth_image(grey_t0, t)
        mae_a = float(np.abs(a.image.astype(float) - ta).mean())
        mae_t = float(np.abs(t.image.astype(float) - tt).mean())
        assert mae_a <= mae_t + MAE_EXCESS, (delta, mae_a, mae_t)
        record_property(f"mae_auto_vs_tuned_{k}", (mae_a, mae_t))


def test_off_shows_the_offset_and_auto_removes_it(dec, record_property):
    """Without noise (which the clip at black and white would bias): OFF pictures are delta / 800 * 255 levels off the
    transmitted grey where no level is clipped, AUTO pictures are not."""
    pcm, _, grey_t = _broadcast(OFFSETS, sigma=0.0)
    off = decode_fm_charts(dec, pcm, SR)
    auto = decode_fm_charts(dec, pcm, SR, levels="auto")
    for k, (o, a, delta) in enumerate(zip(off.charts, auto.charts, OFFSETS)):
        assert o.line_start == a.line_start and a.levels.found
        truth = _truth_image(grey_t, o)
        mid = (truth >= 60) & (truth <= 195)          # no offset up to 150 Hz (48 levels) clips these
        bias_off = float((o.image.astype(float) - truth)[mid].mean())
        bias_auto = float((a.image.astype(float) - truth)[mid].mean())
        assert abs(bias_off - delta / 800.0 * 255.0) <= 1.5, (delta, bias_off)
        assert abs(bias_auto) <= 1.0, (delta, bias_auto)
        record_property(f"bias_off_auto_{k}", (bias_off, bias_auto))


def _raw(dec, pcm, entry, mode=None, max_charts=4, images=True, flags=0, max_offset_hz=0.0):
    """One call of wefax_decode_fm_charts_batch (mode None) or wefax_decode_fm_charts_levels with host buffers."""
    R, n = pcm.shape
    cap = R * 4_000_000 if images else 0
    img = np.zeros(max(1, cap), np.uint8)
    grey = np.zeros((R, n), np.float32)
    tones = np.zeros((R, n // N.FM_TONE_WINDOW, 4), np.float32)
    out = (N.FmChart * (R * max_charts))()
    lev = (N.FmLevelsOut * (R * max_charts))()
    found = (C.c_int * R)()
    desc = N.BatchDesc(R, n, 1, SR, 0.0, 0.0, flags)
    prm = chart_params()
    args = (out, max_charts, found, img.ctypes.data if images else None, cap, tones.ctypes.data, grey.ctypes.data)
    if mode is None:
        rc = dec._lib.wefax_decode_fm_charts_batch(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm),
                                                   *args)
    else:
        lv = N.FmLevels(mode, max_offset_hz)
        rc = dec._lib.wefax_decode_fm_charts_levels(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm),
                                                    C.byref(lv), out, lev, *args[1:])
    return rc, out, lev, list(found), img, tones, grey


def test_off_is_the_batch_entry_point(dec, mixed):
    _, out_b, _, found_b, img_b, tones_b, grey_b = _raw(dec, mixed, "batch")
    rc, out_l, lev, found_l, img_l, tones_l, grey_l = _raw(dec, mixed, "levels", N.FM_LEVELS_OFF)
    assert rc == N.OK and found_l == found_b
    for a, b in zip(out_l, out_b):
        assert [getattr(a, f) for f, _ in N.FmChart._fields_ if f != "slant"] == \
            [getattr(b, f) for f, _ in N.FmChart._fields_ if f != "slant"]
        assert [getattr(a.slant, f) for f, _ in N.FmSlantOut._fields_] == \
            [getattr(b.slant, f) for f, _ in N.FmSlantOut._fields_]
    assert np.array_equal(img_l, img_b) and np.array_equal(tones_l, tones_b) and np.array_equal(grey_l, grey_b)
    for r, k in enumerate(found_l):
        for i in range(min(k, 4)):
            assert lev[r * 4 + i].status == N.FM_LEVELS_NOT_MEASURED
    # and the Python entry points with levels=None report no levels
    assert all(c.levels is None for r in decode_fm_charts_batch(dec, mixed, SR) for c in r.charts)


@pytest.mark.parametrize("slant", [None, "auto"])
@pytest.mark.parametrize("size", [1, 2, 5])
def test_auto_batch_equals_single(dec, mixed, size, slant):
    res = _check(dec, mixed[:size] if size < 5 else mixed, slant=slant)
    assert [r.n_found for r in res] == [1, 1, 0, 2, 1][:size]
    assert all(c.levels is not None and c.levels.found for r in res for c in r.charts)


def test_auto_several_waves(dec, mixed):
    from wefax_b200.decoder import Decoder
    for limit in WAVE_LIMITS:
        with Decoder(0, workspace_limit=limit) as small:
            _check(dec, mixed, batch_dec=small, slant="auto")


def test_auto_device_pcm_and_device_outputs(dec, mixed):
    import torch
    host = decode_fm_charts_batch(dec, mixed, SR, want_grey=True, want_tone_scores=True, levels="auto")
    R, n = mixed.shape
    cap = sum(c.image.size for r in host for c in r.charts) + 4096
    pcm_d = torch.from_numpy(mixed).cuda()
    img_d = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    grey_d = torch.full((R, n), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    out = (N.FmChart * (R * 4))()
    lev = (N.FmLevelsOut * (R * 4))()
    found = (C.c_int * R)()
    desc = N.BatchDesc(R, n, 1, SR, 0.0, 0.0, N.F_PCM_ON_DEVICE | N.F_OUT_ON_DEVICE)
    prm, lv = chart_params(), levels_params("auto")
    dec._check(dec._lib.wefax_decode_fm_charts_levels(dec._h, C.byref(desc), C.c_void_p(pcm_d.data_ptr()),
                                                      C.byref(prm), C.byref(lv), out, lev, 4, found, img_d.data_ptr(),
                                                      cap, None, grey_d.data_ptr()))
    torch.cuda.synchronize()
    assert list(found) == [h.n_found for h in host]
    img = img_d.cpu().numpy()
    for r, h in enumerate(host):
        assert np.array_equal(grey_d[r].cpu().numpy(), h.grey)
        for c, lo, hc in zip(out[r * 4: r * 4 + found[r]], lev[r * 4: r * 4 + found[r]], h.charts):
            assert c.line_start == hc.line_start and lo.status == hc.levels.status
            assert (lo.black_hz, lo.white_hz, lo.offset_hz) == (hc.levels.black_hz, hc.levels.white_hz,
                                                                hc.levels.offset_hz)
            assert np.array_equal(img[c.image_offset: c.image_offset + c.rows * c.width].reshape(c.rows, c.width),
                                  hc.image)
    for a, b in zip(decode_fm_charts_batch(dec, pcm_d, SR, want_grey=True, want_tone_scores=True, levels="auto"), host):
        _same(a, b)


def test_auto_max_charts_and_no_picture_buffer(dec, mixed):
    full = decode_fm_charts_batch(dec, mixed, SR, levels="auto")
    one = decode_fm_charts_batch(dec, mixed, SR, levels="auto", max_charts=1)
    for a, b in zip(one, full):
        assert len(a.charts) == min(1, b.n_found)
        for x, y in zip(a.charts, b.charts):
            assert _same_levels(x.levels, y.levels) and np.array_equal(x.image, y.image)
    rc, out, lev, found, *_ = _raw(dec, mixed, "levels", N.FM_LEVELS_AUTO, images=False)
    assert rc == N.OK and found == [r.n_found for r in full]
    for r, k in enumerate(found):
        for i in range(min(k, 4)):
            assert lev[r * 4 + i].status == N.FM_LEVELS_NOT_MEASURED and out[r * 4 + i].line_start == -1
    res = decode_fm_charts_batch(dec, mixed, SR, levels="auto", want_images=False)
    assert all(c.levels is None for r in res for c in r.charts)


def test_auto_adds_one_launch_per_wave(dec):
    from wefax_b200.decoder import Decoder
    recs = np.stack([synth.synth_recording(40.0, lpm=120, seed=s, carrier_offset_hz=10.0 * s) for s in range(8)])

    def launches(d, pcm, levels):
        decode_fm_charts_batch(d, pcm, SR, levels=levels)
        before = d.launch_count
        res = decode_fm_charts_batch(d, pcm, SR, levels=levels)
        assert all(r.n_found == 1 and r.charts[0].image is not None for r in res)
        return d.launch_count - before

    counts = {size: (launches(dec, recs[:size], None), launches(dec, recs[:size], "auto")) for size in (1, 8)}
    assert counts[1][1] == counts[1][0] + 1 and counts[8][1] == counts[8][0] + 1, counts
    assert counts[1][0] == counts[8][0], counts
    with Decoder(0, workspace_limit=WAVE_LIMITS[1]) as small:     # waves of one recording: one launch more per wave
        off, auto = launches(small, recs[:3], None), launches(small, recs[:3], "auto")
        assert auto == off + 3, (off, auto)


@pytest.mark.parametrize("mode,max_offset_hz", [(2, 0.0), (-1, 0.0), (1, -1.0), (1, 300.5), (1, float("nan")),
                                                (0, 1000.0)])
def test_bad_levels_are_rejected(dec, mode, max_offset_hz):
    pcm = synth.synth_recording(20.0, seed=1)[None, :]
    rc, *_ = _raw(dec, pcm, "levels", mode, max_offset_hz=max_offset_hz)
    assert rc == N.ERR_INVALID
    rc, *_ = _raw(dec, pcm, "levels", N.FM_LEVELS_AUTO, max_offset_hz=0.0)    # 0: the default bound
    assert rc == N.OK
    desc = N.BatchDesc(1, pcm.shape[1], 1, SR, 0.0, 0.0, 0)
    found = (C.c_int * 1)()
    assert dec._lib.wefax_decode_fm_charts_levels(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data),
                                                  C.byref(chart_params()), None, None, None, 0, found, None, 0, None,
                                                  None) == N.ERR_INVALID
