"""GPU tests of the chart finder (wefax_decode_fm_charts, csrc/fm.cu fm_tone_kernel / fm_lpm_kernel, DESIGN.md §4.7b).

  * tone scores against the float64 restatement (tests/fm_charts_oracle.py tone_scores) on the decoder's own grey, within
    1e-4; window classes identical except within 1e-3 of a threshold or of a tie;
  * each candidate's LPM score against lpm_scores on the same grey, within 1e-4, and the same choice;
  * a four-chart broadcast (120/576, 60/288, 90/576, 240/288 with noise gaps) clean, at sigma = 0.05 and at +100 ppm
    with slant="auto": every chart found with its IOC and LPM, spans within one window of the truth, and each picture,
    line start and slant bit for bit what decode_fm returns for that chart's lpm, ioc, search_from and image_end;
    the pictures meet the ground-truth bars of tests/test_gpu_fm.py;
  * 48 kHz stereo input, device PCM and device outputs, max_charts below the charts found, no picture buffer, a
    picture buffer too small, float32 input rejected, and (slow) a 60-minute six-chart broadcast.
"""
import ctypes as C
import math

import numpy as np
import pytest

import fm_charts_oracle as FC
from oracle import fm_oracle as F
from wefax_b200 import _native as N
from wefax_b200 import synth
from wefax_b200.fm import chart_params, decode_fm, decode_fm_charts

pytestmark = pytest.mark.gpu

SR = 11025
T = N.FM_TONE_WINDOW
FOUR = [(120, 576), (60, 288), (90, 576), (240, 288)]


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def _spec(lpm, ioc, block=64):
    return dict(duration_s=20.0 + 60.0 / lpm * 44, lpm=lpm, ioc=ioc, block=block, n_phasing=20)


@pytest.fixture(scope="module")
def four_clean():
    return synth.synth_broadcast([_spec(*c) for c in FOUR], gap_s=3.0, seed=40, return_grey=True)


def _check_found(res, truth):
    assert res.n_found == len(truth) and len(res.charts) == len(truth)
    for c, tr in zip(res.charts, truth):
        assert c.status == N.FM_CHART_OK and c.ioc == tr["ioc"] and c.lpm == tr["lpm"], (c, tr)
        assert abs(c.tone_begin - tr["tone_begin"]) <= T
        assert abs(c.search_from - tr["search_from"]) <= T
        assert abs(c.image_end - tr["stop_begin"]) <= T and c.stop_found
        assert c.width == int(round(math.pi * c.ioc))


def _check_bit_exact(dec, pcm, sr, res, slant=None):
    for c in res.charts:
        one = decode_fm(dec, pcm, sr, lpm=c.lpm, ioc=c.ioc, search_from=c.search_from, image_end=c.image_end,
                        slant=slant)
        assert c.line_start == one.line_start
        assert c.image.shape == one.image.shape and np.array_equal(c.image, one.image)
        assert c.slant == one.slant


def _check_truth(res, truth, tgrey, noisy):
    for c, tr in zip(res.charts, truth):
        assert abs(c.line_start - tr["search_from"]) <= 3
        timg = F.image(tgrey, tr["search_from"], tr["lpm"], tr["ioc"], c.image_end)
        rows = min(timg.shape[0], c.image.shape[0])
        assert rows > 10
        err = np.abs(c.image[:rows].astype(int) - timg[:rows].astype(int))
        assert err.mean() < (14.0 if noisy else 6.0), float(err.mean())
        assert (err <= 16).mean() > (0.75 if noisy else 0.93), float((err <= 16).mean())


def test_tone_scores_and_classes_against_the_restatement(dec, four_clean):
    pcm, truth, _ = four_clean
    res = decode_fm_charts(dec, pcm, SR, want_grey=True, want_tone_scores=True)
    ref = FC.tone_scores(res.grey)
    got = res.tone_scores.astype(np.float64)
    assert got.shape == ref.shape == (len(pcm) // T, 4)
    assert np.abs(got - ref).max() < 1e-4, float(np.abs(got - ref).max())
    cg, cr = FC.tone_classes(got), FC.tone_classes(ref)
    for k in np.nonzero(cg != cr)[0]:
        r = np.sort(ref[k, :3])
        near = abs(r[2] - FC.TONE_MIN_RATIO) < 1e-3 or abs(ref[k, 3] - FC.TONE_MIN_VAR) < 1e-3 or r[2] - r[1] < 1e-3
        assert near, (k, ref[k], got[k])
    # the charts are the restatement's charts of the decoder's own grey
    want = FC.find_charts(cr, len(pcm))
    assert [(c.tone_begin, c.search_from, c.image_end, c.stop_found, c.ioc) for c in res.charts] == \
        [(w["tone_begin"], w["search_from"], w["image_end"], w["stop_found"], w["ioc"]) for w in want]


def test_lpm_scores_against_the_restatement(dec, four_clean):
    pcm, truth, _ = four_clean
    res = decode_fm_charts(dec, pcm, SR, want_grey=True, want_images=False)
    for c in res.charts:
        ref = FC.lpm_scores(res.grey, c.search_from, FC.STANDARD_LPMS)
        lpm, score = FC.best_lpm(ref)
        assert c.lpm == lpm and abs(c.lpm_score - score) < 1e-4
        for cand, r in zip(FC.STANDARD_LPMS, ref):      # each candidate alone: its own score
            one = decode_fm_charts(dec, pcm, SR, lpm_candidates=[cand], want_images=False, max_charts=8)
            got = [o for o in one.charts if o.search_from == c.search_from][0]
            assert abs(got.lpm_score - r) < 1e-4, (cand, got.lpm_score, r)


def test_four_chart_broadcast_clean(dec, four_clean):
    pcm, truth, tgrey = four_clean
    res = decode_fm_charts(dec, pcm, SR)
    _check_found(res, truth)
    _check_bit_exact(dec, pcm, SR, res)
    _check_truth(res, truth, tgrey, noisy=False)


def test_four_chart_broadcast_noisy(dec):
    pcm, truth, tgrey = synth.synth_broadcast([_spec(*c) for c in FOUR], noise_sigma=0.05, gap_s=3.0, seed=41,
                                              return_grey=True)
    res = decode_fm_charts(dec, pcm, SR)
    _check_found(res, truth)
    _check_bit_exact(dec, pcm, SR, res)
    _check_truth(res, truth, tgrey, noisy=True)


def test_four_chart_broadcast_with_drift_and_auto_slant(dec):
    pcm, truth = synth.synth_broadcast([_spec(*c) for c in FOUR], drift_ppm=100.0, gap_s=3.0, seed=42)
    res = decode_fm_charts(dec, pcm, SR, slant="auto")
    _check_found(res, truth)
    _check_bit_exact(dec, pcm, SR, res, slant="auto")
    for c in res.charts:
        assert c.slant.found and abs(c.slant.ppm - 100.0) < 20.0, c.slant


def test_single_ioc288_chart(dec):
    pcm, truth = synth.synth_broadcast([dict(duration_s=60.0, lpm=120, ioc=288, block=64)], seed=3)
    res = decode_fm_charts(dec, pcm, SR)
    assert res.n_found == 1
    c = res.charts[0]
    assert c.ioc == 288 and c.lpm == 120 and c.stop_found
    assert abs(c.search_from - 5 * SR) <= T and abs(c.image_end - 45 * SR) <= T


def test_forced_lpm_and_ioc(dec, four_clean):
    pcm, _, _ = four_clean
    res = decode_fm_charts(dec, pcm, SR, lpm=120, ioc=576, want_images=False)
    assert res.n_found == 4
    assert all(c.lpm == 120 and c.ioc == 576 and c.lpm_score == 0.0 and c.line_start == -1 for c in res.charts)


def test_48k_stereo_input(dec):
    pieces = [_spec(120, 576), _spec(240, 288)]
    pcm48, truth48 = synth.synth_broadcast(pieces, sample_rate=48000, gap_s=2.0, seed=7)
    stereo = np.stack([pcm48, pcm48], axis=1)
    res = decode_fm_charts(dec, stereo, 48000)
    assert res.n_found == 2
    for c, tr in zip(res.charts, truth48):
        assert c.ioc == tr["ioc"] and c.lpm == tr["lpm"] and c.status == N.FM_CHART_OK
        assert abs(c.search_from - tr["search_from"] * SR / 48000) <= T + 1
    _check_bit_exact(dec, stereo, 48000, res)


def test_device_pcm_and_device_outputs(dec, four_clean):
    import torch
    pcm, _, _ = four_clean
    host = decode_fm_charts(dec, pcm, SR, want_grey=True, want_tone_scores=True)
    n, nw = len(pcm), len(pcm) // T
    cap = sum(c.image.size for c in host.charts) + 4 * 1810 * 200
    pcm_d = torch.from_numpy(pcm).cuda()
    img_d = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    grey_d = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
    tone_d = torch.full((nw, 4), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    out = (N.FmChart * 8)()
    found = C.c_int(0)
    desc = N.BatchDesc(1, n, 1, SR, 0.0, 0.0, N.F_PCM_ON_DEVICE | N.F_OUT_ON_DEVICE)
    prm = chart_params()
    dec._check(dec._lib.wefax_decode_fm_charts(dec._h, C.byref(desc), C.c_void_p(pcm_d.data_ptr()), C.byref(prm), out,
                                               8, C.byref(found), img_d.data_ptr(), cap, tone_d.data_ptr(),
                                               grey_d.data_ptr()))
    torch.cuda.synchronize()
    assert found.value == 4
    assert np.array_equal(grey_d.cpu().numpy(), host.grey)
    assert np.array_equal(tone_d.cpu().numpy(), host.tone_scores)
    img = img_d.cpu().numpy()
    for c, h in zip(out[:4], host.charts):
        assert c.line_start == h.line_start and c.lpm == h.lpm
        assert np.array_equal(img[c.image_offset: c.image_offset + c.rows * c.width].reshape(c.rows, c.width), h.image)


def test_max_charts_below_the_charts_found(dec, four_clean):
    pcm, _, _ = four_clean
    full = decode_fm_charts(dec, pcm, SR)
    two = decode_fm_charts(dec, pcm, SR, max_charts=2)
    assert two.n_found == 4 and len(two.charts) == 2
    for a, b in zip(two.charts, full.charts):
        assert (a.tone_begin, a.search_from, a.image_end, a.ioc, a.lpm, a.lpm_score, a.line_start) == \
            (b.tone_begin, b.search_from, b.image_end, b.ioc, b.lpm, b.lpm_score, b.line_start)
        assert np.array_equal(a.image, b.image)
    none = decode_fm_charts(dec, pcm, SR, max_charts=0)
    assert none.n_found == 4 and none.charts == []


def test_no_picture_buffer_and_a_buffer_too_small(dec, four_clean):
    pcm, _, _ = four_clean
    full = decode_fm_charts(dec, pcm, SR)
    lst = decode_fm_charts(dec, pcm, SR, want_images=False)
    assert [(c.tone_begin, c.search_from, c.image_end, c.ioc, c.lpm, c.lpm_score) for c in lst.charts] == \
        [(c.tone_begin, c.search_from, c.image_end, c.ioc, c.lpm, c.lpm_score) for c in full.charts]
    assert all(c.image is None and c.line_start == -1 for c in lst.charts)
    with pytest.raises(ValueError, match="image_capacity 1000 too small"):
        decode_fm_charts(dec, pcm, SR, image_capacity=1000)
    # the library names the bytes it needs; that many is enough
    try:
        decode_fm_charts(dec, pcm, SR, image_capacity=1000)
    except ValueError as e:
        bytes_needed = int(str(e).split("need ")[1].split(")")[0])
    ok = decode_fm_charts(dec, pcm, SR, image_capacity=bytes_needed)
    assert all(np.array_equal(a.image, b.image) for a, b in zip(ok.charts, full.charts))
    with pytest.raises(ValueError):
        decode_fm_charts(dec, pcm, SR, image_capacity=bytes_needed - 1)


def test_float32_input_is_rejected(dec):
    pcm = synth.synth_recording(20.0, seed=1).astype(np.float32) / 32768.0
    out = (N.FmChart * 4)()
    found = C.c_int(-1)
    desc = N.BatchDesc(1, len(pcm), 1, SR, 0.0, 0.0, N.F_PCM_FLOAT32)
    prm = chart_params()
    rc = dec._lib.wefax_decode_fm_charts(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm), out, 4,
                                         C.byref(found), None, 0, None, None)
    assert rc == N.ERR_INVALID and found.value == -1


def test_bad_arguments_are_rejected_before_the_call(dec):
    pcm = synth.synth_recording(20.0, seed=1)
    for bad in (dict(lpm_candidates=[30.0]), dict(lpm_candidates=[60.0] * 9), dict(lpm=0), dict(ioc=-1),
                dict(slant="x"), dict(max_charts=-1)):
        with pytest.raises(ValueError):
            decode_fm_charts(dec, pcm, SR, **bad)


@pytest.mark.slow
def test_sixty_minute_six_chart_broadcast(dec):
    from tools.fm_charts_bench import SIX, six_chart_broadcast
    pcm, truth = six_chart_broadcast()
    assert len(pcm) >= 59 * 60 * SR
    res = decode_fm_charts(dec, pcm, SR, slant="auto")
    assert res.n_found == len(SIX)
    for c, tr in zip(res.charts, truth):
        assert c.ioc == tr["ioc"] and c.lpm == tr["lpm"] and c.status == N.FM_CHART_OK
        assert abs(c.search_from - tr["search_from"]) <= T and abs(c.image_end - tr["stop_begin"]) <= T
        assert c.slant.found
    _check_bit_exact(dec, pcm, SR, res, slant="auto")
