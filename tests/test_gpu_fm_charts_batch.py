"""GPU tests of the batched chart decode (wefax_decode_fm_charts_batch, DESIGN.md §4.7c).

Every recording's chart list, pictures, line starts, slant reports, tone scores and grey stream must equal, bit for bit,
what decode_fm_charts returns for that recording alone: batches of 1, 2 and 5 mixed broadcasts with slant off and
auto, a noise-only recording in the middle, forced lpm / ioc, 48 kHz stereo, a length whose transform half is odd,
several waves, device PCM with device outputs, max_charts below the charts found and no picture buffer.  A buffer
too small, float32 PCM and bad Python arguments are rejected; the launches of a one-wave batch do not grow with it.
"""
import ctypes as C

import numpy as np
import pytest

from wefax_b200 import _native as N
from wefax_b200 import synth
from wefax_b200.fm import chart_params, decode_fm_charts, decode_fm_charts_batch

pytestmark = pytest.mark.gpu

SR = 11025
T = N.FM_TONE_WINDOW
N_MIXED = 85 * SR


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def _spec(lpm, ioc, block=64):
    return dict(duration_s=20.0 + 60.0 / lpm * 44, lpm=lpm, ioc=ioc, block=block, n_phasing=20)


def _fit(pcm, n):
    return np.concatenate([pcm, np.zeros((max(0, n - len(pcm)),) + pcm.shape[1:], np.int16)])[:n]


def _noise(n, seed, sigma=0.05):
    rng = np.random.default_rng(seed)
    return np.clip(np.round(rng.normal(0.0, sigma, n) * 32767.0), -32768, 32767).astype(np.int16)


@pytest.fixture(scope="module")
def mixed():
    """five recordings of N_MIXED samples: one, one, two and one charts, a noise-only one in the middle"""
    recs = [synth.synth_broadcast([_spec(120, 576)], seed=50)[0],
            synth.synth_broadcast([_spec(60, 288)], drift_ppm=60.0, seed=51)[0],
            _noise(N_MIXED, 52),
            synth.synth_broadcast([_spec(240, 288), _spec(90, 576)], gap_s=2.0, seed=53)[0],
            synth.synth_broadcast([_spec(180, 576)], noise_sigma=0.03, seed=54)[0]]
    return np.stack([_fit(r, N_MIXED) for r in recs])


def _same(batch, single):
    assert batch.n_found == single.n_found and len(batch.charts) == len(single.charts)
    for a, b in zip(batch.charts, single.charts):
        assert (a.tone_begin, a.search_from, a.image_end, a.stop_found, a.ioc, a.lpm, a.lpm_score, a.status, a.width,
                a.line_start) == (b.tone_begin, b.search_from, b.image_end, b.stop_found, b.ioc, b.lpm, b.lpm_score,
                                  b.status, b.width, b.line_start)
        assert a.slant == b.slant
        assert (a.image is None) == (b.image is None)
        if a.image is not None:
            assert a.image.shape == b.image.shape and np.array_equal(a.image, b.image)
    for x, y in ((batch.grey, single.grey), (batch.tone_scores, single.tone_scores)):
        assert (x is None) == (y is None)
        if x is not None:
            assert x.shape == y.shape and np.array_equal(x, y)


def _check(dec, pcm, sr, batch_dec=None, **kw):
    res = decode_fm_charts_batch(batch_dec or dec, pcm, sr, want_grey=True, want_tone_scores=True, **kw)
    assert len(res) == len(pcm)
    for r, one in enumerate(res):
        _same(one, decode_fm_charts(dec, pcm[r], sr, want_grey=True, want_tone_scores=True, **kw))
    return res


@pytest.mark.parametrize("slant", [None, "auto"])
@pytest.mark.parametrize("size", [1, 2, 5])
def test_batch_equals_single(dec, mixed, size, slant):
    res = _check(dec, mixed[:size] if size < 5 else mixed, SR, slant=slant)
    assert [r.n_found for r in res] == [1, 1, 0, 2, 1][:size]
    assert all(c.status == N.FM_CHART_OK and c.image is not None for r in res for c in r.charts)


def test_forced_lpm_and_ioc(dec, mixed):
    _check(dec, mixed, SR, lpm=120, ioc=576)


def test_48k_stereo(dec):
    recs = [synth.synth_broadcast([_spec(120, 576)], sample_rate=48000, seed=60)[0],
            synth.synth_broadcast([_spec(240, 288)], sample_rate=48000, seed=61)[0]]
    n = max(len(r) for r in recs)
    mono = np.stack([_fit(r, n) for r in recs])
    res = _check(dec, np.stack([mono, mono], axis=2), 48000)
    assert [r.n_found for r in res] == [1, 1]


def test_odd_half_length(dec):
    # (n + 1) // 2 = 165375 = 3^3 5^3 7^2: the half-length spectrum has an odd length, its rows an even stride
    n = 330750
    pcm = np.stack([_fit(synth.synth_recording(30.0, lpm=240, ioc=288, seed=s, noise_sigma=0.02), n)
                    for s in (11, 12, 13)])
    res = _check(dec, pcm, SR)
    assert all(r.n_found == 1 for r in res)


def test_several_waves(dec, mixed):
    from wefax_b200.decoder import Decoder
    # about 15 bytes per sample and recording: waves of 2, 2 and 1 recordings; then waves of one
    for limit in (40 * N_MIXED, 1):
        with Decoder(0, workspace_limit=limit) as small:
            _check(dec, mixed, SR, batch_dec=small, slant="auto")


def test_device_pcm_and_device_outputs(dec, mixed):
    import torch
    host = decode_fm_charts_batch(dec, mixed, SR, want_grey=True, want_tone_scores=True)
    R, n = mixed.shape
    nw = n // T
    cap = sum(c.image.size for r in host for c in r.charts) + 4096
    pcm_d = torch.from_numpy(mixed).cuda()
    img_d = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    grey_d = torch.full((R, n), float("nan"), dtype=torch.float32, device="cuda")
    tone_d = torch.full((R, nw, 4), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    out = (N.FmChart * (R * 4))()
    found = (C.c_int * R)()
    desc = N.BatchDesc(R, n, 1, SR, 0.0, 0.0, N.F_PCM_ON_DEVICE | N.F_OUT_ON_DEVICE)
    prm = chart_params()
    dec._check(dec._lib.wefax_decode_fm_charts_batch(dec._h, C.byref(desc), C.c_void_p(pcm_d.data_ptr()),
                                                     C.byref(prm), out, 4, found, img_d.data_ptr(), cap,
                                                     tone_d.data_ptr(), grey_d.data_ptr()))
    torch.cuda.synchronize()
    assert list(found) == [h.n_found for h in host]
    img = img_d.cpu().numpy()
    for r, h in enumerate(host):
        assert np.array_equal(grey_d[r].cpu().numpy(), h.grey)
        assert np.array_equal(tone_d[r].cpu().numpy(), h.tone_scores)
        for c, hc in zip(out[r * 4: r * 4 + found[r]], h.charts):
            assert c.line_start == hc.line_start and c.lpm == hc.lpm
            assert np.array_equal(img[c.image_offset: c.image_offset + c.rows * c.width].reshape(c.rows, c.width),
                                  hc.image)
    # a CUDA tensor through the Python entry point: the same charts and pictures
    dev = decode_fm_charts_batch(dec, pcm_d, SR, want_grey=True, want_tone_scores=True)
    for a, b in zip(dev, host):
        _same(a, b)


def test_max_charts_below_the_charts_found(dec, mixed):
    full = decode_fm_charts_batch(dec, mixed, SR)
    one = decode_fm_charts_batch(dec, mixed, SR, max_charts=1)
    assert [r.n_found for r in one] == [r.n_found for r in full]
    for a, b in zip(one, full):
        assert len(a.charts) == min(1, b.n_found)
        for x, y in zip(a.charts, b.charts):
            assert x.line_start == y.line_start and np.array_equal(x.image, y.image)
    none = decode_fm_charts_batch(dec, mixed, SR, max_charts=0)
    assert [r.n_found for r in none] == [r.n_found for r in full] and all(r.charts == [] for r in none)


def test_no_picture_buffer(dec, mixed):
    res = decode_fm_charts_batch(dec, mixed, SR, want_images=False)
    for r in range(len(mixed)):
        _same(res[r], decode_fm_charts(dec, mixed[r], SR, want_images=False))
    assert all(c.image is None and c.line_start == -1 for r in res for c in r.charts)


def test_a_buffer_too_small_names_the_bytes_needed(dec, mixed):
    full = decode_fm_charts_batch(dec, mixed, SR)
    with pytest.raises(ValueError, match="image_capacity 1000 too small") as e:
        decode_fm_charts_batch(dec, mixed, SR, image_capacity=1000)
    need = int(str(e.value).split("need ")[1].split(")")[0])
    single = 0
    for p in mixed:      # the batch needs what its recordings need alone
        try:
            decode_fm_charts(dec, p, SR, image_capacity=1)
        except ValueError as e1:
            single += int(str(e1).split("need ")[1].split(")")[0])
    assert need == single
    ok = decode_fm_charts_batch(dec, mixed, SR, image_capacity=need)
    for a, b in zip(ok, full):
        _same(a, b)
    with pytest.raises(ValueError, match=f"need {need}"):
        decode_fm_charts_batch(dec, mixed, SR, image_capacity=need - 1)


def test_float32_is_rejected(dec):
    pcm = (synth.synth_recording(20.0, seed=1).astype(np.float32) / 32768.0)[None, :].repeat(2, axis=0)
    out = (N.FmChart * 8)()
    found = (C.c_int * 2)(-1, -1)
    desc = N.BatchDesc(2, pcm.shape[1], 1, SR, 0.0, 0.0, N.F_PCM_FLOAT32)
    prm = chart_params()
    rc = dec._lib.wefax_decode_fm_charts_batch(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm), out,
                                               4, found, None, 0, None, None)
    assert rc == N.ERR_INVALID and list(found) == [-1, -1]


def test_launches_do_not_grow_with_the_batch(dec):
    recs = np.stack([synth.synth_recording(40.0, lpm=120, seed=s) for s in range(8)])
    counts = []
    for size in (1, 8):
        decode_fm_charts_batch(dec, recs[:size], SR)      # (plans and tables of this length are built once)
        before = dec.launch_count
        res = decode_fm_charts_batch(dec, recs[:size], SR)
        counts.append(dec.launch_count - before)
        assert all(r.n_found == 1 and r.charts[0].image is not None for r in res)
    assert counts[0] == counts[1], counts
