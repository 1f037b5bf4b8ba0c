"""GPU tests of the FM decode stage by stage, each stage on identical input (csrc/fm.cu, api.cu wefax_decode_fm).

The decode is asked for its grey stream; the float64 restatement (oracle/fm_oracle.py) then computes the line start
and the picture from that very grey stream, so every stage is held to what its kernel should compute from its own
input rather than to the end-to-end bars of tests/test_gpu_fm.py:
  * grey, every sample including both ends, against the restatement with the zero-padded transform: within 2e-3 of
    the 0..1 range (B200 measured maxima are recorded as the `grey_max_err` property of each case);
  * line start exactly (both fold in float32 in the same line order; a difference is allowed only on a float64 tie
    within 1e-6 relative, which is asserted);
  * picture at the decoder's line start and exact line length: same shape, every pixel within +-1, >= 99.99 %
    identical (recorded as `pixels_identical`);
  * edges of the search and image windows, the row count at a line length that is not a binary fraction, more than
    65535 rows, device-resident buffers and context reuse, bit for bit where the same kernels run on the same input.
"""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import fm_oracle as F
from oracle import wefax_oracle as O
from wefax_b200 import _native as N
from wefax_b200 import synth

pytestmark = pytest.mark.gpu

SR = 11025
GREY_TOL = 2.5e-4       # B200: 6.2e-5 at most over every case below (n = 100003)
PIX_IDENTICAL = 0.9999


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


@pytest.fixture(scope="module")
def rec60():
    """60 s at 120 LPM: start tone 0-5 s, 30 phasing lines, picture of 64-sample grey blocks, stop tone, black."""
    return synth.synth_recording(60.0, lpm=120, seed=7, block=64)


def _line_length(lpm, ppm=None):
    Ls = 60.0 / lpm * SR
    return Ls if ppm is None else Ls / (1.0 + ppm * 1e-6)      # as wefax_decode_fm_slant computes it


def run(dec, pcm, sr=SR, lpm=120.0, ioc=576, search_from=0, image_end=0, fold_lines=20, taps=63,
        band=(1200.0, 2600.0), black=1500.0, white=2300.0, ppm=None, flags=0, check=True):
    """One decode through the C-ABI with host buffers sized for any row count; returns rc, grey, line start, image."""
    pcm = np.ascontiguousarray(pcm)
    n_in, ch = pcm.shape[0], (1 if pcm.ndim == 1 else pcm.shape[1])
    n = n_in if sr == SR else N.resampled_length(n_in, sr)
    W = int(round(math.pi * ioc))
    cap = (int(n / _line_length(lpm, ppm)) + 2) * W
    grey = np.full(n, np.nan, dtype=np.float32)
    img = np.zeros(cap, dtype=np.uint8)
    rows, w, ls = C.c_int32(-1), C.c_int32(0), C.c_int64(-1)
    desc = N.BatchDesc(1, n_in, ch, int(sr), 0.0, 0.0, int(flags))
    prm = N.FmParams(float(lpm), int(ioc), float(black), float(white), float(band[0]), float(band[1]), int(taps),
                     int(search_from), int(fold_lines), int(image_end))
    out = N.FmOut(grey.ctypes.data, img.ctypes.data, img.size, C.addressof(rows), C.addressof(w), C.addressof(ls))
    if ppm is None:
        rc = dec._lib.wefax_decode_fm(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm), C.byref(out))
    else:
        sp = N.FmSlant(N.FM_SLANT_FIXED, float(ppm), 0.0, 0.0, 0)
        rc = dec._lib.wefax_decode_fm_slant(dec._h, C.byref(desc), C.c_void_p(pcm.ctypes.data), C.byref(prm),
                                            C.byref(sp), C.byref(out), None)
    if check:
        dec._check(rc)
    return dict(rc=rc, grey=grey, line_start=int(ls.value), rows=int(rows.value), width=int(w.value),
                image=img[: max(0, rows.value) * W].reshape(max(0, rows.value), W), n=n)


def ref_input(pcm, sr=SR):
    """The mono 11025 Hz samples the decode band-passes: L+R wrapped in int16 then halved, resampled if need be."""
    x = O.merge_channels(pcm) if pcm.ndim == 2 else pcm.astype(np.float64)
    return x if sr == SR else O.resample(x, O.resampled_length(x.shape[0], sr))


def check_grey(got, z, black=1500.0, white=2300.0, min_rel_mag=None):
    """Every sample within GREY_TOL; with min_rel_mag only where the float64 |z| >= that fraction of its median."""
    ref = F.grey_of(z, black, white)
    assert got.shape == ref.shape and np.isfinite(got).all()
    keep = np.ones(ref.shape, dtype=bool)
    if min_rel_mag is not None:
        mag = np.abs(z)
        keep = mag >= min_rel_mag * np.median(mag)
    err = np.abs(got.astype(np.float64) - ref)[keep]
    assert err.max() < GREY_TOL, (float(err.max()), int(np.argmax(np.abs(got - ref) * keep)))
    return float(err.max())


def check_line_start(res, search_from, fold_lines, line_length, record=None):
    """The decoder's line start is the restatement's on the decoder's grey, or a float64 near-tie with it."""
    frm = min(max(0, search_from), res["n"] - 1)
    scores = F.phasing_scores(res["grey"], frm, None, fold_lines, line_length=line_length)
    ref = frm + int(np.argmax(scores))
    if res["line_start"] != ref:
        best, got = float(scores.max()), float(scores[res["line_start"] - frm])
        assert best - got <= 1e-6 * best, (res["line_start"], ref, got, best)
        if record:
            record("line_start_near_tie", f"{res['line_start']} vs {ref}")
    return ref


def check_image(res, ioc, image_end, line_length, record=None):
    ref = F.image(res["grey"], res["line_start"], None, ioc, image_end, line_length=line_length)
    assert res["image"].shape == ref.shape, (res["image"].shape, ref.shape)
    if ref.size == 0:
        return 1.0
    d = np.abs(res["image"].astype(int) - ref.astype(int))
    same = float((d == 0).mean())
    assert d.max() <= 1 and same >= PIX_IDENTICAL, (int(d.max()), same)
    if record:
        record("pixels_identical", same)
    return same


# ---- grey stream ----------------------------------------------------------------------------------------------------

# npad == n for 64, 100, 1000 and 661500; the others are zero padded (2047 and 2049 straddle the FIR's 2048-sample tile)
GREY_LENGTHS = [64, 65, 100, 1000, 2047, 2049, 5512, 5513, 11025, 100003, 661500]


def test_grey_lengths_cover_padded_and_unpadded_transforms():
    pads = [F.transform_length(n) > n for n in GREY_LENGTHS]
    assert any(pads) and not all(pads)


@pytest.mark.parametrize("n", GREY_LENGTHS)
def test_grey_every_sample_against_the_padded_transform(dec, rec60, n, record_property):
    pcm = rec60[:n] if n == len(rec60) else rec60[20 * SR: 20 * SR + n]      # picture content, or the whole recording
    res = run(dec, pcm)
    err = check_grey(res["grey"], F.analytic(ref_input(pcm)))
    record_property("grey_max_err", err)
    record_property("npad", F.transform_length(n))


@pytest.mark.parametrize("taps", [3, 15, 19, 23, 31, 47, 63, 40])
def test_grey_with_every_fir_build(dec, rec60, taps, record_property):
    """Band-pass lengths that select each KP build of filtfilt_kernel (16, 16, 20, 24, 32, 48, 64; 40 drops to 39: 48)."""
    pcm = rec60[18 * SR: 21 * SR + 17]
    res = run(dec, pcm, taps=taps)
    record_property("grey_max_err", check_grey(res["grey"], F.analytic(ref_input(pcm), taps=taps)))


@pytest.mark.parametrize("band,black,white", [((1000.0, 3000.0), 1500.0, 2300.0), ((1400.0, 2400.0), 1500.0, 2300.0),
                                              ((1200.0, 2600.0), 1700.0, 2100.0)])
def test_grey_other_bands_and_grey_scales(dec, rec60, band, black, white, record_property):
    pcm = rec60[18 * SR: 22 * SR]
    res = run(dec, pcm, band=band, black=black, white=white, taps=47)
    z = F.analytic(ref_input(pcm), band[0], band[1], 47)
    record_property("grey_max_err", check_grey(res["grey"], z, black, white))
    # black above white (an inverted scale) is not a grey scale the decode accepts
    assert run(dec, pcm, band=band, black=white, white=black, check=False)["rc"] == N.ERR_INVALID


def _stereo(mono, wrap):
    if not wrap:
        rng = np.random.default_rng(3)
        other = np.clip(mono.astype(np.int32) + rng.integers(-300, 300, mono.shape[0]), -32768, 32767)
        return np.stack([mono, other.astype(np.int16)], axis=1)
    loud = np.clip(mono.astype(np.int32) * 4, -32768, 32767).astype(np.int16)     # L + R leaves int16 and wraps
    return np.stack([loud, loud], axis=1)


@pytest.mark.parametrize("wrap", [False, True])
def test_grey_of_stereo_input(dec, rec60, wrap, record_property):
    pcm = _stereo(rec60[18 * SR: 22 * SR + 3], wrap)
    s = pcm[:, 0].astype(np.int32) + pcm[:, 1].astype(np.int32)
    assert ((np.abs(s) > 32767).any()) == wrap
    res = run(dec, pcm)
    # a wrapped sum is a square-wave-like signal: compare where the band-pass leaves a carrier
    err = check_grey(res["grey"], F.analytic(ref_input(pcm)), min_rel_mag=0.01 if wrap else None)
    record_property("grey_max_err", err)


@pytest.mark.parametrize("sr", [48000, 44100, 8000])
def test_grey_of_resampled_input(dec, sr, record_property):
    pcm = synth.synth_recording(12.0, sample_rate=sr, lpm=240, seed=5, block=64)
    res = run(dec, pcm, sr=sr, lpm=240)
    assert res["n"] == O.resampled_length(len(pcm), sr)
    record_property("grey_max_err", check_grey(res["grey"], F.analytic(ref_input(pcm, sr))))


def test_grey_of_silence_and_an_out_of_band_tone(dec, rec60, record_property):
    """Silence, a 500 Hz tone the band-pass removes, then the carrier: the grey is compared where there is signal."""
    t = np.arange(SR // 2) / SR
    tone = np.round(8000 * np.sin(2 * np.pi * 500.0 * t)).astype(np.int16)
    pcm = np.concatenate([np.zeros(SR // 2, dtype=np.int16), tone, rec60[20 * SR: 23 * SR]])
    res = run(dec, pcm)
    z = F.analytic(ref_input(pcm))
    record_property("grey_max_err", check_grey(res["grey"], z, min_rel_mag=0.01))


# ---- line start and picture on the decoder's own grey ---------------------------------------------------------------

@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("lpm", [60, 90, 100, 120, 180, 240, 75, 360])
def test_line_start_and_image_on_the_decoders_grey(dec, lpm, noise, record_property):
    pcm = synth.synth_recording(60.0, lpm=lpm, seed=7, block=64, noise_sigma=noise)
    frm, end = 5 * SR, len(pcm) - 15 * SR
    res = run(dec, pcm, lpm=lpm, search_from=frm, image_end=end)
    Ls = _line_length(lpm)
    check_line_start(res, frm, 20, Ls, record_property)
    assert abs(res["line_start"] - frm) <= 3
    assert res["rows"] == math.floor((end - res["line_start"]) / Ls) > 0
    check_image(res, 576, end, Ls, record_property)


@pytest.mark.parametrize("lpm,ppm", [(120, 29.304888055303476), (120, -137.1), (60, 250.123), (240, -0.7)])
def test_fixed_line_length_fold_and_image(dec, lpm, ppm, record_property):
    """FIXED slant: lines of Ls / (1 + ppm 1e-6) samples, not a binary fraction; fold index floor(l * Ls + o)."""
    pcm = synth.synth_recording(60.0, lpm=lpm, seed=8, block=64, noise_sigma=0.02, drift_ppm=ppm)
    frm, end = 5 * SR, len(pcm) - 15 * SR
    res = run(dec, pcm, lpm=lpm, search_from=frm, image_end=end, ppm=ppm)
    Ls = _line_length(lpm, ppm)
    check_line_start(res, frm, 20, Ls, record_property)
    check_image(res, 576, end, Ls, record_property)


@pytest.mark.parametrize("lpm,ioc", [(120, 288), (60, 50), (240, 1000), (90, 576)])
def test_image_geometry(dec, lpm, ioc, record_property):
    """IOC 288; IOC 50 at 60 LPM (a pixel spans 70 samples); IOC 1000 at 240 LPM (a pixel is 0.88 of a sample)."""
    pcm = synth.synth_recording(60.0, lpm=lpm, ioc=ioc, seed=9, block=16, noise_sigma=0.02)
    frm, end = 5 * SR, len(pcm) - 15 * SR
    res = run(dec, pcm, lpm=lpm, ioc=ioc, search_from=frm, image_end=end)
    assert res["width"] == int(round(math.pi * ioc))
    check_line_start(res, frm, 20, _line_length(lpm), record_property)
    check_image(res, ioc, end, _line_length(lpm), record_property)


# ---- edges ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def rec20():
    return synth.synth_recording(20.0, lpm=120, seed=12, block=64)


@pytest.mark.parametrize("search_from", [0, 20 * SR - 1, 20 * SR + 1000])
def test_search_from_at_and_past_the_ends(dec, rec20, search_from):
    n = len(rec20)
    res = run(dec, rec20, search_from=search_from)
    frm = min(search_from, n - 1)
    check_line_start(res, search_from, 20, _line_length(120))
    assert frm <= res["line_start"] < frm + 5513
    assert res["rows"] == max(0, math.floor((n - res["line_start"]) / 5512.5))
    check_image(res, 576, n, 5512.5)


def test_image_end_edges(dec, rec20):
    n, frm = len(rec20), 2 * SR
    full = run(dec, rec20, search_from=frm, image_end=n)
    assert full["rows"] == math.floor((n - full["line_start"]) / 5512.5) > 0
    check_image(full, 576, n, 5512.5)
    for end in (n + 5000, 0, -7):            # past n, and <= 0, mean n
        r = run(dec, rec20, search_from=frm, image_end=end)
        assert r["line_start"] == full["line_start"] and np.array_equal(r["image"], full["image"]), end
    for end in (frm, frm - 100, frm + 100):  # no whole line between search_from and image_end: no picture, no error
        r = run(dec, rec20, search_from=frm, image_end=end)
        assert r["rc"] == N.OK and r["rows"] == 0 and r["line_start"] == full["line_start"], end


def test_fold_window_past_the_end_and_a_recording_shorter_than_a_line(dec, rec20):
    res = run(dec, rec20, search_from=SR, fold_lines=1000)        # 1000 lines folded, 38 left in the recording
    check_line_start(res, SR, 1000, 5512.5)
    check_image(res, 576, len(rec20), 5512.5)
    short = rec20[6 * SR: 6 * SR + 4000]
    res = run(dec, short)
    check_line_start(res, 0, 20, 5512.5)
    assert res["rows"] == 0 and res["image"].size == 0


def test_lpm_below_the_phasing_search_limit_is_unsupported_and_harmless(dec, rec20):
    before = run(dec, rec20, search_from=SR)
    r = run(dec, rec20, lpm=45.0, search_from=SR, check=False)    # a 14700-sample line: 235 KB of prefix sums
    assert r["rc"] == N.ERR_UNSUPPORTED
    after = run(dec, rec20, search_from=SR)
    assert after["line_start"] == before["line_start"] and np.array_equal(after["image"], before["image"])
    assert np.array_equal(after["grey"], before["grey"])


# ---- the row count (every row the caller is told about is written) --------------------------------------------------

def _fma(a: float, b: float, c: float) -> float:
    return float(Fraction(a) * Fraction(b) + Fraction(c))      # one rounding, as a fused multiply-add


def _row_boundary_case(ls: int, k: int, Ls0: float):
    """A FIXED ppm and a span D such that floor(D / Ls) == k while fma(k, Ls, ls) > ls + D: the last of the k rows
    ends a fraction of an ulp past image_end when the product is not rounded on its own."""
    for D in range(round(k * Ls0) - 40, round(k * Ls0) + 40):
        ppm0 = (Ls0 * k / D - 1.0) * 1e6
        ppm = ppm0
        for _ in range(64):
            ppm = float(np.nextafter(ppm, np.inf))
            Ls = Ls0 / (1.0 + ppm * 1e-6)
            if math.floor(D / Ls) == k and _fma(k, Ls, ls) > ls + D:
                return ppm, D
    return None


@pytest.mark.parametrize("device", [False, True])
def test_last_row_at_a_line_length_that_is_not_a_binary_fraction(dec, rec60, device):
    import torch
    k, Ls0, frm = 65, 5512.5, 5 * SR
    first = run(dec, rec60, search_from=frm, ppm=29.3)
    ls = first["line_start"]
    for _ in range(4):                             # the line start may move with the ppm: search again from the new one
        case = _row_boundary_case(ls, k, Ls0)
        assert case is not None
        ppm, D = case
        probe = run(dec, rec60, search_from=frm, ppm=ppm)
        if probe["line_start"] == ls:
            break
        ls = probe["line_start"]
    else:
        pytest.fail("the line start keeps moving with the ppm")
    Ls = Ls0 / (1.0 + ppm * 1e-6)
    assert math.floor(D / Ls) == k and _fma(k, Ls, ls) > ls + D
    end = ls + D
    ref = F.image(probe["grey"], ls, None, 576, end, line_length=Ls)
    assert ref.shape == (k, 1810)
    if not device:
        white = np.round(8000 * np.sin(2 * np.pi * 2300.0 * np.arange(len(rec60)) / SR)).astype(np.int16)
        primed = run(dec, white, search_from=frm)              # leaves rows of 255 in the context's image buffer
        assert primed["rows"] >= k and primed["image"][:k].mean() > 250
        res = run(dec, rec60, search_from=frm, image_end=end, ppm=ppm)
        img, rows = res["image"], res["rows"]
        assert res["line_start"] == ls
    else:
        W, sentinel = 1810, 0x5A
        pcm_d = torch.from_numpy(rec60).cuda()
        img_d = torch.full(((k + 2) * W,), sentinel, dtype=torch.uint8, device="cuda")
        grey_d = torch.empty(len(rec60), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        rows_c, w_c, ls_c = C.c_int32(-1), C.c_int32(0), C.c_int64(-1)
        desc = N.BatchDesc(1, len(rec60), 1, SR, 0.0, 0.0, N.F_PCM_ON_DEVICE | N.F_OUT_ON_DEVICE)
        prm = N.FmParams(120.0, 576, 1500.0, 2300.0, 1200.0, 2600.0, 63, frm, 20, end)
        out = N.FmOut(grey_d.data_ptr(), img_d.data_ptr(), img_d.numel(), C.addressof(rows_c), C.addressof(w_c),
                      C.addressof(ls_c))
        sp = N.FmSlant(N.FM_SLANT_FIXED, ppm, 0.0, 0.0, 0)
        dec._check(dec._lib.wefax_decode_fm_slant(dec._h, C.byref(desc), C.c_void_p(pcm_d.data_ptr()), C.byref(prm),
                                                  C.byref(sp), C.byref(out), None))
        torch.cuda.synchronize()
        rows = rows_c.value
        assert ls_c.value == ls
        full = img_d.cpu().numpy()
        img = full[: rows * W].reshape(rows, W)
        assert (full[rows * W:] == sentinel).all()            # nothing past the rows it reports
    assert rows == k
    d = np.abs(img.astype(int) - ref.astype(int))
    assert d[-1].max() <= 1, (int(d[-1].max()), img[-1, :8], ref[-1, :8])
    assert d.max() <= 1


def test_more_than_65535_rows(dec):
    """lpm = 30000 (22.05-sample lines), IOC 2 (6 pixels), 140 s: about 67 500 rows, past grid.y's 65535."""
    pcm = synth.synth_recording(140.0, lpm=30000, ioc=2, seed=6, block=4, noise_sigma=0.02)
    res = run(dec, pcm, lpm=30000.0, ioc=2, search_from=5 * SR)
    Ls = 60.0 / 30000 * SR
    assert res["rows"] == math.floor((len(pcm) - res["line_start"]) / Ls) > 65535
    check_line_start(res, 5 * SR, 20, Ls)
    check_image(res, 2, len(pcm), Ls)


# ---- device-resident buffers and context reuse ------------------------------------------------------------------------

def test_device_resident_decode_is_the_host_decode(dec, rec60):
    import torch
    frm, end = 5 * SR, len(rec60) - 15 * SR
    host = run(dec, rec60, search_from=frm, image_end=end)
    W, n = 1810, len(rec60)
    pcm_d = torch.from_numpy(rec60).cuda()
    grey_d = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
    img_d = torch.zeros(host["image"].size + 5 * W, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rows, w, ls = C.c_int32(-1), C.c_int32(0), C.c_int64(-1)
    desc = N.BatchDesc(1, n, 1, SR, 0.0, 0.0, N.F_PCM_ON_DEVICE | N.F_OUT_ON_DEVICE)
    prm = N.FmParams(120.0, 576, 1500.0, 2300.0, 1200.0, 2600.0, 63, frm, 20, end)
    out = N.FmOut(grey_d.data_ptr(), img_d.data_ptr(), img_d.numel(), C.addressof(rows), C.addressof(w),
                  C.addressof(ls))
    dec._check(dec._lib.wefax_decode_fm(dec._h, C.byref(desc), C.c_void_p(pcm_d.data_ptr()), C.byref(prm),
                                        C.byref(out)))
    torch.cuda.synchronize()
    assert ls.value == host["line_start"] and rows.value == host["rows"] and w.value == W
    assert np.array_equal(grey_d.cpu().numpy(), host["grey"])
    assert np.array_equal(img_d.cpu().numpy()[: rows.value * W].reshape(rows.value, W), host["image"])
    # float32 samples are a decode_batch input only: the FM decode must not read them as int16
    f32 = (rec60.astype(np.float32) / 32768.0)
    r = run(dec, f32, flags=N.F_PCM_FLOAT32, check=False)
    assert r["rc"] == N.ERR_INVALID


def test_context_reuse_is_bit_identical_to_fresh_contexts(dec, rec60, rec20):
    from wefax_b200.decoder import Decoder
    other = synth.synth_recording(75.0, lpm=120, seed=21, block=64, noise_sigma=0.03)
    jobs = [dict(pcm=rec60, search_from=5 * SR, image_end=45 * SR), dict(pcm=rec20[3 * SR: 3 * SR + 3000]),
            dict(pcm=other, search_from=5 * SR, lpm=90.0, ioc=288), dict(pcm=rec20, search_from=SR, ppm=-40.5)]
    got = []
    for j, job in enumerate(jobs):
        got.append(run(dec, **job))
        if j % 2 == 0:
            dec.decode(rec20, SR, 120, want=("digitalized", "raster"))      # the batch decode reuses the same buffers
    for job, g in zip(jobs, got):
        with Decoder(0) as fresh:
            f = run(fresh, **job)
        assert g["line_start"] == f["line_start"] and g["rows"] == f["rows"]
        assert np.array_equal(g["grey"], f["grey"]) and np.array_equal(g["image"], f["image"])
