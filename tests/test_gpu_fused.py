"""GPU tests of the fused median-5 + grey map + raster sweep (csrc/greyraster.cu).

The fused kernel must reproduce, bit for bit, what the separate grey-map and raster
kernels produce (those are pinned to the oracle / the reference's golden vectors in
test_gpu_parity.py): same `digitalized_data`, same image, for every line width
(aligned or not), any start_frame, any tiling of the lines, recordings that end in one
of the reference's exceptions, and when the sequential phasing scan has to compute grey
levels that do not exist yet.
"""
import numpy as np
import pytest

from oracle import wefax_oracle as O
from wefax_b200 import synth

pytestmark = pytest.mark.gpu

WANT = ("digitalized", "raster")


def _decoder(monkeypatch, **env):
    from wefax_b200.decoder import Decoder
    for k in ("WEFAX_FUSED", "WEFAX_GR_LINES", "WEFAX_SYNC_FORCE_SCAN"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    return Decoder(0)


def _same(a, b, n_rec):
    assert np.array_equal(a.status, b.status)
    assert np.array_equal(a.start_frame, b.start_frame)
    assert np.array_equal(a.height, b.height)
    assert a.peaks == b.peaks and a.phasing_signals == b.phasing_signals
    if a.digitalized is not None and b.digitalized is not None:
        assert np.array_equal(a.digitalized, b.digitalized)
    for i in range(n_rec):
        assert np.array_equal(a.image(i), b.image(i)), i


@pytest.mark.parametrize("lpm", [60, 90, 100, 120, 180, 240])
def test_fused_equals_separate_kernels_every_width(monkeypatch, lpm):
    """Widths 11025 / 7350 / 6615 / 5512 / 3675 / 2756: odd, even, multiples of 4 and of 8."""
    pcm = np.stack([synth.synth_recording(40.0 + 0.013 * k, lpm=lpm, seed=300 + k, noise_sigma=0.02 * (k + 1))[: 440000]
                    for k in range(3)])
    plain = _decoder(monkeypatch, WEFAX_FUSED=0)
    ref = plain.decode(pcm, 11025, lpm, want=WANT)
    plain.close()
    fused = _decoder(monkeypatch)
    res = fused.decode(pcm, 11025, lpm, want=WANT)
    fused.close()
    _same(res, ref, 3)
    assert any(int(h) > 0 for h in res.height)


@pytest.mark.parametrize("lines", [1, 2, 3, 5, 7, 11, 64])
def test_fused_is_independent_of_the_line_tiling(monkeypatch, lines):
    pcm = np.stack([synth.synth_recording(33.0, lpm=l, seed=17 + l, noise_sigma=0.03) for l in (120, 240)])
    lpms = [120, 240]
    plain = _decoder(monkeypatch, WEFAX_FUSED=0)
    ref = plain.decode(pcm, 11025, lpms, want=WANT)
    plain.close()
    fused = _decoder(monkeypatch, WEFAX_GR_LINES=lines)
    res = fused.decode(pcm, 11025, lpms, want=WANT)
    fused.close()
    _same(res, ref, 2)


def test_fused_with_odd_lengths_offsets_and_outputs(monkeypatch):
    """Odd recording lengths (rows of a batch then start at every alignment), raster without digitalized,
    all outputs at once, device-resident outputs."""
    import torch
    base = synth.synth_recording(37.0, lpm=120, seed=5, noise_sigma=0.04)
    for n in (len(base), len(base) - 1, len(base) - 2, len(base) - 3, len(base) - 5):
        pcm = np.stack([base[:n], np.roll(base, 1234)[:n], base[::-1][:n].copy()])
        plain = _decoder(monkeypatch, WEFAX_FUSED=0)
        ref = plain.decode(pcm, 11025, 120, want=("audio", "demodulated", "digitalized", "raster"))
        plain.close()
        fused = _decoder(monkeypatch)
        res = fused.decode(pcm, 11025, 120, want=("audio", "demodulated", "digitalized", "raster"))
        only_raster = fused.decode(pcm, 11025, 120, want=("raster",))
        dev = fused.decode(torch.from_numpy(pcm).cuda(), 11025, 120, want=WANT, device_outputs=True)
        torch.cuda.synchronize()
        _same(res, ref, 3)
        assert np.array_equal(res.demodulated, ref.demodulated)
        assert only_raster.digitalized is None
        for i in range(3):
            assert np.array_equal(only_raster.image(i), ref.image(i))
            h, w = int(ref.height[i]), ref.width[i]
            assert np.array_equal(dev.raster_flat[i, : h * w].cpu().numpy(), ref.raster_flat[i][: h * w])
        assert np.array_equal(dev.digitalized.cpu().numpy(), ref.digitalized)
        fused.close()


def test_fused_when_the_sequential_scan_needs_grey_levels_that_do_not_exist_yet(monkeypatch):
    """WEFAX_SYNC_FORCE_SCAN=1 sends every recording through the sequential picker, which then reads far
    beyond the head the grey-map pre-pass produced: those levels come from the envelope on the fly."""
    pcm = np.stack([synth.synth_recording(130.0, lpm=120, seed=70 + k, noise_sigma=0.05) for k in range(2)])
    plain = _decoder(monkeypatch, WEFAX_FUSED=0)
    ref = plain.decode(pcm, 11025, 120, want=WANT)
    plain.close()
    forced = _decoder(monkeypatch, WEFAX_SYNC_FORCE_SCAN=1)
    res = forced.decode(pcm, 11025, 120, want=WANT)
    forced.close()
    _same(res, ref, 2)
    for i in range(2):
        consts = O.line_constants(120)
        assert res.peaks[i] == O.pattern_search(res.digitalized[i].astype(np.int64), consts)


def test_fused_recordings_without_an_image_still_get_grey_levels(monkeypatch):
    """A recording that ends in the reference's ValueError (wefax.py:294) or IndexError (wefax.py:304) has
    digitalized_data but no image; a constant recording has neither a finite grey map (wefax.py:216)."""
    rng = np.random.default_rng(3)
    clean = synth.synth_recording(30.0, lpm=120, seed=1)                       # clean synthetic: groups == [[]]
    noise = (rng.normal(0, 3000, size=clean.shape)).astype(np.int16)           # no regular peaks at all
    short = synth.synth_recording(30.0, lpm=120, seed=2, noise_sigma=0.02)
    pcm = np.stack([clean, noise, short])
    plain = _decoder(monkeypatch, WEFAX_FUSED=0)
    ref = plain.decode(pcm, 11025, 120, want=WANT)
    plain.close()
    fused = _decoder(monkeypatch)
    res = fused.decode(pcm, 11025, 120, want=WANT)
    _same(res, ref, 3)
    const = np.full((1, 60000), 1000, dtype=np.int16)
    plain = _decoder(monkeypatch, WEFAX_FUSED=0)
    ref_c = plain.decode(const, 11025, 120, want=WANT)
    plain.close()
    res_c = fused.decode(const, 11025, 120, want=WANT)
    fused.close()
    assert np.array_equal(res_c.status, ref_c.status)
    assert np.array_equal(res_c.digitalized, ref_c.digitalized)


def test_fused_matches_the_oracle_end_to_end(monkeypatch):
    """Same bar as test_decode_matches_oracle_and_digest, on a recording whose start_frame is deep inside it."""
    pcm = synth.synth_recording(100.0, lpm=120, seed=11, noise_sigma=0.06)
    o = O.decode(pcm, 11025, 120)
    fused = _decoder(monkeypatch)
    res = fused.decode(pcm, 11025, 120, want=("audio", "demodulated", "digitalized", "raster"))
    fused.close()
    d = np.abs(res.digitalized[0].astype(np.int64) - o["digitalized_data"])
    assert (d <= 1).mean() >= 0.999
    if o["error"] is None and res.phasing_signals[0] == list(o["phasing_signals"]):
        img, ref_img = res.image(0), o["output_image"]
        assert img.shape == ref_img.shape
        assert (np.abs(img.astype(np.int64) - ref_img.astype(np.int64)) <= 1).mean() >= 0.999
    # on the CUDA path's own grey levels the image is Pillow's, bit for bit
    consts = O.line_constants(120)
    if res.error(0) is None:
        ref_img = O.convert_to_image(res.digitalized[0].astype(np.int64)[int(res.start_frame[0]):], consts["width"])
        assert np.array_equal(res.image(0), ref_img)


def test_graph_replay_of_a_repeated_device_resident_decode(monkeypatch):
    """The third identical device-resident call replays a captured CUDA graph (api.cu, wefax_ctx::graph_exec).
    It must see NEW data in the same buffers, survive other calls on the context in between, and equal the eager path."""
    import torch
    a = np.stack([synth.synth_recording(35.0, lpm=120, seed=40 + k, noise_sigma=0.03) for k in range(3)])
    b = np.stack([synth.synth_recording(35.0, lpm=120, seed=50 + k, noise_sigma=0.05) for k in range(3)])
    eager = _decoder(monkeypatch, WEFAX_GRAPH=0)
    ref_a = eager.decode(a, 11025, 120, want=WANT)
    ref_b = eager.decode(b, 11025, 120, want=WANT)
    eager.close()
    dec = _decoder(monkeypatch)
    buf = torch.from_numpy(a).cuda()
    res = dec.decode(buf, 11025, 120, want=WANT, device_outputs=True)
    launches = []
    for step in range(6):
        src = a if step % 2 == 0 else b
        buf.copy_(torch.from_numpy(src))
        torch.cuda.synchronize()
        before = dec.launch_count
        res = dec.decode(buf, 11025, 120, want=WANT, device_outputs=True, out=res)   # (scalars come back in the new object)
        launches.append(dec.launch_count - before)
        torch.cuda.synchronize()
        ref = ref_a if step % 2 == 0 else ref_b
        assert np.array_equal(res.status, ref.status)
        assert np.array_equal(res.start_frame, ref.start_frame)
        assert np.array_equal(res.height, ref.height)
        assert res.peaks == ref.peaks
        assert np.array_equal(res.digitalized.cpu().numpy(), ref.digitalized)
        for i in range(3):
            h, w = int(ref.height[i]), ref.width[i]
            assert np.array_equal(res.raster_flat[i, : h * w].cpu().numpy(), ref.raster_flat[i][: h * w])
        if step == 3:
            # another call on the context (it may move scratch buffers): the graph must not be replayed blindly
            other = dec.decode(b[:1, :200000], 11025, 120, want=WANT)
            assert other.digitalized.shape == (1, 200000)
    assert len(set(launches)) == 1, launches          # a replay reports the launches it stands for
    dec.close()


def test_both_forms_of_the_greedy_picker_agree(monkeypatch):
    """The chain over the settled-bit mask with its two summary levels (default) and the sequential scan
    (WEFAX_SYNC_FORCE_SCAN=1): same peaks on clean recordings (long plateaus of saturated grey), noisy ones, noise
    only, a signal that settles in thousands of tiny runs and a constant signal, and the same as the reference's
    picker (wefax.py:234-259) on the CUDA path's own grey levels."""
    rng = np.random.default_rng(8)
    n = 700000
    recs = [synth.synth_recording(70.0, lpm=120, seed=1)[:n],
            synth.synth_recording(70.0, lpm=120, seed=2, noise_sigma=0.05)[:n],
            synth.synth_recording(70.0, lpm=120, seed=3, noise_sigma=0.4)[:n],
            rng.normal(0, 2500, size=n).astype(np.int16),
            np.where((np.arange(n) // 3) % 2 == 0, 12000, -12000).astype(np.int16),      # many tiny runs
            np.full(n, 900, dtype=np.int16)]
    pcm = np.stack(recs)
    results = []
    for mode in (None, 1):
        env = {} if mode is None else {"WEFAX_SYNC_FORCE_SCAN": mode}
        dec = _decoder(monkeypatch, **env)
        results.append(dec.decode(pcm, 11025, 120, want=WANT))
        dec.close()
    for other in results[1:]:
        _same(results[0], other, len(recs))
    consts = O.line_constants(120)
    res = results[0]
    for i in range(len(recs)):
        if res.status[i] & 4:          # WEFAX_REC_NAN: no finite grey map (constant recording), the picker never ran
            continue
        assert res.peaks[i] == O.pattern_search(res.digitalized[i].astype(np.int64), consts), i


def test_repeated_decode_into_the_same_result_takes_the_short_way_and_stays_right(monkeypatch):
    """``decode(..., out=res)`` with the arguments of the call that made ``res`` skips argument checking and allocation
    (Decoder.decode fast path): same object back, updated in place, equal to a fresh decode; anything different (other
    input buffer, other settings, a replaced output buffer) goes the long way and is right too."""
    import torch
    a = synth.synth_recording(30.0, lpm=120, seed=81, noise_sigma=0.03)
    b = synth.synth_recording(30.0, lpm=120, seed=82, noise_sigma=0.05)
    dec = _decoder(monkeypatch)
    fresh_a = dec.decode(a, 11025, 120, want=WANT)
    fresh_b = dec.decode(b, 11025, 120, want=WANT)
    host = a.copy()
    res = dec.decode(host, 11025, 120, want=WANT)
    for src, ref in ((b, fresh_b), (a, fresh_a), (b, fresh_b)):
        host[...] = src
        again = dec.decode(host, 11025, 120, want=WANT, out=res)
        assert again is res
        _same(res, ref, 1)
    other = dec.decode(b.copy(), 11025, 120, want=WANT, out=res)           # another input buffer: the long way
    _same(other, fresh_b, 1)
    res90 = dec.decode(host, 11025, 90, want=WANT)                         # other settings never reuse the 120-LPM shortcut
    assert res90.width[0] != res.width[0]
    dev = torch.from_numpy(a).cuda()
    dres = dec.decode(dev, 11025, 120, want=WANT, device_outputs=True)
    dres.digitalized = torch.empty_like(dres.digitalized)                   # a replaced buffer must be written, not the old one
    dev.copy_(torch.from_numpy(b))
    dres2 = dec.decode(dev, 11025, 120, want=WANT, device_outputs=True, out=dres)
    torch.cuda.synchronize()
    assert np.array_equal(dres2.digitalized.cpu().numpy(), fresh_b.digitalized)
    dec.close()
