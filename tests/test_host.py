"""CPU-only tests: the C-ABI library loads and exports what include/wefax_b200.h
declares, the host-side helpers agree with the oracle, the Python surface mirrors
the reference's (constructor errors, file_info, config), and nothing silently
falls back to the CPU when no GPU is present."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import wefax_oracle as O
from wefax_b200 import _native as N
from wefax_b200 import synth, wavio
from wefax_b200.config import Config


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "wefax_b200.h")).read()
    declared = set(re.findall(r"\b(wefax_[a-z0-9_]+)\s*\(", header))
    assert declared == set(N.EXPORTED_SYMBOLS), declared ^ set(N.EXPORTED_SYMBOLS)
    lib = N.load()
    for sym in N.EXPORTED_SYMBOLS:
        assert hasattr(lib, sym), sym
    out = subprocess.run(["nm", "-D", "--defined-only", N.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (wefax_[a-z0-9_]+)", out))
    assert set(N.EXPORTED_SYMBOLS) <= exported
    assert lib.wefax_abi_version() == N.ABI_VERSION == 5


def test_struct_layouts_match_header():
    # sizes the C compiler gives the public structs (LP64)
    assert ctypes.sizeof(N.LineConstants) == 48
    assert ctypes.sizeof(N.BatchDesc) == 48
    assert ctypes.sizeof(N.BatchOut) == 13 * 8


@pytest.mark.parametrize("lpm", [60, 90, 100, 120, 180, 240, 30, 45, 75, 110, 150, 200, 288, 360, 480])
def test_line_constants_match_oracle(lpm):
    c, o = N.line_constants(lpm), O.line_constants(lpm)
    for key in ("frame_len", "n1", "n0", "template_len", "mindistance", "width", "dev_min", "dev_max"):
        assert c[key] == o[key], (lpm, key)


def test_resampled_length_matches_oracle():
    rng = np.random.default_rng(0)
    for sr in (8000, 12000, 22050, 44100, 48000, 96000):
        for n in list(rng.integers(1000, 60_000_000, size=40)) + [48000, 960000, 57_600_000]:
            assert N.resampled_length(int(n), sr) == O.resampled_length(int(n), sr)


@pytest.mark.parametrize("f0,q", [(2600, 1), (2600, 2), (1900, 0.7), (3000, 5)])
def test_notch_coefficients_match_oracle(f0, q):
    b, a = N.notch_coefficients(f0, q, 11025)
    bo, ao = O.notch_coefficients(f0, q, 11025)
    assert np.array_equal(b, bo) and np.array_equal(a, ao)


@pytest.mark.parametrize("n", [1, 2, 9, 4096, 11025, 100003, 330750, 275625, 6_615_000, 13_230_000,
                               39_690_000, 57_600_000, 2 * 3 * 5 * 7 * 11 * 13, 13 ** 5, 999_983])
def test_fft_plan_is_a_factorisation(n):
    lens, blu = N.fft_plan_describe(n)
    target = blu if blu else n
    assert int(np.prod(lens, dtype=np.int64)) == target
    if blu:
        assert blu >= 2 * n - 1
    for r in lens[:-1]:
        assert r <= 1024           # strided passes keep >= 8 columns per 8192-element tile
    assert lens[-1] <= 12000         # tile + tables of the stride-1 pass fit 227 KiB of shared memory
    for r in lens:
        m = r
        for p in (2, 3, 5, 7, 11, 13):
            while m % p == 0:
                m //= p
        assert m == 1


def test_no_cpu_fallback_without_gpu():
    lib = N.load()
    if lib.wefax_device_count() > 0:
        pytest.skip("a GPU is present")
    from wefax_b200.decoder import Decoder, WefaxNativeError
    with pytest.raises(WefaxNativeError):
        Decoder(0)


def test_product_never_imports_oracle():
    """The product path may not route through the oracle, scipy.signal or numpy.fft."""
    pkg = os.path.join(ROOT, "wefax_b200")
    banned = (r"^\s*(from|import)\s+oracle", r"^\s*(from|import)\s+scipy", r"\b(np|numpy)\.fft\.\w+\(")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                for pat in banned:
                    assert not re.search(pat, text, flags=re.M), (f, pat)


def test_demodulator_constructor_errors(tmp_path):
    from wefax_b200.wefax import Demodulator
    with pytest.raises(Exception) as e:
        Demodulator(str(tmp_path / "missing.wav"))
    assert str(e.value) == f"INVALID FILE: file at path: {tmp_path / 'missing.wav'} does not exist"
    p = tmp_path / "x.txt"
    p.write_text("hi")
    with pytest.raises(Exception) as e:
        Demodulator(str(p))
    assert str(e.value) == "INVALID FILETYPE: only .wav files are supported at this moment"
    w = tmp_path / "a.wav"
    synth.write_wav(str(w), synth.synth_recording(1.0, seed=1), 11025)
    d = Demodulator(str(w), lines_per_minute=90, quiet=True)
    assert d.filename == "a.wav" and d.websocket_stack == []
    assert d.time_for_one_frame == 1 / (90 / 60)
    d.update_lines_per_minute(240)
    assert d.lines_per_minute == 240 and d.time_for_one_frame == 0.25
    info = d.file_info()
    assert info == {"filename": "a.wav", "channels": 1, "sample_rate": 11025, "length": 1.0}


def test_wav_reader_matches_scipy(tmp_path):
    from scipy.io import wavfile
    rng = np.random.default_rng(2)
    mono = rng.integers(-32768, 32767, size=12345, dtype=np.int16)
    stereo = rng.integers(-32768, 32767, size=(777, 2), dtype=np.int16)
    for name, data, sr in (("m.wav", mono, 11025), ("s.wav", stereo, 48000)):
        p = str(tmp_path / name)
        wavfile.write(p, sr, data)
        sr2, d2 = wavio.read(p)
        assert sr2 == sr and d2.dtype == np.int16 and np.array_equal(d2, data)
        p2 = str(tmp_path / ("w_" + name))
        synth.write_wav(p2, data, sr)
        sr3, d3 = wavfile.read(p2)
        assert sr3 == sr and np.array_equal(d3, data)
    u8 = rng.integers(0, 255, size=999, dtype=np.uint8)
    p = str(tmp_path / "u8.wav")
    wavfile.write(p, 8000, u8)
    sr2, d2 = wavio.read(p)
    assert sr2 == 8000 and d2.dtype == np.uint8 and np.array_equal(d2, u8)
    # every sample format scipy.io.wavfile.read delivers (wefax.py:349 takes them all): same dtype, same values
    for k, data in enumerate((rng.normal(size=100).astype(np.float32), rng.normal(size=(64, 2)).astype(np.float32),
                              rng.normal(size=77), rng.integers(-2 ** 31, 2 ** 31 - 1, size=500, dtype=np.int32),
                              rng.integers(-2 ** 31, 2 ** 31 - 1, size=(33, 2), dtype=np.int32))):
        p = str(tmp_path / f"fmt{k}.wav")
        wavfile.write(p, 8000, data)
        sr2, d2 = wavio.read(p)
        sr3, d3 = wavfile.read(p)
        assert sr2 == sr3 == 8000 and d2.dtype == d3.dtype == data.dtype and np.array_equal(d2, d3)
    for ch in (1, 2):
        p = str(tmp_path / f"pcm24_{ch}.wav")
        v = rng.integers(-2 ** 23, 2 ** 23 - 1, size=(321, ch), dtype=np.int32)
        write_wav_pcm24(p, v, 22050)
        sr2, d2 = wavio.read(p)
        sr3, d3 = wavfile.read(p)
        assert sr2 == sr3 == 22050 and d2.dtype == d3.dtype == np.int32 and np.array_equal(d2, d3)
        assert np.array_equal(d2.reshape(321, ch), v * 256)   # left-justified, as scipy >= 1.6 stores 24-bit data


def write_wav_pcm24(path, values, sample_rate):
    """values: (n, channels) int32 in [-2^23, 2^23)."""
    import struct
    values = np.asarray(values, dtype=np.int32)
    n, ch = values.shape
    raw = (values.astype("<i4").view(np.uint8).reshape(n, ch, 4)[:, :, :3]).tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(raw)) + b"WAVE"
    hdr += b"fmt " + struct.pack("<IHHIIHH", 16, 1, ch, sample_rate, sample_rate * ch * 3, ch * 3, 24)
    hdr += b"data" + struct.pack("<I", len(raw))
    with open(path, "wb") as fh:
        fh.write(hdr + raw)


def test_config_reads_reference_format(tmp_path, monkeypatch):
    cfgdir = tmp_path / "config"
    cfgdir.mkdir()
    (cfgdir / "config.json").write_text(
        '{"host_settings": {"port": 1}, "notch_filter_settings": {"notch_filter_frequency": 2500, '
        '"notch_filter_quality_factor": 2}}')
    monkeypatch.chdir(tmp_path)
    c = Config()
    assert c.settings["notch_filter_settings"] == {"notch_filter_frequency": 2500, "notch_filter_quality_factor": 2}
    monkeypatch.chdir(tmp_path / "config")          # no config/config.json here: package default
    c = Config()
    assert c.settings["notch_filter_settings"]["notch_filter_frequency"] == 2600
    assert c.settings["notch_filter_settings"]["notch_filter_quality_factor"] == 1


def test_synth_is_deterministic():
    a = synth.synth_recording(3.0, seed=5, noise_sigma=0.05)
    b = synth.synth_recording(3.0, seed=5, noise_sigma=0.05)
    assert a.dtype == np.int16 and np.array_equal(a, b) and a.shape == (33075,)
    assert synth.batch_spec(5) == {"lpm": 90, "ioc": 288, "seed": 1005}


def test_parallel_png_writer_roundtrip(tmp_path):
    from PIL import Image
    from wefax_b200 import pngio
    rng = np.random.default_rng(3)
    for shape, band in (((1, 1), 4 << 20), ((37, 53), 64), ((900, 2756), 1 << 16), ((301, 5512), 1 << 18)):
        img = (rng.integers(0, 256, size=shape) // 8 * 8).astype(np.uint8)
        p = str(tmp_path / f"{shape[0]}x{shape[1]}.png")
        pngio.write_png_gray8(p, img, band_bytes=band)
        with Image.open(p) as im:
            assert im.mode == "L" and im.size == (shape[1], shape[0])
            assert np.array_equal(np.asarray(im), img)
    with pytest.raises(ValueError):
        pngio.write_png_gray8(str(tmp_path / "e.png"), np.zeros((0, 5), np.uint8))
    # zlib's adler32_combine identity
    a, b = rng.bytes(100003), rng.bytes(77)
    import zlib
    assert pngio._adler32_combine(zlib.adler32(a), zlib.adler32(b), len(b)) == zlib.adler32(a + b)


def test_fft_plan_prefers_the_specialised_kernels():
    """The half-length transforms of the BASELINE configs run on fft_fast_strided_kernel (strided pass
    lengths = products of two radices from {12, 14, 15, 16} or 15*7) and hilbert_mid_warp_kernel (last pass
    392 / 300 / 210 / 150 / 140): csrc/fft_fast.cuh, csrc/fft_mid.cuh."""
    fast = {a * b for a in (12, 14, 15, 16) for b in (12, 14, 15, 16)} | {105}
    mid = {392, 300, 210, 150, 140}
    for n_half in (39_690_000 // 2, 6_615_000 // 2, 13_230_000 // 2, 9_922_500):
        lens, blu = N.fft_plan_describe(n_half)
        assert not blu
        assert all(r in fast for r in lens[:-1]), lens
        assert lens[-1] in mid, lens
    assert N.fft_plan_describe(39_690_000 // 2)[0] == [225, 225, 392]


def test_decode_short_way_is_keyed_on_everything_the_native_call_reads():
    """Decoder.decode(out=res): the call that made ``res`` left its ctypes arguments behind; they are reused only when
    the input pointer, shape, dtype, settings AND the large output buffers are the ones of that call.  (Host logic only:
    the native entry point is replaced by a recorder that fills the scalar outputs.)"""
    from wefax_b200.decoder import Decoder

    calls = []

    class FakeLib:
        def wefax_decode_batch(self, h, desc_ref, pcm, lpm, out_ref):
            o = out_ref._obj
            n_rec = desc_ref._obj.n_recordings
            start = np.ctypeslib.as_array(ctypes.cast(o.start_frame, ctypes.POINTER(ctypes.c_int64)), shape=(n_rec,))
            start[:] = len(calls) + 1                      # something that changes from call to call
            calls.append((desc_ref._obj, out_ref._obj, pcm.value, o.digitalized))
            return 0

        def wefax_last_error(self, h):
            return b""

    dec = Decoder.__new__(Decoder)
    dec._lib, dec._h, dec.device = FakeLib(), ctypes.c_void_p(0x1234), 0
    pcm = np.zeros(110250, dtype=np.int16)
    res = dec.decode(pcm, 11025, 120, want=("digitalized",))
    assert res._fast is not None and int(res.start_frame[0]) == 1
    again = dec.decode(pcm, 11025, 120, want=("digitalized",), out=res)
    assert again is res and int(res.start_frame[0]) == 2           # same object, scalars updated in place
    assert calls[1][0] is calls[0][0] and calls[1][1] is calls[0][1] and calls[1][2] == pcm.ctypes.data
    # a view of the same memory is the same input
    assert dec.decode(pcm[:], 11025, 120, want=("digitalized",), out=res) is res
    # anything the native call reads differently goes the long way (a new result object)
    for kwargs, arr in (({"lpm": 90}, pcm), ({"lpm": 120, "notch_q": 2}, pcm), ({"lpm": 120}, pcm.copy()),
                        ({"lpm": 120, "want": ("digitalized", "raster")}, pcm), ({"lpm": 120}, pcm[:-2])):
        kw = dict(want=("digitalized",))
        kw.update(kwargs)
        lpm = kw.pop("lpm")
        other = dec.decode(arr, 11025, lpm, out=res if kw["want"] == ("digitalized",) and len(arr) == len(pcm) else None, **kw)
        assert other is not res
    # a replaced output buffer is written, not the one the shortcut remembers
    n_before = len(calls)
    res.digitalized = np.empty_like(res.digitalized)
    newer = dec.decode(pcm, 11025, 120, want=("digitalized",), out=res)
    assert newer is not res and calls[n_before][3] == res.digitalized.ctypes.data
    # a non-contiguous input is copied by the long way, never handed over by pointer
    strided = np.zeros(2 * len(pcm), dtype=np.int16)[::2]
    r2 = dec.decode(strided, 11025, 120, want=("digitalized",))
    r3 = dec.decode(strided, 11025, 120, want=("digitalized",), out=r2)
    assert r3 is not r2
    dec._h = None                                                   # nothing native to destroy
