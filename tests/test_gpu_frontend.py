"""The input and envelope front end the C-ABI entry points share: one PCM upload (which rejects float32 samples where
an entry point reads int16 only) and one choice of transform form for |hilbert(x)|, used by the decode and by the
stage entry point wefax_hilbert_envelope alike."""
import ctypes as C

import numpy as np
import pytest

from oracle import wefax_oracle as O
from wefax_b200 import _native as N
from wefax_b200 import synth

pytestmark = pytest.mark.gpu

SR = N.TARGET_RATE


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    yield d
    d.close()


def last_error(dec):
    return dec._lib.wefax_last_error(dec._h).decode()


def test_int16_entry_points_reject_float32_samples(dec):
    """Float32 samples are wefax_decode_batch input only; the other entry points that read PCM must not take them
    for int16."""
    pcm = (synth.synth_recording(4.0, lpm=120, seed=3) / 32768.0).astype(np.float32)
    n = pcm.shape[0]
    ptr = C.c_void_p(pcm.ctypes.data)
    desc = N.BatchDesc(1, n, 1, SR, 2600.0, 1.0, N.F_PCM_FLOAT32)
    rc = dec._lib.wefax_segment_envelope(dec._h, C.byref(desc), ptr, 0, 0, 0, n)
    assert rc == N.ERR_INVALID and "int16 samples only" in last_error(dec)
    ts = N.ToneSettings(250.0, 380.0, 0.05, 0.2, 800.0, 3200.0, 4, 6)
    rc = dec._lib.wefax_tone_scan(dec._h, ptr, n, 1, SR, SR, N.F_PCM_FLOAT32, C.byref(ts), None, None, None, None)
    assert rc == N.ERR_INVALID and "int16 samples only" in last_error(dec)
    ps = N.SyncPulseSettings(0.5, 0.2, 1400.0, 1600.0, 2600.0, 1.0)
    rc = dec._lib.wefax_sync_pulse_scan(dec._h, ptr, n, 1, SR, SR, N.F_PCM_FLOAT32, C.byref(ps), None, None, None,
                                        None, None, None, None)
    assert rc == N.ERR_INVALID and "int16 samples only" in last_error(dec)
    prm = N.FmParams(120.0, 576, 1500.0, 2300.0, 1200.0, 2600.0, 63, 0, 20, 0)
    out = N.FmOut(None, None, 0, None, None, None)
    rc = dec._lib.wefax_decode_fm(dec._h, C.byref(desc), ptr, C.byref(prm), C.byref(out))
    assert rc == N.ERR_INVALID and "int16 samples only" in last_error(dec)
    # the context is still usable afterwards
    assert dec.segment_envelope((pcm * 32768.0).astype(np.int16), SR, 0, n) == n


@pytest.mark.parametrize("n,passes,bluestein", [(88200, [225, 196], 0),       # even, half plannable: real-input form
                                                (99225, [225, 441], 0),       # odd, plannable: complex form
                                                (100003, [224, 896], 200704)])   # prime: Bluestein
def test_stage_envelope_is_the_decode_envelope(dec, n, passes, bluestein):
    """demodulated_data of the decode is, bit for bit, the median-5 of wefax_hilbert_envelope applied to the decode's
    own audio_data: the stage entry point runs the decode's envelope for every transform form."""
    p, r, b = C.c_int(), (C.c_int * 8)(), C.c_longlong()
    assert dec._lib.wefax_fft_plan_describe(n // 2 if n % 2 == 0 else n, C.byref(p), r, C.byref(b)) == N.OK
    assert list(r)[: p.value] == passes and b.value == bluestein
    pcm = np.stack([synth.synth_recording(10.0, lpm=120, seed=s, noise_sigma=0.03)[:n] for s in (5, 6)])
    res = dec.decode(pcm, SR, 120, want=("audio", "demodulated"))
    env = dec.hilbert_envelope(res.audio)
    for i in range(2):
        med = O.medfilt5(env[i]).astype(np.float32)
        assert np.array_equal(res.demodulated[i], med), (i, int(np.count_nonzero(res.demodulated[i] != med)))
