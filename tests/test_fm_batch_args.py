"""decode_fm_charts_batch refuses bad arguments before it reaches the native library (no decoder is needed for that)."""
import numpy as np
import pytest

from wefax_b200.fm import decode_fm_charts_batch


@pytest.mark.parametrize("bad", [dict(lpm_candidates=[30.0]), dict(lpm_candidates=[60.0] * 9), dict(lpm=0),
                                 dict(ioc=-1), dict(slant="x"), dict(max_charts=-1), dict(max_charts=1.5)])
def test_bad_keywords(bad):
    with pytest.raises(ValueError):
        decode_fm_charts_batch(None, np.zeros((2, 4096), np.int16), 11025, **bad)


@pytest.mark.parametrize("shape", [(4096,), (2, 4096, 3), (0, 4096), (2, 0), (1, 2, 2, 2)])
def test_bad_shapes(shape):
    with pytest.raises(ValueError):
        decode_fm_charts_batch(None, np.zeros(shape, np.int16), 11025)


@pytest.mark.parametrize("rate", [0, -1, 11025.5, True])
def test_bad_sample_rate(rate):
    with pytest.raises(ValueError):
        decode_fm_charts_batch(None, np.zeros((2, 4096), np.int16), rate)
