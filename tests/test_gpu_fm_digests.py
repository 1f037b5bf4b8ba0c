"""The FM decode's public entry points return, bit for bit, what they returned before the chart decode took batches:
digests of every picture, line start, slant report, tone score array and grey stream of decode_fm (slant off, fixed
+40 ppm, auto) and decode_fm_charts (slant off, auto) against tests/golden/fm_digests.json (written by
tests/golden/make_fm_digests.py from that earlier build)."""
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_fm_outputs_match_the_recorded_digests():
    sys.path.insert(0, GOLDEN)
    try:
        import make_fm_digests
    finally:
        sys.path.remove(GOLDEN)
    from wefax_b200.decoder import Decoder
    with open(os.path.join(GOLDEN, "fm_digests.json")) as f:
        want = json.load(f)
    with Decoder(0) as dec:
        got = make_fm_digests.digests(dec)
    assert sorted(got) == sorted(want)
    bad = [k for k in sorted(want) if got[k] != want[k]]
    assert not bad, {k: (got[k], want[k]) for k in bad[:3]}
