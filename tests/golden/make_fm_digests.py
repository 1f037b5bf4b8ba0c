"""sha256 digests of what the FM decode's public entry points return, for a fixed set of recordings.

    python tests/golden/make_fm_digests.py [--out PATH]      (needs a GPU; default PATH: tests/golden/fm_digests.json)

``fm_digests.json`` was written by this script from the build before the chart decode took batches of recordings;
``tests/test_gpu_fm_digests.py`` recomputes the digests with the current build and compares them, so that every
picture, line start, slant report, tone score array and grey stream of ``decode_fm`` (slant off, fixed +40 ppm, auto)
and ``decode_fm_charts`` (slant off, auto) stays bit for bit what it was.  Only the public Python API is called.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from wefax_b200 import synth  # noqa: E402
from wefax_b200.fm import decode_fm, decode_fm_charts  # noqa: E402

FOUR = [(120, 576), (60, 288), (90, 576), (240, 288)]
ODD_HALF_N = 330750      # (n + 1) // 2 = 165375 = 3^3 5^3 7^2: the transform's half length is odd


def _spec(lpm, ioc, block=64):
    return dict(duration_s=20.0 + 60.0 / lpm * 44, lpm=lpm, ioc=ioc, block=block, n_phasing=20)


def recordings():
    """name -> (pcm int16, sample rate)"""
    clean, _ = synth.synth_broadcast([_spec(*c) for c in FOUR], gap_s=3.0, seed=40)
    drift, _ = synth.synth_broadcast([_spec(*c) for c in FOUR], drift_ppm=100.0, gap_s=3.0, seed=42)
    pcm48, _ = synth.synth_broadcast([_spec(120, 576), _spec(240, 288)], sample_rate=48000, gap_s=2.0, seed=7)
    odd = synth.synth_recording(30.0, lpm=240, ioc=288, seed=11, noise_sigma=0.02)
    odd = np.concatenate([odd, np.zeros(max(0, ODD_HALF_N - len(odd)), np.int16)])[:ODD_HALF_N]
    return {"four_clean": (clean, 11025), "four_drift100": (drift, 11025),
            "stereo48k": (np.stack([pcm48, pcm48], axis=1), 48000), "odd_half": (odd, 11025)}


def _h(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _slant(s):
    if s is None:
        return None
    return [repr(float(s.line_length)), repr(float(s.ppm)), repr(float(s.first_line)), int(s.lines_total),
            int(s.lines_used), repr(float(s.residual_rms)), int(s.status)]


def digests(dec) -> dict:
    out = {}
    for name, (pcm, sr) in recordings().items():
        for mode, slant in (("off", None), ("auto", "auto")):
            res = decode_fm_charts(dec, pcm, sr, slant=slant, want_grey=True, want_tone_scores=True)
            out[f"{name}/charts_{mode}"] = {
                "n_found": res.n_found, "grey": _h(res.grey), "tone_scores": _h(res.tone_scores),
                "charts": [{"tone_begin": c.tone_begin, "search_from": c.search_from, "image_end": c.image_end,
                            "stop_found": c.stop_found, "ioc": c.ioc, "lpm": repr(c.lpm),
                            "lpm_score": repr(c.lpm_score), "status": c.status, "width": c.width,
                            "line_start": c.line_start, "shape": None if c.image is None else list(c.image.shape),
                            "image": None if c.image is None else _h(c.image), "slant": _slant(c.slant)}
                           for c in res.charts]}
            if mode == "off":
                charts = res.charts
        for k, c in enumerate(charts):
            for mode, slant in (("off", None), ("fixed40", 40.0), ("auto", "auto")):
                one = decode_fm(dec, pcm, sr, lpm=c.lpm, ioc=c.ioc, search_from=c.search_from, image_end=c.image_end,
                                slant=slant, want_grey=(k == 0))
                out[f"{name}/fm_{k}_{mode}"] = {"line_start": one.line_start, "shape": list(one.image.shape),
                                                "image": _h(one.image), "slant": _slant(one.slant),
                                                "grey": None if one.grey is None else _h(one.grey)}
    return out


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "fm_digests.json"))
    a = ap.parse_args(argv)
    from wefax_b200.decoder import Decoder
    with Decoder(0) as dec:
        d = digests(dec)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(d, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"{a.out}: {len(d)} entries")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
