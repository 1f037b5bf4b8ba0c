"""Device time of the FM decode's slant correction and its estimate, on a B200-sized input.

Input: a 60-minute 120 LPM synthetic recording with +5 ppm of sample-clock drift and sigma = 0.05 noise.  The FM
decode runs without correction (OFF) and with slant="auto" (AUTO), alternately, after one warm-up call of each;
per-stage device times come from the context's CUDA-event stage timers (wefax_ctx_timings).  The card's name and
power limit are read in the same run.  Writes one JSON file (default profiles/fm_slant_r03.json).

    python tools/fm_slant_bench.py [--reps 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from wefax_b200 import synth  # noqa: E402
from wefax_b200.decoder import Decoder  # noqa: E402
from wefax_b200.fm import decode_fm  # noqa: E402

SR = 11025
SLANT_STAGES = ("fm_slant_profile", "fm_slant_fold", "fm_slant_track")


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError(f"nvidia-smi failed: {r.stderr.strip()}")
    name, power, clock = (x.strip() for x in r.stdout.splitlines()[0].split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--minutes", type=float, default=60.0)
    ap.add_argument("--drift-ppm", type=float, default=5.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fm_slant_r03.json"))
    a = ap.parse_args()

    lpm = 120
    pcm = synth.synth_recording(a.minutes * 60.0, lpm=lpm, seed=2024, block=8, drift_ppm=a.drift_ppm,
                                noise_sigma=0.05)
    frm, end = 5 * SR, len(pcm) - 15 * SR
    kw = dict(lpm=lpm, search_from=frm, image_end=end)
    rec = dict(recording=dict(minutes=a.minutes, lpm=lpm, drift_ppm=a.drift_ppm, noise_sigma=0.05, samples=len(pcm)),
               gpu=gpu_info(), reps=a.reps)
    with Decoder(0) as dec:
        off = decode_fm(dec, pcm, SR, **kw)                       # warm-up: transform plans, buffers, modules
        auto = decode_fm(dec, pcm, SR, slant="auto", **kw)
        dec.enable_timing(True)
        dec.timings(reset=True)
        stages = {"off": [], "auto": []}
        wall = {"off": [], "auto": []}
        for _ in range(a.reps):
            for mode, slant in (("off", None), ("auto", "auto")):
                t = time.perf_counter()
                res = decode_fm(dec, pcm, SR, slant=slant, **kw)
                wall[mode].append((time.perf_counter() - t) * 1e3)
                stages[mode].append({k: v[0] for k, v in dec.timings(reset=True).items()})
                if mode == "auto":
                    auto = res
    s = auto.slant
    per_stage = {}
    for mode in ("off", "auto"):
        names = sorted({k for d in stages[mode] for k in d})
        per_stage[mode] = {k: float(np.median([d.get(k, 0.0) for d in stages[mode]])) for k in names}
    total = {m: float(np.median([sum(d.values()) for d in stages[m]])) for m in ("off", "auto")}
    slant_ms = sum(per_stage["auto"].get(k, 0.0) for k in SLANT_STAGES)
    rec.update(
        device_ms_median=total, device_ms_by_stage_median=per_stage,
        slant_stages_ms=slant_ms, slant_added_ms=total["auto"] - total["off"],
        slant_added_fraction=(total["auto"] - total["off"]) / total["off"],
        host_wall_ms_median={m: float(np.median(wall[m])) for m in wall},
        estimate=dict(status=s.status, ppm=s.ppm, error_ppm=s.ppm - a.drift_ppm, line_length=s.line_length,
                      first_line=s.first_line, lines_total=s.lines_total, lines_used=s.lines_used,
                      residual_rms=s.residual_rms),
        image_rows=dict(off=int(off.image.shape[0]), auto=int(auto.image.shape[0])))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    g = rec["gpu"]
    print(f"{g['name']} (power limit {g['power_limit']}): {a.minutes:g}-min {lpm} LPM, {a.drift_ppm:+g} ppm")
    print(f"device time per decode (median of {a.reps}): OFF {total['off']:.3f} ms, AUTO {total['auto']:.3f} ms "
          f"(+{rec['slant_added_ms']:.3f} ms, {100 * rec['slant_added_fraction']:.1f} %)")
    for k in SLANT_STAGES:
        print(f"  {k:18s} {per_stage['auto'].get(k, 0.0):.4f} ms")
    print(f"estimate {s.ppm:+.4f} ppm (error {s.ppm - a.drift_ppm:+.4f}), {s.lines_used}/{s.lines_total} lines, "
          f"rms {s.residual_rms:.2f} samples; host wall OFF {rec['host_wall_ms_median']['off']:.1f} ms, "
          f"AUTO {rec['host_wall_ms_median']['auto']:.1f} ms")
    print(f"wrote {a.out}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
