"""Time of the chart finder (wefax_decode_fm_charts) on a 60-minute six-chart broadcast, against one plain FM decode.

Input: six synthetic charts of 10 minutes less the gaps, (120, 576), (60, 288), (90, 576), (240, 288), (100, 576),
(180, 288) as (LPM, IOC), with 5 s noise gaps, sigma = 0.05 noise and +5 ppm of sample-clock drift.  After one
warm-up call of each, decode_fm_charts without slant correction (OFF), decode_fm_charts with slant="auto" (AUTO) and
one decode_fm OFF of the first chart's span over the whole recording run alternately; host wall times and per-stage
device times (the context's CUDA-event stage timers, wefax_ctx_timings) are medians over the repetitions.  The card's
name and power limit are read in the same run.  Writes one JSON file (default profiles/fm_charts_r04.json).

    python tools/fm_charts_bench.py [--reps 10] [--out FILE]
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

SR = 11025
SIX = [(120, 576), (60, 288), (90, 576), (240, 288), (100, 576), (180, 288)]
GAP_S = 5.0
CHART_STAGES = ("fm_tone", "fm_lpm")
TAIL_STAGES = ("fm_phasing", "fm_image", "fm_slant_profile", "fm_slant_fold", "fm_slant_track")


def six_chart_broadcast(noise_sigma: float = 0.05, drift_ppm: float = 5.0, seed: int = 2026):
    """60 minutes exactly: six charts of (3600 - 5 gaps) / 6 s each."""
    dur = (3600.0 - GAP_S * (len(SIX) - 1)) / len(SIX)
    return synth.synth_broadcast([dict(duration_s=dur, lpm=lpm, ioc=ioc, block=8) for lpm, ioc in SIX],
                                 noise_sigma=noise_sigma, drift_ppm=drift_ppm, gap_s=GAP_S, seed=seed)


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError(f"nvidia-smi failed: {r.stderr.strip()}")
    name, power, clock = (x.strip() for x in r.stdout.splitlines()[0].split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main() -> int:
    from wefax_b200.decoder import Decoder
    from wefax_b200.fm import decode_fm, decode_fm_charts

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fm_charts_r04.json"))
    a = ap.parse_args()

    pcm, truth = six_chart_broadcast()
    rec = dict(recording=dict(minutes=len(pcm) / SR / 60, charts=SIX, gap_s=GAP_S, noise_sigma=0.05, drift_ppm=5.0,
                              samples=len(pcm)), gpu=gpu_info(), reps=a.reps)
    first = truth[0]
    one_kw = dict(lpm=first["lpm"], ioc=first["ioc"], search_from=first["search_from"], image_end=first["stop_begin"])
    calls = {"charts_off": lambda dec: decode_fm_charts(dec, pcm, SR),
             "charts_auto": lambda dec: decode_fm_charts(dec, pcm, SR, slant="auto"),
             "decode_fm_off": lambda dec: decode_fm(dec, pcm, SR, **one_kw)}
    with Decoder(0) as dec:
        last = {k: f(dec) for k, f in calls.items()}            # warm-up: transform plans, buffers, modules
        dec.enable_timing(True)
        dec.timings(reset=True)
        stages = {k: [] for k in calls}
        wall = {k: [] for k in calls}
        for _ in range(a.reps):
            for k, f in calls.items():
                t = time.perf_counter()
                last[k] = f(dec)
                wall[k].append((time.perf_counter() - t) * 1e3)
                stages[k].append(dec.timings(reset=True))
    per_stage, launches = {}, {}
    for k in calls:
        names = sorted({s for d in stages[k] for s in d})
        per_stage[k] = {s: float(np.median([d.get(s, (0.0, 0))[0] for d in stages[k]])) for s in names}
        launches[k] = {s: int(stages[k][-1].get(s, (0.0, 0))[1]) for s in names}
    total = {k: float(np.median([sum(v[0] for v in d.values()) for d in stages[k]])) for k in calls}
    found = []
    for mode in ("charts_off", "charts_auto"):
        found.append([dict(lpm=c.lpm, ioc=c.ioc, score=round(c.lpm_score, 4), search_from=c.search_from,
                           image_end=c.image_end, rows=None if c.image is None else int(c.image.shape[0]),
                           slant_ppm=None if c.slant is None else c.slant.ppm) for c in last[mode].charts])
    rec.update(device_ms_median=total, device_ms_by_stage_median=per_stage, stage_launches=launches,
               host_wall_ms_median={k: float(np.median(wall[k])) for k in wall},
               charts_found=dict(off=found[0], auto=found[1]), truth=truth)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    g = rec["gpu"]
    print(f"{g['name']} (power limit {g['power_limit']}): {rec['recording']['minutes']:.1f}-min broadcast, "
          f"{len(last['charts_off'].charts)} charts found of {len(SIX)}")
    for k in calls:
        print(f"{k:14s} host wall {rec['host_wall_ms_median'][k]:8.2f} ms, device (sum of stages) {total[k]:8.3f} ms")
        for s in CHART_STAGES + TAIL_STAGES + ("fm_grey",):
            if s in per_stage[k]:
                print(f"    {s:18s} {per_stage[k][s]:.4f} ms ({launches[k][s]} launches)")
    print(f"wrote {a.out}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
