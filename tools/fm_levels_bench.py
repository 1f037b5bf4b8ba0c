"""Accuracy and cost of the chart decode's tuning-offset correction (levels="auto", DESIGN.md §4.7d).

Workload 1: the 60-minute six-chart broadcast of tools/fm_charts_bench.py (sigma = 0.05, +5 ppm), each chart sent with
its own carrier offset (OFFSETS_HZ).  decode_fm_charts OFF and AUTO run alternately --reps times after one warm-up
call of each; per mode the host wall time, the device time (sum of the context's CUDA-event stage timers) and the
fm_levels time are medians over the repetitions.  Per chart: the estimated offset against the truth, and the mean
absolute error of the OFF and the AUTO picture against the picture of the transmitted grey at the same line start.
Workload 2: a C5 batch of 64 distinct ten-minute recordings (synth.batch_spec(k, noisy=True): noise up to 0.1 FS, a
carrier offset within +-50 Hz, +5 ppm) through decode_fm_charts_batch with AUTO: each recording's estimated offset
against its carrier_offset_hz, and the fm_levels time per wave (median over --reps calls).
The card's name and power limit are read in the same run.  Writes one JSON file (default profiles/fm_levels_r06.json).

    python tools/fm_levels_bench.py [--reps 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from oracle import fm_oracle as F  # noqa: E402
from tools.fm_charts_bench import GAP_S, SIX, gpu_info  # noqa: E402
from wefax_b200 import synth  # noqa: E402

SR = 11025
OFFSETS_HZ = (-120.0, -45.0, 0.0, 30.0, 90.0, 150.0)
BATCH, BATCH_DURATION_S = 64, 600.0


def broadcast():
    dur = (3600.0 - GAP_S * (len(SIX) - 1)) / len(SIX)
    return synth.synth_broadcast([dict(duration_s=dur, lpm=lpm, ioc=ioc, block=8, carrier_offset_hz=off)
                                  for (lpm, ioc), off in zip(SIX, OFFSETS_HZ)],
                                 noise_sigma=0.05, drift_ppm=5.0, gap_s=GAP_S, seed=2026, return_grey=True)


def _c5(k):
    return synth.synth_recording(BATCH_DURATION_S, **synth.batch_spec(k, noisy=True))


def _mae(chart, grey_truth):
    truth = F.image(grey_truth, chart.line_start, None, chart.ioc, chart.image_end, line_length=60.0 / chart.lpm * SR)
    return float(np.abs(chart.image.astype(np.float64) - truth).mean())


def _timed(dec, call, reps):
    wall, device, levels, launches = [], [], [], 0
    for _ in range(reps):
        t = time.perf_counter()
        res = call()
        wall.append((time.perf_counter() - t) * 1e3)
        st = dec.timings(reset=True)
        device.append(sum(v[0] for v in st.values()))
        levels.append(st.get("fm_levels", (0.0, 0))[0])
        launches = st.get("fm_levels", (0.0, 0))[1]
    return res, wall, device, levels, launches


def main() -> int:
    from wefax_b200.decoder import Decoder
    from wefax_b200.fm import decode_fm_charts, decode_fm_charts_batch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fm_levels_r06.json"))
    a = ap.parse_args()

    pcm, truth, grey_t = broadcast()
    with Pool(min(16, os.cpu_count() or 1)) as p:
        c5 = np.stack(p.map(_c5, range(BATCH)))
    c5_offsets = [synth.batch_spec(k, noisy=True)["carrier_offset_hz"] for k in range(BATCH)]
    rec = dict(gpu=gpu_info(), reps=a.reps,
               broadcast=dict(minutes=len(pcm) / SR / 60, charts=SIX, offsets_hz=OFFSETS_HZ, gap_s=GAP_S,
                              noise_sigma=0.05, drift_ppm=5.0),
               batch=dict(config="C5", recordings=BATCH, duration_s=BATCH_DURATION_S))
    with Decoder(0) as dec:
        modes = {"off": lambda: decode_fm_charts(dec, pcm, SR), "auto": lambda: decode_fm_charts(dec, pcm, SR, levels="auto")}
        for f in modes.values():
            f()                                           # warm-up: transform plans, buffers, modules
        dec.enable_timing(True)
        dec.timings(reset=True)
        runs = {k: dict(wall=[], device=[], levels=[]) for k in modes}
        last = {}
        for _ in range(a.reps):                           # OFF and AUTO alternate
            for k, f in modes.items():
                last[k], w, d, lv, _ = _timed(dec, f, 1)
                runs[k]["wall"] += w
                runs[k]["device"] += d
                runs[k]["levels"] += lv
        charts = []
        for c_off, c_auto, off in zip(last["off"].charts, last["auto"].charts, OFFSETS_HZ):
            charts.append(dict(lpm=c_auto.lpm, ioc=c_auto.ioc, truth_hz=off, estimate_hz=c_auto.levels.offset_hz,
                               error_hz=c_auto.levels.offset_hz - off, found=c_auto.levels.found,
                               span_hz=c_auto.levels.white_hz - c_auto.levels.black_hz,
                               mae_off=_mae(c_off, grey_t), mae_auto=_mae(c_auto, grey_t)))
        rec["broadcast"].update(
            charts_found=len(last["auto"].charts), charts=charts,
            host_wall_ms_median={k: float(np.median(v["wall"])) for k, v in runs.items()},
            device_ms_median={k: float(np.median(v["device"])) for k, v in runs.items()},
            fm_levels_ms_median=float(np.median(runs["auto"]["levels"])))

        decode_fm_charts_batch(dec, c5, SR, levels="auto")          # warm-up of this length
        dec.timings(reset=True)
        res, wall, device, levels, launches = _timed(dec, lambda: decode_fm_charts_batch(dec, c5, SR, levels="auto"),
                                                     a.reps)
        errs = [(r.charts[0].levels.offset_hz - off) if (r.charts and r.charts[0].levels) else None
                for r, off in zip(res, c5_offsets)]
        rec["batch"].update(
            offsets_hz=c5_offsets, errors_hz=errs,
            found=[bool(r.charts and r.charts[0].levels and r.charts[0].levels.found) for r in res],
            max_abs_error_hz=max(abs(e) for e in errs if e is not None),
            waves=launches, fm_levels_ms_median=float(np.median(levels)),
            fm_levels_ms_per_wave=float(np.median(levels)) / max(1, launches),
            device_ms_median=float(np.median(device)), host_wall_ms_median=float(np.median(wall)))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    g, b, c = rec["gpu"], rec["broadcast"], rec["batch"]
    print(f"{g['name']} (power limit {g['power_limit']})")
    for ch in b["charts"]:
        print(f"  {ch['lpm']:5g} LPM: offset {ch['truth_hz']:+7.1f} Hz, estimate {ch['estimate_hz']:+8.2f} Hz, "
              f"picture MAE off {ch['mae_off']:6.2f} auto {ch['mae_auto']:6.2f}")
    print(f"  broadcast: host wall off {b['host_wall_ms_median']['off']:.2f} ms, auto {b['host_wall_ms_median']['auto']:.2f}"
          f" ms; device off {b['device_ms_median']['off']:.3f} ms, auto {b['device_ms_median']['auto']:.3f} ms; "
          f"fm_levels {b['fm_levels_ms_median'] * 1e3:.1f} us")
    print(f"  C5 x {BATCH}: max |error| {c['max_abs_error_hz']:.2f} Hz, {sum(c['found'])} found; fm_levels "
          f"{c['fm_levels_ms_per_wave'] * 1e3:.1f} us per wave ({c['waves']} waves)")
    print(f"wrote {a.out}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
