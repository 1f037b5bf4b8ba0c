"""Host wall time of the chart decode over the C4 / C5 batch recordings: a loop of decode_fm_charts against one
decode_fm_charts_batch call (host PCM, and PCM resident on the device).

Inputs: ten-minute recordings synth.synth_recording(600, **synth.batch_spec(k, noisy)) (C4 clean, C5 with noise up to
0.1 FS, a carrier offset and a 5 ppm clock drift), a pool of 16 distinct ones replicated to the batch size as bench.py
does.  Under torchrun each rank takes its shard (sharding.local_batches); per batch size and slant mode (off, auto),
after one warm-up call of each, the loop, the host-PCM batch and the device-PCM batch run alternately --reps times.
Times are medians over the repetitions of the maximum over ranks; device times per stage come from the context's
CUDA-event stage timers (wefax_ctx_timings).  Every recording's chart list is gathered (sharding.gather_results) and
checked: one chart, with its batch_spec LPM and IOC.  The card's name and power limit are read in the same run.

    [torchrun --nproc-per-node N] python tools/fm_batch_bench.py [--sizes 8 64 512] [--reps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.fm_charts_bench import gpu_info  # noqa: E402
from wefax_b200 import sharding, synth  # noqa: E402

SR = 11025
DURATION_S = 600.0
DISTINCT = 16


def main() -> int:
    import torch
    import torch.distributed as dist
    from wefax_b200.decoder import Decoder
    from wefax_b200.fm import decode_fm_charts, decode_fm_charts_batch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", type=int, nargs="+", default=[8, 64, 512])
    ap.add_argument("--configs", nargs="+", default=["C4", "C5"], choices=["C4", "C5"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fm_batch_r05.json"))
    a = ap.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rec = dict(gpu=gpu_info() if rank == 0 else None, world_size=world, duration_s=DURATION_S, distinct=DISTINCT,
               reps=a.reps, runs=[])
    dec = Decoder(local_rank)
    for config in a.configs:
        noisy = config == "C5"
        specs = [synth.batch_spec(k, noisy=noisy) for k in range(DISTINCT)]
        pool = np.stack([synth.synth_recording(DURATION_S, **sp) for sp in specs])
        n = int(pool.shape[1])
        for size in a.sizes:
            keys = [(n, SR, 1)] * size
            mine = [i for _, idx in sharding.local_batches(keys, rank, world) for i in idx]
            pcm = pool[[i % DISTINCT for i in mine]]
            pcm_dev = torch.from_numpy(pcm).cuda()
            for slant in (None, "auto"):
                calls = {"loop": lambda: [decode_fm_charts(dec, p, SR, slant=slant) for p in pcm],
                         "batch_host_pcm": lambda: decode_fm_charts_batch(dec, pcm, SR, slant=slant),
                         "batch_device_pcm": lambda: decode_fm_charts_batch(dec, pcm_dev, SR, slant=slant)}
                last = {k: f() for k, f in calls.items()}       # warm-up: plans, buffers, modules
                wall = {k: [] for k in calls}
                stages = {k: [] for k in calls}
                dec.enable_timing(True)
                dec.timings(reset=True)
                for _ in range(a.reps):
                    for k, f in calls.items():
                        torch.cuda.synchronize()
                        if world > 1:
                            dist.barrier()
                        t = time.perf_counter()
                        last[k] = f()
                        wall[k].append(max_over_ranks(time.perf_counter() - t))
                        stages[k].append(dec.timings(reset=True))
                dec.enable_timing(False)
                # every recording's chart list, gathered on rank 0
                local = {i: [(c.lpm, c.ioc, c.status, c.image is not None) for c in r.charts]
                         for i, r in zip(mine, last["batch_host_pcm"])}
                same = all(
                    [(c.lpm, c.ioc, c.status, c.line_start) for c in x.charts] ==
                    [(c.lpm, c.ioc, c.status, c.line_start) for c in y.charts]
                    for key in ("batch_device_pcm", "loop") for x, y in zip(last[key], last["batch_host_pcm"]))
                merged = sharding.gather_results(local)
                same_all = max_over_ranks(0.0 if same else 1.0) == 0.0
                if rank != 0:
                    continue
                ok = [i for i in range(size)
                      if len(merged[i]) == 1 and merged[i][0][:2] == (float(specs[i % DISTINCT]["lpm"]),
                                                                      specs[i % DISTINCT]["ioc"])
                      and merged[i][0][2] == 0 and merged[i][0][3]]
                by_stage = {}
                for k in calls:
                    names = sorted({s for d in stages[k] for s in d})
                    by_stage[k] = {s: dict(ms=float(np.median([d.get(s, (0.0, 0))[0] for d in stages[k]])),
                                           launches=int(stages[k][-1].get(s, (0.0, 0))[1])) for s in names}
                run = dict(config=config, batch=size, slant=slant or "off", samples=n,
                           host_wall_ms_per_recording={k: 1e3 * float(np.median(v)) / size for k, v in wall.items()},
                           input_msamples_per_s={k: size * n / float(np.median(v)) / 1e6 for k, v in wall.items()},
                           device_ms_by_stage_median_rank0=by_stage,
                           charts_right=len(ok), charts_wrong=[i for i in range(size) if i not in set(ok)][:32],
                           loop_and_device_pcm_equal_host_batch=same_all)
                rec["runs"].append(run)
                hw = run["host_wall_ms_per_recording"]
                print(f"{config} batch {size:4d} slant {run['slant']:4s}: per recording loop {hw['loop']:7.2f} ms, "
                      f"batch {hw['batch_host_pcm']:7.2f} ms (host PCM), {hw['batch_device_pcm']:7.2f} ms (device PCM); "
                      f"charts right {len(ok)}/{size}; loop == batch: {same_all}", flush=True)
            del pcm_dev
            torch.cuda.empty_cache()
    dec.close()
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rec, fh, indent=1)
        g = rec["gpu"]
        print(f"{g['name']} (power limit {g['power_limit']}), {world} GPU(s): wrote {a.out}")
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
