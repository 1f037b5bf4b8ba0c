#!/usr/bin/env python
"""Benchmark of the WEFAX file-decoding hot path on B200.

    python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

Metric (BASELINE.json): decoded audio Msamples/s.  A step is one pass of the whole
hot path (ingest -> zero-phase notch -> Hilbert envelope -> median/percentile grey
map -> phasing search -> x4 raster) over one synthetic recording per GPU; at N=1
that is BASELINE.json configs[1]: a 60-min mono 11025 Hz recording at 120 LPM.
With N ranks every rank decodes its own recording (independent units, no
collective on the data path): weak scaling.

value : inputs and outputs resident in HBM, CUDA events on the decoder's stream,
        max over ranks.
e2e   : the same decode through the C-ABI call with HOST (pinned) buffers: the
        int16 PCM is copied to the device and digitalized + raster are copied back
        inside the timed region (wall clock between stream syncs, max over ranks).

--dump-outputs DIR writes what the last timed step returned (rank 0's recording; the inputs are seeded, so two
builds run with the same arguments can be compared output for output): start_frame, height, status, low_high,
peaks and phasing_signals (-1 padded to MAX_PEAKS per recording) whole as float64, and digitalized (the grey levels) and image (the pixels of
every recording's image, concatenated) as float32, whole up to DUMP_SAMPLE elements, else at DUMP_SAMPLE positions
drawn with DUMP_SEED.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "decoded audio Msamples/s"
UNIT = "Msamples/s"
ALGO_BYTES_PER_SAMPLE = 7.0      # SURVEY.md §8(d): int16 in + uint8 grey out + x4 uint8 raster out @ 11025 Hz
HBM_FALLBACK_GBS = 6650.0        # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_SAMPLE = 1 << 22            # --dump-outputs: elements kept of one large output (16 MiB as float32)
DUMP_SEED = 12345


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--duration", type=float, default=3600.0, help="seconds of audio per recording")
    ap.add_argument("--lpm", type=int, default=120)
    ap.add_argument("--sample-rate", type=int, default=11025,
                    help="input sample rate; != 11025 exercises the FFT-domain resampler (configs[2]: 48000, 1200 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-depth", type=int, default=3,
                    help="decoder contexts (one host thread each) the end-to-end measurement keeps in flight")
    ap.add_argument("--workspace-mb", type=int, default=0, help="cap on the scratch of one decode wave (0 = library default)")
    ap.add_argument("--batch", type=int, default=1,
                    help="recordings per GPU per step; > 1 selects the batch workload (BASELINE.json configs[3] shape: "
                         "--duration 600 --batch 64, LPM cycling 60/90/120/240)")
    ap.add_argument("--noisy", action="store_true",
                    help="with --batch: BASELINE configs[4] recordings (AWGN 0.02-0.1 FS, +-50 Hz carrier offset, 5 ppm "
                         "clock drift; synth.batch_spec(k, noisy=True)), 16 distinct ones replicated to the batch size")
    ap.add_argument("--segments", action="store_true",
                    help="BASELINE configs[2]: ONE recording (default 20 min at 48 kHz) decoded in overlapping segments, "
                         "one per GPU (strong scaling; wefax_b200/segments.py).  Not the headline workload.")
    ap.add_argument("--local-segments", type=int, default=1, help="with --segments: contexts (segments) per GPU")
    ap.add_argument("--devices", type=int, default=1,
                    help="with --segments, without torchrun: ONE process drives this many GPUs, one segment and one "
                         "host thread each; no process group, the histogram sums are plain host additions")
    ap.add_argument("--halo", type=int, default=65536, help="with --segments: halo in 11025-Hz samples")
    ap.add_argument("--config", default=None, choices=(None, "batch4096", "noisy4096"),
                    help="BASELINE.json configs[3] / configs[4] as written: --total (default 4096) ten-minute recordings "
                         "with mixed LPM 60/90/120/240 and IOC 288/576 dealt over the ranks by wefax_b200/sharding.py")
    ap.add_argument("--total", type=int, default=4096, help="with --config: recordings in the whole job")
    ap.add_argument("--repeat", type=int, default=1,
                    help="with --segments: the synthetic recording tiled this many times (a very long recording)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy "
                         "(see the module docstring)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.segments or args.config):
        ap.error("--dump-outputs covers the default decode path (also with --batch / --noisy / --sample-rate)")
    return args


def workload_name(args) -> str:
    if args.sample_rate != 11025:
        return (f"synthetic {args.duration / 60:g}-min mono {args.sample_rate} Hz recording resampled to 11025 Hz, "
                f"{args.lpm} LPM, one per GPU (BASELINE.json configs[2] on one GPU)")
    if args.batch > 1 and getattr(args, "noisy", False):
        return (f"batch of {args.batch} noisy synthetic {args.duration / 60:g}-min mono 11025 Hz recordings per GPU (AWGN, "
                f"+-50 Hz carrier offset, 5 ppm drift), mixed LPM and IOC (BASELINE.json configs[4] shape)")
    if args.batch > 1:
        return (f"batch of {args.batch} synthetic {args.duration / 60:g}-min mono 11025 Hz recordings per GPU, mixed LPM "
                f"60/90/120/240 (BASELINE.json configs[3] shape)")
    return (f"synthetic {args.duration / 60:g}-min mono 11025 Hz WEFAX recording, IOC576/{args.lpm} LPM, "
            f"one per GPU (BASELINE.json configs[1])")


JSON_OUT = sys.stdout


def bind_to_gpu_numa_node(index: int) -> None:
    """Pin this rank (and the threads it starts) to the CPU cores NVML reports as local to its GPU, BEFORE any pinned
    buffer is allocated: pinned staging then lives on the GPU's own NUMA node, and eight ranks do not push their
    PCIe traffic through the inter-socket link.  Best effort (single-socket hosts / containers: no-op)."""
    if os.environ.get("WEFAX_BENCH_NOBIND") == "1":   # (A/B switch)
        return
    global _FULL_AFFINITY
    if _FULL_AFFINITY is None:
        try:
            _FULL_AFFINITY = os.sched_getaffinity(0)
        except Exception:
            _FULL_AFFINITY = set()
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
    except Exception:
        pass


_FULL_AFFINITY = None


def unbind_from_numa_node() -> None:
    """Give the rank all its cores back.  The binding above is for WHERE pinned staging memory lands; while the
    device-resident loop runs it only makes the launching thread share a few cores with the NCCL / sampler threads
    (measured at 2 GPUs: 0.770 ms per step bound, 0.738 ms unbound)."""
    if _FULL_AFFINITY:
        try:
            os.sched_setaffinity(0, _FULL_AFFINITY)
        except Exception:
            pass


def claim_stdout() -> None:
    """stdout carries exactly one JSON line: keep a private handle on it and point fd 1 at stderr, so that
    banners of native libraries (NCCL's version line) cannot land in front of the JSON."""
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def copy_ceiling(world: int):
    """What the host can move with NO kernels (tools/copy_ceiling.py: one process per GPU, this step's pinned H2D + D2H
    traffic, full duplex), measured on this pool's 8 x B200 box and kept under profiles/: the end-to-end figure cannot
    exceed it.  None when no measurement exists for this GPU count."""
    try:
        with open(os.path.join(ROOT, "profiles", f"copy_ceiling_r02_n{world}.json")) as fh:
            c = json.load(fh)
        return {"msamples_s": round(c["e2e_ceiling_msamples_s"], 1), "d2h_gbs": round(c["duplex_d2h_gbs"], 1),
                "h2d_gbs": round(c["duplex_h2d_gbs"], 1), "source": f"profiles/copy_ceiling_r02_n{world}.json (measured, static)"}
    except Exception:
        return None


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._active = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            if self._active.is_set() and self.nv is not None:
                try:
                    self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    for bit, name in self.REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.004)

    def start(self):
        self.t.start()

    def region(self, on: bool):
        (self._active.set if on else self._active.clear)()

    def stop(self) -> dict:
        self._stop.set()
        self.t.join(timeout=1.0)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------- reference arm (CPU)
REFERENCE_SLEEP_S = 7.0   # wefax.py:59,73,75,77,193,202: fixed sleeps per process(), patched out and reported apart


def _oracle_decode(job):
    pcm, lpm = job
    from oracle import wefax_oracle as O
    out = O.decode(pcm, 11025, lpm)
    return int(out["digitalized_data"].shape[0])


def _reference_decode(job):
    """One process() of the UNMODIFIED reference (oracle/_ref or /root/reference) on a WAV file."""
    wav, lpm = job
    from oracle import ref_runner
    _dt, n = ref_runner.time_reference_process(wav, lpm)
    return int(n)


def reference_kind() -> str:
    try:
        from oracle import ref_runner
        return "reference" if ref_runner.reference_available() else "port"
    except Exception:
        return "port"


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank: int) -> None:
    """The reference's own CPU implementation of the path on the host cores: the unmodified
    `wefax.Demodulator.process()` staged under oracle/_ref (oracle/make_ref.py), one process per host core
    (the reference is single-threaded), each decoding one bounded recording of the same synthetic model per
    step.  Falls back to the numpy port (oracle/wefax_oracle.py) only where the reference files are absent."""
    if rank != 0:
        return
    import multiprocessing as mp
    import tempfile
    from wefax_b200 import synth
    kind = reference_kind()
    workers = max(1, min(host_cores(), 64))
    # per-core cost of the reference: ~1.15 us per sample + up to 6.6 s of pattern_search per recording
    # (BASELINE.md section 2); keep the whole run within a few minutes
    budget_s = 240.0 / max(1, args.steps)
    sample_s = 600.0 if kind == "port" else float(min(600.0, max(120.0, (budget_s - 6.6) / 1.27e-2)))
    sample_s = min(sample_s, args.duration)
    pcm = synth.synth_recording(sample_s, lpm=args.lpm, seed=0)
    tiny = synth.synth_recording(20.0, lpm=args.lpm, seed=0)
    tmp = tempfile.mkdtemp(prefix="wefax_ref_")
    if kind == "reference":
        wav, wav_tiny = os.path.join(tmp, "sample.wav"), os.path.join(tmp, "warm.wav")
        synth.write_wav(wav, pcm, 11025)
        synth.write_wav(wav_tiny, tiny, 11025)
        fn, jobs, warm_jobs = _reference_decode, [(wav, args.lpm)] * workers, [(wav_tiny, args.lpm)] * workers
    else:
        fn, jobs, warm_jobs = _oracle_decode, [(pcm, args.lpm)] * workers, [(tiny, args.lpm)] * workers
    with mp.get_context("fork").Pool(workers) as pool:
        for _ in range(args.warmup):          # CPU code has nothing to warm but the page cache: a 20-s clip
            pool.map(fn, warm_jobs)
        t0 = time.perf_counter()
        total = 0
        for _ in range(args.steps):
            total += sum(pool.map(fn, jobs))
        dt = time.perf_counter() - t0
    value = total / dt / 1e6
    what = ("the UNMODIFIED reference wefax.Demodulator.process() (oracle/_ref), matplotlib stubbed, its fixed "
            f"{REFERENCE_SLEEP_S:g} s of time.sleep per call patched out") if kind == "reference" else \
        "oracle/wefax_oracle.py numpy port (reference files not staged)"
    sample = (f"per step {workers} x one {sample_s:g} s recording ({pcm.shape[0]} samples) of the same synthetic model, "
              f"one process per host core; {what}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": kind, "sample": sample,
                         "sleep_s_per_file_not_counted": REFERENCE_SLEEP_S if kind == "reference" else 0.0},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)


# --------------------------------------------------------------------------- our arm (GPU)
def stage_bytes(name: str, n: int, half: bool) -> float:
    """Algorithmic bytes one launch of a stage must move for an n-sample recording
    (DESIGN.md 'Kernels'): what it has to read + write once.  With the real-input
    transform (even n) every FFT pass works on n/2 complex values."""
    m = n // 2 if half else n
    if name.startswith("fft_fwd_"):
        return m * 16.0
    if name.startswith("fft_inv_"):
        i = int(name.rsplit("_", 1)[1])
        if half:
            return m * 16.0 + (n * 4.0 if i == 0 else 0.0)   # the last pass also re-reads x for sqrt(x^2 + y^2)
        return m * (8.0 + (4.0 if i == 0 else 8.0))           # the last pass (index 0) writes |z| fp32
    return {"filtfilt": n * (2 + 4.0), "hilbert_pairs": m * 16.0, "hilbert_mid": m * 16.0, "percentiles": n * 4.0 * 3,
            "quantise": n * (4 + 1.0), "raster": n * (1 + 4.0), "median5": n * 8.0, "sync_search": 0.0,
            # fused demod-to-pixel sweep: envelope in (4 B), digitalized (1 B) + x4 raster (4 B) out
            "grey_raster": n * (4 + 1 + 4.0)}.get(name, 0.0)


def sample_index(sizes, stride: int) -> np.ndarray:
    """Flat indices into a (len(sizes), stride) buffer whose row i holds sizes[i] valid elements: all of them when
    they number at most DUMP_SAMPLE, else DUMP_SAMPLE positions drawn with DUMP_SEED (sorted), the same in every run
    whose outputs have the same sizes."""
    sizes = np.asarray(sizes, dtype=np.int64)
    total = int(sizes.sum())
    if total <= DUMP_SAMPLE:
        g = np.arange(total, dtype=np.int64)
    else:
        g = np.sort(np.random.default_rng(DUMP_SEED).integers(0, total, DUMP_SAMPLE))
    starts = np.cumsum(sizes) - sizes
    row = np.searchsorted(starts, g, side="right") - 1
    return row * stride + (g - starts[row])


def snapshot_outputs(res) -> dict:
    """What one decode call with device outputs handed back, copied out of buffers the next call overwrites: the
    per-recording results whole, the grey levels and the images (the first height x width bytes of each raster row;
    the rest of the row is not written) whole or sampled by sample_index."""
    import torch
    from wefax_b200 import _native as N
    B = len(res.lpm)
    out = {}
    for name, buf, sizes in (("digitalized", res.digitalized, [res.n_out] * B),
                             ("image", res.raster_flat, [int(h) * int(w) for h, w in zip(res.height, res.width)])):
        idx = torch.from_numpy(sample_index(sizes, buf.shape[1])).to(buf.device)
        out[name] = buf.reshape(-1).index_select(0, idx).cpu().numpy().astype(np.float32)
    for name in ("start_frame", "height", "status", "low_high"):
        out[name] = np.asarray(getattr(res, name), dtype=np.float64).copy()
    # ragged per recording: padded with -1 to the MAX_PEAKS slots the decoder fills, so that the shape does not depend
    # on the results (a recording may have no phasing lines at all)
    for name in ("peaks", "phasing_signals"):
        a = np.full((B, N.MAX_PEAKS), -1.0)
        for i, r in enumerate(getattr(res, name)):
            a[i, :len(r)] = r
        out[name] = a
    return out


def run_ours(args, rank: int, world: int, local_rank: int) -> None:
    import torch
    import torch.distributed as dist
    from wefax_b200 import synth
    from wefax_b200 import _native as N
    from wefax_b200.decoder import Decoder

    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when NCCL_DEBUG=VERSION; stdout carries exactly one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.batch > 1:
        # a pool of distinct recordings (one per LPM), replicated to the batch size: every copy is
        # decoded in full, nothing is cached between copies
        if args.noisy:
            specs = [synth.batch_spec(16 * rank + k, noisy=True) for k in range(min(16, args.batch))]
            distinct = [synth.synth_recording(args.duration, **sp) for sp in specs]
            lpms = [specs[k % len(specs)]["lpm"] for k in range(args.batch)]
            pcm = np.stack([distinct[k % len(distinct)] for k in range(args.batch)])
        else:
            pool = {l: synth.synth_recording(args.duration, lpm=l, seed=1000 * rank + l, noise_sigma=0.02)
                    for l in synth.BATCH_LPMS}
            lpms = [synth.BATCH_LPMS[k % 4] for k in range(args.batch)]
            pcm = np.stack([pool[l] for l in lpms])
        lpm_arg = lpms
    else:
        pcm = synth.synth_recording(args.duration, sample_rate=args.sample_rate, lpm=args.lpm, seed=rank)
        lpm_arg = args.lpm
    n = int(pcm.shape[-1]) * (args.batch if args.batch > 1 else 1)   # samples per GPU per step
    n_rec = int(pcm.shape[-1])
    stream = torch.cuda.Stream(device=local_rank)
    dec = Decoder(local_rank, stream=stream.cuda_stream, workspace_limit=(args.workspace_mb << 20) or None)
    pcm_dev = torch.from_numpy(pcm).cuda()
    pcm_pin = torch.empty(pcm.shape, dtype=torch.int16, pin_memory=True)
    pcm_pin.numpy()[...] = pcm
    want = ("digitalized", "raster")
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- value: everything resident in HBM -------------------------------------------
    if world > 1:
        unbind_from_numa_node()       # (pcm_pin is allocated: the device-resident loop needs no NUMA placement)
    res = dec.decode(pcm_dev, args.sample_rate, lpm_arg, want=want, device_outputs=True)
    # (a noisy recording may legitimately end in the reference's own ValueError of wefax.py:294; its decode still ran)
    ref_errors = sum(res.error(i) is not None for i in range(len(res.lpm)))
    if ref_errors and not args.noisy:
        raise RuntimeError(f"decode failed: {res.error(0)!r}")
    for _ in range(args.warmup):
        dec.decode(pcm_dev, args.sample_rate, lpm_arg, want=want, device_outputs=True, out=res)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = dec.launch_count
    sampler.region(True)
    ev0.record(stream)
    for _ in range(args.steps):
        dec.decode(pcm_dev, args.sample_rate, lpm_arg, want=want, device_outputs=True, out=res)
    ev1.record(stream)
    barrier()
    sampler.region(False)
    launches = dec.launch_count - launches0
    dumped = snapshot_outputs(res) if args.dump_outputs and rank == 0 else None
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_per_step = ms_total / args.steps
    value = world * n / (ms_per_step * 1e-3) / 1e6

    # ---- per-stage device times (same loop, stage launches bracketed by CUDA events) --
    dec.enable_timing(True)
    dec.timings(reset=True)
    sampler.region(True)
    for _ in range(args.steps):
        dec.decode(pcm_dev, args.sample_rate, lpm_arg, want=want, device_outputs=True, out=res)
    sampler.region(False)
    stage_ms = dec.timings(reset=True)
    dec.enable_timing(False)

    # ---- e2e: host buffers through the C-ABI -------------------------------------------
    # A stream of recordings through the public API: `depth` decoder contexts (own stream, own pinned
    # result buffers), one host thread each, take the steps round-robin, so the device->host copy of
    # one recording overlaps the host->device copy and the kernels of the next (PCIe is full duplex).
    # Every step still copies its PCM in and its digitalized data + raster out inside the timed region.
    if world > 1:
        bind_to_gpu_numa_node(local_rank)   # the pinned result buffers allocated next should be local to the GPU
    depth = max(1, min(args.e2e_depth, args.steps))
    decs = [dec] + [Decoder(local_rank, workspace_limit=(args.workspace_mb << 20) or None) for _ in range(depth - 1)]
    hosts = [d.decode(pcm_pin.numpy(), args.sample_rate, lpm_arg, want=want, pinned=True) for d in decs]
    for _ in range(max(1, args.warmup // 2)):
        for d, h in zip(decs, hosts):
            d.decode(pcm_pin.numpy(), args.sample_rate, lpm_arg, want=want, pinned=True, out=h)
    host = hosts[0]

    def e2e_worker(i):
        for _ in range(i, args.steps, depth):
            decs[i].decode(pcm_pin.numpy(), args.sample_rate, lpm_arg, want=want, pinned=True, out=hosts[i])
        decs[i].synchronize()

    barrier()
    sampler.region(True)
    t0 = time.perf_counter()
    workers = [threading.Thread(target=e2e_worker, args=(i,)) for i in range(depth)]
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    sampler.region(False)
    barrier()
    for d in decs[1:]:
        d.close()
    # ---- the same traffic with NO kernels, on THIS box (what the e2e figure cannot exceed): this step's pinned PCM up
    # and its results (digitalized + raster buffers as allocated) down, full duplex on two streams, all ranks at once
    live_ceiling = None
    try:
        outs = [t for t in (res.digitalized, res.raster_flat) if t is not None]
        pins = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in outs]
        s_up, s_dn = torch.cuda.Stream(device=local_rank), torch.cuda.Stream(device=local_rank)
        reps = max(5, min(20, args.steps))

        def copy_only(k):
            barrier()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            for _ in range(k):
                with torch.cuda.stream(s_up):
                    pcm_dev.copy_(pcm_pin, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    for dst, src in zip(pins, outs):
                        dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            return max_over_ranks(time.perf_counter() - t1)

        copy_only(2)
        copy_s = copy_only(reps)
        up_b = pcm_pin.numel() * pcm_pin.element_size()
        dn_b = sum(t.numel() * t.element_size() for t in outs)
        live_ceiling = {"msamples_s": round(world * n * reps / copy_s / 1e6, 1),
                        "h2d_gbs": round(world * up_b * reps / copy_s / 1e9, 1),
                        "d2h_gbs": round(world * dn_b * reps / copy_s / 1e9, 1),
                        "d2h_bytes_per_step_as_allocated": int(dn_b),
                        "source": "measured in this run on this box: the step's pinned copies alone, full duplex, no kernels"}
        del pins
    except Exception as exc:   # the ceiling is a reference figure, never a reason to lose the bench line
        live_ceiling = {"error": repr(exc)}
    e2e_value = world * n * args.steps / e2e_s / 1e6
    h2d = n * 2
    d2h = int(host.n_out) * max(1, args.batch) + int(sum(int(h) * int(w) for h, w in zip(host.height, host.width)))
    clocks = sampler.stop()

    # ---- multi-GPU correctness visible to the driver: ONE recording decoded in `world` overlapping segments
    # (wefax_b200/segments.py, configs[2] mode), one per rank, against rank 0's exact single-GPU decode ----------
    segments_check = None
    if world > 1 and args.batch == 1:
        from wefax_b200 import segments as S
        chk = synth.synth_recording(600.0, lpm=args.lpm, seed=777, noise_sigma=0.03)   # the same on every rank
        seg = S.decode_segmented(chk, 11025, args.lpm, [dec], exchange=S.HostExchange(device=local_rank),
                                 want=("raster",), gather=True)
        if rank == 0:
            whole = dec.decode(chk, 11025, args.lpm, want=("raster",))
            same_start = int(seg.start_frame) == int(whole.start_frame[0])
            img, ref_img = seg.image, whole.image(0)
            within = None
            if same_start and img is not None and img.shape == ref_img.shape and img.size:
                d = np.abs(img.astype(np.int16) - ref_img.astype(np.int16))
                within = [float((d <= 1).mean()), float((d == 0).mean())]
            segments_check = {"recording": "synthetic 10 min, 11025 Hz, AWGN 0.03 FS, seed 777", "segments": world,
                              "start_frame_equal": bool(same_start),
                              "start_frame": [int(seg.start_frame), int(whole.start_frame[0])],
                              "pixels_within_1_and_identical": within,
                              "stated_tolerance": ">= 99.5 % of pixels within +-1 (DESIGN.md section 6)"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = hbm_peak()
    n_rec = int(res.n_out)            # samples per recording at 11025 Hz (after the resampler)
    half = n_rec % 2 == 0 and not os.environ.get("WEFAX_NO_REAL_FFT")
    lens, blu = N.fft_plan_describe(n_rec // 2 if half else n_rec)
    if half and blu:                 # n/2 not smooth: the library falls back to the full-length transform
        half = False
        lens, blu = N.fft_plan_describe(n_rec)
    kernels = {}
    for name, (ms, cnt) in stage_ms.items():
        avg = ms / max(cnt, 1)
        # a large batch runs in waves that fit the workspace: one launch then moves 1/waves of the step's bytes
        b = stage_bytes(name, n, half) / max(1.0, cnt / args.steps)
        kernels[name] = {"ms": round(avg, 5), "launches_per_step": cnt / args.steps,
                         "algo_bytes": b, "gbs": round(b / (avg * 1e-3) / 1e9, 1) if avg > 0 and b else None}
    sub = {k: kernels.pop(k) for k in list(kernels) if k.startswith("pct_")}   # parts of "percentiles"
    sub.update({k: kernels.pop(k) for k in list(kernels) if k.startswith("sync_") and k != "sync_search"})
    # kernel families: which CUDA kernel runs each timed stage
    fast_lengths = {a * b for a in (12, 14, 15, 16) for b in (12, 14, 15, 16)} | {105}
    tma_lengths = {225, 240, 256, 210, 196, 105}
    fast_on = os.environ.get("WEFAX_FFT_FAST", "1") != "0" and len(lens) >= 2
    tma_on = fast_on and os.environ.get("WEFAX_FFT_TMAFAST", "1") != "0"
    npass = len(lens)

    def family(stage: str) -> str:
        if not stage.startswith("fft_"):
            mid = "hilbert_mid_kernel" if os.environ.get("WEFAX_MID_WARP") == "0" else "hilbert_mid_warp_kernel"
            return {"hilbert_mid": mid, "filtfilt": "notch_sym_kernel", "raster": "raster_kernel",
                    "grey_raster": "grey_raster_kernel",
                    "quantise": "quantise_kernel", "percentiles": "pct_*_kernel (4 launches)",
                    "sync_search": "sync_*_kernel (5 launches)"}.get(stage, stage)
        i = int(stage.rsplit("_", 1)[1])
        if i == npass - 1 or not fast_on or lens[i] not in fast_lengths:
            return "fft_pass_kernel"                      # generic (stride-1 pass, or a length outside the menu)
        if stage == "fft_inv_0" or not tma_on or lens[i] not in tma_lengths:
            return "fft_fast_strided_kernel"              # register-direct (envelope store)
        # TMA-staged plain complex pass (three tiles in flight unless WEFAX_TMA_PIPE=0)
        return "fft_fast_tma_kernel" if os.environ.get("WEFAX_TMA_PIPE") == "0" else "fft_fast_tma3_kernel"

    # "percentiles" and "sync_search" bracket several small kernels plus their host-side launch work: they are
    # reported as stages but are not candidates for the dominant KERNEL
    fam = {}
    for k, v in kernels.items():
        if k in ("percentiles", "sync_search"):
            continue
        f = fam.setdefault(family(k), {"ms": 0.0, "launches": 0.0, "bytes": 0.0})
        f["ms"] += v["ms"] * v["launches_per_step"]
        f["launches"] += v["launches_per_step"]
        f["bytes"] += v["algo_bytes"] * v["launches_per_step"]
    dom_name = max(fam, key=lambda k: fam[k]["ms"])
    dom_ms = fam[dom_name]["ms"] / max(fam[dom_name]["launches"], 1.0)
    dom_bytes = fam[dom_name]["bytes"] / max(fam[dom_name]["launches"], 1.0)
    dom_total_ms = fam[dom_name]["ms"]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            traffic = json.load(fh).get(dom_name)
    except Exception:
        pass
    stage_sum = sum(v["ms"] * v["launches_per_step"] for v in kernels.values())
    roofline_valid = args.sample_rate == 11025   # with the resampler, its passes share the fft_* tags of the Hilbert transform
    path_gbs = ALGO_BYTES_PER_SAMPLE * (n / (ms_per_step * 1e-3)) / 1e9

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "samples_per_recording": n_rec, "recordings_per_step": world * max(1, args.batch),
                   "fft_passes": lens, "fft_length": n_rec // 2 if half else n_rec,
                   "real_input_transform": bool(half), "bluestein": bool(blu), "outputs": list(want),
                   "l2": "no explicit flush: one step streams ~1.3 GB (>> 126 MB L2) through HBM",
                   "parallelism": f"{world} independent recordings, no collective",
                   "recordings_ending_in_a_reference_exception": int(ref_errors)},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s / args.steps * 1e3, "pipeline_depth": depth,
                "copy_only_ceiling": live_ceiling,
                "fraction_of_copy_only_ceiling": (round(e2e_value / live_ceiling["msamples_s"], 3)
                                                  if live_ceiling and live_ceiling.get("msamples_s") else None),
                "copy_only_ceiling_other_box": copy_ceiling(world),
                "api": "Decoder.decode -> wefax_decode_batch (host pinned buffers), one host thread + context per pipeline slot"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": dom_name if roofline_valid else None,
                     "achieved": round(achieved, 1) if roofline_valid else None, "peak": peak,
                     "unit": "GB/s", "frac": round(achieved / peak, 4) if roofline_valid else None, "traffic": traffic,
                     "peak_source": peak_src, "algo_bytes_per_launch": dom_bytes, "avg_launch_ms": round(dom_ms, 5),
                     "share_of_step": round(dom_total_ms / stage_sum, 3) if stage_sum else None,
                     "launches_per_step": fam[dom_name]["launches"],
                     "whole_path": {"algo_bytes_per_sample": ALGO_BYTES_PER_SAMPLE, "achieved": round(path_gbs, 1),
                                    "frac": round(path_gbs / peak, 4)}},
        "stages": kernels, "stage_parts": sub,
    }
    if segments_check is not None:
        line["segments_check"] = segments_check
    # every kernel family against the HBM roofline (the dominant one is `roofline` itself); the fused
    # demod-to-pixel sweep is the kernel north_star sets the >= 60 % target for
    line["roofline"]["kernels"] = {
        k: {"ms": round(v["ms"] / max(v["launches"], 1.0), 5), "launches_per_step": v["launches"],
            "algo_bytes_per_launch": v["bytes"] / max(v["launches"], 1.0),
            "achieved": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] > 0 else None,
            "frac": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak, 4) if v["ms"] > 0 else None}
        for k, v in fam.items() if v["bytes"] > 0}
    if world == 1 and not args.no_cpu_baseline and args.batch == 1 and args.sample_rate == 11025:
        from oracle import wefax_oracle as O
        t0 = time.perf_counter()
        o = O.decode(pcm, 11025, args.lpm)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": n / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": f"the full {args.duration:g} s recording ({n} samples), one pass of "
                                          f"oracle/wefax_oracle.py on one host core"}
        # same-run sanity: the CUDA result against the oracle on this very workload
        dig = res.digitalized[0].cpu().numpy().astype(np.int64)
        line["parity"] = {"grey_within_1": float((np.abs(dig - o["digitalized_data"]) <= 1).mean()),
                          "start_frame_equal": bool(int(res.start_frame[0]) == int(o.get("start_frame", -1)))}
    else:
        line["cpu_baseline"] = None
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_segments(args, rank: int, world: int, local_rank: int) -> None:
    """ONE recording over world x local-segments contexts.  The timed region is the whole protocol with the
    segments' PCM resident in HBM: per-segment kernels, the three histogram exchanges + start_frame broadcast
    through the host, image rows left in each GPU's memory (`value`), or copied to pinned host memory and
    gathered on rank 0 (`e2e`).  Host exchanges are part of the path, so the clock is the host's, bracketed by
    barrier + synchronize, max over ranks."""
    import torch
    import torch.distributed as dist
    from wefax_b200 import segments as S
    from wefax_b200 import synth
    from wefax_b200.decoder import Decoder

    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rate = args.sample_rate
    pcm = synth.synth_recording(args.duration, sample_rate=rate, lpm=args.lpm, seed=1)   # same on every rank
    if args.repeat > 1:
        pcm = np.tile(pcm, args.repeat)
    n_frames = int(pcm.shape[0])
    single = world == 1 and args.devices > 1
    L = args.devices if single else args.local_segments
    G = world * L
    workers = [Decoder(d) for d in range(L)] if single else [Decoder(local_rank) for _ in range(L)]
    ex = S.HostExchange(device=local_rank)
    segs = S.plan_decode(n_frames, rate, args.lpm, G, args.halo)
    mine = {sg.index: torch.from_numpy(np.ascontiguousarray(S.segment_frames(pcm, sg))).cuda(workers[k].device)
            for k, sg in enumerate(segs[rank * L:(rank + 1) * L])}
    pinned = {sg.index: torch.from_numpy(np.ascontiguousarray(S.segment_frames(pcm, sg))).pin_memory()
              for sg in segs[rank * L:(rank + 1) * L]}
    sampler = ClockSampler(local_rank)
    sampler.start()

    def step(device_resident: bool):
        src = mine if device_resident else pinned
        return S.decode_segmented(None, rate, args.lpm, workers, halo=args.halo, exchange=ex, n_frames=n_frames,
                                  segment_pcm=lambda sg: src[sg.index], want=("raster",), segments=segs,
                                  rows_on_device=True, gather=not device_resident)

    res = step(True)
    if res.error() is not None:
        raise RuntimeError(f"decode failed: {res.error()!r}")
    for _ in range(args.warmup):
        step(True)
    barrier()
    l0 = sum(w.launch_count for w in workers)
    sampler.region(True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(True)
    barrier()
    ms_per_step = max_over_ranks(time.perf_counter() - t0) * 1e3 / args.steps
    sampler.region(False)
    launches = sum(w.launch_count for w in workers) - l0

    for _ in range(max(1, args.warmup // 2)):
        step(False)
    barrier()
    sampler.region(True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host = step(False)
    barrier()
    e2e_ms = max_over_ranks(time.perf_counter() - t0) * 1e3 / args.steps
    sampler.region(False)
    clocks = sampler.stop()

    # per-stage device times of this rank's first context (one more pass)
    workers[0].enable_timing(True)
    workers[0].timings(reset=True)
    step(True)
    stage_ms = workers[0].timings(reset=True)
    workers[0].enable_timing(False)

    if rank == 0:
        n_total = res.n_out
        algo = 2.0 * n_frames + 4.0 * res.width * ((n_total - res.start_frame) // res.width)   # int16 in, x4 raster out
        peak, src_peak = hbm_peak()
        line = {
            "metric": "decoded audio Msamples/s", "value": n_frames / (ms_per_step * 1e-3) / 1e6, "unit": "Msamples/s",
            "n_gpus": L if single else world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"synthetic {args.duration * args.repeat / 60:g}-min mono {rate} Hz WEFAX recording"
                                   f"{' (a ' + format(args.duration / 60, 'g') + '-min one tiled)' if args.repeat > 1 else ''}, {args.lpm} LPM, "
                                   f"split into {G} overlapping segments over {L if single else world} GPU(s)"
                                   f"{' driven by one process' if single else ''} (BASELINE.json configs[2])",
                       "frames": n_frames, "samples_at_11025": n_total, "segments": G, "halo": args.halo,
                       "segment_samples": [sg.n_out for sg in segs], "outputs": ["raster"],
                       "exchange": "3 x 32 KiB histograms all-reduced + start_frame broadcast through the host; no "
                                   "collective on the data path",
                       "timing": "host clock around the whole protocol (it contains host exchanges), barrier + "
                                 "synchronize both sides, max over ranks",
                       "l2": "no explicit flush; note: an 8-way split leaves ~2 M-sample segments that fit in L2"},
            "clocks": clocks,
            "e2e": {"value": n_frames / (e2e_ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(sum(2 * (sg.in_end - sg.in_begin) for sg in segs)),
                    "d2h_bytes_per_step": int(host.image.nbytes),
                    "api": "segments.decode_segmented -> wefax_segment_* (pinned host PCM per segment, image rows "
                           "sent GPU to GPU to rank 0, one pinned device->host copy of the image)"},
            "gpu_launches": int(launches) * world,   # this rank's launches x ranks (every rank runs the same kernels)
            "roofline": {"bound": "hbm", "kernel": "whole segmented path (A = 2 B per input frame + 4 B per raster byte)",
                         "achieved": algo / (ms_per_step * 1e-3) / 1e9, "peak": peak * (L if single else world),
                         "unit": "GB/s",
                         "frac": algo / (ms_per_step * 1e-3) / 1e9 / (peak * (L if single else world)), "traffic": None,
                         "peak_source": src_peak},
            "stages_rank0_ms": {k: v[0] for k, v in sorted(stage_ms.items())},
            "cpu_baseline": None,
        }
        print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_batch_config(args, rank: int, world: int, local_rank: int) -> None:
    """BASELINE.json configs[3] (batch4096) / configs[4] (noisy4096): `--total` ten-minute recordings, recording k
    with synth.batch_spec(k) (LPM (60, 90, 120, 240)[k % 4], IOC (576, 288)[(k // 4) % 2]; noisy: AWGN 0.02-0.1 FS,
    +-50 Hz carrier offset, 5 ppm drift), dealt over the ranks by sharding.local_batches, decoded by Decoder with
    inputs and outputs resident in HBM, start_frame / status gathered on rank 0, a subset checked against the oracle.
    The PCM of the job is TILED from 16 distinct recordings (k % 16; generating 4096 distinct ones on the host would
    take an hour): every copy is decoded in full, nothing is cached between copies."""
    import torch
    import torch.distributed as dist
    from wefax_b200 import sharding, synth
    from wefax_b200.decoder import Decoder

    noisy = args.config == "noisy4096"
    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    total = args.total
    duration = 600.0
    distinct = 16
    specs = [synth.batch_spec(k, noisy=noisy) for k in range(distinct)]
    pool = np.stack([synth.synth_recording(duration, **sp) for sp in specs])          # (16, n) int16, same on all ranks
    n = int(pool.shape[1])
    keys = [(n, 11025, 1)] * total
    batches = sharding.local_batches(keys, rank, world)                                # [(key, [indices])]
    mine = [i for _, idx in batches for i in idx]
    pool_dev = torch.from_numpy(pool).cuda()
    sel = torch.tensor([i % distinct for i in mine], dtype=torch.long, device=pool_dev.device)
    pcm_dev = pool_dev.index_select(0, sel).contiguous()                               # this rank's share, in HBM
    lpms = [specs[i % distinct]["lpm"] for i in mine]
    stream = torch.cuda.Stream(device=local_rank)
    dec = Decoder(local_rank, stream=stream.cuda_stream)
    want = ("digitalized", "raster")
    sampler = ClockSampler(local_rank)
    sampler.start()
    res = dec.decode(pcm_dev, 11025, lpms, want=want, device_outputs=True)
    for _ in range(max(0, args.warmup - 1)):
        dec.decode(pcm_dev, 11025, lpms, want=want, device_outputs=True, out=res)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = dec.launch_count
    sampler.region(True)
    ev0.record(stream)
    for _ in range(args.steps):
        dec.decode(pcm_dev, 11025, lpms, want=want, device_outputs=True, out=res)
    ev1.record(stream)
    barrier()
    sampler.region(False)
    launches = dec.launch_count - l0
    ms_per_step = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    clocks = sampler.stop()
    # ---- parity on a subset: every rank checks the first copy of each distinct recording it holds against the oracle
    # (2 per rank at 8 ranks, all 16 at one rank: 16 decodes of the float64 restatement in total, in parallel) --------
    from oracle import wefax_oracle as O
    first_copy = {}
    for j, i in enumerate(mine):
        first_copy.setdefault(i % distinct, j)
    checks = []
    for d, j in sorted(first_copy.items()):
        if world > 1 and d % world != rank % min(world, distinct):
            continue   # (every kind is held by every rank when world < 16: split the oracle work)
        o = O.decode(pool[d], 11025, specs[d]["lpm"])
        dig = res.digitalized[j].cpu().numpy().astype(np.int64)
        diff = np.abs(dig - o["digitalized_data"])
        err = res.error(j)
        agree = (err is None) == (o["error"] is None) and (
            int(res.start_frame[j]) == int(o["start_frame"]) if err is None else type(err).__name__ == o["error"][0])
        pix = None
        if err is None and agree:
            img, ref_img = res.image(j).cpu().numpy(), o["output_image"]
            pix = float((np.abs(img.astype(np.int16) - ref_img.astype(np.int16)) <= 1).mean()) if img.shape == ref_img.shape else 0.0
        checks.append((d, bool(agree), float((diff <= 1).mean()), float((diff == 0).mean()), pix))
    # ---- the only exchange: small per-recording results to rank 0 ---------------------------------------------
    local = {i: (int(res.start_frame[j]), int(res.status[j]), int(res.height[j])) for j, i in enumerate(mine)}
    merged = sharding.gather_results(local, 0)
    all_checks = sharding.gather_results({(rank, c[0]): c for c in checks}, 0)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    by_kind_check = {}
    for (_, d), c in all_checks.items():
        by_kind_check.setdefault(d, c)
    checked = len(by_kind_check)
    same_start = sum(1 for c in by_kind_check.values() if c[1])
    within1 = [c[2] for c in by_kind_check.values()]
    ident = [c[3] for c in by_kind_check.values()]
    pixels = [c[4] for c in by_kind_check.values() if c[4] is not None]
    # every copy of a distinct recording must decode to the same small results, whichever rank had it
    by_kind = {}
    consistent = True
    for i, v in merged.items():
        consistent &= by_kind.setdefault(i % distinct, v) == v
    value = total * n / (ms_per_step * 1e-3) / 1e6
    peak, peak_src = hbm_peak()
    path_gbs = ALGO_BYTES_PER_SAMPLE * value * 1e6 / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"batch of {total} {'noisy ' if noisy else ''}synthetic 10-min mono 11025 Hz recordings, mixed LPM "
                               f"60/90/120/240 and IOC 288/576, sharded over {world} GPU(s) by wefax_b200/sharding.py "
                               f"(BASELINE.json configs[{4 if noisy else 3}])",
                   "recordings": total, "recordings_per_gpu": len(mine), "samples_per_recording": n,
                   "pcm": "tiled from 16 distinct recordings (k % 16), every copy decoded in full",
                   "outputs": list(want), "parallelism": f"{world} ranks, no collective on the data path; host gather of "
                                                         "start_frame / status / height only",
                   "l2": "no explicit flush: one step streams > 10 GB per GPU through HBM"},
        "clocks": clocks, "gpu_launches": int(launches) * world,
        "roofline": {"bound": "hbm", "kernel": "whole path (A = 7 B per sample)", "achieved": round(path_gbs, 1),
                     "peak": peak * world, "unit": "GB/s", "frac": round(path_gbs / (peak * world), 4), "traffic": None,
                     "peak_source": peak_src},
        "parity": {"checked_against_oracle": checked, "start_frame_or_error_equal": same_start,
                   "grey_within_1_min": min(within1), "grey_identical_min": min(ident),
                   "pixels_within_1_min": min(pixels) if pixels else None,
                   "all_copies_of_a_recording_agree_across_ranks": bool(consistent),
                   "recordings_gathered": len(merged)},
        "e2e": None, "cpu_baseline": None,
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: `python bench.py --gpus N` without torchrun re-launches itself under it
        import subprocess
        port = 29500 + (os.getpid() % 2000)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    claim_stdout()
    if args.config:
        run_batch_config(args, rank, world, local_rank)
        return
    if args.segments:
        if "--duration" not in " ".join(sys.argv):
            args.duration = 1200.0
        if "--sample-rate" not in " ".join(sys.argv):
            args.sample_rate = 48000
        run_segments(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
