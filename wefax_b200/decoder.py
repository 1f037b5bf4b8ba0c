"""Batched decode on one GPU: thin Python over ``wefax_decode_batch`` (C-ABI).

``Decoder`` owns one native context (one GPU, one stream).  ``decode`` takes a
batch of equal-length recordings — host ``numpy`` int16 (pageable or pinned) or
a CUDA ``torch`` int16 tensor — and returns the reference decoder's
post-``process()`` quantities for each of them (wefax.py:55-84).  PyTorch is
used only to allocate pinned / device buffers and to hand over a stream.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _native as N

ALL_OUTPUTS = ("audio", "demodulated", "digitalized", "raster")


class WefaxNativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"wefax_b200 native error {code}: {message}")
        self.code = code
        self.message = message


@dataclass
class BatchResult:
    """Outputs of one ``Decoder.decode`` call; arrays are indexed by recording."""
    n_out: int                      # samples per recording at 11025 Hz
    sample_rate: int                # always 11025 after the call (wefax.py:392)
    lpm: list
    width: list                     # image width per recording (wefax.py:298)
    status: np.ndarray              # WEFAX_REC_* bits
    peaks: list                     # pattern_search() positions (wefax.py:261)
    phasing_signals: list           # wefax.py:78
    start_frame: np.ndarray         # wefax.py:80
    height: np.ndarray              # raster rows
    low_high: np.ndarray            # (B, 2) the 0.5 / 99.5 percentiles
    audio: object = None            # (B, n_out) float32   wefax.py:72
    demodulated: object = None      # (B, n_out) float32   wefax.py:74
    digitalized: object = None      # (B, n_out) uint8     wefax.py:76
    raster_flat: object = None      # (B, raster_stride) uint8
    on_device: bool = False
    _keepalive: list = field(default_factory=list, repr=False)
    # what a repeated ``decode(..., out=this)`` with identical arguments needs to skip the argument checking and the
    # allocation of the small result arrays (set by Decoder.decode; the arrays above are then updated in place)
    _fast: object = field(default=None, repr=False, compare=False)

    def image(self, i: int):
        """Raster of recording ``i`` as a ``(height, width)`` uint8 array (a view)."""
        if self.raster_flat is None:
            raise ValueError("decode() was called without 'raster' in want")
        h, w = int(self.height[i]), int(self.width[i])
        return self.raster_flat[i][: h * w].reshape(h, w)

    def error(self, i: int):
        """The exception the reference's process() would raise for recording ``i`` (or None)."""
        s = int(self.status[i])
        if s & N.REC_NAN:
            return ValueError("cannot convert float NaN to integer")       # wefax.py:216
        if s & N.REC_NO_GROUPS:
            return ValueError("max() iterable argument is empty")           # wefax.py:294
        if s & N.REC_NO_LINES:
            return IndexError("image index out of range")                   # wefax.py:304
        return None


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class Decoder:
    """One native context = one GPU + one stream.  Not thread-safe; use one per thread."""

    def __init__(self, device: int = 0, stream: int | None = None, workspace_limit: int | None = None):
        lib = N.load()
        if lib.wefax_abi_version() != N.ABI_VERSION:
            raise RuntimeError("libwefax_b200.so ABI mismatch; rebuild")
        handle = C.c_void_p()
        rc = lib.wefax_ctx_create(int(device), C.c_void_p(stream or 0), C.byref(handle))
        if rc != N.OK:
            raise WefaxNativeError(rc, "cannot create a CUDA context on device %d "
                                       "(wefax_b200 needs a Blackwell GPU; there is no CPU fallback)" % device)
        self._lib = lib
        self._h = handle
        self.device = int(device)
        if workspace_limit:
            lib.wefax_ctx_set_workspace_limit(self._h, int(workspace_limit))

    # -- plumbing -----------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.wefax_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int) -> None:
        if rc != N.OK:
            msg = self._lib.wefax_last_error(self._h).decode(errors="replace")
            if rc == N.ERR_INVALID:
                raise ValueError(msg)
            raise WefaxNativeError(rc, msg)

    @property
    def stream(self) -> int:
        return int(self._lib.wefax_ctx_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._lib.wefax_ctx_launch_count(self._h))

    def synchronize(self) -> None:
        self._check(self._lib.wefax_ctx_sync(self._h))

    def enable_timing(self, enable: bool = True) -> None:
        """Bracket every stage launch with CUDA events on the context's stream."""
        self._check(self._lib.wefax_ctx_enable_timing(self._h, int(enable)))

    def timings(self, reset: bool = True) -> dict:
        """``{stage: (total_ms, launches)}`` accumulated since the last reset."""
        buf = C.create_string_buffer(1 << 16)
        self._check(self._lib.wefax_ctx_timings(self._h, buf, len(buf), int(reset)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, ms, cnt = line.split()
            out[name] = (float(ms), int(cnt))
        return out

    # -- the decode path ------------------------------------------------------
    def decode(self, pcm, sample_rate: int, lpm=120, notch_freq=2600, notch_q=1,
               want=("digitalized", "raster"), device_outputs: bool = False, pinned: bool = False,
               out: BatchResult | None = None) -> BatchResult:
        """Decode a batch.

        pcm: int16, shape ``(n,)``, ``(n, 2)``, ``(B, n)`` or ``(B, n, 2)`` (numpy / CUDA torch
        tensor; a 2-D array whose last dim is 2 is taken as one stereo recording).
        lpm: one value or one per recording.  want: which large outputs to produce.
        device_outputs: leave the large outputs on the GPU (torch tensors).
        pinned: allocate host outputs in pinned memory (faster D2H).
        out: a previous result with the same shapes whose buffers are reused.
        """
        on_dev_in = _is_torch(pcm) and pcm.is_cuda
        shape = tuple(pcm.shape)
        # ---- the steady state of a service: the same buffers and settings again, results into the same object --------
        if out is not None and out._fast is not None:
            f = out._fast
            ptr = pcm.data_ptr() if on_dev_in else (pcm.ctypes.data if isinstance(pcm, np.ndarray) else None)
            key = (self._h.value if hasattr(self._h, "value") else id(self._h), ptr, shape, str(pcm.dtype), int(sample_rate),
                   lpm if np.isscalar(lpm) else tuple(lpm), notch_freq, notch_q, tuple(want), device_outputs, pinned)
            same_bufs = (out.audio is f["bufs"].get("audio") and out.demodulated is f["bufs"].get("demodulated")
                         and out.digitalized is f["bufs"].get("digitalized") and out.raster_flat is f["bufs"].get("raster"))
            if (ptr is not None and same_bufs and key == f["key"]
                    and (pcm.is_contiguous() if on_dev_in else pcm.flags["C_CONTIGUOUS"])):
                self._check(self._lib.wefax_decode_batch(self._h, f["desc"], C.c_void_p(ptr), f["lpm"], f["out"]))
                peaks, n_peaks, phasing, n_phasing = f["peaks"], f["n_peaks"], f["phasing"], f["n_phasing"]
                B = len(out.lpm)
                out.peaks = [peaks[i, : n_peaks[i]].tolist() for i in range(B)]
                out.phasing_signals = [phasing[i, : n_phasing[i]].tolist() for i in range(B)]
                return out
        if len(shape) == 1:
            B, n, ch = 1, shape[0], 1
        elif len(shape) == 2 and shape[1] == 2 and shape[0] != 2:
            B, n, ch = 1, shape[0], 2
        elif len(shape) == 2:
            B, n, ch = shape[0], shape[1], 1
        elif len(shape) == 3 and shape[2] == 2:
            B, n, ch = shape[0], shape[1], 2
        else:
            raise ValueError(f"unsupported pcm shape {shape}")
        as_float = False
        if on_dev_in:
            import torch
            if pcm.dtype not in (torch.int16, torch.float32) or not pcm.is_contiguous():
                raise ValueError("device pcm must be a contiguous int16 (or mono float32) tensor")
            as_float = pcm.dtype == torch.float32
            pcm_ptr = pcm.data_ptr()
        else:
            if _is_torch(pcm):
                pcm = pcm.numpy()
            if pcm.dtype == np.float32:
                as_float = True   # WAV sample formats other than 16-bit PCM, converted by the caller (wefax.py:349)
            elif pcm.dtype != np.int16:
                raise TypeError(f"pcm must be int16 or float32 (got {pcm.dtype}); convert other WAV sample formats "
                                "first (wefax_b200.wefax.Demodulator does)")
            pcm = np.ascontiguousarray(pcm)
            pcm_ptr = pcm.ctypes.data
        if as_float and ch != 1:
            raise ValueError("float32 input must be mono: merge the channels first (wefax.py:360-373)")
        lpms = [float(lpm)] * B if np.isscalar(lpm) else [float(v) for v in lpm]
        if len(lpms) != B:
            raise ValueError("need one lpm per recording")
        sample_rate = int(sample_rate)
        n_out = n if sample_rate == N.TARGET_RATE else N.resampled_length(n, sample_rate)
        widths = [N.line_constants(v)["width"] for v in lpms]
        rstride = max(4 * (n_out // w) * w for w in widths) if n_out > 0 else 0
        for name in want:
            if name not in ALL_OUTPUTS:
                raise ValueError(f"unknown output {name!r}")

        keep = [pcm]
        if out is not None:
            keep.extend(out._keepalive)   # pinned tensors behind reused host buffers
        bufs = {}

        def alloc(name, shape_, dtype):
            prev = getattr(out, name if name != "raster" else "raster_flat") if out is not None else None
            if prev is not None:
                # a reused buffer must be exactly what this call would allocate: the native side writes
                # B * n_out (or raster_stride) elements through the raw pointer
                prev_dev = _is_torch(prev) and prev.is_cuda
                prev_dtype = str(prev.dtype).replace("torch.", "")
                if (tuple(prev.shape) != tuple(shape_) or prev_dtype != np.dtype(dtype).name
                        or prev_dev != bool(device_outputs)
                        or (prev_dev and prev.device.index != self.device)
                        or (_is_torch(prev) and not prev.is_contiguous())
                        or (not _is_torch(prev) and not prev.flags["C_CONTIGUOUS"])):
                    raise ValueError(f"out.{name} has shape {tuple(prev.shape)} / dtype {prev_dtype} / "
                                     f"{'device' if prev_dev else 'host'} memory; this call needs shape "
                                     f"{tuple(shape_)}, {np.dtype(dtype).name}, "
                                     f"{'device' if device_outputs else 'host'} memory")
                return prev
            if device_outputs:
                import torch
                tdt = {np.float32: torch.float32, np.uint8: torch.uint8}[dtype]
                return torch.empty(shape_, dtype=tdt, device=f"cuda:{self.device}")
            if pinned:
                import torch
                tdt = {np.float32: torch.float32, np.uint8: torch.uint8}[dtype]
                t = torch.empty(shape_, dtype=tdt, pin_memory=True)
                keep.append(t)
                return t.numpy()
            return np.empty(shape_, dtype=dtype)

        def ptr(a):
            return a.data_ptr() if _is_torch(a) else a.ctypes.data

        o = N.BatchOut()
        for name, dtype in (("audio", np.float32), ("demodulated", np.float32), ("digitalized", np.uint8)):
            if name in want:
                bufs[name] = alloc(name, (B, n_out), dtype)
                setattr(o, name, ptr(bufs[name]))
        if "raster" in want:
            bufs["raster"] = alloc("raster", (B, max(rstride, 1)), np.uint8)
            o.raster = ptr(bufs["raster"])
        o.raster_stride = max(rstride, 1)
        peaks = np.zeros((B, N.MAX_PEAKS), dtype=np.int32)
        n_peaks = np.zeros(B, dtype=np.int32)
        phasing = np.zeros((B, N.MAX_PEAKS), dtype=np.int32)
        n_phasing = np.zeros(B, dtype=np.int32)
        start = np.zeros(B, dtype=np.int64)
        height = np.zeros(B, dtype=np.int32)
        status = np.zeros(B, dtype=np.int32)
        low_high = np.zeros((B, 2), dtype=np.float64)
        o.peaks, o.n_peaks = peaks.ctypes.data, n_peaks.ctypes.data
        o.phasing, o.n_phasing = phasing.ctypes.data, n_phasing.ctypes.data
        o.start_frame, o.height = start.ctypes.data, height.ctypes.data
        o.status, o.low_high = status.ctypes.data, low_high.ctypes.data

        desc = N.BatchDesc(B, n, ch, sample_rate, float(notch_freq), float(notch_q),
                           (N.F_PCM_ON_DEVICE if on_dev_in else 0) | (N.F_OUT_ON_DEVICE if device_outputs else 0) |
                           (N.F_PCM_FLOAT32 if as_float else 0))
        lpm_arr = (C.c_double * B)(*lpms)
        lpm_ptr = C.cast(lpm_arr, C.c_void_p)
        self._check(self._lib.wefax_decode_batch(self._h, C.byref(desc), C.c_void_p(pcm_ptr), lpm_ptr, C.byref(o)))
        result = BatchResult(
            n_out=n_out, sample_rate=N.TARGET_RATE, lpm=lpms, width=widths, status=status,
            peaks=[peaks[i, : n_peaks[i]].tolist() for i in range(B)],
            phasing_signals=[phasing[i, : n_phasing[i]].tolist() for i in range(B)],
            start_frame=start, height=height, low_high=low_high,
            audio=bufs.get("audio"), demodulated=bufs.get("demodulated"),
            digitalized=bufs.get("digitalized"), raster_flat=bufs.get("raster"),
            on_device=device_outputs, _keepalive=keep)
        if on_dev_in or isinstance(pcm, np.ndarray):
            result._fast = {
                "key": (self._h.value if hasattr(self._h, "value") else id(self._h), pcm_ptr, shape, str(pcm.dtype),
                        sample_rate, lpm if np.isscalar(lpm) else tuple(lpm), notch_freq, notch_q, tuple(want),
                        device_outputs, pinned),
                "desc": C.byref(desc), "lpm": lpm_ptr, "out": C.byref(o),
                "hold": (desc, lpm_arr, o),           # the ctypes objects behind the references above
                "bufs": bufs,                         # the large buffers the native side writes through raw pointers
                "peaks": peaks, "n_peaks": n_peaks, "phasing": phasing, "n_phasing": n_phasing}
        return result

    # -- stage-level entry points (parity tests) --------------------------------
    def fft(self, x: np.ndarray, inverse: bool = False) -> np.ndarray:
        """Complex DFT along the last axis (complex64 in/out); numpy.fft conventions."""
        x = np.ascontiguousarray(x, dtype=np.complex64)
        batch = int(np.prod(x.shape[:-1])) if x.ndim > 1 else 1
        y = np.empty_like(x)
        self._check(self._lib.wefax_fft_c2c(self._h, x.shape[-1], batch, x.ctypes.data, y.ctypes.data, int(inverse)))
        return y

    def hilbert_envelope(self, x: np.ndarray) -> np.ndarray:
        """``abs(scipy.signal.hilbert(x))`` along the last axis (float32)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        batch = int(np.prod(x.shape[:-1])) if x.ndim > 1 else 1
        y = np.empty_like(x)
        self._check(self._lib.wefax_hilbert_envelope(self._h, x.shape[-1], batch, x.ctypes.data, y.ctypes.data))
        return y

    def resample(self, x: np.ndarray, num: int) -> np.ndarray:
        """``scipy.signal.resample(x, num)`` along the last axis (float32)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        batch = int(np.prod(x.shape[:-1])) if x.ndim > 1 else 1
        y = np.empty(x.shape[:-1] + (int(num),), dtype=np.float32)
        self._check(self._lib.wefax_resample(self._h, x.shape[-1], int(num), batch, x.ctypes.data, y.ctypes.data))
        return y

    def filtfilt(self, x: np.ndarray, notch_freq=2600, notch_q=1) -> np.ndarray:
        """``scipy.signal.filtfilt(*iirnotch(f0, Q, 11025), x)`` along the last axis (float32)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        batch = int(np.prod(x.shape[:-1])) if x.ndim > 1 else 1
        y = np.empty_like(x)
        self._check(self._lib.wefax_filtfilt(self._h, x.shape[-1], batch, float(notch_freq), float(notch_q),
                                             x.ctypes.data, y.ctypes.data))
        return y

    def digitalize(self, envelope: np.ndarray, demodulated: bool = True):
        """median-5 + percentile stretch + rounding of a raw |hilbert| envelope
        (wefax.py:175,196-216).  Returns ``(demodulated, digitalized, low_high, status)``;
        ``demodulated=False`` skips the median-5 output (returned as None) and its host buffer."""
        e = np.ascontiguousarray(envelope, dtype=np.float32)
        batch = int(np.prod(e.shape[:-1])) if e.ndim > 1 else 1
        dem = np.empty_like(e) if demodulated else None
        dig = np.empty(e.shape, dtype=np.uint8)
        lh = np.zeros((batch, 2), dtype=np.float64)
        st = np.zeros(batch, dtype=np.int32)
        self._check(self._lib.wefax_digitalize(self._h, e.shape[-1], batch, e.ctypes.data,
                                               C.c_void_p(dem.ctypes.data if dem is not None else None),
                                               dig.ctypes.data, lh.ctypes.data, st.ctypes.data))
        return dem, dig, lh, st

    def sync_raster(self, digitalized: np.ndarray, lpm) -> BatchResult:
        """Phasing search + raster on given digitalized data ``(B, n)`` uint8 (wefax.py:218-327)."""
        dig = np.ascontiguousarray(digitalized, dtype=np.uint8)
        if dig.ndim == 1:
            dig = dig[None]
        B, n = dig.shape
        lpms = [float(lpm)] * B if np.isscalar(lpm) else [float(v) for v in lpm]
        widths = [N.line_constants(v)["width"] for v in lpms]
        rstride = max(max(4 * (n // w) * w for w in widths), 1)
        raster = np.zeros((B, rstride), dtype=np.uint8)
        peaks = np.zeros((B, N.MAX_PEAKS), dtype=np.int32)
        n_peaks = np.zeros(B, dtype=np.int32)
        phasing = np.zeros((B, N.MAX_PEAKS), dtype=np.int32)
        n_phasing = np.zeros(B, dtype=np.int32)
        start = np.zeros(B, dtype=np.int64)
        height = np.zeros(B, dtype=np.int32)
        status = np.zeros(B, dtype=np.int32)
        o = N.BatchOut()
        o.raster, o.raster_stride = raster.ctypes.data, rstride
        o.peaks, o.n_peaks = peaks.ctypes.data, n_peaks.ctypes.data
        o.phasing, o.n_phasing = phasing.ctypes.data, n_phasing.ctypes.data
        o.start_frame, o.height, o.status = start.ctypes.data, height.ctypes.data, status.ctypes.data
        lpm_arr = (C.c_double * B)(*lpms)
        self._check(self._lib.wefax_sync_raster(self._h, n, B, dig.ctypes.data, C.cast(lpm_arr, C.c_void_p),
                                                C.byref(o)))
        return BatchResult(
            n_out=n, sample_rate=N.TARGET_RATE, lpm=lpms, width=widths, status=status,
            peaks=[peaks[i, : n_peaks[i]].tolist() for i in range(B)],
            phasing_signals=[phasing[i, : n_phasing[i]].tolist() for i in range(B)],
            start_frame=start, height=height, low_high=np.zeros((B, 2)), digitalized=dig, raster_flat=raster)

    # -- segment mode (one long recording over several contexts / GPUs; wefax_b200/segments.py) ----
    def segment_envelope(self, pcm, sample_rate: int, core_begin: int, core_end: int,
                         notch_freq=2600, notch_q=1, n_out: int | None = None, seam: int = 0) -> int:
        """Ingest (+ resample) + notch + |hilbert| of one extended segment; the envelope stays on the
        GPU.  ``[core_begin, core_end)``: the 11025-Hz samples this segment owns, relative to the
        extended segment; ``n_out``: its planned length at 11025 Hz (None: the reference's formula);
        ``seam``: where, inside the extended segment, the recording's end meets its start (0: nowhere).
        Returns the extended segment's length at 11025 Hz."""
        on_dev = _is_torch(pcm) and pcm.is_cuda
        shape = tuple(pcm.shape)
        ch = 2 if len(shape) == 2 else 1
        if len(shape) not in (1, 2) or (len(shape) == 2 and shape[1] != 2):
            raise ValueError(f"unsupported pcm shape {shape}")
        if on_dev:
            import torch
            if pcm.dtype != torch.int16 or not pcm.is_contiguous():
                raise ValueError("device pcm must be a contiguous int16 tensor")
            ptr = pcm.data_ptr()
        else:
            if _is_torch(pcm):
                pcm = pcm.numpy()
            if pcm.dtype != np.int16:
                raise TypeError(f"pcm must be int16 (got {pcm.dtype})")
            pcm = np.ascontiguousarray(pcm)
            ptr = pcm.ctypes.data
        desc = N.BatchDesc(1, shape[0], ch, int(sample_rate), float(notch_freq), float(notch_q),
                           N.F_PCM_ON_DEVICE if on_dev else 0)
        sample_rate = int(sample_rate)
        if n_out is None:
            n_out = shape[0] if sample_rate == N.TARGET_RATE else N.resampled_length(shape[0], sample_rate)
        self._check(self._lib.wefax_segment_envelope(self._h, C.byref(desc), C.c_void_p(ptr), int(n_out), int(seam),
                                                     int(core_begin), int(core_end)))
        self._seg_core = (int(core_begin), int(core_end))
        return int(n_out)

    def segment_histogram(self, level: int, prefix=(0, 0, 0, 0)) -> np.ndarray:
        """``(4, 2048)`` uint32 radix-digit histogram of the core's median-filtered envelope."""
        hist = np.zeros((4, 2048), dtype=np.uint32)
        pre = (C.c_uint32 * 4)(*[int(v) for v in prefix])
        self._check(self._lib.wefax_segment_histogram(self._h, int(level), pre, hist.ctypes.data))
        return hist

    def segment_quantise(self, low: float, high: float, want=("digitalized",)) -> dict:
        """Grey map of the extended segment with the global percentiles; returns the core's share of
        the outputs named in ``want`` (``digitalized`` uint8, ``demodulated`` float32)."""
        lo, hi = self._seg_core
        out = {}
        dig = np.empty(hi - lo, dtype=np.uint8) if "digitalized" in want else None
        dem = np.empty(hi - lo, dtype=np.float32) if "demodulated" in want else None
        self._check(self._lib.wefax_segment_quantise(
            self._h, float(low), float(high),
            C.c_void_p(dig.ctypes.data if dig is not None and dig.size else None),
            C.c_void_p(dem.ctypes.data if dem is not None and dem.size else None)))
        if dig is not None:
            out["digitalized"] = dig
        if dem is not None:
            out["demodulated"] = dem
        return out

    # device-resident form of the percentile exchange (state: CUDA int32 tensor of N.SEG_STATE_WORDS; nothing syncs)
    def segment_select_init(self, state, ranks, t_lo: float, t_hi: float) -> None:
        r = (C.c_uint32 * 4)(*[int(v) for v in ranks])
        self._check(self._lib.wefax_segment_select_init(self._h, C.c_void_p(state.data_ptr()), r, float(t_lo), float(t_hi)))

    def segment_histogram_dev(self, level: int, state) -> None:
        self._check(self._lib.wefax_segment_histogram_dev(self._h, int(level), C.c_void_p(state.data_ptr())))

    def segment_select_dev(self, level: int, state) -> None:
        self._check(self._lib.wefax_segment_select_dev(self._h, int(level), C.c_void_p(state.data_ptr())))

    def segment_quantise_dev(self, state, want=("digitalized",)) -> dict:
        """Grey map with the low / high held in the device state; the core's share of ``want`` comes back in pinned
        host arrays that are valid after the next synchronisation of this context."""
        lo, hi = self._seg_core
        out = {}
        dig = np.empty(hi - lo, dtype=np.uint8) if "digitalized" in want else None
        dem = np.empty(hi - lo, dtype=np.float32) if "demodulated" in want else None
        self._check(self._lib.wefax_segment_quantise_dev(
            self._h, C.c_void_p(state.data_ptr()),
            C.c_void_p(dig.ctypes.data if dig is not None and dig.size else None),
            C.c_void_p(dem.ctypes.data if dem is not None and dem.size else None)))
        if dig is not None or dem is not None:
            self.synchronize()   # pageable destinations: the copies above were staged, make them visible
        if dig is not None:
            out["digitalized"] = dig
        if dem is not None:
            out["demodulated"] = dem
        return out

    def segment_sync(self, lpm) -> dict:
        """Phasing search on the resident grey levels (the segment that starts the recording)."""
        peaks = np.zeros(N.MAX_PEAKS, dtype=np.int32)
        phasing = np.zeros(N.MAX_PEAKS, dtype=np.int32)
        n_peaks, n_phasing = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
        start, status = np.zeros(1, dtype=np.int64), np.zeros(1, dtype=np.int32)
        o = N.BatchOut()
        o.peaks, o.n_peaks = peaks.ctypes.data, n_peaks.ctypes.data
        o.phasing, o.n_phasing = phasing.ctypes.data, n_phasing.ctypes.data
        o.start_frame, o.status = start.ctypes.data, status.ctypes.data
        self._check(self._lib.wefax_segment_sync(self._h, float(lpm), C.byref(o)))
        return {"peaks": peaks[: n_peaks[0]].tolist(), "phasing_signals": phasing[: n_phasing[0]].tolist(),
                "start_frame": int(start[0]), "status": int(status[0])}

    def segment_raster(self, lpm, first_sample: int, n_lines: int, skip_lines: int, keep_lines: int,
                       out=None) -> np.ndarray:
        """``(4 * keep_lines, width)`` rows of the image lines this segment owns."""
        w = N.line_constants(float(lpm))["width"]
        if out is None:
            out = np.empty((4 * keep_lines, w), dtype=np.uint8)
        if keep_lines > 0:
            ptr = out.data_ptr() if _is_torch(out) else out.ctypes.data
            self._check(self._lib.wefax_segment_raster(self._h, float(lpm), int(first_sample), int(n_lines),
                                                       int(skip_lines), int(keep_lines), C.c_void_p(ptr)))
        return out
