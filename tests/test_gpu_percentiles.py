"""The 0.5 / 99.5 percentile stage against numpy on every selection path, at the batch sizes and lengths that select it.

``launch_percentiles`` (wefax_b200/csrc/stages.cu) picks its algorithm from the length ``n``, the batch size and the
device's SM count ``S``.  ``pct_path`` below restates that dispatch; every case names the path the model predicts, the
stage timers confirm that the kernels of that path (and only those) ran, and ``test_cases_cover_every_path`` requires the
case table to reach every path the model can produce on this device.  Each row is compared, exactly, with
``O.medfilt5`` + ``O.digitalize``: ``low``, ``high``, the status and every grey level.

Rows of a batch differ by distinct powers of two: median-5, numpy's lerp and the grey map commute exactly with such a
scaling, so the float64 reference is computed once per base row and every row still catches a row-stride error.
``bracket_falls_back`` restates the bracket test of ``pct_final_kernel`` on the host: the period-127 data (which the
stride-127 sample cannot see) must fall back, noise must not, and every bracket path gets rows of both sorts.
"""
import math

import numpy as np
import pytest

from oracle import wefax_oracle as O

pytestmark = pytest.mark.gpu

# --------------------------------------------------------------------------- the dispatch of launch_percentiles
K_PCT_STRIDE = 127                 # stages.cu:692  kPctStride: every 127th median goes into the sample
RADIX_BELOW = 1 << 20              # stages.cu:1170 radix select below 2^20 samples (WEFAX_PCT_MODE overrides)
MAX_NCTA = 128                     # stages.cu:1225 ncta = max(1, min(128, S / batch))
HIST_WORDS = 4 * 2048              # stages.cu:1228 the bracket kernel's histogram ahead of its sample slice
FUSED_SMEM = 200 * 1024            # stages.cu:1230 sample slice in pct_bracket2_kernel's shared memory up to this
FINAL_SMEM = 160 * 1024            # stages.cu:1280 list slice in pct_final_kernel's shared memory up to this
FUSED_PER_MAX = FUSED_SMEM // 4 - HIST_WORDS   # 43008 sample keys per CTA
REC_NAN = 4
N_MAX = 1 << 26                    # lengths the coverage check ranges over: 101 minutes at 11025 Hz


def pct_geometry(n):
    """PctGeom of stages.cu:1162-1213 (ranks, sample ranks, open ends, list capacity)."""
    v_lo, v_hi = (n - 1) * (0.5 / 100), (n - 1) * (99.5 / 100)
    i_lo, i_hi = math.floor(v_lo), math.floor(v_hi)
    r = [min(x, n - 1) for x in (i_lo, i_lo + 1, i_hi, i_hi + 1)]
    ns = (n + K_PCT_STRIDE - 1) // K_PCT_STRIDE
    delta = max(64, math.ceil(12.0 * math.sqrt(ns * 0.005)))
    a_lo, b_lo = r[0] // K_PCT_STRIDE - delta, r[1] // K_PCT_STRIDE + 1 + delta
    a_hi, b_hi = r[2] // K_PCT_STRIDE - delta, r[3] // K_PCT_STRIDE + 1 + delta
    s_rank = [min(max(x, 0), ns - 1) for x in (a_lo, b_lo, a_hi, b_hi)]
    cap = min(n, 4 * (2 * delta + 2) * K_PCT_STRIDE + 4096)
    return dict(r=r, ns=ns, delta=delta, s_rank=s_rank, open_lo=a_lo <= 0, open_hi=b_hi >= ns - 1, cap=cap)


def pct_path(n, batch, S, force=None):
    """``("radix",)`` or ``(sample, final)``: sample "fused" (pct_bracket2_kernel, in shared memory) or "global"
    (pct_sample_kernel + pct_bracket_kernel); final "local" / "global" (two cooperative CTA groups, list slices in
    shared / global memory) or "serial" (ncta == 1, launched without the cooperative API).  stages.cu:1170-1296."""
    bracket = force == "bracket" if force else n >= RADIX_BELOW
    if not bracket:
        return ("radix",)
    g = pct_geometry(n)
    ncta = max(1, min(MAX_NCTA, S // batch))
    per = -(-g["ns"] // ncta)
    sample = "fused" if (HIST_WORDS + per) * 4 <= FUSED_SMEM else "global"
    if ncta == 1:
        final = "serial"
    else:
        per_max = -(-g["cap"] // (ncta // 2))
        final = "local" if per_max * 4 <= FINAL_SMEM else "global"
    return (sample, final)


def ncta_of(batch, S):
    return max(1, min(MAX_NCTA, S // batch))


def reachable_paths(S, n_max=N_MAX):
    """Every path pct_path produces for 1 <= n <= n_max, any batch and either mode.  For a given ncta the sample and
    final choices are monotone in n, so the ends of the range and both sides of every switch are enough."""
    paths = {("radix",)}
    batches = {}
    for b in range(1, S + 2):
        batches.setdefault(ncta_of(b, S), b)
    for ncta, b in batches.items():
        cand = {1, RADIX_BELOW - 1, RADIX_BELOW, n_max}
        n_sw = FUSED_PER_MAX * ncta * K_PCT_STRIDE
        cand |= {n_sw, n_sw + 1}
        if ncta >= 2:
            lo, hi = 1, n_max          # last n whose final slices fit in shared memory
            if pct_path(lo, b, S, "bracket")[1] == "local":
                while lo < hi:
                    mid = (lo + hi + 1) // 2
                    if pct_path(mid, b, S, "bracket")[1] == "local":
                        lo = mid
                    else:
                        hi = mid - 1
                cand |= {lo, lo + 1}
        for n in cand:
            if 1 <= n <= n_max:
                paths.add(pct_path(n, b, S, "bracket" if n < RADIX_BELOW else None))
    return paths


def bracket_falls_back(m32, n, sample):
    """Host restatement of the bracket test (pct_bracket*_kernel keys, pct_collect2_kernel counts, pct_final_kernel
    check) on one row's float32 median-5 values.  Returns (falls back, shared leading key bits of the low and the high
    bracket as pct_final_kernel's level skip sees them: 0, 11 or 22)."""
    g = pct_geometry(n)
    keys = m32.view(np.uint32)
    samp = np.sort(keys[: g["ns"] * K_PCT_STRIDE: K_PCT_STRIDE])
    k = [int(samp[s]) for s in g["s_rank"]]
    if sample == "fused":   # two radix levels: the lower ends round down, the upper ends up to their 1024-key bin
        k = [k[0] & ~0x3FF, k[1] | 0x3FF, k[2] & ~0x3FF, k[3] | 0x3FF]
    if g["open_lo"]:
        k[0] = 0
    if g["open_hi"]:
        k[3] = 0xFFFFFFFF
    below0 = int(np.count_nonzero(keys < k[0]))
    len0 = int(np.count_nonzero((keys >= k[0]) & (keys <= k[1])))
    len1 = int(np.count_nonzero((keys >= k[2]) & (keys <= k[3])))
    below1 = n - int(np.count_nonzero(keys > k[3])) - len1
    r, cap = g["r"], g["cap"]
    ok = (len0 <= cap and len1 <= cap and below0 <= r[0] and r[1] < below0 + len0
          and below1 <= r[2] and r[3] < below1 + len1)

    def shared(a, b):
        return 0 if (a ^ b) >> 21 else (11 if (a ^ b) >> 10 else 22)
    return (not ok), (shared(k[0], k[1]), shared(k[2], k[3]))


# --------------------------------------------------------------------------- data
KINDS = ("noise", "ramp", "duplicates", "two_level", "periodic", "narrow", "zero_subnormal")


def make_base(kind, n):
    rng = np.random.default_rng(1000 + KINDS.index(kind))
    if kind == "noise":
        env = np.abs(rng.normal(size=n)) * 2000
    elif kind == "ramp":
        env = np.linspace(1.0, 9000.0, n)
    elif kind == "duplicates":
        env = rng.integers(0, 40, size=n).astype(np.float64) * 100.0
    elif kind == "two_level":
        env = np.where(rng.random(n) < 0.004, 50.0, 3000.0) + rng.random(n)
    elif kind == "periodic":       # period = the sampling stride: the sample sees one phase only
        env = 1000.0 + 900.0 * np.sin(2 * np.pi * np.arange(n) / 127.0) + rng.random(n)
    elif kind == "narrow":
        # 3000 + 12.5 U in runs of 8 (so the medians keep the distribution): 51200 keys above float32(3000), whose
        # low 10 bits are zero.  Where the brackets are not open, each lies inside one 1024-key bin: its ends share
        # 22 leading bits, and pct_final_kernel skips two of its three radix levels.
        env = np.repeat(3000.0 + 12.5 * rng.random(n // 8 + 1), 8)[:n]
    else:   # exact zeros below the 0.5 percentile, subnormals across it
        env = np.abs(rng.normal(size=n)) * 2000
        nz, nsub = max(1, 3 * n // 1000), max(1, 6 * n // 1000)
        a = n // 3
        env[a: a + nz] = 0.0
        sub = env[a + nz: a + nz + nsub]
        sub[:] = np.repeat(rng.random(nsub // 8 + 1) * 1e-39, 8)[: sub.size]
    return env.astype(np.float32)


class _Refs:
    """float64 references of the base rows of one length (only the latest length is held: the large ones are GBs)."""

    def __init__(self):
        self.n = None
        self.rows = {}

    def get(self, n, kind):
        if n != self.n:
            self.n, self.rows = n, {}
        if kind not in self.rows:
            base = make_base(kind, n)
            m = O.medfilt5(base.astype(np.float64))
            with np.errstate(invalid="ignore"):   # a constant row (n <= 2) has no grey levels, only the NaN status
                d, low, high = O.digitalize(m)
            ok = high - low > 0 and math.isfinite(high - low)
            self.rows[kind] = dict(base=base, m32=m.astype(np.float32), d=d.astype(np.uint8) if ok else None,
                                   low=low, high=high, ok=ok)
        return self.rows[kind]


_REFS = _Refs()


def device_sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def odd_ncta_batch(S):
    """Smallest batch >= 3 whose ncta is odd (batch 3: 49 CTAs on 148 SMs)."""
    return next(b for b in range(3, S) if ncta_of(b, S) % 2 == 1 and ncta_of(b, S) >= 5)


# id -> S -> (n, batch, WEFAX_PCT_MODE, kinds); ordered by length so that each length's references are made once
N_MOD4_2 = 1_300_006
ALL = KINDS
CASES = {
    "radix-b1": lambda S: (700_001, 1, None, ALL),
    "radix-b9": lambda S: (700_001, 9, None, ALL),
    "radix-bS+1": lambda S: (700_001, S + 1, None, ALL),
    "tiny-1": lambda S: (1, len(ALL), "bracket", ALL),
    "tiny-2": lambda S: (2, len(ALL), "bracket", ALL),
    "tiny-5": lambda S: (5, len(ALL), "bracket", ALL),
    "tiny-127": lambda S: (127, len(ALL), "bracket", ALL),
    "tiny-128": lambda S: (128, len(ALL), "bracket", ALL),
    "tiny-129": lambda S: (129, len(ALL), "bracket", ALL),
    "tiny-5000": lambda S: (5000, len(ALL), "bracket", ALL),
    "serial-bS/2+1": lambda S: (RADIX_BELOW + 7, S // 2 + 1, None, ALL),
    "serial-b2S+1": lambda S: (RADIX_BELOW + 7, 2 * S + 1, None, ALL),
    "local-even-b2": lambda S: (1_300_007, 2, None, ALL),
    "local-odd": lambda S: (1_300_007, odd_ncta_batch(S), None, ALL),
    "global-final-bS/2": lambda S: (1_300_007, S // 2, None, ALL),
    "mod4-local-even-b2": lambda S: (N_MOD4_2, 2, None, ALL),
    "mod4-local-odd": lambda S: (N_MOD4_2, odd_ncta_batch(S), None, ALL),
    "mod4-global-final-bS/2": lambda S: (N_MOD4_2, S // 2, None, ALL),
    "serial-fused-edge": lambda S: (FUSED_PER_MAX * K_PCT_STRIDE, S // 2 + 1, None, ALL),
    "serial-global-sample": lambda S: (FUSED_PER_MAX * K_PCT_STRIDE + 1, S // 2 + 1, None, ALL),
    "local-long-b2": lambda S: (FUSED_PER_MAX * K_PCT_STRIDE + 1, 2, None, ALL),
    "global-sample-coop": lambda S: (FUSED_PER_MAX * K_PCT_STRIDE * ncta_of(S // 4, S) + 1, S // 4, None,
                                     ("noise", "ramp", "periodic", "narrow", "zero_subnormal")),
}
SLOW = {"serial-fused-edge", "serial-global-sample", "local-long-b2", "global-sample-coop", "serial-b2S+1"}
# rows that must fall back (True) or must not (False) wherever n >= 2^20
MEANT_FALLBACK = {"periodic": True, "noise": False}


@pytest.fixture(scope="module")
def dec():
    from wefax_b200.decoder import Decoder
    d = Decoder(0)
    d.enable_timing(True)
    yield d
    d.close()


def check_timings(t, path, where):
    assert "percentiles" in t, (where, t)
    assert ("pct_sample" in t) == (path[0] == "global"), (where, path, sorted(t))
    for name in ("pct_bracket", "pct_collect", "pct_final"):
        assert (name in t) == (path != ("radix",)), (where, path, name, sorted(t))


def test_path_model_matches_the_documented_switches():
    """The restatement at the sizes DESIGN.md §4.3 names (148 SMs)."""
    assert pct_path(700_001, 1, 148) == ("radix",)
    assert pct_path(1_300_007, 1, 148) == ("fused", "local")
    assert pct_path(1_300_007, 3, 148) == ("fused", "local") and ncta_of(3, 148) == 49
    assert pct_path(1_300_007, 74, 148) == ("fused", "global")
    assert pct_path(6_615_000, 64, 148) == ("fused", "global")
    assert pct_path(6_615_000, 75, 148) == ("global", "serial")
    assert pct_path(5_462_016, 75, 148) == ("fused", "serial")
    assert pct_path(5_462_017, 75, 148) == ("global", "serial")
    assert pct_path(21_848_065, 37, 148) == ("global", "global")
    assert pct_geometry(5000)["cap"] == 5000 and pct_geometry(5000)["open_lo"] and pct_geometry(5000)["open_hi"]


def test_cases_cover_every_path():
    """Every path the model produces on this device has a case, and every bracket path has a case whose rows must
    fall back and rows that must not."""
    S = device_sm_count()
    covered = {}
    for cid, f in CASES.items():
        n, b, force, kinds = f(S)
        p = pct_path(n, b, S, force)
        covered.setdefault(p, set())
        if n >= RADIX_BELOW:
            covered[p] |= {MEANT_FALLBACK[k] for k in kinds if k in MEANT_FALLBACK}
    missing = reachable_paths(S) - set(covered)
    assert not missing, (S, missing)
    for p, fb in covered.items():
        if p != ("radix",):
            assert fb == {True, False}, (p, fb)


@pytest.mark.parametrize("cid", [pytest.param(c, marks=pytest.mark.slow) if c in SLOW else c for c in CASES])
def test_stage_matches_numpy(dec, cid, monkeypatch):
    S = device_sm_count()
    n, batch, force, kinds = CASES[cid](S)
    if force:
        monkeypatch.setenv("WEFAX_PCT_MODE", force)
    else:
        monkeypatch.delenv("WEFAX_PCT_MODE", raising=False)
    path = pct_path(n, batch, S, force)
    K = len(kinds)
    calls = -(-K // batch)
    # the median-5 output is checked on small inputs; the large ones skip it (and its host buffer)
    with_dem = batch * n <= 16_000_000
    seen_fallback = {}
    for c in range(calls):
        row_kind = [kinds[(c * batch + i) % K] for i in range(batch)]
        row_exp = [(c * batch + i) // K for i in range(batch)]
        env = np.empty((batch, n), dtype=np.float32)
        for i in range(batch):
            np.multiply(_REFS.get(n, row_kind[i])["base"], np.float32(2.0 ** row_exp[i]), out=env[i])
        dec.timings(reset=True)
        dem, dig, lh, st = dec.digitalize(env, demodulated=with_dem)
        check_timings(dec.timings(reset=True), path, cid)
        del env
        for i in range(batch):
            ref = _REFS.get(n, row_kind[i])
            s = 2.0 ** row_exp[i]
            where = (cid, path, c, i, row_kind[i])
            assert lh[i, 0] == ref["low"] * s and lh[i, 1] == ref["high"] * s, (where, lh[i], ref["low"], ref["high"])
            if ref["ok"]:
                assert st[i] == 0, where
                assert np.array_equal(dig[i], ref["d"]), (where, int(np.count_nonzero(dig[i] != ref["d"])))
            else:
                assert st[i] == REC_NAN, where
            if dem is not None:
                assert np.array_equal(dem[i], ref["m32"] * np.float32(s)), where
            if path != ("radix",):
                fb, shared = bracket_falls_back(ref["m32"] * np.float32(s), n, path[0])
                seen_fallback.setdefault(row_kind[i], set()).add(fb)
                if n >= RADIX_BELOW and row_kind[i] in MEANT_FALLBACK:
                    assert fb == MEANT_FALLBACK[row_kind[i]], where
                if row_kind[i] == "narrow" and not pct_geometry(n)["open_lo"] and not pct_geometry(n)["open_hi"]:
                    assert not fb and shared == (22, 22), (where, shared)
    if path != ("radix",) and n >= RADIX_BELOW:
        assert {True, False} <= set().union(*seen_fallback.values()), (cid, seen_fallback)


# --------------------------------------------------------------------------- the paths inside the decode
TEN_MINUTES = 600 * 11025


@pytest.fixture(scope="module")
def ten_minute_pcm():
    from wefax_b200 import synth
    return synth.synth_recording(600.0, lpm=120, seed=5, noise_sigma=0.03)


def am_period_127(n):
    """A 1500 Hz carrier amplitude-modulated with period 127: its envelope defeats the stride-127 sample."""
    i = np.arange(n, dtype=np.float64)
    x = 0.25 * 32767 * (1.0 + 0.9 * np.sin(2 * np.pi * i / 127.0)) * np.sin(2 * np.pi * 1500.0 * i / 11025.0) / 1.9
    return np.round(x).astype(np.int16)


def decode_batch_pcm(base, B, am_row=1):
    pcm = np.empty((B, base.shape[0]), dtype=np.int16)
    for r in range(B):
        if r == am_row:
            pcm[r] = am_period_127(base.shape[0])
            continue
        # rolled and scaled a little differently per row: every row has its own percentiles
        np.right_shift(np.roll(base, 7919 * r).astype(np.int32) * (200 + r), 8, out=pcm[r], casting="unsafe")
    return pcm


def check_decode_rows(res, B, path, am_row=1):
    """Every row's low / high and grey levels equal O.digitalize of its own float32 medians."""
    import torch
    n = res.n_out
    fallback = []
    for i in range(B):
        dem = res.demodulated[i]
        dig = res.digitalized[i]
        if isinstance(dem, torch.Tensor):
            dem, dig = dem.cpu().numpy(), dig.cpu().numpy()
        d, low, high = O.digitalize(dem)
        assert res.low_high[i, 0] == low and res.low_high[i, 1] == high, (i, res.low_high[i], low, high)
        assert not (int(res.status[i]) & REC_NAN), i
        assert np.array_equal(dig, d.astype(np.uint8)), (i, int(np.count_nonzero(dig != d)))
        fallback.append(bracket_falls_back(dem, n, path[0])[0])
    assert fallback[am_row], "the period-127 row must defeat the sample"
    assert not all(fallback)
    return fallback


@pytest.mark.slow
@pytest.mark.parametrize("which", ["ncta2", "ncta1"])
def test_decode_percentile_paths(dec, ten_minute_pcm, which, monkeypatch):
    """Ten-minute recordings decoded in one wave: 64 of them (ncta = 2, list slices in global memory) and S/2 + 1
    (ncta = 1, the sample in global memory, serial final).  The fused grey map reads the threshold table that the
    last percentile kernel leaves behind, also where it fell back."""
    import torch
    monkeypatch.delenv("WEFAX_PCT_MODE", raising=False)
    S = device_sm_count()
    B = (1 << ((S // 2).bit_length() - 1)) if which == "ncta2" else S // 2 + 1
    path = pct_path(TEN_MINUTES, B, S)
    assert path == (("fused", "global") if which == "ncta2" else ("global", "serial")), (S, B, path)
    pcm = torch.from_numpy(decode_batch_pcm(ten_minute_pcm, B)).cuda()
    dec.timings(reset=True)
    res = dec.decode(pcm, 11025, 120, want=("demodulated", "digitalized", "raster"), device_outputs=True)
    t = dec.timings(reset=True)
    del pcm
    check_timings(t, path, which)
    assert t["pct_bracket"][1] == 1, "one wave"
    check_decode_rows(res, B, path)


@pytest.mark.slow
def test_decode_percentiles_depth_first(ten_minute_pcm, monkeypatch):
    """The same check with the recordings spread over concurrent decode lanes, four recordings per lane wave."""
    from wefax_b200.decoder import Decoder
    monkeypatch.delenv("WEFAX_PCT_MODE", raising=False)
    monkeypatch.setenv("WEFAX_DEPTH_FIRST", "1")
    monkeypatch.setenv("WEFAX_LANE_WAVE", "4")
    S = device_sm_count()
    B = 12
    pcm = decode_batch_pcm(ten_minute_pcm, B)
    with Decoder(0) as d:
        res = d.decode(pcm, 11025, 120, want=("demodulated", "digitalized", "raster"))
    check_decode_rows(res, B, pct_path(TEN_MINUTES, 4, S))
