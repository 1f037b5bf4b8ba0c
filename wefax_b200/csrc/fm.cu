// N4 (SURVEY.md §8(f)): a true WEFAX demodulator as an EXTENSION of the reference path.
//
// The reference decodes by slope detection (notch + envelope, wefax.py:63-74) and rasters
// int(samples-per-line) columns.  Its README (README.md:85-101) describes what a radiofax receiver
// really does: the grey level is the instantaneous frequency (black 1500 Hz, white 2300 Hz), a
// line lasts 60/LPM seconds exactly (5512.5 samples at 120 LPM), and a line has pi*IOC pixels.
// None of that exists in the reference's code, so there is no reference parity here: this mode is
// off by default, is checked against a float64 restatement (oracle/fm_oracle.py) and against the
// ground truth of the synthetic generator, and never touches the reference-exact path.
//
//   band-limit   zero-phase FIR band-pass around the 1900 Hz +- 400 Hz carrier: the notch kernel
//                (stages.cu: filtfilt_kernel) run with windowed-sinc taps instead of the notch's
//   analytic     y = Hilbert(x) from the same real-input transform (fft_exec.cu), y stored
//   FM demod     phase difference of consecutive analytic samples -> Hz -> grey in [0, 1]
//   phasing      fold `fold_lines` lines of grey modulo the exact line length, boxcar of the 5 %
//                white pulse, arg max = line start (block-wide reduction)
//   image        pixel (row, col) = box average of grey over its exact fractional sample span,
//                one thread per pixel: demod -> grey map -> line resample in one pass over x, y
//   slant        (optional) the recording's true line length from the white line pulses: sheared folds of a
//                binned profile, per-line pulse tracking, a line fit on the host (api.cu; DESIGN.md §4.7a)
//   levels       (optional) each chart's tuning offset: lower medians of the grey over the phasing lines' body and
//                pulse, the picture shifted by their midpoint's distance from 0.5 (DESIGN.md §4.7d)
#include <cmath>
#include <vector>

#include "stages.cuh"

namespace wefax {

// windowed-sinc (Hamming) band-pass, unit gain at the band centre; applied forwards and backwards
FirParams make_bandpass_fir(double lo_hz, double hi_hz, double fs, int taps) {
    if (taps < 3 || taps > kMaxFirTaps - 1 || !(lo_hz > 0.0) || !(hi_hz > lo_hz) || !(hi_hz < fs / 2))
        WEFAX_THROW(WEFAX_ERR_INVALID, "bad band-pass parameters");
    if ((taps & 1) == 0) taps -= 1;
    std::vector<double> h(taps);
    const double fl = lo_hz / fs, fh = hi_hz / fs, mid = (taps - 1) / 2.0, fc = 0.5 * (fl + fh);
    double gr = 0.0, gi = 0.0;
    for (int i = 0; i < taps; ++i) {
        const double t = i - mid;
        const double ideal = t == 0.0 ? 2.0 * (fh - fl) : (sin(2.0 * M_PI * fh * t) - sin(2.0 * M_PI * fl * t)) / (M_PI * t);
        const double win = 0.54 - 0.46 * cos(2.0 * M_PI * i / (taps - 1));
        h[i] = ideal * win;
        gr += h[i] * cos(2.0 * M_PI * fc * t);
        gi += h[i] * sin(2.0 * M_PI * fc * t);
    }
    const double gain = sqrt(gr * gr + gi * gi);
    FirParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.K = taps;
    const int sizes[] = {16, 20, 24, 32, 48, 64};
    for (int s : sizes)
        if (taps <= s) {
            fp.KP = s;
            break;
        }
    for (int i = 0; i < taps; ++i) fp.h[i] = (float)(h[i] / gain);
    for (int j = 0; j < fp.KP; ++j) fp.hr[j] = fp.h[fp.KP - 1 - j];
    return fp;
}

// grey[i] = (f_inst - black) / (white - black), f_inst from the phase step z[i] * conj(z[i-1]); blockIdx.y = recording
__global__ void __launch_bounds__(256)
fm_grey_kernel(const float *x, const float *y, size_t xs, float *g, long long n, float hz_per_rad, float black,
               float inv_span) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    x += blockIdx.y * xs;
    y += blockIdx.y * xs;
    g += blockIdx.y * (size_t)n;
    const long long j = i > 0 ? i - 1 : 0, k = i > 0 ? i : 1;   // sample 0 repeats the first step
    const float xr = __ldg(x + k), yr = __ldg(y + k), xp = __ldg(x + j), yp = __ldg(y + j);
    const float re = fmaf(xr, xp, yr * yp), im = fmaf(yr, xp, -xr * yp);
    const float f = atan2f(im, re) * hz_per_rad;
    g[i] = (f - black) * inv_span;
}

__device__ __forceinline__ float clip01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }

// P[o] = sum over lines of clip(grey[from + floor(l * Ls + o)]), o < Lc = ceil(Ls); l * Ls and the sum each rounded
// (no fused multiply-add: at a line length that is not a binary fraction the fused form can pick the next sample).
// blockIdx.y = chart of the table (charts with phase = 0 are skipped), P of chart c at P + c * ps
__global__ void __launch_bounds__(256)
fm_fold_kernel(const FmChartJob *tab, int lines, float *P, int ps) {
    const FmChartJob &job = tab[blockIdx.y];
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const int Lc = job.Lc;
    if (!job.phase || o >= Lc) return;
    const float *g = job.g;
    const long long n = job.n, from = job.from;
    const double Ls = job.Ls;
    P += (size_t)blockIdx.y * ps;
    float acc = 0.f;
    for (int l = 0; l < lines; ++l) {
        const long long i = from + (long long)floor(__dadd_rn(__dmul_rn((double)l, Ls), (double)o));
        if (i < n) acc += clip01(__ldg(g + i));
    }
    P[o] = acc;
}

// line start = from + arg max_o sum_{j < wb} P[(o + j) mod Lc]  (smallest o on ties); one CTA per chart with phase = 1
__global__ void __launch_bounds__(1024)
fm_phase_kernel(const FmChartJob *tab, const float *P, int ps, long long *line_start) {
    extern __shared__ double pre[];    // pre[i] = sum_{j < i} P[j mod Lc], i <= 2*Lc (two periods: circular boxcar)
    __shared__ double s_part[1024];
    __shared__ unsigned long long s_best[32];
    const FmChartJob &job = tab[blockIdx.x];
    if (!job.phase) return;
    const int Lc = job.Lc, wb = job.wb;
    const long long from = job.from;
    P += (size_t)blockIdx.x * ps;
    line_start += blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x, total = 2 * Lc;
    // chunked scan: each thread sums a contiguous chunk, thread 0 scans the chunk totals
    const int chunk = (total + nt - 1) / nt;
    const int b = tid * chunk, e = min(b + chunk, total);
    double sum = 0.0;
    for (int i = b; i < e; ++i) sum += (double)P[i % Lc];
    s_part[tid] = sum;
    __syncthreads();
    if (tid == 0) {
        double run = 0.0;
        for (int t = 0; t < nt; ++t) {
            const double v = s_part[t];
            s_part[t] = run;
            run += v;
        }
    }
    __syncthreads();
    double run = s_part[tid];
    for (int i = b; i < e; ++i) {
        pre[i] = run;
        run += (double)P[i % Lc];
    }
    if (tid == nt - 1) pre[total] = run;
    __syncthreads();
    // key: score as ordered bits in the high word, (0x7fffffff - o) in the low word
    unsigned long long best = 0ull;
    for (int o = tid; o < Lc; o += nt) {
        const float score = (float)(pre[o + wb] - pre[o]);   // >= 0
        const unsigned long long key = ((unsigned long long)__float_as_uint(score) << 32) | (unsigned)(0x7fffffff - o);
        best = key > best ? key : best;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, d);
        best = other > best ? other : best;
    }
    if ((tid & 31) == 0) s_best[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < nt / 32; ++w) best = s_best[w] > best ? s_best[w] : best;
        *line_start = from + (long long)(0x7fffffff - (int)(unsigned)(best & 0xffffffffull));
    }
}

// pixel (r, p): box average of clip(grey - shift) over [a, a + Ls / W), a = line_start + r * Ls + p * Ls / W.
// rows = min(rows_max, floor((image_end - line_start) / Ls)), the host's expression (wefax_decode_fm_slant), so
// every row the caller is told about is written; grid.y strides over the rows (it is capped at 65535), grid.z is the
// chart of the table, grid.x covers the widest picture.  shift = 0 leaves every grey value as it is (g - 0.f == g).
__global__ void __launch_bounds__(256)
fm_image_kernel(const FmChartJob *tab, const long long *line_start, uint8_t *img) {
    const FmChartJob &job = tab[blockIdx.z];
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int W = job.W, rows_max = job.rows_max;
    if (p >= W || rows_max <= 0) return;
    const float *g = job.g;
    const float shift = job.shift;
    const long long n = job.n, image_end = job.image_end;
    const double Ls = job.Ls;
    img += job.out;
    const long long ls_i = line_start[blockIdx.z];
    const double ls = (double)ls_i;
    const long long rows = min((long long)rows_max, (long long)floor(__ddiv_rn((double)(image_end - ls_i), Ls)));
    const double step = Ls / (double)W;
    for (long long r = blockIdx.y; r < rows; r += gridDim.y) {
        const double a = ls + (double)r * Ls + (double)p * step, b = a + step;
        const long long i0 = (long long)floor(a), i1 = (long long)ceil(b);
        float acc = 0.f;
        for (long long i = i0; i < i1; ++i) {
            const double lo = fmax(a, (double)i), hi = fmin(b, (double)(i + 1));
            const float wgt = (float)(hi - lo);
            if (i >= 0 && i < n && wgt > 0.f) acc = fmaf(wgt, clip01(__ldg(g + i) - shift), acc);
        }
        const float v = rintf(255.f * acc / (float)step);
        img[(size_t)r * W + p] = (uint8_t)fminf(fmaxf(v, 0.f), 255.f);
    }
}

// ---- tuning offset: the black and white levels of the phasing lines (DESIGN.md §4.7d) ----

// order-preserving key: a < b as floats <=> key(a) < key(b) as unsigned integers (NaN aside)
__device__ __forceinline__ unsigned int float_key(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// One CTA per (set, chart): blockIdx.x = 0 is the body set, offsets o in [wb + e, floor(Ls) - e); 1 is the pulse set,
// o in [e, wb - e); e = ceil(wb / 4).  Its samples are i = s + floor(l * Ls + o) for lines l < lines (fm_fold_kernel's
// rounding), s = line_start[chart], kept where 0 <= i < min(n, image_end).  Out: the lower median of their unclipped
// grey (element floor((m - 1) / 2) of the m values in ascending order) and m.  The median is an exact radix select
// over the order-preserving keys, 11, 11 and 10 bits, each pass walking the set again (it is read from L2).
constexpr int kLevelsThreads = 1024;
__global__ void __launch_bounds__(kLevelsThreads)
fm_levels_kernel(const FmChartJob *tab, int lines, const long long *line_start, FmLevel *lev) {
    __shared__ unsigned int hist[2048];
    __shared__ unsigned int s_warp[kLevelsThreads / 32];
    __shared__ unsigned int s_prefix, s_rank;
    const FmChartJob &job = tab[blockIdx.y];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *g = job.g;
    const double Ls = job.Ls;
    const int wb = job.wb, e = (wb + 3) / 4;
    const int o0 = blockIdx.x == 0 ? wb + e : e;
    const int o1 = blockIdx.x == 0 ? (int)floor(Ls) - e : wb - e;
    const long long s = line_start[blockIdx.y], end = min(job.n, job.image_end);
    // line l starts at or after s + l * Ls - 1: the lines past this bound hold no sample below end
    const long long ln = end > s ? min((long long)lines, (long long)floor((double)(end - s) / Ls) + 2) : 0;
    lev += 2 * (size_t)blockIdx.y + blockIdx.x;
    unsigned int prefix = 0u, rank = 0u, count = 0u;
    for (int pass = 0; pass < 3; ++pass) {
        const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
        const unsigned int digit = pass == 2 ? 0x3ffu : 0x7ffu;
        const unsigned int chosen = pass == 0 ? 0u : (pass == 1 ? 0xffe00000u : 0xfffffc00u);   // bits already found
        for (int b = tid; b < 2048; b += kLevelsThreads) hist[b] = 0u;
        __syncthreads();
        for (long long l = 0; l < ln; ++l) {
            const double base = __dmul_rn((double)l, Ls);
            for (int o = o0 + tid; o < o1; o += kLevelsThreads) {
                const long long i = s + (long long)floor(__dadd_rn(base, (double)o));
                if (i < 0 || i >= end) continue;
                const unsigned int k = float_key(__ldg(g + i));
                if ((k & chosen) == prefix) atomicAdd(&hist[(k >> shift) & digit], 1u);
            }
        }
        __syncthreads();
        // exclusive scan of the bins, two per thread: the bin holding the rank extends the prefix
        const unsigned int h0 = hist[2 * tid], h1 = hist[2 * tid + 1], mine = h0 + h1;
        unsigned int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned int w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned int v = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += v;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        if (pass == 0) {
            count = s_warp[kLevelsThreads / 32 - 1];
            if (count == 0u) break;     // (every thread sees the same count)
            rank = (count - 1u) / 2u;
        }
        const unsigned int start = (warp ? s_warp[warp - 1] : 0u) + incl - mine;
        if (rank >= start && rank < start + h0) {
            s_prefix = prefix | ((unsigned int)(2 * tid) << shift);
            s_rank = rank - start;
        } else if (rank >= start + h0 && rank < start + mine) {
            s_prefix = prefix | ((unsigned int)(2 * tid + 1) << shift);
            s_rank = rank - start - h0;
        }
        __syncthreads();
        prefix = s_prefix;
        rank = s_rank;
    }
    if (tid == 0) {
        lev->value = count ? key_float(prefix) : __int_as_float(0x7fc00000);
        lev->pad = 0;
        lev->count = (long long)count;
    }
}

// ---- slant: the sample-clock error measured from the white line pulses (DESIGN.md §4.7a) ----

// Q[l][b] = mean of clip(grey) over [from + floor(l * Ls) + b * D, +D); samples at or past n count as 0.  One CTA per
// (line, chart), Ls = the chart's sLs, lines l < q_lines
__global__ void __launch_bounds__(256)
fm_slant_profile_kernel(const FmChartJob *tab, float *Q) {
    const FmChartJob &job = tab[blockIdx.y];
    const int l = blockIdx.x;
    if (l >= job.q_lines) return;
    const float *g = job.g;
    const long long n = job.n, from = job.from;
    const double Ls = job.sLs;
    const int D = job.D, Bn = job.Bn;
    Q += job.q_off;
    const long long base = from + (long long)floor((double)l * Ls);
    for (int b = threadIdx.x; b < Bn; b += blockDim.x) {
        const long long i0 = base + (long long)b * D;
        float acc = 0.f;
        for (int j = 0; j < D; ++j)
            if (i0 + j < n) acc += clip01(__ldg(g + i0 + j));
        Q[(size_t)l * Bn + b] = acc / (float)D;
    }
}

__device__ __forceinline__ int floor_div(int a, int b) { return a / b - ((a % b != 0) && ((a < 0) != (b < 0))); }

// One CTA per candidate c of the total shift k over `lines` lines (c = 0, 1, 2, 3, 4, ... -> k = 0, -2, +2, -4, +4, ...):
// S_k[b] = sum_l Q[l][(b + round(l * k / lines)) mod Bn], circular boxcar of wbb bins, arg max over (c, b) into *best as
// (score bits << 32) | (0x7fffffff - (c * Bn + b)): the highest score wins, then the smallest |k|, then the smallest b.
// blockIdx.y = chart (lines = q_lines, candidates c < n_cand), its key into best[chart]
__global__ void __launch_bounds__(1024)
fm_slant_fold_kernel(const FmChartJob *tab, const float *Q, unsigned long long *best) {
    extern __shared__ float S[];
    __shared__ unsigned long long s_best[32];
    const FmChartJob &job = tab[blockIdx.y];
    const int c = blockIdx.x, tid = threadIdx.x;
    if (c >= job.n_cand) return;
    const int lines = job.q_lines, Bn = job.Bn, wbb = job.wbb;
    Q += job.q_off;
    best += blockIdx.y;
    const int k = c == 0 ? 0 : ((c + 1) / 2) * 2 * ((c & 1) ? -1 : 1);
    for (int b = tid; b < Bn; b += blockDim.x) {
        float acc = 0.f;
        for (int l = 0; l < lines; ++l) {
            const int sh = floor_div(2 * l * k + lines, 2 * lines);
            const int col = ((b + sh) % Bn + Bn) % Bn;
            acc += __ldg(Q + (size_t)l * Bn + col);
        }
        S[b] = acc;
    }
    __syncthreads();
    unsigned long long key = 0ull;
    for (int b = tid; b < Bn; b += blockDim.x) {
        float score = 0.f;
        for (int j = 0; j < wbb; ++j) score += S[(b + j) % Bn];
        const unsigned long long kb = ((unsigned long long)__float_as_uint(fmaxf(score, 0.f)) << 32) |
                                      (unsigned)(0x7fffffff - (c * Bn + b));
        key = kb > key ? kb : key;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, d);
        key = other > key ? other : key;
    }
    if ((tid & 31) == 0) s_best[tid >> 5] = key;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < (int)(blockDim.x + 31) / 32; ++w) key = s_best[w] > key ? s_best[w] : key;
        atomicMax(best, key);
    }
}

// One warp per line l < lines: the pulse is the arg max over x in [c - R, c + R], c = floor(a + l * s + 0.5), of the
// width-wb boxcar of clip(grey) (smallest x on ties); contrast = boxcar mean - mean of the guard bands [x - wb, x) and
// [x + wb, x + 2 wb).  pos[l] = x when the contrast reaches min_contrast, else -1 (also when the window leaves the
// recording).  Boxcars from float64 prefix sums of the window in shared memory.  blockIdx.y = chart (a, s, wb = swb,
// R; lines l < track_lines), pos / contrast from its pos_off.
__global__ void __launch_bounds__(32)
fm_slant_track_kernel(const FmChartJob *tab, double min_contrast, long long *pos, float *contrast) {
    extern __shared__ double pre[];    // pre[i] = sum_{j < i} clip(g[lo + j]), i <= span
    const FmChartJob &job = tab[blockIdx.y];
    const int l = blockIdx.x, lane = threadIdx.x;
    if (l >= job.track_lines) return;
    const float *g = job.g;
    const long long n = job.n;
    const double a = job.a, s = job.s;
    const int wb = job.swb, R = job.R;
    pos += job.pos_off;
    contrast += job.pos_off;
    const long long c = (long long)floor(a + (double)l * s + 0.5);
    const long long lo = c - R - wb;
    const int span = 2 * R + 3 * wb;
    if (lo < 0 || lo + span > n) {
        if (lane == 0) {
            pos[l] = -1;
            contrast[l] = 0.f;
        }
        return;
    }
    for (int i = lane; i < span; i += 32) pre[i + 1] = (double)clip01(__ldg(g + lo + i));
    if (lane == 0) pre[0] = 0.0;
    __syncwarp();
    // in-place scan: each lane sums a contiguous chunk, the lanes scan their totals with shuffles
    const int chunk = (span + 31) / 32, b = 1 + lane * chunk, e = min(b + chunk, span + 1);
    double sum = 0.0;
    for (int i = b; i < e; ++i) sum += pre[i];
    double incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    double run = incl - sum;
    __syncwarp();
    for (int i = b; i < e; ++i) {
        run += pre[i];
        pre[i] = run;
    }
    __syncwarp();
    // x = c - R + t  <->  pre index u = t + wb
    double best = -1.0;
    int bt = 0;
    for (int t = lane; t <= 2 * R; t += 32) {
        const double box = pre[t + 2 * wb] - pre[t + wb];
        if (box > best) {
            best = box;
            bt = t;
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, d);
        const int ot = __shfl_xor_sync(0xffffffffu, bt, d);
        if (ob > best || (ob == best && ot < bt)) {
            best = ob;
            bt = ot;
        }
    }
    if (lane == 0) {
        const int u = bt + wb;
        const double guard = (pre[u] - pre[u - wb]) + (pre[u + 2 * wb] - pre[u + wb]);
        const double ctr = best / wb - guard / (2.0 * wb);
        pos[l] = ctr >= min_contrast ? c - R + bt : -1;
        contrast[l] = (float)ctr;
    }
}

// ---- charts of a recording: tone windows and the LPM from the phasing lines (DESIGN.md §4.7b) ----

// sum of K values over the CTA (every thread gets the totals); s: 32 * K doubles of shared memory
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double *s) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) / 32;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
        for (int d = 16; d; d >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], d);
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < K; ++k) s[warp * K + k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double t = 0.0;
        for (int w = 0; w < nw; ++w) t += s[w * K + k];
        v[k] = t;
    }
    __syncthreads();
}

// One CTA per whole window k of T samples: u = clip(grey), mu = mean, V = mean((u - mu)^2),
// C_f = sum_j (u_j - mu) exp(-2 pi i f j / 11025) for f = 300, 450, 675 Hz with the phase from the exact integer
// (f * j) mod 11025, r_f = 2 |C_f|^2 / (T^2 V) (0 when V = 0).  out[k] = (r_300, r_450, r_675, V)
constexpr int kToneThreads = 256;
__global__ void __launch_bounds__(kToneThreads)
fm_tone_kernel(const float *g, long long n, long long nw, float4 *out) {
    constexpr int T = WEFAX_FM_TONE_WINDOW;
    constexpr int F[3] = {300, 450, 675};
    __shared__ float u[T];
    __shared__ double s_red[32 * 7];
    const float *w = g + blockIdx.y * (size_t)n + (size_t)blockIdx.x * T;   // blockIdx.y = recording
    double m[1] = {0.0};
    for (int j = threadIdx.x; j < T; j += blockDim.x) {
        const float v = clip01(__ldg(w + j));
        u[j] = v;
        m[0] += (double)v;
    }
    block_sum<1>(m, s_red);    // (its barrier also publishes u)
    const double mu = m[0] / T;
    double a[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // sum d^2, then (re, im) of C_300, C_450, C_675
    for (int j = threadIdx.x; j < T; j += blockDim.x) {
        const double d = (double)u[j] - mu;
        a[0] += d * d;
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            float sn, cs;
            sincospif((float)(2 * ((F[f] * j) % WEFAX_TARGET_RATE)) / (float)WEFAX_TARGET_RATE, &sn, &cs);
            a[1 + 2 * f] += d * (double)cs;
            a[2 + 2 * f] -= d * (double)sn;
        }
    }
    block_sum<7>(a, s_red);
    if (threadIdx.x == 0) {
        float r[3];
#pragma unroll
        for (int f = 0; f < 3; ++f)
            r[f] = a[0] > 0.0 ? (float)(2.0 * (a[1 + 2 * f] * a[1 + 2 * f] + a[2 + 2 * f] * a[2 + 2 * f]) / ((double)T * a[0]))
                              : 0.f;
        out[blockIdx.y * (size_t)nw + blockIdx.x] = make_float4(r[0], r[1], r[2], (float)(a[0] / T));
    }
}

// One CTA per (chart, candidate): the phasing fold of fm_fold_kernel (same index, same float32 sums in line order) for
// the candidate's line length from the chart's `from` in its grey stream, kept in shared memory, then
// score = max_o sum_{j < wb} P[(o + j) mod Lc] / (wb * lines) - mean(P) / lines  (boxcar sums in float64)
__global__ void __launch_bounds__(1024)
fm_lpm_kernel(const FmChartJob *tab, LpmCandidates cand, int lines, double *score) {
    __shared__ float P[kLpmMaxLine];
    __shared__ double s_red[32 * 2];
    const int chart = blockIdx.x / cand.n, c = blockIdx.x % cand.n, tid = threadIdx.x, nt = blockDim.x;
    const double Ls = cand.Ls[c];
    const int Lc = cand.Lc[c], wb = cand.wb[c];
    const float *g = tab[chart].g;
    const long long n = tab[chart].n, f0 = tab[chart].from;
    double tot[1] = {0.0};
    for (int o = tid; o < Lc; o += nt) {
        float acc = 0.f;
        for (int l = 0; l < lines; ++l) {
            const long long i = f0 + (long long)floor(__dadd_rn(__dmul_rn((double)l, Ls), (double)o));
            if (i < n) acc += clip01(__ldg(g + i));
        }
        P[o] = acc;
        tot[0] += (double)acc;
    }
    block_sum<1>(tot, s_red);   // (its barrier also publishes P)
    // each thread slides the boxcar over a contiguous chunk of offsets
    const int chunk = (Lc + nt - 1) / nt, b = tid * chunk, e = min(b + chunk, Lc);
    double best = 0.0;
    if (b < e) {
        double box = 0.0;
        for (int j = 0; j < wb; ++j) box += (double)P[(b + j) % Lc];
        best = box;
        for (int o = b + 1; o < e; ++o) {
            box += (double)P[(o + wb - 1) % Lc] - (double)P[o - 1];
            best = fmax(best, box);
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, d));
    if ((tid & 31) == 0) s_red[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < (nt + 31) / 32; ++w) best = fmax(best, s_red[w]);
        score[blockIdx.x] = best / ((double)wb * lines) - tot[0] / Lc / lines;
    }
}

void launch_fm_tone(wefax_ctx *ctx, const float *g, long long n, long long n_windows, int batch, float4 *out) {
    if (n_windows <= 0 || batch <= 0) return;
    StageTimer timer(ctx, "fm_tone");
    fm_tone_kernel<<<dim3((unsigned)n_windows, batch), kToneThreads, 0, ctx->stream>>>(g, n, n_windows, out);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_lpm(wefax_ctx *ctx, const FmChartJob *d_tab, int n_charts, const LpmCandidates &cand, int lines,
                   double *d_score) {
    if (n_charts <= 0) return;
    StageTimer timer(ctx, "fm_lpm");
    fm_lpm_kernel<<<(unsigned)(n_charts * cand.n), 1024, 0, ctx->stream>>>(d_tab, cand, lines, d_score);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_grey(wefax_ctx *ctx, const float *x, const float *y, size_t xs, float *g, long long n, int batch,
                    double black_hz, double white_hz) {
    StageTimer timer(ctx, "fm_grey");
    const float hz_per_rad = (float)((double)WEFAX_TARGET_RATE / (2.0 * M_PI));
    fm_grey_kernel<<<dim3((unsigned)((n + 255) / 256), batch), 256, 0, ctx->stream>>>(
        x, y, xs, g, n, hz_per_rad, (float)black_hz, (float)(1.0 / (white_hz - black_hz)));
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_phasing(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts, int lines,
                       float *P, long long *d_line_start) {
    int Lc = 0;
    for (int c = 0; c < n_charts; ++c)
        if (h_tab[c].phase) Lc = std::max(Lc, h_tab[c].Lc);
    if (Lc == 0) return;
    StageTimer timer(ctx, "fm_phasing");
    fm_fold_kernel<<<dim3((Lc + 255) / 256, n_charts), 256, 0, ctx->stream>>>(d_tab, lines, P, Lc);
    const size_t smem = (size_t)(2 * Lc + 1) * sizeof(double);
    if (smem > 200 * 1024) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "line of %d samples is too long for the phasing search", Lc);
    const void *fn = (const void *)fm_phase_kernel;
    if (!ctx->smem_configured.count(fn)) {
        CUDA_CHECK(cudaFuncSetAttribute(fm_phase_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        ctx->smem_configured[fn] = 1;
    }
    fm_phase_kernel<<<n_charts, 1024, smem, ctx->stream>>>(d_tab, P, Lc, d_line_start);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches += 2;
}

void launch_fm_levels(wefax_ctx *ctx, const FmChartJob *d_tab, int n_charts, int lines, const long long *d_line_start,
                      FmLevel *lev) {
    if (n_charts <= 0) return;
    StageTimer timer(ctx, "fm_levels");
    fm_levels_kernel<<<dim3(2, n_charts), kLevelsThreads, 0, ctx->stream>>>(d_tab, lines, d_line_start, lev);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_image(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                     const long long *d_line_start, uint8_t *img) {
    int W = 0, rows = 0;
    for (int c = 0; c < n_charts; ++c)
        if (h_tab[c].rows_max > 0) {
            W = std::max(W, h_tab[c].W);
            rows = std::max(rows, h_tab[c].rows_max);
        }
    if (rows <= 0 || W <= 0) return;
    StageTimer timer(ctx, "fm_image");
    dim3 grid((W + 255) / 256, std::min(rows, 65535), n_charts);
    fm_image_kernel<<<grid, 256, 0, ctx->stream>>>(d_tab, d_line_start, img);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_profile(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts, float *Q) {
    int lines = 0;
    for (int c = 0; c < n_charts; ++c) lines = std::max(lines, h_tab[c].q_lines);
    if (lines <= 0) return;
    StageTimer timer(ctx, "fm_slant_profile");
    fm_slant_profile_kernel<<<dim3(lines, n_charts), 256, 0, ctx->stream>>>(d_tab, Q);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_fold(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                          const float *Q, unsigned long long *d_best) {
    int Bn = 0, n_cand = 0;
    for (int c = 0; c < n_charts; ++c) {
        const FmChartJob &j = h_tab[c];
        if (j.q_lines <= 0) continue;
        if (j.Bn > 8192 || (long long)j.n_cand * j.Bn > 0x7fffffffLL)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "slant search of %d bins x %d candidates is too large", j.Bn, j.n_cand);
        Bn = std::max(Bn, j.Bn);
        n_cand = std::max(n_cand, j.n_cand);
    }
    CUDA_CHECK(cudaMemsetAsync(d_best, 0, (size_t)n_charts * sizeof(unsigned long long), ctx->stream));
    if (n_cand <= 0) return;
    StageTimer timer(ctx, "fm_slant_fold");
    const int threads = std::min(1024, (Bn + 31) / 32 * 32);
    fm_slant_fold_kernel<<<dim3(n_cand, n_charts), threads, (size_t)Bn * sizeof(float), ctx->stream>>>(d_tab, Q, d_best);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_track(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                           double min_contrast, long long *pos, float *contrast) {
    int lines = 0;
    size_t smem = 0;
    for (int c = 0; c < n_charts; ++c) {
        const FmChartJob &j = h_tab[c];
        if (j.track_lines <= 0) continue;
        lines = std::max(lines, j.track_lines);
        const size_t sm = (size_t)(2 * j.R + 3 * j.swb + 1) * sizeof(double);
        if (sm > 48 * 1024)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "line pulse of %d samples is too long for the slant search", j.swb);
        smem = std::max(smem, sm);
    }
    if (lines <= 0) return;
    StageTimer timer(ctx, "fm_slant_track");
    fm_slant_track_kernel<<<dim3(lines, n_charts), 32, smem, ctx->stream>>>(d_tab, min_contrast, pos, contrast);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

}  // namespace wefax
