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

// grey[i] = (f_inst - black) / (white - black), f_inst from the phase step z[i] * conj(z[i-1])
__global__ void __launch_bounds__(256)
fm_grey_kernel(const float *x, const float *y, float *g, long long n, float hz_per_rad, float black, float inv_span) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long j = i > 0 ? i - 1 : 0, k = i > 0 ? i : 1;   // sample 0 repeats the first step
    const float xr = __ldg(x + k), yr = __ldg(y + k), xp = __ldg(x + j), yp = __ldg(y + j);
    const float re = fmaf(xr, xp, yr * yp), im = fmaf(yr, xp, -xr * yp);
    const float f = atan2f(im, re) * hz_per_rad;
    g[i] = (f - black) * inv_span;
}

__device__ __forceinline__ float clip01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }

// P[o] = sum over lines of clip(grey[from + floor(l * Ls + o)]), o < Lc = ceil(Ls); l * Ls and the sum each rounded
// (no fused multiply-add: at a line length that is not a binary fraction the fused form can pick the next sample)
__global__ void __launch_bounds__(256)
fm_fold_kernel(const float *g, long long n, long long from, double Ls, int lines, int Lc, float *P) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= Lc) return;
    float acc = 0.f;
    for (int l = 0; l < lines; ++l) {
        const long long i = from + (long long)floor(__dadd_rn(__dmul_rn((double)l, Ls), (double)o));
        if (i < n) acc += clip01(__ldg(g + i));
    }
    P[o] = acc;
}

// line start = from + arg max_o sum_{j < wb} P[(o + j) mod Lc]  (smallest o on ties); one CTA
__global__ void __launch_bounds__(1024)
fm_phase_kernel(const float *P, int Lc, int wb, long long from, long long *line_start) {
    extern __shared__ double pre[];    // pre[i] = sum_{j < i} P[j mod Lc], i <= 2*Lc (two periods: circular boxcar)
    __shared__ double s_part[1024];
    __shared__ unsigned long long s_best[32];
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

// pixel (r, p): box average of clip(grey) over [a, a + Ls / W), a = line_start + r * Ls + p * Ls / W.
// rows = min(rows_max, floor((image_end - line_start) / Ls)), the host's expression (wefax_decode_fm_slant), so
// every row the caller is told about is written; grid.y strides over the rows (it is capped at 65535)
__global__ void __launch_bounds__(256)
fm_image_kernel(const float *g, long long n, const long long *line_start, double Ls, int W, int rows_max,
                long long image_end, uint8_t *img) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= W) return;
    const long long ls_i = *line_start;
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
            if (i >= 0 && i < n && wgt > 0.f) acc = fmaf(wgt, clip01(__ldg(g + i)), acc);
        }
        const float v = rintf(255.f * acc / (float)step);
        img[(size_t)r * W + p] = (uint8_t)fminf(fmaxf(v, 0.f), 255.f);
    }
}

// ---- slant: the sample-clock error measured from the white line pulses (DESIGN.md §4.7a) ----

// Q[l][b] = mean of clip(grey) over [from + floor(l * Ls) + b * D, +D); samples at or past n count as 0.  One CTA per line.
__global__ void __launch_bounds__(256)
fm_slant_profile_kernel(const float *g, long long n, long long from, double Ls, int D, int Bn, float *Q) {
    const int l = blockIdx.x;
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
__global__ void __launch_bounds__(1024)
fm_slant_fold_kernel(const float *Q, int lines, int Bn, int wbb, unsigned long long *best) {
    extern __shared__ float S[];
    __shared__ unsigned long long s_best[32];
    const int c = blockIdx.x, tid = threadIdx.x;
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
// recording).  Boxcars from float64 prefix sums of the window in shared memory.
__global__ void __launch_bounds__(32)
fm_slant_track_kernel(const float *g, long long n, double a, double s, int wb, int R, double min_contrast,
                      long long *pos, float *contrast) {
    extern __shared__ double pre[];    // pre[i] = sum_{j < i} clip(g[lo + j]), i <= span
    const int l = blockIdx.x, lane = threadIdx.x;
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

void launch_fm_grey(wefax_ctx *ctx, const float *x, const float *y, float *g, long long n, double black_hz,
                    double white_hz) {
    StageTimer timer(ctx, "fm_grey");
    const float hz_per_rad = (float)((double)WEFAX_TARGET_RATE / (2.0 * M_PI));
    fm_grey_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(x, y, g, n, hz_per_rad, (float)black_hz,
                                                                       (float)(1.0 / (white_hz - black_hz)));
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_phasing(wefax_ctx *ctx, const float *g, long long n, long long from, double Ls, int lines, float *P,
                       long long *d_line_start) {
    StageTimer timer(ctx, "fm_phasing");
    const int Lc = (int)ceil(Ls);
    const int wb = std::max(1, (int)llround(0.05 * Ls));
    fm_fold_kernel<<<(Lc + 255) / 256, 256, 0, ctx->stream>>>(g, n, from, Ls, lines, Lc, P);
    const size_t smem = (size_t)(2 * Lc + 1) * sizeof(double);
    if (smem > 200 * 1024) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "line of %d samples is too long for the phasing search", Lc);
    const void *fn = (const void *)fm_phase_kernel;
    if (!ctx->smem_configured.count(fn)) {
        CUDA_CHECK(cudaFuncSetAttribute(fm_phase_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        ctx->smem_configured[fn] = 1;
    }
    fm_phase_kernel<<<1, 1024, smem, ctx->stream>>>(P, Lc, wb, from, d_line_start);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches += 2;
}

void launch_fm_image(wefax_ctx *ctx, const float *g, long long n, const long long *d_line_start, double Ls, int W,
                     int rows_max, long long image_end, uint8_t *img) {
    if (rows_max <= 0) return;
    StageTimer timer(ctx, "fm_image");
    dim3 grid((W + 255) / 256, std::min(rows_max, 65535));
    fm_image_kernel<<<grid, 256, 0, ctx->stream>>>(g, n, d_line_start, Ls, W, rows_max, image_end, img);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_profile(wefax_ctx *ctx, const float *g, long long n, long long from, double Ls, int D, int Bn,
                             int lines, float *Q) {
    StageTimer timer(ctx, "fm_slant_profile");
    fm_slant_profile_kernel<<<lines, 256, 0, ctx->stream>>>(g, n, from, Ls, D, Bn, Q);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_fold(wefax_ctx *ctx, const float *Q, int lines, int Bn, int wbb, int n_cand,
                          unsigned long long *d_best) {
    StageTimer timer(ctx, "fm_slant_fold");
    if (Bn > 8192 || (long long)n_cand * Bn > 0x7fffffffLL)
        WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "slant search of %d bins x %d candidates is too large", Bn, n_cand);
    const int threads = std::min(1024, (Bn + 31) / 32 * 32);
    CUDA_CHECK(cudaMemsetAsync(d_best, 0, sizeof(unsigned long long), ctx->stream));
    fm_slant_fold_kernel<<<n_cand, threads, (size_t)Bn * sizeof(float), ctx->stream>>>(Q, lines, Bn, wbb, d_best);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void launch_fm_slant_track(wefax_ctx *ctx, const float *g, long long n, double a, double s, int lines, int wb, int R,
                           double min_contrast, long long *pos, float *contrast) {
    if (lines <= 0) return;
    StageTimer timer(ctx, "fm_slant_track");
    const size_t smem = (size_t)(2 * R + 3 * wb + 1) * sizeof(double);
    if (smem > 48 * 1024) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "line pulse of %d samples is too long for the slant search", wb);
    fm_slant_track_kernel<<<lines, 32, smem, ctx->stream>>>(g, n, a, s, wb, R, min_contrast, pos, contrast);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

}  // namespace wefax
