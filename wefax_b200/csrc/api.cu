// extern "C" surface of libwefax_b200.so: context management, host helpers and
// the batched decode that strings the kernels together (see include/wefax_b200.h).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "stages.cuh"

using namespace wefax;

namespace {

template <class F>
int guarded(wefax_ctx *ctx, F &&f, bool touches_scratch = true) {
    if (ctx && touches_scratch) ctx->api_calls++;
    try {
        f();
        return WEFAX_OK;
    } catch (const Error &e) {
        if (ctx) {
            ctx->last_error = e.msg;
            // (a call that failed half way: nothing of it may still be running when the caller reuses its buffers)
            if (ctx->stream && cudaStreamQuery(ctx->stream) != cudaErrorStreamCaptureUnsupported) {
                cudaStreamSynchronize(ctx->stream);
                (void)cudaGetLastError();
            }
        }
        return e.code;
    } catch (const std::bad_alloc &) {
        if (ctx) ctx->last_error = "host allocation failed";
        return WEFAX_ERR_NOMEM;
    } catch (const std::exception &e) {
        if (ctx) ctx->last_error = e.what();
        return WEFAX_ERR_INVALID;
    }
}

// scipy.signal.iirnotch (wefax.py:68-70)
void notch_coefficients(double f0, double q, double fs, double b[3], double a[3]) {
    double w0 = 2.0 * f0 / fs;
    if (w0 > 1.0 || w0 < 0.0) WEFAX_THROW(WEFAX_ERR_INVALID, "w0 should be such that 0 < w0 < 1");
    double bw = w0 / q * M_PI;
    w0 = w0 * M_PI;
    double beta = tan(bw / 2.0);
    double gain = 1.0 / (1.0 + beta);
    b[0] = gain;
    b[1] = gain * (-2.0 * cos(w0));
    b[2] = gain;
    a[0] = 1.0;
    a[1] = -2.0 * gain * cos(w0);
    a[2] = 2.0 * gain - 1.0;
}

// impulse response of the biquad (direct form II transposed, as scipy's lfilter),
// truncated where the remaining tail is below 3e-9 of the total
FirParams make_fir(double f0, double q, double fs) {
    double b[3], a[3];
    notch_coefficients(f0, q, fs, b, a);
    const int NMAX = 1 << 16;
    std::vector<double> h(NMAX);
    double z0 = 0.0, z1 = 0.0, x = 1.0;
    for (int i = 0; i < NMAX; ++i) {
        double y = b[0] * x + z0;
        z0 = b[1] * x - a[1] * y + z1;
        z1 = b[2] * x - a[2] * y;
        x = 0.0;
        h[i] = y;
    }
    double total = 0.0;
    for (double v : h) total += fabs(v);
    double tail = 0.0;
    int K = NMAX;
    while (K > 1 && tail + fabs(h[K - 1]) < 3e-9 * total) tail += fabs(h[--K]);
    if (K > kMaxFirTaps) {
        // too long for the FIR form: the recursion itself (float64, blocks with a warm-up of K samples)
        if (K >= NMAX)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "notch impulse response longer than %d samples: quality factor too high", NMAX);
        FirParams fp;
        memset(&fp, 0, sizeof(fp));
        fp.K = K;
        fp.iir = 1;
        fp.warm = K;
        for (int i = 0; i < 3; ++i) {
            fp.b[i] = b[i];
            fp.a[i] = a[i];
        }
        // lfilter_zi: steady state for a unit step, y = H(1)
        const double g1 = (b[0] + b[1] + b[2]) / (1.0 + a[1] + a[2]);
        fp.zi[1] = b[2] - a[2] * g1;
        fp.zi[0] = b[1] - a[1] * g1 + fp.zi[1];
        return fp;
    }
    FirParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.K = K;
    const int sizes[] = {16, 20, 24, 32, 48, 64};
    for (int s : sizes)
        if (K <= s) {
            fp.KP = s;
            break;
        }
    for (int i = 0; i < K; ++i) fp.h[i] = (float)h[i];
    for (int j = 0; j < fp.KP; ++j) fp.hr[j] = fp.h[fp.KP - 1 - j];
    // interior form: autocorrelation of the (untruncated) impulse response, cut where the rest is below fp32
    // resolution of the sum (1e-7 of the total; 12 taps each side for Q = 1)
    {
        const int GM = 256;
        std::vector<double> g(GM);
        double gtot = 0.0;
        for (int k = 0; k < GM; ++k) {
            double acc = 0.0;
            for (int m = 0; m + k < NMAX; ++m) acc += h[m] * h[m + k];
            g[k] = acc;
            gtot += (k ? 2.0 : 1.0) * fabs(acc);
        }
        double gtail = 0.0;
        int KG = GM - 1;
        while (KG > 1 && gtail + 2.0 * fabs(g[KG]) < 1e-7 * gtot) gtail += 2.0 * fabs(g[KG--]);
        fp.KC = 0;
        const int csizes[] = {8, 12, 16, 24, 32};
        for (int s : csizes)
            if (KG <= s) {
                fp.KC = s;
                break;
            }
        for (int k = 0; k <= fp.KC; ++k) fp.g[k] = (float)g[k];
    }
    return fp;
}

// the notch of a context rarely changes between calls: the 4096-step impulse response is computed once per (f0, Q)
const FirParams &cached_fir(wefax_ctx *ctx, double f0, double q) {
    if (!(ctx->fir_valid && ctx->fir_f0 == f0 && ctx->fir_q == q)) {
        ctx->fir_valid = false;
        ctx->fir = make_fir(f0, q, (double)WEFAX_TARGET_RATE);
        ctx->fir_f0 = f0;
        ctx->fir_q = q;
        ctx->fir_valid = true;
    }
    return ctx->fir;
}

void line_constants(double lpm, int sr, wefax_line_constants *o) {
    // Python: 1 / (lpm / 60); int(x * frame_len * sample_rate) evaluated left to right
    volatile double frame_len = 1.0 / (lpm / 60.0);
    volatile double t5 = 0.005 * frame_len;
    volatile double t1 = 0.001 * frame_len;
    volatile double f = frame_len * (double)sr;
    o->frame_len = frame_len;
    o->n1 = (int)(t5 * (double)sr);
    o->n0 = (int)(t1 * (double)sr);
    o->template_len = 2 * o->n1 + o->n0;
    o->mindistance = (int)(f * 0.8);
    o->width = (int)f;
    o->dev_min = f - 500.0;
    o->dev_max = f + 500.0;
}

void *pinned(wefax_ctx *ctx, size_t bytes) {
    if (bytes > ctx->pinned_cap) {
        if (ctx->pinned) cudaFreeHost(ctx->pinned);
        ctx->pinned = nullptr;
        ctx->pinned_cap = 0;
        CUDA_CHECK(cudaMallocHost(&ctx->pinned, bytes + 4096));
        ctx->pinned_cap = bytes + 4096;
    }
    return ctx->pinned;
}

constexpr long long kSegMinPiece = 64;   // shortest piece either side of a segment's seam

void use_device(wefax_ctx *ctx) { CUDA_CHECK(cudaSetDevice(ctx->device)); }

// The caller's PCM as a device pointer: pcm itself under WEFAX_F_PCM_ON_DEVICE, else a copy of its first `samples`
// samples staged in ctx->pcm.  Samples are int16, or float32 under WEFAX_F_PCM_FLOAT32, which only the batch decode
// takes (float_ok).
const void *upload_pcm(wefax_ctx *ctx, const void *pcm, size_t samples, unsigned flags, bool float_ok) {
    const bool f32 = flags & WEFAX_F_PCM_FLOAT32;
    if (f32 && !float_ok)
        WEFAX_THROW(WEFAX_ERR_INVALID, "WEFAX_F_PCM_FLOAT32: this entry point takes int16 samples only");
    if (flags & WEFAX_F_PCM_ON_DEVICE) return pcm;
    const size_t bytes = samples * (f32 ? sizeof(float) : sizeof(int16_t));
    void *buf = ctx->pcm.reserve(bytes);
    StageTimer timer(ctx, "h2d_pcm");
    CUDA_CHECK(cudaMemcpyAsync(buf, pcm, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return buf;
}

// What the notch reads: the uploaded PCM as it is, or the resampled float stream for input not at 11025 Hz.
// stride: samples from one recording to the next.
struct NotchInput {
    IngestMode mode;
    const void *x;
    size_t stride;
    // the input from sample i on (a stereo int16 frame and a float sample are 4 bytes each)
    const void *at(long long i) const { return (const char *)x + (size_t)i * (mode == kInMonoI16 ? 2 : 4); }
};

// desc: frames, channels, sample rate and sample type of the uploaded d_pcm; n: the length at 11025 Hz.  The
// resampler reserves work_z: take any scratch from work_z after this call.
NotchInput notch_input(wefax_ctx *ctx, const wefax_batch_desc &desc, const void *d_pcm, long long n, int batch) {
    const long long n_in = desc.n_frames;
    const bool f32 = desc.flags & WEFAX_F_PCM_FLOAT32;
    if (desc.sample_rate == WEFAX_TARGET_RATE)
        return NotchInput{f32 ? kInFloat : (desc.channels == 2 ? kInStereoI16 : kInMonoI16), d_pcm, (size_t)n_in};
    // (wefax.py:60-62)
    float *xin = (float *)ctx->resample_in.reserve(((size_t)batch * n_in + (size_t)batch * n) * sizeof(float));
    float *xrs = xin + (size_t)batch * n_in;
    const float *src = (const float *)d_pcm;   // already float: the resampler reads it in place
    if (!f32) {
        launch_ingest_float(ctx, (const int16_t *)d_pcm, (size_t)n_in, desc.channels, xin, (size_t)n_in, n_in, batch);
        src = xin;
    }
    resample_real(ctx, n_in, n, src, (size_t)n_in, xrs, (size_t)n, batch);
    return NotchInput{kInFloat, xrs, (size_t)n};
}

// Segment mode: grey map of the resident envelope into seg.dig with the percentiles in d_res, then the core's share of
// the optional outputs (no synchronisation)
void segment_grey_map(wefax_ctx *ctx, const RecResult *d_res, uint8_t *digitalized, float *demodulated) {
    cudaStream_t st = ctx->stream;
    const long long n = ctx->seg.n, lo = ctx->seg.core_lo, hi = ctx->seg.core_hi;
    uint8_t *d_dig = (uint8_t *)ctx->seg.dig.reserve((size_t)n);
    const float *d_env = ctx->seg.env.as<float>() + ctx->seg.base;
    launch_quantise(ctx, d_env, (size_t)n, d_dig, (size_t)n, n, 1, d_res, 0, n, st, "quantise");
    if (digitalized && hi > lo)
        CUDA_CHECK(cudaMemcpyAsync(digitalized, d_dig + lo, (size_t)(hi - lo), cudaMemcpyDefault, st));
    if (demodulated && hi > lo) {
        float *d_med = (float *)ctx->work_a.reserve((size_t)(hi - lo) * sizeof(float));
        launch_segment_median(ctx, d_env, n, lo, hi, d_med);
        CUDA_CHECK(cudaMemcpyAsync(demodulated, d_med, (size_t)(hi - lo) * sizeof(float), cudaMemcpyDefault, st));
    }
}

struct LineSet {
    std::vector<LineDev> lines;
    int max_width = 0, min_width = 1 << 30, min_mind = 1 << 30;
    long long raster_need = 0;
};

LineSet prepare_lines(const double *lpm, int nrec, long long n) {
    LineSet ls;
    ls.lines.resize(nrec);
    for (int r = 0; r < nrec; ++r) {
        if (!(lpm[r] > 0.0)) WEFAX_THROW(WEFAX_ERR_INVALID, "lines per minute must be positive");
        wefax_line_constants lc;
        line_constants(lpm[r], WEFAX_TARGET_RATE, &lc);
        if (lc.width < 1 || lc.template_len < 1 || lc.template_len > 2048 || lc.mindistance < 1024)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "lines per minute %g outside the supported range (4..500)", lpm[r]);
        ls.lines[r] = LineDev{lc.n1, lc.n0, lc.template_len, lc.mindistance, lc.width, lc.dev_min, lc.dev_max,
                              lc.width % 8 == 0 ? 2 : (lc.width % 4 == 0 ? 1 : 0), 0};
        ls.max_width = std::max(ls.max_width, lc.width);
        ls.min_width = std::min(ls.min_width, lc.width);
        ls.min_mind = std::min(ls.min_mind, lc.mindistance);
        ls.raster_need = std::max(ls.raster_need, 4 * (n / lc.width) * lc.width);
    }
    return ls;
}

// small per-recording results -> the caller's host arrays; rasters of host-output calls
void deliver_results(wefax_ctx *ctx, const RecResult *h_res, int g, int w0, const LineSet &ls,
                     const wefax_batch_out *out, const uint8_t *d_raster, size_t rs, bool out_dev) {
    bool copied = false;
    for (int r = 0; r < g; ++r) {
        const RecResult &rr = h_res[r];
        const int R = w0 + r;
        if (out->n_peaks) out->n_peaks[R] = rr.n_peaks;
        if (out->peaks) memcpy(out->peaks + (size_t)R * WEFAX_MAX_PEAKS, rr.peaks, sizeof(rr.peaks));
        if (out->n_phasing) out->n_phasing[R] = rr.n_phasing;
        if (out->phasing) memcpy(out->phasing + (size_t)R * WEFAX_MAX_PEAKS, rr.phasing, sizeof(rr.phasing));
        if (out->start_frame) out->start_frame[R] = rr.start_frame;
        if (out->height) out->height[R] = rr.height;
        if (out->status) out->status[R] = rr.status;
        if (out->low_high) {
            out->low_high[2 * R] = rr.low;
            out->low_high[2 * R + 1] = rr.high;
        }
        if (out->raster && !out_dev && rr.height > 0) {
            const size_t bytes = (size_t)rr.height * ls.lines[R].width;
            CUDA_CHECK(cudaMemcpyAsync(out->raster + (size_t)R * out->raster_stride, d_raster + (size_t)r * rs, bytes,
                                       cudaMemcpyDeviceToHost, ctx->stream));
            copied = true;
        }
    }
    if (copied) CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}


// Depth-first form of a batch (see wefax_ctx::max_wave).  Returns false when the batch should run breadth-first on
// the context itself: single recordings, working sets larger than the L2 cache, stage timing on (the per-stage
// event pairs belong to one stream), or WEFAX_DEPTH_FIRST=0.
bool decode_depth_first(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, const double *lpm,
                        const wefax_batch_out *out, long long n) {
    const int nrec = desc->n_recordings;
    if (ctx->is_lane || ctx->timing || ctx->depth_first == 0 || ctx->lanes < 1 || nrec < 2) return false;
    // Measured on B200 (profiles/bench_r02_lanes.md): with everything resident in HBM a lane is bound by its ~25
    // kernel launches per recording (the host, not the GPU), so device-resident batches stay breadth-first unless
    // WEFAX_DEPTH_FIRST=1 asks otherwise.  With HOST buffers the lanes are a copy / compute pipeline: the PCM of one
    // chunk goes up and the results of another come down while a third is in the kernels (1.7x end to end).
    const bool host_io = !(desc->flags & WEFAX_F_PCM_ON_DEVICE) || !(desc->flags & WEFAX_F_OUT_ON_DEVICE);
    int lane_wave = ctx->lane_wave;
    if (ctx->depth_first < 0) {
        if (!host_io || nrec < 2 * ctx->lanes) return false;
        if (!getenv("WEFAX_LANE_WAVE")) lane_wave = (int)std::max(1ll, std::min(16ll, (long long)nrec / (4 * ctx->lanes)));
    }
    (void)n;
    const int L = std::min(ctx->lanes, nrec);
    while ((int)ctx->lane_ctx.size() < L) {
        wefax_ctx *lane = nullptr;
        const int rc = wefax_ctx_create(ctx->device, nullptr, &lane);
        if (rc != WEFAX_OK) WEFAX_THROW(rc, "cannot create a decode lane on device %d", ctx->device);
        lane->is_lane = true;
        lane->workspace_limit = ctx->workspace_limit;
        ctx->lane_ctx.push_back(lane);
        cudaEvent_t e;
        CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->ev_lane_join.push_back(e);
    }
    if (!ctx->ev_lane_fork) CUDA_CHECK(cudaEventCreateWithFlags(&ctx->ev_lane_fork, cudaEventDisableTiming));
    // the lanes start after whatever the caller queued on the context's stream (e.g. the producer of a device PCM)
    CUDA_CHECK(cudaEventRecord(ctx->ev_lane_fork, ctx->stream));
    const size_t esz = (desc->flags & WEFAX_F_PCM_FLOAT32) ? sizeof(float) : sizeof(int16_t);
    const long long n_in = desc->n_frames;
    std::vector<int> rc(L, WEFAX_OK);
    std::vector<std::thread> threads;
    for (int l = 0; l < L; ++l) {
        const int r0 = (int)((long long)nrec * l / L), r1 = (int)((long long)nrec * (l + 1) / L);
        wefax_ctx *lane = ctx->lane_ctx[l];
        lane->max_wave = lane_wave;
        lane->use_fused = ctx->use_fused;
        threads.emplace_back([=, &rc] {
            cudaSetDevice(lane->device);
            if (cudaStreamWaitEvent(lane->stream, ctx->ev_lane_fork, 0) != cudaSuccess) {
                rc[l] = WEFAX_ERR_CUDA;
                return;
            }
            wefax_batch_desc d = *desc;
            d.n_recordings = r1 - r0;
            wefax_batch_out o = *out;
            const size_t R = (size_t)r0;
            if (o.audio) o.audio += R * (size_t)n;
            if (o.demodulated) o.demodulated += R * (size_t)n;
            if (o.digitalized) o.digitalized += R * (size_t)n;
            if (o.peaks) o.peaks += R * WEFAX_MAX_PEAKS;
            if (o.n_peaks) o.n_peaks += R;
            if (o.phasing) o.phasing += R * WEFAX_MAX_PEAKS;
            if (o.n_phasing) o.n_phasing += R;
            if (o.start_frame) o.start_frame += R;
            if (o.height) o.height += R;
            if (o.status) o.status += R;
            if (o.low_high) o.low_high += 2 * R;
            if (o.raster) o.raster += R * (size_t)o.raster_stride;
            const int16_t *p = (const int16_t *)((const char *)pcm + R * (size_t)n_in * (size_t)desc->channels * esz);
            rc[l] = wefax_decode_batch(lane, &d, p, lpm + r0, &o);
        });
    }
    for (auto &t : threads) t.join();
    for (int l = 0; l < L; ++l) {
        wefax_ctx *lane = ctx->lane_ctx[l];
        ctx->launches += lane->launches;
        lane->launches = 0;
        // (every lane call ends with a synchronisation of its stream; the event keeps the stream semantics explicit)
        CUDA_CHECK(cudaEventRecord(ctx->ev_lane_join[l], lane->stream));
        CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->ev_lane_join[l], 0));
    }
    for (int l = 0; l < L; ++l)
        if (rc[l] != WEFAX_OK) WEFAX_THROW(rc[l], "%s", ctx->lane_ctx[l]->last_error.c_str());
    return true;
}

// ---- slant search of the FM decode (DESIGN.md §4.7a; float64 restatement: tests/fm_slant_oracle.py) ----

constexpr int kSlantCoarseLines = 1024;

struct SlantGeometry {
    double Ls;
    int wb, D, Bn, wbb, R;
    long long L;   // whole lines in [from, image_end) at the longest allowed line
    int Lc;        // lines of the coarse stage
    int J;         // coarse candidates k = 2j, |j| <= J
};

SlantGeometry slant_geometry(double Ls, long long from, long long image_end, double max_ppm) {
    SlantGeometry s;
    s.Ls = Ls;
    s.wb = std::max(1, (int)llround(0.05 * Ls));
    s.D = std::max(1, (int)llround(s.wb / 16.0));
    s.Bn = (int)ceil(Ls / s.D);
    s.wbb = std::max(1, (int)llround((double)s.wb / s.D));
    s.R = 5 * s.D;
    const long long span = image_end - from;
    s.L = span > 0 ? (long long)floor((double)span / (Ls / (1.0 - max_ppm * 1e-6))) : 0;
    s.Lc = (int)std::min<long long>(s.L, kSlantCoarseLines);
    const int K = (int)ceil(max_ppm * 1e-6 * Ls * s.Lc / s.D);
    s.J = (K + 1) / 2;
    return s;
}

struct LineFit {
    double a = 0.0, s = 0.0, rms = 0.0;
    int used = 0;
};

void least_squares(const std::vector<double> &l, const std::vector<double> &y, double &a, double &s) {
    double ml = 0.0, my = 0.0;
    for (size_t i = 0; i < l.size(); ++i) {
        ml += l[i];
        my += y[i];
    }
    ml /= (double)l.size();
    my /= (double)l.size();
    double sxy = 0.0, sxx = 0.0;
    for (size_t i = 0; i < l.size(); ++i) {
        sxy += (l[i] - ml) * (y[i] - my);
        sxx += (l[i] - ml) * (l[i] - ml);
    }
    s = sxy / sxx;
    a = my - s * ml;
}

// least squares of pulse position against line index, then twice: drop |residual| > max(1, 3 * 1.4826 * MAD), refit.
// false: fewer than min_lines lines at some fit
bool robust_line_fit(std::vector<double> l, std::vector<double> y, int min_lines, LineFit &fit) {
    const size_t need = (size_t)std::max(2, min_lines);
    if (l.size() < need) return false;
    least_squares(l, y, fit.a, fit.s);
    for (int pass = 0; pass < 2; ++pass) {
        std::vector<double> r(l.size());
        for (size_t i = 0; i < l.size(); ++i) r[i] = fabs(y[i] - (fit.a + fit.s * l[i]));
        std::vector<double> sorted = r;
        std::sort(sorted.begin(), sorted.end());
        const size_t m = sorted.size();
        const double mad = (m & 1) ? sorted[m / 2] : 0.5 * (sorted[m / 2 - 1] + sorted[m / 2]);
        const double thr = std::max(1.0, 3.0 * 1.4826 * mad);
        size_t k = 0;
        for (size_t i = 0; i < l.size(); ++i)
            if (r[i] <= thr) {
                l[k] = l[i];
                y[k] = y[i];
                ++k;
            }
        l.resize(k);
        y.resize(k);
        if (k < need) return false;
        least_squares(l, y, fit.a, fit.s);
    }
    double ss = 0.0;
    for (size_t i = 0; i < l.size(); ++i) {
        const double r = y[i] - (fit.a + fit.s * l[i]);
        ss += r * r;
    }
    fit.used = (int)l.size();
    fit.rms = sqrt(ss / (double)l.size());
    return true;
}

// ---- FM decode: the stages every FM entry point shares ----

// the caller's slant parameters with their defaults filled in
wefax_fm_slant checked_slant(const wefax_fm_slant &slant) {
    wefax_fm_slant sp = slant;
    if (sp.mode == WEFAX_FM_SLANT_FIXED) {
        if (!(fabs(sp.ppm) <= 2000.0)) WEFAX_THROW(WEFAX_ERR_INVALID, "slant ppm must be within +-2000");
    } else if (sp.mode == WEFAX_FM_SLANT_AUTO) {
        if (sp.min_contrast == 0.0) sp.min_contrast = 0.3;
        if (sp.min_lines == 0) sp.min_lines = 8;
        if (!(sp.max_ppm > 0.0 && sp.max_ppm <= 2000.0))
            WEFAX_THROW(WEFAX_ERR_INVALID, "max_ppm must be in (0, 2000]");
        if (!(sp.min_contrast > 0.0 && sp.min_contrast <= 1.0) || sp.min_lines < 2)
            WEFAX_THROW(WEFAX_ERR_INVALID, "min_contrast must be in (0, 1] and min_lines >= 2");
    } else if (sp.mode != WEFAX_FM_SLANT_OFF) {
        WEFAX_THROW(WEFAX_ERR_INVALID, "unknown slant mode %d", sp.mode);
    }
    return sp;
}

// One picture's line lengths: the one FIXED uses (OFF: Ls) and the shortest one the mode may use, which sizes the
// picture to rows_max rows
struct FmGeometry {
    double Ls, Ls_fixed, Ls_min;
    int W, rows_max;
};

FmGeometry fm_geometry(double lpm, int ioc, const wefax_fm_slant &sp, long long from, long long image_end) {
    FmGeometry f;
    f.Ls = 60.0 / lpm * (double)WEFAX_TARGET_RATE;   // exact (fractional) samples per line
    f.W = (int)llround(M_PI * (double)ioc);
    f.Ls_fixed = sp.mode == WEFAX_FM_SLANT_FIXED ? f.Ls / (1.0 + sp.ppm * 1e-6) : f.Ls;
    f.Ls_min = sp.mode == WEFAX_FM_SLANT_AUTO ? f.Ls / (1.0 + sp.max_ppm * 1e-6) : f.Ls_fixed;
    f.rows_max = (int)std::max<long long>(0, (long long)floor((double)(image_end - from) / f.Ls_min));
    return f;
}

// The FM front end's layout for recordings of n samples at 11025 Hz: the real-input transform runs on the next even
// length npad = 2 * half_len whose half is smooth (zero padded).  zs, the row stride of the half-length spectrum, is
// even so that a batch takes the same fused Hilbert middle as one recording.
struct FmFront {
    long long n, half_len, npad, zs;
    FftPlan *half;
};

FmFront fm_front_plan(wefax_ctx *ctx, long long n) {
    FmFront f;
    f.n = n;
    f.half_len = next_smooth_length((n + 1) / 2);
    f.half = f.half_len > 0 ? get_plan(ctx, f.half_len) : nullptr;
    if (!f.half) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "no transform length for n=%lld", n);
    f.npad = 2 * f.half_len;
    f.zs = f.half_len + (f.half_len & 1);
    return f;
}

// Band-pass, analytic signal and discriminator of `batch` recordings (d_pcm: their uploaded PCM, desc as the caller's):
// the grey streams, rows of n samples at 11025 Hz, in g_out when it is not null (a device buffer), else in work_z
float *fm_front_end(wefax_ctx *ctx, const wefax_batch_desc &desc, const void *d_pcm, const wefax_fm_params &prm,
                    const FmFront &f, int batch, float *g_out) {
    cudaStream_t st = ctx->stream;
    const FirParams fp = make_bandpass_fir(prm.band_lo_hz, prm.band_hi_hz, (double)WEFAX_TARGET_RATE, prm.fir_taps);
    const long long n = f.n, npad = f.npad;
    float *x = (float *)ctx->work_a.reserve((size_t)batch * npad * sizeof(float));
    float *y = (float *)ctx->work_e.reserve((size_t)batch * npad * sizeof(float));
    if (npad > n)
        CUDA_CHECK(cudaMemset2DAsync(x + n, (size_t)npad * sizeof(float), 0, (size_t)(npad - n) * sizeof(float), batch, st));
    const NotchInput in = notch_input(ctx, desc, d_pcm, n, batch);
    launch_filtfilt(ctx, in.mode, in.x, in.stride, x, (size_t)npad, nullptr, 0, n, fp, batch);
    float2 *z = (float2 *)ctx->work_z.reserve((size_t)batch * f.zs * sizeof(float2));
    hilbert_envelope_real(ctx, f.half, x, (size_t)npad, z, (size_t)f.zs, y, (size_t)npad, batch, /*want_y=*/true);
    float *g = g_out ? g_out : (float *)ctx->work_z.reserve((size_t)batch * n * sizeof(float));
    launch_fm_grey(ctx, x, y, (size_t)npad, g, n, batch, prm.black_hz, prm.white_hz);
    return g;
}

// One chart of the picture stage: its recording's grey stream and its span in; its line start, rows, slant report and
// picture offset out
struct FmTail {
    const float *g;
    long long n, from, image_end;
    FmGeometry fg;
    bool picture;              // write its picture (rows_max rows at most)
    long long line_start = 0;
    int rows = 0;
    long long offset = 0;      // of its picture from d_img (fm_tail)
    wefax_fm_slant_out so;
    wefax_fm_levels_out lv;    // tuning offset (NOT_MEASURED unless the levels mode is AUTO)
};

// The picture stage of every chart in cs, each launch once over one chart table (DESIGN.md §4.7c):
//   AUTO: coarse sheared fold of each chart's first Lc lines, per-line pulse tracking, robust line fit (twice: Lc
//         lines, then all L lines from the first fit), three synchronisations for all charts together; a chart whose
//         search finds too few pulses or leaves +-max_ppm keeps its phasing line start (status NOT_FOUND);
//   the phasing fold of every chart without a fitted line; levels AUTO: every chart's black and white levels from its
//   line start (DESIGN.md §4.7d); one synchronisation for all line starts and levels;
//   packed picture offsets from d_img on (rows * W bytes each), each chart's tuning shift; one image launch.
// Returns the bytes of pictures written to d_img (device); the image launch may still be running.
long long fm_tail(wefax_ctx *ctx, std::vector<FmTail> &cs, const wefax_fm_params &prm, const wefax_fm_slant &sp,
                  const wefax_fm_levels &lv, uint8_t *d_img) {
    cudaStream_t st = ctx->stream;
    const int nc = (int)cs.size();
    if (nc == 0) return 0;
    const int fold_lines = prm.fold_lines;
    const bool levels = lv.mode == WEFAX_FM_LEVELS_AUTO;
    std::vector<FmChartJob> tab(nc);
    int max_lc = 0;
    for (int i = 0; i < nc; ++i) {
        FmTail &c = cs[i];
        FmChartJob &j = tab[i];
        memset(&c.lv, 0, sizeof(c.lv));
        c.lv.status = WEFAX_FM_LEVELS_NOT_MEASURED;
        memset(&j, 0, sizeof(j));
        j.g = c.g;
        j.n = c.n;
        j.from = c.from;
        j.image_end = c.image_end;
        j.Ls = c.fg.Ls_fixed;
        j.phase = 1;
        j.W = c.fg.W;
        max_lc = std::max(max_lc, (int)ceil(j.Ls));
        memset(&c.so, 0, sizeof(c.so));
        c.so.status = WEFAX_FM_SLANT_OK;
        if (sp.mode == WEFAX_FM_SLANT_FIXED) c.so.ppm = sp.ppm;
    }
    const size_t tab_bytes = ((size_t)nc * sizeof(FmChartJob) + 255) / 256 * 256;
    const size_t key_bytes = ((size_t)nc * sizeof(long long) + 255) / 256 * 256;
    const size_t lev_bytes = ((size_t)2 * nc * sizeof(FmLevel) + 255) / 256 * 256;
    char *dev = (char *)ctx->out_small.reserve(tab_bytes + 2 * key_bytes + lev_bytes +
                                               (size_t)nc * max_lc * sizeof(float));
    FmChartJob *d_tab = (FmChartJob *)dev;
    long long *d_ls = (long long *)(dev + tab_bytes);
    unsigned long long *d_best = (unsigned long long *)(dev + tab_bytes + key_bytes);
    FmLevel *d_lev = (FmLevel *)(dev + tab_bytes + 2 * key_bytes);
    float *P = (float *)(dev + tab_bytes + 2 * key_bytes + lev_bytes);
    // (pageable source: the copy is staged before the call returns, so the host table may change right after it)
    auto upload = [&] {
        CUDA_CHECK(cudaMemcpyAsync(d_tab, tab.data(), (size_t)nc * sizeof(FmChartJob), cudaMemcpyHostToDevice, st));
    };
    std::vector<long long> ls0(nc, 0);

    if (sp.mode == WEFAX_FM_SLANT_AUTO) {
        std::vector<SlantGeometry> sg(nc);
        std::vector<char> alive(nc, 0);
        long long q_total = 0, pos_total = 0;
        for (int i = 0; i < nc; ++i) {
            FmTail &c = cs[i];
            sg[i] = slant_geometry(c.fg.Ls, c.from, c.image_end, sp.max_ppm);
            c.so.status = WEFAX_FM_SLANT_NOT_FOUND;
            c.so.lines_total = (int)std::min<long long>(sg[i].L, INT32_MAX);
            if (sg[i].L < std::max(2, sp.min_lines) || sg[i].L > INT32_MAX) continue;
            alive[i] = 1;
            FmChartJob &j = tab[i];
            j.sLs = sg[i].Ls;
            j.D = sg[i].D;
            j.Bn = sg[i].Bn;
            j.wbb = sg[i].wbb;
            j.R = sg[i].R;
            j.swb = sg[i].wb;
            j.q_lines = sg[i].Lc;
            j.n_cand = 2 * sg[i].J + 1;
            j.q_off = q_total;
            j.pos_off = pos_total;
            q_total += (long long)sg[i].Lc * sg[i].Bn;
            pos_total += sg[i].L;
        }
        if (pos_total > 0) {
            const size_t q_bytes = ((size_t)q_total * sizeof(float) + 255) / 256 * 256;
            char *scratch = (char *)ctx->work_misc.reserve(q_bytes + (size_t)pos_total * (sizeof(long long) + sizeof(float)));
            float *Q = (float *)scratch;
            long long *d_pos = (long long *)(scratch + q_bytes);
            float *d_ctr = (float *)(d_pos + pos_total);
            upload();
            launch_fm_slant_profile(ctx, d_tab, tab.data(), nc, Q);
            launch_fm_slant_fold(ctx, d_tab, tab.data(), nc, Q, d_best);
            long long *h = (long long *)pinned(ctx, (size_t)std::max<long long>(nc, pos_total) * sizeof(long long) + 64);
            CUDA_CHECK(cudaMemcpyAsync(h, d_best, (size_t)nc * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            std::vector<double> a(nc, 0.0), s(nc, 0.0);
            std::vector<LineFit> fit(nc);
            for (int i = 0; i < nc; ++i) {
                if (!alive[i]) continue;
                const int rank = 0x7fffffff - (int)(unsigned)((unsigned long long)h[i] & 0xffffffffull);
                const int c = rank / sg[i].Bn, b = rank % sg[i].Bn;
                const int k = c == 0 ? 0 : ((c + 1) / 2) * 2 * ((c & 1) ? -1 : 1);
                a[i] = (double)(cs[i].from + (long long)b * sg[i].D);
                s[i] = sg[i].Ls + (double)k * sg[i].D / sg[i].Lc;
            }
            for (int pass = 0; pass < 2; ++pass) {
                for (int i = 0; i < nc; ++i) {
                    tab[i].track_lines = alive[i] ? (pass == 0 ? sg[i].Lc : (int)sg[i].L) : 0;
                    tab[i].a = a[i];
                    tab[i].s = s[i];
                }
                upload();
                launch_fm_slant_track(ctx, d_tab, tab.data(), nc, sp.min_contrast, d_pos, d_ctr);
                CUDA_CHECK(cudaMemcpyAsync(h, d_pos, (size_t)pos_total * sizeof(long long), cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaStreamSynchronize(st));
                for (int i = 0; i < nc; ++i) {
                    if (!alive[i]) continue;
                    std::vector<double> li, yi;
                    const long long *hp = h + tab[i].pos_off;
                    for (int l = 0; l < tab[i].track_lines; ++l)
                        if (hp[l] >= 0) {
                            li.push_back((double)l);
                            yi.push_back((double)hp[l]);
                        }
                    if (!robust_line_fit(std::move(li), std::move(yi), sp.min_lines, fit[i])) {
                        alive[i] = 0;
                        continue;
                    }
                    a[i] = fit[i].a;
                    s[i] = fit[i].s;
                }
            }
            for (int i = 0; i < nc; ++i) {
                tab[i].q_lines = tab[i].track_lines = 0;
                if (!alive[i]) continue;
                const double ppm = (sg[i].Ls / s[i] - 1.0) * 1e6;
                if (!(fabs(ppm) <= sp.max_ppm)) continue;
                wefax_fm_slant_out &so = cs[i].so;
                so.status = WEFAX_FM_SLANT_OK;
                so.line_length = s[i];
                so.ppm = ppm;
                so.first_line = a[i] - floor((a[i] - (double)cs[i].from) / s[i]) * s[i];
                so.lines_used = fit[i].used;
                so.residual_rms = fit[i].rms;
                ls0[i] = llround(so.first_line);
                tab[i].Ls = so.line_length;
                tab[i].phase = 0;
            }
        }
    }
    for (int i = 0; i < nc; ++i) {
        tab[i].Lc = (int)ceil(tab[i].Ls);
        tab[i].wb = std::max(1, (int)llround(0.05 * tab[i].Ls));
    }

    // line starts: the fitted ones as given, the others from the phasing fold
    upload();
    CUDA_CHECK(cudaMemcpyAsync(d_ls, ls0.data(), (size_t)nc * sizeof(long long), cudaMemcpyHostToDevice, st));
    launch_fm_phasing(ctx, d_tab, tab.data(), nc, fold_lines, P, d_ls);
    if (levels) launch_fm_levels(ctx, d_tab, nc, fold_lines, d_ls, d_lev);
    long long *h_ls = (long long *)pinned(ctx, (size_t)nc * sizeof(long long) + (size_t)2 * nc * sizeof(FmLevel) + 64);
    FmLevel *h_lev = (FmLevel *)(h_ls + nc);
    CUDA_CHECK(cudaMemcpyAsync(h_ls, d_ls, (size_t)nc * sizeof(long long), cudaMemcpyDeviceToHost, st));
    if (levels) CUDA_CHECK(cudaMemcpyAsync(h_lev, d_lev, (size_t)2 * nc * sizeof(FmLevel), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));

    // rows, packed offsets and tuning shifts, then every picture in one launch
    const double span = prm.white_hz - prm.black_hz;
    long long off = 0;
    for (int i = 0; i < nc; ++i) {
        FmTail &c = cs[i];
        const double line_length = tab[i].Ls;
        if (levels) {
            const FmLevel &body = h_lev[2 * i], &pulse = h_lev[2 * i + 1];
            const double b = body.value, w = pulse.value, delta = (b + w) / 2.0 - 0.5;
            wefax_fm_levels_out &o = c.lv;
            o.black_hz = prm.black_hz + b * span;
            o.white_hz = prm.black_hz + w * span;
            o.offset_hz = delta * span;
            o.black_samples = body.count;
            o.white_samples = pulse.count;
            const bool ok = body.count > 0 && pulse.count > 0 && w - b >= 0.75 && w - b <= 1.25 &&
                            fabs(o.offset_hz) <= lv.max_offset_hz;
            o.status = ok ? WEFAX_FM_LEVELS_OK : WEFAX_FM_LEVELS_NOT_FOUND;
            if (ok) tab[i].shift = (float)delta;
        }
        c.line_start = h_ls[i];
        c.rows = (int)std::min<long long>(
            c.fg.rows_max, std::max<long long>(0, (long long)floor((double)(c.image_end - c.line_start) / line_length)));
        if (tab[i].phase) {
            c.so.line_length = line_length;
            c.so.first_line = (double)c.line_start;
        }
        c.offset = off;
        tab[i].out = off;
        tab[i].rows_max = (d_img && c.picture) ? c.fg.rows_max : 0;
        if (tab[i].rows_max > 0) off += (long long)c.rows * c.fg.W;
    }
    if (off > 0) {
        upload();
        launch_fm_image(ctx, d_tab, tab.data(), nc, d_ls, d_img);
    }
    return off;
}

// ---- charts of a recording (DESIGN.md §4.7b; float64 restatement: tests/fm_charts_oracle.py) ----

int tone_class(const float *s) {   // s = (r_300, r_450, r_675, V) of one window
    int k = 0;
    for (int f = 1; f < 3; ++f)
        if (s[f] > s[k]) k = f;
    if (!(s[k] >= WEFAX_FM_TONE_MIN_RATIO && s[3] >= WEFAX_FM_TONE_MIN_VAR)) return WEFAX_FM_TONE_NONE;
    static const int cls[3] = {WEFAX_FM_TONE_START_576, WEFAX_FM_TONE_STOP, WEFAX_FM_TONE_START_288};
    return cls[k];
}

std::vector<wefax_fm_chart> find_charts(const std::vector<int> &cls, long long n) {
    std::vector<wefax_fm_chart> charts;
    const long long T = WEFAX_FM_TONE_WINDOW, nw = (long long)cls.size();
    bool open = false;
    for (long long k = 0; k < nw;) {
        long long e = k + 1;
        while (e < nw && cls[e] == cls[k]) ++e;
        const int c = cls[k];
        if (e - k >= WEFAX_FM_TONE_MIN_RUN && c != WEFAX_FM_TONE_NONE) {
            if (open) {
                charts.back().image_end = k * T;
                charts.back().stop_found = c == WEFAX_FM_TONE_STOP;
                open = false;
            }
            if (c != WEFAX_FM_TONE_STOP) {
                wefax_fm_chart ch;
                memset(&ch, 0, sizeof(ch));
                ch.tone_begin = k * T;
                ch.search_from = e * T;
                ch.ioc = c == WEFAX_FM_TONE_START_576 ? 576 : 288;
                ch.line_start = -1;
                charts.push_back(ch);
                open = true;
            }
        }
        k = e;
    }
    if (open) charts.back().image_end = n;
    return charts;
}

}  // namespace

extern "C" {

int wefax_abi_version(void) { return WEFAX_ABI_VERSION; }

int wefax_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

int wefax_ctx_create(int device, void *stream, wefax_ctx **out) {
    if (!out) return WEFAX_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
        (void)cudaGetLastError();
        return WEFAX_ERR_CUDA;   // no CUDA device: there is no CPU fallback
    }
    wefax_ctx *ctx = new (std::nothrow) wefax_ctx();
    if (!ctx) return WEFAX_ERR_NOMEM;
    int rc = guarded(ctx, [&] {
        ctx->device = device;
        use_device(ctx);
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "built for sm_100a (Blackwell); device %d is sm_%d%d", device, prop.major,
                        prop.minor);
        ctx->sm_count = prop.multiProcessorCount;
        if (const char *gr = getenv("WEFAX_GRAPH")) ctx->use_graph = gr[0] != '0';
        if (const char *df = getenv("WEFAX_DEPTH_FIRST")) ctx->depth_first = atoi(df) != 0 ? 1 : 0;
        if (const char *ln = getenv("WEFAX_LANES")) ctx->lanes = std::max(1, std::min(8, atoi(ln)));
        if (const char *lw = getenv("WEFAX_LANE_WAVE")) ctx->lane_wave = std::max(1, atoi(lw));
        const char *fused = getenv("WEFAX_FUSED");   // WEFAX_FUSED=0: separate grey-map and raster kernels
        ctx->use_fused = !(fused && fused[0] == '0');
        int prio_least = 0, prio_greatest = 0;
        CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
        if (stream) {
            ctx->stream = (cudaStream_t)stream;
        } else {
            // highest priority: its small latency-bound kernels get SM slots before other work on the device
            CUDA_CHECK(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_greatest));
            ctx->own_stream = true;
        }
    });
    if (rc != WEFAX_OK) {
        delete ctx;
        return rc;
    }
    *out = ctx;
    return WEFAX_OK;
}

void wefax_ctx_destroy(wefax_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    for (wefax_ctx *lane : ctx->lane_ctx) wefax_ctx_destroy(lane);
    ctx->lane_ctx.clear();
    if (ctx->ev_lane_fork) cudaEventDestroy(ctx->ev_lane_fork);
    for (cudaEvent_t e : ctx->ev_lane_join) cudaEventDestroy(e);
    ctx->plans.clear();
    ctx->bluestein.clear();
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->pinned_up) cudaFreeHost(ctx->pinned_up);
    for (auto &sp : ctx->spans) {
        cudaEventDestroy(sp.e0);
        cudaEventDestroy(sp.e1);
    }
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *wefax_last_error(const wefax_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }

int wefax_ctx_sync(wefax_ctx *ctx) {
    return guarded(ctx, [&] {
        use_device(ctx);
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    }, false);
}

void *wefax_ctx_stream(wefax_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
long long wefax_ctx_launch_count(const wefax_ctx *ctx) { return ctx ? ctx->launches : 0; }

int wefax_ctx_set_workspace_limit(wefax_ctx *ctx, long long bytes) {
    if (!ctx || bytes < (1ll << 20)) return WEFAX_ERR_INVALID;
    ctx->workspace_limit = bytes;
    return WEFAX_OK;
}

int wefax_ctx_enable_timing(wefax_ctx *ctx, int enable) {
    if (!ctx) return WEFAX_ERR_INVALID;
    ctx->timing = enable != 0;
    return WEFAX_OK;
}

// Resolves the pending event pairs and writes "name total_ms launches\n" lines
// (accumulated since the last reset) into buf.
int wefax_ctx_timings(wefax_ctx *ctx, char *buf, long long buf_len, int reset) {
    if (!ctx || !buf || buf_len < 1) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        use_device(ctx);
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        for (auto &sp : ctx->spans) {
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, sp.e0, sp.e1));
            auto &acc = ctx->stage_ms[sp.name];
            acc.first += ms;
            acc.second += 1;
            ctx->event_pool.push_back(sp.e0);
            ctx->event_pool.push_back(sp.e1);
        }
        ctx->spans.clear();
        std::string out;
        for (auto &kv : ctx->stage_ms) {
            char line[128];
            snprintf(line, sizeof(line), "%s %.6f %lld\n", kv.first.c_str(), kv.second.first, kv.second.second);
            out += line;
        }
        if ((long long)out.size() + 1 > buf_len) WEFAX_THROW(WEFAX_ERR_INVALID, "timing buffer too small");
        memcpy(buf, out.c_str(), out.size() + 1);
        if (reset) ctx->stage_ms.clear();
    }, false);
}

int wefax_line_constants_for(double lpm, int sample_rate, wefax_line_constants *out) {
    if (!out || !(lpm > 0.0) || sample_rate <= 0) return WEFAX_ERR_INVALID;
    line_constants(lpm, sample_rate, out);
    return WEFAX_OK;
}

long long wefax_resampled_length(long long n_frames, int sample_rate) {
    volatile double length = (double)n_frames / (double)sample_rate;
    return (long long)((double)WEFAX_TARGET_RATE * length);
}

int wefax_notch_coefficients(double f0, double q, double fs, double b[3], double a[3]) {
    return guarded(nullptr, [&] { notch_coefficients(f0, q, fs, b, a); });
}

int wefax_fft_plan_describe(long long n, int *n_passes, int pass_len[8], long long *bluestein_len) {
    if (n < 1 || !n_passes || !pass_len || !bluestein_len) return WEFAX_ERR_INVALID;
    std::vector<int> Rs;
    long long m = 0;
    if (!plan_factors(n, Rs)) {
        m = next_smooth_length(2 * n - 1);
        if (m <= 0 || !plan_factors(m, Rs)) return WEFAX_ERR_UNSUPPORTED;
    }
    *bluestein_len = m;
    *n_passes = (int)Rs.size();
    for (int i = 0; i < 8; ++i) pass_len[i] = i < (int)Rs.size() ? Rs[i] : 0;
    return WEFAX_OK;
}

// ---------------------------------------------------------------------------
int wefax_decode_batch(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, const double *lpm,
                       const wefax_batch_out *out) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!desc || !pcm || !lpm || !out) WEFAX_THROW(WEFAX_ERR_INVALID, "null argument");
        const int nrec = desc->n_recordings;
        const long long n_in = desc->n_frames;
        const int ch = desc->channels;
        if (nrec < 1 || n_in < 1 || (ch != 1 && ch != 2) || desc->sample_rate <= 0)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad batch description");
        // ---- replay of the CUDA graph of the previous, identical call (see wefax_ctx::graph_exec): decided before any
        // other host work - the GPU idles for as long as the host takes between two replays
        auto graph_key_of = [&]() {
            std::vector<unsigned long long> key = {
                (unsigned long long)nrec, (unsigned long long)n_in, (unsigned long long)ch, (unsigned long long)desc->sample_rate,
                (unsigned long long)desc->flags, (unsigned long long)(uintptr_t)pcm, (unsigned long long)(uintptr_t)out->audio,
                (unsigned long long)(uintptr_t)out->demodulated, (unsigned long long)(uintptr_t)out->digitalized,
                (unsigned long long)(uintptr_t)out->raster, (unsigned long long)out->raster_stride,
                (unsigned long long)ctx->workspace_limit};
            auto bits = [](double v) { unsigned long long u; memcpy(&u, &v, sizeof(u)); return u; };
            key.reserve(key.size() + 2 + (size_t)nrec);
            key.push_back(bits(desc->notch_freq));
            key.push_back(bits(desc->notch_q));
            for (int r = 0; r < nrec; ++r) key.push_back(bits(lpm[r]));
            return key;
        };
        if (ctx->graph_exec && !ctx->timing && ctx->api_calls == ctx->graph_epoch + 1 && ctx->stream) {
            if (graph_key_of() == ctx->graph_key) {
                use_device(ctx);
                CUDA_CHECK(cudaGraphLaunch(ctx->graph_exec, ctx->stream));
                ctx->launches += ctx->graph_launches;
                ctx->graph_epoch = ctx->api_calls;
                CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
                deliver_results(ctx, (const RecResult *)ctx->graph_h_res, nrec, 0, LineSet(), out, nullptr, 0, true);
                return;
            }
        }
        const bool resample = desc->sample_rate != WEFAX_TARGET_RATE;
        const long long n = resample ? wefax_resampled_length(n_in, desc->sample_rate) : n_in;
        if (n <= 9)
            WEFAX_THROW(WEFAX_ERR_INVALID, "The length of the input vector x must be greater than padlen, which is 9.");
        if (n_in >= (1ll << 31) - 4096 || n >= (1ll << 31) - 4096) WEFAX_THROW(WEFAX_ERR_INVALID, "recording too long");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        if (decode_depth_first(ctx, desc, pcm, lpm, out, n)) return;
        const bool pcm_dev = desc->flags & WEFAX_F_PCM_ON_DEVICE;
        const bool out_dev = desc->flags & WEFAX_F_OUT_ON_DEVICE;
        // float32 samples (the host side of WAV formats other than 16-bit PCM: int32 / 24-bit / float, wefax.py:349)
        const bool pcm_f32 = desc->flags & WEFAX_F_PCM_FLOAT32;
        if (pcm_f32 && ch != 1) WEFAX_THROW(WEFAX_ERR_INVALID, "float32 input must be mono (merge the channels on the host)");
        const size_t esz = pcm_f32 ? sizeof(float) : sizeof(int16_t);

        // wefax.py:63: the frequency goes through int()
        const FirParams &fp = cached_fir(ctx, (double)(long long)desc->notch_freq, desc->notch_q);

        const LineSet ls = prepare_lines(lpm, nrec, n);
        const std::vector<LineDev> &lines = ls.lines;
        const int max_width = ls.max_width, min_width = ls.min_width, min_mind = ls.min_mind;
        const long long raster_cap = 4 * n;   // >= 4 * (n / w) * w for every w
        const long long rstride_user = out->raster_stride;
        if (out->raster && rstride_user < ls.raster_need)
            WEFAX_THROW(WEFAX_ERR_INVALID, "raster_stride %lld too small (need %lld)", rstride_user, ls.raster_need);

        // transform scratch per recording
        const EnvelopeForm form = envelope_form(ctx, n);
        long long zlen_rs = 0;
        if (resample) {
            std::vector<int> tmp;
            long long a = plan_factors(n_in, tmp) ? n_in : next_smooth_length(2 * n_in - 1);
            zlen_rs = std::max(a, form.zlen);
        }
        const long long per_rec = (pcm_dev ? 0 : n_in * ch * (long long)esz) + (resample ? n_in * 4 + (n_in + n) * 8 : 0) +
                                  std::max(form.zlen, zlen_rs) * 8 + n * (4 + 4 + 4 + 1 + 4) + 4096;
        int wave = (int)std::max<long long>(1, std::min<long long>(nrec, ctx->workspace_limit / per_rec));
        wave = std::min(wave, 32768);
        if (ctx->max_wave > 0) wave = std::min(wave, ctx->max_wave);

        LineDev *d_lines = (LineDev *)ctx->out_small.reserve((sizeof(LineDev) + sizeof(RecResult)) * (size_t)wave +
                                                             sizeof(SelState) * (size_t)wave + 256);
        RecResult *d_res = (RecResult *)(d_lines + wave);
        SelState *d_sel = (SelState *)(((uintptr_t)(d_res + wave) + 255) & ~(uintptr_t)255);
        RecResult *h_res = (RecResult *)pinned(ctx, sizeof(RecResult) * (size_t)wave + sizeof(LineDev) * (size_t)wave);
        LineDev *h_lines = (LineDev *)(h_res + wave);

        uint8_t *d_raster = nullptr;
        size_t rs = 0;
        // everything of one wave up to (not including) the final synchronisation: asynchronous work on `st` only
        auto issue_wave = [&](int w0, int g) {
            // ---- inputs ------------------------------------------------------------
            const void *d_pcm = upload_pcm(ctx, (const char *)pcm + (size_t)w0 * n_in * ch * esz, (size_t)g * n_in * ch,
                                           desc->flags, true);
            memcpy(h_lines, lines.data() + w0, sizeof(LineDev) * g);
            CUDA_CHECK(cudaMemcpyAsync(d_lines, h_lines, sizeof(LineDev) * g, cudaMemcpyHostToDevice, st));
            CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult) * g, st));
            const SyncPlan splan = prepare_sync(ctx, lines.data() + w0, g, n);   // (asynchronous upload from pinned staging)
            // the phasing search's scratch is cleared among the first operations of the wave instead of between two
            // latency-bound kernels
            clear_sync_scratch(ctx, splan, g);

            float *d_env = (float *)ctx->work_e.reserve((size_t)g * n * sizeof(float));
            uint8_t *d_dig = (out_dev && out->digitalized) ? out->digitalized + (size_t)w0 * n
                                                           : (uint8_t *)ctx->out_dig.reserve((size_t)g * n);
            rs = out_dev ? (size_t)rstride_user : (size_t)raster_cap;
            d_raster = nullptr;
            if (out->raster)
                d_raster = out_dev ? out->raster + (size_t)w0 * rs : (uint8_t *)ctx->out_raster.reserve((size_t)g * rs);

            // ---- resample (wefax.py:60-62) + zero-phase notch (wefax.py:63-72) -------
            // The notch writes the float audio_data where the caller wants it or the envelope's form reads it, and
            // the complex copy (x, 0) where the form is the full-length complex transform.
            const bool need_audio = out->audio != nullptr || !form.plan;
            float *d_audio = nullptr;
            if (need_audio)
                d_audio = (out_dev && out->audio) ? out->audio + (size_t)w0 * n
                                                  : (float *)ctx->work_a.reserve((size_t)g * n * sizeof(float));
            const NotchInput in = notch_input(ctx, *desc, d_pcm, n, g);
            float2 *z = envelope_scratch(ctx, form, g);
            launch_filtfilt(ctx, in.mode, in.x, in.stride, d_audio, (size_t)n, form.plan ? z : nullptr, (size_t)n, n, fp, g);
            // ---- analytic-signal envelope (wefax.py:174) ------------------------------
            launch_envelope(ctx, form, d_audio, (size_t)n, z, d_env, (size_t)n, g);
            // ---- median-5, percentiles, grey map (wefax.py:175,196-200) ---------------
            const bool fused = d_raster && ctx->use_fused;
            GreyTable *d_tab = fused ? (GreyTable *)ctx->grey_tab.reserve(sizeof(GreyTable) * (size_t)g) : nullptr;
            const bool have_table = launch_percentiles(ctx, d_env, (size_t)n, n, g, d_sel, d_res, 5, d_tab);
            if (fused) {
                // fused demod-to-pixel path: grey levels of the head for the phasing search (wefax.py:218-294),
                // then ONE sweep over the envelope writes digitalized_data and the raster (wefax.py:296-327)
                // (the threshold table is first read by the search's sequential fallback; the percentile stage may have
                //  left it behind already)
                if (!have_table) launch_grey_table(ctx, d_res, d_tab, g);
                const long long head = sync_head(splan, n);
                launch_quantise(ctx, d_env, (size_t)n, d_dig, (size_t)n, n, g, d_res, 0, head, st, "quantise_head");
                LazyGrey lazy;
                lazy.env = d_env;
                lazy.es = (size_t)n;
                lazy.tables = d_tab;
                lazy.valid = head;
                launch_sync_search(ctx, d_dig, (size_t)n, n, g, d_lines, d_res, min_mind, splan, lazy);
                launch_grey_raster(ctx, d_env, (size_t)n, out->digitalized ? d_dig : nullptr, (size_t)n, d_raster, rs, n, g,
                                   d_lines, lines.data() + w0, d_res, d_tab);
            } else {
                launch_quantise(ctx, d_env, (size_t)n, d_dig, (size_t)n, n, g, d_res, 0, n, st, "quantise");
                // ---- phasing search (wefax.py:218-294) and raster (wefax.py:296-327) -----
                launch_sync_search(ctx, d_dig, (size_t)n, n, g, d_lines, d_res, min_mind, splan);
                if (d_raster)
                    launch_raster(ctx, d_dig, (size_t)n, n, g, d_lines, d_res, d_raster, rs, max_width, (int)(n / min_width));
            }
            float *d_demod = nullptr;
            if (out->demodulated) {
                d_demod = out_dev ? out->demodulated + (size_t)w0 * n
                                  : (float *)ctx->work_z.reserve((size_t)g * n * sizeof(float));
                launch_median5(ctx, d_env, (size_t)n, d_demod, (size_t)n, n, g);
            }

            // ---- results ---------------------------------------------------------------
            CUDA_CHECK(cudaMemcpyAsync(h_res, d_res, sizeof(RecResult) * g, cudaMemcpyDeviceToHost, st));
            if (!out_dev) {
                StageTimer timer(ctx, "d2h_outputs");
                if (out->audio)
                    CUDA_CHECK(cudaMemcpyAsync(out->audio + (size_t)w0 * n, d_audio, (size_t)g * n * sizeof(float),
                                               cudaMemcpyDeviceToHost, st));
                if (out->demodulated)
                    CUDA_CHECK(cudaMemcpyAsync(out->demodulated + (size_t)w0 * n, d_demod, (size_t)g * n * sizeof(float),
                                               cudaMemcpyDeviceToHost, st));
                if (out->digitalized)
                    CUDA_CHECK(cudaMemcpyAsync(out->digitalized + (size_t)w0 * n, d_dig, (size_t)g * n,
                                               cudaMemcpyDeviceToHost, st));
            }
        };

        // ---- CUDA graph of a device-resident single-wave decode (see wefax_ctx::graph_exec) --------------------
        const bool graphable = ctx->use_graph && !ctx->graph_failed && pcm_dev && out_dev && wave >= nrec && !ctx->timing &&
                               out->raster && ctx->use_fused && !ctx->is_lane && st != nullptr;
        if (graphable) {
            std::vector<unsigned long long> key = graph_key_of();
            // (an identical call right after the one that captured the graph was answered at the top of this function)
            if (ctx->graph_exec) {
                cudaGraphExecDestroy(ctx->graph_exec);
                ctx->graph_exec = nullptr;
            }
            if (ctx->api_calls == ctx->graph_cand_epoch + 1 && key == ctx->graph_candidate) {
                // second identical call in a row: every scratch buffer has its size, capture this one
                const long long launches0 = ctx->launches;
                cudaGraph_t graph = nullptr;
                bool ok = cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) == cudaSuccess;
                if (ok) {
                    try {
                        issue_wave(0, nrec);
                    } catch (...) {
                        ok = false;
                    }
                    if (cudaStreamEndCapture(st, &graph) != cudaSuccess || !graph) ok = false;
                }
                if (ok && cudaGraphInstantiate(&ctx->graph_exec, graph, 0) != cudaSuccess) ok = false;
                if (graph) cudaGraphDestroy(graph);
                if (ok) {
                    ctx->graph_launches = ctx->launches - launches0;
                    ctx->graph_key = key;
                    ctx->graph_h_res = h_res;
                    CUDA_CHECK(cudaGraphLaunch(ctx->graph_exec, st));
                    ctx->graph_epoch = ctx->api_calls;
                    CUDA_CHECK(cudaStreamSynchronize(st));
                    deliver_results(ctx, h_res, nrec, 0, ls, out, nullptr, 0, true);
                    return;
                }
                // capture is not possible here (e.g. a launch the driver cannot record): stay eager on this context
                (void)cudaGetLastError();
                ctx->graph_exec = nullptr;
                ctx->graph_failed = true;
                ctx->launches = launches0;
            } else {
                ctx->graph_candidate = key;
                ctx->graph_cand_epoch = ctx->api_calls;
            }
        }

        for (int w0 = 0; w0 < nrec; w0 += wave) {
            const int g = std::min(wave, nrec - w0);
            issue_wave(w0, g);
            CUDA_CHECK(cudaStreamSynchronize(st));
            deliver_results(ctx, h_res, g, w0, ls, out, d_raster, rs, out_dev);
        }
    });
}

// ---------------------------------------------------------------------------
// stage-level entry points (host pointers)
// ---------------------------------------------------------------------------
int wefax_fft_c2c(wefax_ctx *ctx, long long n, int batch, const float *in, float *out, int inverse) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || batch < 1 || !in || !out) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        FftPlan *plan = get_plan(ctx, n);
        if (!plan) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "n=%lld has a prime factor > 13 (Bluestein is used on the decode path)", n);
        const size_t bytes = (size_t)n * batch * sizeof(float2);
        float2 *a = (float2 *)ctx->work_z.reserve(bytes * 2);
        float2 *scratch = a + (size_t)n * batch;
        float2 *o = (float2 *)ctx->work_misc.reserve(bytes);
        CUDA_CHECK(cudaMemcpyAsync(a, in, bytes, cudaMemcpyHostToDevice, ctx->stream));
        fft_c2c_natural(ctx, plan, a, o, scratch, batch, inverse != 0);
        CUDA_CHECK(cudaMemcpyAsync(out, o, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    });
}

int wefax_hilbert_envelope(wefax_ctx *ctx, long long n, int batch, const float *x, float *env) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || batch < 1 || !x || !env) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        const size_t bytes = (size_t)n * batch * sizeof(float);
        float *dx = (float *)ctx->work_a.reserve(bytes);
        float *de = (float *)ctx->work_e.reserve(bytes);
        CUDA_CHECK(cudaMemcpyAsync(dx, x, bytes, cudaMemcpyHostToDevice, ctx->stream));
        const EnvelopeForm form = envelope_form(ctx, n);
        float2 *z = envelope_scratch(ctx, form, batch);
        std::vector<float2> xz;
        if (form.plan) {
            // the complex form reads (x, 0), as the decode's notch writes it
            xz.assign((size_t)n * batch, make_float2(0.f, 0.f));
            for (size_t i = 0; i < xz.size(); ++i) xz[i].x = x[i];
            CUDA_CHECK(cudaMemcpyAsync(z, xz.data(), xz.size() * sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));
        }
        launch_envelope(ctx, form, dx, (size_t)n, z, de, (size_t)n, batch);
        CUDA_CHECK(cudaMemcpyAsync(env, de, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    });
}

int wefax_resample(wefax_ctx *ctx, long long n, long long num, int batch, const float *x, float *y) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || num < 1 || batch < 1 || !x || !y) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        float *dx = (float *)ctx->work_a.reserve((size_t)n * batch * sizeof(float));
        float *dy = (float *)ctx->work_e.reserve((size_t)num * batch * sizeof(float));
        CUDA_CHECK(cudaMemcpyAsync(dx, x, (size_t)n * batch * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        resample_real(ctx, n, num, dx, (size_t)n, dy, (size_t)num, batch);
        CUDA_CHECK(cudaMemcpyAsync(y, dy, (size_t)num * batch * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    });
}

int wefax_filtfilt(wefax_ctx *ctx, long long n, int batch, double notch_freq, double notch_q, const float *x,
                   float *y) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || batch < 1 || !x || !y) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        if (n <= 9)
            WEFAX_THROW(WEFAX_ERR_INVALID, "The length of the input vector x must be greater than padlen, which is 9.");
        use_device(ctx);
        const FirParams fp = make_fir(notch_freq, notch_q, (double)WEFAX_TARGET_RATE);
        const size_t bytes = (size_t)n * batch * sizeof(float);
        float *dx = (float *)ctx->work_a.reserve(bytes);
        float *dy = (float *)ctx->work_e.reserve(bytes);
        CUDA_CHECK(cudaMemcpyAsync(dx, x, bytes, cudaMemcpyHostToDevice, ctx->stream));
        launch_filtfilt(ctx, kInFloat, dx, (size_t)n, dy, (size_t)n, nullptr, 0, n, fp, batch);
        CUDA_CHECK(cudaMemcpyAsync(y, dy, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    });
}

int wefax_digitalize(wefax_ctx *ctx, long long n, int batch, const float *envelope, float *demodulated,
                     uint8_t *digitalized, double *low_high, int32_t *status) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || batch < 1 || !envelope) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const size_t bytes = (size_t)n * batch * sizeof(float);
        float *de = (float *)ctx->work_e.reserve(bytes);
        float *dm = (float *)ctx->work_a.reserve(bytes);
        uint8_t *dd = (uint8_t *)ctx->out_dig.reserve((size_t)n * batch);
        RecResult *d_res = (RecResult *)ctx->out_small.reserve((sizeof(RecResult) + sizeof(SelState)) * (size_t)batch + 256);
        SelState *d_sel = (SelState *)(((uintptr_t)(d_res + batch) + 255) & ~(uintptr_t)255);
        RecResult *h_res = (RecResult *)pinned(ctx, sizeof(RecResult) * (size_t)batch);
        CUDA_CHECK(cudaMemcpyAsync(de, envelope, bytes, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult) * batch, st));
        launch_percentiles(ctx, de, (size_t)n, n, batch, d_sel, d_res);
        launch_quantise(ctx, de, (size_t)n, dd, (size_t)n, n, batch, d_res, 0, n, ctx->stream, "quantise");
        if (demodulated) {
            launch_median5(ctx, de, (size_t)n, dm, (size_t)n, n, batch);
            CUDA_CHECK(cudaMemcpyAsync(demodulated, dm, bytes, cudaMemcpyDeviceToHost, st));
        }
        if (digitalized) CUDA_CHECK(cudaMemcpyAsync(digitalized, dd, (size_t)n * batch, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(h_res, d_res, sizeof(RecResult) * batch, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (int r = 0; r < batch; ++r) {
            if (low_high) {
                low_high[2 * r] = h_res[r].low;
                low_high[2 * r + 1] = h_res[r].high;
            }
            if (status) status[r] = h_res[r].status;
        }
    });
}

int wefax_sync_raster(wefax_ctx *ctx, long long n, int batch, const uint8_t *digitalized, const double *lpm,
                      const wefax_batch_out *out) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (n < 1 || batch < 1 || !digitalized || !lpm || !out) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const LineSet ls = prepare_lines(lpm, batch, n);
        if (out->raster && out->raster_stride < ls.raster_need)
            WEFAX_THROW(WEFAX_ERR_INVALID, "raster_stride %lld too small (need %lld)", out->raster_stride, ls.raster_need);
        uint8_t *dd = (uint8_t *)ctx->out_dig.reserve((size_t)n * batch);
        LineDev *d_lines = (LineDev *)ctx->out_small.reserve((sizeof(LineDev) + sizeof(RecResult)) * (size_t)batch);
        RecResult *d_res = (RecResult *)(d_lines + batch);
        RecResult *h_res = (RecResult *)pinned(ctx, sizeof(RecResult) * (size_t)batch);
        const size_t rs = (size_t)(4 * n);
        uint8_t *d_raster = out->raster ? (uint8_t *)ctx->out_raster.reserve((size_t)batch * rs) : nullptr;
        CUDA_CHECK(cudaMemcpyAsync(dd, digitalized, (size_t)n * batch, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(d_lines, ls.lines.data(), sizeof(LineDev) * batch, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult) * batch, st));
        const SyncPlan splan = prepare_sync(ctx, ls.lines.data(), batch, n);
        clear_sync_scratch(ctx, splan, batch);
        launch_sync_search(ctx, dd, (size_t)n, n, batch, d_lines, d_res, ls.min_mind, splan);
        if (d_raster)
            launch_raster(ctx, dd, (size_t)n, n, batch, d_lines, d_res, d_raster, rs, ls.max_width, (int)(n / ls.min_width));
        CUDA_CHECK(cudaMemcpyAsync(h_res, d_res, sizeof(RecResult) * batch, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        deliver_results(ctx, h_res, batch, 0, ls, out, d_raster, rs, false);
    });
}

// ---------------------------------------------------------------------------
// segment mode: one long recording as overlapping segments, one per context / GPU
// (SURVEY.md 8(e); host protocol in wefax_b200/segments.py)
// ---------------------------------------------------------------------------
int wefax_segment_envelope(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, long long n_resampled,
                           long long seam, long long core_begin, long long core_end) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!desc || !pcm) WEFAX_THROW(WEFAX_ERR_INVALID, "null argument");
        const long long n_in = desc->n_frames;
        const int ch = desc->channels;
        if (desc->n_recordings != 1 || n_in < 1 || (ch != 1 && ch != 2) || desc->sample_rate <= 0)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad segment description");
        const bool resample = desc->sample_rate != WEFAX_TARGET_RATE;
        // the planner's exact length (cut points fall on whole 11025-Hz samples); 0: the reference's formula
        const long long n = !resample ? n_in : (n_resampled > 0 ? n_resampled : wefax_resampled_length(n_in, desc->sample_rate));
        if (!resample && n_resampled > 0 && n_resampled != n_in)
            WEFAX_THROW(WEFAX_ERR_INVALID, "n_resampled %lld != n_frames %lld at 11025 Hz", n_resampled, n_in);
        if (n <= 9)
            WEFAX_THROW(WEFAX_ERR_INVALID, "The length of the input vector x must be greater than padlen, which is 9.");
        if (n_in >= (1ll << 31) - 4096 || n >= (1ll << 31) - 4096) WEFAX_THROW(WEFAX_ERR_INVALID, "segment too long");
        if (core_begin < 0 || core_end < core_begin || core_end > n)
            WEFAX_THROW(WEFAX_ERR_INVALID, "core [%lld, %lld) outside the extended segment of %lld samples", core_begin,
                        core_end, n);
        // The recording's end meets its start at `seam` (circular halo of the first / last segment): the
        // transforms see the junction exactly as the whole-recording circular transforms do, while the notch
        // and the median treat the two sides as the two ends of the recording they are.
        if (seam < 0 || seam >= n || (seam > 0 && (seam <= kSegMinPiece || n - seam <= kSegMinPiece)))
            WEFAX_THROW(WEFAX_ERR_INVALID, "seam %lld outside the extended segment of %lld samples", seam, n);
        if (seam > 0 && !(seam <= core_begin || core_end <= seam))
            WEFAX_THROW(WEFAX_ERR_INVALID, "core [%lld, %lld) straddles the seam %lld", core_begin, core_end, seam);
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        ctx->seg.have_env = ctx->seg.have_dig = false;
        const FirParams &fp = cached_fir(ctx, (double)(long long)desc->notch_freq, desc->notch_q);

        const EnvelopeForm form = envelope_form(ctx, n);
        const void *d_pcm = upload_pcm(ctx, pcm, (size_t)n_in * ch, desc->flags, false);
        float *d_env = (float *)ctx->seg.env.reserve((size_t)n * sizeof(float));
        float *d_audio = (float *)ctx->work_a.reserve((size_t)n * sizeof(float));
        const NotchInput in = notch_input(ctx, *desc, d_pcm, n, 1);
        float2 *z = envelope_scratch(ctx, form, 1);
        float2 *zc = form.plan ? z : nullptr;
        if (seam > 0)
            launch_filtfilt(ctx, in.mode, in.x, in.stride, d_audio, (size_t)n, zc, (size_t)n, seam, fp, 1);
        launch_filtfilt(ctx, in.mode, in.at(seam), in.stride, d_audio + seam, (size_t)n, zc ? zc + seam : nullptr,
                        (size_t)n, n - seam, fp, 1);
        launch_envelope(ctx, form, d_audio, (size_t)n, z, d_env, (size_t)n, 1);
        CUDA_CHECK(cudaStreamSynchronize(st));
        // only the side of the seam that holds the core is needed from here on
        const bool tail_side = seam > 0 && seam <= core_begin;
        ctx->seg.base = tail_side ? seam : 0;
        ctx->seg.n = seam > 0 ? (tail_side ? n - seam : seam) : n;
        ctx->seg.core_lo = core_begin - ctx->seg.base;
        ctx->seg.core_hi = core_end - ctx->seg.base;
        ctx->seg.have_env = true;
    });
}

int wefax_segment_histogram(wefax_ctx *ctx, int level, const uint32_t prefix[4], uint32_t *hist) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (level < 0 || level > 2 || !hist || (level > 0 && !prefix)) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        if (!ctx->seg.have_env) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_envelope has not run on this context");
        use_device(ctx);
        const uint32_t zero[4] = {0, 0, 0, 0};
        uint32_t *d_hist = (uint32_t *)ctx->out_small.reserve(4 * 2048 * sizeof(uint32_t));
        uint32_t *h_hist = (uint32_t *)pinned(ctx, 4 * 2048 * sizeof(uint32_t));
        launch_segment_hist(ctx, ctx->seg.env.as<float>() + ctx->seg.base, ctx->seg.n, ctx->seg.core_lo, ctx->seg.core_hi, level,
                            level > 0 ? prefix : zero, d_hist);
        CUDA_CHECK(cudaMemcpyAsync(h_hist, d_hist, 4 * 2048 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        memcpy(hist, h_hist, 4 * 2048 * sizeof(uint32_t));
    });
}

int wefax_segment_quantise(wefax_ctx *ctx, double low, double high, uint8_t *digitalized, float *demodulated) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!ctx->seg.have_env) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_envelope has not run on this context");
        use_device(ctx);
        RecResult *d_res = (RecResult *)ctx->out_small.reserve(sizeof(RecResult));
        RecResult *h_res = (RecResult *)pinned(ctx, sizeof(RecResult));
        memset(h_res, 0, sizeof(RecResult));
        h_res->low = low;
        h_res->high = high;
        CUDA_CHECK(cudaMemcpyAsync(d_res, h_res, sizeof(RecResult), cudaMemcpyHostToDevice, ctx->stream));
        segment_grey_map(ctx, d_res, digitalized, demodulated);
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        ctx->seg.have_dig = true;
    });
}

int wefax_segment_select_init(wefax_ctx *ctx, uint32_t *state, const uint32_t ranks[4], double t_lo, double t_hi) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!state || !ranks) WEFAX_THROW(WEFAX_ERR_INVALID, "null argument");
        use_device(ctx);
        launch_segment_state_init(ctx, state, ranks, t_lo, t_hi);
    });
}

int wefax_segment_histogram_dev(wefax_ctx *ctx, int level, uint32_t *state) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (level < 0 || level > 2 || !state) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        if (!ctx->seg.have_env) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_envelope has not run on this context");
        use_device(ctx);
        launch_segment_hist(ctx, ctx->seg.env.as<float>() + ctx->seg.base, ctx->seg.n, ctx->seg.core_lo, ctx->seg.core_hi, level,
                            nullptr, state + WEFAX_SEG_STATE_HIST, level > 0 ? state + 4 : nullptr);
    });
}

int wefax_segment_select_dev(wefax_ctx *ctx, int level, uint32_t *state) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (level < 0 || level > 2 || !state) WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        use_device(ctx);
        launch_segment_select_dev(ctx, state, level);
    });
}

int wefax_segment_quantise_dev(wefax_ctx *ctx, const uint32_t *state, uint8_t *digitalized, float *demodulated) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!state) WEFAX_THROW(WEFAX_ERR_INVALID, "null argument");
        if (!ctx->seg.have_env) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_envelope has not run on this context");
        use_device(ctx);
        RecResult *d_res = (RecResult *)ctx->out_small.reserve(sizeof(RecResult));
        CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult), ctx->stream));
        launch_segment_state_to_result(ctx, state, d_res);
        segment_grey_map(ctx, d_res, digitalized, demodulated);
        ctx->seg.have_dig = true;   // (stream-ordered: the search / raster calls that follow run on the same stream)
    });
}

int wefax_segment_sync(wefax_ctx *ctx, double lpm, const wefax_batch_out *out) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!out) WEFAX_THROW(WEFAX_ERR_INVALID, "null argument");
        if (!ctx->seg.have_dig) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_quantise has not run on this context");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const long long n = ctx->seg.n;
        const LineSet ls = prepare_lines(&lpm, 1, n);
        LineDev *d_lines = (LineDev *)ctx->out_small.reserve(sizeof(LineDev) + sizeof(RecResult));
        RecResult *d_res = (RecResult *)(d_lines + 1);
        RecResult *h_res = (RecResult *)pinned(ctx, sizeof(RecResult));
        CUDA_CHECK(cudaMemcpyAsync(d_lines, ls.lines.data(), sizeof(LineDev), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult), st));
        const SyncPlan splan = prepare_sync(ctx, ls.lines.data(), 1, n);
        clear_sync_scratch(ctx, splan, 1);
        launch_sync_search(ctx, ctx->seg.dig.as<uint8_t>(), (size_t)n, n, 1, d_lines, d_res, ls.min_mind, splan);
        CUDA_CHECK(cudaMemcpyAsync(h_res, d_res, sizeof(RecResult), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        wefax_batch_out small = *out;
        small.raster = nullptr;   // the raster of a segment comes from wefax_segment_raster
        small.height = nullptr;   // (the height of the whole image is the host's to compute)
        small.low_high = nullptr;
        // a segment shorter than one line is not an error of the recording
        h_res->status &= ~WEFAX_REC_NO_LINES;
        deliver_results(ctx, h_res, 1, 0, ls, &small, nullptr, 0, false);
    });
}

int wefax_segment_raster(wefax_ctx *ctx, double lpm, long long first_sample, int n_lines, int skip_lines,
                         int keep_lines, uint8_t *raster) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&, first_sample]() mutable {
        if (!raster || n_lines < 0 || skip_lines < 0 || keep_lines < 0 || skip_lines + keep_lines > n_lines)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        if (!ctx->seg.have_dig) WEFAX_THROW(WEFAX_ERR_INVALID, "wefax_segment_quantise has not run on this context");
        if (keep_lines == 0) return;
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const long long n = ctx->seg.n;
        const LineSet ls = prepare_lines(&lpm, 1, n);
        const int w = ls.lines[0].width;
        first_sample -= ctx->seg.base;   // positions of the API are relative to the extended segment
        if (first_sample < 0 || first_sample + (long long)n_lines * w > n)
            WEFAX_THROW(WEFAX_ERR_INVALID, "lines [%lld, +%d x %d) outside the extended segment of %lld samples",
                        first_sample, n_lines, w, n);
        LineDev *d_lines = (LineDev *)ctx->out_small.reserve(sizeof(LineDev) + sizeof(RecResult));
        RecResult *d_res = (RecResult *)(d_lines + 1);
        char *h_up = (char *)pinned(ctx, sizeof(LineDev) + sizeof(RecResult));
        RecResult h_res;
        memset(&h_res, 0, sizeof(h_res));
        h_res.start_frame = first_sample;
        h_res.height = 4 * n_lines;
        memcpy(h_up, &ls.lines[0], sizeof(LineDev));
        memcpy(h_up + sizeof(LineDev), &h_res, sizeof(RecResult));
        CUDA_CHECK(cudaMemcpyAsync(d_lines, h_up, sizeof(LineDev) + sizeof(RecResult), cudaMemcpyHostToDevice, st));
        const size_t rs = (size_t)4 * n_lines * w;
        uint8_t *d_raster = (uint8_t *)ctx->out_raster.reserve(rs);
        launch_raster(ctx, ctx->seg.dig.as<uint8_t>(), (size_t)n, n, 1, d_lines, d_res, d_raster, rs, w, n_lines);
        CUDA_CHECK(cudaMemcpyAsync(raster, d_raster + (size_t)4 * skip_lines * w, (size_t)4 * keep_lines * w,
                                   cudaMemcpyDefault, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
    });
}

int wefax_tone_scan(wefax_ctx *ctx, const int16_t *pcm, long long n_frames, int channels, int sample_rate,
                    long long packet_frames, unsigned flags, const wefax_tone_settings *settings,
                    uint8_t *start_flags, uint8_t *stop_flags, int32_t *n_start_peaks, int32_t *n_stop_peaks) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!pcm || !settings || n_frames < 0 || packet_frames < 4 || sample_rate < 1 || (channels != 1 && channels != 2))
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        const long long n_packets = n_frames / packet_frames;
        if (n_packets == 0) return;
        if (n_packets > 0x7fffffff) WEFAX_THROW(WEFAX_ERR_INVALID, "too many packets");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const size_t P = (size_t)packet_frames;
        const uint32_t half = (uint32_t)(P / 2);
        // packets per wave: float samples + complex transform scratch + kept bins within the workspace cap
        const size_t per_packet = P * (sizeof(float) + sizeof(float2) * 4) + (size_t)half * sizeof(float2);
        long long wave = (long long)((size_t)ctx->workspace_limit / per_packet);
        if (wave < 1) wave = 1;
        if (wave > n_packets) wave = n_packets;
        if (wave > 65535) wave = 65535;   // grid.y of the transform passes
        const size_t frame_elems = (size_t)channels;
        uint8_t *h_flags = (uint8_t *)pinned(ctx, (size_t)n_packets * (2 + 2 * sizeof(int32_t)) + 16);
        int32_t *h_counts = (int32_t *)(h_flags + (((size_t)n_packets * 2 + 15) & ~(size_t)15));
        uint8_t *d_flags = (uint8_t *)ctx->out_small.reserve((size_t)n_packets * (2 + 2 * sizeof(int32_t)) + 16);
        int32_t *d_counts = (int32_t *)(d_flags + (((size_t)n_packets * 2 + 15) & ~(size_t)15));
        for (long long p0 = 0; p0 < n_packets; p0 += wave) {
            const int np = (int)std::min(wave, n_packets - p0);
            const int16_t *d_pcm =
                (const int16_t *)upload_pcm(ctx, pcm + (size_t)p0 * P * frame_elems, (size_t)np * P * frame_elems, flags, false);
            float *x = (float *)ctx->work_a.reserve((size_t)np * P * sizeof(float));
            float2 *X = (float2 *)ctx->work_e.reserve((size_t)np * half * sizeof(float2));
            launch_ingest_float(ctx, d_pcm, P, channels, x, P, (long long)P, np);   // stride in frames
            spectrum_natural(ctx, (long long)P, x, P, X, half, half, np);
            launch_tone_peaks(ctx, X, half, (long long)P, sample_rate, np, *settings, d_flags + 2 * p0, d_counts + 2 * p0);
        }
        CUDA_CHECK(cudaMemcpyAsync(h_flags, d_flags, (size_t)n_packets * 2, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(h_counts, d_counts, (size_t)n_packets * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (long long k = 0; k < n_packets; ++k) {
            if (start_flags) start_flags[k] = h_flags[2 * k];
            if (stop_flags) stop_flags[k] = h_flags[2 * k + 1];
            if (n_start_peaks) n_start_peaks[k] = h_counts[2 * k];
            if (n_stop_peaks) n_stop_peaks[k] = h_counts[2 * k + 1];
        }
    });
}

// DataPacket.find_sync_pulse() (data_packet.py:301-343) for every consecutive packet of a recording: the packet's
// spectrum must hold exactly one peak (height / prominence, no distance rule) inside [min, max] Hz, and the template
// search over the packet's OWN grey levels (its own notch at the packet's sample rate, |hilbert|, median-3, 0.5 / 99.5
// percentile stretch with delta + 1e-6: data_packet.py:408-465) must return at least one pulse.
int wefax_sync_pulse_scan(wefax_ctx *ctx, const int16_t *pcm, long long n_frames, int channels, int sample_rate,
                          long long packet_frames, unsigned flags, const wefax_sync_pulse_settings *settings,
                          uint8_t *pulse_found, uint8_t *frequency_peak_found, int32_t *n_fft_peaks, int32_t *n_pulses,
                          int32_t *last_pulse, int32_t *pulses, uint8_t *samples) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!pcm || !settings || n_frames < 0 || packet_frames < 16 || sample_rate < 1 || (channels != 1 && channels != 2))
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        const long long n_packets = n_frames / packet_frames;
        if (n_packets == 0) return;
        if (n_packets > 0x7fffffff) WEFAX_THROW(WEFAX_ERR_INVALID, "too many packets");
        if (packet_frames >= (1ll << 31) - 4096) WEFAX_THROW(WEFAX_ERR_INVALID, "packet too long");
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const long long P = packet_frames;
        const uint32_t half_bins = (uint32_t)(P / 2);
        // samples(x) = int((x / (len / rate)) * len)  (data_packet.py:315), Python float arithmetic
        volatile double length = (double)P / (double)sample_rate;
        auto nsamp = [&](double x) { volatile double q = x / length; return (int)(q * (double)P); };
        const int k0 = nsamp(0.025), mind = nsamp(0.4);
        if (k0 + 2 > 2048 || mind < 1024 || P <= k0 + 2)
            WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "packet geometry outside the supported range (template %d, distance %d)",
                        k0 + 2, mind);
        const FirParams fp = make_fir(settings->notch_freq, settings->notch_q, (double)sample_rate);
        wefax_tone_settings ts;
        ts.start_distance = ts.stop_distance = 1.0;   // find_peaks without a distance rule
        ts.height = settings->height;
        ts.prominence = settings->prominence;
        ts.min_frequency = settings->min_frequency;
        ts.max_frequency = settings->max_frequency;
        ts.min_amount = ts.max_amount = 1;

        const EnvelopeForm form = envelope_form(ctx, P);
        const size_t per_packet = (size_t)P * (sizeof(float) * 3 + sizeof(float2) * 4 + 1) + (size_t)half_bins * sizeof(float2) +
                                  (size_t)form.zlen * sizeof(float2) + sizeof(RecResult) + sizeof(SelState);
        long long wave = (long long)((size_t)ctx->workspace_limit / per_packet);
        wave = std::max<long long>(1, std::min<long long>(std::min<long long>(wave, n_packets), 32768));

        LineDev line;
        memset(&line, 0, sizeof(line));
        line.n1 = k0;
        line.L = k0 + 2;
        line.mindistance = mind;
        line.width = (int)P;
        char *small = (char *)ctx->out_small.reserve(sizeof(LineDev) + 256 + (sizeof(RecResult) + sizeof(SelState)) * (size_t)wave +
                                                     (size_t)wave * (2 + 2 * sizeof(int32_t)) + 64);
        LineDev *d_line = (LineDev *)small;
        RecResult *d_res = (RecResult *)(small + 256);
        SelState *d_sel = (SelState *)(((uintptr_t)(d_res + wave) + 255) & ~(uintptr_t)255);
        uint8_t *d_flags = (uint8_t *)(d_sel + wave);
        int32_t *d_counts = (int32_t *)(d_flags + (((size_t)wave * 2 + 15) & ~(size_t)15));
        char *hbuf = (char *)pinned(ctx, sizeof(LineDev) + (sizeof(RecResult)) * (size_t)wave +
                                             (size_t)wave * (2 + 2 * sizeof(int32_t)) + 64);
        LineDev *h_line = (LineDev *)hbuf;
        RecResult *h_res = (RecResult *)(h_line + 1);
        uint8_t *h_flags = (uint8_t *)(h_res + wave);
        int32_t *h_counts = (int32_t *)(h_flags + (((size_t)wave * 2 + 15) & ~(size_t)15));
        *h_line = line;
        CUDA_CHECK(cudaMemcpyAsync(d_line, h_line, sizeof(LineDev), cudaMemcpyHostToDevice, st));

        for (long long p0 = 0; p0 < n_packets; p0 += wave) {
            const int np = (int)std::min(wave, n_packets - p0);
            const int16_t *d_pcm =
                (const int16_t *)upload_pcm(ctx, pcm + (size_t)p0 * P * channels, (size_t)np * P * channels, flags, false);
            // ---- the spectral test on the raw samples (data_packet.py:302-311) -----------------------------
            float *x = (float *)ctx->resample_in.reserve((size_t)np * P * sizeof(float));
            float2 *X = (float2 *)ctx->work_misc.reserve((size_t)np * half_bins * sizeof(float2));
            launch_ingest_float(ctx, d_pcm, (size_t)P, channels, x, (size_t)P, P, np);
            spectrum_natural(ctx, P, x, (size_t)P, X, half_bins, half_bins, np);
            launch_tone_peaks(ctx, X, half_bins, P, sample_rate, np, ts, d_flags, d_counts);
            // ---- the packet's grey levels (data_packet.py:408-465) ----------------------------------------
            float *d_audio = (float *)ctx->work_a.reserve((size_t)np * P * sizeof(float));
            float *d_env = (float *)ctx->work_e.reserve((size_t)np * P * sizeof(float));
            uint8_t *d_dig = (uint8_t *)ctx->out_dig.reserve((size_t)np * P);
            float2 *z = envelope_scratch(ctx, form, np);
            launch_filtfilt(ctx, kInFloat, x, (size_t)P, d_audio, (size_t)P, form.plan ? z : nullptr, (size_t)P, P, fp, np);
            launch_envelope(ctx, form, d_audio, (size_t)P, z, d_env, (size_t)P, np);
            CUDA_CHECK(cudaMemsetAsync(d_res, 0, sizeof(RecResult) * np, st));
            launch_percentiles(ctx, d_env, (size_t)P, P, np, d_sel, d_res, 3);
            launch_quantise(ctx, d_env, (size_t)P, d_dig, (size_t)P, P, np, d_res, 0, P, st, "packet_quantise", 3, 0.000001);
            // ---- the template search (data_packet.py:313-331) -----------------------------------------------
            launch_packet_pulse_search(ctx, d_dig, (size_t)P, P, np, d_line, d_res, mind);
            CUDA_CHECK(cudaMemcpyAsync(h_res, d_res, sizeof(RecResult) * np, cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaMemcpyAsync(h_flags, d_flags, (size_t)np * 2, cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaMemcpyAsync(h_counts, d_counts, (size_t)np * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            if (samples) CUDA_CHECK(cudaMemcpyAsync(samples + (size_t)p0 * P, d_dig, (size_t)np * P, cudaMemcpyDefault, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            for (int k = 0; k < np; ++k) {
                const long long K = p0 + k;
                const bool freq_ok = h_flags[2 * k] != 0;
                const int npl = h_res[k].n_peaks;
                if (frequency_peak_found) frequency_peak_found[K] = freq_ok ? 1 : 0;
                if (n_fft_peaks) n_fft_peaks[K] = h_counts[2 * k];
                if (n_pulses) n_pulses[K] = npl;
                if (last_pulse) last_pulse[K] = npl > 0 ? h_res[k].peaks[npl - 1] : -1;
                if (pulse_found) pulse_found[K] = (freq_ok && npl > 0) ? 1 : 0;
                if (pulses)
                    for (int t = 0; t < WEFAX_MAX_PULSES; ++t) pulses[(size_t)K * WEFAX_MAX_PULSES + t] = t < npl ? h_res[k].peaks[t] : -1;
            }
        }
    });
}

int wefax_decode_fm(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, const wefax_fm_params *prm,
                    const wefax_fm_out *out) {
    wefax_fm_slant off;
    memset(&off, 0, sizeof(off));
    off.mode = WEFAX_FM_SLANT_OFF;
    return wefax_decode_fm_slant(ctx, desc, pcm, prm, &off, out, nullptr);
}

int wefax_decode_fm_slant(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, const wefax_fm_params *prm,
                          const wefax_fm_slant *slant, const wefax_fm_out *out, wefax_fm_slant_out *slant_out) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!desc || !pcm || !prm || !slant || !out || desc->n_recordings != 1 || desc->n_frames < 64 ||
            (desc->channels != 1 && desc->channels != 2) || desc->sample_rate < 1)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        if (!(prm->lpm > 0.0) || prm->ioc < 1 || !(prm->white_hz > prm->black_hz) || prm->fold_lines < 1)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad FM parameters");
        const wefax_fm_slant sp = checked_slant(*slant);
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const long long n_in = desc->n_frames;
        const bool resample = desc->sample_rate != WEFAX_TARGET_RATE;
        const long long n = resample ? wefax_resampled_length(n_in, desc->sample_rate) : n_in;
        if (n < 64) WEFAX_THROW(WEFAX_ERR_INVALID, "recording too short");
        const bool out_dev = desc->flags & WEFAX_F_OUT_ON_DEVICE;
        const long long image_end = (prm->image_end > 0 && prm->image_end <= n) ? prm->image_end : n;
        const long long from = std::max<long long>(0, std::min<long long>(prm->search_from, n - 1));
        const FmGeometry fg = fm_geometry(prm->lpm, prm->ioc, sp, from, image_end);
        if (out->image && (long long)fg.rows_max * fg.W > out->image_capacity)
            WEFAX_THROW(WEFAX_ERR_INVALID, "image_capacity %lld too small (need %lld)", out->image_capacity,
                        (long long)fg.rows_max * fg.W);

        // grey stream (in the transform scratch, or straight into the caller's device buffer)
        const FmFront ff = fm_front_plan(ctx, n);
        const void *d_pcm = upload_pcm(ctx, pcm, (size_t)n_in * desc->channels, desc->flags, false);
        const float *g = fm_front_end(ctx, *desc, d_pcm, *prm, ff, 1, (out_dev && out->grey) ? out->grey : nullptr);
        if (!out_dev && out->grey)
            CUDA_CHECK(cudaMemcpyAsync(out->grey, g, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
        // the picture stage with a table of one chart: the caller's span
        std::vector<FmTail> cs(1);
        cs[0].g = g;
        cs[0].n = n;
        cs[0].from = from;
        cs[0].image_end = image_end;
        cs[0].fg = fg;
        cs[0].picture = out->image != nullptr;
        uint8_t *d_img = nullptr;
        if (out->image && fg.rows_max > 0)
            d_img = out_dev ? out->image : (uint8_t *)ctx->out_raster.reserve((size_t)fg.rows_max * fg.W);
        const wefax_fm_levels off = {WEFAX_FM_LEVELS_OFF, 200.0};
        const long long bytes = fm_tail(ctx, cs, *prm, sp, off, d_img);
        if (!out_dev && bytes > 0)
            CUDA_CHECK(cudaMemcpyAsync(out->image, d_img, (size_t)bytes, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        if (out->rows) *out->rows = cs[0].rows;
        if (out->width) *out->width = fg.W;
        if (out->line_start) *out->line_start = cs[0].line_start;
        if (slant_out) *slant_out = cs[0].so;
    });
}

int wefax_decode_fm_charts(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                           const wefax_fm_chart_params *params, wefax_fm_chart *charts, int max_charts, int *n_charts,
                           uint8_t *images, long long image_capacity, float *tone_scores, float *grey) {
    if (ctx && desc && desc->n_recordings != 1)
        return guarded(ctx, [] { WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument"); });
    return wefax_decode_fm_charts_batch(ctx, desc, pcm, params, charts, max_charts, n_charts, images, image_capacity,
                                        tone_scores, grey);
}

int wefax_decode_fm_charts_batch(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                                 const wefax_fm_chart_params *params, wefax_fm_chart *charts, int max_charts,
                                 int *n_charts, uint8_t *images, long long image_capacity, float *tone_scores,
                                 float *grey) {
    const wefax_fm_levels off = {WEFAX_FM_LEVELS_OFF, 0.0};
    return wefax_decode_fm_charts_levels(ctx, desc, pcm, params, &off, charts, nullptr, max_charts, n_charts, images,
                                         image_capacity, tone_scores, grey);
}

int wefax_decode_fm_charts_levels(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                                  const wefax_fm_chart_params *params, const wefax_fm_levels *levels,
                                  wefax_fm_chart *charts, wefax_fm_levels_out *levels_out, int max_charts,
                                  int *n_charts, uint8_t *images, long long image_capacity, float *tone_scores,
                                  float *grey) {
    if (!ctx) return WEFAX_ERR_INVALID;
    return guarded(ctx, [&] {
        if (!desc || !pcm || !params || !levels || !n_charts || max_charts < 0 || (max_charts > 0 && !charts) ||
            desc->n_recordings < 1 || desc->n_frames < 64 || (desc->channels != 1 && desc->channels != 2) ||
            desc->sample_rate < 1)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad argument");
        const wefax_fm_params &prm = params->fm;
        if (!(prm.lpm >= 0.0) || prm.ioc < 0 || !(prm.white_hz > prm.black_hz) || prm.fold_lines < 1)
            WEFAX_THROW(WEFAX_ERR_INVALID, "bad FM parameters");
        const wefax_fm_slant sp = checked_slant(params->slant);
        wefax_fm_levels lv = *levels;
        if (lv.mode != WEFAX_FM_LEVELS_OFF && lv.mode != WEFAX_FM_LEVELS_AUTO)
            WEFAX_THROW(WEFAX_ERR_INVALID, "unknown levels mode %d", lv.mode);
        if (lv.max_offset_hz == 0.0) lv.max_offset_hz = 200.0;
        if (!(lv.max_offset_hz > 0.0 && lv.max_offset_hz <= WEFAX_FM_LEVELS_MAX_OFFSET_HZ))
            WEFAX_THROW(WEFAX_ERR_INVALID, "max_offset_hz must be in (0, %g]", WEFAX_FM_LEVELS_MAX_OFFSET_HZ);
        static const double kStandardLpm[] = {60.0, 90.0, 100.0, 120.0, 180.0, 240.0};
        const int n_cand = params->n_lpm_candidates ? params->n_lpm_candidates : 6;
        const double *cand_lpm = params->n_lpm_candidates ? params->lpm_candidates : kStandardLpm;
        if (n_cand < 1 || n_cand > WEFAX_FM_MAX_LPM_CANDIDATES)
            WEFAX_THROW(WEFAX_ERR_INVALID, "1 to %d LPM candidates, not %d", WEFAX_FM_MAX_LPM_CANDIDATES, n_cand);
        LpmCandidates cand;
        memset(&cand, 0, sizeof(cand));
        cand.n = n_cand;
        for (int c = 0; c < n_cand; ++c) {
            if (!(cand_lpm[c] >= 60.0 && cand_lpm[c] <= 240.0))
                WEFAX_THROW(WEFAX_ERR_INVALID, "LPM candidate %g is outside [60, 240]", cand_lpm[c]);
            cand.Ls[c] = 60.0 / cand_lpm[c] * (double)WEFAX_TARGET_RATE;
            cand.Lc[c] = (int)ceil(cand.Ls[c]);
            cand.wb[c] = std::max(1, (int)llround(0.05 * cand.Ls[c]));
        }
        use_device(ctx);
        cudaStream_t st = ctx->stream;
        const int nrec = desc->n_recordings, ch = desc->channels;
        const long long n_in = desc->n_frames;
        const bool resample = desc->sample_rate != WEFAX_TARGET_RATE;
        const long long n = resample ? wefax_resampled_length(n_in, desc->sample_rate) : n_in;
        if (n < 64) WEFAX_THROW(WEFAX_ERR_INVALID, "recording too short");
        const bool out_dev = desc->flags & WEFAX_F_OUT_ON_DEVICE, pcm_dev = desc->flags & WEFAX_F_PCM_ON_DEVICE;
        const long long nw = n / WEFAX_FM_TONE_WINDOW;
        const size_t tone_row = (size_t)nw * 4;   // floats of one recording's tone scores
        const FmFront ff = fm_front_plan(ctx, n);

        // waves: the front end's buffers, the grey streams and the pictures of every recording of a wave stay resident
        const long long per_rec = (pcm_dev ? 0 : n_in * ch * 2) + (resample ? n_in * 4 + (n_in + n) * 4 : 0) +
                                  ff.npad * 8 + ff.zs * 8 + nw * 16 + n + 4096;
        int wave = (int)std::max<long long>(1, std::min<long long>(nrec, ctx->workspace_limit / per_rec));
        wave = std::min(wave, 32768);

        long long need = 0, img_off = 0;
        bool too_small = false;
        for (int w0 = 0; w0 < nrec; w0 += wave) {
            const int gw = std::min(wave, nrec - w0);
            // ---- front end and tone windows of the whole wave -----------------------------------------------------
            const void *d_pcm = upload_pcm(ctx, pcm + (size_t)w0 * n_in * ch, (size_t)gw * n_in * ch, desc->flags, false);
            float *grey_w = grey ? grey + (size_t)w0 * n : nullptr;
            const float *g = fm_front_end(ctx, *desc, d_pcm, prm, ff, gw, out_dev ? grey_w : nullptr);
            if (!out_dev && grey_w)
                CUDA_CHECK(cudaMemcpyAsync(grey_w, g, (size_t)gw * n * sizeof(float), cudaMemcpyDeviceToHost, st));
            const size_t tone_bytes = (size_t)gw * tone_row * sizeof(float);
            float4 *d_tone = (float4 *)ctx->work_misc.reserve(tone_bytes + 16);
            launch_fm_tone(ctx, g, n, nw, gw, d_tone);
            if (out_dev && tone_scores && nw > 0)
                CUDA_CHECK(cudaMemcpyAsync(tone_scores + (size_t)w0 * tone_row, d_tone, tone_bytes,
                                           cudaMemcpyDeviceToDevice, st));
            float *h_tone = (float *)pinned(ctx, tone_bytes + 16);
            if (nw > 0) CUDA_CHECK(cudaMemcpyAsync(h_tone, d_tone, tone_bytes, cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            if (!out_dev && tone_scores && nw > 0) memcpy(tone_scores + (size_t)w0 * tone_row, h_tone, tone_bytes);

            // ---- charts of each recording; the LPM of every chart of the wave in one launch ------------------------
            std::vector<std::vector<wefax_fm_chart>> found(gw);
            std::vector<FmChartJob> lpm_tab;
            std::vector<int> cls((size_t)nw);
            for (int r = 0; r < gw; ++r) {
                for (long long k = 0; k < nw; ++k) cls[k] = tone_class(h_tone + (size_t)r * tone_row + 4 * k);
                found[r] = find_charts(cls, n);
                n_charts[w0 + r] = (int)found[r].size();
                found[r].resize(std::min<size_t>(found[r].size(), (size_t)max_charts));
                for (wefax_fm_chart &c : found[r]) {
                    c.lpm = prm.lpm;
                    if (prm.ioc > 0) c.ioc = prm.ioc;
                    if (prm.lpm > 0.0) continue;
                    FmChartJob j;
                    memset(&j, 0, sizeof(j));
                    j.g = g + (size_t)r * n;
                    j.n = n;
                    j.from = std::min<long long>(c.search_from, n - 1);
                    lpm_tab.push_back(j);
                }
            }
            if (!lpm_tab.empty()) {
                const int nl = (int)lpm_tab.size();
                const size_t tab_bytes = ((size_t)nl * sizeof(FmChartJob) + 255) / 256 * 256;
                char *buf = (char *)ctx->work_misc.reserve(tab_bytes + (size_t)nl * n_cand * sizeof(double));
                FmChartJob *d_tab = (FmChartJob *)buf;
                double *d_score = (double *)(buf + tab_bytes);
                CUDA_CHECK(cudaMemcpyAsync(d_tab, lpm_tab.data(), (size_t)nl * sizeof(FmChartJob), cudaMemcpyHostToDevice, st));
                launch_fm_lpm(ctx, d_tab, nl, cand, prm.fold_lines, d_score);
                double *h_score = (double *)pinned(ctx, (size_t)nl * n_cand * sizeof(double));
                CUDA_CHECK(cudaMemcpyAsync(h_score, d_score, (size_t)nl * n_cand * sizeof(double), cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaStreamSynchronize(st));
                int t = 0;
                for (auto &rec : found)
                    for (wefax_fm_chart &c : rec) {
                        const double *sc = h_score + (size_t)(t++) * n_cand;
                        int best = 0;
                        for (int k = 1; k < n_cand; ++k)
                            if (sc[k] > sc[best]) best = k;
                        c.lpm = cand_lpm[best];
                        c.lpm_score = sc[best];
                        if (c.lpm_score < WEFAX_FM_LPM_MIN_SCORE) c.status = WEFAX_FM_CHART_NO_LPM;
                    }
            }

            // ---- every picture of the wave: one table, packed from img_off on --------------------------------------
            std::vector<FmTail> cs;
            long long wave_need = 0;
            for (int r = 0; r < gw; ++r)
                for (wefax_fm_chart &c : found[r]) {
                    const long long from = std::min<long long>(c.search_from, n - 1);
                    const FmGeometry fg = fm_geometry(c.lpm, c.ioc, sp, from, c.image_end);
                    c.width = fg.W;
                    if (c.status != WEFAX_FM_CHART_OK) continue;
                    wave_need += (long long)fg.rows_max * fg.W;
                    if (!images) continue;
                    FmTail t;
                    t.g = g + (size_t)r * n;
                    t.n = n;
                    t.from = from;
                    t.image_end = c.image_end;
                    t.fg = fg;
                    t.picture = true;
                    cs.push_back(t);
                }
            need += wave_need;
            if (images && need > image_capacity) too_small = true;   // (the remaining waves still count what they need)
            long long bytes = 0;
            if (!too_small && !cs.empty()) {
                uint8_t *d_img = out_dev ? images + img_off : (uint8_t *)ctx->out_raster.reserve((size_t)wave_need + 1);
                bytes = fm_tail(ctx, cs, prm, sp, lv, d_img);
                if (!out_dev && bytes > 0)
                    CUDA_CHECK(cudaMemcpyAsync(images + img_off, d_img, (size_t)bytes, cudaMemcpyDeviceToHost, st));
            }
            CUDA_CHECK(cudaStreamSynchronize(st));
            size_t t = 0;
            long long off = img_off;
            for (int r = 0; r < gw; ++r)
                for (size_t i = 0; i < found[r].size(); ++i) {
                    wefax_fm_chart &c = found[r][i];
                    wefax_fm_levels_out lo;
                    memset(&lo, 0, sizeof(lo));
                    lo.status = WEFAX_FM_LEVELS_NOT_MEASURED;
                    c.image_offset = off;
                    if (images && c.status == WEFAX_FM_CHART_OK && !too_small) {
                        const FmTail &p = cs[t++];
                        c.image_offset = img_off + p.offset;
                        c.rows = p.rows;
                        c.line_start = p.line_start;
                        c.slant = p.so;
                        lo = p.lv;
                        off = c.image_offset + (long long)p.rows * p.fg.W;
                    }
                    charts[(size_t)(w0 + r) * max_charts + i] = c;
                    if (levels_out) levels_out[(size_t)(w0 + r) * max_charts + i] = lo;
                }
            img_off += bytes;
        }
        if (too_small) WEFAX_THROW(WEFAX_ERR_INVALID, "image_capacity %lld too small (need %lld)", image_capacity, need);
    });
}

}  // extern "C"
