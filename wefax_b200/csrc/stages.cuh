// Non-FFT stages of the decode path: declarations shared by stages.cu and api.cu.
#pragma once

#include "ctx.cuh"

namespace wefax {

// per-recording line geometry (wefax_line_constants, device copy)
struct LineDev {
    int n1, n0, L, mindistance, width;
    double dev_min, dev_max;
    int gr_class;   // fused grey map + raster: 2 = width % 8 == 0, 1 = width % 4 == 0, else 0
    int pad;
};

// per-recording results produced on the device
struct RecResult {
    int32_t n_peaks;
    int32_t peaks[WEFAX_MAX_PEAKS];
    int32_t n_phasing;
    int32_t phasing[WEFAX_MAX_PEAKS];
    long long start_frame;
    int32_t height;      // raster rows (4 * image lines)
    int32_t status;
    double low, high;
};

// per-recording geometry of the parallel phasing search (host-computed)
struct SyncDev {
    long long m;      // number of correlation positions = n - L
    long long lim;    // settled bits are computed for [0, lim)
    long long limc;   // correlation / window maxima are computed for [0, limc)
    int fast;         // 0: this recording only runs the sequential scan
};

// device scratch of the parallel phasing search for one wave
struct SyncPlan {
    bool any_fast = false;
    SyncDev *sd = nullptr;
    int *corr = nullptr;
    size_t cs = 0;             // ints per recording in corr
    uint32_t *bits = nullptr;
    size_t bs = 0;             // words per recording in bits
    int *first_pos = nullptr, *need_scan = nullptr;
    long long max_lim = 0, max_limc = 0;
    int max_w = 0, max_wblocks = 0;
};

// percentile selection state, one per recording
struct SelState {
    uint32_t rank[4];      // remaining rank of each target inside its prefix class
    uint32_t prefix[4];    // key prefix found so far
    uint32_t hist[3][4][2048];
};

// grey map of one recording as a table (greyraster.cu): level(m) = largest k with T[k] <= float bits of m
struct GreyTable {
    uint32_t T[260];     // T[0] = 0, T[k]: smallest non-negative float bit pattern whose level is >= k, T[256..] = ~0
    float scale, off;    // fp32 estimate of the level: rint(m * scale + off)
    int est_ok;          // the estimate is proven to be within +-1 of the exact level for every float
    int pad;
};

// the sequential phasing scan may run past the grey levels that exist when it starts (fused grey map + raster):
// levels at positions >= valid are then computed from the envelope on the fly
struct LazyGrey {
    const float *env = nullptr;
    size_t es = 0;
    const GreyTable *tables = nullptr;
    long long valid = 0;
};

enum IngestMode { kInMonoI16 = 0, kInStereoI16 = 1, kInFloat = 2 };

void launch_ingest_float(wefax_ctx *ctx, const int16_t *pcm, size_t pcm_stride, int channels, float *x, size_t xs,
                         long long n, int batch);
// out (float, may be null) and / or zout (complex (x, 0), may be null)
void launch_filtfilt(wefax_ctx *ctx, IngestMode mode, const void *in, size_t in_stride, float *out, size_t out_stride,
                     float2 *zout, size_t z_stride, long long n, const FirParams &fp, int batch);
void launch_median5(wefax_ctx *ctx, const float *env, size_t es, float *out, size_t os, long long n, int batch);
// 0.5 / 99.5 percentiles of median5(env) -> RecResult.low/high (+ WEFAX_REC_NAN)
// med: median window in front of the percentiles (5: file path, wefax.py:175; 3: packets, data_packet.py:440)
// tables != nullptr: the stage also leaves the grey threshold table of every recording there when it can (returns
// true; false: the caller launches launch_grey_table itself)
struct GreyTable;
bool launch_percentiles(wefax_ctx *ctx, const float *env, size_t es, long long n, int batch, SelState *sel,
                        RecResult *res, int med = 5, GreyTable *tables = nullptr);
// eps: added to high - low (0 on the file path, 0.000001 for packets: data_packet.py:461)
void launch_quantise(wefax_ctx *ctx, const float *env, size_t es, uint8_t *dig, size_t ds, long long n, int batch,
                     const RecResult *res, long long i_begin, long long i_end, cudaStream_t stream, const char *tag,
                     int med = 5, double eps = 0.0);
// min_mindistance: smallest LineDev.mindistance of the batch (sizes the scan chunk; must be >= 1024).
// Expects the scratch cleared by clear_sync_scratch() earlier on the context's stream.
void launch_sync_search(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int batch, const LineDev *lines,
                        RecResult *res, int min_mindistance, const SyncPlan &sp, const LazyGrey &lazy = LazyGrey());
// the scratch the parallel search expects cleared (first positive correlation, settled bits)
void clear_sync_scratch(wefax_ctx *ctx, const SyncPlan &sp, int batch);
void launch_packet_pulse_search(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int n_packets,
                                const LineDev *line, RecResult *res, int mindistance);
// samples the parallel phasing search reads: [0, sync_head(sp, n))
long long sync_head(const SyncPlan &sp, long long n);
// sizes the parallel search for recordings [first, first+count) and uploads its geometry
SyncPlan prepare_sync(wefax_ctx *ctx, const LineDev *host_lines, int count, long long n);
void launch_raster(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int batch, const LineDev *lines,
                   const RecResult *res, uint8_t *raster, size_t rs, int max_width, int max_lines);
// ---- fused median-5 + grey map + raster (greyraster.cu) ----
// threshold tables of the grey map from RecResult.low/high (one per recording)
void launch_grey_table(wefax_ctx *ctx, const RecResult *res, GreyTable *tables, int batch);
// envelope -> digitalized (all n samples; dig may be null) + raster (rows of recordings with status OK; raster may
// be null).  Needs RecResult.start_frame / height / status, i.e. runs after the phasing search.
void launch_grey_raster(wefax_ctx *ctx, const float *env, size_t es, uint8_t *dig, size_t ds, uint8_t *raster, size_t rs,
                        long long n, int batch, const LineDev *d_lines, const LineDev *h_lines, const RecResult *res,
                        const GreyTable *tables);

// ---- segment mode (segment.cu): radix-digit histograms of the median-filtered envelope of the core
// samples [core_lo, core_hi) of an extended segment of n samples; hist: 4 x 2048 counters (device)
// prefix_dev (may be null): the four prefixes in DEVICE memory (device-resident exchange) instead of `prefix`
void launch_segment_hist(wefax_ctx *ctx, const float *env, long long n, long long core_lo, long long core_hi, int level,
                         const uint32_t prefix[4], uint32_t *hist, const uint32_t *prefix_dev = nullptr);
void launch_segment_state_init(wefax_ctx *ctx, uint32_t *state, const uint32_t ranks[4], double t_lo, double t_hi);
void launch_segment_select_dev(wefax_ctx *ctx, uint32_t *state, int level);
void launch_segment_state_to_result(wefax_ctx *ctx, const uint32_t *state, RecResult *res);
void launch_segment_median(wefax_ctx *ctx, const float *env, long long n, long long core_lo, long long core_hi,
                           float *out);

// find_peaks-based start / stop tone decision on the spectra of n_packets packets (tones.cu);
// flags / counts hold 2 entries per packet (start, stop), device pointers
void launch_tone_peaks(wefax_ctx *ctx, const float2 *X, size_t xs, long long packet_len, int sample_rate,
                       int n_packets, const wefax_tone_settings &s, uint8_t *flags, int32_t *counts);

// ---- N4 extension: FM-discriminator demodulation and IOC pixel columns (fm.cu) ----
FirParams make_bandpass_fir(double lo_hz, double hi_hz, double fs, int taps);
// grey of `batch` recordings: x / y rows of stride xs, g rows of n samples
void launch_fm_grey(wefax_ctx *ctx, const float *x, const float *y, size_t xs, float *g, long long n, int batch,
                    double black_hz, double white_hz);
// One chart of the FM decode's picture stage, which runs once over a table of charts (DESIGN.md §4.7c): where its grey
// stream lies, its span, the phasing fold and picture geometry, its output offset, and its slant search state
struct FmChartJob {
    const float *g;         // grey stream of the chart's recording, n samples
    long long n, from, image_end;
    double Ls;              // line length of the phasing fold and of the picture
    int Lc, wb;             // phasing fold: ceil(Ls) offsets, boxcar of wb samples
    int phase;              // 1: line start from the phasing fold; 0: given (the slant fit)
    int W, rows_max;        // picture: W pixels per row, rows_max rows at most (0: no picture)
    long long out;          // offset (bytes) of the picture in the output
    float shift;            // picture of clip(grey - shift): the measured tuning offset in grey units (0: none)
    // slant search (AUTO): profile of q_lines lines of the nominal line sLs in Bn bins of D samples (Q from q_off),
    // n_cand sheared folds; pulse tracking of track_lines lines around a + l * s (pos / contrast from pos_off)
    double sLs, a, s;
    int D, Bn, wbb, R, swb, q_lines, n_cand, track_lines;
    long long q_off, pos_off;
};
// line start of every chart with phase = 1 into d_line_start[chart]: the fold of `lines` lines (P: max Lc floats per chart)
void launch_fm_phasing(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts, int lines,
                       float *P, long long *d_line_start);
// tuning offset (DESIGN.md §4.7d): lower median of the unclipped grey over each chart's pulse and body sets of its first
// `lines` lines from d_line_start[chart] (Ls, wb; samples below min(n, image_end)), one (value, count) per set
struct FmLevel {
    float value;            // the order statistic (NaN when the set is empty)
    int pad;
    long long count;        // samples in the set
};
// lev[2 * chart] = body (black), lev[2 * chart + 1] = pulse (white)
void launch_fm_levels(wefax_ctx *ctx, const FmChartJob *d_tab, int n_charts, int lines, const long long *d_line_start,
                      FmLevel *lev);
// every chart's picture (rows_max > 0) into img + out
void launch_fm_image(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                     const long long *d_line_start, uint8_t *img);
// slant search (DESIGN.md §4.7a), per chart with q_lines > 0: Q = q_lines x Bn bin means of D samples from `from`
void launch_fm_slant_profile(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts, float *Q);
// sheared folds of each chart's Q for its n_cand candidate total shifts, best (score, candidate, bin) key into
// d_best[chart] (device)
void launch_fm_slant_fold(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                          const float *Q, unsigned long long *d_best);
// pulse position (or -1) and contrast of lines [0, track_lines) of each chart around a + l * s, +-R samples, pulse width swb
void launch_fm_slant_track(wefax_ctx *ctx, const FmChartJob *d_tab, const FmChartJob *h_tab, int n_charts,
                           double min_contrast, long long *pos, float *contrast);
// charts (DESIGN.md §4.7b): (r_300, r_450, r_675, V) of each whole WEFAX_FM_TONE_WINDOW window of g into out, for
// `batch` recordings of n samples (g) and n_windows windows (out) each
void launch_fm_tone(wefax_ctx *ctx, const float *g, long long n, long long n_windows, int batch, float4 *out);
// the LPM candidates' line lengths Ls = 60 / lpm * 11025, Lc = ceil(Ls) <= kLpmMaxLine, boxcars wb = max(1, round(0.05 Ls))
constexpr int kLpmMaxLine = 11025;
struct LpmCandidates {
    int n;
    double Ls[WEFAX_FM_MAX_LPM_CANDIDATES];
    int Lc[WEFAX_FM_MAX_LPM_CANDIDATES], wb[WEFAX_FM_MAX_LPM_CANDIDATES];
};
// phasing score of every (chart, candidate), chart-major, folding `lines` lines from each chart's `from` in its grey
// stream (d_tab: g, n, from)
void launch_fm_lpm(wefax_ctx *ctx, const FmChartJob *d_tab, int n_charts, const LpmCandidates &cand, int lines,
                   double *d_score);

}  // namespace wefax
