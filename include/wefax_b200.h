/*
 * wefax_b200 — C-ABI of the B200-native WEFAX file-decoding hot path.
 *
 * The reference (wojlin/WEFAX) has no plugin / FFI interface: its decode path is
 * the Python class wefax.Demodulator (wefax.py:18-408) whose process()
 * (wefax.py:46-93) calls scipy / numpy / Pillow.  This library sits BELOW a
 * Demodulator-compatible Python class (wefax_b200/wefax.py) and replaces, call
 * for call, the third-party routines process() runs:
 *
 *   wefax.py:349,360-373  wavfile.read + __merge_channels   -> int16 ingest (+ wrapping stereo merge)
 *   wefax.py:384          scipy.signal.resample             -> FFT-domain resample to 11025 Hz
 *   wefax.py:68-72        iirnotch + filtfilt               -> zero-phase notch (exact edge handling)
 *   wefax.py:174-175      hilbert + medfilt(abs, 5)         -> length-N analytic signal, envelope, median-5
 *   wefax.py:196-200,216  percentile / round / clip         -> global 0.5 / 99.5 percentile grey map
 *   wefax.py:221-294      pattern_search + peak grouping    -> phasing search, start_frame
 *   wefax.py:296-327      putpixel loop + Image.resize      -> line raster, x4 vertical bicubic (Pillow-exact)
 *
 * Plain pointers and sizes only; no torch / numpy types.  One context is used
 * from one host thread at a time; several contexts (one per GPU / stream) may be
 * used concurrently.  Every entry point returns a wefax_status; the message of
 * the last failure of a context is available from wefax_last_error().
 * There is NO CPU fallback: without a CUDA device wefax_ctx_create() fails.
 */
#ifndef WEFAX_B200_H
#define WEFAX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WEFAX_ABI_VERSION 5
#define WEFAX_TARGET_RATE 11025   /* wefax.py:60 */
#define WEFAX_MAX_PEAKS 100       /* wefax.py:251 */

typedef struct wefax_ctx wefax_ctx;

typedef enum {
    WEFAX_OK = 0,
    WEFAX_ERR_INVALID = 1,      /* bad argument */
    WEFAX_ERR_CUDA = 2,         /* CUDA runtime failure (message in wefax_last_error) */
    WEFAX_ERR_NOMEM = 3,        /* device allocation failed */
    WEFAX_ERR_UNSUPPORTED = 4   /* e.g. notch impulse response too long for the FIR path */
} wefax_status;

/* Per-recording outcome (wefax_batch_out.status), mirrors the exceptions the
 * reference's process() propagates. */
#define WEFAX_REC_OK 0
#define WEFAX_REC_NO_GROUPS 1   /* wefax.py:294  max([]) -> ValueError            */
#define WEFAX_REC_NO_LINES 2    /* wefax.py:304  putpixel on a 0-line image -> IndexError */
#define WEFAX_REC_NAN 4         /* wefax.py:216  int(nan): high == low percentile  */

/* wefax_batch_desc.flags */
#define WEFAX_F_PCM_ON_DEVICE 1u   /* pcm points to device memory                 */
#define WEFAX_F_OUT_ON_DEVICE 2u   /* every non-NULL output points to device mem  */
#define WEFAX_F_PCM_FLOAT32 4u     /* wefax_decode_batch only: pcm points to float32 mono samples (WAV sample formats
                                      other than 16-bit PCM, converted by the caller as scipy.io.wavfile.read would
                                      deliver them, wefax.py:349); channels must be 1.  The other entry points that
                                      read pcm take int16 only and reject it (WEFAX_ERR_INVALID).  */

/* ---- context -------------------------------------------------------------- */

/* stream: a cudaStream_t owned by the caller, or NULL to let the context create
 * its own.  All work of this context is issued on that stream. */
int wefax_ctx_create(int device, void *stream, wefax_ctx **out);
void wefax_ctx_destroy(wefax_ctx *ctx);
const char *wefax_last_error(const wefax_ctx *ctx);
int wefax_ctx_sync(wefax_ctx *ctx);
void *wefax_ctx_stream(wefax_ctx *ctx);
/* number of kernels this context has launched so far (bench accounting) */
long long wefax_ctx_launch_count(const wefax_ctx *ctx);
/* cap on the scratch memory one decode wave may use (default 24 GiB); recordings
 * of a batch are processed in waves that fit. */
int wefax_ctx_set_workspace_limit(wefax_ctx *ctx, long long bytes);
/* Per-stage device timing with CUDA events on the context's stream.  After
 * wefax_ctx_enable_timing(ctx, 1) every stage launch is bracketed by an event pair;
 * wefax_ctx_timings() synchronises, accumulates and writes one line per stage
 * ("name total_ms launches\n") into buf; reset != 0 clears the accumulators. */
int wefax_ctx_enable_timing(wefax_ctx *ctx, int enable);
int wefax_ctx_timings(wefax_ctx *ctx, char *buf, long long buf_len, int reset);
int wefax_abi_version(void);
int wefax_device_count(void);

/* ---- host-side helpers (no GPU needed) ------------------------------------ */

/* Constants the reference derives from LPM with Python float semantics
 * (wefax.py:33,223,225,229,264-266,298). */
typedef struct {
    double frame_len;     /* 1 / (lpm / 60)                         */
    int n1, n0;           /* samples(0.005), samples(0.001)         */
    int template_len;     /* 2*n1 + n0                              */
    int mindistance;      /* int(frame_len * sr * 0.8)              */
    int width;            /* int(frame_len * sr)                    */
    double dev_min, dev_max;   /* frame_len*sr -/+ 500 (exclusive)  */
} wefax_line_constants;
int wefax_line_constants_for(double lpm, int sample_rate, wefax_line_constants *out);

/* int(11025 * (n_frames / sample_rate))  (wefax.py:357,384) */
long long wefax_resampled_length(long long n_frames, int sample_rate);

/* scipy.signal.iirnotch(f0, Q, fs) (wefax.py:68-70) */
int wefax_notch_coefficients(double f0, double q, double fs, double b[3], double a[3]);

/* How an n-point transform is decomposed: number of passes, the radix-R of each
 * pass, and (bluestein != 0) the padded length used for non-smooth n. */
int wefax_fft_plan_describe(long long n, int *n_passes, int pass_len[8], long long *bluestein_len);

/* ---- the decode path ------------------------------------------------------ */

typedef struct {
    int n_recordings;
    long long n_frames;      /* input frames per recording (all recordings of a batch are equal) */
    int channels;            /* 1, or 2 = interleaved L,R merged as in wefax.py:372 */
    int sample_rate;         /* of the input; != 11025 triggers the FFT resample   */
    double notch_freq;       /* config.json notch_filter_frequency (wefax.py:63: int()) */
    double notch_q;          /* config.json notch_filter_quality_factor            */
    unsigned flags;
} wefax_batch_desc;

/* Outputs.  Any pointer may be NULL (that output is then not produced / copied).
 * audio / demodulated / digitalized / raster live where WEFAX_F_OUT_ON_DEVICE says;
 * the small per-recording results (peaks .. low_high) are ALWAYS host pointers.
 * n_out = n_frames if sample_rate == 11025 else wefax_resampled_length().
 * Per-recording strides: audio/demodulated/digitalized n_out elements; peaks and
 * phasing WEFAX_MAX_PEAKS ints; raster raster_stride bytes (>= 4*(n_out/width)*width). */
typedef struct {
    float *audio;            /* wefax.py:72   audio_data after filtfilt (int16 scale)  */
    float *demodulated;      /* wefax.py:74   demodulated_data                          */
    uint8_t *digitalized;    /* wefax.py:76   digitalized_data (0..255)                 */
    int32_t *peaks;          /* wefax.py:261  pattern_search() positions                */
    int32_t *n_peaks;
    int32_t *phasing;        /* wefax.py:78   phasing_signals                           */
    int32_t *n_phasing;
    int64_t *start_frame;    /* wefax.py:80                                             */
    int32_t *height;         /* raster rows = 4 * ((n_out - start_frame) / width)       */
    int32_t *status;         /* WEFAX_REC_* bits                                        */
    double *low_high;        /* 2 per recording: the 0.5 / 99.5 percentiles             */
    uint8_t *raster;         /* wefax.py:82-84 output_image, row-major (height, width)  */
    long long raster_stride;
} wefax_batch_out;

/* lpm: one value per recording (wefax.py:20,42). */
int wefax_decode_batch(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                       const double *lpm, const wefax_batch_out *out);

/* ---- stage-level entry points (parity tests of single stages) -------------- */

/* Complex DFT of `batch` sequences of length n, natural order in and out, host
 * pointers, interleaved (re, im) float32.  inverse != 0 applies the 1/n scale. */
int wefax_fft_c2c(wefax_ctx *ctx, long long n, int batch, const float *in, float *out, int inverse);

/* |scipy.signal.hilbert(x)| without the median filter; host pointers. */
int wefax_hilbert_envelope(wefax_ctx *ctx, long long n, int batch, const float *x, float *env);

/* scipy.signal.resample(x, num) for real float32 input; host pointers. */
int wefax_resample(wefax_ctx *ctx, long long n, long long num, int batch, const float *x, float *y);

/* scipy.signal.filtfilt(*iirnotch(f0, q, 11025), x) on float32 input; host pointers. */
int wefax_filtfilt(wefax_ctx *ctx, long long n, int batch, double notch_freq, double notch_q, const float *x,
                   float *y);

/* medfilt(env, 5) -> demodulated (optional), percentiles -> low_high (2 per recording),
 * grey map -> digitalized; status gets WEFAX_REC_NAN per recording.  Host pointers.
 * (wefax.py:175,196-200,216 on a given |hilbert| envelope) */
int wefax_digitalize(wefax_ctx *ctx, long long n, int batch, const float *envelope, float *demodulated,
                     uint8_t *digitalized, double *low_high, int32_t *status);

/* Phasing search + raster on given digitalized data (wefax.py:218-327).  Host pointers;
 * uses out->peaks .. out->status and out->raster / raster_stride; other fields ignored. */
int wefax_sync_raster(wefax_ctx *ctx, long long n, int batch, const uint8_t *digitalized, const double *lpm,
                      const wefax_batch_out *out);

/* ---- one long recording in overlapping segments, one per GPU (SURVEY.md 8(e), configs[2]) -----
 * process() (wefax.py:46-93) couples a whole recording three times: resample / hilbert are length-N
 * circular transforms (wefax.py:384,174), the two percentiles are global order statistics
 * (wefax.py:196) and start_frame shifts every image row (wefax.py:80,300-304).  Segment mode keeps the
 * last two EXACT across segments (histogram exchange below; start_frame from the first segment) and
 * approximates the first with a halo that is discarded (tolerance stated in DESIGN.md section 6).
 * All positions are 11025-Hz samples relative to the extended segment (core + halo) this context
 * holds.  Call order per context: envelope -> histogram x3 -> quantise -> [sync] -> raster.  The host
 * side (wefax_b200/segments.py) sums the histograms of all segments between the calls; no NCCL. */

/* ingest (+ resample) + notch + |hilbert| of one extended segment; the envelope stays resident in the
 * context.  desc: n_recordings == 1, n_frames = input frames of the extended segment; pcm as for
 * wefax_decode_batch, except that it is always int16: WEFAX_F_PCM_FLOAT32 is rejected (WEFAX_ERR_INVALID).  n_resampled = length of the extended segment at 11025 Hz (the planner cuts on
 * whole 11025-Hz samples, so this is exact; 0 = wefax_resampled_length(n_frames), the reference's float
 * formula for a whole recording).  [core_begin, core_end) = the samples this segment owns.
 * seam (0 = none): the transforms of the reference are circular, so the halo in front of the FIRST segment
 * is the END of the recording and the halo behind the LAST segment is its START; seam is the 11025-Hz
 * position inside the extended segment where the recording's end meets its start.  The transforms run
 * across the seam (as the whole-recording transforms do), the notch (filtfilt edge rules, wefax.py:72) and
 * the median (zero padding, wefax.py:175) treat it as the two ends of the recording.  The core must lie on
 * one side of it. */
int wefax_segment_envelope(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, long long n_resampled,
                           long long seam, long long core_begin, long long core_end);

/* Radix-digit histogram of the float bit patterns of medfilt(envelope, 5) over the core samples.
 * level 0: bin = bits >> 21 of every core sample -> hist[0][..]; level 1: samples with
 * bits >> 21 == prefix[t] -> hist[t][(bits >> 10) & 0x7FF]; level 2: samples with bits >> 10 == prefix[t]
 * -> hist[t][bits & 0x3FF].  hist: HOST pointer, 4 x 2048 uint32. */
int wefax_segment_histogram(wefax_ctx *ctx, int level, const uint32_t prefix[4], uint32_t *hist);

/* Grey map of the whole extended segment with the GLOBAL percentiles (wefax.py:197-216); stays
 * resident.  Optional outputs of the core samples only (host or device pointers, may be NULL):
 * digitalized (uint8) and demodulated = medfilt(envelope, 5) (float32). */
int wefax_segment_quantise(wefax_ctx *ctx, double low, double high, uint8_t *digitalized, float *demodulated);

/* ---- the same percentile exchange with everything resident on the devices (no host round trip per level) ----
 * `state` is a DEVICE buffer of WEFAX_SEG_STATE_WORDS uint32 owned by the caller (one per context):
 *   [0..3] remaining ranks, [4..7] prefixes, [8..9] t_lo, [10..11] t_hi, [12..13] low, [14..15] high (doubles),
 *   [16] WEFAX_REC_* status bits, [WEFAX_SEG_STATE_HIST ..) the 4 x 2048 histogram of the current level.
 * wefax_segment_select_init once, then per level 0, 1, 2:  wefax_segment_histogram_dev  ->  the caller sums
 * state[WEFAX_SEG_STATE_HIST ..] over all segments ON THE CONTEXT'S STREAM (e.g. ncclAllReduce, 32 KiB of control
 * data, not the compute path)  ->  wefax_segment_select_dev (every rank narrows the same targets redundantly).
 * After level 2 low / high / status are in the state and wefax_segment_quantise_dev maps the grey levels.  None of
 * these calls synchronises; with one segment the result is bit-identical to the host protocol's. */
#define WEFAX_SEG_STATE_HIST 32
#define WEFAX_SEG_STATE_WORDS (32 + 4 * 2048)
int wefax_segment_select_init(wefax_ctx *ctx, uint32_t *state, const uint32_t ranks[4], double t_lo, double t_hi);
int wefax_segment_histogram_dev(wefax_ctx *ctx, int level, uint32_t *state);
int wefax_segment_select_dev(wefax_ctx *ctx, int level, uint32_t *state);
int wefax_segment_quantise_dev(wefax_ctx *ctx, const uint32_t *state, uint8_t *digitalized, float *demodulated);

/* Phasing search (wefax.py:218-294) on the resident grey levels; meaningful on the segment that starts
 * at sample 0 of the recording (the search reads at most the first 100 peaks).  Fills out->peaks,
 * n_peaks, phasing, n_phasing, start_frame, status (host pointers, 1 recording). */
int wefax_segment_sync(wefax_ctx *ctx, double lpm, const wefax_batch_out *out);

/* Line raster + x4 vertical bicubic (wefax.py:296-327) of n_lines lines of width w = int(frame_len*11025)
 * starting at first_sample; the lines [skip_lines, skip_lines + keep_lines) are this segment's own (the
 * others are the bicubic margin: 2 lines each side unless the image ends there) and only their
 * 4 * keep_lines rows are written to raster (host or device pointer, 4 * keep_lines * w bytes). */
int wefax_segment_raster(wefax_ctx *ctx, double lpm, long long first_sample, int n_lines, int skip_lines,
                         int keep_lines, uint8_t *raster);

/* ---- start / stop tone test of packets (SURVEY.md 8(f) N2) ------------------- */

/* config/config.json "tones_settings" as data_packet.py:43-57 reads them. */
typedef struct {
    double start_distance;   /* start_tone_peaks_minimum_distance (bins)  data_packet.py:352 */
    double stop_distance;    /* stop_tone_peaks_minimum_distance (bins)   data_packet.py:362 */
    double height;           /* tones_peaks_minimum_height                data_packet.py:374 */
    double prominence;       /* tones_peaks_minimum_prominence            data_packet.py:375 */
    double min_frequency;    /* tones_peaks_minimum_frequency (Hz)        data_packet.py:380-381 */
    double max_frequency;    /* tones_peaks_maximum_frequency (Hz)                            */
    int min_amount;          /* tones_peaks_minimum_amount                data_packet.py:383-384 */
    int max_amount;          /* tones_peaks_maximum_amount                                    */
} wefax_tone_settings;

/* DataPacket.contain_start_tone() / contain_stop_tone() (data_packet.py:345-406) for every
 * consecutive packet of packet_frames frames of ONE recording: n_packets = n_frames / packet_frames
 * (a trailing partial packet is ignored).  pcm: int16, mono or interleaved stereo (merged as in
 * wefax.py:372), host pointer unless flags has WEFAX_F_PCM_ON_DEVICE; WEFAX_F_PCM_FLOAT32 is rejected
 * (WEFAX_ERR_INVALID).  Outputs are HOST pointers
 * of n_packets entries each; any may be NULL.  n_*_peaks = number of peaks find_peaks returned
 * (after the distance / height / prominence filters). */
int wefax_tone_scan(wefax_ctx *ctx, const int16_t *pcm, long long n_frames, int channels, int sample_rate,
                    long long packet_frames, unsigned flags, const wefax_tone_settings *settings,
                    uint8_t *start_flags, uint8_t *stop_flags, int32_t *n_start_peaks, int32_t *n_stop_peaks);

/* config/config.json "sync_pulse_settings" + "notch_filter_settings" as data_packet.py:20-46 reads them
 * (peaks_minimum_distance is read there but never used). */
typedef struct {
    double height;           /* peaks_minimum_height      data_packet.py:304 */
    double prominence;       /* peaks_minimum_prominence  data_packet.py:305 */
    double min_frequency;    /* peaks_minimum_frequency (Hz)  data_packet.py:309-311 */
    double max_frequency;    /* peaks_maximum_frequency (Hz)                          */
    double notch_freq;       /* notch_filter_frequency    data_packet.py:428 (designed at the PACKET's sample rate) */
    double notch_q;          /* notch_filter_quality_factor                           */
} wefax_sync_pulse_settings;

#define WEFAX_MAX_PULSES 16   /* pulse positions reported per packet (a 1-s packet holds at most 3) */

/* DataPacket.find_sync_pulse() (data_packet.py:301-343) for every consecutive packet of packet_frames frames of
 * ONE recording - the phasing gate of the live decoder's state machine (wefax_live.py:187-192): exactly one
 * spectral peak, inside [min_frequency, max_frequency], and at least one pulse from the template search over
 * the packet's own grey levels (data_packet.py:408-465: notch at the packet's rate, |hilbert|, median-3,
 * percentile stretch).  pcm / flags as for wefax_tone_scan (int16 only: WEFAX_F_PCM_FLOAT32 is rejected with
 * WEFAX_ERR_INVALID).  Outputs are HOST pointers of n_packets entries
 * (pulses: n_packets x WEFAX_MAX_PULSES, -1 padded; samples: n_packets x packet_frames grey levels, host or
 * device per cudaMemcpyDefault); any may be NULL.  last_pulse = peaks_samples[-1] (-1: none): where the live
 * decoder starts the picture inside the packet (wefax_live.py:191). */
int wefax_sync_pulse_scan(wefax_ctx *ctx, const int16_t *pcm, long long n_frames, int channels, int sample_rate,
                          long long packet_frames, unsigned flags, const wefax_sync_pulse_settings *settings,
                          uint8_t *pulse_found, uint8_t *frequency_peak_found, int32_t *n_fft_peaks, int32_t *n_pulses,
                          int32_t *last_pulse, int32_t *pulses, uint8_t *samples);

/* ---- EXTENSION (SURVEY.md 8(f) N4): FM-discriminator demodulation, IOC pixel columns ---------
 * Not in the reference's code (only described in its README.md:85-101): grey = instantaneous
 * frequency mapped black_hz..white_hz -> 0..255, exact line length 60/lpm s, pi*ioc pixels per line.
 * No reference parity exists for this entry point; it is checked against oracle/fm_oracle.py and the
 * synthetic generator's ground truth. */
typedef struct {
    double lpm;               /* lines per minute                                         */
    int ioc;                  /* index of cooperation: 576 or 288 -> round(pi*ioc) pixels  */
    double black_hz, white_hz;        /* 1500 / 2300 (README.md:87-88)                     */
    double band_lo_hz, band_hi_hz;    /* zero-phase FIR band-pass cut-offs, e.g. 1200 / 2600 */
    int fir_taps;             /* odd, <= 63                                                */
    long long search_from;    /* sample (at 11025 Hz) where the phasing search starts      */
    int fold_lines;           /* lines folded by the phasing search                        */
    long long image_end;      /* sample where the image ends (<= n_out; <= 0: n_out)       */
} wefax_fm_params;

typedef struct {
    float *grey;              /* optional: per-sample grey in [0,1] before clipping, n_out floats */
    uint8_t *image;           /* rows x width, row-major                                    */
    long long image_capacity; /* bytes available at image                                   */
    int32_t *rows, *width;    /* HOST pointers                                              */
    int64_t *line_start;      /* HOST pointer: sample index of the first image line         */
} wefax_fm_out;

/* One recording (desc->n_recordings must be 1); desc->flags as for wefax_decode_batch (grey / image
 * follow WEFAX_F_OUT_ON_DEVICE), except that pcm is always int16: WEFAX_F_PCM_FLOAT32 is rejected
 * (WEFAX_ERR_INVALID).  desc->notch_* are ignored.  The image has floor((image_end - line_start) / line
 * length) rows, computed in float64 without contraction, and every one of them is written. */
int wefax_decode_fm(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm, const wefax_fm_params *params,
                    const wefax_fm_out *out);

/* Slant (sample-clock error) correction of the FM decode.  A recording whose sample clock is off by p ppm has lines
 * of Ls / (1 + p * 1e-6) samples, Ls = 60 / lpm * 11025; ppm below is that p (positive: the recording's clock runs
 * slow, lines are shorter in samples; for resampled input it is the same as at the input rate). */
#define WEFAX_FM_SLANT_OFF 0     /* lines of exactly Ls samples: the output of the plain FM decode           */
#define WEFAX_FM_SLANT_FIXED 1   /* lines of Ls / (1 + ppm * 1e-6) samples, line start from the phasing fold  */
#define WEFAX_FM_SLANT_AUTO 2    /* line length and first line measured from the white line pulses          */

#define WEFAX_FM_SLANT_OK 0
#define WEFAX_FM_SLANT_NOT_FOUND 1   /* AUTO: too few pulses (or a fit outside +-max_ppm); the output is OFF's */

typedef struct {
    int mode;                 /* WEFAX_FM_SLANT_*                                                         */
    double ppm;               /* FIXED: the clock error, |ppm| <= 2000                                    */
    double max_ppm;           /* AUTO: largest clock error searched, in (0, 2000]                         */
    double min_contrast;      /* AUTO: pulse minus guard bands a line must show, (0, 1]; 0 = 0.3          */
    int min_lines;            /* AUTO: fewest lines with a pulse for a fit, >= 2; 0 = 8                   */
} wefax_fm_slant;

typedef struct {
    double line_length;       /* samples (at 11025 Hz) per image line used for the image                  */
    double ppm;               /* (Ls / line_length - 1) * 1e6                                             */
    double first_line;        /* fractional sample of the first image line (line_start = its rounding)    */
    int32_t lines_total;      /* AUTO: lines tracked in the last pass                                     */
    int32_t lines_used;       /* AUTO: lines whose pulse entered the final fit                            */
    double residual_rms;      /* AUTO: rms of the final fit's residuals (samples); large: the drift is not linear */
    int32_t status;           /* WEFAX_FM_SLANT_OK or WEFAX_FM_SLANT_NOT_FOUND                            */
} wefax_fm_slant_out;

/* The FM decode with slant correction; params / out as for the plain FM decode above, which equals this call with
 * mode WEFAX_FM_SLANT_OFF.  The image is sized for the shortest line the mode allows (FIXED: its line; AUTO:
 * Ls / (1 + max_ppm * 1e-6)).  slant_out (HOST pointer) may be NULL. */
int wefax_decode_fm_slant(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                          const wefax_fm_params *params, const wefax_fm_slant *slant, const wefax_fm_out *out,
                          wefax_fm_slant_out *slant_out);

/* ---- every chart of a recording (DESIGN.md 4.7b) --------------------------------------------------------------------
 * Tone windows: the grey stream is cut into whole windows of WEFAX_FM_TONE_WINDOW samples (0.2 s).  With u = clip(grey,
 * 0, 1), window mean mu and variance V = mean((u - mu)^2), r_f = 2 |sum_j (u_j - mu) exp(-2 pi i f j / 11025)|^2 /
 * (T^2 V) is the share of V in the line at f = 300, 450, 675 Hz (1 for a sinusoid, 8 / pi^2 for a square wave; 0 when
 * V = 0).  A window is START_576 / STOP / START_288 when r_300 / r_450 / r_675 is the largest of the three, that
 * largest r >= WEFAX_FM_TONE_MIN_RATIO and V >= WEFAX_FM_TONE_MIN_VAR; otherwise NONE.
 * Charts: a run is >= WEFAX_FM_TONE_MIN_RUN consecutive windows of one class, taken at its full length.  A start run
 * opens a chart (tone_begin = its first sample, search_from = the sample after it); the chart ends at the first later
 * STOP run (image_end = its first sample, stop_found = 1), at the next start run (which opens the next chart), or at
 * the end of the recording.  A STOP run with no chart open is ignored.
 * LPM: for each candidate c, the phasing fold of fold_lines lines of 60 / c * 11025 samples from search_from (the
 * index of the plain decode's fold) scores (best circular boxcar of 5 % of a line) / (boxcar width * lines) - (fold
 * mean) / lines; the highest score wins (the first listed on ties).  Below WEFAX_FM_LPM_MIN_SCORE the chart has status
 * WEFAX_FM_CHART_NO_LPM and no picture. */
#define WEFAX_FM_TONE_WINDOW 2205
#define WEFAX_FM_TONE_MIN_RATIO 0.5
#define WEFAX_FM_TONE_MIN_VAR 0.01
#define WEFAX_FM_TONE_MIN_RUN 10
#define WEFAX_FM_LPM_MIN_SCORE 0.3
#define WEFAX_FM_MAX_LPM_CANDIDATES 8   /* each within [60, 240] LPM */

#define WEFAX_FM_TONE_NONE 0
#define WEFAX_FM_TONE_START_576 1
#define WEFAX_FM_TONE_STOP 2
#define WEFAX_FM_TONE_START_288 3

#define WEFAX_FM_CHART_OK 0
#define WEFAX_FM_CHART_NO_LPM 1         /* no candidate reached WEFAX_FM_LPM_MIN_SCORE: reported, not decoded */

typedef struct {
    wefax_fm_params fm;       /* lpm / ioc: 0 = detect per chart, > 0 = that value for every chart (IOC 576 and 288
                                 start tones both open charts); search_from / image_end are ignored              */
    wefax_fm_slant slant;     /* applies to every chart                                                           */
    int n_lpm_candidates;     /* 0: the standard 60, 90, 100, 120, 180, 240                                       */
    double lpm_candidates[WEFAX_FM_MAX_LPM_CANDIDATES];
} wefax_fm_chart_params;

typedef struct {
    int64_t tone_begin;       /* first sample (at 11025 Hz) of the start tone run                                */
    int64_t search_from;      /* sample after the start tone run: the phasing search starts here                 */
    int64_t image_end;        /* first sample of the stop tone run, of the next start tone run, or n_out         */
    int32_t stop_found;       /* 1: image_end is a stop tone                                                     */
    int32_t ioc;              /* 576 or 288 from the start tone (or the forced value)                            */
    double lpm;               /* the best candidate (or the forced value)                                        */
    double lpm_score;         /* its score (0 when the LPM is forced)                                            */
    int32_t status;           /* WEFAX_FM_CHART_*                                                                */
    int32_t rows, width;      /* the picture: rows x width bytes at images + image_offset (rows 0: none)         */
    int64_t line_start;       /* sample of the first picture line (-1: no picture decoded)                       */
    int64_t image_offset;
    wefax_fm_slant_out slant; /* as wefax_decode_fm_slant reports it                                             */
} wefax_fm_chart;

/* Every chart of one recording, from one band-pass / Hilbert / discriminator pass: tone windows, charts, each
 * chart's IOC and LPM, then for each of the first max_charts charts (status OK) the picture exactly as
 * wefax_decode_fm_slant computes it with that chart's lpm, ioc, search_from and image_end.  desc / pcm / flags as for
 * wefax_decode_fm (WEFAX_F_PCM_FLOAT32 is rejected).  charts: HOST array of max_charts entries; *n_charts (HOST) = the
 * number of charts found, also when it is above max_charts.  images: the pictures back to back (host, or device under
 * WEFAX_F_OUT_ON_DEVICE), or NULL for the chart list only (no pictures, line_start -1); image_capacity must hold
 * sum over the decoded charts of floor((image_end - search_from) / shortest line) * width bytes (the shortest line as
 * wefax_decode_fm_slant sizes its image), else WEFAX_ERR_INVALID naming the bytes needed.  Optional outputs (host or
 * device as images): tone_scores, n_out / WEFAX_FM_TONE_WINDOW windows x (r_300, r_450, r_675, V) floats; grey,
 * n_out floats. */
int wefax_decode_fm_charts(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                           const wefax_fm_chart_params *params, wefax_fm_chart *charts, int max_charts,
                           int *n_charts, uint8_t *images, long long image_capacity, float *tone_scores, float *grey);

/* Every chart of desc->n_recordings >= 1 recordings of equal length (int16, host or WEFAX_F_PCM_ON_DEVICE), each
 * recording's charts and pictures exactly what wefax_decode_fm_charts returns for it alone.  The recordings run in
 * waves sized by wefax_ctx_set_workspace_limit; each wave takes a fixed number of launches and synchronisations
 * however many recordings and charts it holds (DESIGN.md 4.7c).  charts: HOST array of n_recordings x max_charts
 * entries, recording r's at r * max_charts; n_charts: HOST array of one count per recording (the charts found, also
 * when above max_charts; 0 when none is found, which is not an error).  images: the pictures of every recording back
 * to back, in recording then chart order, image_offset counted from images; image_capacity covers the whole batch,
 * else WEFAX_ERR_INVALID naming the bytes needed.  tone_scores: (n_out / WEFAX_FM_TONE_WINDOW) x 4 floats per
 * recording; grey: n_out floats per recording. */
int wefax_decode_fm_charts_batch(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                                 const wefax_fm_chart_params *params, wefax_fm_chart *charts, int max_charts,
                                 int *n_charts, uint8_t *images, long long image_capacity, float *tone_scores,
                                 float *grey);

/* ---- tuning offset of each chart from its phasing lines (DESIGN.md 4.7d) --------------------------------------------
 * A receiver mistuned by D Hz moves every grey value by D / (white_hz - black_hz).  For each chart with a picture, with
 * s its line start, Ls its line length (the slant fit's under AUTO slant), wb = max(1, round(0.05 Ls)), e = ceil(wb / 4)
 * and end = min(n_out, image_end), the samples i = s + floor(l * Ls + o) of lines l < fold_lines that lie in [0, end)
 * form two sets: the pulse, o in [e, wb - e), and the body, o in [wb + e, floor(Ls) - e).  b and w are the lower
 * medians (element floor((m - 1) / 2) in ascending order) of the unclipped grey over the body and the pulse; d = (b +
 * w) / 2 - 0.5.  Status OK when both sets hold samples, w - b is within [0.75, 1.25] and |d (white_hz - black_hz)| <=
 * max_offset_hz: the picture is then made of clip(grey - (float)d), a shift with no stretch (the discriminator's scale
 * is exact; noise pulls the measured levels toward the band centre, so the span is not a measure of it).  Otherwise the
 * picture is the uncorrected one.  The grey stream and the tone scores are never corrected. */
#define WEFAX_FM_LEVELS_OFF 0
#define WEFAX_FM_LEVELS_AUTO 1
#define WEFAX_FM_LEVELS_OK 0
#define WEFAX_FM_LEVELS_NOT_FOUND 1      /* measured, failed the checks: picture uncorrected */
#define WEFAX_FM_LEVELS_NOT_MEASURED 2   /* mode OFF, or the chart got no picture            */
#define WEFAX_FM_LEVELS_MAX_OFFSET_HZ 300.0

typedef struct {
    int mode;                 /* WEFAX_FM_LEVELS_*                                                                */
    double max_offset_hz;     /* largest offset corrected, (0, WEFAX_FM_LEVELS_MAX_OFFSET_HZ]; 0 = 200          */
} wefax_fm_levels;

typedef struct {
    double black_hz, white_hz, offset_hz;   /* measured (NaN from an empty set); offset_hz is applied only when status
                                               is OK; all 0 when not measured                                   */
    int64_t black_samples, white_samples;   /* samples in the body and the pulse set                              */
    int32_t status;                         /* WEFAX_FM_LEVELS_*                                                  */
} wefax_fm_levels_out;

/* wefax_decode_fm_charts_batch with the tuning offset measured and corrected per chart (levels: HOST pointer, not
 * NULL; a bad mode or max_offset_hz is WEFAX_ERR_INVALID).  levels_out: HOST array laid out like charts
 * (n_recordings x max_charts), or NULL.  With mode OFF every output equals wefax_decode_fm_charts_batch's, which is
 * this call with mode OFF and levels_out NULL.  AUTO adds one launch per wave with pictures and no synchronisation. */
int wefax_decode_fm_charts_levels(wefax_ctx *ctx, const wefax_batch_desc *desc, const int16_t *pcm,
                                  const wefax_fm_chart_params *params, const wefax_fm_levels *levels,
                                  wefax_fm_chart *charts, wefax_fm_levels_out *levels_out, int max_charts,
                                  int *n_charts, uint8_t *images, long long image_capacity, float *tone_scores,
                                  float *grey);

#ifdef __cplusplus
}
#endif
#endif /* WEFAX_B200_H */
