// The context behind the C-ABI handle: device, stream, cached FFT plans, scratch.
#pragma once

#include <cstring>
#include <vector>

#include "common.cuh"
#include "fft.cuh"
#include "fft_fast.cuh"

namespace wefax {
// chirp-z (Bluestein) data for a transform length with a prime factor > 13
struct Bluestein {
    long long n = 0, m = 0;
    FftPlan *plan = nullptr;   // length m (owned by the context's plan cache)
    DevBuf chirp;              // c[i] = exp(-i*pi*i^2/n), i < n
    DevBuf vhat;               // FFT_m of the wrapped conj(chirp), engine order, scaled by 1/m
};

constexpr int kMaxFirTaps = 64;
constexpr int kMaxSymTaps = 32;

// Truncated impulse response of the notch section (wefax.py:68-72): filtfilt is
// evaluated as a causal FIR h followed by an anti-causal FIR h with scipy's exact
// edge treatment (odd extension by 9, steady-state initial conditions).
struct FirParams {
    int K;                    // taps actually used (<= kMaxFirTaps), padded to KP
    int KP;                   // K rounded up to a multiple of 4
    float h[kMaxFirTaps];     // h[m], zero padded
    float hr[kMaxFirTaps];    // reversed: hr[j] = h[KP-1-j]
    // Away from the ends of the signal the two sections collapse into ONE symmetric FIR g = h * reversed(h):
    // out[i] = g[0] x[i] + sum_k g[k] (x[i-k] + x[i+k]), k <= KC (0: not available, use the two sections)
    int KC;
    float g[kMaxSymTaps + 1];
    // Impulse response longer than kMaxFirTaps (high quality factor, or a high sample rate in front of the notch
    // as in the live path's packets): the recursive form itself, in float64, in blocks that warm up over `warm`
    // samples (the response has decayed below 3e-9 of its sum by then); K then only reports the length.
    int iir;
    int warm;
    double b[3], a[3];
    double zi[2];             // scipy.signal.lfilter_zi(b, a): steady state of the transposed direct form II for a unit step
};
}  // namespace wefax

struct wefax_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string last_error;
    long long launches = 0;
    long long workspace_limit = 24ll << 30;
    // Lanes: a batch is split over child contexts (own stream and scratch, one host thread each) that take their
    // recordings through ALL stages a few at a time.  With host buffers that is a copy / compute pipeline; with
    // device-resident data it keeps a recording's working set in L2 (depth first), at the price of more launches.
    int max_wave = 0;                         // > 0: cap on the recordings of one wave (set on the lanes)
    int depth_first = -1;                     // WEFAX_DEPTH_FIRST: -1 auto, 0 off, 1 on
    int lanes = 3;                            // WEFAX_LANES
    int lane_wave = 1;                        // WEFAX_LANE_WAVE: recordings per wave on a lane
    // CUDA graph of the last device-resident single-wave decode: when the very next decode has identical arguments the
    // ~25 launches, memsets and small copies are replayed as ONE graph launch (the step then does not depend on how fast
    // the host can launch).  Any other call on the context in between invalidates it (scratch may move).
    bool use_graph = true;                    // WEFAX_GRAPH=0 turns it off
    bool graph_failed = false;                // a capture failed on this context: stay eager
    cudaGraphExec_t graph_exec = nullptr;
    std::vector<unsigned long long> graph_key, graph_candidate;
    long long api_calls = 0, graph_epoch = -1, graph_cand_epoch = -1;
    long long graph_launches = 0;
    void *graph_h_res = nullptr;              // pinned result records (RecResult[]) the graph's last copy fills
    bool is_lane = false;
    std::vector<wefax_ctx *> lane_ctx;        // owned
    cudaEvent_t ev_lane_fork = nullptr;
    std::vector<cudaEvent_t> ev_lane_join;
    int sm_count = 148;
    bool use_fused = true;  // WEFAX_FUSED=0: grey map and raster as two kernels instead of the fused sweep
    std::map<long long, std::unique_ptr<wefax::FftPlan>> plans;
    std::map<long long, std::unique_ptr<wefax::Bluestein>> bluestein;
    std::map<const void *, int> smem_configured;   // kernels whose dynamic-smem limit was raised
    // scratch (grown on demand, reused between calls)
    wefax::DevBuf pcm, work_a, work_z, work_e, work_misc, out_dig, out_raster, out_small, resample_in, sync_buf, pct_buf, grey_tab, iir_tmp;
    // segment mode: the extended segment's envelope and grey levels stay resident between the calls
    struct Segment {
        bool have_env = false, have_dig = false;
        long long base = 0;                          // start, in env, of the side of the seam that holds the core
        long long n = 0, core_lo = 0, core_hi = 0;   // length of that side and the core inside it (11025-Hz samples)
        wefax::DevBuf env, dig;
    } seg;
    // FIR form of the notch for the last (f0, Q) seen (api.cu: cached_fir)
    bool fir_valid = false;
    double fir_f0 = 0.0, fir_q = 0.0;
    wefax::FirParams fir;
    // pinned staging for small results
    void *pinned = nullptr;
    size_t pinned_cap = 0;
    void *pinned_up = nullptr;   // pinned staging of small host->device uploads (no stream sync needed to reuse the source)
    size_t pinned_up_cap = 0;
    // optional per-stage device timing (CUDA events on the context's stream)
    bool timing = false;
    struct Span {
        char name[24];   // copied: pass tags live in short-lived PassDev copies
        cudaEvent_t e0, e1;
    };
    std::vector<Span> spans;
    std::vector<cudaEvent_t> event_pool;
    std::map<std::string, std::pair<double, long long>> stage_ms;   // name -> (total ms, launches)
};

namespace wefax {

FftPlan *get_plan(wefax_ctx *ctx, long long n);   // nullptr when n needs Bluestein

// Brackets one stage with CUDA events when ctx->timing is on (no host sync here;
// wefax_ctx_timings() resolves them).
struct StageTimer {
    wefax_ctx *ctx;
    cudaEvent_t e1 = nullptr;
    cudaStream_t stream;
    StageTimer(wefax_ctx *c, const char *name, cudaStream_t on = nullptr) : ctx(c), stream(on ? on : c->stream) {
        if (!ctx->timing) return;
        cudaEvent_t ev[2];
        for (auto &e : ev) {
            if (!ctx->event_pool.empty()) {
                e = ctx->event_pool.back();
                ctx->event_pool.pop_back();
            } else {
                CUDA_CHECK(cudaEventCreate(&e));
            }
        }
        CUDA_CHECK(cudaEventRecord(ev[0], stream));
        e1 = ev[1];
        wefax_ctx::Span sp;
        strncpy(sp.name, name, sizeof(sp.name) - 1);
        sp.name[sizeof(sp.name) - 1] = 0;
        sp.e0 = ev[0];
        sp.e1 = ev[1];
        ctx->spans.push_back(sp);
    }
    ~StageTimer() {
        if (e1) cudaEventRecord(e1, stream);
    }
};

template <class LoadOp, class StoreOp, int MINB>
void launch_pass_variant(wefax_ctx *ctx, const PassDev &p, const LoadOp &ld, const StoreOp &st, int batch,
                         const CUtensorMap &map, const float2 *base, size_t bstride) {
    const void *fn = (const void *)fft_pass_kernel<LoadOp, StoreOp, MINB>;
    if (!ctx->smem_configured.count(fn)) {
        CUDA_CHECK(cudaFuncSetAttribute(fft_pass_kernel<LoadOp, StoreOp, MINB>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        ctx->smem_configured[fn] = 1;
    }
    dim3 grid(p.ntiles, batch);
    fft_pass_kernel<LoadOp, StoreOp, MINB><<<grid, p.nthreads, p.smem_bytes, ctx->stream>>>(p, ld, st, map, base, bstride);
}

template <int R1, int R2, class StoreOp>
void launch_fast_variant(wefax_ctx *ctx, const PassDev &p, const float2 *src, size_t bstride, const StoreOp &st,
                         int batch) {
    using K = fast::Cfg<R1, R2, fast::kFastC>;
    auto kern = fast::fft_fast_strided_kernel<R1, R2, fast::kFastC, StoreOp>;
    const void *fn = (const void *)kern;
    auto it = ctx->smem_configured.find(fn);
    int per_sm;
    if (it == ctx->smem_configured.end()) {
        CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM));
        CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, K::T, K::SMEM));
        if (per_sm < 1) per_sm = 1;
        ctx->smem_configured[fn] = per_sm;
    } else {
        per_sm = it->second;
    }
    const long long total = (long long)p.fast_ntiles * batch;
    const int grid = (int)std::min<long long>(total, (long long)ctx->sm_count * per_sm);
    kern<<<grid, K::T, K::SMEM, ctx->stream>>>(p, src, bstride, st, (int)total);
}

// The strided pass with its tiles by tensor TMA (fft_fast_tma3_kernel); false when the pass does not fit the boxes
template <int R1, int R2>
bool launch_fast_tma(wefax_ctx *ctx, const PassDev &p, const float2 *src, size_t src_bs, float2 *dst, size_t dst_bs,
                     int batch) {
    using K = fast::TmaCfg<R1, R2>;
    static_assert(fast::kFastCW == K::C, "tile geometry of the plan");
    int rbox = 0;
    for (int rb = std::min(K::R, 256); rb >= 1; --rb)
        if (K::R % rb == 0) {
            rbox = rb;
            break;
        }
    if (K::R / rbox > 8) return false;
    alignas(64) CUtensorMap in_map, out_map;
    if (!encode_strided_map(p, src, src_bs, batch, K::C, rbox, &in_map)) return false;
    if (!encode_strided_map(p, dst, dst_bs, batch, K::C, rbox, &out_map)) return false;
    auto kern = fast::fft_fast_tma3_kernel<R1, R2>;
    const void *fn = (const void *)kern;
    if (!ctx->smem_configured.count(fn)) {
        CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM));
        ctx->smem_configured[fn] = 1;
    }
    const long long total = (long long)p.fast_ntiles * batch;
    const int grid = (int)std::min<long long>(total, (long long)ctx->sm_count);
    kern<<<grid, K::T + 32, K::SMEM, ctx->stream>>>(p, in_map, out_map, rbox, (int)total);   // + the copy warp
    return true;
}

// Strided passes whose length has a compiled (R1, R2) pair go to the specialised kernel when the
// tile comes from plain complex memory and the store functor is one of the hot-path ones.
template <class LoadOp, class StoreOp>
bool try_launch_fast(wefax_ctx *ctx, const PassDev &p, const LoadOp &ld, const StoreOp &st, int batch) {
    if constexpr (std::is_same<LoadOp, LoadComplex>::value &&
                  (std::is_same<StoreOp, StoreComplex>::value || std::is_same<StoreOp, StoreEnvPairs>::value)) {
        if (!p.fast_R1 || p.contiguous || ld.conj) return false;
        if ((long long)p.fast_ntiles * batch > 0x7fffffffll) return false;
        StageTimer timer(ctx, p.tag);
        if constexpr (std::is_same<StoreOp, StoreComplex>::value) {
            // plain complex in and out: the TMA-staged variant (tile loads and stores by the copy engine)
            if (st.scale == 1.f && !st.conj) {
                bool done = false;
                switch (p.fast_R1 * 100 + p.fast_R2) {
                    case 1515: done = launch_fast_tma<15, 15>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    case 1615: done = launch_fast_tma<16, 15>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    case 1616: done = launch_fast_tma<16, 16>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    case 1514: done = launch_fast_tma<15, 14>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    case 1414: done = launch_fast_tma<14, 14>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    case 1507: done = launch_fast_tma<15, 7>(ctx, p, ld.src, ld.bstride, st.dst, st.bstride, batch); break;
                    default: break;
                }
                if (done) {
                    CUDA_CHECK(cudaGetLastError());
                    ctx->launches++;
                    return true;
                }
            }
        }
        switch (p.fast_R1 * 100 + p.fast_R2) {
#define WEFAX_FAST_CASE(a, b) \
    case (a) * 100 + (b): launch_fast_variant<a, b, StoreOp>(ctx, p, ld.src, ld.bstride, st, batch); break;
            WEFAX_FAST_CASE(15, 7)
            WEFAX_FAST_CASE(12, 12)
            WEFAX_FAST_CASE(14, 12)
            WEFAX_FAST_CASE(15, 12)
            WEFAX_FAST_CASE(16, 12)
            WEFAX_FAST_CASE(14, 14)
            WEFAX_FAST_CASE(15, 14)
            WEFAX_FAST_CASE(16, 14)
            WEFAX_FAST_CASE(15, 15)
            WEFAX_FAST_CASE(16, 15)
            WEFAX_FAST_CASE(16, 16)
#undef WEFAX_FAST_CASE
            default: return false;
        }
        CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
        return true;
    } else {
        return false;
    }
}

template <class LoadOp, class StoreOp>
void launch_pass(wefax_ctx *ctx, const PassDev &p_in, const LoadOp &ld, const StoreOp &st, int batch) {
    if (try_launch_fast(ctx, p_in, ld, st, batch)) return;
    PassDev p = p_in;
    alignas(64) CUtensorMap map;
    memset(&map, 0, sizeof(map));
    const float2 *base = nullptr;
    size_t bstride = 0;
    p.load_mode = 0;
    if (ld.tma_source(&base, &bstride)) p.load_mode = choose_load_mode(p, base, bstride, batch, &map);
    StageTimer timer(ctx, p.tag);
    // three CTAs of this pass fit one SM (227 KiB shared memory, 1 KiB reserved per CTA)?
    if ((size_t)p.smem_bytes + 1024 <= (size_t)(227 * 1024) / 3)
        launch_pass_variant<LoadOp, StoreOp, 3>(ctx, p, ld, st, batch, map, base, bstride);
    else
        launch_pass_variant<LoadOp, StoreOp, 2>(ctx, p, ld, st, batch, map, base, bstride);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// |hilbert(x)| for even n through a half-length transform of the packed real input
// (half = plan of n/2; x and env strides even).  x must stay intact until the end.
// want_y: env receives the Hilbert transform y of x instead of the envelope sqrt(x^2 + y^2)
void hilbert_envelope_real(wefax_ctx *ctx, FftPlan *half, const float *x, size_t xs, float2 *z, size_t zs, float *env,
                           size_t es, int batch, bool want_y = false);

// How |hilbert(x)| is computed at length n: a half-length transform of the packed real signal (half: even n whose half
// can be planned), a full-length transform of the complex copy (x, 0) (plan), or Bluestein (neither).
// zlen: complex scratch per sequence (n / 2, n, or Bluestein's padded length).
struct EnvelopeForm {
    FftPlan *half = nullptr, *plan = nullptr;
    long long n = 0, zlen = 0;
};
EnvelopeForm envelope_form(wefax_ctx *ctx, long long n);
// work_z scratch of `batch` sequences for launch_envelope, and for the complex copy the notch writes (nullptr for
// Bluestein, which reserves its own).  Take it after anything else that reserves work_z (the resampler): a larger
// reserve moves the buffer.
float2 *envelope_scratch(wefax_ctx *ctx, const EnvelopeForm &f, int batch);
// env = |hilbert(audio)| of `batch` sequences (no median filter).  The complex form reads (audio, 0) from z, where the
// notch leaves it, and not audio.
void launch_envelope(wefax_ctx *ctx, const EnvelopeForm &f, const float *audio, size_t as, float2 *z, float *env,
                     size_t es, int batch);

// natural-order complex DFT (test entry / Bluestein building block)
void fft_c2c_natural(wefax_ctx *ctx, FftPlan *plan, const float2 *in, float2 *out, float2 *scratch,
                     int batch, bool inverse);

// forward DFT of `batch` real sequences of length n (any n), first `keep` bins in natural
// order into X (stride xs_out); scratch: ctx->work_z
void spectrum_natural(wefax_ctx *ctx, long long n, const float *x, size_t xs, float2 *X, size_t xs_out,
                      uint32_t keep, int batch);

// scipy.signal.resample(x, num) on real float input (any n, num)
void resample_real(wefax_ctx *ctx, long long n, long long num, const float *x, size_t xs, float *y,
                   size_t ys, int batch);

}  // namespace wefax
