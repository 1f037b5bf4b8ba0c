// Non-FFT stages: ingest, zero-phase notch, median-5, percentile selection,
// grey-level quantisation, phasing search, line raster with x4 bicubic.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "grey.cuh"

namespace wefax {

// ===========================================================================
// ingest (only needed in front of the resampler; the notch reads PCM directly)
// ===========================================================================
template <int MODE>
__device__ __forceinline__ float load_sample(const void *in, size_t base, long long i) {
    if (MODE == kInMonoI16) return (float)__ldg((const int16_t *)in + base + i);
    if (MODE == kInStereoI16) {
        // wefax.py:372: np.add on two int16 scalars wraps, then /2 in float64
        const int16_t *p = (const int16_t *)in + 2 * (base + i);
        int16_t s = (int16_t)(__ldg(p) + __ldg(p + 1));
        return 0.5f * (float)s;
    }
    return __ldg((const float *)in + base + i);
}

template <int MODE>
__global__ void ingest_kernel(const void *in, size_t in_stride, float *x, size_t xs, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[(size_t)blockIdx.y * xs + i] = load_sample<MODE>(in, (size_t)blockIdx.y * in_stride, i);
}

// mono int16 -> float, 8 samples per thread (16-byte load, two 16-byte stores)
__global__ void __launch_bounds__(256)
ingest_mono8_kernel(const int16_t *in, size_t in_stride, float *x, size_t xs, long long n) {
    const long long i = 8 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= n) return;
    const int16_t *src = in + (size_t)blockIdx.y * in_stride + i;
    float *dst = x + (size_t)blockIdx.y * xs + i;
    if (i + 8 <= n) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(src));
        const int w[4] = {v.x, v.y, v.z, v.w};
        float f[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f[2 * k] = (float)(short)(w[k] & 0xffff);
            f[2 * k + 1] = (float)(short)(w[k] >> 16);
        }
        reinterpret_cast<float4 *>(dst)[0] = make_float4(f[0], f[1], f[2], f[3]);
        reinterpret_cast<float4 *>(dst)[1] = make_float4(f[4], f[5], f[6], f[7]);
    } else {
        for (long long k = i; k < n; ++k) dst[k - i] = (float)__ldg(src + (k - i));
    }
}

void launch_ingest_float(wefax_ctx *ctx, const int16_t *pcm, size_t pcm_stride, int channels, float *x, size_t xs,
                         long long n, int batch) {
    StageTimer timer(ctx, "ingest");
    if (channels == 1 && (reinterpret_cast<uintptr_t>(pcm) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
        (batch == 1 || (pcm_stride % 8 == 0 && xs % 4 == 0))) {
        dim3 g8((unsigned)((n + 2047) / 2048), batch);
        ingest_mono8_kernel<<<g8, 256, 0, ctx->stream>>>(pcm, pcm_stride, x, xs, n);
        CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
        return;
    }
    dim3 grid((unsigned)((n + 255) / 256), batch);
    if (channels == 2)
        ingest_kernel<kInStereoI16><<<grid, 256, 0, ctx->stream>>>(pcm, pcm_stride, x, xs, n);
    else
        ingest_kernel<kInMonoI16><<<grid, 256, 0, ctx->stream>>>(pcm, pcm_stride, x, xs, n);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// ===========================================================================
// zero-phase notch == scipy.signal.filtfilt(b, a, x)   (wefax.py:72)
// ===========================================================================
constexpr int kFirTile = 2048;
constexpr int kFirThreads = 256;
constexpr int kPadLen = 9;   // 3 * max(len(a), len(b))

template <int MODE, int KP>
__global__ void __launch_bounds__(kFirThreads)
filtfilt_kernel(const void *in, size_t in_stride, float *out, size_t out_stride, float2 *zout, size_t z_stride,
                long long n, const FirParams fp, int tiles_first, int tiles_skip) {
    constexpr int TS = kFirTile;
    constexpr int NEXT = TS + 2 * (KP - 1);          // extended-signal samples a tile needs
    constexpr int NEXT_AL = (NEXT + 16 + 3) & ~3;
    constexpr int NYF = TS + KP - 1;                 // forward-filtered samples a tile needs
    constexpr int NYF_AL = (NYF + 16 + 7) & ~7;
    constexpr int W = KP + 8;                        // register window: 8 outputs + KP - 1 history
    __shared__ __align__(16) float s_ext[NEXT_AL];
    __shared__ __align__(16) float s_yf[NYF_AL];

    const int tid = threadIdx.x;
    const size_t base = (size_t)blockIdx.y * in_stride;
    // the tiles between tiles_first and tiles_first + tiles_skip belong to notch_sym_kernel
    const long long tile = (int)blockIdx.x < tiles_first ? blockIdx.x : blockIdx.x + tiles_skip;
    const long long E = n + 2 * kPadLen;                              // length of the odd-extended signal
    const long long e0 = kPadLen + tile * TS;                         // first output of this tile, extended coords

    const long long e_first = e0 - (KP - 1);                          // extended index of s_ext[0]
    if (e_first >= kPadLen && e_first + NEXT <= n + kPadLen) {
        // interior tile: every sample is a plain input sample; keep all loads in flight
        const long long g0 = e_first - kPadLen;
        constexpr int ITER = (NEXT_AL + kFirThreads - 1) / kFirThreads;
        float v[ITER];
#pragma unroll
        for (int it = 0; it < ITER; ++it) {
            const int j = tid + it * kFirThreads;
            v[it] = j < NEXT ? load_sample<MODE>(in, base, g0 + j) : 0.f;
        }
#pragma unroll
        for (int it = 0; it < ITER; ++it) {
            const int j = tid + it * kFirThreads;
            if (j < NEXT_AL) s_ext[j] = v[it];
        }
    } else {
        for (int j = tid; j < NEXT_AL; j += kFirThreads) {
            long long e = e_first + j;
            float v = 0.f;
            if (j < NEXT) {
                if (e < 0) e = 0;   // steady-state initial condition: constant ext[0] to the left
                if (e < E) {
                    if (e < kPadLen)
                        v = 2.f * load_sample<MODE>(in, base, 0) - load_sample<MODE>(in, base, kPadLen - e);
                    else if (e >= n + kPadLen)
                        v = 2.f * load_sample<MODE>(in, base, n - 1) - load_sample<MODE>(in, base, 2 * n + 7 - e);
                    else
                        v = load_sample<MODE>(in, base, e - kPadLen);
                }
            }
            s_ext[j] = v;
        }
    }
    __syncthreads();

    // forward (causal) section: yf_rel[i] = sum_j hr[j] * ext_rel[i + j]
    for (int i0 = 8 * tid; i0 < NYF; i0 += 8 * kFirThreads) {
        float w[W];
#pragma unroll
        for (int q = 0; q < W / 4; ++q) {
            float4 t = *reinterpret_cast<const float4 *>(&s_ext[i0 + 4 * q]);
            w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
        }
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            const float c = fp.hr[j];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(c, w[i + j], acc[i]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) s_yf[i0 + i] = acc[i];
    }
    __syncthreads();

    // backward section starts from the steady state of the last forward sample
    const long long last_rel = (E - 1) - e0;
    if (last_rel < NYF - 1) {
        const float vlast = s_yf[last_rel];
        for (int j = (int)last_rel + 1 + tid; j < NYF_AL; j += kFirThreads) s_yf[j] = vlast;
    }
    __syncthreads();

    // backward (anti-causal) section: out[i] = sum_m h[m] * yf_rel[i + m]
    {
        const int i0 = 8 * tid;
        float w[W];
#pragma unroll
        for (int q = 0; q < W / 4; ++q) {
            float4 t = *reinterpret_cast<const float4 *>(&s_yf[i0 + 4 * q]);
            w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
        }
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
        for (int m = 0; m < KP; ++m) {
            const float c = fp.h[m];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(c, w[i + m], acc[i]);
        }
        // each thread owns 8 consecutive outputs: two 16-byte stores per thread, 1 KiB contiguous per warp
        const long long g = tile * TS + i0;
        if (out) {
            float *o = out + (size_t)blockIdx.y * out_stride + g;
            if (g + 7 < n && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {
                reinterpret_cast<float4 *>(o)[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
                reinterpret_cast<float4 *>(o)[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (g + i < n) o[i] = acc[i];
            }
        }
        // the complex copy (x, 0) a full-length transform reads through TMA
        if (zout) {
            float2 *z = zout + (size_t)blockIdx.y * z_stride + g;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (g + i < n) z[i] = make_float2(acc[i], 0.f);
        }
    }
}

// packed fp32 pairs (SASS FADD2 / FMUL2 / FFMA2): two samples per instruction, same IEEE roundings as the scalar forms
__device__ __forceinline__ float2 fir_add2(float2 a, float2 b) {
    float2 r;
    asm("{.reg .b64 ta, tb, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%5}; add.rn.f32x2 tr, ta, tb; mov.b64 {%0,%1}, tr;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 fir_mul2(float c, float2 a) {
    float2 r;
    asm("{.reg .b64 ta, tb, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%4}; mul.rn.f32x2 tr, ta, tb; mov.b64 {%0,%1}, tr;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(c));
    return r;
}
__device__ __forceinline__ float2 fir_fma2(float c, float2 a, float2 acc) {
    float2 r;
    asm("{.reg .b64 ta, tb, tc, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%4}; mov.b64 tc, {%5,%6}; "
        "fma.rn.f32x2 tr, ta, tb, tc; mov.b64 {%0,%1}, tr;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(c), "f"(acc.x), "f"(acc.y));
    return r;
}

// Interior tiles (further than the filter's memory from both ends of the signal): the two sections are one
// symmetric FIR, out[i] = g0 x[i] + sum_k g_k (x[i-k] + x[i+k]).  One shared-memory stage instead of two, half the
// multiplies; mono int16 comes in as one 16-byte load per thread.
// Persistent CTAs, kNotchSymCtas per SM with the window and both partial sums in registers (62).  Five per SM cap the
// registers at 48 and spill; they were measured no faster (DESIGN.md 4.1).
constexpr int kNotchSymCtas = 4;

template <int MODE, int KC>
__global__ void __launch_bounds__(kFirThreads, kNotchSymCtas)
notch_sym_kernel(const void *in, size_t in_stride, float *out, size_t out_stride, float2 *zout, size_t z_stride,
                 long long n, const FirParams fp, int tile0, int ntiles) {
    constexpr int TS = kFirTile;
    constexpr int NX = TS + 2 * KC;
    constexpr int W = 8 + 2 * KC;
    // Shared-memory layout: chunks of 8 samples, 12 floats apart.  A thread's window is W / 8 whole chunks; with a
    // 48-byte chunk pitch the 16-byte reads of the 8 lanes of a quarter-warp fall into 8 different bank groups (with
    // the natural 32-byte pitch lanes t and t + 4 collide on every read).
    constexpr int NXP = (NX / 8) * 12;
    static_assert(KC % 4 == 0 && NX % 8 == 0, "chunked layout needs whole chunks");
    auto sidx = [](int i) { return (i >> 3) * 12 + (i & 7); };
    __shared__ __align__(16) float s_x[2][NXP];
    const int tid = threadIdx.x;
    const size_t base = (size_t)blockIdx.y * in_stride;
    int t = blockIdx.x;                                   // persistent: tiles t, t + gridDim.x, ...
    if (t >= ntiles) return;
    // mono int16 whose tiles start on 16-byte boundaries: one 16-byte load per thread (+ the halo), issued a whole
    // tile ahead of its use
    bool vec = false;
    const int16_t *pcm16 = nullptr;
    if (MODE == kInMonoI16) {
        pcm16 = (const int16_t *)in + base + (long long)tile0 * TS;
        vec = (reinterpret_cast<uintptr_t>(pcm16) & 15) == 0;
    }
    int4 pv = make_int4(0, 0, 0, 0);
    int16_t ph = 0;
    auto prefetch = [&](int tile) {
        const int16_t *src = pcm16 + (long long)tile * TS;     // [src - KC, src + TS + KC) is inside the recording
        pv = __ldg(reinterpret_cast<const int4 *>(src) + tid);
        if (tid < 2 * KC) ph = __ldg(tid < KC ? src - KC + tid : src + TS + (tid - KC));
    };
    if (vec) prefetch(t);
    int buf = 0;
    while (true) {
        float *sx = s_x[buf];
        const long long t0 = (long long)(t + tile0) * TS;   // first output of the tile
        if (vec) {
            const int wv[4] = {pv.x, pv.y, pv.z, pv.w};
            float f[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                f[2 * k] = (float)(short)(wv[k] & 0xffff);
                f[2 * k + 1] = (float)(short)(wv[k] >> 16);
            }
            *reinterpret_cast<float4 *>(&sx[sidx(KC + 8 * tid)]) = make_float4(f[0], f[1], f[2], f[3]);
            *reinterpret_cast<float4 *>(&sx[sidx(KC + 8 * tid + 4)]) = make_float4(f[4], f[5], f[6], f[7]);
            if (tid < 2 * KC) sx[sidx(tid < KC ? tid : TS + tid)] = (float)ph;
        } else {
            constexpr int ITER = (NX + kFirThreads - 1) / kFirThreads;
            float v[ITER];
#pragma unroll
            for (int it = 0; it < ITER; ++it) {
                const int j = tid + it * kFirThreads;
                v[it] = j < NX ? load_sample<MODE>(in, base, t0 - KC + j) : 0.f;
            }
#pragma unroll
            for (int it = 0; it < ITER; ++it) {
                const int j = tid + it * kFirThreads;
                if (j < NX) sx[sidx(j)] = v[it];
            }
        }
        // one barrier per tile: the other buffer was last read before the previous barrier
        __syncthreads();
        const int tn = t + gridDim.x;
        if (vec && tn < ntiles) prefetch(tn);

        const int i0 = 8 * tid;
        // The window as aligned pairs wp[m] = (w[2m], w[2m+1]) (they are register pairs as the 16-byte loads deliver them),
        // so that one packed instruction (FADD2 / FFMA2) works on two outputs.  Even taps pair up outputs (2m, 2m+1),
        // odd taps outputs (2m+1, 2m+2): both then read only aligned pairs, and the two partial sums meet in 8 scalar adds.
        float2 wp[W / 2];
#pragma unroll
        for (int q = 0; q < W / 4; ++q) {
            const float4 x4 = *reinterpret_cast<const float4 *>(&sx[sidx(i0 + 4 * q)]);
            wp[2 * q] = make_float2(x4.x, x4.y);
            wp[2 * q + 1] = make_float2(x4.z, x4.w);
        }
        constexpr int H = KC / 2;               // wp[H + m] holds outputs (2m, 2m+1)
        float2 ae[4], ao[5];                    // ae[m]: outputs (2m, 2m+1);  ao[m]: outputs (2m-1, 2m)
#pragma unroll
        for (int m = 0; m < 4; ++m) ae[m] = fir_mul2(fp.g[0], wp[H + m]);
#pragma unroll
        for (int m = 0; m < 5; ++m) ao[m] = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 1; k <= KC; ++k) {
            const float c = fp.g[k];
            if (k % 2 == 0) {
#pragma unroll
                for (int m = 0; m < 4; ++m) ae[m] = fir_fma2(c, fir_add2(wp[H + m - k / 2], wp[H + m + k / 2]), ae[m]);
            } else {
                // outputs (2m-1, 2m): samples (KC + 2m - 1 -+ k, +1) = pairs H + m - (k+1)/2 and H + m + (k-1)/2
#pragma unroll
                for (int m = 0; m < 5; ++m)
                    ao[m] = fir_fma2(c, fir_add2(wp[H + m - (k + 1) / 2], wp[H + m + (k - 1) / 2]), ao[m]);
            }
        }
        float acc[8];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            acc[2 * m] = ae[m].x + ao[m].y;
            acc[2 * m + 1] = ae[m].y + ao[m + 1].x;
        }
        const long long g = t0 + i0;
        if (out) {
            float *o = out + (size_t)blockIdx.y * out_stride + g;
            if ((reinterpret_cast<uintptr_t>(o) & 15) == 0) {
                reinterpret_cast<float4 *>(o)[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
                reinterpret_cast<float4 *>(o)[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = acc[i];
            }
        }
        if (zout) {
            float2 *z = zout + (size_t)blockIdx.y * z_stride + g;
#pragma unroll
            for (int i = 0; i < 8; ++i) z[i] = make_float2(acc[i], 0.f);
        }
        if (tn >= ntiles) break;
        t = tn;
        buf ^= 1;
    }
}

template <int MODE, int KC>
static void launch_notch_sym(wefax_ctx *ctx, const void *in, size_t in_stride, float *out, size_t out_stride, float2 *zout,
                             size_t z_stride, long long n, const FirParams &fp, int batch, int tile0, int ntiles) {
    const int per_rec = std::max(1, (ctx->sm_count * kNotchSymCtas + batch - 1) / batch);
    dim3 grid((unsigned)std::min(ntiles, per_rec), batch);
    notch_sym_kernel<MODE, KC><<<grid, kFirThreads, 0, ctx->stream>>>(in, in_stride, out, out_stride, zout, z_stride, n, fp,
                                                                      tile0, ntiles);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

template <int MODE>
static void launch_filtfilt_mode(wefax_ctx *ctx, const void *in, size_t in_stride, float *out, size_t out_stride,
                                 float2 *zout, size_t z_stride, long long n, const FirParams &fp, int batch) {
    StageTimer timer(ctx, "filtfilt");
    const int ntiles = (int)((n + kFirTile - 1) / kFirTile);
    // tiles [ti_lo, ti_hi) are further than the filter's memory from both ends: symmetric single-stage form
    int ti_lo = 0, ti_hi = 0;
    if (fp.KC > 0) {
        const long long margin = 2ll * fp.KP + 16;
        ti_lo = (int)((margin + kFirTile - 1) / kFirTile);
        ti_hi = (int)std::max<long long>(0, (n - margin) / kFirTile);
        if (ti_hi <= ti_lo) ti_lo = ti_hi = 0;
    }
    if (ti_hi > ti_lo) {
        switch (fp.KC) {
#define WEFAX_SYM_CASE(KC_) \
    case KC_: launch_notch_sym<MODE, KC_>(ctx, in, in_stride, out, out_stride, zout, z_stride, n, fp, batch, ti_lo, ti_hi - ti_lo); break;
            WEFAX_SYM_CASE(8)
            WEFAX_SYM_CASE(12)
            WEFAX_SYM_CASE(16)
            WEFAX_SYM_CASE(24)
            WEFAX_SYM_CASE(32)
#undef WEFAX_SYM_CASE
            default: ti_lo = ti_hi = 0; break;
        }
    }
    const int tiles_first = ti_lo, tiles_skip = ti_hi - ti_lo;
    dim3 grid((unsigned)(ntiles - tiles_skip), batch);
#define WEFAX_FIR_CASE(KP_)                                                                                   \
    if (fp.KP == KP_) {                                                                                       \
        filtfilt_kernel<MODE, KP_><<<grid, kFirThreads, 0, ctx->stream>>>(in, in_stride, out, out_stride, zout, z_stride, n, fp, \
                                                                          tiles_first, tiles_skip);         \
        CUDA_CHECK(cudaGetLastError());                                                                       \
        ctx->launches++;                                                                                      \
        return;                                                                                               \
    }
    WEFAX_FIR_CASE(16)
    WEFAX_FIR_CASE(20)
    WEFAX_FIR_CASE(24)
    WEFAX_FIR_CASE(32)
    WEFAX_FIR_CASE(48)
    WEFAX_FIR_CASE(64)
#undef WEFAX_FIR_CASE
    WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "notch impulse response needs %d taps (max %d)", fp.K, kMaxFirTaps);
}

// ---------------------------------------------------------------------------
// Recursive form for notches whose impulse response is too long for the FIR kernels (high quality factor, or a
// high sample rate in front of the filter as in the live path's packets, data_packet.py:421-431): scipy's
// filtfilt itself - odd extension by 9, lfilter with zi * ext[0], the same backwards - in float64, one thread per
// block of kIirBlock samples.  A block that does not start at the signal's edge warms up from zero state over
// `warm` samples, by which the response has decayed below 3e-9 of its sum (the FIR form's truncation rule).
// ---------------------------------------------------------------------------
constexpr int kIirBlock = 2048;

template <int MODE>
__device__ __forceinline__ double iir_ext(const void *in, size_t base, long long e, long long n) {
    // odd extension (scipy signaltools.odd_ext, padlen 9) of the ingested signal, extended index e in [0, n + 18)
    if (e < kPadLen) return 2.0 * (double)load_sample<MODE>(in, base, 0) - (double)load_sample<MODE>(in, base, kPadLen - e);
    if (e >= n + kPadLen)
        return 2.0 * (double)load_sample<MODE>(in, base, n - 1) - (double)load_sample<MODE>(in, base, 2 * n + 7 - e);
    return (double)load_sample<MODE>(in, base, e - kPadLen);
}

template <int MODE>
__global__ void __launch_bounds__(128)
iir_forward_kernel(const void *in, size_t in_stride, double *yf, size_t yf_stride, long long n, const FirParams fp) {
    const long long E = n + 2 * kPadLen;
    const long long blk = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long start = blk * kIirBlock;
    if (start >= E) return;
    const long long end = min(start + kIirBlock, E);
    const size_t base = (size_t)blockIdx.y * in_stride;
    double *y_out = yf + (size_t)blockIdx.y * yf_stride;
    const double b0 = fp.b[0], b1 = fp.b[1], b2 = fp.b[2], a1 = fp.a[1], a2 = fp.a[2];
    long long i = start - fp.warm;
    double z0 = 0.0, z1 = 0.0;
    if (i <= 0) {
        i = 0;
        const double x0 = iir_ext<MODE>(in, base, 0, n);
        z0 = fp.zi[0] * x0;
        z1 = fp.zi[1] * x0;
    }
    for (; i < end; ++i) {
        const double x = iir_ext<MODE>(in, base, i, n);
        const double y = b0 * x + z0;
        z0 = b1 * x - a1 * y + z1;
        z1 = b2 * x - a2 * y;
        if (i >= start) y_out[i] = y;
    }
}

__global__ void __launch_bounds__(128)
iir_backward_kernel(const double *yf, size_t yf_stride, float *out, size_t out_stride, float2 *zout, size_t z_stride,
                    long long n, const FirParams fp) {
    // reversed coordinate j = E - 1 - i: lfilter over yf reversed, zi * yf[E - 1]; sample j is output E - 1 - j - 9
    const long long E = n + 2 * kPadLen;
    const long long blk = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long start = blk * kIirBlock;
    if (start >= E) return;
    const long long end = min(start + kIirBlock, E);
    const double *y_in = yf + (size_t)blockIdx.y * yf_stride;
    const double b0 = fp.b[0], b1 = fp.b[1], b2 = fp.b[2], a1 = fp.a[1], a2 = fp.a[2];
    long long j = start - fp.warm;
    double z0 = 0.0, z1 = 0.0;
    if (j <= 0) {
        j = 0;
        const double x0 = y_in[E - 1];
        z0 = fp.zi[0] * x0;
        z1 = fp.zi[1] * x0;
    }
    for (; j < end; ++j) {
        const double x = y_in[E - 1 - j];
        const double y = b0 * x + z0;
        z0 = b1 * x - a1 * y + z1;
        z1 = b2 * x - a2 * y;
        const long long o = E - 1 - j - kPadLen;
        if (j >= start && o >= 0 && o < n) {
            if (out) out[(size_t)blockIdx.y * out_stride + o] = (float)y;
            if (zout) zout[(size_t)blockIdx.y * z_stride + o] = make_float2((float)y, 0.f);
        }
    }
}

static void launch_filtfilt_iir(wefax_ctx *ctx, IngestMode mode, const void *in, size_t in_stride, float *out,
                                size_t out_stride, float2 *zout, size_t z_stride, long long n, const FirParams &fp,
                                int batch) {
    StageTimer timer(ctx, "filtfilt");
    const long long E = n + 2 * kPadLen;
    const size_t ys = (size_t)((E + 1) & ~1ll);
    double *yf = (double *)ctx->iir_tmp.reserve(ys * (size_t)batch * sizeof(double));
    const long long nblk = (E + kIirBlock - 1) / kIirBlock;
    dim3 grid((unsigned)((nblk + 127) / 128), batch);
    switch (mode) {
        case kInMonoI16: iir_forward_kernel<kInMonoI16><<<grid, 128, 0, ctx->stream>>>(in, in_stride, yf, ys, n, fp); break;
        case kInStereoI16: iir_forward_kernel<kInStereoI16><<<grid, 128, 0, ctx->stream>>>(in, in_stride, yf, ys, n, fp); break;
        default: iir_forward_kernel<kInFloat><<<grid, 128, 0, ctx->stream>>>(in, in_stride, yf, ys, n, fp); break;
    }
    iir_backward_kernel<<<grid, 128, 0, ctx->stream>>>(yf, ys, out, out_stride, zout, z_stride, n, fp);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches += 2;
}

void launch_filtfilt(wefax_ctx *ctx, IngestMode mode, const void *in, size_t in_stride, float *out, size_t out_stride,
                     float2 *zout, size_t z_stride, long long n, const FirParams &fp, int batch) {
    if (fp.iir) {
        launch_filtfilt_iir(ctx, mode, in, in_stride, out, out_stride, zout, z_stride, n, fp, batch);
        return;
    }
    switch (mode) {
        case kInMonoI16:
            launch_filtfilt_mode<kInMonoI16>(ctx, in, in_stride, out, out_stride, zout, z_stride, n, fp, batch);
            break;
        case kInStereoI16:
            launch_filtfilt_mode<kInStereoI16>(ctx, in, in_stride, out, out_stride, zout, z_stride, n, fp, batch);
            break;
        default:
            launch_filtfilt_mode<kInFloat>(ctx, in, in_stride, out, out_stride, zout, z_stride, n, fp, batch);
            break;
    }
}

__global__ void median5_kernel(const float *env, size_t es, float *out, size_t os, long long n) {
    const float *e = env + (size_t)blockIdx.y * es;
    float *o = out + (size_t)blockIdx.y * os;
    long long i0 = 4 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
    if (i0 >= n) return;
    float m[4];
    load_med4(e, i0, n, m);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (i0 + j < n) o[i0 + j] = m[j];
}

void launch_median5(wefax_ctx *ctx, const float *env, size_t es, float *out, size_t os, long long n, int batch) {
    StageTimer timer(ctx, "median5");
    dim3 grid((unsigned)((n + 1023) / 1024), batch);
    median5_kernel<<<grid, 256, 0, ctx->stream>>>(env, es, out, os, n);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// ===========================================================================
// numpy.percentile(env, (0.5, 99.5))  (wefax.py:196): exact order statistics by a
// 3-level radix select on the float bit pattern (11 + 11 + 10 bits), then numpy's
// linear interpolation in double.
// ===========================================================================
__device__ __forceinline__ int level_shift(int level) { return level == 0 ? 21 : (level == 1 ? 10 : 0); }
__device__ __forceinline__ uint32_t level_mask(int level) { return level == 2 ? 0x3FFu : 0x7FFu; }

template <int LEVEL, int MED>
__global__ void __launch_bounds__(256) hist_kernel(const float *env, size_t es, long long n, SelState *sel_all) {
    constexpr int NH = LEVEL == 0 ? 1 : 4;
    __shared__ uint32_t s_hist[NH][2048];
    SelState *sel = sel_all + blockIdx.y;
    const float *e = env + (size_t)blockIdx.y * es;
    for (int i = threadIdx.x; i < NH * 2048; i += blockDim.x) (&s_hist[0][0])[i] = 0;
    uint32_t prefix[4];
    if (LEVEL > 0) {
#pragma unroll
        for (int t = 0; t < 4; ++t) prefix[t] = sel->prefix[t];
    }
    __syncthreads();

    const long long stride = 4ll * blockDim.x * gridDim.x;
    for (long long i0 = 4 * ((long long)blockIdx.x * blockDim.x + threadIdx.x); i0 < ((n + stride - 1) / stride) * stride;
         i0 += stride) {
        float m[4] = {0.f, 0.f, 0.f, 0.f};
        if (i0 < n) load_med4<MED>(e, i0, n, m);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool valid = i0 + j < n;
            const uint32_t key = __float_as_uint(m[j]);
            if (LEVEL == 0) {
                // warp-aggregated: the envelope is concentrated in a few exponent bins
                const uint32_t bin = valid ? (key >> 21) : 0xFFFFFFFFu;
                const unsigned peers = __match_any_sync(0xFFFFFFFFu, bin);
                if (valid && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[0][bin], __popc(peers));
            } else if (valid) {
                const uint32_t hi = key >> (LEVEL == 1 ? 21 : 10);
                const uint32_t bin = (key >> level_shift(LEVEL)) & level_mask(LEVEL);
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (hi == prefix[t]) atomicAdd(&s_hist[t % NH][bin], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NH * 2048; i += blockDim.x) {
        uint32_t c = (&s_hist[0][0])[i];
        if (c) atomicAdd(&sel->hist[LEVEL][i >> 11][i & 2047], c);
    }
}

__global__ void select_init_kernel(SelState *sel_all, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    SelState *sel = sel_all + blockIdx.x;
    if (threadIdx.x == 0) {
        sel->rank[0] = r0; sel->rank[1] = r1; sel->rank[2] = r2; sel->rank[3] = r3;
        sel->prefix[0] = sel->prefix[1] = sel->prefix[2] = sel->prefix[3] = 0;
    }
}

// one block (256 threads) per recording: locate, for each of the 4 target ranks, the
// histogram bin that contains it
__global__ void __launch_bounds__(256)
select_kernel(SelState *sel_all, int level, RecResult *res_all, double t_lo, double t_hi) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_bin[4], s_before[4];
    SelState *sel = sel_all + blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int bits = level == 2 ? 10 : 11;
    for (int t = 0; t < 4; ++t) {
        const uint32_t *hist = sel->hist[level][level == 0 ? 0 : t];
        const uint32_t rank = sel->rank[t];
        uint32_t c[8], local = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c[j] = hist[8 * tid + j];
            local += c[j];
        }
        uint32_t incl = local;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        uint32_t woff = 0;
        for (int w = 0; w < wid; ++w) woff += s_warp[w];
        uint32_t before = woff + incl - local;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (rank >= before && rank < before + c[j]) {
                s_bin[t] = 8 * tid + j;
                s_before[t] = before;
            }
            before += c[j];
        }
        __syncthreads();
    }
    if (tid < 4) {
        sel->prefix[tid] = (sel->prefix[tid] << bits) | s_bin[tid];
        sel->rank[tid] -= s_before[tid];
    }
    __syncthreads();
    if (level == 2 && tid == 0) {
        // numpy _lerp: a + (b-a)*t for t < 0.5, b - (b-a)*(1-t) otherwise (no FMA contraction)
        double v[4];
        for (int t = 0; t < 4; ++t) v[t] = (double)__uint_as_float(sel->prefix[t]);
        double d0 = __dsub_rn(v[1], v[0]), d1 = __dsub_rn(v[3], v[2]);
        double low = t_lo >= 0.5 ? __dsub_rn(v[1], __dmul_rn(d0, __dsub_rn(1.0, t_lo))) : __dadd_rn(v[0], __dmul_rn(d0, t_lo));
        double high = t_hi >= 0.5 ? __dsub_rn(v[3], __dmul_rn(d1, __dsub_rn(1.0, t_hi))) : __dadd_rn(v[2], __dmul_rn(d1, t_hi));
        RecResult *res = res_all + blockIdx.x;
        res->low = low;
        res->high = high;
        double delta = __dsub_rn(high, low);
        if (!(delta > 0.0) || isinf(delta)) res->status |= WEFAX_REC_NAN;
    }
}

// ---------------------------------------------------------------------------
// Bracketed selection for long recordings: one light pass over the data instead of
// three histogram passes.
//   1. every 61st median-filtered sample goes into a small array;
//   2. one CTA selects, exactly, four order statistics of that sample: values that
//      bracket the 0.5 and 99.5 percentile with a wide safety margin;
//   3. one pass over the data counts the elements below each bracket and copies the
//      (few) elements inside into a list;
//   4. one CTA selects the exact order statistics inside the lists and checks that
//      the wanted ranks really fell inside the brackets.  If not (or a list
//      overflowed) a flag makes the fallback kernel redo the selection exactly over
//      the whole data, so the result is always the exact numpy.percentile value.
// ---------------------------------------------------------------------------
constexpr int kPctStride = 127;
constexpr int kSelThreads = 1024;

struct PctGeom {
    long long n, ns;               // samples, sub-sampled count
    uint32_t s_rank[4];            // sample ranks of the bracket ends: lo_a, lo_b, hi_a, hi_b
    int open_lo, open_hi;          // bracket reaches the end of the sample: extend to -inf / +inf
    uint32_t r[4];                 // wanted ranks: i_lo, i_lo+1, i_hi, i_hi+1 (clipped)
    double t_lo, t_hi;             // numpy lerp weights
    uint32_t cap;                  // capacity of each candidate list
};

struct PctState {                  // per recording, device
    uint32_t key[4];               // bracket keys lo_a, lo_b, hi_a, hi_b
    unsigned long long below[2];   // elements with key < lo_a / key > hi_b (pct_collect2_kernel)
    uint32_t len[2];               // candidates collected in each list (may exceed cap: overflow)
    int fallback;
    uint32_t out_key[4];           // order statistics found by the two halves of the final selection
    unsigned int done;             // halves that have delivered their keys
};

// Exact selection of NT order statistics among `count` keys produced by key_at(i),
// by the `ncta` co-resident CTAs (kSelThreads threads each) that serve one
// recording: 3 radix levels (11 + 11 + 10 bits); every CTA histograms its slice in
// shared memory, adds it to the recording's global histogram, the CTAs meet at a
// barrier and each of them locates the targets' bins (so all hold the same state).
// ranks[] in (s_rank), keys out (s_prefix).  ghist: 3 levels x NT x 2048 zeroed words.
struct CoopSync {
    unsigned int arrived;   // monotonically increasing barrier counter
};

__device__ __forceinline__ void coop_barrier(CoopSync *cs, unsigned ncta, unsigned &phase) {
    __syncthreads();
    if (threadIdx.x == 0) {
        ++phase;
        if (ncta > 1) {
            __threadfence();
            atomicAdd(&cs->arrived, 1u);
            while (*((volatile unsigned int *)&cs->arrived) < phase * ncta) {
            }
            __threadfence();
        }
    }
    __syncthreads();
}

// nbar: CTAs that meet at the barrier (0: ncta).  With ncta = 1, cta = 0 and nbar = the real number of CTAs every CTA
// histograms its OWN keys (e.g. a slice it holds in shared memory) and the CTAs still select together.
template <int NT, class KeyAt>
__device__ void coop_select(KeyAt key_at, long long count, int cta, unsigned ncta, CoopSync *cs, unsigned &phase,
                            uint32_t *ghist, uint32_t *s_hist /* NT*2048 */, uint32_t *s_rank, uint32_t *s_prefix,
                            uint32_t *s_scan /* 32 */, unsigned nbar = 0, int nlevels = 3, int first_level = 0,
                            uint32_t known_prefix = 0) {
    if (nbar == 0) nbar = ncta;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // first_level > 0: every key is known to start with known_prefix (11 or 22 bits), those levels are skipped
    if (tid < NT) s_prefix[tid] = known_prefix;
    // nlevels < 3: the prefixes stop after 11 or 22 bits (the caller completes them conservatively)
    for (int level = first_level; level < nlevels; ++level) {
        const int shift = level == 0 ? 21 : (level == 1 ? 10 : 0);
        const uint32_t mask = level == 2 ? 0x3FFu : 0x7FFu;
        const int nh = level == 0 ? 1 : NT;           // level 0: all targets share one histogram
        uint32_t *gh = ghist + (size_t)level * NT * 2048;
        for (int i = tid; i < nh * 2048; i += kSelThreads) s_hist[i] = 0;
        __syncthreads();
        uint32_t pre[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) pre[t] = s_prefix[t];
        // 8 independent loads per thread are issued before any of them is consumed
        constexpr int U = 8;
        const long long span = (long long)U * kSelThreads;
        const long long rounds = (count + span * ncta - 1) / (span * ncta);
        for (long long it = 0; it < rounds; ++it) {
            uint32_t key[U];
            bool valid[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const long long i = ((it * ncta + cta) * U + u) * kSelThreads + tid;
                valid[u] = i < count;
                key[u] = valid[u] ? key_at(i) : 0xFFFFFFFFu;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (level == 0) {
                    // keys are concentrated in a few bins: lanes with equal bins share one atomic
                    const uint32_t bin = valid[u] ? (key[u] >> 21) : 0xFFFFFFFFu;
                    const unsigned peers = __match_any_sync(0xFFFFFFFFu, bin);
                    if (valid[u] && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (uint32_t)__popc(peers));
                } else if (valid[u]) {
                    const uint32_t hi = key[u] >> (level == 1 ? 21 : 10);
                    const uint32_t bin = (key[u] >> shift) & mask;
#pragma unroll
                    for (int t = 0; t < NT; ++t)
                        if (hi == pre[t]) atomicAdd(&s_hist[t * 2048 + bin], 1u);
                }
            }
        }
        __syncthreads();
        for (int i = tid; i < nh * 2048; i += kSelThreads) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(&gh[i], c);
        }
        coop_barrier(cs, nbar, phase);
        // locate each target in the recording-wide histogram: thread tid owns bins 2*tid, 2*tid+1
        for (int t = 0; t < NT; ++t) {
            const int hsel = level == 0 ? 0 : t;
            const uint32_t c0 = __ldcg(&gh[hsel * 2048 + 2 * tid]), c1 = __ldcg(&gh[hsel * 2048 + 2 * tid + 1]);
            uint32_t incl = c0 + c1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= d) incl += v;
            }
            if (lane == 31) s_scan[wid] = incl;
            __syncthreads();
            uint32_t woff = 0;
            for (int w = 0; w < wid; ++w) woff += s_scan[w];
            uint32_t before = woff + incl - (c0 + c1);
            const uint32_t rank = s_rank[t];
            uint32_t found_bin = 0xFFFFFFFFu, found_before = 0;
            if (rank >= before && rank < before + c0) {
                found_bin = 2 * tid;
                found_before = before;
            } else if (rank >= before + c0 && rank < before + c0 + c1) {
                found_bin = 2 * tid + 1;
                found_before = before + c0;
            }
            __syncthreads();
            if (found_bin != 0xFFFFFFFFu) {
                s_prefix[t] = (pre[t] << (level == 2 ? 10 : 11)) | found_bin;
                s_rank[t] = rank - found_before;
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(256)
pct_sample_kernel(const float *env, size_t es, PctGeom g, float *samp, size_t ss) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= g.ns) return;
    const float *e = env + (size_t)blockIdx.y * es;
    const long long i = s * kPctStride;
    float w[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const long long k = i - 2 + j;
        w[j] = (k >= 0 && k < g.n) ? __ldg(e + k) : 0.f;
    }
    samp[(size_t)blockIdx.y * ss + s] = med5(w[0], w[1], w[2], w[3], w[4]);
}

// scratch of the cooperative selections of one recording (zeroed before every use)
struct PctCoop {
    CoopSync sync[3];                // bracket kernel, final kernel (low list, high list)
    uint32_t hist[3][3 * 4 * 2048];  // [sample | low list | high list][level][target][bin]
};

__global__ void __launch_bounds__(kSelThreads)
pct_bracket_kernel(const float *samp, size_t ss, PctGeom g, PctState *st_all, PctCoop *coop_all, int ncta) {
    __shared__ uint32_t s_hist[4 * 2048];
    __shared__ uint32_t s_rank[4], s_prefix[4], s_scan[32];
    const int rec = blockIdx.x / ncta, cta = blockIdx.x % ncta;
    const float *sp = samp + (size_t)rec * ss;
    PctCoop *coop = coop_all + rec;
    if (threadIdx.x < 4) s_rank[threadIdx.x] = g.s_rank[threadIdx.x];
    __syncthreads();
    unsigned phase = 0;
    coop_select<4>([&](long long i) { return __float_as_uint(__ldg(sp + i)); }, g.ns, cta, (unsigned)ncta, &coop->sync[0],
                   phase, coop->hist[0], s_hist, s_rank, s_prefix, s_scan);
    if (cta == 0 && threadIdx.x == 0) {
        PctState *st = st_all + rec;
        st->key[0] = g.open_lo ? 0u : s_prefix[0];
        st->key[1] = s_prefix[1];
        st->key[2] = s_prefix[2];
        st->key[3] = g.open_hi ? 0xFFFFFFFFu : s_prefix[3];
        st->below[0] = st->below[1] = 0;
        st->len[0] = st->len[1] = 0;
        st->fallback = 0;
        st->done = 0;
    }
}

// pct_sample_kernel + pct_bracket_kernel in one: every CTA takes its slice of the sample positions, keeps the
// medians' keys in shared memory, and the three radix levels of the cooperative selection read them from there.
__global__ void __launch_bounds__(kSelThreads)
pct_bracket2_kernel(const float *env, size_t es, PctGeom g, PctState *st_all, PctCoop *coop_all, int ncta, int per) {
    extern __shared__ uint32_t s_brk[];
    uint32_t *s_hist = s_brk;                 // 4 * 2048
    uint32_t *s_keys = s_brk + 4 * 2048;      // per
    __shared__ uint32_t s_rank[4], s_prefix[4], s_scan[32];
    const int rec = blockIdx.x / ncta, cta = blockIdx.x % ncta;
    const float *e = env + (size_t)rec * es;
    PctCoop *coop = coop_all + rec;
    const long long s0 = (long long)cta * per;
    const int cnt = (int)max(0ll, min((long long)per, g.ns - s0));
#pragma unroll 4
    for (int j = threadIdx.x; j < cnt; j += kSelThreads) {
        const long long i = (s0 + j) * kPctStride;
        float w[5];
#pragma unroll
        for (int t = 0; t < 5; ++t) {
            const long long k = i - 2 + t;
            w[t] = (k >= 0 && k < g.n) ? __ldg(e + k) : 0.f;
        }
        s_keys[j] = __float_as_uint(med5(w[0], w[1], w[2], w[3], w[4]));
    }
    if (threadIdx.x < 4) s_rank[threadIdx.x] = g.s_rank[threadIdx.x];
    __syncthreads();
    unsigned phase = 0;
    // Two radix levels (22 of the 32 key bits) are enough for a BRACKET: its lower ends round down, its upper ends
    // round up to the 1024-pattern bin that holds the sample's order statistic (a few hundred more candidates out
    // of tens of thousands), and one grid-wide barrier round less.
    coop_select<4>([&](long long i) { return s_keys[i]; }, (long long)cnt, 0, 1u, &coop->sync[0], phase, coop->hist[0], s_hist,
                   s_rank, s_prefix, s_scan, (unsigned)ncta, 2);
    if (cta == 0 && threadIdx.x == 0) {
        PctState *st = st_all + rec;
        st->key[0] = g.open_lo ? 0u : (s_prefix[0] << 10);
        st->key[1] = (s_prefix[1] << 10) | 0x3FFu;
        st->key[2] = s_prefix[2] << 10;
        st->key[3] = g.open_hi ? 0xFFFFFFFFu : ((s_prefix[3] << 10) | 0x3FFu);
        st->below[0] = st->below[1] = 0;
        st->len[0] = st->len[1] = 0;
        st->fallback = 0;
        st->done = 0;
    }
}

constexpr int kPctStage = 1024;   // per-CTA staging of candidates before one global append

// Candidates of both brackets into their lists.  The samples outside the two brackets' span (99 % of them lie
// strictly between the brackets) cost one subtract, one compare and one warp vote each; only warps that hold a
// sample in a tail or a bracket enter the classification.  Counts: below[0] = samples under the low bracket,
// below[1] = samples ABOVE the high bracket (the final selection derives its rank offset from it).
__global__ void __launch_bounds__(256)
pct_collect2_kernel(const float *env, size_t es, PctGeom g, PctState *st_all, float *lists, size_t ls) {
    __shared__ unsigned long long s_cnt_out[2];
    __shared__ float s_cand[2][kPctStage];
    __shared__ uint32_t s_cnt[2], s_base[2];
    PctState *st = st_all + blockIdx.y;
    const float *e = env + (size_t)blockIdx.y * es;
    float *list[2] = {lists + (size_t)blockIdx.y * ls, lists + (size_t)blockIdx.y * ls + g.cap};
    const uint32_t k0 = st->key[0], k1 = st->key[1], k2 = st->key[2], k3 = st->key[3];
    if (threadIdx.x < 2) {
        s_cnt_out[threadIdx.x] = 0;
        s_cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    auto append = [&](int h, float v) {
        const uint32_t slot = atomicAdd(&s_cnt[h], 1u);
        if (slot < kPctStage) {
            s_cand[h][slot] = v;
        } else {                                    // staging full (pathological data): append directly
            const uint32_t gslot = atomicAdd(&st->len[h], 1u);
            if (gslot < g.cap) list[h][gslot] = v;
        }
    };
    // middle = k1 < key < k2  <=>  key - (k1 + 1) < k2 - k1 - 1 (unsigned); brackets that touch or overlap make
    // the span empty: every sample is then classified
    const uint32_t mid_lo = k1 + 1u, mid_span = k2 > k1 ? k2 - k1 - 1u : 0u;
    uint32_t n_under = 0, n_over = 0;
    const long long n = g.n;
    const long long stride = 8ll * blockDim.x * gridDim.x;
    const long long rounds = (n + stride - 1) / stride;   // every thread runs every round: the votes are warp-wide
    long long i0 = 8 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
    for (long long it = 0; it < rounds; ++it, i0 += stride) {
        float m[8];
        int nvalid = 0;
        bool need = false;   // this thread may hold a median outside the middle
        float f[16];
        bool fast = false;
        if (i0 < n) {
            nvalid = (int)min(8ll, n - i0);
            fast = i0 >= 4 && i0 + 12 <= n && (reinterpret_cast<uintptr_t>(e + i0) & 15) == 0;
            if (fast) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 v = __ldg(reinterpret_cast<const float4 *>(e + i0 - 4) + q);
                    f[4 * q] = v.x; f[4 * q + 1] = v.y; f[4 * q + 2] = v.z; f[4 * q + 3] = v.w;
                }
                // A median of 5 lies outside the middle only if at least 3 of its 5 values do: fewer than 3 such
                // values among the 12 this thread's 8 windows cover settles all 8 at once (the usual case: 99 % of
                // the samples are in the middle), without a single median.
                int outside = 0;
#pragma unroll
                for (int j = 2; j < 14; ++j) outside += (__float_as_uint(f[j]) - mid_lo >= mid_span) ? 1 : 0;
                need = outside >= 3;
            } else {
                need = true;
            }
        }
        if (!__any_sync(0xFFFFFFFFu, need)) continue;
        if (i0 < n) {
            if (fast) med8_from16<2>(f, m);
            else load_med8(e, i0, n, m);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) m[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t key = __float_as_uint(m[j]);
            const bool out_mid = (key - mid_lo >= mid_span) && j < nvalid;
            if (__any_sync(0xFFFFFFFFu, out_mid)) {
                if (out_mid) {
                    if (key <= k1) {
                        if (key < k0) n_under++;
                        else append(0, m[j]);
                    }
                    if (key >= k2) {
                        if (key > k3) n_over++;
                        else append(1, m[j]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        n_under += __shfl_xor_sync(0xFFFFFFFFu, n_under, d);
        n_over += __shfl_xor_sync(0xFFFFFFFFu, n_over, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_cnt_out[0], (unsigned long long)n_under);
        atomicAdd(&s_cnt_out[1], (unsigned long long)n_over);
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        atomicAdd(&st->below[threadIdx.x], s_cnt_out[threadIdx.x]);
        const uint32_t c = min(s_cnt[threadIdx.x], (uint32_t)kPctStage);
        s_cnt[threadIdx.x] = c;
        s_base[threadIdx.x] = c ? atomicAdd(&st->len[threadIdx.x], c) : 0u;
    }
    __syncthreads();
    for (int h = 0; h < 2; ++h)
        for (uint32_t i = threadIdx.x; i < s_cnt[h]; i += blockDim.x)
            if (s_base[h] + i < g.cap) list[h][s_base[h] + i] = s_cand[h][i];
}

__device__ void write_percentiles(RecResult *res, const uint32_t key[4], double t_lo, double t_hi) {
    // numpy _lerp: a + (b-a)*t for t < 0.5, b - (b-a)*(1-t) otherwise (no FMA contraction)
    double v[4];
    for (int t = 0; t < 4; ++t) v[t] = (double)__uint_as_float(key[t]);
    double d0 = __dsub_rn(v[1], v[0]), d1 = __dsub_rn(v[3], v[2]);
    double low = t_lo >= 0.5 ? __dsub_rn(v[1], __dmul_rn(d0, __dsub_rn(1.0, t_lo))) : __dadd_rn(v[0], __dmul_rn(d0, t_lo));
    double high = t_hi >= 0.5 ? __dsub_rn(v[3], __dmul_rn(d1, __dsub_rn(1.0, t_hi))) : __dadd_rn(v[2], __dmul_rn(d1, t_hi));
    res->low = low;
    res->high = high;
    double delta = __dsub_rn(high, low);
    if (!(delta > 0.0) || isinf(delta)) res->status |= WEFAX_REC_NAN;
}

__global__ void __launch_bounds__(kSelThreads)
pct_final_kernel(PctGeom g, PctState *st_all, const float *lists, size_t ls, RecResult *res_all, PctCoop *coop_all,
                 int ncta, int local_per) {
    __shared__ uint32_t s_hist[2 * 2048];
    __shared__ uint32_t s_rank[2], s_prefix[2], s_scan[32], s_key[4];
    const int rec = blockIdx.x / ncta, cta = blockIdx.x % ncta;
    PctState *st = st_all + rec;
    PctCoop *coop = coop_all + rec;
    const float *list_lo = lists + (size_t)rec * ls, *list_hi = list_lo + g.cap;
    // every CTA of the recording takes the same decision from the same data
    bool ok = st->len[0] <= g.cap && st->len[1] <= g.cap;
    // samples under each bracket
    const unsigned long long below_of[2] = {st->below[0], (unsigned long long)g.n - st->below[1] - st->len[1]};
    for (int h = 0; h < 2 && ok; ++h) {
        const unsigned long long b = below_of[h];
        ok = b <= g.r[2 * h] && (unsigned long long)g.r[2 * h + 1] < b + st->len[h];
    }
    if (!ok) {
        if (cta == 0 && threadIdx.x == 0) st->fallback = 1;
        return;
    }
    unsigned phase = 0;
    if (ncta >= 2) {
        // the CTAs of the recording split into two groups that select in the two lists at the same time
        const int h = cta & 1, gcta = cta >> 1;
        const unsigned gn = (unsigned)((ncta + 1 - h) >> 1);
        const float *lst = h ? list_hi : list_lo;
        if (threadIdx.x < 2) s_rank[threadIdx.x] = g.r[2 * h + threadIdx.x] - (uint32_t)below_of[h];
        // every key of the list lies inside its bracket: the leading bits the bracket's two ends share are known, and a
        // radix level that only confirms them (one grid-wide barrier round each) is skipped
        const uint32_t klo = st->key[2 * h], khi = st->key[2 * h + 1];
        const int first = ((klo ^ khi) >> 21) != 0u ? 0 : (((klo ^ khi) >> 10) != 0u ? 1 : 2);
        const uint32_t known = first == 0 ? 0u : (first == 1 ? klo >> 21 : klo >> 10);
        if (local_per > 0) {
            // this CTA's slice of the list goes to shared memory once; the three radix levels read it from there
            extern __shared__ uint32_t s_fin[];
            const long long len = (long long)st->len[h];
            const long long per = (len + gn - 1) / gn, s0 = (long long)gcta * per;
            const int cnt = (int)max(0ll, min(per, len - s0));   // per <= local_per (the launcher sized it from cap)
            for (int j = threadIdx.x; j < cnt; j += kSelThreads) s_fin[j] = __float_as_uint(__ldg(lst + s0 + j));
            __syncthreads();
            coop_select<2>([&](long long i) { return s_fin[i]; }, (long long)cnt, 0, 1u, &coop->sync[1 + h], phase,
                           coop->hist[1 + h], s_hist, s_rank, s_prefix, s_scan, gn, 3, first, known);
        } else {
            __syncthreads();
            coop_select<2>([&](long long i) { return __float_as_uint(__ldg(lst + i)); }, (long long)st->len[h], gcta, gn,
                           &coop->sync[1 + h], phase, coop->hist[1 + h], s_hist, s_rank, s_prefix, s_scan, 0, 3, first, known);
        }
        if (gcta == 0 && threadIdx.x == 0) {
            st->out_key[2 * h] = s_prefix[0];
            st->out_key[2 * h + 1] = s_prefix[1];
            __threadfence();
            if (atomicAdd(&st->done, 1u) == 1u) {   // the other half delivered first: finish
                __threadfence();
                uint32_t key[4];
                for (int t = 0; t < 4; ++t) key[t] = *((volatile uint32_t *)&st->out_key[t]);
                write_percentiles(res_all + rec, key, g.t_lo, g.t_hi);
            }
        }
        return;
    }
    for (int h = 0; h < 2; ++h) {
        const float *lst = h ? list_hi : list_lo;
        if (threadIdx.x < 2) s_rank[threadIdx.x] = g.r[2 * h + threadIdx.x] - (uint32_t)below_of[h];
        __syncthreads();
        coop_select<2>([&](long long i) { return __float_as_uint(__ldg(lst + i)); }, (long long)st->len[h], cta,
                       (unsigned)ncta, &coop->sync[1 + h], phase, coop->hist[1 + h], s_hist, s_rank, s_prefix, s_scan);
        phase = 0;   // each list has its own barrier counter
        if (threadIdx.x < 2) s_key[2 * h + threadIdx.x] = s_prefix[threadIdx.x];
        __syncthreads();
    }
    if (cta == 0 && threadIdx.x == 0) write_percentiles(res_all + rec, s_key, g.t_lo, g.t_hi);
}

// exact selection over the whole recording by one CTA (only when a bracket failed)
// ... and, bracket or not, the last kernel of the percentile stage: it leaves the recording's grey threshold table
// behind (tables != nullptr) so that the fused grey map needs no kernel of its own for it.
__global__ void __launch_bounds__(kSelThreads)
pct_fallback_kernel(const float *env, size_t es, PctGeom g, const PctState *st_all, RecResult *res_all,
                    PctCoop *coop_all, GreyTable *tables) {
    __shared__ uint32_t s_hist[4 * 2048];
    __shared__ uint32_t s_rank[4], s_prefix[4], s_scan[32];
    if (!st_all[blockIdx.x].fallback) {
        if (tables) build_grey_table(res_all + blockIdx.x, tables + blockIdx.x);
        return;
    }
    const float *e = env + (size_t)blockIdx.x * es;
    PctCoop *coop = coop_all + blockIdx.x;
    // reuse the sample histogram space (its selection is long finished): clear it first
    for (int i = threadIdx.x; i < 3 * 4 * 2048; i += kSelThreads) coop->hist[0][i] = 0;
    if (threadIdx.x < 4) s_rank[threadIdx.x] = g.r[threadIdx.x];
    __threadfence();
    __syncthreads();
    const long long n = g.n;
    unsigned phase = 0;
    coop_select<4>(
        [&](long long i) {
            float w[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const long long k = i - 2 + j;
                w[j] = (k >= 0 && k < n) ? __ldg(e + k) : 0.f;
            }
            return __float_as_uint(med5(w[0], w[1], w[2], w[3], w[4]));
        },
        n, 0, 1u, &coop->sync[0], phase, coop->hist[0], s_hist, s_rank, s_prefix, s_scan);
    if (threadIdx.x == 0) write_percentiles(res_all + blockIdx.x, s_prefix, g.t_lo, g.t_hi);
    if (tables) {
        __threadfence_block();
        __syncthreads();
        build_grey_table(res_all + blockIdx.x, tables + blockIdx.x);
    }
}

bool launch_percentiles(wefax_ctx *ctx, const float *env, size_t es, long long n, int batch, SelState *sel,
                        RecResult *res, int med, GreyTable *tables) {
    StageTimer timer(ctx, "percentiles");
    cudaStream_t st = ctx->stream;
    // numpy 'linear' method: virtual index (n-1)*q, q = 0.5/100 and 99.5/100
    const double v_lo = (double)(n - 1) * (0.5 / 100), v_hi = (double)(n - 1) * (99.5 / 100);
    const long long i_lo = (long long)floor(v_lo), i_hi = (long long)floor(v_hi);
    const double t_lo = v_lo - (double)i_lo, t_hi = v_hi - (double)i_hi;
    auto clip = [&](long long r) { return (uint32_t)std::min(r, n - 1); };
    const char *force = getenv("WEFAX_PCT_MODE");   // "radix" | "bracket" (tests); default by length
    if (med != 5 && med != 3) WEFAX_THROW(WEFAX_ERR_INVALID, "median window %d", med);
    // (the bracketed selection is written for the file path's median-5; packets are short anyway)
    const bool bracket = med == 5 && (force ? (force[0] == 'b') : (n >= (1ll << 20)));
    if (!bracket) {
        CUDA_CHECK(cudaMemsetAsync(sel, 0, sizeof(SelState) * batch, st));
        select_init_kernel<<<batch, 32, 0, st>>>(sel, clip(i_lo), clip(i_lo + 1), clip(i_hi), clip(i_hi + 1));
        long long per_block = 4 * 256;
        int blocks = (int)std::min<long long>((n + per_block - 1) / per_block, (long long)ctx->sm_count * 8);
        blocks = std::max(1, blocks / std::max(1, std::min(batch, 8)));
        dim3 grid(blocks, batch);
        if (med == 3) {
            hist_kernel<0, 3><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 0, res, t_lo, t_hi);
            hist_kernel<1, 3><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 1, res, t_lo, t_hi);
            hist_kernel<2, 3><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 2, res, t_lo, t_hi);
        } else {
            hist_kernel<0, 5><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 0, res, t_lo, t_hi);
            hist_kernel<1, 5><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 1, res, t_lo, t_hi);
            hist_kernel<2, 5><<<grid, 256, 0, st>>>(env, es, n, sel);
            select_kernel<<<batch, 256, 0, st>>>(sel, 2, res, t_lo, t_hi);
        }
        CUDA_CHECK(cudaGetLastError());
        ctx->launches += 7;
        return false;   // (short recordings: the caller builds the threshold table itself)
    }
    PctGeom g;
    memset(&g, 0, sizeof(g));
    g.n = n;
    g.ns = (n + kPctStride - 1) / kPctStride;
    g.r[0] = clip(i_lo); g.r[1] = clip(i_lo + 1); g.r[2] = clip(i_hi); g.r[3] = clip(i_hi + 1);
    g.t_lo = t_lo;
    g.t_hi = t_hi;
    // bracket half-width in sample ranks: 12 sigma of a binomial tail count, at least 64
    const double q = 0.005;
    const long long delta = std::max<long long>(64, (long long)std::ceil(12.0 * std::sqrt((double)g.ns * q)));
    const long long a_lo = (long long)(g.r[0] / kPctStride) - delta, b_lo = (long long)(g.r[1] / kPctStride) + 1 + delta;
    const long long a_hi = (long long)(g.r[2] / kPctStride) - delta, b_hi = (long long)(g.r[3] / kPctStride) + 1 + delta;
    g.open_lo = a_lo <= 0;
    g.open_hi = b_hi >= g.ns - 1;
    auto sclip = [&](long long r) { return (uint32_t)std::min<long long>(std::max<long long>(r, 0), g.ns - 1); };
    g.s_rank[0] = sclip(a_lo); g.s_rank[1] = sclip(b_lo); g.s_rank[2] = sclip(a_hi); g.s_rank[3] = sclip(b_hi);
    g.cap = (uint32_t)std::min<long long>(n, 4 * (2 * delta + 2) * kPctStride + 4096);
    const size_t ss = (size_t)((g.ns + 63) & ~63ll), ls = 2 * (size_t)g.cap;
    char *base = (char *)ctx->pct_buf.reserve((ss + ls) * sizeof(float) * batch +
                                              (sizeof(PctState) + sizeof(PctCoop)) * batch + 512);
    float *samp = (float *)base;
    float *lists = samp + ss * batch;
    PctState *pst = (PctState *)(((uintptr_t)(lists + ls * batch) + 15) & ~(uintptr_t)15);
    PctCoop *coop = (PctCoop *)(((uintptr_t)(pst + batch) + 255) & ~(uintptr_t)255);
    CUDA_CHECK(cudaMemsetAsync(coop, 0, sizeof(PctCoop) * batch, st));
    // CTAs of one recording spin at a barrier, so all of them must be resident at once:
    // 1024-thread CTAs, two per SM.  Up to 128 CTAs per recording: 41 -> 31 us for the bracket kernel against 32 CTAs,
    // whose latency-bound sample read gets four times shorter.
    const int ncta = std::max(1, std::min(128, ctx->sm_count / batch));

    const int per = (int)((g.ns + ncta - 1) / ncta);
    const size_t fused_smem = ((size_t)4 * 2048 + (size_t)per) * sizeof(uint32_t);
    // the sample taken in the bracket kernel's shared memory when it fits, else a separate sampling pass
    if (fused_smem <= 200 * 1024) {
        StageTimer t1(ctx, "pct_bracket");
        const void *fn = (const void *)pct_bracket2_kernel;
        if (!ctx->smem_configured.count(fn)) {
            CUDA_CHECK(cudaFuncSetAttribute(pct_bracket2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            ctx->smem_configured[fn] = 1;
        }
        int ncta_arg = ncta, per_arg = per;
        size_t es_arg = es;
        void *args[] = {(void *)&env, (void *)&es_arg, (void *)&g, (void *)&pst, (void *)&coop, (void *)&ncta_arg, (void *)&per_arg};
        if (ncta > 1)
            CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)pct_bracket2_kernel, dim3(batch * ncta), dim3(kSelThreads), args,
                                                   fused_smem, st));
        else
            pct_bracket2_kernel<<<batch, kSelThreads, fused_smem, st>>>(env, es, g, pst, coop, 1, per);
        ctx->launches -= 1;   // (one kernel instead of two; the total below counts five)
    } else {
    dim3 g1((unsigned)((g.ns + 255) / 256), batch);
    {
        StageTimer t1(ctx, "pct_sample");
        pct_sample_kernel<<<g1, 256, 0, st>>>(env, es, g, samp, ss);
    }
    {
        StageTimer t1(ctx, "pct_bracket");
        // cooperative launch: the runtime only starts the grid when all its CTAs fit at once
        int ncta_arg = ncta;
        size_t ss_arg = ss;
        void *args[] = {(void *)&samp, (void *)&ss_arg, (void *)&g, (void *)&pst, (void *)&coop, (void *)&ncta_arg};
        if (ncta > 1)
            CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)pct_bracket_kernel, dim3(batch * ncta),
                                                   dim3(kSelThreads), args, 0, st));
        else   // one CTA per recording: no cross-CTA barrier, any grid size
            pct_bracket_kernel<<<batch, kSelThreads, 0, st>>>(samp, ss, g, pst, coop, 1);
    }
    }
    int blocks = (int)std::min<long long>((n + 2047) / 2048, (long long)ctx->sm_count * 8);
    blocks = std::max(1, blocks / std::max(1, std::min(batch, 8)));
    {
        StageTimer t1(ctx, "pct_collect");
        pct_collect2_kernel<<<dim3(blocks, batch), 256, 0, st>>>(env, es, g, pst, lists, ls);
    }
    {
        StageTimer t1(ctx, "pct_final");
        int ncta_arg = ncta;
        size_t ls_arg = ls;
        // keys of a CTA's slice of a candidate list in shared memory (two groups of ncta / 2 CTAs, one per list)
        int local_per = 0;
        size_t fin_smem = 0;
        if (ncta >= 2) {
            const long long per_max = ((long long)g.cap + (ncta / 2) - 1) / (ncta / 2);
            if (per_max * 4 <= 160 * 1024) {
                local_per = (int)per_max;
                fin_smem = (size_t)per_max * sizeof(uint32_t);
                const void *fn = (const void *)pct_final_kernel;
                if (!ctx->smem_configured.count(fn)) {
                    CUDA_CHECK(cudaFuncSetAttribute(pct_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
                    ctx->smem_configured[fn] = 1;
                }
            }
        }
        void *args[] = {(void *)&g, (void *)&pst, (void *)&lists, (void *)&ls_arg, (void *)&res, (void *)&coop,
                        (void *)&ncta_arg, (void *)&local_per};
        if (ncta > 1)
            CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)pct_final_kernel, dim3(batch * ncta), dim3(kSelThreads),
                                                   args, fin_smem, st));
        else
            pct_final_kernel<<<batch, kSelThreads, 0, st>>>(g, pst, lists, ls, res, coop, 1, 0);
        pct_fallback_kernel<<<batch, kSelThreads, 0, st>>>(env, es, g, pst, res, coop, tables);
    }
    CUDA_CHECK(cudaGetLastError());
    ctx->launches += 5;
    return tables != nullptr;
}

// ===========================================================================
// grey map  (wefax.py:197-200,216): round(255*(env-low)/(high-low)), clip, int
// ===========================================================================
template <int MED>
__global__ void __launch_bounds__(256)
quantise_kernel(const float *env, size_t es, uint8_t *dig, size_t ds, long long n, const RecResult *res_all,
                long long i_begin, long long i_end, double eps) {
    const RecResult *res = res_all + blockIdx.y;
    const float *e = env + (size_t)blockIdx.y * es;
    uint8_t *d = dig + (size_t)blockIdx.y * ds;
    const double low = res->low;
    // the file path divides by high - low (wefax.py:198), the live path's packets by high - low + 0.000001
    // (data_packet.py:461)
    const double delta = __dadd_rn(__dsub_rn(res->high, low), eps);
    long long i0 = i_begin + 8 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);   // i_begin % 8 == 0
    if (i0 >= i_end) return;
    float m[8];
    load_med8<MED>(e, i0, n, m);
    // numpy: round(255 * (env - low) / delta) in float64 (rint = half to even = numpy.round).
    // The float64 divide is only needed when the value is close to a rounding boundary: an
    // fp32 estimate (error << 1e-3 grey levels) decides every other element.
    const float low_f = (float)low, scale_f = (float)(255.0 / delta);
    // estimate error ~ |low|*scale*2^-24 + |est|*3*2^-24: must stay far below the 2e-3 guard band
    const bool fast_ok = delta > 0.0 && isfinite(scale_f) && fabs(low) * (255.0 / delta) * 1.2e-7 < 5e-4;
    uint32_t packed[2] = {0u, 0u};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float est = (m[j] - low_f) * scale_f;
        const float fr = est - floorf(est);
        float v;
        if (fast_ok && fabsf(fr - 0.5f) > 2e-3f && fabsf(est) < 1e6f) {
            v = rintf(est);
        } else {
            v = (float)rint(__ddiv_rn(__dmul_rn(255.0, __dsub_rn((double)m[j], low)), delta));
        }
        v = fminf(fmaxf(v, 0.f), 255.f);
        packed[j >> 2] |= (uint32_t)(int)v << (8 * (j & 3));
    }
    if (i0 + 7 < n && ((reinterpret_cast<uintptr_t>(d + i0) & 7) == 0)) {
        *reinterpret_cast<uint2 *>(d + i0) = make_uint2(packed[0], packed[1]);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (i0 + j < n) d[i0 + j] = (uint8_t)(packed[j >> 2] >> (8 * (j & 3)));
    }
}

// Grey levels of samples [i_begin, i_end) (i_begin a multiple of 8) on `stream`.
void launch_quantise(wefax_ctx *ctx, const float *env, size_t es, uint8_t *dig, size_t ds, long long n, int batch,
                     const RecResult *res, long long i_begin, long long i_end, cudaStream_t stream, const char *tag,
                     int med, double eps) {
    if (i_end <= i_begin) return;
    StageTimer timer(ctx, tag, stream);
    dim3 grid((unsigned)((i_end - i_begin + 2047) / 2048), batch);
    if (med == 3)
        quantise_kernel<3><<<grid, 256, 0, stream>>>(env, es, dig, ds, n, res, i_begin, i_end, eps);
    else
        quantise_kernel<5><<<grid, 256, 0, stream>>>(env, es, dig, ds, n, res, i_begin, i_end, eps);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// ===========================================================================
// phasing search  (wefax.py:218-294)
// ===========================================================================
constexpr int kSyncThreads = 1024;
constexpr int kSyncMaxL = 2048;

__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long *s_red) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, v, d);
        v = o > v ? o : v;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();   // protect s_red from the previous reduction's readers
    if (lane == 0) s_red[wid] = v;
    __syncthreads();
    unsigned long long r = s_red[lane];   // kSyncThreads / 32 == 32 partials
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, r, d);
        r = o > r ? o : r;
    }
    return r;
}

// key orders by correlation, ties by smallest index (the picker's strict '>')
__device__ __forceinline__ unsigned long long sync_key(int corr, int idx) {
    return ((unsigned long long)((uint32_t)corr ^ 0x80000000u) << 32) | (uint32_t)(0x7FFFFFFF - idx);
}
__device__ __forceinline__ int key_corr(unsigned long long k) { return (int)((uint32_t)(k >> 32) ^ 0x80000000u); }
__device__ __forceinline__ int key_idx(unsigned long long k) { return 0x7FFFFFFF - (int)(uint32_t)k; }

// wefax.py:263-294 (find_sync_pulses / find_peak_groups, quirks included), then
// start_frame (wefax.py:80) and the image height (wefax.py:299).  One thread.
__device__ void finish_sync(const int *peaks, int np, const LineDev &ln, long long n, RecResult *res) {
    // dev_max > x > dev_min (wefax.py:268) on integers: x <= ceil(dev_max) - 1 and x >= floor(dev_min) + 1
    const int reg_hi = (int)ceil(ln.dev_max) - 1, reg_lo = (int)floor(ln.dev_min) + 1;
    auto regular = [&](int x) { return x <= reg_hi && x >= reg_lo; };
    int nclear = 0;
    for (int i = 1; i < np - 1; ++i)
        if (regular(peaks[i] - peaks[i - 1])) nclear++;
    int best_start = 0, best_len = -1, cur_start = 1, cur_len = 0;
    for (int i = 1; i < nclear - 1; ++i) {
        if (regular(peaks[i] - peaks[i - 1])) {
            if (cur_len == 0) cur_start = i;
            cur_len++;
        } else {
            if (cur_len > best_len) {
                best_len = cur_len;
                best_start = cur_start;
            }
            cur_len = 0;
        }
    }
    res->n_peaks = np;
    for (int i = 0; i < np; ++i) res->peaks[i] = peaks[i];
    int status = res->status;
    long long start = 0;
    if (best_len < 0) {
        status |= WEFAX_REC_NO_GROUPS;
        res->n_phasing = 0;
    } else {
        res->n_phasing = best_len;
        for (int i = 0; i < best_len; ++i) res->phasing[i] = peaks[best_start + i];
        if (best_len > 0) start = peaks[best_start + best_len - 1];
    }
    res->start_frame = start;
    long long h = (n - start) / ln.width;
    if (!(status & WEFAX_REC_NO_GROUPS) && h == 0) status |= WEFAX_REC_NO_LINES;
    res->height = (status == WEFAX_REC_OK) ? (int32_t)(4 * h) : 0;
    res->status = status;
}

// PACKET: the live path's per-packet picker (data_packet.py:313-331) instead of the file path's: template
// [255] + [0] * n1 + [255] shifted by -128 (LineDev.n1 zeros, L = n1 + 2), sentinel (-mindistance, 0) instead of
// (0, 0), no 100-peak stop, and the first entry of the list is dropped on return (one CTA per packet).
template <int PER, bool PACKET>
__global__ void __launch_bounds__(kSyncThreads)
sync_search_kernel(const uint8_t *dig_all, size_t ds, long long n, const LineDev *lines, RecResult *res_all,
                   const int *need_scan, const LazyGrey lazy) {
    if (need_scan && !need_scan[blockIdx.x]) return;   // the windowed-maximum path already finished this recording
    constexpr int CH = kSyncThreads * PER;            // positions handled per iteration
    constexpr int TOTMAX = CH + kSyncMaxL;
    constexpr int EPT = (TOTMAX + kSyncThreads - 1) / kSyncThreads;
    __shared__ int s_p[TOTMAX + 1];                   // exclusive prefix sums of (d - 128)
    __shared__ int s_wsum[32];
    __shared__ unsigned long long s_red[32];
    __shared__ int s_peaks[WEFAX_MAX_PEAKS];

    const LineDev ln = lines[PACKET ? 0 : blockIdx.x];   // packets of one scan share their geometry
    RecResult *res = res_all + blockIdx.x;
    const uint8_t *dig = dig_all + (size_t)blockIdx.x * ds;
    const float *lazy_env = lazy.env ? lazy.env + (size_t)blockIdx.x * lazy.es : nullptr;
    const GreyTable *lazy_tab = lazy.env ? lazy.tables + blockIdx.x : nullptr;
    auto grey_at = [&](long long i) -> int {
        if (lazy_env && i >= lazy.valid) return grey_at_from_envelope(lazy_env, i, n, lazy_tab);
        return (int)__ldg(dig + i);
    };
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = ln.L, n1 = ln.n1, n0 = ln.n0, mind = ln.mindistance;
    const long long m = n - L;                        // range(len(data) - len(sync))

    long long p = PACKET ? -(long long)mind : 0;   // position of the newest peak
    int v = 0;             // its correlation
    int npeaks = 1;        // peaks = [(0, 0)]  /  [(-mindistance, 0)]
    bool done = false;
    if (tid == 0) s_peaks[0] = (int)p;
    // correlation at position i of the chunk from the exclusive prefix sums of (d - 128)
    auto corr_at = [&](int i) -> int {
        if (PACKET) {
            const int a = s_p[i], b = s_p[i + 1], cc = s_p[i + L - 1], d = s_p[i + L];
            return 127 * (b - a) - 128 * (cc - b) + 127 * (d - cc);
        }
        const int a = s_p[i], b = s_p[i + n1], cc = s_p[i + n1 + n0], d = s_p[i + L];
        return -127 * (b - a) - 128 * (cc - b) - 127 * (d - cc);
    };

    for (long long base = 0; base < m && !done; base += CH) {
        const int valid = (int)min((long long)CH, m - base);
        const int tot = valid + L;
        // ---- exclusive prefix sums of (d - 128) over [base, base + tot) -----------------
        int vals[EPT], run = 0;
        const int j0 = tid * EPT;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            int idx = j0 + j;
            int x = idx < tot ? grey_at(base + idx) - 128 : 0;
            run += x;
            vals[j] = run;
        }
        int incl = run;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += o;
        }
        __syncthreads();   // previous iteration's readers of s_p / s_wsum are done
        if (lane == 31) s_wsum[wid] = incl;
        __syncthreads();
        int woff = 0;
        {
            int t = lane < wid ? s_wsum[lane] : 0;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, d);
            woff = t;
        }
        const int excl = woff + incl - run;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            int idx = j0 + j;
            if (idx < TOTMAX) s_p[idx + 1] = excl + vals[j];
        }
        if (tid == 0) s_p[0] = 0;
        __syncthreads();

        // ---- correlation of this thread's positions -------------------------------------
        int corr[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            int i = tid + u * kSyncThreads;
            int c = 0;
            if (i < valid) c = corr_at(i);
            corr[u] = c;
        }
        auto range_max = [&](int lo, int hi) -> unsigned long long {   // max over positions [lo, hi)
            unsigned long long k = 0;
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                int i = tid + u * kSyncThreads;
                if (i >= lo && i < hi) {
                    unsigned long long kk = sync_key(corr[u], i);
                    k = kk > k ? kk : k;
                }
            }
            return block_max_u64(k, s_red);
        };

        const long long i_exp = p + mind + 1;          // first i with i - p > mindistance
        if (i_exp < base + valid) {
            const int a_exp = (int)(i_exp - base);
            unsigned long long k1 = a_exp > 0 ? range_max(0, a_exp) : 0ull;
            if (k1 != 0ull && key_corr(k1) > v) {
                // a replacement happens first: the peak moves into this chunk, no opening here
                unsigned long long k = range_max(0, valid);
                p = base + key_idx(k);
                v = key_corr(k);
            } else {
                // open a new peak at i_exp
                p = i_exp;
                v = corr_at(a_exp);
                npeaks++;
                if (npeaks == WEFAX_MAX_PEAKS) {   // wefax.py:251 (a packet never gets there: <= n / mindistance peaks)
                    done = true;
                } else if (a_exp + 1 < valid) {
                    unsigned long long k2 = range_max(a_exp + 1, valid);
                    if (k2 != 0ull && key_corr(k2) > v) {
                        p = base + key_idx(k2);
                        v = key_corr(k2);
                    }
                }
            }
        } else {
            unsigned long long k = range_max(0, valid);
            if (k != 0ull && key_corr(k) > v) {
                p = base + key_idx(k);
                v = key_corr(k);
            }
        }
        if (tid == 0) s_peaks[npeaks - 1] = (int)p;
    }
    __syncthreads();

    if (PACKET) {
        if (tid == 0) {
            res->n_peaks = npeaks - 1;
            for (int i = 1; i < npeaks; ++i) res->peaks[i - 1] = s_peaks[i];
            res->start_frame = npeaks > 1 ? s_peaks[npeaks - 1] : -1;   // the last pulse: where the live decoder starts
        }
        return;
    }
    if (tid == 0) finish_sync(s_peaks, npeaks, ln, n, res);
}

// ---------------------------------------------------------------------------
// Parallel form of the greedy picker.  Let corr[i] be the correlation and
// W[i] = max corr over (i, min(i + mindistance, m-1)].  Position i is "settled"
// when corr[i] >= W[i]: once the picker's newest peak sits there, nothing replaces it
// before the next peak opens.  The picker's trajectory is then
//     P_k = first settled position >= a_k,     a_{k+1} = P_k + mindistance + 1,
// with a_0 = first i <= mindistance with corr[i] > 0 (the initial peak (0, 0) only
// moves to a strictly positive correlation; if there is none, P_0 = 0).  corr, W
// (van Herk prefix/suffix maxima over blocks of mindistance) and the settled bits
// are data-parallel; only the <= 100-step chain over a bitmask in shared memory is
// sequential.  Equivalence with wefax.py:234-259 is checked bit for bit in the tests.
// ---------------------------------------------------------------------------
constexpr int kCorrTile = 4096;

__global__ void __launch_bounds__(kSyncThreads)
sync_corr_kernel(const uint8_t *dig_all, size_t ds, long long n, const LineDev *lines, const SyncDev *sd_all,
                 int *corr_all, size_t cs, int *first_pos) {
    constexpr int TOTMAX = kCorrTile + kSyncMaxL;
    constexpr int EPT = (TOTMAX + kSyncThreads - 1) / kSyncThreads;
    __shared__ int s_p[TOTMAX + 1];
    __shared__ int s_wsum[32];
    const LineDev ln = lines[blockIdx.y];
    const SyncDev sd = sd_all[blockIdx.y];
    const long long base = (long long)blockIdx.x * kCorrTile;
    if (!sd.fast || base >= sd.limc) return;
    const uint8_t *dig = dig_all + (size_t)blockIdx.y * ds;
    int *corr = corr_all + (size_t)blockIdx.y * cs;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = ln.L, n1 = ln.n1, n0 = ln.n0;
    const int valid = (int)min((long long)kCorrTile, sd.limc - base);
    const int tot = valid + L;
    int vals[EPT], run = 0;
    const int j0 = tid * EPT;
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
        int idx = j0 + j;
        int x = idx < tot ? (int)__ldg(dig + base + idx) - 128 : 0;
        run += x;
        vals[j] = run;
    }
    int incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_wsum[wid] = incl;
    __syncthreads();
    int woff;
    {
        int t = lane < wid ? s_wsum[lane] : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, d);
        woff = t;
    }
    const int excl = woff + incl - run;
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
        int idx = j0 + j;
        if (idx < TOTMAX) s_p[idx + 1] = excl + vals[j];
    }
    if (tid == 0) s_p[0] = 0;
    __syncthreads();
    int first = 0x7FFFFFFF;
    for (int i = tid; i < valid; i += kSyncThreads) {
        int a = s_p[i], b = s_p[i + n1], cc = s_p[i + n1 + n0], d = s_p[i + L];
        int c = -127 * (b - a) - 128 * (cc - b) - 127 * (d - cc);
        corr[base + i] = c;
        if (c > 0 && base + i <= ln.mindistance) first = min(first, (int)(base + i));
    }
    if (base <= ln.mindistance) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) first = min(first, __shfl_xor_sync(0xFFFFFFFFu, first, d));
        if (lane == 0 && first != 0x7FFFFFFF) atomicMin(first_pos + blockIdx.y, first);
    }
}

// inclusive running maximum of s[0..len) (dir 0: left to right, dir 1: right to left) by one CTA
__device__ __forceinline__ void block_running_max(const int *src, int *dst, int len, int dir, int *s_w) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int per = (len + kSyncThreads - 1) / kSyncThreads;
    const int NEG = (int)0x80000000;
    const int lo = tid * per, hi = min(lo + per, len);
    int run = NEG;
    for (int i = lo; i < hi; ++i) run = max(run, src[dir ? len - 1 - i : i]);
    int incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl = max(incl, o);
    }
    __syncthreads();
    if (lane == 31) s_w[wid] = incl;
    __syncthreads();
    int carry = NEG;
    for (int k = 0; k < wid; ++k) carry = max(carry, s_w[k]);
    int prev = __shfl_up_sync(0xFFFFFFFFu, incl, 1);
    if (lane > 0) carry = max(carry, prev);
    run = carry;
    // src and dst may alias: a thread only rewrites its own chunk, after reading it
    for (int i = lo; i < hi; ++i) {
        const int idx = dir ? len - 1 - i : i;
        run = max(run, src[idx]);
        dst[idx] = run;
    }
    __syncthreads();
}

// settled bits: corr[i] >= max corr over (i, min(i + w, m - 1)], with the window maximum from
// van Herk / Gil-Werman prefix and suffix maxima over blocks of w = mindistance positions.
// CTA j holds block j and block j+1 of the correlation in shared memory: suffix maxima of
// block j, prefix maxima of block j+1; nothing but the bit mask goes back to global memory.
__global__ void __launch_bounds__(kSyncThreads)
sync_settled_kernel(const LineDev *lines, const SyncDev *sd_all, const int *corr_all, size_t cs, uint32_t *bits_all,
                    size_t bs) {
    extern __shared__ int s_dyn[];
    __shared__ int s_w[32];
    const LineDev ln = lines[blockIdx.y];
    const SyncDev sd = sd_all[blockIdx.y];
    const int w = ln.mindistance;
    const long long b0 = (long long)blockIdx.x * w;
    if (!sd.fast || b0 >= sd.lim) return;
    int *s_c = s_dyn, *s_suf = s_dyn + w, *s_pre = s_dyn + 2 * w;
    const int len0 = (int)min((long long)w, sd.limc - b0);
    const int len1 = (int)max(0ll, min((long long)w, sd.limc - (b0 + w)));
    const int *corr = corr_all + (size_t)blockIdx.y * cs;
    for (int i = threadIdx.x; i < len0; i += kSyncThreads) s_c[i] = corr[b0 + i];
    for (int i = threadIdx.x; i < len1; i += kSyncThreads) s_pre[i] = corr[b0 + w + i];
    __syncthreads();
    block_running_max(s_c, s_suf, len0, 1, s_w);
    if (len1 > 0) block_running_max(s_pre, s_pre, len1, 0, s_w);
    uint32_t *bits = bits_all + (size_t)blockIdx.y * bs;
    const long long p_first = b0 & ~31ll;
    const long long p_end = min(b0 + len0, sd.lim);
    for (long long p = p_first + threadIdx.x; p < ((p_end + 31) & ~31ll); p += kSyncThreads) {
        bool settled = false;
        if (p >= b0 && p < p_end) {
            const int i = (int)(p - b0);
            const long long a = p + 1, e = min(p + w, sd.m - 1);
            int wmax = (int)0x80000000;
            if (a <= e) {
                if (a < b0 + w && i + 1 < len0) wmax = s_suf[i + 1];              // rest of block j
                if (e >= b0 + w) wmax = max(wmax, s_pre[e - (b0 + w)]);           // head of block j+1
            }
            settled = s_c[i] >= wmax;
        }
        const unsigned word = __ballot_sync(0xFFFFFFFFu, settled);
        if ((threadIdx.x & 31) == 0 && word) atomicOr(&bits[p >> 5], word);       // words straddle CTAs
    }
}

__device__ __forceinline__ uint32_t smem_addr_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// the sequential part: <= 100 jumps over the settled-bit mask held in shared memory
__global__ void __launch_bounds__(1024)
sync_chain_kernel(long long n, const LineDev *lines, const SyncDev *sd_all, const uint32_t *bits_all, size_t bs,
                  const int *first_pos, RecResult *res_all, int *need_scan, int force_scan) {
    extern __shared__ uint32_t s_bits[];
    __shared__ int s_peaks[WEFAX_MAX_PEAKS];
    const LineDev ln = lines[blockIdx.x];
    const SyncDev sd = sd_all[blockIdx.x];
    if (!sd.fast || force_scan == 1) {   // test hook: WEFAX_SYNC_FORCE_SCAN=1, the sequential scan decides
        if (threadIdx.x == 0) need_scan[blockIdx.x] = 1;
        return;
    }
    const int nwords = (int)((sd.lim + 31) >> 5);
    const uint32_t *bits = bits_all + (size_t)blockIdx.x * bs;
    {
        // 128-bit loads, several in flight per thread (bs is a multiple of 4 words)
        const int nvec = (nwords + 3) >> 2;
        const uint4 *src = reinterpret_cast<const uint4 *>(bits);
        uint4 *dst = reinterpret_cast<uint4 *>(s_bits);
#pragma unroll 4
        for (int i = threadIdx.x; i < nvec; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    // Summary of the mask, built by warp votes and a short parallel walk:
    //   s_l1[j]   bit k: word 32 j + k is non-empty                         (one word per 1024 positions)
    //   s_l2[j]   bit k: s_l1[32 j + k] != 0                                 (only used to build s_nxt)
    //   s_nxt[b]  first settled position >= 1024 b, or -1                    (one int per 1024 positions)
    // "First settled position >= a" is then ONE round of three independent shared-memory loads for the usual case
    // (the word of a, the summary word of its 1024-block, s_nxt of the next block) and a second load only when the
    // answer lies in the same block but another word - however the settled positions are spread: isolated maxima of
    // a noisy correlation, plateaus of saturated grey, or everything at once (a constant signal).
    uint32_t *s_l1 = s_bits + (((size_t)nwords + 3) & ~(size_t)3);
    const int nl1 = (nwords + 31) >> 5, nl2 = (nl1 + 31) >> 5;
    uint32_t *s_l2 = s_l1 + ((nl1 + 1 + 3) & ~3);
    int *s_nxt = reinterpret_cast<int *>(s_l2 + ((nl2 + 3) & ~3));   // nl1 + 1 entries
    {
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
        for (int j = wid; j <= nl1; j += nwarps) {          // (one zero word past the end: the chain reads s_l1[nl1])
            const int wi = 32 * j + lane;
            const unsigned word = __ballot_sync(0xFFFFFFFFu, wi < nwords && s_bits[wi] != 0u);
            if (lane == 0) s_l1[j] = word;
        }
        __syncthreads();
        for (int j = wid; j < nl2; j += nwarps) {
            const int k = 32 * j + lane;
            const unsigned word = __ballot_sync(0xFFFFFFFFu, k < nl1 && s_l1[k] != 0u);
            if (lane == 0) s_l2[j] = word;
        }
        __syncthreads();
        for (int b = threadIdx.x; b <= nl1; b += blockDim.x) {
            int pos = -1;
            if (b < nl1) {
                int j = -1;                                   // first non-empty summary word at or after b
                if (s_l1[b] != 0u) {
                    j = b;
                } else if (b + 1 < nl1) {
                    int jj = (b + 1) >> 5;
                    uint32_t t = s_l2[jj] & (~0u << ((b + 1) & 31));
                    while (t == 0u && ++jj < nl2) t = s_l2[jj];
                    if (t != 0u) j = (jj << 5) + (__ffs(t) - 1);
                }
                if (j >= 0) {
                    const int wi = (j << 5) + (__ffs(s_l1[j]) - 1);
                    pos = (wi << 5) + (__ffs(s_bits[wi]) - 1);
                }
            }
            s_nxt[b] = pos;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // One thread, pure latency (a dependent instruction of a lone warp issues every ~5 cycles): the loop is kept
        // to a few dozen instructions - 32-bit shared addresses, one bound check per step (the 100-peak stop and both
        // range ends are sorted out after the loop), the three look-ups issued side by side.
        const int w = ln.mindistance;
        const int lim = (int)sd.lim;
        const int last = (int)min(sd.m - 1, (long long)0x7ffffff0);   // a > last ends the picker
        const int amax = min(last, lim - 1);                          // a > amax: the picker ends or the mask does
        const uint32_t a_bits = smem_addr_u32(s_bits), a_l1 = smem_addr_u32(s_l1), a_nxt = smem_addr_u32(s_nxt);
        // first settled position >= x (0 <= x < lim); -1 when the mask ends first
        auto next_settled = [&](int x) -> int {
            const int wi = x >> 5, blk = x >> 10;
            const uint32_t v0 = lds_u32(a_bits + 4u * (uint32_t)wi) & (~0u << (x & 31));
            // words wi + 1 .. 31 of this block (bit 31 shifted out when wi is the block's last word)
            const uint32_t u0 = lds_u32(a_l1 + 4u * (uint32_t)blk) & ((0xFFFFFFFEu << (wi & 31)));
            const int far = (int)lds_u32(a_nxt + 4u * (uint32_t)(blk + 1));
            if (v0 != 0u) return (wi << 5) + (__ffs(v0) - 1);
            if (u0 != 0u) {
                const int w2 = (blk << 5) + (__ffs(u0) - 1);
                return (w2 << 5) + (__ffs(lds_u32(a_bits + 4u * (uint32_t)w2)) - 1);
            }
            return far;
        };
        int np = 1, ok = 1;
        int P = 0;
        const int j0 = first_pos[blockIdx.x];
        if (sd.m > 0 && j0 != 0x7F7F7F7F) {
            P = j0 < lim ? next_settled(j0) : -1;
            if (P < 0) ok = 0;
        }
        s_peaks[0] = P;
        if (ok && sd.m > 0) {
            int a = P + w + 1;
#pragma unroll 1
            while (np < WEFAX_MAX_PEAKS - 1 && a <= amax) {
                P = next_settled(a);
                if (P < 0) {
                    ok = 0;
                    break;
                }
                s_peaks[np++] = P;
                a = P + w + 1;
            }
            if (ok && a <= last) {
                // the loop stopped at the 100-peak limit (the 100th peak is never refined, wefax.py:251) or at the
                // end of the precomputed region
                if (np == WEFAX_MAX_PEAKS - 1) s_peaks[np++] = a;
                else ok = 0;
            }
        }
        if (ok) {
            need_scan[blockIdx.x] = 0;
            finish_sync(s_peaks, np, ln, n, res_all + blockIdx.x);
        } else {
            need_scan[blockIdx.x] = 1;   // ran out of precomputed region: let the sequential scan do it
        }
    }
}

long long sync_head(const SyncPlan &sp, long long n) {
    // the parallel search reads positions < max_limc + template length
    return sp.any_fast ? std::min(n, ((sp.max_limc + kSyncMaxL + 2047) / 2048) * 2048) : n;
}

void clear_sync_scratch(wefax_ctx *ctx, const SyncPlan &sp, int batch) {
    if (!sp.any_fast) return;
    CUDA_CHECK(cudaMemsetAsync(sp.first_pos, 0x7F, sizeof(int) * batch, ctx->stream));   // 0x7F7F7F7F = no positive correlation yet
    CUDA_CHECK(cudaMemsetAsync(sp.bits, 0, sp.bs * batch * sizeof(uint32_t), ctx->stream));
}

void launch_sync_search(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int batch, const LineDev *lines,
                        RecResult *res, int min_mindistance, const SyncPlan &sp, const LazyGrey &lazy) {
    StageTimer timer(ctx, "sync_search");
    cudaStream_t st = ctx->stream;
    const char *fs = getenv("WEFAX_SYNC_FORCE_SCAN");
    const int force_scan = fs ? atoi(fs) : 0;
    if (sp.any_fast) {
        dim3 g1((unsigned)std::max<long long>(1, (sp.max_limc + kCorrTile - 1) / kCorrTile), batch);
        {
            StageTimer t1(ctx, "sync_corr");
            sync_corr_kernel<<<g1, kSyncThreads, 0, st>>>(dig, ds, n, lines, sp.sd, sp.corr, sp.cs, sp.first_pos);
        }
        dim3 g2((unsigned)std::max(1, sp.max_wblocks), batch);
        const void *fn = (const void *)sync_settled_kernel;
        if (!ctx->smem_configured.count(fn)) {
            CUDA_CHECK(cudaFuncSetAttribute(sync_settled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            CUDA_CHECK(cudaFuncSetAttribute(sync_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
            ctx->smem_configured[fn] = 1;
        }
        {
            StageTimer t1(ctx, "sync_settled");
            // (1024 threads per block of `mindistance` positions also in batches: with 256 / 512 threads per CTA - and the
            //  thread count a run-time value - the kernel took 877 / 609 us instead of 434 us on 64 recordings: its 53 KB of
            //  shared memory per CTA, not its thread count, limits residency, and the compile-time stride matters)
            sync_settled_kernel<<<g2, kSyncThreads, (size_t)3 * sp.max_w * sizeof(int), st>>>(lines, sp.sd, sp.corr, sp.cs,
                                                                                           sp.bits, sp.bs);
        }
        {
            StageTimer t1(ctx, "sync_chain");
            // the settled bits, their two summary levels (1/32 and 1/1024 of the mask) and one int per 1024 positions
            const size_t chain_words = (size_t)(((sp.max_lim + 31) / 32 + 4 + 3) & ~3ll);
            const size_t chain_aux = (2 * (chain_words / 32 + 8) + chain_words / 1024 + 8) * sizeof(uint32_t);
            sync_chain_kernel<<<batch, 1024, chain_words * sizeof(uint32_t) + chain_aux, st>>>(
                n, lines, sp.sd, sp.bits, sp.bs, sp.first_pos, res, sp.need_scan, force_scan);
        }
        ctx->launches += 3;
    } else {
        CUDA_CHECK(cudaMemsetAsync(sp.need_scan, 1, sizeof(int) * batch, st));
    }
    if (min_mindistance >= 4096)
        sync_search_kernel<4, false><<<batch, kSyncThreads, 0, st>>>(dig, ds, n, lines, res, sp.need_scan, lazy);
    else if (min_mindistance >= 2048)
        sync_search_kernel<2, false><<<batch, kSyncThreads, 0, st>>>(dig, ds, n, lines, res, sp.need_scan, lazy);
    else
        sync_search_kernel<1, false><<<batch, kSyncThreads, 0, st>>>(dig, ds, n, lines, res, sp.need_scan, lazy);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// data_packet.py:313-331 for n_packets packets of n grey levels each (stride ds); line: one LineDev on the device
// with n1 = samples(0.025), L = n1 + 2, mindistance = samples(0.4).  RecResult.peaks / n_peaks / start_frame (= last
// pulse or -1) per packet.
void launch_packet_pulse_search(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int n_packets,
                                const LineDev *line, RecResult *res, int mindistance) {
    StageTimer timer(ctx, "packet_pulses");
    if (mindistance >= 4096)
        sync_search_kernel<4, true><<<n_packets, kSyncThreads, 0, ctx->stream>>>(dig, ds, n, line, res, nullptr, LazyGrey());
    else if (mindistance >= 2048)
        sync_search_kernel<2, true><<<n_packets, kSyncThreads, 0, ctx->stream>>>(dig, ds, n, line, res, nullptr, LazyGrey());
    else
        sync_search_kernel<1, true><<<n_packets, kSyncThreads, 0, ctx->stream>>>(dig, ds, n, line, res, nullptr, LazyGrey());
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

// ===========================================================================
// line raster + x4 vertical bicubic == Image.new/putpixel/resize  (wefax.py:296-327)
// Pillow Resample.c: BICUBIC (a = -0.5), support 2, coefficients normalised per
// output row, fixed point with PRECISION_BITS = 22.
// ===========================================================================
constexpr int kRasterRows = 16;      // input lines per tile (-> 64 output rows)
constexpr int kRasterThreads = 256;  // x 4 columns per thread

__device__ __forceinline__ double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// Each thread owns 4 adjacent columns and walks down kRasterRows input lines with a
// 5-line luminance window (lines r-2 .. r+2) in registers; every input line yields 4
// output rows whose Pillow coefficients sit in shared memory as 5 "window slot" weights.
__global__ void __launch_bounds__(kRasterThreads)
raster_kernel(const uint8_t *dig_all, size_t ds, long long n, const LineDev *lines, const RecResult *res_all,
              uint8_t *raster_all, size_t rs) {
    __shared__ int s_k[4 * kRasterRows][5];

    const RecResult *res = res_all + blockIdx.z;
    const int w = lines[blockIdx.z].width;
    const int h = res->height / 4;
    const int r0 = blockIdx.y * kRasterRows;
    const int x0 = (blockIdx.x * kRasterThreads + threadIdx.x) * 4;
    if (res->status != WEFAX_REC_OK || r0 >= h || blockIdx.x * kRasterThreads * 4 >= w) return;
    const uint8_t *dig = dig_all + (size_t)blockIdx.z * ds + res->start_frame;
    uint8_t *out = raster_all + (size_t)blockIdx.z * rs;

    // Pillow precompute_coeffs + normalize_coeffs_8bpc for this tile's output rows
    if (threadIdx.x < 4 * kRasterRows) {
        const int yy = 4 * r0 + threadIdx.x;
        const int r = yy >> 2;
        const double scale = 0.25, support = 2.0;
        const double center = (yy + 0.5) * scale;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > h) xmax = h;
        xmax -= xmin;
        double kw[5], ww = 0.0;
        for (int t = 0; t < 5; ++t) {
            kw[t] = t < xmax ? bicubic_filter((t + xmin - center + 0.5)) : 0.0;
            ww += kw[t];
        }
        int slot[5] = {0, 0, 0, 0, 0};
        for (int t = 0; t < 5; ++t) {
            if (t >= xmax) break;
            double kv = (ww != 0.0) ? kw[t] / ww : kw[t];
            int ki = kv < 0 ? (int)(-0.5 + kv * 4194304.0) : (int)(0.5 + kv * 4194304.0);
            int sl = xmin + t - (r - 2);          // window slot of input line xmin + t
            if (sl >= 0 && sl < 5) slot[sl] = ki;
        }
        for (int t = 0; t < 5; ++t) s_k[threadIdx.x][t] = slot[t];
    }
    __syncthreads();
    if (x0 >= w) return;

    auto load_line = [&](int r, int *l) {
        // luminance 255 - value (wefax.py:303); lines outside the image only meet zero weights
        if (r < 0 || r >= h) {
            l[0] = l[1] = l[2] = l[3] = 0;
            return;
        }
        const uint8_t *p = dig + (size_t)r * w + x0;
#pragma unroll
        for (int c = 0; c < 4; ++c) l[c] = (x0 + c < w) ? 255 - (int)__ldg(p + c) : 0;
    };
    int win[5][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) load_line(r0 - 2 + j, win[j]);
    const bool full = x0 + 3 < w;
    // Interior tiles (no line of the tile within 2 lines of the image's first / last line): Pillow's coefficients
    // depend on the phase only (the filter argument t + xmin - center + 0.5 is exact in binary), phases 0,1 use
    // lines r-2..r+1 and phases 2,3 lines r-1..r+2.  The 16 weights live in registers for the whole tile.
    if (r0 >= 2 && r0 + kRasterRows + 2 <= h) {
        int k[4][4];
#pragma unroll
        for (int ph = 0; ph < 4; ++ph)
#pragma unroll
            for (int t = 0; t < 4; ++t) k[ph][t] = s_k[ph][ph < 2 ? t : t + 1];
#pragma unroll
        for (int rr = 0; rr < kRasterRows; ++rr) {
            const int r = r0 + rr;
            load_line(r + 2, win[4]);
#pragma unroll
            for (int ph = 0; ph < 4; ++ph) {
                const int b = ph < 2 ? 0 : 1;
                int v[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    int acc = (1 << 21) + win[b][c] * k[ph][0] + win[b + 1][c] * k[ph][1] + win[b + 2][c] * k[ph][2] +
                              win[b + 3][c] * k[ph][3];
                    acc >>= 22;
                    v[c] = __vimin_s32_relu(acc, 255);   // clamp to [0, 255] in one instruction
                }
                uint8_t *o = out + (size_t)(4 * r + ph) * w + x0;
                if (full && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
                    *reinterpret_cast<uint32_t *>(o) = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) |
                                                       ((uint32_t)v[3] << 24);
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (x0 + c < w) o[c] = (uint8_t)v[c];
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) win[j][c] = win[j + 1][c];
        }
        return;
    }
#pragma unroll
    for (int rr = 0; rr < kRasterRows; ++rr) {
        const int r = r0 + rr;
        if (r >= h) break;
        load_line(r + 2, win[4]);
#pragma unroll
        for (int ph = 0; ph < 4; ++ph) {
            const int k0 = s_k[4 * rr + ph][0], k1 = s_k[4 * rr + ph][1], k2 = s_k[4 * rr + ph][2],
                      k3 = s_k[4 * rr + ph][3], k4 = s_k[4 * rr + ph][4];
            int v[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                int acc = (1 << 21) + win[0][c] * k0 + win[1][c] * k1 + win[2][c] * k2 + win[3][c] * k3 + win[4][c] * k4;
                acc >>= 22;
                v[c] = __vimin_s32_relu(acc, 255);   // clamp to [0, 255] in one instruction
            }
            uint8_t *o = out + (size_t)(4 * r + ph) * w + x0;
            if (full && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
                *reinterpret_cast<uint32_t *>(o) = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) |
                                                   ((uint32_t)v[3] << 24);
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (x0 + c < w) o[c] = (uint8_t)v[c];
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) win[j][c] = win[j + 1][c];
    }
}

void launch_raster(wefax_ctx *ctx, const uint8_t *dig, size_t ds, long long n, int batch, const LineDev *lines,
                   const RecResult *res, uint8_t *raster, size_t rs, int max_width, int max_lines) {
    StageTimer timer(ctx, "raster");
    if (max_lines <= 0) return;
    const int cols_per_block = kRasterThreads * 4;
    dim3 grid((max_width + cols_per_block - 1) / cols_per_block, (max_lines + kRasterRows - 1) / kRasterRows, batch);
    raster_kernel<<<grid, kRasterThreads, 0, ctx->stream>>>(dig, ds, n, lines, res, raster, rs);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

}  // namespace wefax

namespace wefax {

SyncPlan prepare_sync(wefax_ctx *ctx, const LineDev *host_lines, int count, long long n) {
    SyncPlan sp;
    std::vector<SyncDev> sd(count);
    for (int r = 0; r < count; ++r) {
        const LineDev &ln = host_lines[r];
        SyncDev d;
        d.m = n - ln.L;
        d.fast = 3ll * ln.mindistance * (long long)sizeof(int) <= 200 * 1024;
        if (d.m <= 0) {
            d.m = d.m < 0 ? 0 : d.m;
            d.lim = d.limc = 0;
        } else {
            const long long w = ln.mindistance;
            d.lim = std::min<long long>(d.m, std::min<long long>(160ll * ln.width, 1500000ll));
            d.limc = std::min<long long>(d.m, ((d.lim + w + 1 + w - 1) / w) * w);
        }
        if (d.fast) {
            sp.any_fast = true;
            sp.max_lim = std::max(sp.max_lim, d.lim);
            sp.max_limc = std::max(sp.max_limc, d.limc);
            sp.max_w = std::max(sp.max_w, ln.mindistance);
            if (d.limc > 0)
                sp.max_wblocks = std::max(sp.max_wblocks, (int)((d.limc + ln.mindistance - 1) / ln.mindistance));
        }
        sd[r] = d;
    }
    sp.cs = (size_t)((sp.max_limc + 63) & ~63ll);
    sp.bs = (size_t)(((sp.max_lim + 31) / 32 + 4) & ~3ll);   // whole uint4s, 16-byte aligned rows
    const size_t ints = sp.cs * count;
    const size_t bytes = ints * sizeof(int) + sp.bs * count * sizeof(uint32_t) + (size_t)count * (sizeof(SyncDev) + 8) + 256;
    char *base = (char *)ctx->sync_buf.reserve(bytes);
    sp.corr = (int *)base;
    sp.bits = (uint32_t *)(sp.corr + sp.cs * count);
    sp.first_pos = (int *)(sp.bits + sp.bs * count);
    sp.need_scan = sp.first_pos + count;
    sp.sd = (SyncDev *)(((uintptr_t)(sp.need_scan + count) + 15) & ~(uintptr_t)15);
    // staged through pinned memory owned by the context: the copy is truly asynchronous and nothing has to wait
    // for it on the host (every API call ends with a stream synchronisation before the staging area is reused)
    const size_t up = sizeof(SyncDev) * (size_t)count;
    if (up > ctx->pinned_up_cap) {
        if (ctx->pinned_up) cudaFreeHost(ctx->pinned_up);
        ctx->pinned_up = nullptr;
        ctx->pinned_up_cap = 0;
        CUDA_CHECK(cudaMallocHost(&ctx->pinned_up, up + 4096));
        ctx->pinned_up_cap = up + 4096;
    }
    memcpy(ctx->pinned_up, sd.data(), up);
    CUDA_CHECK(cudaMemcpyAsync(sp.sd, ctx->pinned_up, up, cudaMemcpyHostToDevice, ctx->stream));
    return sp;
}

}  // namespace wefax
