// Transform drivers on top of the pass kernel: Hilbert envelope (smooth lengths
// and Bluestein), natural-order DFT for tests, FFT-domain resampling.
#include "ctx.cuh"
#include "fft_mid.cuh"

namespace wefax {

// ----------------------------- generic functors (cold paths) ---------------
struct LoadGeneric {
    int mode;               // 0 complex, 1 real zero-padded, 2 real*chirp zero-padded, 3 complex*chirp zero-padded
    const void *src;
    const float2 *chirp;
    size_t bstride;
    size_t n_valid;
    int conj;
    bool tma_source(const float2 **base, size_t *stride) const {
        *base = (const float2 *)src;
        *stride = bstride;
        return mode == 0 && conj == 0;
    }
    __device__ __forceinline__ float2 operator()(size_t i, int b) const {
        switch (mode) {
            case 0: {
                float2 v = __ldg((const float2 *)src + (size_t)b * bstride + i);
                if (conj) v.y = -v.y;
                return v;
            }
            case 1:
                return make_float2(i < n_valid ? __ldg((const float *)src + (size_t)b * bstride + i) : 0.f, 0.f);
            case 2: {
                if (i >= n_valid) return make_float2(0.f, 0.f);
                float x = __ldg((const float *)src + (size_t)b * bstride + i);
                float2 c = __ldg(chirp + i);
                return make_float2(x * c.x, x * c.y);
            }
            default: {
                if (i >= n_valid) return make_float2(0.f, 0.f);
                float2 v = __ldg((const float2 *)src + (size_t)b * bstride + i);
                if (conj) v.y = -v.y;
                return cmul(v, __ldg(chirp + i));
            }
        }
    }
};

struct StoreGeneric {
    int mode;   // 0 complex, 1 mul-table+conj, 2 bluestein hilbert mid, 3 abs, 4 real part,
                // 5 bluestein spectrum (natural), 6 bluestein real part
    void *dst;
    const float2 *table;    // mode 1: by position; modes 5/6: chirp
    size_t bstride;
    size_t n_valid;
    uint32_t n;             // transform length of the Hilbert mask
    float scale;
    int conj;
    using Side = NoSide;
    __device__ __forceinline__ Side side_load(size_t, int) const { return Side{}; }
    __device__ __forceinline__ int column_aux(int) const { return 0; }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int, int, Side = Side{}) const {
        switch (mode) {
            case 0:
                v.x *= scale;
                v.y *= conj ? -scale : scale;
                ((float2 *)dst)[(size_t)b * bstride + i] = v;
                break;
            case 1: {
                float2 w = cmul(v, __ldg(table + i));
                ((float2 *)dst)[(size_t)b * bstride + i] = make_float2(w.x, -w.y);
                break;
            }
            case 2: {
                float h = 0.f;
                if (i < n) {
                    uint64_t k2 = 2ull * i;
                    h = i == 0 ? 1.f : (k2 < n ? 2.f : (k2 == n ? 1.f : 0.f));
                }
                h *= scale;
                ((float2 *)dst)[(size_t)b * bstride + i] = make_float2(v.x * h, v.y * h);
                break;
            }
            case 3:
                if (i < n_valid) ((float *)dst)[(size_t)b * bstride + i] = scale * sqrtf(fmaf(v.x, v.x, v.y * v.y));
                break;
            case 4:
                if (i < n_valid) ((float *)dst)[(size_t)b * bstride + i] = scale * v.x;
                break;
            case 5:
                if (i < n_valid) {
                    float2 w = cmul(make_float2(v.x, -v.y), __ldg(table + i));
                    ((float2 *)dst)[(size_t)b * bstride + i] = make_float2(w.x * scale, w.y * scale);
                }
                break;
            default:
                if (i < n_valid) {
                    float2 w = cmul(make_float2(v.x, -v.y), __ldg(table + i));
                    ((float *)dst)[(size_t)b * bstride + i] = scale * w.x;
                }
                break;
        }
    }
};

// ----------------------------- position <-> frequency ----------------------
struct PosMap {
    int npass;
    int R[kMaxPasses];
    uint32_t S[kMaxPasses];
    __device__ __forceinline__ uint32_t freq(uint32_t pos) const {
        uint32_t k = 0, mult = 1;
#pragma unroll
        for (int i = 0; i < kMaxPasses; ++i)
            if (i < npass) {
                uint32_t d = (pos / S[i]) % (uint32_t)R[i];
                k += d * mult;
                mult *= (uint32_t)R[i];
            }
        return k;
    }
    __device__ __forceinline__ uint32_t pos(uint32_t k) const {
        uint32_t p = 0;
#pragma unroll
        for (int i = 0; i < kMaxPasses; ++i)
            if (i < npass) {
                uint32_t d = k % (uint32_t)R[i];
                k /= (uint32_t)R[i];
                p += d * S[i];
            }
        return p;
    }
};

static PosMap pos_map(const FftPlan *plan) {
    PosMap m{};
    m.npass = plan->npass;
    for (int i = 0; i < plan->npass; ++i) {
        m.R[i] = plan->Rs[i];
        m.S[i] = (uint32_t)plan->S[i];
    }
    return m;
}

// engine order -> natural order (first `keep` frequencies), or the reverse with zero fill
__global__ void engine_to_natural_kernel(const float2 *z, size_t zs, float2 *out, size_t os, uint32_t keep, PosMap pm) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= keep) return;
    out[(size_t)blockIdx.y * os + k] = z[(size_t)blockIdx.y * zs + pm.pos(k)];
}
__global__ void natural_to_engine_kernel(const float2 *in, size_t is, uint32_t have, float2 *z, size_t zs, uint32_t n,
                                         PosMap pm, int conj) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    uint32_t k = pm.freq(p);
    float2 v = make_float2(0.f, 0.f);
    if (k < have) {
        v = in[(size_t)blockIdx.y * is + k];
        if (conj) v.y = -v.y;
    }
    z[(size_t)blockIdx.y * zs + p] = v;
}

// ----------------------------- plans ---------------------------------------
FftPlan *get_plan(wefax_ctx *ctx, long long n) {
    auto it = ctx->plans.find(n);
    if (it != ctx->plans.end()) return it->second.get();
    std::unique_ptr<FftPlan> plan = make_plan(n, ctx->stream);
    FftPlan *raw = plan.get();
    ctx->plans[n] = std::move(plan);   // nullptr is cached too: "needs Bluestein"
    return raw;
}

static LoadComplex load_c(const float2 *p, size_t bs, int conj = 0) { return LoadComplex{p, bs, conj}; }

// forward passes 0..P-1 with `ld` feeding pass 0 and `st` finishing pass P-1
template <class LoadFirst, class StoreLast>
static void run_forward(wefax_ctx *ctx, FftPlan *plan, const LoadFirst &ld, const StoreLast &st, float2 *z, size_t zs,
                        int batch) {
    const int P = plan->npass;
    if (P == 1) {
        launch_pass(ctx, plan->fwd[0], ld, st, batch);
        return;
    }
    launch_pass(ctx, plan->fwd[0], ld, StoreComplex{z, zs, 1.f, 0}, batch);
    for (int i = 1; i < P - 1; ++i) launch_pass(ctx, plan->fwd[i], load_c(z, zs), StoreComplex{z, zs, 1.f, 0}, batch);
    launch_pass(ctx, plan->fwd[P - 1], load_c(z, zs), st, batch);
}

// inverse-structure passes P-1..0 (engine order in, natural order out); the data
// must already be conjugated/scaled by whoever produced it
template <class LoadFirst, class StoreLast>
static void run_inverse(wefax_ctx *ctx, FftPlan *plan, const LoadFirst &ld, const StoreLast &st, float2 *z, size_t zs,
                        int batch) {
    const int P = plan->npass;
    if (P == 1) {
        launch_pass(ctx, plan->inv[0], ld, st, batch);
        return;
    }
    launch_pass(ctx, plan->inv[P - 1], ld, StoreComplex{z, zs, 1.f, 0}, batch);
    for (int i = P - 2; i >= 1; --i) launch_pass(ctx, plan->inv[i], load_c(z, zs), StoreComplex{z, zs, 1.f, 0}, batch);
    launch_pass(ctx, plan->inv[0], load_c(z, zs), st, batch);
}

// |hilbert(x)| for `batch` real sequences of length plan->n (no median filter).
// x: real input (stride xs) or nullptr when z already holds (x, 0); z: complex scratch
// (stride zs >= n); env: output (stride es).
static void hilbert_envelope(wefax_ctx *ctx, FftPlan *plan, const float *x, size_t xs, float2 *z, size_t zs,
                             float *env, size_t es, int batch) {
    const size_t n = (size_t)plan->n;
    StoreHilbert sh{z, zs, plan->outer(), (uint32_t)n, (int)(n / plan->Rs[plan->npass - 1]), (float)(1.0 / (double)n)};
    if (x)
        run_forward(ctx, plan, LoadReal{x, xs, n}, sh, z, zs, batch);
    else   // z already holds (x, 0): every pass can take its tile through TMA
        run_forward(ctx, plan, load_c(z, zs), sh, z, zs, batch);
    run_inverse(ctx, plan, load_c(z, zs), StoreAbs{env, es, n, 1.f}, z, zs, batch);
}

// ----------------------------- real-input Hilbert envelope ------------------
// x real, n = 2M.  z[m] = x[2m] + i*x[2m+1]; Z = DFT_M(z).  With E/O the spectra of the
// even/odd samples (E = (Z[k] + conj Z[M-k])/2, O = (Z[k] - conj Z[M-k])/(2i)) the
// spectrum of x is X[k] = E + w^k O, w = exp(-2*pi*i/n).  The Hilbert transform
// y = H[x] has Y[k] = -i X[k] (0 < k < M), Y[0] = Y[M] = 0; packing y the same way,
// Z'[k] = conj(w^k) (Z[k] + conj Z[M-k])/2 - w^k (Z[k] - conj Z[M-k])/2,  Z'[0] = 0,
// and IDFT_M(Z') = y[2m] + i*y[2m+1].  This kernel turns Z into conj(Z')/M in place
// (conjugated so the inverse can run on the forward kernels); engine order throughout.
// One CTA per engine-order row (all digits but the last fixed): frequency
// k = kb + ncols*j for j = 0..R_last-1; its mirror M-k lives in the row of
// kb' = (ncols - kb) mod ncols at j' = R_last-1-j (kb > 0) or (R_last-j) mod R_last
// (kb = 0): both rows are walked contiguously, one forwards and one backwards.
struct PairGeom {
    int nouter;                 // passes - 1
    int Rout[kMaxPasses];       // R_0 .. R_{P-2}
    int R_last, ncols;
};

constexpr int kPairRows = 8;   // engine-order rows per CTA

__global__ void __launch_bounds__(256)
hilbert_pairs_kernel(float2 *z_all, size_t zs, uint32_t M, PairGeom g, const float2 *tw_lo, const float2 *tw_hi,
                     float inv_m) {
    __shared__ int s_kb[kPairRows], s_o2[kPairRows];
    float2 *z = z_all + (size_t)blockIdx.y * zs;
    const int o0 = blockIdx.x * kPairRows;
    if (threadIdx.x < kPairRows) {
        // digits of this row (most significant first in o), its base frequency and the mirrored row
        const int o = o0 + threadIdx.x;
        int kb = 0, o2 = -1;
        if (o < g.ncols) {
            int d[kMaxPasses], rem = o;
#pragma unroll
            for (int i = kMaxPasses - 1; i >= 0; --i)
                if (i < g.nouter) {
                    d[i] = rem % g.Rout[i];
                    rem /= g.Rout[i];
                }
            int mult = 1;
#pragma unroll
            for (int i = 0; i < kMaxPasses; ++i)
                if (i < g.nouter) {
                    kb += d[i] * mult;
                    mult *= g.Rout[i];
                }
            int rem2 = kb ? g.ncols - kb : 0;
            o2 = 0;
#pragma unroll
            for (int i = 0; i < kMaxPasses; ++i)
                if (i < g.nouter) {
                    o2 = o2 * g.Rout[i] + rem2 % g.Rout[i];
                    rem2 /= g.Rout[i];
                }
        }
        s_kb[threadIdx.x] = kb;
        s_o2[threadIdx.x] = o2;
    }
    __syncthreads();
    for (int r = 0; r < kPairRows; ++r) {
        const int o = o0 + r, o2 = s_o2[r], kb = s_kb[r];
        if (o >= g.ncols || o2 < o) continue;             // the mirrored row's CTA owns these pairs
        float2 *row = z + (size_t)o * g.R_last;
        float2 *row2 = z + (size_t)o2 * g.R_last;
        for (int j = threadIdx.x; j < g.R_last; j += blockDim.x) {
            const int j2 = kb ? g.R_last - 1 - j : (j ? g.R_last - j : 0);
            if (o2 == o && j2 < j) continue;              // self-mirrored row: each pair once
            const uint32_t k = (uint32_t)kb + (uint32_t)g.ncols * (uint32_t)j;
            if (k == 0) {
                row[0] = make_float2(0.f, 0.f);
                continue;
            }
            const float2 zk = row[j], zm = row2[j2];
            const float2 lo = __ldg(tw_lo + (k & ((1u << kTwLoBits) - 1))), hi = __ldg(tw_hi + (k >> kTwLoBits));
            const float2 w = cmul(lo, hi);                // w_n^k
            const float2 s = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));   // (zk + conj zm)/2
            const float2 d = make_float2(0.5f * (zk.x - zm.x), 0.5f * (zk.y + zm.y));   // (zk - conj zm)/2
            const float2 a = cmul(make_float2(w.x, -w.y), s), b = cmul(w, d);           // Z'[k] = conj(w) s - w d
            row[j] = make_float2((a.x - b.x) * inv_m, -(a.y - b.y) * inv_m);
            if (!(o2 == o && j2 == j)) {
                // Z'[M-k] = -w conj(s) - conj(w) conj(d)
                const float2 a2 = cmul(w, make_float2(s.x, -s.y)),
                             b2 = cmul(make_float2(w.x, -w.y), make_float2(d.x, -d.y));
                row2[j2] = make_float2(-(a2.x + b2.x) * inv_m, (a2.y + b2.y) * inv_m);
            }
        }
    }
}

// row pairs (o, mirrored o, base frequency) and w_{2R}^j for the fused middle kernel, built once per plan
static void ensure_mid_tables(wefax_ctx *ctx, FftPlan *half) {
    if (half->mid_npairs) return;
    const int P = half->npass;
    const int nouter = P - 1;
    const int R = half->Rs[P - 1];
    const int ncols = (int)(half->n / R);
    std::vector<fast::MidRow> rows;
    rows.reserve(ncols / 2 + 2);
    for (int o = 0; o < ncols; ++o) {
        int d[kMaxPasses] = {0, 0, 0, 0}, rem = o;
        for (int i = nouter - 1; i >= 0; --i) {
            d[i] = rem % half->Rs[i];
            rem /= half->Rs[i];
        }
        int kb = 0, mult = 1;
        for (int i = 0; i < nouter; ++i) {
            kb += d[i] * mult;
            mult *= half->Rs[i];
        }
        int rem2 = kb ? ncols - kb : 0, o2 = 0;
        for (int i = 0; i < nouter; ++i) {
            o2 = o2 * half->Rs[i] + rem2 % half->Rs[i];
            rem2 /= half->Rs[i];
        }
        if (o2 >= o) rows.push_back(fast::MidRow{o, o2, kb, 0});
    }
    std::vector<float2> twB(R);
    for (int j = 0; j < R; ++j) {
        const double ang = -M_PI * (double)j / (double)R;   // w_{2R}^j
        twB[j] = make_float2((float)cos(ang), (float)sin(ang));
    }
    const size_t rows_bytes = (rows.size() * sizeof(fast::MidRow) + 255) & ~size_t(255);
    char *base = (char *)half->mid_tab.reserve(rows_bytes + R * sizeof(float2));
    CUDA_CHECK(cudaMemcpyAsync(base, rows.data(), rows.size() * sizeof(fast::MidRow), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_CHECK(cudaMemcpyAsync(base + rows_bytes, twB.data(), R * sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));   // the host vectors go out of scope
    half->mid_npairs = (int)rows.size();
}

template <int R1, int R2>
static void launch_mid(wefax_ctx *ctx, FftPlan *half, float2 *z, size_t zs, int batch) {
    using K = fast::MidWarpCfg<R1, R2>;
    auto kern = fast::hilbert_mid_warp_kernel<R1, R2>;
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
    const int P = half->npass;
    const PassDev &pi = half->inv[P - 1];
    fast::MidArgs a{};
    a.z = z;
    a.zs = zs;
    const size_t rows_bytes = ((size_t)half->mid_npairs * sizeof(fast::MidRow) + 255) & ~size_t(255);
    a.rows = half->mid_tab.as<fast::MidRow>();
    a.twB = (const float2 *)(half->mid_tab.as<char>() + rows_bytes);
    a.npairs = half->mid_npairs;
    a.total_tiles = a.npairs * batch;               // one pair per warp and round
    a.ncols = (int)(half->n / K::R);
    a.twR = pi.twR;
    a.tw2_lo = half->tw2_lo;
    a.tw2_hi = half->tw2_hi;
    a.tw_lo = pi.tw_lo;
    a.tw_hi = pi.tw_hi;
    a.tw_mode = pi.tw_mode;
    a.ko_R = pi.ko_R;
    a.inv_m = (float)(1.0 / (double)half->n);
    const int ctas = (a.total_tiles + K::WARPS - 1) / K::WARPS;
    const int grid = std::min(ctas, ctx->sm_count * per_sm);
    StageTimer timer(ctx, "hilbert_mid");
    kern<<<grid, K::T, K::SMEM, ctx->stream>>>(a);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

void hilbert_envelope_real(wefax_ctx *ctx, FftPlan *half, const float *x, size_t xs, float2 *z, size_t zs, float *env,
                           size_t es, int batch, bool want_y) {
    const size_t M = (size_t)half->n;
    const int P = half->npass;
    // x / env strides are in floats and must be even so that pair views stay aligned
    const StoreEnvPairs store_env{(float2 *)env, (const float2 *)x, es / 2, xs / 2, want_y ? 1 : 0};
    int R1 = 0, R2 = 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(z) & 15) == 0 && (batch == 1 || (zs & 1) == 0);
    if (P >= 2 && aligned && (long long)batch * (long long)(M / half->Rs[P - 1]) < (1ll << 30) &&
        fast::mid_pair(half->Rs[P - 1], &R1, &R2)) {
        // passes 0 .. P-2 forward, the fused middle, passes P-2 .. 0 inverse
        ensure_mid_tables(ctx, half);
        launch_pass(ctx, half->fwd[0], load_c((const float2 *)x, xs / 2), StoreComplex{z, zs, 1.f, 0}, batch);
        for (int i = 1; i < P - 1; ++i) launch_pass(ctx, half->fwd[i], load_c(z, zs), StoreComplex{z, zs, 1.f, 0}, batch);
        switch (R1 * 100 + R2) {
            case 1428: launch_mid<14, 28>(ctx, half, z, zs, batch); break;
            case 1014: launch_mid<10, 14>(ctx, half, z, zs, batch); break;
            case 1520: launch_mid<15, 20>(ctx, half, z, zs, batch); break;
            case 1415: launch_mid<14, 15>(ctx, half, z, zs, batch); break;
            default: launch_mid<10, 15>(ctx, half, z, zs, batch); break;
        }
        for (int i = P - 2; i >= 1; --i) launch_pass(ctx, half->inv[i], load_c(z, zs), StoreComplex{z, zs, 1.f, 0}, batch);
        launch_pass(ctx, half->inv[0], load_c(z, zs), store_env, batch);
        return;
    }
    run_forward(ctx, half, load_c((const float2 *)x, xs / 2), StoreComplex{z, zs, 1.f, 0}, z, zs, batch);
    {
        StageTimer timer(ctx, "hilbert_pairs");
        PairGeom g{};
        g.nouter = half->npass - 1;
        for (int i = 0; i < g.nouter; ++i) g.Rout[i] = half->Rs[i];
        g.R_last = half->Rs[half->npass - 1];
        g.ncols = (int)(M / g.R_last);
        dim3 grid((unsigned)((g.ncols + kPairRows - 1) / kPairRows), batch);
        hilbert_pairs_kernel<<<grid, 256, 0, ctx->stream>>>(z, zs, (uint32_t)M, g, half->tw2_lo, half->tw2_hi,
                                                           (float)(1.0 / (double)M));
        CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
    run_inverse(ctx, half, load_c(z, zs), store_env, z, zs, batch);
}

void fft_c2c_natural(wefax_ctx *ctx, FftPlan *plan, const float2 *in, float2 *out, float2 *scratch, int batch,
                     bool inverse) {
    const size_t n = (size_t)plan->n;
    PosMap pm = pos_map(plan);
    dim3 grid((unsigned)((n + 255) / 256), batch);
    if (!inverse) {
        run_forward(ctx, plan, load_c(in, n), StoreComplex{scratch, n, 1.f, 0}, scratch, n, batch);
        engine_to_natural_kernel<<<grid, 256, 0, ctx->stream>>>(scratch, n, out, n, (uint32_t)n, pm);
        ctx->launches++;
    } else {
        natural_to_engine_kernel<<<grid, 256, 0, ctx->stream>>>(in, n, (uint32_t)n, scratch, n, (uint32_t)n, pm, 1);
        ctx->launches++;
        run_inverse(ctx, plan, load_c(scratch, n), StoreComplex{out, n, (float)(1.0 / (double)n), 1}, scratch, n, batch);
    }
    CUDA_CHECK(cudaGetLastError());
}

// ----------------------------- Bluestein -----------------------------------
__global__ void chirp_kernel(float2 *c, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long e = ((unsigned long long)i * i) % (2ull * n);
    double s, co;
    sincospi(-(double)e / (double)n, &s, &co);
    c[i] = make_float2((float)co, (float)s);
}
__global__ void chirp_wrap_kernel(const float2 *c, float2 *v, uint32_t n, uint32_t m) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    float2 out = make_float2(0.f, 0.f);
    if (j < n) out = make_float2(c[j].x, -c[j].y);
    else if (m - j < n) out = make_float2(c[m - j].x, -c[m - j].y);
    v[j] = out;
}

static Bluestein *get_bluestein(wefax_ctx *ctx, long long n) {
    auto it = ctx->bluestein.find(n);
    if (it != ctx->bluestein.end()) return it->second.get();
    auto b = std::make_unique<Bluestein>();
    b->n = n;
    b->m = next_smooth_length(2 * n - 1);
    if (b->m <= 0) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "no FFT length found for Bluestein n=%lld", n);
    b->plan = get_plan(ctx, b->m);
    if (!b->plan) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "Bluestein length %lld not plannable", b->m);
    float2 *c = (float2 *)b->chirp.reserve((size_t)n * sizeof(float2));
    float2 *vh = (float2 *)b->vhat.reserve((size_t)b->m * sizeof(float2));
    DevBuf tmp;
    float2 *v = (float2 *)tmp.reserve((size_t)b->m * sizeof(float2));
    chirp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(c, (uint32_t)n);
    chirp_wrap_kernel<<<(unsigned)((b->m + 255) / 256), 256, 0, ctx->stream>>>(c, v, (uint32_t)n, (uint32_t)b->m);
    ctx->launches += 2;
    run_forward(ctx, b->plan, load_c(v, (size_t)b->m), StoreComplex{vh, (size_t)b->m, (float)(1.0 / (double)b->m), 0},
                vh, (size_t)b->m, 1);
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    Bluestein *raw = b.get();
    ctx->bluestein[n] = std::move(b);
    return raw;
}

static LoadGeneric lg(int mode, const void *src, const float2 *chirp, size_t bs, size_t n_valid, int conj = 0) {
    return LoadGeneric{mode, src, chirp, bs, n_valid, conj};
}
static StoreGeneric sg(int mode, void *dst, const float2 *table, size_t bs, size_t n_valid, uint32_t n, float scale,
                       int conj = 0) {
    return StoreGeneric{mode, dst, table, bs, n_valid, n, scale, conj};
}

// Bluestein path for lengths with a large prime factor
static void hilbert_envelope_bluestein(wefax_ctx *ctx, long long n, const float *x, size_t xs, float *env, size_t es,
                                       int batch) {
    Bluestein *b = get_bluestein(ctx, n);
    const size_t m = (size_t)b->m;
    float2 *z = (float2 *)ctx->work_z.reserve(m * sizeof(float2) * batch);
    const float2 *c = b->chirp.as<float2>();
    const float2 *vh = b->vhat.as<float2>();
    // DFT_n(x) by chirp convolution; r = conj(conv)
    run_forward(ctx, b->plan, lg(2, x, c, xs, (size_t)n), sg(1, z, vh, m, m, 0, 1.f), z, m, batch);
    // u2 = (h/n) * r for k < n, zero beyond (|chirp| = 1 cancels, see DESIGN.md)
    run_inverse(ctx, b->plan, lg(0, z, nullptr, m, m), sg(2, z, nullptr, m, m, (uint32_t)n, (float)(1.0 / (double)n)),
                z, m, batch);
    run_forward(ctx, b->plan, lg(0, z, nullptr, m, m), sg(1, z, vh, m, m, 0, 1.f), z, m, batch);
    run_inverse(ctx, b->plan, lg(0, z, nullptr, m, m), sg(3, env, nullptr, es, (size_t)n, 0, 1.f), z, m, batch);
}

EnvelopeForm envelope_form(wefax_ctx *ctx, long long n) {
    EnvelopeForm f;
    f.n = n;
    f.half = (n % 2 == 0) ? get_plan(ctx, n / 2) : nullptr;
    f.plan = f.half ? nullptr : get_plan(ctx, n);
    f.zlen = f.half ? n / 2 : (f.plan ? n : next_smooth_length(2 * n - 1));
    if (f.zlen <= 0) WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "no transform length for n=%lld", n);
    return f;
}

float2 *envelope_scratch(wefax_ctx *ctx, const EnvelopeForm &f, int batch) {
    if (!f.half && !f.plan) return nullptr;
    return (float2 *)ctx->work_z.reserve((size_t)batch * f.zlen * sizeof(float2));
}

void launch_envelope(wefax_ctx *ctx, const EnvelopeForm &f, const float *audio, size_t as, float2 *z, float *env,
                     size_t es, int batch) {
    if (f.half)
        hilbert_envelope_real(ctx, f.half, audio, as, z, (size_t)f.zlen, env, es, batch);
    else if (f.plan)
        hilbert_envelope(ctx, f.plan, nullptr, 0, z, (size_t)f.zlen, env, es, batch);
    else
        hilbert_envelope_bluestein(ctx, f.n, audio, as, env, es, batch);
}

// ----------------------------- resample ------------------------------------
// scipy.signal.resample(x, num) for real x (wefax.py:384): X = rfft(x); keep
// m2 = min(num, n)//2 + 1 bins; unpaired bin m/2 doubled (down) or halved (up)
// when m is even and num != n; y = irfft(X * num/n, num).
__global__ void resample_spectrum_kernel(const float2 *X, size_t xs, float2 *Zc, size_t zs, uint32_t m2, uint32_t m,
                                         uint32_t n, uint32_t num, float scale) {
    // Zc[k] = conj of the one-sided inverse-transform input (irfft as Re(IDFT) of a one-sided spectrum)
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m2) return;
    float2 v = X[(size_t)blockIdx.y * xs + k];
    if ((m & 1u) == 0 && num != n && k == m / 2) {
        float f = num < n ? 2.f : 0.5f;
        v.x *= f;
        v.y *= f;
    }
    float w = 2.f;
    if (k == 0) {
        w = 1.f;
        v.y = 0.f;   // irfft ignores the imaginary part of DC
    } else if ((num & 1u) == 0 && k == num / 2) {
        w = 1.f;
        v.y = 0.f;   // ... and of the Nyquist bin
    }
    w *= scale;
    Zc[(size_t)blockIdx.y * zs + k] = make_float2(v.x * w, -v.y * w);
}

// forward DFT of real x, first `keep` bins in natural order into X (stride xs_out)
void spectrum_natural(wefax_ctx *ctx, long long n, const float *x, size_t xs, float2 *X, size_t xs_out,
                      uint32_t keep, int batch) {
    FftPlan *plan = get_plan(ctx, n);
    if (plan) {
        float2 *z = (float2 *)ctx->work_z.reserve((size_t)n * sizeof(float2) * batch);
        run_forward(ctx, plan, LoadReal{x, xs, (size_t)n}, StoreComplex{z, (size_t)n, 1.f, 0}, z, (size_t)n, batch);
        dim3 grid((keep + 255) / 256, batch);
        engine_to_natural_kernel<<<grid, 256, 0, ctx->stream>>>(z, (size_t)n, X, xs_out, keep, pos_map(plan));
        ctx->launches++;
        CUDA_CHECK(cudaGetLastError());
        return;
    }
    Bluestein *b = get_bluestein(ctx, n);
    const size_t m = (size_t)b->m;
    float2 *z = (float2 *)ctx->work_z.reserve(m * sizeof(float2) * batch);
    run_forward(ctx, b->plan, lg(2, x, b->chirp.as<float2>(), xs, (size_t)n), sg(1, z, b->vhat.as<float2>(), m, m, 0, 1.f),
                z, m, batch);
    run_inverse(ctx, b->plan, lg(0, z, nullptr, m, m), sg(5, X, b->chirp.as<float2>(), xs_out, keep, 0, 1.f), z, m, batch);
}

// y = Re(DFT_num(Zc)) where Zc (natural order, `have` bins, zero beyond) is the
// conjugated one-sided spectrum
static void real_from_onesided(wefax_ctx *ctx, long long num, const float2 *Zc, size_t zcs, uint32_t have, float *y,
                               size_t ys, int batch) {
    FftPlan *plan = get_plan(ctx, num);
    if (plan) {
        float2 *z = (float2 *)ctx->work_z.reserve((size_t)num * sizeof(float2) * batch);
        dim3 grid((unsigned)((num + 255) / 256), batch);
        natural_to_engine_kernel<<<grid, 256, 0, ctx->stream>>>(Zc, zcs, have, z, (size_t)num, (uint32_t)num,
                                                                pos_map(plan), 0);
        ctx->launches++;
        CUDA_CHECK(cudaGetLastError());
        run_inverse(ctx, plan, load_c(z, (size_t)num), StoreRealPart{y, ys, (size_t)num, 1.f}, z, (size_t)num, batch);
        return;
    }
    Bluestein *b = get_bluestein(ctx, num);
    const size_t m = (size_t)b->m;
    float2 *z = (float2 *)ctx->work_z.reserve(m * sizeof(float2) * batch);
    run_forward(ctx, b->plan, lg(3, Zc, b->chirp.as<float2>(), zcs, have), sg(1, z, b->vhat.as<float2>(), m, m, 0, 1.f), z,
                m, batch);
    run_inverse(ctx, b->plan, lg(0, z, nullptr, m, m), sg(6, y, b->chirp.as<float2>(), ys, (size_t)num, 0, 1.f), z, m,
                batch);
}

// ---- real-input fast path of the resampler (n and num even, both halves plannable) ----------------
// rfft through a half-length complex transform of the packed signal z[m] = x[2m] + i*x[2m+1]:
// X[k] = E + w_n^k * O with E = (Z[k] + conj Z[M-k]) / 2, O = (Z[k] - conj Z[M-k]) / (2i), Z in engine order.
__global__ void rfft_gather_kernel(const float2 *z, size_t zs, float2 *X, size_t xs, uint32_t keep, uint32_t M,
                                   PosMap pm, const float2 *tw_lo, const float2 *tw_hi) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= keep) return;
    const float2 *zb = z + (size_t)blockIdx.y * zs;
    const uint32_t ka = k % M, kb = (M - ka) % M;
    const float2 zk = zb[pm.pos(ka)], zm = zb[pm.pos(kb)];
    const float2 E = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
    const float2 O = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));   // (zk - conj zm) / (2i)
    const float2 w = cmul(__ldg(tw_lo + (k & ((1u << kTwLoBits) - 1))), __ldg(tw_hi + (k >> kTwLoBits)));   // w_n^k
    X[(size_t)blockIdx.y * xs + k] = cadd(E, cmul(w, O));
}

// scipy's bin selection and scaling (see resample_spectrum_kernel) on the fly, then the packed spectrum of the
// half-length inverse: Z'[k] = A + i*B, A = (Y[k] + conj Y[M'-k]) / 2, B = (Y[k] - conj Y[M'-k]) * w_num^(-k) / 2,
// stored conjugated and scaled at its engine position (the inverse runs the forward kernels on conjugated data).
__global__ void irfft_scatter_kernel(const float2 *X, size_t xs, uint32_t m2, uint32_t m, uint32_t n, uint32_t num,
                                     float2 *z, size_t zs, uint32_t Mp, PosMap pm, const float2 *tw_lo,
                                     const float2 *tw_hi, float scale) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Mp) return;
    const float2 *Xb = X + (size_t)blockIdx.y * xs;
    auto Y = [&](uint32_t k) {   // one-sided spectrum handed to irfft(., num): bins >= m2 are zero
        float2 v = make_float2(0.f, 0.f);
        if (k < m2) {
            v = Xb[k];
            if ((m & 1u) == 0 && num != n && k == m / 2) {
                const float f = num < n ? 2.f : 0.5f;
                v.x *= f;
                v.y *= f;
            }
            if (k == 0 || k == Mp) v.y = 0.f;   // irfft ignores the imaginary part of DC and Nyquist
        }
        return v;
    };
    const uint32_t k = pm.freq(p);
    const float2 yk = Y(k), ym = Y(Mp - k);                       // k = 0 pairs with the Nyquist bin
    const float2 A = make_float2(0.5f * (yk.x + ym.x), 0.5f * (yk.y - ym.y));
    const float2 D = make_float2(0.5f * (yk.x - ym.x), 0.5f * (yk.y + ym.y));
    const float2 w = cmul(__ldg(tw_lo + (k & ((1u << kTwLoBits) - 1))), __ldg(tw_hi + (k >> kTwLoBits)));   // w_num^k
    const float2 B = cmul(D, make_float2(w.x, -w.y));
    // Z' = A + i*B;  store conj(Z') * scale
    z[(size_t)blockIdx.y * zs + p] = make_float2((A.x - B.y) * scale, -(A.y + B.x) * scale);
}

static bool resample_real_fast(wefax_ctx *ctx, long long n, long long num, const float *x, size_t xs, float *y,
                               size_t ys, int batch) {
    if ((n & 1) || (num & 1) || (xs & 1) || (ys & 1)) return false;
    if ((reinterpret_cast<uintptr_t>(x) & 7) || (reinterpret_cast<uintptr_t>(y) & 7)) return false;
    FftPlan *hin = get_plan(ctx, n / 2), *hout = get_plan(ctx, num / 2);
    if (!hin || !hout) return false;
    const uint32_t M = (uint32_t)(n / 2), Mp = (uint32_t)(num / 2);
    const uint32_t m = (uint32_t)std::min(n, num), m2 = m / 2 + 1;
    float2 *z = (float2 *)ctx->work_z.reserve((size_t)std::max(M, Mp) * sizeof(float2) * batch);
    float2 *X = (float2 *)ctx->work_misc.reserve((size_t)m2 * sizeof(float2) * batch);
    run_forward(ctx, hin, load_c((const float2 *)x, xs / 2), StoreComplex{z, (size_t)M, 1.f, 0}, z, (size_t)M, batch);
    {
        StageTimer timer(ctx, "rfft_gather");
        dim3 grid((m2 + 255) / 256, batch);
        rfft_gather_kernel<<<grid, 256, 0, ctx->stream>>>(z, (size_t)M, X, (size_t)m2, m2, M, pos_map(hin), hin->tw2_lo,
                                                         hin->tw2_hi);
    }
    {
        StageTimer timer(ctx, "irfft_scatter");
        dim3 grid((Mp + 255) / 256, batch);
        // X * (num / n), the 1/2 of A and B is in the kernel, 1/M' of the inverse transform: together 2/n ... / 2 = 1/n * (num/Mp)/...
        const float scale = (float)(((double)num / (double)n) / (double)Mp);
        irfft_scatter_kernel<<<grid, 256, 0, ctx->stream>>>(X, (size_t)m2, m2, m, (uint32_t)n, (uint32_t)num, z, (size_t)Mp,
                                                           Mp, pos_map(hout), hout->tw2_lo, hout->tw2_hi, scale);
    }
    ctx->launches += 2;
    CUDA_CHECK(cudaGetLastError());
    run_inverse(ctx, hout, load_c(z, (size_t)Mp), StoreComplex{(float2 *)y, ys / 2, 1.f, 1}, z, (size_t)Mp, batch);
    return true;
}

void resample_real(wefax_ctx *ctx, long long n, long long num, const float *x, size_t xs, float *y, size_t ys,
                   int batch) {
    if (resample_real_fast(ctx, n, num, x, xs, y, ys, batch)) return;
    const uint32_t m = (uint32_t)std::min(n, num);
    const uint32_t m2 = m / 2 + 1;
    float2 *X = (float2 *)ctx->work_misc.reserve((size_t)m2 * sizeof(float2) * 2 * batch);
    float2 *Zc = X + (size_t)m2 * batch;
    spectrum_natural(ctx, n, x, xs, X, m2, m2, batch);
    dim3 grid((m2 + 255) / 256, batch);
    // X * (num/n) and the 1/num of irfft combine to 1/n
    resample_spectrum_kernel<<<grid, 256, 0, ctx->stream>>>(X, m2, Zc, m2, m2, m, (uint32_t)n, (uint32_t)num,
                                                           (float)(1.0 / (double)n));
    ctx->launches++;
    CUDA_CHECK(cudaGetLastError());
    real_from_onesided(ctx, num, Zc, m2, m2, y, ys, batch);
}

}  // namespace wefax
