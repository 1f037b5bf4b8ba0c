// Mixed-radix, multi-pass, in-place complex FFT for one long 1-D sequence (or a
// batch of them).  Replaces the pocketfft calls under scipy.signal.hilbert /
// scipy.signal.resample on the reference's path (wefax.py:174,384).
//
// n = R_0 * R_1 * ... * R_{P-1}.  Element index i = sum_i n_i * S_i with
// S_i = prod_{j>i} R_j.  The forward transform is P decimation-in-frequency
// passes: pass i transforms, for every "column" (all other digits fixed), the R_i
// elements spaced S_i apart, multiplies by w_{L_i}^{k_i * m} (L_i = R_i*S_i, m the
// column offset inside its length-L_i sub-problem) and stores in place.  After the
// last pass the value of frequency k = k_0 + R_0*k_1 + R_0*R_1*k_2 + ... sits at
// position sum_i k_i*S_i ("engine order").  The inverse runs the mirrored
// decimation-in-time passes P-1..0 (twiddle on load) and ends in natural order,
// so a forward/inverse pair needs no transposition at all; point-wise spectral
// work (Hilbert mask, Bluestein products) is fused into the stores and only needs
// the position -> frequency map.
//
// One CTA owns a tile of C adjacent columns x R rows in shared memory, runs the
// radix-2..32 stages there (prime radices 2,3,5,7,11,13 and in-register composites
// such as 14, 15, 16, 25, 28; in-place DIF, digit-reversed read-out),
// and touches global memory exactly once per element per pass: coalesced C*8-byte
// row segments for strided passes, one contiguous C*R*8-byte chunk for the last
// (stride-1) pass.
#pragma once

#include <type_traits>

#include <cuda.h>   // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "common.cuh"

namespace wefax {

constexpr int kMaxStages = 14;
constexpr int kMaxPasses = 4;
constexpr int kFftThreads = 256;
constexpr int kTwLoBits = 11;
constexpr int kTwStep = 16;     // rows between two exact inter-pass twiddle anchors   // two-level inter-pass twiddle table: 2^11 "lo" entries

struct PassDev {
    int R, S, ncols;          // transform length, element stride, number of columns (= n / R)
    int C, log2C;             // columns per tile (power of two)
    int contiguous;           // S == 1
    int nstages;
    int radix[kMaxStages];
    FastDiv divM[kMaxStages];     // M = L / r of each stage
    FastDiv divNbf[kMaxStages];   // R / r of each stage
    FastDiv divR, divTpo;
    const float2 *twR;            // w_R^e, e < R
    const uint16_t *perm;         // smem position of output k after the in-place DIF stages
    const float2 *tw_lo, *tw_hi;  // inter-pass twiddle w_L^e = tw_lo[e & mask] * tw_hi[e >> bits]
    int tw_mode;                  // applied on store: 0 none, 1 forward e = k*m, 2 inverse e = ko*(k*S + m)
    int ko_R;                     // inverse: length of the pass that runs next (ko = o % ko_R)
    int tiles_per_o;              // strided passes: ceil(S / C) tiles per outer index
    int load_mode;                // 0 functor (LDG), 1 TMA tensor tile (strided), 2 TMA bulk copy (contiguous)
    int rbox, nbox;               // TMA box rows / boxes per tile
    int nthreads;
    int smem_bytes;
    int ntiles;
    char tag[16];                 // "fft_fwd_0", "fft_inv_2", ... (stage timing label)
    // specialised two-stage kernel (fft_fast.cuh) for strided passes with R = fast_R1 * fast_R2; 0 = none
    int fast_R1, fast_R2;
    int fast_tiles_per_o, fast_ntiles;
    FastDiv fast_divTpo;
};

// ----------------------------- load / store functors -----------------------
struct LoadComplex {
    const float2 *src;
    size_t bstride;
    int conj;
    // a plain (unconjugated) complex load can be replaced by a TMA tile copy
    bool tma_source(const float2 **base, size_t *stride) const {
        *base = src;
        *stride = bstride;
        return conj == 0;
    }
    __device__ __forceinline__ float2 operator()(size_t i, int b) const {
        float2 v = __ldg(src + (size_t)b * bstride + i);
        if (conj) v.y = -v.y;
        return v;
    }
};
struct LoadReal {
    const float *src;
    size_t bstride;
    size_t n_valid;   // elements >= n_valid read as zero (zero padding)
    bool tma_source(const float2 **, size_t *) const { return false; }
    __device__ __forceinline__ float2 operator()(size_t i, int b) const {
        return make_float2(i < n_valid ? __ldg(src + (size_t)b * bstride + i) : 0.f, 0.f);
    }
};

struct NoSide {};   // store functors without a side input

struct StoreComplex {
    float2 *dst;
    size_t bstride;
    float scale;
    int conj;
    using Side = NoSide;
    __device__ __forceinline__ Side side_load(size_t, int) const { return Side{}; }
    __device__ __forceinline__ int column_aux(int) const { return 0; }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int, int, Side = Side{}) const {
        v.x *= scale;
        v.y *= conj ? -scale : scale;
        dst[(size_t)b * bstride + i] = v;
    }
};

// position -> frequency for the LAST forward pass (stride 1): the column index o
// encodes the digits k_0..k_{P-2} (most significant first); k = rev(o) + ncols*k_last.
struct OuterDigits {
    int nouter;
    int Rout[kMaxPasses];
    __device__ __forceinline__ int rev(int o) const {
        int d[kMaxPasses];
#pragma unroll
        for (int i = kMaxPasses - 1; i >= 0; --i)
            if (i < nouter) {
                d[i] = o % Rout[i];
                o /= Rout[i];
            }
        int k = 0, mult = 1;
#pragma unroll
        for (int i = 0; i < kMaxPasses; ++i)
            if (i < nouter) {
                k += d[i] * mult;
                mult *= Rout[i];
            }
        return k;
    }
};

// scipy.signal.hilbert's spectral mask (wefax.py:174), the 1/n of the inverse
// transform and the conjugation that lets the inverse reuse the forward kernels.
struct StoreHilbert {
    float2 *dst;
    size_t bstride;
    OuterDigits od;
    uint32_t n;
    int ncols;
    float inv_n;
    using Side = NoSide;
    __device__ __forceinline__ Side side_load(size_t, int) const { return Side{}; }
    __device__ __forceinline__ int column_aux(int col) const { return od.rev(col); }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int k, int aux, Side = Side{}) const {
        uint32_t kf = (uint32_t)aux + (uint32_t)ncols * (uint32_t)k;
        uint64_t k2 = 2ull * kf;
        float h = kf == 0 ? 1.f : (k2 < n ? 2.f : (k2 == n ? 1.f : 0.f));
        h *= inv_n;
        dst[(size_t)b * bstride + i] = make_float2(v.x * h, -v.y * h);
    }
};

// |z| of the analytic signal (numpy.abs in wefax.py:175), only the first n_valid
struct StoreAbs {
    float *dst;
    size_t bstride;
    size_t n_valid;
    float scale;
    using Side = NoSide;
    __device__ __forceinline__ Side side_load(size_t, int) const { return Side{}; }
    __device__ __forceinline__ int column_aux(int) const { return 0; }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int, int, Side = Side{}) const {
        if (i < n_valid) dst[(size_t)b * bstride + i] = scale * sqrtf(fmaf(v.x, v.x, v.y * v.y));
    }
};

// Real-input path: the last inverse pass yields conj(y[2m] + i*y[2m+1]) with y the
// Hilbert transform of x; the envelope is sqrt(x^2 + y^2) for the sample pair (2m, 2m+1).
struct StoreEnvPairs {
    float2 *env;            // envelope viewed as pairs
    const float2 *x;        // the real input viewed as pairs
    size_t ebstride, xbstride;
    int want_y = 0;         // 1: store the Hilbert transform y itself (FM discriminator, csrc/fm.cu) instead of |x + iy|
    using Side = float2;    // the x pair, fetched a few iterations ahead of its use
    __device__ __forceinline__ Side side_load(size_t i, int b) const { return __ldg(x + (size_t)b * xbstride + i); }
    __device__ __forceinline__ int column_aux(int) const { return 0; }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int, int, Side xs) const {
        env[(size_t)b * ebstride + i] =
            want_y ? make_float2(v.x, -v.y)
                   : make_float2(sqrtf(fmaf(xs.x, xs.x, v.x * v.x)), sqrtf(fmaf(xs.y, xs.y, v.y * v.y)));
    }
};

struct StoreRealPart {
    float *dst;
    size_t bstride;
    size_t n_valid;
    float scale;
    using Side = NoSide;
    __device__ __forceinline__ Side side_load(size_t, int) const { return Side{}; }
    __device__ __forceinline__ int column_aux(int) const { return 0; }
    __device__ __forceinline__ void operator()(size_t i, int b, float2 v, int, int, Side = Side{}) const {
        if (i < n_valid) dst[(size_t)b * bstride + i] = scale * v.x;
    }
};

// ----------------------------- butterflies ---------------------------------
template <int r> struct Bfly;

template <> struct Bfly<2> {
    __device__ __forceinline__ static void run(float2 *v, const float2 *) {
        float2 a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    }
};
template <> struct Bfly<4> {
    __device__ __forceinline__ static void run(float2 *v, const float2 *) {
        float2 t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
        float2 t2 = cadd(v[1], v[3]), t3 = csub(v[1], v[3]);
        v[0] = cadd(t0, t2);
        v[2] = csub(t0, t2);
        v[1] = make_float2(t1.x + t3.y, t1.y - t3.x);
        v[3] = make_float2(t1.x - t3.y, t1.y + t3.x);
    }
};
template <> struct Bfly<8> {
    __device__ __forceinline__ static void run(float2 *v, const float2 *) {
        float2 e[4] = {v[0], v[2], v[4], v[6]};
        float2 o[4] = {v[1], v[3], v[5], v[7]};
        Bfly<4>::run(e, nullptr);
        Bfly<4>::run(o, nullptr);
        const float h = 0.70710678118654752440f;
        float2 o1 = make_float2(h * (o[1].x + o[1].y), h * (o[1].y - o[1].x));    // * (1-i)/sqrt2
        float2 o2 = make_float2(o[2].y, -o[2].x);                                  // * -i
        float2 o3 = make_float2(h * (o[3].y - o[3].x), -h * (o[3].x + o[3].y));   // * (-1-i)/sqrt2
        v[0] = cadd(e[0], o[0]);
        v[4] = csub(e[0], o[0]);
        v[1] = cadd(e[1], o1);
        v[5] = csub(e[1], o1);
        v[2] = cadd(e[2], o2);
        v[6] = csub(e[2], o2);
        v[3] = cadd(e[3], o3);
        v[7] = csub(e[3], o3);
    }
};
// odd prime radix: pair (t, r-t); cs[j] = (cos, sin)(2*pi*(j+1)/r)
template <int r> struct Bfly {
    static constexpr int h = (r - 1) / 2;
    __device__ __forceinline__ static void run(float2 *v, const float2 *cs) {
        float2 a[h], b[h];
#pragma unroll
        for (int t = 1; t <= h; ++t) {
            a[t - 1] = cadd(v[t], v[r - t]);
            b[t - 1] = csub(v[t], v[r - t]);
        }
        float2 v0 = v[0];
        float2 s = v0;
#pragma unroll
        for (int t = 0; t < h; ++t) s = cadd(s, a[t]);
        v[0] = s;
#pragma unroll
        for (int u = 1; u <= h; ++u) {
            float2 p = v0, q = make_float2(0.f, 0.f);
#pragma unroll
            for (int t = 1; t <= h; ++t) {
                int j = (t * u) % r;
                float c = j <= h ? cs[j - 1].x : cs[r - j - 1].x;
                float sn = j <= h ? cs[j - 1].y : -cs[r - j - 1].y;
                p.x = fmaf(c, a[t - 1].x, p.x);
                p.y = fmaf(c, a[t - 1].y, p.y);
                q.x = fmaf(sn, b[t - 1].x, q.x);
                q.y = fmaf(sn, b[t - 1].y, q.y);
            }
            v[u] = make_float2(p.x + q.y, p.y - q.x);
            v[r - u] = make_float2(p.x - q.y, p.y + q.x);
        }
    }
};

// Length-(A*B) DFT held in registers: B radix-A butterflies over stride B, the
// inner twiddles w_{AB}^{t_b*u_a} (from the w_R table), then A radix-B butterflies.
// Output u = u_a + A*u_b ends up in v[u_a*B + u_b].
template <int A, int B> struct Composite {
    static constexpr int r = A * B;
    __device__ __forceinline__ static void run(float2 *v, const float2 *twR, int tw_stride, const float2 *csA,
                                               const float2 *csB) {
        if constexpr (B == 1) {
            Bfly<A>::run(v, csA);
        } else {
#pragma unroll
        for (int tb = 0; tb < B; ++tb) {
            float2 x[A];
#pragma unroll
            for (int ta = 0; ta < A; ++ta) x[ta] = v[ta * B + tb];
            Bfly<A>::run(x, csA);
#pragma unroll
            for (int ua = 0; ua < A; ++ua) v[ua * B + tb] = x[ua];
        }
#pragma unroll
        for (int ua = 1; ua < A; ++ua)
#pragma unroll
            for (int tb = 1; tb < B; ++tb) v[ua * B + tb] = cmul(v[ua * B + tb], twR[(ua * tb) * tw_stride]);
#pragma unroll
        for (int ua = 0; ua < A; ++ua) Bfly<B>::run(&v[ua * B], csB);
        }
    }
};

template <int r> __device__ __forceinline__ void load_cs(float2 *cs, const float2 *twR, int R) {
    if constexpr ((r & 1) && r > 1) {
#pragma unroll
        for (int j = 1; j <= (r - 1) / 2; ++j) {
            float2 w = twR[j * (R / r)];
            cs[j - 1] = make_float2(w.x, -w.y);
        }
    }
}

// One in-place DIF stage of radix A*B over the whole tile: each thread takes A*B
// elements spaced M = L/(A*B) apart into registers, transforms them, applies the
// stage twiddles w_L^{q*u} and writes them back to the same places.
template <int A, int B>
__device__ __forceinline__ void dif_stage(float2 *tile, const float2 *twR, const PassDev &p, int s, int L) {
    constexpr int r = A * B;
    const int M = L / r;
    const int nb = p.R / L;
    const int nbf = p.R / r;
    const int total = nbf * p.C;
    float2 csA[(A - 1) / 2 + 1], csB[(B - 1) / 2 + 1];
    load_cs<A>(csA, twR, p.R);
    load_cs<B>(csB, twR, p.R);
    const int tw_stride = p.R / r;
    for (int b = threadIdx.x; b < total; b += blockDim.x) {
        int cc, qp, base, step;
        if (p.contiguous) {
            cc = p.divNbf[s].div(b);
            qp = b - cc * nbf;
        } else {
            cc = b & (p.C - 1);
            qp = b >> p.log2C;
        }
        const int blk = p.divM[s].div(qp);
        const int q = qp - blk * M;
        const int j0 = blk * L + q;
        if (p.contiguous) {
            base = cc * p.R + j0;
            step = M;
        } else {
            base = j0 * p.C + cc;
            step = M * p.C;
        }
        float2 v[r];
#pragma unroll
        for (int t = 0; t < r; ++t) v[t] = tile[base + t * step];
        Composite<A, B>::run(v, twR, tw_stride, csA, csB);
        const int e1 = q * nb;
#pragma unroll
        for (int ua = 0; ua < A; ++ua)
#pragma unroll
            for (int ub = 0; ub < B; ++ub) {
                const int u = ua + A * ub;
                float2 x = v[ua * B + ub];
                if (M > 1 && u > 0) x = cmul(x, twR[e1 * u]);
                tile[base + u * step] = x;
            }
    }
}

__device__ __forceinline__ float2 pass_twiddle(const PassDev &p, uint32_t e) {
    float2 lo = __ldg(p.tw_lo + (e & ((1u << kTwLoBits) - 1)));
    float2 hi = __ldg(p.tw_hi + (e >> kTwLoBits));
    return cmul(lo, hi);
}

// ---- TMA / mbarrier primitives (sm_90+ PTX; SASS: UTMALDG / UBLKCP / SYNCS) -------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_bulk(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// One pass over one tile.  Global memory is touched once per element: the tile comes
// in through TMA (one tensor box per <=256 rows for strided passes, one bulk copy for
// the stride-1 pass) or, for fused prologues, through the load functor; it leaves
// through coalesced stores with the inter-pass twiddle and the store functor applied.
// MINB = CTAs per SM the register allocation aims for: 3 when the tile is small enough for
// three CTAs to share an SM (a few spills, better latency hiding), else 2.
template <class LoadOp, class StoreOp, int MINB>
__global__ void __launch_bounds__(kFftThreads, MINB)
fft_pass_kernel(const PassDev p, const LoadOp ld, const StoreOp st, const __grid_constant__ CUtensorMap tmap,
                const float2 *bulk_src, size_t bulk_bstride) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float2 *tile = reinterpret_cast<float2 *>(smem_raw);
    float2 *twR = tile + (size_t)p.C * p.R;
    uint16_t *perm = reinterpret_cast<uint16_t *>(twR + p.R);
    int *aux = reinterpret_cast<int *>(perm + ((p.R + 1) & ~1));
    int *aux2 = aux + p.C;
    uint64_t *mbar = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(aux2 + p.C) + 7) & ~uintptr_t(7));
    // inter-pass twiddles of this tile, factored as anchor[k / 16] * step[k % 16] per column / row
    float2 *twA = reinterpret_cast<float2 *>(mbar + 2);
    const int NA = (p.R + kTwStep - 1) / kTwStep;
    float2 *twS = twA + p.C * NA;

    const int tid = threadIdx.x, nt = blockDim.x;
    const int batch = blockIdx.y;

    // tile geometry
    int o, m0, c0;                       // strided: outer index and first column offset; contiguous: first row
    if (p.contiguous) {
        c0 = blockIdx.x * p.C;
        o = 0;
        m0 = 0;
    } else {
        o = p.divTpo.div(blockIdx.x);
        m0 = (blockIdx.x - o * p.tiles_per_o) * p.C;
        c0 = 0;
    }
    const int rows_valid = p.contiguous ? min(p.C, p.ncols - c0) : 0;

    if (p.load_mode != 0 && tid == 0) {
        mbar_init(mbar, 1);
    }
    if (p.load_mode != 0) __syncthreads();
    if (p.load_mode == 1 && tid == 0) {
        mbar_expect_tx(mbar, (uint32_t)(p.R * p.C * sizeof(float2)));
        for (int b = 0; b < p.nbox; ++b)
            tma_load_4d(tile + (size_t)b * p.rbox * p.C, &tmap, mbar, 2 * m0, b * p.rbox, o, batch);
    } else if (p.load_mode == 2 && tid == 0) {
        const uint32_t bytes = (uint32_t)(rows_valid * p.R * sizeof(float2));
        mbar_expect_tx(mbar, bytes);
        tma_load_bulk(tile, bulk_src + (size_t)batch * bulk_bstride + (size_t)c0 * p.R, bytes, mbar);
    }

    for (int i = tid; i < p.R; i += nt) {
        twR[i] = __ldg(p.twR + i);
        perm[i] = __ldg(p.perm + i);
    }
    // per-column constants: store-functor aux, inter-pass twiddle exponent e = e0 + k*de
    const int cc_s = tid & (p.C - 1);
    const uint32_t m_s = (uint32_t)(m0 + cc_s);
    const bool valid_s = !p.contiguous && m_s < (uint32_t)p.S;
    const size_t cbase = (size_t)o * (size_t)p.R * (size_t)p.S + m_s;
    const int jstep = nt >> p.log2C;
    uint32_t tw_e0 = 0, tw_de = 0;
    if (!p.contiguous) {
        if (p.tw_mode == 1) {
            tw_de = m_s;
        } else if (p.tw_mode == 2) {
            const uint32_t ko = (uint32_t)o % (uint32_t)p.ko_R;
            tw_e0 = ko * m_s;
            tw_de = ko * (uint32_t)p.S;
        }
    }
    if (tid < p.C) {
        const int col = p.contiguous ? c0 + tid : o * p.S + m0 + tid;
        const bool ok = p.contiguous ? (tid < rows_valid) : (m0 + tid < p.S);
        aux[tid] = ok ? st.column_aux(col) : 0;
        aux2[tid] = (p.contiguous && p.tw_mode == 2) ? (c0 + tid) % p.ko_R : 0;
    }

    if (p.tw_mode != 0) {
        // exact two-level lookups once per (column, anchor) and (column, step) while the tile is in flight
        if (p.contiguous) __syncthreads();   // aux2 (ko per row) is needed below
        const int total = p.C * (NA + kTwStep);
        for (int idx = tid; idx < total; idx += nt) {
            int cc, x;
            uint32_t e0, de;
            if (p.contiguous) {               // layout [cc][x]; e = ko * k
                cc = idx / (NA + kTwStep);
                x = idx - cc * (NA + kTwStep);
                e0 = 0;
                de = (uint32_t)aux2[cc];
            } else {                          // layout [x][cc]; e = e0 + k * de of column cc
                x = idx >> p.log2C;
                cc = idx & (p.C - 1);
                const uint32_t m = (uint32_t)(m0 + cc);
                if (p.tw_mode == 1) {
                    e0 = 0;
                    de = m;
                } else {
                    const uint32_t ko = (uint32_t)o % (uint32_t)p.ko_R;
                    e0 = ko * m;
                    de = ko * (uint32_t)p.S;
                }
                if (m >= (uint32_t)p.S) e0 = de = 0;   // padding column
            }
            const bool anchor = x < NA;
            const uint32_t e = anchor ? e0 + (uint32_t)(x * kTwStep) * de : (uint32_t)(x - NA) * de;
            const float2 w = pass_twiddle(p, e);
            if (p.contiguous)
                (anchor ? twA[cc * NA + x] : twS[cc * kTwStep + (x - NA)]) = w;
            else
                (anchor ? twA[x * p.C + cc] : twS[(x - NA) * p.C + cc]) = w;
        }
    }

    const int tile_elems = p.C * p.R;
    if (p.load_mode == 0) {
        if (p.contiguous) {
            const size_t gbase = (size_t)c0 * p.R;
            const int nvalid = rows_valid * p.R;
#pragma unroll 8
            for (int e = tid; e < tile_elems; e += nt)
                tile[e] = e < nvalid ? ld(gbase + e, batch) : make_float2(0.f, 0.f);
        } else {
#pragma unroll 8
            for (int j = tid >> p.log2C; j < p.R; j += jstep)
                tile[j * p.C + cc_s] = valid_s ? ld(cbase + (size_t)j * p.S, batch) : make_float2(0.f, 0.f);
        }
        __syncthreads();
    } else {
        __syncthreads();          // tables visible to everyone
        mbar_wait(mbar, 0);       // tile has landed (async proxy writes are visible after the wait)
    }

    int L = p.R;
    for (int s = 0; s < p.nstages; ++s) {
        const int r = p.radix[s];
        switch (r) {
            case 2: dif_stage<2, 1>(tile, twR, p, s, L); break;
            case 3: dif_stage<3, 1>(tile, twR, p, s, L); break;
            case 4: dif_stage<4, 1>(tile, twR, p, s, L); break;
            case 5: dif_stage<5, 1>(tile, twR, p, s, L); break;
            case 7: dif_stage<7, 1>(tile, twR, p, s, L); break;
            case 8: dif_stage<8, 1>(tile, twR, p, s, L); break;
            case 11: dif_stage<11, 1>(tile, twR, p, s, L); break;
            case 13: dif_stage<13, 1>(tile, twR, p, s, L); break;
            case 6: dif_stage<2, 3>(tile, twR, p, s, L); break;
            case 9: dif_stage<3, 3>(tile, twR, p, s, L); break;
            case 10: dif_stage<2, 5>(tile, twR, p, s, L); break;
            case 12: dif_stage<4, 3>(tile, twR, p, s, L); break;
            case 14: dif_stage<2, 7>(tile, twR, p, s, L); break;
            case 15: dif_stage<3, 5>(tile, twR, p, s, L); break;
            case 16: dif_stage<4, 4>(tile, twR, p, s, L); break;
            case 20: dif_stage<4, 5>(tile, twR, p, s, L); break;
            case 21: dif_stage<3, 7>(tile, twR, p, s, L); break;
            case 24: dif_stage<8, 3>(tile, twR, p, s, L); break;
            case 25: dif_stage<5, 5>(tile, twR, p, s, L); break;
            case 28: dif_stage<4, 7>(tile, twR, p, s, L); break;
            default: dif_stage<8, 4>(tile, twR, p, s, L); break;   // 32
        }
        L /= r;
        __syncthreads();
    }

    // Functors with a side input (e.g. the x pair of the envelope store) get their side
    // loads of SU elements requested before any is used; the others keep the plain loop.
    constexpr bool kHasSide = !std::is_empty<typename StoreOp::Side>::value;
    constexpr int SU = kHasSide ? 8 : 1;
    if (p.contiguous) {
        const size_t gbase = (size_t)c0 * p.R;
        const int nvalid = rows_valid * p.R;
#pragma unroll(kHasSide ? 1 : 4)
        for (int e0 = tid; e0 < nvalid; e0 += SU * nt) {
            typename StoreOp::Side side[SU];
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int e = e0 + u * nt;
                if (e < nvalid) side[u] = st.side_load(gbase + e, batch);
            }
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int e = e0 + u * nt;
                if (e < nvalid) {
                    const int cc = p.divR.div(e);
                    const int k = e - cc * p.R;
                    float2 v = tile[cc * p.R + perm[k]];
                    if (p.tw_mode == 2)
                        v = cmul(v, cmul(twA[cc * NA + (k >> 4)], twS[cc * kTwStep + (k & (kTwStep - 1))]));
                    st(gbase + e, batch, v, k, aux[cc], side[u]);
                }
            }
        }
    } else if (valid_s) {
        const int a = aux[cc_s];
#pragma unroll(kHasSide ? 1 : 4)
        for (int k0 = tid >> p.log2C; k0 < p.R; k0 += SU * jstep) {
            typename StoreOp::Side side[SU];
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int k = k0 + u * jstep;
                if (k < p.R) side[u] = st.side_load(cbase + (size_t)k * p.S, batch);
            }
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int k = k0 + u * jstep;
                if (k < p.R) {
                    float2 v = tile[(int)perm[k] * p.C + cc_s];
                    if (p.tw_mode != 0)
                        v = cmul(v, cmul(twA[(k >> 4) * p.C + cc_s], twS[(k & (kTwStep - 1)) * p.C + cc_s]));
                    st(cbase + (size_t)k * p.S, batch, v, k, a, side[u]);
                }
            }
        }
    }
}

// ----------------------------- host-side plan ------------------------------
struct FftPlan {
    long long n = 0;
    int npass = 0;
    int Rs[kMaxPasses] = {0, 0, 0, 0};
    long long S[kMaxPasses] = {0, 0, 0, 0};
    PassDev fwd[kMaxPasses];   // tw_mode 1 on all but the last pass
    PassDev inv[kMaxPasses];   // tw_mode 2 on all but pass 0 (the last one to run)
    DevBuf tables;             // twR / perm / tw_lo / tw_hi of every pass
    const float2 *tw2_lo = nullptr, *tw2_hi = nullptr;   // w_{2n}^e (real-input packing), two-level like tw_lo/hi
    // fused "last forward pass + pair untangling + first inverse pass" (fft_mid.cuh): row pairs and w_{2R}^j
    DevBuf mid_tab;
    int mid_npairs = 0;
    OuterDigits outer() const {
        OuterDigits od{};
        od.nouter = npass - 1;
        for (int i = 0; i < npass - 1; ++i) od.Rout[i] = Rs[i];
        return od;
    }
};

// Factor n into pass lengths; returns false when n has a prime factor > 13 or no
// feasible split exists (the caller then uses Bluestein).
bool plan_factors(long long n, std::vector<int> &Rs);
// smallest 2^a 3^b 5^c 7^d >= m that plan_factors accepts
long long next_smooth_length(long long m);
std::unique_ptr<FftPlan> make_plan(long long n, cudaStream_t stream);
// Chooses how a pass reads its tile from `base` (see PassDev::load_mode) and, for
// strided passes, encodes the 4-D tensor map {2S floats, R, outer, batch}.
int choose_load_mode(const PassDev &p, const float2 *base, size_t bstride, int batch, CUtensorMap *map);
bool encode_strided_map(const PassDev &p, const float2 *base, size_t bstride, int batch, int cols, int rbox,
                        CUtensorMap *map);

}  // namespace wefax
