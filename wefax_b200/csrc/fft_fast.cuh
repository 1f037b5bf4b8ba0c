// Specialised two-stage strided FFT pass: compile-time pass length R = R1 * R2.
//
// The generic pass kernel (fft.cuh) is instruction-bound: ~120 thread instructions per
// point per pass (run-time radices, strides and divisions; three shared-memory round
// trips; a separate read-out loop).  For the strided passes of the long transforms on the
// decode path this kernel does the same arithmetic with everything but the global stride
// known at compile time:
//
//   stage 1  thread (q, cc): R1 rows  q + R2*t  of column cc straight from global memory
//            into registers (two 128-byte row segments per warp), length-R1 DFT in
//            registers (prime-factor / constant-twiddle codelets, no table look-ups),
//            stage twiddles w_R^(q*u) from a [q][u] table at immediate offsets, one
//            shared-memory write;
//   stage 2  thread (u, cc): the R2 contiguous rows of block u from shared memory, length-R2
//            DFT in registers, inter-pass twiddle, and the store functor straight from
//            registers (row k = u + R1*k2, again 128-byte segments per row).
//
// One shared-memory round trip, one __syncthreads per tile (double-buffered tile), persistent
// CTAs striding over the tiles.  The inter-pass twiddle w^(e0 + k*de) of row k = u + R1*k2
// is A[u] * P[k2] with A = w^(e0 + u*de) (one exact two-level look-up per thread) and
// P[k2] = w^(k2*R1*de) (one look-up per thread, shared through the tile buffer).
//
// Output convention, tables and twiddle exponents are those of fft_pass_kernel with stage
// radices {R1, R2}; a plan may mix both kernels freely.
#pragma once

#include "fft.cuh"

// Tile-shape knobs of the strided pass.  Defaults are the measured best on B200 for the 60-min recording
// (us per plain pass / last inverse pass):  C=16 NBUF=2: 78 / 105   C=32 NBUF=1: 72 / 101 (default)
// C=32 NBUF=2 (one CTA per SM): 100 / 120   C=16 H=2 NBUF=1: 86 / 237 (spills)
#ifndef WEFAX_FAST_NBUF
#define WEFAX_FAST_NBUF 1   // exchange-tile buffers: 2 = one barrier per tile, 1 = two barriers, half the memory
#endif
#ifndef WEFAX_FAST_H
#define WEFAX_FAST_H 1      // column groups per thread
#endif
#ifndef WEFAX_FAST_C
#define WEFAX_FAST_C 32     // adjacent columns per thread group: 32 = 256-byte row segments
#endif

namespace wefax {
namespace fast {

// ----------------------------- packed fp32 arithmetic ------------------------
// Blackwell issues two fp32 operations per instruction on a 64-bit register pair (SASS FADD2 /
// FMUL2 / FFMA2; PTX add/mul/fma.rn.f32x2) and can swap or negate the halves of an operand for
// free.  A complex number is exactly such a pair, so complex add/sub cost one instruction, a
// real-constant scale-and-accumulate one, and a complex multiply two (w given as (wx, wx) and
// (-wy, wy)) or three (w given as (wx, wy)) instead of two, two and four.  Same IEEE roundings as
// the scalar forms (no contraction beyond the explicit fma).
#ifndef WEFAX_FAST_PACKED
#define WEFAX_FAST_PACKED 1   // 0: the same formulas on scalar FADD / FMUL / FFMA (A/B measurements)
#endif
#if WEFAX_FAST_PACKED
#define WEFAX_P2(op)                                                                                          \
    __device__ __forceinline__ float2 p##op(float2 a, float2 b) {                                             \
        float2 r;                                                                                             \
        asm("{.reg .b64 ta, tb, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%5}; " #op                           \
            ".rn.f32x2 tr, ta, tb; mov.b64 {%0,%1}, tr;}"                                                      \
            : "=f"(r.x), "=f"(r.y)                                                                            \
            : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                                        \
        return r;                                                                                             \
    }
WEFAX_P2(add)
WEFAX_P2(sub)
WEFAX_P2(mul)
#undef WEFAX_P2
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c) {
    float2 r;
    asm("{.reg .b64 ta, tb, tc, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%5}; mov.b64 tc, {%6,%7}; "
        "fma.rn.f32x2 tr, ta, tb, tc; mov.b64 {%0,%1}, tr;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return r;
}
#else
__device__ __forceinline__ float2 padd(float2 a, float2 b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
__device__ __forceinline__ float2 psub(float2 a, float2 b) { return make_float2(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y)); }
__device__ __forceinline__ float2 pmul(float2 a, float2 b) { return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c) {
    return make_float2(__fmaf_rn(a.x, b.x, c.x), __fmaf_rn(a.y, b.y, c.y));
}
#endif
__device__ __forceinline__ float2 swp(float2 a) { return make_float2(a.y, a.x); }
__device__ __forceinline__ float2 bc(float c) { return make_float2(c, c); }
// v * w with w = (wx, wy) given as wa = (wx, wx), wb = (-wy, wy)
__device__ __forceinline__ float2 pcmul2(float2 v, float2 wa, float2 wb) { return pfma(v, wa, pmul(swp(v), wb)); }
// v * w with w = (wx, wy) as stored: wx*v + wy*(-v.y, v.x)
__device__ __forceinline__ float2 pcmul3(float2 v, float2 w) {
    return pfma(v, bc(w.x), pmul(bc(w.y), pmul(swp(v), make_float2(-1.f, 1.f))));
}
// v * (cx + i*cy) for literal cx, cy
__device__ __forceinline__ float2 pcmulc(float2 v, float cx, float cy) {
    return pfma(v, bc(cx), pmul(swp(v), make_float2(-cy, cy)));
}

// ----------------------------- codelets -------------------------------------
// In-register butterflies, natural order in and out, X_u = sum_t x_t exp(-2*pi*i*t*u/r).
template <int r> struct Cs;
template <> struct Cs<2> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float2 a = v[0], b = v[1];
        v[0] = padd(a, b);
        v[1] = psub(a, b);
    }
};
template <> struct Cs<4> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float2 t0 = padd(v[0], v[2]), t1 = psub(v[0], v[2]);
        const float2 t2 = padd(v[1], v[3]), t3 = swp(psub(v[1], v[3]));
        v[0] = padd(t0, t2);
        v[2] = psub(t0, t2);
        v[1] = pfma(make_float2(1.f, -1.f), t3, t1);    // t1 + (t3.y, -t3.x)
        v[3] = pfma(make_float2(-1.f, 1.f), t3, t1);
    }
};
// odd prime r: pair (t, r-t); CS[j-1] = (cos, sin)(2*pi*j/r)
template <int r> struct OddCs {
    static constexpr int h = (r - 1) / 2;
    __device__ __forceinline__ static void run(float2 *v, const float (&co)[h], const float (&si)[h]) {
        float2 a[h], b[h];
#pragma unroll
        for (int t = 1; t <= h; ++t) {
            a[t - 1] = padd(v[t], v[r - t]);
            b[t - 1] = swp(psub(v[t], v[r - t]));      // (d.y, d.x) of the difference d
        }
        const float2 v0 = v[0];
        float2 s = v0;
#pragma unroll
        for (int t = 0; t < h; ++t) s = padd(s, a[t]);
        v[0] = s;
#pragma unroll
        for (int u = 1; u <= h; ++u) {
            float2 p = v0, q = make_float2(0.f, 0.f);
#pragma unroll
            for (int t = 1; t <= h; ++t) {
                const int j = (t * u) % r;
                const float c = j <= h ? co[j - 1] : co[r - j - 1];
                const float sn = j <= h ? si[j - 1] : -si[r - j - 1];
                p = pfma(bc(c), a[t - 1], p);
                // q = sum sn * (d.y, -d.x) = -i * sum sn * d
                q = t == 1 ? pmul(make_float2(sn, -sn), b[t - 1]) : pfma(make_float2(sn, -sn), b[t - 1], q);
            }
            v[u] = padd(p, q);
            v[r - u] = psub(p, q);
        }
    }
};
template <> struct Cs<3> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float co[1] = {-0.5f}, si[1] = {0.86602540378443865f};
        OddCs<3>::run(v, co, si);
    }
};
template <> struct Cs<5> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float co[2] = {0.30901699437494742f, -0.80901699437494742f};
        const float si[2] = {0.95105651629515357f, 0.58778525229247313f};
        OddCs<5>::run(v, co, si);
    }
};
template <> struct Cs<7> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float co[3] = {0.62348980185873353f, -0.22252093395631440f, -0.90096886790241913f};
        const float si[3] = {0.78183148246802981f, 0.97492791218182361f, 0.43388373911755812f};
        OddCs<7>::run(v, co, si);
    }
};

__host__ __device__ constexpr int mod_inverse(int a, int m) {
    for (int i = 1; i < m; ++i)
        if ((a * i) % m == 1) return i;
    return 1;
}

// Good-Thomas prime-factor DFT of length A*B (gcd(A, B) = 1): no inner twiddles, index
// maps resolved at compile time.  Natural order in, natural order out.
template <int A, int B> struct Pfa {
    static constexpr int N = A * B;
    __device__ __forceinline__ static void run(float2 *v) {
        float2 t[A][B];
#pragma unroll
        for (int n1 = 0; n1 < A; ++n1)
#pragma unroll
            for (int n2 = 0; n2 < B; ++n2) t[n1][n2] = v[(B * n1 + A * n2) % N];
#pragma unroll
        for (int n2 = 0; n2 < B; ++n2) {
            float2 x[A];
#pragma unroll
            for (int n1 = 0; n1 < A; ++n1) x[n1] = t[n1][n2];
            Cs<A>::run(x);
#pragma unroll
            for (int k1 = 0; k1 < A; ++k1) t[k1][n2] = x[k1];
        }
        static_assert(A > 1 && B > 1, "coprime factors");
        constexpr int ia = B * mod_inverse(B % A, A), ib = A * mod_inverse(A % B, B);
#pragma unroll
        for (int k1 = 0; k1 < A; ++k1) {
            Cs<B>::run(t[k1]);
#pragma unroll
            for (int k2 = 0; k2 < B; ++k2) v[(ia * k1 + ib * k2) % N] = t[k1][k2];
        }
    }
};

template <int N> struct Dft;
template <> struct Dft<7> {
    __device__ __forceinline__ static void run(float2 *v) { Cs<7>::run(v); }
};
template <> struct Dft<12> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<3, 4>::run(v); }
};
template <> struct Dft<14> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<2, 7>::run(v); }
};
template <> struct Dft<15> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<3, 5>::run(v); }
};
// 16 = 4 x 4 Cooley-Tukey with literal twiddles w16^e = exp(-2*pi*i*e/16)
template <> struct Dft<16> {
    __device__ __forceinline__ static void run(float2 *v) {
        const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, h = 0.70710678118654752f;
        float2 t[4][4];   // t[ua][tb]
#pragma unroll
        for (int tb = 0; tb < 4; ++tb) {
            float2 x[4] = {v[tb], v[4 + tb], v[8 + tb], v[12 + tb]};
            Cs<4>::run(x);
#pragma unroll
            for (int ua = 0; ua < 4; ++ua) t[ua][tb] = x[ua];
        }
        // inner twiddles w16^(ua*tb)
        t[1][1] = pcmulc(t[1][1], c1, -s1);
        t[1][2] = pcmulc(t[1][2], h, -h);
        t[1][3] = pcmulc(t[1][3], s1, -c1);
        t[2][1] = pcmulc(t[2][1], h, -h);
        t[2][2] = pmul(swp(t[2][2]), make_float2(1.f, -1.f));   // w16^4 = -i
        t[2][3] = pcmulc(t[2][3], -h, -h);
        t[3][1] = pcmulc(t[3][1], s1, -c1);
        t[3][2] = pcmulc(t[3][2], -h, -h);
        t[3][3] = pcmulc(t[3][3], -c1, s1);
#pragma unroll
        for (int ua = 0; ua < 4; ++ua) {
            Cs<4>::run(t[ua]);
#pragma unroll
            for (int ub = 0; ub < 4; ++ub) v[ua + 4 * ub] = t[ua][ub];
        }
    }
};

// ----------------------------- the pass -------------------------------------
// A tile is R rows x (C*H) adjacent columns.  Thread (row, cc) owns columns cc + h*C, h < H: with H = 2
// the two 128-byte halves of a 256-byte row segment are requested back to back by the same warp, which is
// what the HBM controller needs to keep a mixed read+write stream near the copy rate
// (tools/strided_copy_bench.cu: 128-byte segments 3.5 TB/s, 256-byte segments 5.4 TB/s).
template <int R1, int R2, int C> struct Cfg {
    static constexpr int R = R1 * R2;
    static constexpr int H = WEFAX_FAST_H;
    static constexpr int CW = C * H;                                // columns per tile
    static constexpr int ROWS = R1 > R2 ? R1 : R2;
    static constexpr int T = ((ROWS * C + 31) / 32) * 32;
    static constexpr int BUF = R * CW + R2 * CW;                    // tile + P table, in float2
    static constexpr int NBUF = WEFAX_FAST_NBUF;                    // 2: one barrier per tile; 1: two barriers, half the memory
    static constexpr int SMEM = (R + NBUF * BUF) * (int)sizeof(float2);
    // CTAs per SM: shared memory, and a register budget of 64 * H per thread
    static constexpr int BY_SMEM = (227 * 1024) / (SMEM + 1024);
    static constexpr int BY_REGS = 1024 / (T * H);
    static constexpr int MINB_ = BY_SMEM < BY_REGS ? BY_SMEM : BY_REGS;
    static constexpr int MINB = MINB_ < 1 ? 1 : (MINB_ > 3 ? 3 : MINB_);
};

template <int R1, int R2, int C, class StoreOp>
__global__ void __launch_bounds__((Cfg<R1, R2, C>::T), (Cfg<R1, R2, C>::MINB))
fft_fast_strided_kernel(const PassDev p, const float2 *src, size_t src_bstride, const StoreOp st, int total_tiles) {
    using K = Cfg<R1, R2, C>;
    constexpr int R = K::R, H = K::H, CW = K::CW;
    extern __shared__ __align__(16) unsigned char fast_smem[];
    // tables stay plain (wx, wy): a 16-byte (wx, wx, -wy, wy) layout would make the multiply two instructions
    // instead of three but doubles the shared-memory traffic of the twiddles, which costs more (measured)
    float2 *twQ = reinterpret_cast<float2 *>(fast_smem);   // [q][u] stage twiddles w_R^(q*u)
    float2 *buf0 = twQ + R;

    const int tid = threadIdx.x;
    const int cc = tid % C, row = tid / C;                 // row = q in stage 1, = u in stage 2
    for (int i = tid; i < R; i += K::T) {
        const int q = i / R1, u = i - q * R1;
        twQ[i] = __ldg(p.twR + q * u);
    }
    __syncthreads();
    const bool act1 = row < R2, act2 = row < R1;
    const size_t rstride = (size_t)p.S;
    constexpr bool kHasSide = !std::is_empty<typename StoreOp::Side>::value;

    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        float2 *tb = buf0 + (K::NBUF == 2 ? (it & 1) * K::BUF : 0);
        float2 *P = tb + R * CW;
        const int batch = tile / p.fast_ntiles;
        const int t_in = tile - batch * p.fast_ntiles;
        const int o = p.fast_divTpo.div(t_in);
        const uint32_t m0 = (uint32_t)((t_in - o * p.fast_tiles_per_o) * CW + cc);
        const size_t obase = (size_t)o * (size_t)R * rstride;
        bool colok[H];
        float2 Pval[H], Aval[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const uint32_t m = m0 + h * C;
            colok[h] = m < (uint32_t)p.S;
            // inter-pass twiddle factors of this thread (exact two-level look-ups, in flight with the data)
            uint32_t e0 = 0, de = 0;
            if (p.tw_mode == 1) {
                de = m;
            } else if (p.tw_mode == 2) {
                const uint32_t ko = (uint32_t)o % (uint32_t)p.ko_R;
                e0 = ko * m;
                de = ko * (uint32_t)p.S;
            }
            if (!colok[h]) e0 = de = 0;
            Pval[h] = Aval[h] = make_float2(1.f, 0.f);
            if (p.tw_mode != 0) {
                if (act1) Pval[h] = pass_twiddle(p, (uint32_t)(row * R1) * de);
                if (act2) Aval[h] = pass_twiddle(p, e0 + (uint32_t)row * de);
            }
        }

        float2 v[H][R1];
        if (act1) {
            const float2 *g = src + (size_t)batch * src_bstride + obase + m0 + (size_t)row * rstride;
#pragma unroll
            for (int t = 0; t < R1; ++t)
#pragma unroll
                for (int h = 0; h < H; ++h)
                    v[h][t] = colok[h] ? __ldg(g + (size_t)(R2 * t) * rstride + h * C) : make_float2(0.f, 0.f);
#pragma unroll
            for (int h = 0; h < H; ++h) Dft<R1>::run(v[h]);
        }
        if (K::NBUF == 1) __syncthreads();   // stage-2 readers of the previous tile are done with the buffer
        if (act1) {
            const float2 *tq = twQ + row * R1;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const int col = cc + h * C;
                if (p.tw_mode != 0) P[row * CW + col] = Pval[h];
                tb[row * CW + col] = v[h][0];
#pragma unroll
                for (int u = 1; u < R1; ++u) tb[(row + R2 * u) * CW + col] = pcmul3(v[h][u], tq[u]);
            }
        }
        __syncthreads();
        if (act2) {
            float2 y[H][R2];
            typename StoreOp::Side side[H][R2];
            if constexpr (kHasSide) {
#pragma unroll
                for (int k2 = 0; k2 < R2; ++k2)
#pragma unroll
                    for (int h = 0; h < H; ++h)
                        if (colok[h])
                            side[h][k2] = st.side_load(obase + m0 + h * C + (size_t)(row + R1 * k2) * rstride, batch);
            }
#pragma unroll
            for (int h = 0; h < H; ++h) {
#pragma unroll
                for (int t = 0; t < R2; ++t) y[h][t] = tb[(row * R2 + t) * CW + cc + h * C];
                Dft<R2>::run(y[h]);
            }
            float2 Aa[H], Ab[H];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                Aa[h] = bc(Aval[h].x);
                Ab[h] = make_float2(-Aval[h].y, Aval[h].y);
            }
#pragma unroll
            for (int k2 = 0; k2 < R2; ++k2) {
                const int k = row + R1 * k2;
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    if (!colok[h]) continue;
                    float2 val = y[h][k2];
                    if (p.tw_mode != 0) {
                        val = pcmul2(val, Aa[h], Ab[h]);
                        if (k2 > 0) val = pcmul3(val, P[k2 * CW + cc + h * C]);
                    }
                    st(obase + m0 + h * C + (size_t)k * rstride, batch, val, k, 0, side[h][k2]);
                }
            }
        }
    }
}

// ----------------------------- the pass, TMA-staged -----------------------------------------------------------------
// Same arithmetic, but the R x 32 tile travels by tensor TMA in both directions (256-byte row segments, no global-memory
// instructions or 64-bit address arithmetic in the workers' loop), and the copy engine runs two tiles ahead of the
// arithmetic.  Both register stages work IN PLACE on the tile buffer (stage 1 reads and writes the same rows of a
// column; stage 2 reads its R2 rows, meets the other workers at a barrier, and writes the permuted rows), so there is no
// exchange tile and the shared memory holds three tile buffers: one being computed, one landing, one leaving.  A 17th
// warp does nothing but drive the copy engine: it learns through an mbarrier that a tile is finished, stores it, waits
// (alone) until the store has read the buffer, and at once loads the tile three ahead into it.  The 16 worker warps
// never wait for a store and meet only each other (named barrier), twice a tile.  Plain complex in, plain complex out
// (scale 1, no conjugation): the strided passes that are not the envelope store.  One CTA of 544 threads per SM.
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap *map, const void *src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}

template <int R1, int R2> struct TmaCfg {
    static constexpr int R = R1 * R2;
    static constexpr int C = 32;
    static constexpr int T = 512;
    static constexpr int TILE = R * C;                               // float2 per tile buffer
    static constexpr int SMEM = (R + 3 * TILE + 2 * R2 * C) * (int)sizeof(float2) + 64 + 1024;   // + alignment slack
    static_assert(R1 <= 16 && R2 <= 16, "512 threads = 16 rows x 32 columns");
};

template <int R1, int R2>
__global__ void __launch_bounds__(512 + 32, 1)
fft_fast_tma3_kernel(const PassDev p, const __grid_constant__ CUtensorMap in_map, const __grid_constant__ CUtensorMap out_map,
                     int rbox, int total_tiles) {
    using K = TmaCfg<R1, R2>;
    constexpr int R = K::R, C = K::C;
    extern __shared__ unsigned char tma_smem_raw[];
    float2 *B0 = reinterpret_cast<float2 *>(tma_smem_raw + ((1024u - (smem_u32(tma_smem_raw) & 1023u)) & 1023u));
    float2 *P0 = B0 + 3 * K::TILE;             // [2][R2][C] inter-pass twiddle columns, double-buffered
    float2 *twQ = P0 + 2 * R2 * C;             // [q][u]
    uint64_t *full = reinterpret_cast<uint64_t *>(twQ + R);   // [3] tile landed
    uint64_t *done = full + 3;                                 // [3] tile computed

    const int tid = threadIdx.x;
    const int cc = tid % C, row = tid / C;
    for (int i = tid; i < R; i += K::T) {
        const int q = i / R1, u = i - q * R1;
        twQ[i] = __ldg(p.twR + q * u);
    }
    if (tid == 0) {
        for (int b = 0; b < 3; ++b) {
            mbar_init(full + b, 1);
            mbar_init(done + b, K::T / 32);
        }
    }
    __syncthreads();
    const int nt = (int)blockIdx.x < total_tiles ? (total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    constexpr uint32_t kTileBytes = (uint32_t)(K::TILE * sizeof(float2));
    const int nbox = R / rbox;
    auto tile_coords = [&](int k, int &batch, int &o, int &m0) {
        const int tile = blockIdx.x + k * gridDim.x;
        batch = tile / p.fast_ntiles;
        const int t_in = tile - batch * p.fast_ntiles;
        o = p.fast_divTpo.div(t_in);
        m0 = (t_in - o * p.fast_tiles_per_o) * C;
    };

    if (tid >= K::T) {
        // ---- the copy warp ------------------------------------------------------------------------------------------
        if (tid == K::T) {
            auto issue_load = [&](int k) {
                int batch, o, m0;
                tile_coords(k, batch, o, m0);
                float2 *dst = B0 + (size_t)(k % 3) * K::TILE;
                uint64_t *bar = full + (k % 3);
                mbar_expect_tx(bar, kTileBytes);
                for (int b = 0; b < nbox; ++b) tma_load_4d(dst + (size_t)b * rbox * C, &in_map, bar, 2 * m0, b * rbox, o, batch);
            };
            for (int k = 0; k < 3 && k < nt; ++k) issue_load(k);
            for (int k = 0; k < nt; ++k) {
                while (!mbar_try_wait(done + (k % 3), (uint32_t)((k / 3) & 1))) {
                }
                int batch, o, m0;
                tile_coords(k, batch, o, m0);
                const float2 *src = B0 + (size_t)(k % 3) * K::TILE;
                for (int b = 0; b < nbox; ++b) tma_store_4d(&out_map, src + (size_t)b * rbox * C, 2 * m0, b * rbox, o, batch);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                if (k + 3 < nt) {
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the buffer has been read out
                    issue_load(k + 3);
                }
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
        return;
    }

    // ---- the sixteen worker warps ---------------------------------------------------------------------------------------
    const bool act1 = row < R2, act2 = row < R1;
    for (int k = 0; k < nt; ++k) {
        float2 *A = B0 + (size_t)(k % 3) * K::TILE;
        float2 *P = P0 + (size_t)(k & 1) * R2 * C;
        int batch, o, m0;
        tile_coords(k, batch, o, m0);
        const uint32_t m = (uint32_t)(m0 + cc);
        const bool colok = m < (uint32_t)p.S;
        uint32_t e0 = 0, de = 0;
        if (p.tw_mode == 1) {
            de = m;
        } else if (p.tw_mode == 2) {
            const uint32_t ko = (uint32_t)o % (uint32_t)p.ko_R;
            e0 = ko * m;
            de = ko * (uint32_t)p.S;
        }
        if (!colok) e0 = de = 0;
        float2 Pval = make_float2(1.f, 0.f), Aval = make_float2(1.f, 0.f);
        if (p.tw_mode != 0) {
            if (act1) Pval = pass_twiddle(p, (uint32_t)(row * R1) * de);
            if (act2) Aval = pass_twiddle(p, e0 + (uint32_t)row * de);
        }
        while (!mbar_try_wait(full + (k % 3), (uint32_t)((k / 3) & 1))) {
        }
        if (act1) {
            float2 v[R1];
#pragma unroll
            for (int t = 0; t < R1; ++t) v[t] = A[(row + R2 * t) * C + cc];
            Dft<R1>::run(v);
            if (p.tw_mode != 0) P[row * C + cc] = Pval;
            const float2 *tq = twQ + row * R1;
            A[row * C + cc] = v[0];
#pragma unroll
            for (int u = 1; u < R1; ++u) A[(row + R2 * u) * C + cc] = pcmul3(v[u], tq[u]);   // the rows it read
        }
        asm volatile("bar.sync 1, 512;" ::: "memory");
        float2 y[R2];
        if (act2) {
#pragma unroll
            for (int t = 0; t < R2; ++t) y[t] = A[(row * R2 + t) * C + cc];
            Dft<R2>::run(y);
            const float2 Aa = bc(Aval.x), Ab = make_float2(-Aval.y, Aval.y);
#pragma unroll
            for (int k2 = 0; k2 < R2; ++k2) {
                if (p.tw_mode != 0) {
                    y[k2] = pcmul2(y[k2], Aa, Ab);
                    if (k2 > 0) y[k2] = pcmul3(y[k2], P[k2 * C + cc]);
                }
            }
        }
        asm volatile("bar.sync 1, 512;" ::: "memory");   // every block of rows has been read: they may be overwritten
        if (act2) {
#pragma unroll
            for (int k2 = 0; k2 < R2; ++k2) A[(row + R1 * k2) * C + cc] = y[k2];   // natural row order
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if ((tid & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(done + (k % 3))) : "memory");
    }
}

// (R1, R2) pairs with a compiled kernel; 0 when R has none
inline bool fast_pair(int R, int *R1, int *R2) {
    static const int pairs[][2] = {{15, 7},  {12, 12}, {14, 12}, {15, 12}, {16, 12}, {14, 14},
                                   {15, 14}, {16, 14}, {15, 15}, {16, 15}, {16, 16}};
    for (auto &pr : pairs)
        if (pr[0] * pr[1] == R) {
            if (R1) *R1 = pr[0];
            if (R2) *R2 = pr[1];
            return true;
        }
    return false;
}

// 16 columns = 128-byte row segments.  Wider tiles were tried (32 columns with 512 threads, or two 16-column
// halves per thread): the memory system likes them (tools/strided_copy_bench.cu) but the SM side loses more
// to registers / occupancy than the 256-byte segments win (75-95 us against 80 us per pass on B200).
constexpr int kFastC = WEFAX_FAST_C;
constexpr int kFastCW = WEFAX_FAST_C * WEFAX_FAST_H;   // columns per tile

}  // namespace fast
}  // namespace wefax
