// Fused demod-to-pixel kernel: median-5 of the envelope, grey map, `digitalized` and the x4 bicubic
// raster in ONE sweep (wefax.py:175, 197-200, 216, 296-327).  The envelope is read once (4 B / sample),
// `digitalized` (1 B) and the raster (4 B) are written once; nothing else touches HBM.
//
//  * grey map without float64 in the hot loop: round(255 * (m - low) / delta) is a monotone step function of
//    the fp32 median m, so a 256-entry table of the smallest float bit pattern of every level (found once per
//    recording by bisection with the exact float64 formula) decides the level exactly: an fp32 estimate of the
//    level, proven by the table builder to be within +-1 of the truth, is corrected by two compares against the
//    neighbouring thresholds.
//  * one thread owns 8 adjacent image columns and walks down `lines_per_item` lines with a 5-line window of grey
//    levels in registers (compile-time rotation, no moves); every line yields 4 raster rows as 8-byte stores.
//  * image lines start at start_frame + r * width: the envelope rows are misaligned with respect to the raster
//    rows by an amount that is fixed per row.  The envelope comes in as four aligned 16-byte loads (one row
//    prefetched ahead) and the median network is instantiated for the four possible offsets.
#include <algorithm>
#include <cmath>

#include "grey.cuh"

namespace wefax {

constexpr int kGrThreads = 128;
constexpr int kGrCols = 8;   // columns per thread

// One CTA of 256 threads per recording.
__global__ void __launch_bounds__(256) grey_table_kernel(const RecResult *res_all, GreyTable *tables) {
    build_grey_table(res_all + blockIdx.x, tables + blockIdx.x);
}

struct GreyRasterParams {
    const float *env;
    size_t es;
    uint8_t *dig;      // may be null
    size_t ds;
    uint8_t *raster;   // may be null: grey map only
    size_t rs;
    long long n;
    const LineDev *lines;
    const RecResult *res;
    const GreyTable *tables;
    int lines_per_item;
    int only_class;    // >= 0: only recordings whose LineDev.gr_class equals it (mixed-width batches: one launch per class)
    int nk[4][4];      // negated interior Pillow coefficients of the 4 phases (taps in line order)
    int ck[4];         // (1 << 21) + 255 * sum of the phase's coefficients
};

__device__ __forceinline__ double gr_bicubic(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// Pillow precompute_coeffs + normalize_coeffs_8bpc for output row yy of an image of h lines, as weights of
// the input lines r-2 .. r+2 (r = yy / 4); lines outside the image get weight 0.
__device__ void pillow_row_weights(int yy, int h, int kw5[5]) {
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
        kw[t] = t < xmax ? gr_bicubic((t + xmin - center + 0.5)) : 0.0;
        ww += kw[t];
    }
    for (int t = 0; t < 5; ++t) kw5[t] = 0;
    for (int t = 0; t < 5 && t < xmax; ++t) {
        const double kv = (ww != 0.0) ? kw[t] / ww : kw[t];
        const int ki = kv < 0 ? (int)(-0.5 + kv * 4194304.0) : (int)(0.5 + kv * 4194304.0);
        const int sl = xmin + t - (r - 2);
        if (sl >= 0 && sl < 5) kw5[sl] = ki;
    }
}

// d = v0 | v1 << 8 | v2 << 16 | v3 << 24, every value clamped to [0, 255]
__device__ __forceinline__ uint32_t pack4_sat(int v0, int v1, int v2, int v3) {
    uint32_t t, d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(v3), "r"(v2), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(v1), "r"(v0), "r"(t));
    return d;
}

// 8 bytes (lo = bytes 0..3) to an address of any alignment, inline: the alignment is the same for every thread of a warp
// (adjacent threads own adjacent groups of 8 columns), so the branches are uniform.  (The out-of-line store_any below
// costs ~50 instructions a call under the ABI - measured 2.4x on the whole sweep for widths that are not multiples of 8.)
__device__ __forceinline__ void store8_inline(uint8_t *p, uint32_t lo, uint32_t hi) {
    const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7u);
    if (a == 0u) {
        *reinterpret_cast<uint2 *>(p) = make_uint2(lo, hi);
    } else if (a == 4u) {
        reinterpret_cast<uint32_t *>(p)[0] = lo;
        reinterpret_cast<uint32_t *>(p)[1] = hi;
    } else if ((a & 1u) == 0u) {   // 2 or 6
        *reinterpret_cast<uint16_t *>(p) = (uint16_t)lo;
        *reinterpret_cast<uint32_t *>(p + 2) = __funnelshift_r(lo, hi, 16);
        *reinterpret_cast<uint16_t *>(p + 6) = (uint16_t)(hi >> 16);
    } else if ((a & 3u) == 3u) {   // 3 or 7: p + 1 is 4-byte aligned
        p[0] = (uint8_t)lo;
        *reinterpret_cast<uint32_t *>(p + 1) = __funnelshift_r(lo, hi, 8);
        *reinterpret_cast<uint16_t *>(p + 5) = (uint16_t)(hi >> 8);
        p[7] = (uint8_t)(hi >> 24);
    } else {                       // 1 or 5: p + 3 is 4-byte aligned
        p[0] = (uint8_t)lo;
        *reinterpret_cast<uint16_t *>(p + 1) = (uint16_t)(lo >> 8);
        *reinterpret_cast<uint32_t *>(p + 3) = __funnelshift_r(lo, hi, 24);
        p[7] = (uint8_t)(hi >> 24);
    }
}

// kGrCols bytes (lo = bytes 0..3) to an address of any alignment, first `count` bytes only when count < kGrCols
// (out of line: the hot loop only comes here for rows of unaligned widths; the generic items use it throughout)
__device__ __noinline__ void store_any(uint8_t *p, uint32_t lo, uint32_t hi, int count) {
    if (count >= kGrCols) {
        const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7u);
        if (a == 0u) {
            *reinterpret_cast<uint2 *>(p) = make_uint2(lo, hi);
        } else if (a == 4u) {
            reinterpret_cast<uint32_t *>(p)[0] = lo;
            reinterpret_cast<uint32_t *>(p)[1] = hi;
        } else if ((a & 1u) == 0u) {   // 2 or 6
            *reinterpret_cast<uint16_t *>(p) = (uint16_t)lo;
            *reinterpret_cast<uint32_t *>(p + 2) = __funnelshift_r(lo, hi, 16);
            *reinterpret_cast<uint16_t *>(p + 6) = (uint16_t)(hi >> 16);
        } else if ((a & 3u) == 3u) {   // 3 or 7: p + 1 is 4-byte aligned
            p[0] = (uint8_t)lo;
            *reinterpret_cast<uint32_t *>(p + 1) = __funnelshift_r(lo, hi, 8);
            *reinterpret_cast<uint16_t *>(p + 5) = (uint16_t)(hi >> 8);
            p[7] = (uint8_t)(hi >> 24);
        } else {                       // 1 or 5: p + 3 is 4-byte aligned
            p[0] = (uint8_t)lo;
            *reinterpret_cast<uint16_t *>(p + 1) = (uint16_t)(lo >> 8);
            *reinterpret_cast<uint32_t *>(p + 3) = __funnelshift_r(lo, hi, 24);
            p[7] = (uint8_t)(hi >> 24);
        }
    } else {
        for (int c = 0; c < count; ++c) p[c] = (uint8_t)((c < 4 ? lo >> (8 * c) : hi >> (8 * (c - 4))) & 0xFFu);
    }
}

struct GreyQuant {
    const uint2 *pairs;   // shared: (T[k], T[k + 1] - T[k])
    const uint32_t *T;    // shared: T[0 .. 256]
    float scale, off;
    int est_ok;
    // estimate (within +-1, proven by the table builder) corrected by the two neighbouring thresholds
    __device__ __forceinline__ int level_fast(float m) const {
        const uint32_t bits = __float_as_uint(m);
        const int k0 = grey_estimate(m, scale, off);
        const uint2 t = pairs[k0];
        return k0 + (bits - t.x >= t.y && bits >= t.x ? 1 : 0) - (bits < t.x ? 1 : 0);
    }
    __device__ __forceinline__ int level(float m) const {
        return est_ok ? level_fast(m) : grey_from_table(T, __float_as_uint(m));
    }
};

// fp32 estimate of the level, clamped to 0..255 by the conversion itself
__device__ __forceinline__ uint32_t grey_estimate_u8(float m, float scale, float off) {
    uint32_t k;
    asm("cvt.rni.u8.f32 %0, %1;" : "=r"(k) : "f"(fmaf(m, scale, off)));
    return k;
}

// Pillow's BICUBIC coefficients for the x4 up-scaling, rows whose 4 taps are all inside the image (precompute_coeffs
// with a = -0.5, normalised, round(k * 2^22)): they depend on the phase yy % 4 only.  Phases 0 / 1 weigh lines
// r-2 .. r+1, phases 2 / 3 (the mirror images) lines r-1 .. r+2.  launch_grey_raster() recomputes them with
// Pillow's arithmetic and refuses to run if they differ.
__host__ __device__ constexpr int bic_coeff(int ph, int t) {
    // phases 2 / 3 mirror phases 1 / 0
    return ph >= 2 ? bic_coeff(3 - ph, 3 - t)
                   : (ph == 0 ? (t == 0 ? -184320 : t == 1 ? 1634304 : t == 2 ? 3051520 : -307200)
                              : (t == 0 ? -28672 : t == 1 ? 380928 : t == 2 ? 4042752 : -200704));
}
constexpr int kBicBias = (1 << 21) + 255 * 4194304;   // (1 << 21) + 255 * sum: the raster works on 255 - level

// The same row in fp32, two columns per instruction (FFMA2).  Every coefficient is a multiple of 4096 and the four
// of a phase sum to 2^22, so   ((1 << 21) + sum k_t (255 - g_t)) >> 22  =  floor(255.5 - sum (k_t / 2^22) g_t)
// and every partial sum is a multiple of 2^-10 below 2^11 in magnitude: exact in fp32.
static_assert(bic_coeff(0, 0) % 4096 == 0 && bic_coeff(0, 1) % 4096 == 0 && bic_coeff(0, 2) % 4096 == 0 &&
              bic_coeff(0, 3) % 4096 == 0 && bic_coeff(1, 0) % 4096 == 0 && bic_coeff(1, 1) % 4096 == 0 &&
              bic_coeff(1, 2) % 4096 == 0 && bic_coeff(1, 3) % 4096 == 0, "coefficients are multiples of 2^12");
static_assert(bic_coeff(0, 0) + bic_coeff(0, 1) + bic_coeff(0, 2) + bic_coeff(0, 3) == 4194304 &&
              bic_coeff(1, 0) + bic_coeff(1, 1) + bic_coeff(1, 2) + bic_coeff(1, 3) == 4194304, "coefficients sum to 2^22");

__device__ __forceinline__ float2 gr_fma2(float w, float2 x, float2 acc) {
    float2 r;
    asm("{.reg .b64 ta, tb, tc, tr; mov.b64 ta, {%2,%3}; mov.b64 tb, {%4,%4}; mov.b64 tc, {%5,%6}; "
        "fma.rn.f32x2 tr, ta, tb, tc; mov.b64 {%0,%1}, tr;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(x.x), "f"(x.y), "f"(w), "f"(acc.x), "f"(acc.y));
    return r;
}
__device__ __forceinline__ int gr_floor(float x) {
    int k;
    asm("cvt.rmi.s32.f32 %0, %1;" : "=r"(k) : "f"(x));
    return k;
}

template <int PH>
__device__ __forceinline__ float2 bic_phase2(float2 a, float2 b, float2 c, float2 d) {
    constexpr float w0 = -(float)bic_coeff(PH, 0) / 4194304.f, w1 = -(float)bic_coeff(PH, 1) / 4194304.f;
    constexpr float w2 = -(float)bic_coeff(PH, 2) / 4194304.f, w3 = -(float)bic_coeff(PH, 3) / 4194304.f;
    float2 acc = make_float2(255.5f, 255.5f);
    acc = gr_fma2(w0, a, acc);
    acc = gr_fma2(w1, b, acc);
    acc = gr_fma2(w2, c, acc);
    acc = gr_fma2(w3, d, acc);
    return acc;
}

// One interior item: all its lines are image lines at least 2 lines from the image's first / last line, every
// load stays inside the recording, the fp32 estimate is valid, the column group is complete.  OFF: offset (in
// floats, mod 4) of the envelope element two to the left of the item's first column from a 16-byte boundary, the
// same for every line when the width is a multiple of 4; OFF < 0: evaluated per line.  ALIGN: alignment every
// raster row of the item is known to have (8, 4, or 0 = anything).  HAS_DIG: digitalized is written.
// The line loop is deliberately NOT unrolled: its body stays resident in the instruction cache; the price is the
// moves that shift the 5-line window (grey levels as floats, two columns per register pair: 17 % of the kernel's
// instructions).  Measured alternatives on B200, 60-min recording, 94.8 us as it stands: the loop unrolled five times
// (window positions become register names) 120 us, instruction-cache misses; only the bicubic part five times, one copy
// per position of a 5-line ring chosen by a switch, 100.8 us (10 880 instructions of code per kernel, 32 bytes spilled).
template <int OFF, int ALIGN, bool HAS_DIG>
__device__ __forceinline__ void interior_item(const GreyQuant &Q, const float *e, uint8_t *dg, uint8_t *out,
                                              long long i_first, long long r_a, int nrows, int w, int c0, int ncols) {
    // ncols < kGrCols: the last, partial column group of a line (widths that are not multiples of 8).  All 8 columns
    // are computed (the loads run on into the next line, which is inside the recording); only the stores are cut.
    const bool whole = ALIGN == 8 || ncols == kGrCols;
    constexpr int NP = kGrCols / 2;
    float2 win[5][NP];
    const float *prow = e + i_first - 2;   // x[0] of the line being fetched
    float4 nx[4];
    auto fetch = [&]() {
        const float4 *pa = reinterpret_cast<const float4 *>(reinterpret_cast<uintptr_t>(prow) & ~(uintptr_t)15);
#pragma unroll
        for (int q = 0; q < 4; ++q) nx[q] = __ldg(pa + q);
    };
    fetch();
    uint8_t *drow = dg + i_first;                       // digitalized of the line being computed
    uint8_t *orow = out + (size_t)(4 * r_a) * w + c0;   // raster rows of the line being emitted
#pragma unroll
    for (int t = 0; t < 5; ++t)
#pragma unroll
        for (int c = 0; c < NP; ++c) win[t][c] = make_float2(0.f, 0.f);

#pragma unroll 1
    for (int j = 0; j < nrows; ++j) {
        // ---- grey levels of line r_a - 2 + j ----------------------------------------------------------------
        float f[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            f[4 * q] = nx[q].x; f[4 * q + 1] = nx[q].y; f[4 * q + 2] = nx[q].z; f[4 * q + 3] = nx[q].w;
        }
        float m[kGrCols];
        if (OFF >= 0) {
            med8_from16<(OFF >= 0 ? OFF : 0)>(f, m);
        } else {
            switch ((int)((reinterpret_cast<uintptr_t>(prow) >> 2) & 3u)) {
                case 0: med8_from16<0>(f, m); break;
                case 1: med8_from16<1>(f, m); break;
                case 2: med8_from16<2>(f, m); break;
                default: med8_from16<3>(f, m); break;
            }
        }
        prow += w;
        if (j + 1 < nrows) fetch();   // the medians have consumed nx: the next line streams in under the rest of this one
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int c = 0; c < NP; ++c) win[t][c] = win[t + 1][c];
        uint32_t g[kGrCols];
        uint32_t bad = 0u;
#pragma unroll
        for (int c = 0; c < kGrCols; ++c) {
            g[c] = grey_estimate_u8(m[c], Q.scale, Q.off);
            const uint2 t = Q.pairs[g[c]];
            bad |= (__float_as_uint(m[c]) - t.x >= t.y) ? 1u : 0u;
        }
        if (bad) {   // some estimate is one level off (rare): redo the line with the corrected form
#pragma unroll
            for (int c = 0; c < kGrCols; ++c) g[c] = (uint32_t)Q.level_fast(m[c]);
        }
#pragma unroll
        for (int c = 0; c < NP; ++c) win[4][c] = make_float2((float)g[2 * c], (float)g[2 * c + 1]);
        if (HAS_DIG) {
            if (j >= 2 && j < nrows - 2) {
                const uint32_t lo = g[0] | (g[1] << 8) | (g[2] << 16) | (g[3] << 24);
                const uint32_t hi = g[4] | (g[5] << 8) | (g[6] << 16) | (g[7] << 24);
                // (start_frame fixes the alignment of the digitalized rows: the same for every line when the width is
                //  a multiple of 8, changing from line to line otherwise; always the same across a warp)
                if (whole) store8_inline(drow, lo, hi);
                else store_any(drow, lo, hi, ncols);
            }
            drow += w;
        }
        // ---- line r_a + j - 4 is complete: its 4 raster rows ---------------------------------------------------
        if (j >= 4) {
            uint8_t *o = orow;
            auto put = [&](const float2 (&v)[NP]) {
                const uint32_t lo = pack4_sat(gr_floor(v[0].x), gr_floor(v[0].y), gr_floor(v[1].x), gr_floor(v[1].y));
                const uint32_t hi = pack4_sat(gr_floor(v[2].x), gr_floor(v[2].y), gr_floor(v[3].x), gr_floor(v[3].y));
                if (ALIGN == 8) {
                    *reinterpret_cast<uint2 *>(o) = make_uint2(lo, hi);
                } else if (!whole) {
                    store_any(o, lo, hi, ncols);
                } else if (ALIGN == 4) {
                    reinterpret_cast<uint32_t *>(o)[0] = lo;
                    reinterpret_cast<uint32_t *>(o)[1] = hi;
                } else {
                    store8_inline(o, lo, hi);
                }
                o += w;
            };
            float2 v[NP];
#pragma unroll
            for (int c = 0; c < NP; ++c) v[c] = bic_phase2<0>(win[0][c], win[1][c], win[2][c], win[3][c]);
            put(v);
#pragma unroll
            for (int c = 0; c < NP; ++c) v[c] = bic_phase2<1>(win[0][c], win[1][c], win[2][c], win[3][c]);
            put(v);
#pragma unroll
            for (int c = 0; c < NP; ++c) v[c] = bic_phase2<2>(win[1][c], win[2][c], win[3][c], win[4][c]);
            put(v);
#pragma unroll
            for (int c = 0; c < NP; ++c) v[c] = bic_phase2<3>(win[1][c], win[2][c], win[3][c], win[4][c]);
            put(v);
            orow = o;
        }
    }
}

// ALIGN: alignment every raster row of the launch's recordings is known to have: 8 (width % 8 == 0), 4 (width % 4 == 0)
// or 0 (anything); for 8 and 4 the envelope rows of a recording also share one 16-byte phase.
// (5 CTAs per SM at 96 registers when the rows keep their alignment; odd widths carry per-line alignments, and at 96
//  registers the allocator reused a destination of the in-flight envelope load as a temporary, a full DRAM latency per
//  line: they get 128 registers and 4 CTAs)
template <int ALIGN>
__global__ void __launch_bounds__(kGrThreads, ALIGN == 0 ? 4 : 5) grey_raster_kernel(const __grid_constant__ GreyRasterParams P) {
    __shared__ uint32_t s_T[260];
    __shared__ uint2 s_pairs[256];
    const int rec = blockIdx.y;
    if (P.only_class >= 0 && P.lines[rec].gr_class != P.only_class) return;
    const RecResult *res = P.res + rec;
    const GreyTable *tab = P.tables + rec;
    for (int i = threadIdx.x; i < 257; i += kGrThreads) s_T[i] = tab->T[i];
    for (int i = threadIdx.x; i < 256; i += kGrThreads) {
        const uint32_t t0 = tab->T[i], t1 = tab->T[i + 1];
        s_pairs[i] = make_uint2(t0, t1 - t0);
    }
    GreyQuant Q;
    Q.pairs = s_pairs;
    Q.T = s_T;
    Q.scale = tab->scale;
    Q.off = tab->off;
    Q.est_ok = tab->est_ok;
    const int w = P.lines[rec].width;
    const long long s = res->start_frame;
    const int h = (P.raster && res->status == WEFAX_REC_OK) ? res->height / 4 : 0;
    const long long n = P.n;
    __syncthreads();

    // line space anchored at start_frame: line r holds samples s + r*w .. s + r*w + w - 1; the partial lines in
    // front of start_frame and behind the image only produce grey levels
    const long long r_lo = -((s + w - 1) / w);
    const long long r_hi = (n - s + w - 1) / w;
    const int ng = (w + kGrCols - 1) / kGrCols;
    const int U = P.lines_per_item;
    const long long ntiles = (r_hi - r_lo + U - 1) / U;
    const long long item = (long long)blockIdx.x * kGrThreads + threadIdx.x;
    if (item >= ntiles * ng) return;
    // the first CTAs take the LAST tile (image / recording edge: the slow generic form), then tiles 0, 1, ...
    long long tile = item / ng;
    const int grp = (int)(item - tile * ng);
    tile = tile == 0 ? ntiles - 1 : tile - 1;
    // the last column group of a width that is not a multiple of 8 is moved left so that it is whole: it recomputes a
    // few columns of its neighbour (both write the same bytes) instead of being the one partial group whose stores
    // have to be cut - that one thread used to hold its whole warp back in every tile
    const int c0 = w >= kGrCols ? min(grp * kGrCols, w - kGrCols) : 0;
    const int ncols = min(kGrCols, w - c0);
    const long long r_a = r_lo + tile * U, r_b = min(r_a + U, r_hi);

    const float *e = P.env + (size_t)rec * P.es;
    uint8_t *dg = P.dig ? P.dig + (size_t)rec * P.ds : nullptr;
    uint8_t *out = P.raster ? P.raster + (size_t)rec * P.rs : nullptr;

    const long long i_first = s + (r_a - 2) * w + c0;   // sample (line r_a - 2, column c0)
    const bool interior = Q.est_ok && r_a >= 2 && r_b + 2 <= h && i_first - 2 >= 4 && s + (r_b + 1) * w + c0 + 14 <= n;
    if (interior) {
        const int nrows = (int)(r_b - r_a) + 4;
#define WEFAX_GR_RUN(OFF_)                                                                        \
    if (dg) interior_item<OFF_, ALIGN, true>(Q, e, dg, out, i_first, r_a, nrows, w, c0, ncols);   \
    else interior_item<OFF_, ALIGN, false>(Q, e, dg, out, i_first, r_a, nrows, w, c0, ncols);
        if (ALIGN >= 4) {
            switch ((int)((reinterpret_cast<uintptr_t>(e + i_first - 2) >> 2) & 3u)) {
                case 0: WEFAX_GR_RUN(0) break;
                case 1: WEFAX_GR_RUN(1) break;
                case 2: WEFAX_GR_RUN(2) break;
                default: WEFAX_GR_RUN(3) break;
            }
        } else {
            WEFAX_GR_RUN(-1)
        }
#undef WEFAX_GR_RUN
        return;
    }

    // ---- generic items: recording / image edges, recordings without an image ------------------------------
    int win[5][kGrCols];
#pragma unroll
    for (int t = 0; t < 5; ++t)
#pragma unroll
        for (int c = 0; c < kGrCols; ++c) win[t][c] = 0;
    // only lines that feed a raster row of this item or are its own need grey levels
    const bool any_raster = out && r_a < h && r_b > 0;
    const long long r_from = any_raster ? r_a - 2 : r_a, r_to = any_raster ? r_b + 2 : r_b;
#pragma unroll 1
    for (long long r = r_from; r < r_to; ++r) {
        const long long i0 = s + r * w + c0;
        float f[16];
#pragma unroll
        for (int j = 0; j < 12; ++j) {
            const long long i = i0 - 2 + j;
            f[j] = (i >= 0 && i < n) ? __ldg(e + i) : 0.f;
        }
        f[12] = f[13] = f[14] = f[15] = 0.f;
        float m[kGrCols];
        med8_from16<0>(f, m);
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int c = 0; c < kGrCols; ++c) win[t][c] = win[t + 1][c];
#pragma unroll
        for (int c = 0; c < kGrCols; ++c) win[4][c] = Q.level(m[c]);
        if (dg && r >= r_a && r < r_b) {
#pragma unroll
            for (int c = 0; c < kGrCols; ++c) {
                const long long i = i0 + c;
                if (c < ncols && i >= 0 && i < n) dg[i] = (uint8_t)win[4][c];
            }
        }
        const long long q = r - 2;
        if (out && q >= r_a && q < r_b && q >= 0 && q < h) {
            const bool inner = q >= 2 && q + 2 < h;
#pragma unroll 1
            for (int ph = 0; ph < 4; ++ph) {
                int kw[5];
                if (inner) {
                    kw[0] = ph < 2 ? -P.nk[ph][0] : 0;
                    kw[1] = ph < 2 ? -P.nk[ph][1] : -P.nk[ph][0];
                    kw[2] = ph < 2 ? -P.nk[ph][2] : -P.nk[ph][1];
                    kw[3] = ph < 2 ? -P.nk[ph][3] : -P.nk[ph][2];
                    kw[4] = ph < 2 ? 0 : -P.nk[ph][3];
                } else {
                    pillow_row_weights((int)(4 * q + ph), h, kw);
                }
                int v[kGrCols];
#pragma unroll
                for (int c = 0; c < kGrCols; ++c) {
                    int acc = 1 << 21;
#pragma unroll
                    for (int t = 0; t < 5; ++t) acc += kw[t] * (255 - win[t][c]);   // luminance 255 - value (wefax.py:303)
                    v[c] = acc >> 22;
                }
                store_any(out + (size_t)(4 * q + ph) * w + c0, pack4_sat(v[0], v[1], v[2], v[3]),
                          pack4_sat(v[4], v[5], v[6], v[7]), ncols);
            }
        }
    }
}

void launch_grey_table(wefax_ctx *ctx, const RecResult *res, GreyTable *tables, int batch) {
    StageTimer timer(ctx, "grey_table");
    grey_table_kernel<<<batch, 256, 0, ctx->stream>>>(res, tables);
    CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
}

namespace {
double host_bicubic(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}
}  // namespace

void launch_grey_raster(wefax_ctx *ctx, const float *env, size_t es, uint8_t *dig, size_t ds, uint8_t *raster, size_t rs,
                        long long n, int batch, const LineDev *d_lines, const LineDev *h_lines, const RecResult *res,
                        const GreyTable *tables) {
    StageTimer timer(ctx, "grey_raster");
    GreyRasterParams P;
    P.env = env; P.es = es; P.dig = dig; P.ds = ds; P.raster = raster; P.rs = rs; P.n = n;
    P.lines = d_lines; P.res = res; P.tables = tables;
    // interior rows: Pillow's coefficients depend on the phase only (filter arguments are exact binary fractions
    // and sum to exactly 1), so they are computed here once, with Pillow's own arithmetic
    for (int ph = 0; ph < 4; ++ph) {
        const double center = (ph + 0.5) * 0.25 + 8.0;   // any line far from the edges
        const int xmin = (int)(center - 2.0 + 0.5), xmax = (int)(center + 2.0 + 0.5) - xmin;
        double kw[5], ww = 0.0;
        for (int t = 0; t < 5; ++t) {
            kw[t] = t < xmax ? host_bicubic(t + xmin - center + 0.5) : 0.0;
            ww += kw[t];
        }
        long long sum = 0;
        for (int t = 0; t < 4; ++t) {
            const double kv = (ww != 0.0) ? kw[t] / ww : kw[t];
            const int ki = kv < 0 ? (int)(-0.5 + kv * 4194304.0) : (int)(0.5 + kv * 4194304.0);
            P.nk[ph][t] = -ki;
            sum += ki;
        }
        P.ck[ph] = (int)((1ll << 21) + 255 * sum);
        for (int t = 0; t < 4; ++t) {
            const int expect = bic_coeff(ph, t);
            if (P.nk[ph][t] != -expect || P.ck[ph] != kBicBias)
                WEFAX_THROW(WEFAX_ERR_UNSUPPORTED, "bicubic coefficient table does not match Pillow's arithmetic on this host");
        }
    }
    // recordings by alignment class (LineDev.gr_class, set by api.cu from the width): the raster rows of a recording
    // are all 8- / 4-byte aligned when its width is a multiple of 8 / 4 and so are the raster base and stride
    const bool base8 = (reinterpret_cast<uintptr_t>(raster) & 7) == 0 && rs % 8 == 0;
    const bool base4 = (reinterpret_cast<uintptr_t>(raster) & 3) == 0 && rs % 4 == 0;
    int count[3] = {0, 0, 0};   // 0: generic widths, 1: width % 4 == 0, 2: width % 8 == 0
    for (int r = 0; r < batch; ++r) count[h_lines[r].gr_class]++;
    auto resident_ctas = [&](const void *fn, int fallback) {
        auto it = ctx->smem_configured.find(fn);
        if (it != ctx->smem_configured.end()) return it->second;
        int per_sm = fallback;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kGrThreads, 0) != cudaSuccess || per_sm < 1) {
            (void)cudaGetLastError();
            per_sm = fallback;
        }
        ctx->smem_configured[fn] = per_sm;
        return per_sm;
    };
    for (int cls = 2; cls >= 0; --cls) {
        if (!count[cls]) continue;
        const int align = (cls == 2 && base8) ? 8 : ((cls >= 1 && base4) ? 4 : 0);
        const int per_sm = align == 8   ? resident_ctas((const void *)grey_raster_kernel<8>, 5)
                           : align == 4 ? resident_ctas((const void *)grey_raster_kernel<4>, 5)
                                        : resident_ctas((const void *)grey_raster_kernel<0>, 4);
        const double resident = (double)ctx->sm_count * per_sm * kGrThreads;
        auto items_for = [&](int U, long long *max_items) {
            double total = 0;
            long long mx = 0;
            for (int r = 0; r < batch; ++r) {
                if (h_lines[r].gr_class != cls) continue;
                const int w = h_lines[r].width;
                const long long nl = n / w + 2;
                const long long it = ((nl + U - 1) / U) * ((w + kGrCols - 1) / kGrCols);
                total += (double)it;
                mx = std::max(mx, it);
            }
            if (max_items) *max_items = mx;
            return total;
        };
        // lines per item: a long walk amortises the 4 extra lines of every item (they cost the grey map only, ~40 % of
        // a line), but the grid should be several waves of resident CTAs and end close to a whole one
        int best_u = 16;
        double best_eff = -1.0;
        for (int U = 8; U <= 40; ++U) {
            const double waves = items_for(U, nullptr) / resident;
            const double eff = (double)U / (U + 1.6) * (waves / std::ceil(waves - 1e-9)) * (waves >= 3.0 ? 1.0 : 0.8);
            if (eff > best_eff) {
                best_eff = eff;
                best_u = U;
            }
        }
        const char *force_u = getenv("WEFAX_GR_LINES");
        if (force_u && atoi(force_u) >= 1) best_u = atoi(force_u);
        P.lines_per_item = best_u;
        P.only_class = count[cls] == batch ? -1 : cls;
        long long max_items = 0;
        items_for(best_u, &max_items);
        dim3 grid((unsigned)((max_items + kGrThreads - 1) / kGrThreads), batch);
        if (align == 8)
            grey_raster_kernel<8><<<grid, kGrThreads, 0, ctx->stream>>>(P);
        else if (align == 4)
            grey_raster_kernel<4><<<grid, kGrThreads, 0, ctx->stream>>>(P);
        else
            grey_raster_kernel<0><<<grid, kGrThreads, 0, ctx->stream>>>(P);
        CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
}

}  // namespace wefax
