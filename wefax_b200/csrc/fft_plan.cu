// Host-side FFT planning: factor n into pass lengths, size the shared-memory
// tiles, build the twiddle / permutation tables on the device.
#include <algorithm>
#include <mutex>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>

#include "fft.cuh"
#include "fft_fast.cuh"
#include "fft_mid.cuh"

namespace wefax {

namespace {

// tile budget in complex elements (64 KiB of float2 => 3 CTAs / SM)
constexpr int kTileMax = 8192;
// strided passes keep at least this many adjacent columns per tile (coalescing)
constexpr int kMinCols = 8;
// ... and at most this many
constexpr int kMaxCols = 64;
// the stride-1 pass keeps tile + w_R table + permutation (18 bytes per point) within 227 KiB
constexpr long long kLastPassMax = 12000;

bool smooth13(long long n) {
    for (int p : {2, 3, 5, 7, 11, 13})
        while (n % p == 0) n /= p;
    return n == 1;
}

std::vector<long long> divisors_upto(long long n, long long cap) {
    std::vector<long long> small, out;
    for (long long d = 1; d * d <= n; ++d)
        if (n % d == 0) {
            if (d <= cap) out.push_back(d);
            long long e = n / d;
            if (e != d && e <= cap) out.push_back(e);
        }
    std::sort(out.begin(), out.end());
    return out;
}

// stage radices the kernel implements (primes and two-factor in-register composites)
const int kRadixMenu[] = {2, 3, 4, 5, 7, 8, 11, 13, 6, 9, 10, 12, 14, 15, 16, 20, 21, 24, 25, 28, 32};

// rough thread-instructions per element of one shared-memory stage of radix r
double stage_cost(int r) { return 14.0 + 30.0 / r + 2.5 * std::log2((double)r); }
constexpr double kPassCost = 40.0;   // global load/store + inter-pass twiddle, per element

// cheapest split of R into menu radices (memoised); cost < 0 when impossible
struct StagePlan {
    double cost = -1.0;
    std::vector<int> radices;
};
const StagePlan &stage_plan(int R) {
    // per host thread: contexts are driven from several threads at once (one context per thread), and the memo
    // is mutated while references into it are alive
    thread_local std::map<int, StagePlan> memo;
    auto it = memo.find(R);
    if (it != memo.end()) return it->second;
    StagePlan best;
    if (R == 1) {
        best.cost = 0.0;
    } else {
        for (int r : kRadixMenu) {
            if (R % r) continue;
            const StagePlan &sub = stage_plan(R / r);
            if (sub.cost < 0) continue;
            double c = stage_cost(r) + sub.cost;
            if (best.cost < 0 || c < best.cost - 1e-9) {
                best.cost = c;
                best.radices = sub.radices;
                best.radices.push_back(r);   // larger radices tend to come last: the last stage has no twiddles
            }
        }
    }
    return memo[R] = best;
}

// Columns per tile of a pass of length R.  Strided passes want >= 32 adjacent columns
// (256-byte row segments); the budget is 8192 complex (64 KiB, 2-3 CTAs per SM) and is
// raised to 16384 (one CTA per SM) only when that is what it takes to get there.
int tile_cols(int R, int ncols, bool strided) {
    int C = 1;
    while (C * 2 * R <= kTileMax && C * 2 <= kMaxCols) C *= 2;
    if (strided && C < 32)
        while (C * 2 * R <= 2 * kTileMax && C < 32) C *= 2;
    while (C > 1 && C / 2 >= ncols) C /= 2;
    return C;
}

// per-element cost of one pass of length R: its stages, each divided by the fraction
// of the 256 threads that have a butterfly in the last round, plus the global traffic,
// scaled by how badly short row segments and single-CTA occupancy hurt (measured on B200)
double pass_cost(int R, long long n, bool strided) {
    const StagePlan &sp = stage_plan(R);
    if (sp.cost < 0) return -1.0;
    // specialised two-stage kernel (fft_fast.cuh): ~45 instructions per point
    if (strided && n >= (1 << 16) && fast::fast_pair(R, nullptr, nullptr)) return 50.0;
    // stride-1 pass lengths the fused middle kernel of the real-input Hilbert transform handles (fft_mid.cuh)
    if (!strided && n >= (1 << 16) && fast::mid_pair(R, nullptr, nullptr)) return 60.0;
    const int C = tile_cols(R, (int)std::min<long long>(n / R, 1 << 30), strided);
    double c = kPassCost;
    for (int r : sp.radices) {
        const int total = C * (R / r);
        const int rounds = (total + kFftThreads - 1) / kFftThreads;
        c += stage_cost(r) * (double)(rounds * kFftThreads) / (double)total;
    }
    if (strided && C < 32) c *= 1.0 + 0.5 * (32.0 / C - 1.0);     // 64-byte segments cost ~2.5x
    // CTAs per SM by shared memory (tile + w_R table + permutation): measured per-element
    // pass times on B200 are ~5 ps with three resident CTAs, ~6 ps with two, ~10 ps with one
    const double smem = (double)C * R * 8.0 + R * 10.0 + 8192.0;
    const int ctas = (int)std::min(3.0, std::floor(227.0 * 1024.0 / smem));
    c *= ctas >= 3 ? 1.0 : (ctas == 2 ? 1.15 : 1.9);
    return c;
}

struct Search {
    long long n, cap_s, cap_l, min_r;
    double best_cost = 1e300;
    std::vector<int> best;
    std::vector<int> cur;
    // strided factors are chosen non-decreasing; the remainder is the last pass
    void go(long long rem, int left, long long lo) {
        if (left == 0) {
            if (rem > cap_l || rem < 2 || (!cur.empty() && rem < min_r)) return;
            // an even last pass keeps every stride even: TMA tensor loads need 16-byte row pitches
            if (!cur.empty() && n % 2 == 0 && rem % 2 != 0) return;
            double cost = pass_cost((int)rem, n, false);
            if (cost < 0) return;
            for (int r : cur) cost += pass_cost(r, n, true);
            if (cost < best_cost - 1e-9) {
                best_cost = cost;
                best = cur;
                best.push_back((int)rem);
            }
            return;
        }
        for (long long d : divisors_upto(rem, cap_s)) {
            if (d < lo || d < 2 || d < min_r) continue;
            if (stage_plan((int)d).cost < 0) continue;
            cur.push_back((int)d);
            go(rem / d, left - 1, d);
            cur.pop_back();
        }
    }
};

std::vector<int> stage_radices(int R) { return stage_plan(R).radices; }

__global__ void twiddle_table_kernel(float2 *dst, int count, double L, double mult) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    // w_L^(i*mult) = exp(-2*pi*i * (i*mult mod L) / L), evaluated in double
    double e = fmod((double)i * mult, L);
    double s, c;
    sincospi(-2.0 * e / L, &s, &c);
    dst[i] = make_float2((float)c, (float)s);
}

}  // namespace

bool plan_factors(long long n, std::vector<int> &Rs) {
    Rs.clear();
    if (n < 1) return false;
    if (n == 1) {
        Rs.push_back(1);
        return true;
    }
    if (!smooth13(n)) return false;
    double best_cost = 1e300;
    for (int P = 1; P <= kMaxPasses; ++P) {
        Search s;
        s.n = n;
        s.cap_s = kTileMax / kMinCols;
        s.cap_l = kLastPassMax;
        s.min_r = n >= 64 * 64 ? 64 : 2;   // no degenerate passes on long transforms
        s.go(n, P - 1, 2);
        if (!s.best.empty() && s.best_cost < best_cost - 1e-9) {
            best_cost = s.best_cost;
            Rs = s.best;
        }
    }
    return !Rs.empty();
}

long long next_smooth_length(long long m) {
    long long best = -1;
    // enumerate 2^a 3^b 5^c 7^d in [m, 2m)
    for (long long p7 = 1; p7 < 2 * m; p7 *= 7)
        for (long long p5 = p7; p5 < 2 * m; p5 *= 5)
            for (long long p3 = p5; p3 < 2 * m; p3 *= 3) {
                long long v = p3;
                while (v < m) v *= 2;
                if (best < 0 || v < best) {
                    std::vector<int> tmp;
                    if (plan_factors(v, tmp)) best = v;
                }
            }
    return best;
}

std::unique_ptr<FftPlan> make_plan(long long n, cudaStream_t stream) {
    std::vector<int> Rs;
    if (!plan_factors(n, Rs)) return nullptr;
    auto plan = std::make_unique<FftPlan>();
    plan->n = n;
    plan->npass = (int)Rs.size();
    const int P = plan->npass;
    for (int i = 0; i < P; ++i) plan->Rs[i] = Rs[i];
    for (int i = P - 1; i >= 0; --i) plan->S[i] = (i == P - 1) ? 1 : plan->S[i + 1] * Rs[i + 1];

    // table layout
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) & ~size_t(255);
        return o;
    };
    size_t o_twR[kMaxPasses], o_perm[kMaxPasses], o_lo[kMaxPasses], o_hi[kMaxPasses];
    long long n_hi[kMaxPasses];
    for (int i = 0; i < P; ++i) {
        o_twR[i] = take((size_t)Rs[i] * sizeof(float2));
        o_perm[i] = take((size_t)Rs[i] * sizeof(uint16_t));
        long long L = (long long)Rs[i] * plan->S[i];
        n_hi[i] = (L >> kTwLoBits) + 1;
        o_lo[i] = take(sizeof(float2) << kTwLoBits);
        o_hi[i] = take((size_t)n_hi[i] * sizeof(float2));
    }
    const long long n2_hi = ((2 * n) >> kTwLoBits) + 1;
    const size_t o2_lo = take(sizeof(float2) << kTwLoBits), o2_hi = take((size_t)n2_hi * sizeof(float2));
    char *base = (char *)plan->tables.reserve(off);
    plan->tw2_lo = (const float2 *)(base + o2_lo);
    plan->tw2_hi = (const float2 *)(base + o2_hi);
    twiddle_table_kernel<<<((1 << kTwLoBits) + 255) / 256, 256, 0, stream>>>((float2 *)(base + o2_lo), 1 << kTwLoBits,
                                                                           2.0 * (double)n, 1.0);
    twiddle_table_kernel<<<(unsigned)((n2_hi + 255) / 256), 256, 0, stream>>>((float2 *)(base + o2_hi), (int)n2_hi,
                                                                           2.0 * (double)n, (double)(1 << kTwLoBits));

    for (int i = 0; i < P; ++i) {
        PassDev d;
        memset(&d, 0, sizeof(d));
        const int R = Rs[i];
        d.R = R;
        d.S = (int)plan->S[i];
        d.ncols = (int)(n / R);
        d.contiguous = (i == P - 1);
        const int C = tile_cols(R, d.ncols, !d.contiguous);
        d.C = C;
        d.log2C = 0;
        while ((1 << d.log2C) < C) ++d.log2C;
        std::vector<int> rad = stage_radices(R);
        if ((int)rad.size() > kMaxStages) return nullptr;
        d.nstages = (int)rad.size();
        int L = R;
        for (int s = 0; s < d.nstages; ++s) {
            d.radix[s] = rad[s];
            d.divM[s].init(L / rad[s]);
            d.divNbf[s].init(R / rad[s]);
            L /= rad[s];
        }
        d.divR.init(R);
        const long long nouter = n / ((long long)R * d.S);
        if (d.contiguous) {
            d.tiles_per_o = 1;
            d.ntiles = (d.ncols + C - 1) / C;
        } else {
            d.tiles_per_o = (d.S + C - 1) / C;
            d.ntiles = (int)(nouter * d.tiles_per_o);
        }
        d.divTpo.init(d.tiles_per_o);
        d.fast_R1 = d.fast_R2 = 0;
        d.fast_tiles_per_o = d.fast_ntiles = 1;
        if (!d.contiguous && fast::fast_pair(R, &d.fast_R1, &d.fast_R2)) {
            d.fast_tiles_per_o = (d.S + fast::kFastCW - 1) / fast::kFastCW;
            d.fast_ntiles = (int)(nouter * d.fast_tiles_per_o);
        }
        d.fast_divTpo.init(d.fast_tiles_per_o);
        // TMA box: the most rows (<= 256) that divide R and keep every box 128-byte aligned in smem
        d.rbox = 0;
        for (int rb = std::min(R, 256); rb >= 1; --rb)
            if (R % rb == 0 && ((size_t)rb * C * sizeof(float2)) % 128 == 0) {
                d.rbox = rb;
                break;
            }
        d.nbox = d.rbox ? R / d.rbox : 0;
        if (d.nbox > 16) d.rbox = d.nbox = 0;
        d.nthreads = std::max(C, kFftThreads);
        d.twR = (const float2 *)(base + o_twR[i]);
        d.perm = (const uint16_t *)(base + o_perm[i]);
        d.smem_bytes = (int)((size_t)C * R * sizeof(float2) + (size_t)R * sizeof(float2) +
                             (size_t)((R + 1) & ~1) * sizeof(uint16_t) + (size_t)2 * C * sizeof(int) + 48 +
                             (size_t)C * ((R + kTwStep - 1) / kTwStep + kTwStep) * sizeof(float2));

        // digit-reversal: smem position of output k after the in-place DIF stages
        std::vector<uint16_t> perm(R);
        for (int k = 0; k < R; ++k) {
            int pos = 0, kk = k, span = R;
            for (int r : rad) {
                int dg = kk % r;
                kk /= r;
                span /= r;
                pos += dg * span;
            }
            perm[k] = (uint16_t)pos;
        }
        CUDA_CHECK(cudaMemcpyAsync(base + o_perm[i], perm.data(), R * sizeof(uint16_t),
                                   cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));   // perm is a stack temporary

        const double Lp = (double)R * (double)plan->S[i];
        twiddle_table_kernel<<<(R + 255) / 256, 256, 0, stream>>>((float2 *)(base + o_twR[i]), R, (double)R, 1.0);
        twiddle_table_kernel<<<((1 << kTwLoBits) + 255) / 256, 256, 0, stream>>>(
            (float2 *)(base + o_lo[i]), 1 << kTwLoBits, Lp, 1.0);
        twiddle_table_kernel<<<(unsigned)((n_hi[i] + 255) / 256), 256, 0, stream>>>(
            (float2 *)(base + o_hi[i]), (int)n_hi[i], Lp, (double)(1 << kTwLoBits));
        CUDA_CHECK(cudaGetLastError());

        // forward: multiply by w_{L_i}^{k*m} on store (all but the last pass)
        d.tw_mode = (i < P - 1) ? 1 : 0;
        d.ko_R = 1;
        d.tw_lo = (const float2 *)(base + o_lo[i]);
        d.tw_hi = (const float2 *)(base + o_hi[i]);
        snprintf(d.tag, sizeof(d.tag), "fft_fwd_%d", i);
        plan->fwd[i] = d;
        // inverse (passes run P-1 .. 0): the twiddle the NEXT pass (i-1) needs on its input,
        // w_{L_{i-1}}^{k_{i-1} * (position inside its sub-problem)}, is applied on this pass's store
        d.tw_mode = (i > 0) ? 2 : 0;
        d.ko_R = (i > 0) ? Rs[i - 1] : 1;
        d.tw_lo = (const float2 *)(base + o_lo[i > 0 ? i - 1 : 0]);
        d.tw_hi = (const float2 *)(base + o_hi[i > 0 ? i - 1 : 0]);
        snprintf(d.tag, sizeof(d.tag), "fft_inv_%d", i);
        plan->inv[i] = d;
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
    return plan;
}

}  // namespace wefax

namespace wefax {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)ptr;
        else
            (void)cudaGetLastError();
    });
    return fn;
}

int choose_load_mode(const PassDev &p, const float2 *base, size_t bstride, int batch, CUtensorMap *map) {
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return 0;
    if (batch > 1 && (bstride & 1)) return 0;               // every batch element must stay 16-byte aligned
    if (p.contiguous) {
        // one bulk copy per tile: source and size must be multiples of 16 bytes
        const bool full_ok = (((size_t)p.C * p.R) & 1) == 0 || p.ntiles == 1;
        const int tail = p.ncols % p.C;
        const bool tail_ok = ((size_t)(tail ? tail : p.C) * p.R & 1) == 0;
        const bool first_ok = p.ntiles > 1 || tail_ok;
        return (full_ok && tail_ok && first_ok) ? 2 : 0;
    }
    if ((p.S & 1) || !p.rbox) return 0;                      // row pitch S*8 bytes must be a multiple of 16
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return 0;
    const unsigned long long nouter = (unsigned long long)p.ncols / (unsigned long long)p.S;
    cuuint64_t dims[4] = {2ull * (unsigned long long)p.S, (cuuint64_t)p.R, nouter, (cuuint64_t)batch};
    cuuint64_t strides[3] = {(cuuint64_t)p.S * 8ull, (cuuint64_t)p.R * (cuuint64_t)p.S * 8ull,
                             (cuuint64_t)(batch > 1 ? bstride : (size_t)p.R * p.S * nouter) * 8ull};
    cuuint32_t box[4] = {2u * (cuuint32_t)p.C, (cuuint32_t)p.rbox, 1u, 1u};
    cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    CUresult rc = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void *)base, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return rc == CUDA_SUCCESS ? 1 : 0;
}

// 4-D tensor map {2S floats, R, outer, batch} with a box of `cols` complex columns x `rbox` rows for the
// TMA-staged strided pass (fft_fast.cuh: fft_fast_tma3_kernel); false when the geometry cannot be encoded.
bool encode_strided_map(const PassDev &p, const float2 *base, size_t bstride, int batch, int cols, int rbox,
                        CUtensorMap *map) {
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (p.S & 1) || rbox < 1 || rbox > 256) return false;
    if (batch > 1 && (bstride & 1)) return false;
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    const unsigned long long nouter = (unsigned long long)p.ncols / (unsigned long long)p.S;
    cuuint64_t dims[4] = {2ull * (unsigned long long)p.S, (cuuint64_t)p.R, nouter, (cuuint64_t)batch};
    cuuint64_t strides[3] = {(cuuint64_t)p.S * 8ull, (cuuint64_t)p.R * (cuuint64_t)p.S * 8ull,
                             (cuuint64_t)(batch > 1 ? bstride : (size_t)p.R * p.S * nouter) * 8ull};
    cuuint32_t box[4] = {2u * (cuuint32_t)cols, (cuuint32_t)rbox, 1u, 1u};
    cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void *)base, dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace wefax
