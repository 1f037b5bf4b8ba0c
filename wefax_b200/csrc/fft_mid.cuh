// Real-input Hilbert transform, middle of the sandwich in ONE kernel:
//
//     last forward pass (stride 1)  ->  pair untangling  ->  first inverse pass (stride 1)
//
// All three work on engine-order rows of R = R1*R2 contiguous elements (fft_exec.cu:
// hilbert_pairs_kernel explains the pairing: the mirror M-k of frequency k = kb + ncols*j of
// row o lives in row o2 at j2 = R-1-j).  Every warp owns one (row, mirrored row) pair at a
// time: two bulk TMA copies bring the rows into shared memory, both transforms and the
// untangling run there, two bulk TMA stores write them back.  Compared with three separate
// kernels this removes two full read+write sweeps over the transform buffer.  A warp meets
// nobody (__syncwarp between the phases, no CTA-wide barrier), so the sixteen warps of an SM
// drift apart and one warp's copies hide behind the arithmetic of the others.
//
// Row transform = two register stages (fft_fast.cuh codelets):
//   stage 1  item (row, q):  R1 elements q + R2*t of the natural-order row -> DFT_R1 ->
//            * w_R^(q*u) -> block u of the exchange buffer (block pitch R2|1: conflict-free)
//   stage 2  item (row, u):  the R2 elements of block u -> DFT_R2 -> frequency u + R1*k2,
//            natural order, (inverse only) times the inter-pass twiddle w^(ko*k).
#pragma once

#include "fft_fast.cuh"

namespace wefax {
namespace fast {

template <> struct Dft<28> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<4, 7>::run(v); }
};
template <> struct Dft<20> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<4, 5>::run(v); }
};
template <> struct Dft<21> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<3, 7>::run(v); }
};
template <> struct Dft<10> {
    __device__ __forceinline__ static void run(float2 *v) { Pfa<2, 5>::run(v); }
};

struct MidRow {
    int o, o2;      // engine-order row and its mirrored row (o2 >= o; o2 == o: self-mirrored)
    int kb;         // base frequency of row o
    int pad;
};

struct MidArgs {
    float2 *z;
    size_t zs;                     // batch stride (complex elements)
    const MidRow *rows;            // npairs entries
    int npairs;                    // row pairs per sequence
    int total_tiles;               // npairs * batch
    int ncols;                     // rows per sequence
    const float2 *twR;             // w_R^e, e < R
    const float2 *twB;             // w_{2R}^j, j < R   (= w_n^(ncols*j), n = 2*ncols*R)
    const float2 *tw2_lo, *tw2_hi; // w_n^e two-level (row factor w_n^kb)
    const float2 *tw_lo, *tw_hi;   // inter-pass twiddle tables of the pass that follows the first inverse pass
    int tw_mode;                   // 2 when a pass follows (e = ko*k), 0 when R is the whole transform
    int ko_R;
    float inv_m;
};

__device__ __forceinline__ void tma_store_bulk(void *gdst, const void *ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int R1, int R2> struct MidWarpCfg {
    static constexpr int R = R1 * R2;
    static constexpr int WARPS = 4, T = 32 * WARPS;
    static constexpr int BP = R2 | 1, MIDP = R1 * BP;            // block and row pitch of the exchange buffer
    static constexpr int PER_WARP = 2 * R + 2 * MIDP + 2 * R2;   // float2: rows, exchange rows, inter-pass twiddles
    static constexpr int SMEM = (R + WARPS * PER_WARP) * (int)sizeof(float2) + WARPS * 8 + 16;
    static_assert(R % 2 == 0 && PER_WARP % 2 == 0, "bulk copies need 16-byte aligned rows");
};

// ROWS rows (R apart in nat, MIDP apart in mid) shared by T threads
template <int R1, int R2, int ROWS, int T>
__device__ __forceinline__ void mid_stage1(const float2 *nat, float2 *mid, const float2 *twQ, int tid) {
    using K = MidWarpCfg<R1, R2>;
    // G1 lanes per row (power of two >= R2): a half-warp never straddles two rows, so the 64-bit
    // shared-memory accesses stay conflict-free
    constexpr int G1 = R2 <= 16 ? 16 : 32;
    static_assert(R2 <= 32, "stage-1 lane group");
#pragma unroll 1
    for (int item = tid; item < G1 * ROWS; item += T) {
        const int row = item / G1, q = item % G1;
        if (q >= R2) continue;
        float2 v[R1];
        const float2 *src = nat + row * K::R + q;
#pragma unroll
        for (int t = 0; t < R1; ++t) v[t] = src[R2 * t];
        Dft<R1>::run(v);
        float2 *dst = mid + row * K::MIDP + q;
        const float2 *tq = twQ + q * R1;
        dst[0] = v[0];
#pragma unroll
        for (int u = 1; u < R1; ++u) dst[u * K::BP] = pcmul3(v[u], tq[u]);
    }
}

// pre_aval (optional, only when every thread has at most one item): the item's inter-pass twiddle, fetched earlier
template <int R1, int R2, bool TW, int ROWS, int T>
__device__ __forceinline__ void mid_stage2(const float2 *mid, float2 *nat, const float2 *P, const MidArgs &a,
                                           const int *s_ko, int tid, const float2 *pre_aval = nullptr) {
    using K = MidWarpCfg<R1, R2>;
    constexpr int G2 = R1 <= 16 ? 16 : 32;
    static_assert(R1 <= 32, "stage-2 lane group");
#pragma unroll 1
    for (int item = tid; item < G2 * ROWS; item += T) {
        const int row = item / G2, u = item % G2;
        if (u >= R1) continue;
        float2 Aval = make_float2(1.f, 0.f);
        if (TW) {
            if (G2 * ROWS <= T && pre_aval) {
                Aval = *pre_aval;
            } else {
                const uint32_t e = (uint32_t)s_ko[row] * (uint32_t)u;
                Aval = cmul(__ldg(a.tw_lo + (e & ((1u << kTwLoBits) - 1))), __ldg(a.tw_hi + (e >> kTwLoBits)));
            }
        }
        float2 y[R2];
        const float2 *src = mid + row * K::MIDP + u * K::BP;
#pragma unroll
        for (int t = 0; t < R2; ++t) y[t] = src[t];
        Dft<R2>::run(y);
        float2 *dst = nat + row * K::R + u;
        const float2 Aa = bc(Aval.x), Ab = make_float2(-Aval.y, Aval.y);
#pragma unroll
        for (int k2 = 0; k2 < R2; ++k2) {
            float2 val = y[k2];
            if (TW) {
                val = pcmul2(val, Aa, Ab);
                if (k2 > 0) val = pcmul3(val, P[row * R2 + k2]);
            }
            dst[R1 * k2] = val;
        }
    }
}

template <int R1, int R2>
__global__ void __launch_bounds__(128, 4)
hilbert_mid_warp_kernel(const MidArgs a) {
    using K = MidWarpCfg<R1, R2>;
    constexpr int R = K::R;
    extern __shared__ __align__(128) unsigned char mid_smem[];
    float2 *twQ = reinterpret_cast<float2 *>(mid_smem);               // [q][u] stage twiddles (shared by the warps)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float2 *nat = twQ + R + warp * K::PER_WARP;                        // [2][R] natural-order rows
    float2 *mid = nat + 2 * R;                                         // [2][R1][BP] exchange rows
    float2 *P = mid + 2 * K::MIDP;                                     // [2][R2] w^(ko*R1*k2)
    uint64_t *mbar = reinterpret_cast<uint64_t *>(twQ + R + K::WARPS * K::PER_WARP) + warp;
    __shared__ int s_ko[K::WARPS][2];

    for (int i = tid; i < R; i += K::T) {
        const int q = i / R1, u = i - q * R1;
        twQ[i] = __ldg(a.twR + q * u);
    }
    if (lane == 0) mbar_init(mbar, 1);
    __syncthreads();

    constexpr uint32_t kRowBytes = R * sizeof(float2);
    int it = 0;
    for (int tile = blockIdx.x * K::WARPS + warp; tile < a.total_tiles; tile += gridDim.x * K::WARPS, ++it) {
        const int batch = tile / a.npairs;
        const MidRow r = a.rows[tile - batch * a.npairs];
        float2 *zb = a.z + (size_t)batch * a.zs;
        const int o = r.o, o2 = r.o2 == r.o ? -1 : r.o2, kb = r.kb;
        const bool self = o2 < 0;
        if (lane == 0) {
            mbar_expect_tx(mbar, self ? kRowBytes : 2 * kRowBytes);
            tma_load_bulk(nat, zb + (size_t)o * R, kRowBytes, mbar);
            if (!self) tma_load_bulk(nat + R, zb + (size_t)o2 * R, kRowBytes, mbar);
            s_ko[warp][0] = o % a.ko_R;
            s_ko[warp][1] = self ? 0 : o2 % a.ko_R;
        }
        if (self)   // the second slot transforms zeros
            for (int i = lane; i < R; i += 32) nat[R + i] = make_float2(0.f, 0.f);
        float2 wkb;   // (inv_m / 2) * w_n^kb
        {
            const uint32_t e = (uint32_t)kb;
            const float2 wk = cmul(__ldg(a.tw2_lo + (e & ((1u << kTwLoBits) - 1))), __ldg(a.tw2_hi + (e >> kTwLoBits)));
            wkb = make_float2(wk.x * (0.5f * a.inv_m), wk.y * (0.5f * a.inv_m));
        }
        __syncwarp();
        if (a.tw_mode != 0) {
            for (int i = lane; i < 2 * R2; i += 32) {
                const int row = i / R2, k2 = i - row * R2;
                const uint32_t e = (uint32_t)s_ko[warp][row] * (uint32_t)(R1 * k2);
                P[i] = cmul(__ldg(a.tw_lo + (e & ((1u << kTwLoBits) - 1))), __ldg(a.tw_hi + (e >> kTwLoBits)));
            }
        }
        // this lane's inter-pass twiddle of the inverse pass (its one stage-2 item: row lane / G2, u = lane % G2):
        // the two table reads travel while the rows are still landing
        float2 aval = make_float2(1.f, 0.f);
        {
            constexpr int G2 = R1 <= 16 ? 16 : 32;
            const int row = lane / G2, u = lane % G2;
            if (a.tw_mode != 0 && 2 * G2 <= 32 && u < R1) {
                const uint32_t e = (uint32_t)s_ko[warp][row] * (uint32_t)u;
                aval = cmul(__ldg(a.tw_lo + (e & ((1u << kTwLoBits) - 1))), __ldg(a.tw_hi + (e >> kTwLoBits)));
            }
        }
        __syncwarp();
        mbar_wait(mbar, it & 1);

        // ---- last forward pass
        mid_stage1<R1, R2, 2, 32>(nat, mid, twQ, lane);
        __syncwarp();
        mid_stage2<R1, R2, false, 2, 32>(mid, nat, P, a, s_ko[warp], lane);
        __syncwarp();

        // ---- untangle the real-input spectrum, apply -i*sgn, re-tangle, conjugate, scale
        // With s = zk + conj(zm), d = zk - conj(zm), w = (inv_m / 2) * w_n^k:  a = conj(w) s,  b = w d,
        //   row[j]   = conj(a - b)            row2[j2] = -(a + b)
        // (the mirror's products are the conjugates of a and b, so one pair of complex multiplies serves both rows)
        {
            float2 *row = nat;
            float2 *row2 = self ? row : row + R;
#pragma unroll 2
            for (int j = lane; j < R; j += 32) {
                const int j2 = kb ? R - 1 - j : (j ? R - j : 0);
                if (self && j2 < j) continue;
                if (kb == 0 && j == 0) {
                    row[0] = make_float2(0.f, 0.f);
                    continue;
                }
                const float2 zk = row[j], zm = row2[j2];
                const float2 w = pcmul3(__ldg(a.twB + j), wkb);                       // (inv_m / 2) * w_n^k, k = kb + ncols*j
                const float2 sp = pfma(zm, make_float2(1.f, -1.f), zk);                 // zk + conj zm
                const float2 dm = pfma(zm, make_float2(-1.f, 1.f), zk);                 // zk - conj zm
                const float2 wa = bc(w.x);
                const float2 aa = pfma(sp, wa, pmul(swp(sp), make_float2(w.y, -w.y)));  // conj(w) * sp
                const float2 bb = pfma(dm, wa, pmul(swp(dm), make_float2(-w.y, w.y)));  // w * dm
                row[j] = pmul(psub(aa, bb), make_float2(1.f, -1.f));
                if (!(self && j2 == j)) row2[j2] = pmul(padd(aa, bb), make_float2(-1.f, -1.f));
            }
        }
        __syncwarp();

        // ---- first inverse pass (forward kernels on conjugated data)
        mid_stage1<R1, R2, 2, 32>(nat, mid, twQ, lane);
        __syncwarp();
        if (a.tw_mode != 0)
            mid_stage2<R1, R2, true, 2, 32>(mid, nat, P, a, s_ko[warp], lane, &aval);
        else
            mid_stage2<R1, R2, false, 2, 32>(mid, nat, P, a, s_ko[warp], lane);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            tma_store_bulk(zb + (size_t)o * R, nat, kRowBytes);
            if (!self) tma_store_bulk(zb + (size_t)o2 * R, nat + R, kRowBytes);
            tma_store_commit();
            tma_store_wait_read();   // the rows may be overwritten by the next pair's loads
        }
        __syncwarp();
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

inline bool mid_pair(int R, int *R1, int *R2) {
    static const int pairs[][2] = {{14, 28}, {10, 14}, {15, 20}, {10, 15}, {14, 15}};   // keep in step with hilbert_envelope_real (fft_exec.cu)
    for (auto &pr : pairs)
        if (pr[0] * pr[1] == R) {
            if (R1) *R1 = pr[0];
            if (R2) *R2 = pr[1];
            return true;
        }
    return false;
}

}  // namespace fast
}  // namespace wefax
