// sweep_fused.cuh — ONE kernel for the whole candidate sweep of a scalar GP (p = 1):
//     K(X*, X) tile  ->  W = L^-1 K*^T on the FP64 tensor pipe  ->  sum_i W_ic^2 (variance) and sum_i W_ic beta_i
//     (mean: k*^T alpha = (L^-1 k*)^T (L^-1 delta))  ->  EI / PI / UCB  ->  scores
// replacing the three launches per chunk of the large-n path (ks_build_kernel, gemm_tma_kernel<EPI_COLSUMSQ>,
// acq_epilogue_kernel) and the HBM round trip of the K* chunk between them.
// Reference call sites: acq(surrogate, grid) in optimize_acquisition (acq_utils.jl:44-52) ->
// ExpectedImprovement.jl:40-66 / ProbabilityImprovement.jl:38-63 / UpperConfidenceBound.jl:38-45 ->
// posterior_mean / posterior_var (StandardGP.jl:361-379).
//
// Persistent, one CTA per SM; a CTA OWNS whole candidate tiles (128 candidates) and walks all row tiles
// of L^-1 for them, so
//   * the K* tile (128 x n) of a candidate tile is private to its CTA: the eight DMMA warps BUILD the tile
//     of the CTA's next candidate tile into a double-buffered private scratch (2 x 128 x ceil16(n) doubles per
//     CTA, written once and read back by TMA; it stays in L2 only for small n: 4 MiB per CTA at n = 2048, 32 MiB
//     at n = 16384) before contracting the current one — the kernel
//     evaluations and the DMMA work share the FP64 pipe anyway, so running them back to back in the same
//     warps loses nothing and needs no cross-CTA synchronisation;
//   * every candidate tile costs the same, so the static schedule tile = b, b + G, ... is balanced;
//   * the column sums accumulate across row tiles in shared memory: no [T][m] partial array, no epilogue launch.
// The TMA producer warp runs ahead across row tiles and candidate tiles (5-stage full/empty mbarrier ring);
// it waits on a `built` mbarrier before the first load of a candidate tile; the builders order their
// generic-proxy stores before the async-proxy (TMA) reads with fence.proxy.async.
// k runs over ceil16(n) columns only and the row fragments of a tile are dealt to the warps interleaved
// (fragment f = 4 i + q to warp q), so a partial last row tile costs ceil(rows / 32) / 4 of a full one:
// no padding of n to 128 in the executed work.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>
#include <type_traits>

#include "kernels.cuh"
#include "tma_pipe.cuh"

namespace abo {

constexpr int FS_STAGES = 5;
constexpr int FS_THREADS = 256 + 32;
// Largest padded system (Npad) of a scalar GP that takes the fused sweep; larger systems take the three-kernel path.  The
// bound is the private K* scratch, 2 x 128 x Kld x 8 B per CTA, allocated for every SM: 32 MiB per CTA and 4.97 GB on 148 SMs
// at n = 16384.
constexpr int64_t FS_MAX_NPAD = 16384;

struct FusedParams {
    KSpec spec;
    AcqSpec acq;
    const double* XsT;      // scaled training coordinates, coordinate-major [d][ldx]
    int64_t ldx;
    int64_t n;              // observations (= system size, p == 1)
    int T;                  // row tiles of L^-1
    int Kld;                // ceil16(n): k extent and row stride of the K* scratch
    const double* Xc;       // candidates, point-major [m][d] (device)
    int64_t m;
    const double* beta;     // L^-1 (y - mean), zero in the padding
    double* scratch;        // [gridDim.x][2][128][Kld]
    double* mean_out;       // each nullable, length m
    double* var_out;
    double* score_out;
    int ntiles;             // candidate tiles = ceil(m / 128)
};

template <int DT>
constexpr int fused_smem_bytes() {
    return FS_STAGES * SW_STAGE_BYTES + 128 * DT * 8 + 2 * 4 * 128 * 8 + 2 * 128 * 8 + (2 * FS_STAGES + 2) * 8 + 128;
}

__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;\n" ::: "memory"); }
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }

// one k16 stage of the 128 x 128 product; fragment rows interleaved: warp q owns rows 8 (4 i + q) + fr.  Only the row
// fragments ilo <= i < ihi of this warp are live; partial ranges occur in the last row tile of a system that is not a
// multiple of 128, and inside the diagonal block (rows above the diagonal).
__device__ __forceinline__ void fused_stage_range(const double* __restrict__ a_s, const double* __restrict__ b_s, double (&acc)[4][8][2],
                                                  int ilo, int ihi) {
    switch (ilo * 5 + ihi) {
        case 0 * 5 + 4: dmma_stage<0, 4, 128>(a_s, b_s, acc); break;
        case 0 * 5 + 3: dmma_stage<0, 3, 128>(a_s, b_s, acc); break;
        case 0 * 5 + 2: dmma_stage<0, 2, 128>(a_s, b_s, acc); break;
        case 0 * 5 + 1: dmma_stage<0, 1, 128>(a_s, b_s, acc); break;
        case 1 * 5 + 4: dmma_stage<1, 4, 128>(a_s, b_s, acc); break;
        case 1 * 5 + 3: dmma_stage<1, 3, 128>(a_s, b_s, acc); break;
        case 1 * 5 + 2: dmma_stage<1, 2, 128>(a_s, b_s, acc); break;
        case 2 * 5 + 4: dmma_stage<2, 4, 128>(a_s, b_s, acc); break;
        case 2 * 5 + 3: dmma_stage<2, 3, 128>(a_s, b_s, acc); break;
        case 3 * 5 + 4: dmma_stage<3, 4, 128>(a_s, b_s, acc); break;
        default: break;                                              // empty range
    }
}

// kernel profile value by FAMILY (0: SE, 1: Matern-5/2 kinds, 2: Matern-7/2 kinds): the family switch is taken once per
// candidate tile, not once per entry (ncu: the per-entry dispatch branches and their re-convergence were ~15 % of the
// builder's issue slots, plus instruction-cache misses on three inlined copies of the profile code)
template <int FAM>
__device__ __forceinline__ double phi_value(int kind, double u) {
    if (FAM == 0) return exp(-u / 2);
    const double r = sqrt(u);
    if (FAM == 1) {
        const double q5 = 2.23606797749978969641;
        const double v = (1 + q5 * r + u * (5.0 / 3.0)) * exp(-q5 * r);          // 5 u / 3 without the FP64 division (1 ulp of one term)
        return (kind == K_AM52 && u < 1e-10) ? 1.0 - (5.0 / 6.0) * u : v;
    }
    const double q7 = 2.64575131106459059050;
    const double v = (1 + q7 * r + u * (14.0 / 5.0) + (7.0 / 15.0) * q7 * r * u) * exp(-q7 * r);
    return (kind == K_AM72 && u < 1e-10) ? 1.0 - (7.0 / 10.0) * u : v;
}

template <int DT>
__global__ void __launch_bounds__(FS_THREADS, 1)
sweep_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const FusedParams p) {
    extern __shared__ __align__(128) unsigned char fs_smem[];
    double* stage_base = reinterpret_cast<double*>(fs_smem);
    double* sc = reinterpret_cast<double*>(fs_smem + FS_STAGES * SW_STAGE_BYTES);        // [128][DT] scaled candidate coordinates
    double* red = sc + 128 * DT;                                                           // [2][4][128]
    double* qacc = red + 2 * 4 * 128;                                                      // [128] sum of squares so far
    double* macc = qacc + 128;                                                             // [128] w . beta so far
    uint64_t* full = reinterpret_cast<uint64_t*>(macc + 128);
    uint64_t* empty = full + FS_STAGES;
    uint64_t* built = empty + FS_STAGES;                                                   // [2]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x, b = blockIdx.x;
    const int ntl = (b < p.ntiles) ? (p.ntiles - b + G - 1) / G : 0;                       // candidate tiles of this CTA
    const int nk_max = p.Kld / 16;

    if (tid == 0) {
        for (int s = 0; s < FS_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        mbar_init(&built[0], 1); mbar_init(&built[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (tid < 128) { qacc[tid] = 0.0; macc[tid] = 0.0; }
    __syncthreads();

    if (warp == 8) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int j = 0; j < ntl; ++j) {
                mbar_wait(&built[j & 1], (uint32_t)((j >> 1) & 1));                       // K* tile of candidate tile j is in the scratch
                const int brow = (b * 2 + (j & 1)) * 128;
                for (int ib = 0; ib < p.T; ++ib) {
                    const int nk = min((ib + 1) * 8, nk_max);
                    const int m0 = ib * 128;
                    for (int kt = 0; kt < nk; ++kt) {
                        mbar_wait(&empty[stage], phase ^ 1);
                        tma_stage_load(stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES), &full[stage], &tmA, kt * 16, m0,
                                       &tmB, kt * 16, brow);
                        if (++stage == FS_STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
        return;
    }

    // ------------------------------ builders / DMMA consumers (warps 0..7) ------------------------------
    const int q = warp & 3, wn = (warp >> 2) * 64;
    const int fr = lane >> 2, fk = lane & 3;
    const int d = p.spec.d;
    const int64_t n = p.n;
    double* my_scratch = p.scratch + (size_t)b * 2 * 128 * p.Kld;

    // zero the k-padding columns [n, Kld) of both scratch tiles once (they meet zero columns of L^-1, but must be finite)
    {
        const int padw = p.Kld - (int)n;
        for (int e = tid; e < 2 * 128 * padw; e += 256) my_scratch[(size_t)(e / padw) * p.Kld + n + (e % padw)] = 0.0;
    }

    // K* tile of candidate tile j -> scratch slot j & 1.  Work items of (32 training points) x (32 candidates), lane = point
    // (coalesced 256-byte stores along k); BCU candidates in flight per lane: with two warps per scheduler that is 2 x BCU
    // independent FP64 chains, enough to cover the DADD -> DFMA latency (4 left the FP64 pipe ~50 % idle, ncu stall_wait).
    constexpr int BCU = 8;
    auto build = [&](int j) {
        const int64_t c_base = ((int64_t)b + (int64_t)j * G) * 128;
        double* tile = my_scratch + (size_t)(j & 1) * 128 * p.Kld;
        for (int e = tid; e < 128 * DT; e += 256) {
            const int c = e / DT, k = e - c * DT;
            const int64_t gc = c_base + c;
            sc[e] = (k < d && gc < p.m) ? p.spec.sk(k) * p.Xc[gc * d + k] : 0.0;
        }
        bar_consumers();
        const int nitems = (int)((n + 31) / 32) * 4;
        auto items = [&](auto fam_tag) {
            constexpr int FAM = decltype(fam_tag)::value;
            constexpr bool PREF = DT <= 12;                           // next item's coordinates loaded one item ahead (register budget)
            double xn[PREF ? DT : 1];
            if (PREF) {
                const int64_t i0 = (int64_t)(warp >> 2) * 32 + lane;
#pragma unroll
                for (int k = 0; k < DT; ++k) xn[PREF ? k : 0] = (k < d && i0 < n && warp < nitems) ? p.XsT[(int64_t)k * p.ldx + i0] : 0.0;
            }
            for (int item = warp; item < nitems; item += 8) {
                const int64_t i = (int64_t)(item >> 2) * 32 + lane;
                const int c0 = (item & 3) * 32;
                const bool live = i < n;
                double x[DT];
                if (PREF) {
#pragma unroll
                    for (int k = 0; k < DT; ++k) x[k] = xn[PREF ? k : 0];
                    const int64_t i2 = (int64_t)((item + 8) >> 2) * 32 + lane;
                    const bool nxt = (item + 8 < nitems) && i2 < n;
#pragma unroll
                    for (int k = 0; k < DT; ++k) xn[PREF ? k : 0] = (k < d && nxt) ? p.XsT[(int64_t)k * p.ldx + i2] : 0.0;
                } else {
#pragma unroll
                    for (int k = 0; k < DT; ++k) x[k] = (k < d && live) ? p.XsT[(int64_t)k * p.ldx + i] : 0.0;
                }
                double* col = tile + i;
#pragma unroll 1
                for (int c = c0; c < c0 + 32; c += BCU) {
                    double u[BCU];
#pragma unroll
                    for (int r = 0; r < BCU; ++r) u[r] = 0.0;
#pragma unroll
                    for (int k = 0; k < DT; ++k) {
#pragma unroll
                        for (int r = 0; r < BCU; ++r) { const double df = x[k] - sc[(c + r) * DT + k]; u[r] = fma(df, df, u[r]); }
                    }
#pragma unroll
                    for (int r = 0; r < BCU; ++r) {
                        const double v = p.spec.scale * phi_value<FAM>(p.spec.kind, u[r]);
                        if (live) col[(size_t)(c + r) * p.Kld] = v;
                    }
                }
            }
        };
        const int kind = p.spec.kind;
        if (kind == K_SE) items(std::integral_constant<int, 0>{});
        else if (kind == K_M52 || kind == K_AM52 || kind == K_ADM52) items(std::integral_constant<int, 1>{});
        else items(std::integral_constant<int, 2>{});
        fence_proxy_async_global();                                   // generic-proxy stores before the TMA (async-proxy) reads
        __threadfence();
        bar_consumers();
        if (tid == 0) mbar_arrive(&built[j & 1]);
    };

    int stage = 0;
    uint32_t phase = 0;
    for (int j = -1; j < ntl; ++j) {
        if (j + 1 < ntl) build(j + 1);                                // one tile ahead of the contraction (single call site: one copy of the code)
        if (j < 0) continue;
        const int64_t c_base = ((int64_t)b + (int64_t)j * G) * 128;
        for (int ib = 0; ib < p.T; ++ib) {
            const int nk = min((ib + 1) * 8, nk_max);
            const int m0 = ib * 128;
            const int rows = (int)min((int64_t)128, n - m0);          // live rows of this tile (the rest is identity padding: W = 0)
            const int nfrag = (rows + 7) >> 3;
            const int ni = max(0, min(4, (nfrag - q + 3) >> 2));      // live fragments of this warp (f = 4 i + q < nfrag)
            double acc[4][8][2];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) { acc[i][jj][0] = 0.0; acc[i][jj][1] = 0.0; }
            const int a_off = ((8 * q + fr) << 2) + fk;
            const int b_off = SW_OPER_DOUBLES + ((wn + fr) << 2) + fk;
            // k16 steps left of the diagonal block: every live row fragment; inside the diagonal block (k0 = m0 + 16 t) only the
            // rows >= k0 are non-zero in L^-1: fragments f >= 2 t, i.e. i >= ceil((2 t - q) / 4) for this warp — the
            // upper-triangle half of the diagonal tile is never multiplied (it is (T + 1) / T of the work at T row tiles)
            const int nk_full = (rows == 128) ? min(nk, ib * 8) : 0;
            for (int kt = 0; kt < nk_full; ++kt) {
                mbar_wait(&full[stage], phase);
                const double* st = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
                dmma_stage<0, 4, 128>(st + a_off, st + b_off, acc);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == FS_STAGES) { stage = 0; phase ^= 1; }
            }
            for (int kt = nk_full; kt < nk; ++kt) {
                mbar_wait(&full[stage], phase);
                const double* st = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
                const int t = kt - ib * 8;                            // < 0 left of the diagonal block
                const int ilo = t > 0 ? max(0, (2 * t - q + 3) >> 2) : 0;
                fused_stage_range(st + a_off, st + b_off, acc, ilo, ni);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == FS_STAGES) { stage = 0; phase ^= 1; }
            }
            // ---- tile epilogue: column sums of W^2 and of W * beta over the tile's rows
            double bt[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) bt[i] = p.beta[m0 + 8 * (4 * i + q) + fr];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    double s2 = 0.0, sm = 0.0;
#pragma unroll
                    for (int i = 0; i < 4; ++i) { s2 = fma(acc[i][jj][e], acc[i][jj][e], s2); sm = fma(acc[i][jj][e], bt[i], sm); }
                    s2 += __shfl_xor_sync(0xffffffffu, s2, 4);  sm += __shfl_xor_sync(0xffffffffu, sm, 4);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, 8);  sm += __shfl_xor_sync(0xffffffffu, sm, 8);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, 16); sm += __shfl_xor_sync(0xffffffffu, sm, 16);
                    if (fr == 0) {
                        const int col = wn + jj * 8 + 2 * fk + e;
                        red[q * 128 + col] = s2;
                        red[512 + q * 128 + col] = sm;
                    }
                }
            }
            bar_consumers();
            if (tid < 128) {
                qacc[tid] += ((red[tid] + red[128 + tid]) + red[256 + tid]) + red[384 + tid];
                macc[tid] += ((red[512 + tid] + red[640 + tid]) + red[768 + tid]) + red[896 + tid];
            }
            bar_consumers();
        }
        // ---- candidate-tile epilogue: mean, variance (+1e-18), acquisition in the reference's operation order
        if (tid < 128) {
            const int64_t gc = c_base + tid;
            if (gc < p.m) {
                const double mu = macc[tid] + p.acq.mean_c;
                const double var = (p.acq.kss - qacc[tid]) + JITTER;
                if (p.mean_out) p.mean_out[gc] = mu;
                if (p.var_out) p.var_out[gc] = var;
                if (p.score_out && p.acq.acq >= 0) p.score_out[gc] = acq_value(p.acq, mu, var);
            }
            qacc[tid] = 0.0; macc[tid] = 0.0;
        }
    }
}

}  // namespace abo
