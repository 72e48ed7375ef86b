// kernels.cuh — the non-GEMM device code of libabo_cuda: kernel profiles, kernel-matrix
// construction (value and derivative blocks), the 128x128 diagonal-block factor+inverse, the
// cross-kernel K(X*, X) tile builder with fused posterior-mean partials, the acquisition
// epilogue and a few O(n^2) vector kernels.
//
// Index conventions on the device
//   system index  idx = i * p + a   (POINT-major: point i, output a; a = 0 value, a >= 1 d/dx_a)
//   — the reference's out-major order (GradientGP.jl:919-922) only exists at the ABI.
//   Coordinates are stored pre-scaled (s * x, ScaleTransform first — SURVEY H4) and
//   coordinate-major:  XsT[k * ldx + i].
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "gemm_dmma.cuh"

namespace abo {

constexpr int NB = 128;                 // tile / panel width everywhere
constexpr double JITTER = 1e-18;        // AbstractGPs default_σ² (StandardGP.jl:361-379 via FiniteGP)

enum KernelId { K_SE = 0, K_M52 = 1, K_M72 = 2, K_AM52 = 3, K_AM72 = 4, K_ADM52 = 5, K_ADM72 = 6 };
enum AcqId { ACQ_EI = 0, ACQ_PI = 1, ACQ_UCB = 2 };

constexpr int ARD_MAXD = 32;
struct KSpec {
    int kind, d, p;
    double s, scale, noise;      // s: the isotropic ScaleTransform 1/l (also what the d > 32 kernels use)
    double sv[ARD_MAXD];         // per-dimension inverse length scales s_k = 1/l_k (ARD; all equal to s for an isotropic kernel)
    __host__ __device__ __forceinline__ double sk(int k) const { return d <= ARD_MAXD ? sv[k] : s; }
};

// phi(u), phi'(u), phi''(u), u = squared scaled distance.
// SE: KernelFunctions SqExponentialKernel; Matern: KernelFunctions Matern52/72Kernel and
// src/surrogates/GradientGP.jl:94-101,176-209,320-327,400-437 (Approx: Taylor branch u < 1e-10).
__device__ __forceinline__ void phi_eval(int kind, double u, double& p, double& dp, double& ddp) {
    if (kind == K_SE) {
        p = exp(-u / 2);
        dp = -p / 2;
        ddp = p / 4;
        return;
    }
    const double r = sqrt(u);
    if (kind == K_M52 || kind == K_AM52 || kind == K_ADM52) {
        const double q5 = 2.23606797749978969641;   // sqrt(5)
        if (kind == K_AM52 && u < 1e-10) { p = 1.0 - (5.0 / 6.0) * u; dp = -5.0 / 6.0; ddp = 0.0; return; }
        const double z = exp(-q5 * r);
        p = (1 + q5 * r + 5 * u / 3) * z;
        dp = (-5.0 / 6.0) * (1 + q5 * r) * z;
        ddp = (25.0 / 12.0) * z;
        return;
    }
    const double q7 = 2.64575131106459059050;       // sqrt(7)
    if (kind == K_AM72 && u < 1e-10) { p = 1.0 - (7.0 / 10.0) * u; dp = -7.0 / 10.0; ddp = 0.0; return; }
    const double z = exp(-q7 * r);
    p = (1 + q7 * r + 14 * u / 5 + 7 * q7 * r * u / 15) * z;
    dp = (-7.0 / 10.0) * (1 + q7 * r + 7 * u / 3) * z;
    ddp = (49.0 / 60.0) * (1 + q7 * r) * z;
}

// gradKernel entry (src/surrogates/GradientGP.jl:573-606) in closed form; D = s*(x - y).
//   (0,0) sig2 phi ; (a,0) 2 s_a sig2 phi' D_a ; (0,b) -2 s_b sig2 phi' D_b ;
//   (a,b) -sig2 [ 4 s_a s_b phi'' D_a D_b + 2 s_a^2 phi' delta_ab ]        (s_a = s for an isotropic kernel)
__device__ __forceinline__ double gk_entry(const KSpec& ks, double p, double dp, double ddp, int a, int b,
                                           double Da, double Db) {
    if (a == 0 && b == 0) return ks.scale * p;
    if (b == 0) return 2 * ks.sk(a - 1) * ks.scale * dp * Da;
    if (a == 0) return -2 * ks.sk(b - 1) * ks.scale * dp * Db;
    const double sa = ks.sk(a - 1), sb = ks.sk(b - 1);
    return -ks.scale * (4 * sa * sb * ddp * Da * Db + (a == b ? 2 * sa * sa * dp : 0.0));
}

// ------------------------------------------------------------------------------------------
// coordinates:  XsT[k*ldx + i] = s * X[i*d + k]
// ------------------------------------------------------------------------------------------
__global__ void scale_transpose_kernel(const double* __restrict__ X, double* __restrict__ XsT, int64_t n,
                                       int d, int64_t ldx, KSpec spec) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ldx * d) return;
    int k = (int)(t / ldx);
    int64_t i = t % ldx;
    XsT[t] = (i < n) ? spec.sk(k) * X[i * d + k] : 0.0;
}

// ------------------------------------------------------------------------------------------
// K + noise*I, lower tiles, identity in the padding  (StandardGP.jl:80, GradientGP.jl:662-665)
// grid (T, T, batch); tile (blockIdx.y, blockIdx.x), skipped above the diagonal.
// Batched form (NLML restarts): per-batch KSpec parameters come from arrays.
// ------------------------------------------------------------------------------------------
struct KmatBatch {
    const double* s;       // per batch inverse lengthscale (nullptr: use spec.s); with ARD: [batch][d] (see `ard`)
    const double* scale;   // per batch sigma^2
    int64_t strideX;       // XsT stride per batch
    int64_t strideK;
    int ard;               // 1: s holds d inverse length scales per batch
};
// hyper-parameters of batch entry z into the by-value KSpec copy of a kernel
__device__ __forceinline__ void apply_batch(KSpec& spec, const KmatBatch& bt, int z) {
    if (!bt.s) return;
    spec.scale = bt.scale[z];
    if (bt.ard) {
        for (int k = 0; k < spec.d && k < ARD_MAXD; ++k) spec.sv[k] = bt.s[(int64_t)z * spec.d + k];
        spec.s = spec.sv[0];
    } else {
        spec.s = bt.s[z];
        for (int k = 0; k < ARD_MAXD; ++k) spec.sv[k] = spec.s;
    }
}

__global__ void __launch_bounds__(256) kmat_kernel(KSpec spec, const double* __restrict__ XsT, int64_t ldx,
                                                   int64_t N, double* __restrict__ Kmat, int64_t ld,
                                                   KmatBatch bt) {
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    apply_batch(spec, bt, blockIdx.z);
    const double* X = XsT + (int64_t)blockIdx.z * bt.strideX;
    double* Kb = Kmat + (int64_t)blockIdx.z * bt.strideK;
    const int c = threadIdx.x & 127;
    const int64_t gc = (int64_t)bj * NB + c;
    const bool p1 = spec.p == 1;                       // scalar GP: no 64-bit divisions in the entry loop
    const int64_t j = p1 ? gc : gc / spec.p;
    const int b = p1 ? 0 : (int)(gc % spec.p);
    for (int r = threadIdx.x >> 7; r < NB; r += 2) {
        const int64_t gr = (int64_t)bi * NB + r;
        double v;
        if (gr >= N || gc >= N) {
            v = (gr == gc) ? 1.0 : 0.0;
        } else {
            const int64_t i = p1 ? gr : gr / spec.p;
            const int a = p1 ? 0 : (int)(gr % spec.p);
            double u = 0.0, Da = 0.0, Db = 0.0;
            for (int k = 0; k < spec.d; ++k) {
                double df = X[k * ldx + i] - X[k * ldx + j];
                u = fma(df, df, u);
                if (k == a - 1) Da = df;
                if (k == b - 1) Db = df;
            }
            double p, dp, ddp;
            phi_eval(spec.kind, u, p, dp, ddp);
            v = gk_entry(spec, p, dp, ddp, a, b, Da, Db);
            if (gr == gc) v += spec.noise;
        }
        Kb[gr * ld + gc] = v;
    }
}

// scalar GP (p = 1), d <= DT: the same tile with the coordinates in registers / shared memory.  A thread owns CPT
// columns (x_j in registers) and walks the rows of its row group (x_i broadcast from shared memory), so one shared
// load feeds CPT distance terms and there is no index arithmetic in the entry loop.  Bit-identical to kmat_kernel
// (same k order; the zero padding of the coordinates adds exact zeros).
template <int DT, int CPT>
__global__ void __launch_bounds__(256) kmat_p1_kernel(KSpec spec, const double* __restrict__ XsT, int64_t ldx, int64_t N,
                                                      double* __restrict__ Kmat, int64_t ld, KmatBatch bt) {
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    apply_batch(spec, bt, blockIdx.z);
    const double* X = XsT + (int64_t)blockIdx.z * bt.strideX;
    double* Kb = Kmat + (int64_t)blockIdx.z * bt.strideK;
    __shared__ double sxi[DT][NB];
    const int tid = threadIdx.x;
    for (int e = tid; e < DT * NB; e += 256) {
        const int k = e >> 7, r = e & 127;
        const int64_t gr = (int64_t)bi * NB + r;
        sxi[k][r] = (k < spec.d && gr < N) ? X[k * ldx + gr] : 0.0;
    }
    constexpr int TPG = NB / CPT, NG = 256 / TPG, RPG = NB / NG;
    const int tg = tid % TPG, grp = tid / TPG;
    double xj[CPT][DT];
#pragma unroll
    for (int q = 0; q < CPT; ++q) {
        const int64_t gc = (int64_t)bj * NB + tg + q * TPG;
#pragma unroll
        for (int k = 0; k < DT; ++k) xj[q][k] = (k < spec.d && gc < N) ? X[k * ldx + gc] : 0.0;
    }
    __syncthreads();
    for (int rr = 0; rr < RPG; ++rr) {
        const int r = grp * RPG + rr;
        const int64_t gr = (int64_t)bi * NB + r;
        double u[CPT];
#pragma unroll
        for (int q = 0; q < CPT; ++q) u[q] = 0.0;
#pragma unroll
        for (int k = 0; k < DT; ++k) {
            const double xi = sxi[k][r];
#pragma unroll
            for (int q = 0; q < CPT; ++q) { const double df = xi - xj[q][k]; u[q] = fma(df, df, u[q]); }
        }
#pragma unroll
        for (int q = 0; q < CPT; ++q) {
            const int64_t gc = (int64_t)bj * NB + tg + q * TPG;
            double v;
            if (gr >= N || gc >= N) {
                v = (gr == gc) ? 1.0 : 0.0;
            } else {
                double p, dp, ddp;
                phi_eval(spec.kind, u[q], p, dp, ddp);
                v = spec.scale * p;
                if (gr == gc) v += spec.noise;
            }
            Kb[gr * ld + gc] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// 128 x 128 diagonal block of the blocked Cholesky:  A = L L^T in shared memory and L^-1 of the
// block.  Writes L (upper part zeroed) back in place and L^-1 to Dinv.  A non-positive pivot
// sets *info (1-based global pivot, first failure wins).  One CTA of 512 threads per matrix
// (blockIdx.x = batch).
// ------------------------------------------------------------------------------------------
__device__ long long g_potf2_clk[16];     // phase timestamps of CTA 0 of the last launch (inspection)
constexpr int POTF2_LD = 129;                                    // block [128][129]
constexpr int POTF2_PLD = 132;                                   // sub-panel buffer [32][132]

// ------------------------------------------------------------------------------------------
// potf2_ws_kernel — warp-specialised diagonal-block kernel: the FACTOR group (warps 0-7) runs the
// Cholesky of the 128 x 128 block (four 32-column sub-panels, see the comments inside), while
// the INVERSE group (warps 8-15) builds L^-1 one 32-row block behind it:
//     round s (after the diagonal block D_s is final):
//        X_ss = inv(D_s)                              (8x8 scalar level + two DMMA levels)
//        S_st = sum_{u=t}^{s-1} L_su X_ut   (t < s)   (DMMA, X_ut read back from global Dinv)
//        X_st = - X_ss S_st                           (DMMA)  -> global Dinv
// so that when the last diagonal block is done only X_33 and one multiply remain, overlapped with
// the write-back of L.  Groups synchronise internally with named barriers (1: factor, 2: inverse);
// the factor group never waits for the inverse group: it only ARRIVES on per-round barriers
// (4+s: D_s final, 8+s: rows below column block s final) that the inverse group syncs on.
// ------------------------------------------------------------------------------------------
constexpr int PW_XLD = 36;
constexpr int PW_F_SCRATCH = 32 * POTF2_PLD + 64 + 2 * 32 + 2 * 32 * 32;    // panel | col ping-pong | 1/diag x 2 | D^T x 2 (look-ahead)
constexpr int PW_I_SCRATCH = 32 * PW_XLD + 3 * 32 * PW_XLD + 320;            // X_ss | S_s0..S_s2 | T of the 32-block levels
constexpr int PW_SMEM_BYTES = (128 * POTF2_LD + PW_F_SCRATCH + PW_I_SCRATCH + 16) * (int)sizeof(double);

__device__ __forceinline__ void bar_named(int id, int count) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}

__global__ void __launch_bounds__(512) potf2_ws_kernel(double* __restrict__ Ablk, int64_t ld, int64_t strideA,
                                                       double* __restrict__ Dinv, int64_t strideD,
                                                       int* __restrict__ info, int pivot_base) {
    extern __shared__ __align__(16) double sm[];
    double* sL = sm;                                   // [128][129]
    double* sP = sm + 128 * POTF2_LD;                  // factor group: panel [32][132]
    double* sCol = sP + 32 * POTF2_PLD;                // two 32-entry column buffers
    double* sRinv = sCol + 64;                         // reciprocals of the block's diagonal, two sub-panels (ping-pong)
    double* sDT = sRinv + 2 * 32;                      // transposed diagonal block [32][32], two sub-panels
    double* sXs = sDT + 2 * 32 * 32;                   // inverse group: X_ss [32][36]
    double* sS = sXs + 32 * PW_XLD;                    // S_st, t = 0..2, [32][36] each
    double* sTi = sS + 3 * 32 * PW_XLD;                // T staging of the levels inside a 32-block
    __shared__ int s_fail;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5, fr = lane >> 2, fk = lane & 3;
    double* A = Ablk + (int64_t)blockIdx.x * strideA;
    double* Di = Dinv + (int64_t)blockIdx.x * strideD;
    if (tid == 0) s_fail = 0;
    pdl_launch_dependents();
    pdl_wait();
    const bool stamp = (tid == 0 && blockIdx.x == 0);
    if (stamp) g_potf2_clk[0] = clock64();
    // warps 1..15 stage the block in shared memory; warp 0 takes the first diagonal block D_0 straight
    // from global memory into registers and factors it meanwhile (its result is what everybody waits for)
    if (warp > 0) {
        // 16-byte loads, eight in flight per thread before the first shared-memory store: the staging must not be a chain of
        // dependent global-memory latencies (it gates the first substitution: everybody waits for "block staged AND D_0 final")
        constexpr int NV = 128 * 64;                       // double2 elements of the block
        for (int e0 = tid - 32; e0 < NV; e0 += 480 * 8) {
            double2 v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int e = e0 + q * 480;
                if (e < NV) v[q] = *reinterpret_cast<const double2*>(A + (int64_t)(e >> 6) * ld + 2 * (e & 63));
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int e = e0 + q * 480;
                if (e < NV) {
                    const int r = e >> 6, c = 2 * (e & 63);
                    if (r >= 32 || c >= 32) { sL[r * POTF2_LD + c] = v[q].x; sL[r * POTF2_LD + c + 1] = v[q].y; }
                }
            }
        }
    }
    if (stamp) g_potf2_clk[1] = clock64();

    if (warp < 8) {
        // =============================== FACTOR GROUP ===============================
        // Look-ahead inside the block: warp 0 only factors the 32 x 32 diagonal blocks.  As soon as D_sp is final the other
        // seven warps substitute the rows below it; the three 16 x 16 tiles of the trailing update that make up the NEXT
        // diagonal block go first (warps 1-3, one tile each) and release warp 0 into diag(sp + 1), which then runs concurrently
        // with the write-back of column block sp and the rest of the rank-32 update.  The chain per sub-panel is
        // diag -> substitution -> one tile -> diag instead of diag -> substitution -> write-back -> whole update -> diag.
        //   named barriers: 1 "D_sp final" (warp 0 arrives, 256) | 3 "panel substituted" (warps 1-7, 224)
        //                   12 "next diagonal block updated" (warps 1-3 arrive, warp 0 syncs, 128) | 13 "update done" (warps 1-7, 224)
        for (int sp = 0; sp < 4; ++sp) {
            const int c0 = sp * 32, c1 = c0 + 32;
            double* sDTp = sDT + (sp & 1) * (32 * 32);     // ping-pong: warp 0 runs one sub-panel ahead of the readers
            double* sRinvp = sRinv + (sp & 1) * 32;
            if (warp == 0) {
                if (sp > 0) bar_named(12, 128);            // block (c0..c1)^2 carries the updates of all previous sub-panels
                if (stamp && sp == 1) g_potf2_clk[5] = clock64();
                double a[32];
                if (sp == 0) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) a[c] = A[(int64_t)lane * ld + c];
                } else {
#pragma unroll
                    for (int c = 0; c < 32; ++c) a[c] = sL[(c0 + lane) * POTF2_LD + c0 + c];
                }
                int failcol = -1;
                double d = __shfl_sync(0xffffffffu, a[0], 0);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (failcol < 0 && !(d > 0.0)) failcol = j;
                    const double rinv = rsqrt(d);
                    const double lj = (lane == j) ? d * rinv : a[j] * rinv;
                    a[j] = lj;
                    if (j < 31) {
                        const double own = fma(-lj, lj, a[(j + 1) & 31]);
                        d = __shfl_sync(0xffffffffu, own, (j + 1) & 31);
                    }
                    if (lane == j) sRinvp[j] = rinv;
                    double* col = sCol + (j & 1) * 32;
                    col[lane] = lj;
                    __syncwarp();
#pragma unroll
                    for (int c2 = 0; c2 < 16; ++c2) {
                        if (2 * c2 + 1 > j) {
                            const double2 lc = *reinterpret_cast<const double2*>(col + 2 * c2);
                            if (2 * c2 > j) a[2 * c2] = fma(-lj, lc.x, a[2 * c2]);
                            a[2 * c2 + 1] = fma(-lj, lc.y, a[2 * c2 + 1]);
                        }
                    }
                }
                if (failcol >= 0) {
                    if (lane == 0) { s_fail = 1; atomicCAS(info + blockIdx.x, 0, pivot_base + c0 + failcol + 1); }
                } else {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        // the block's strictly-upper part is zeroed: the inverse group reads it as a full tile
                        sL[(c0 + lane) * POTF2_LD + c0 + c] = (c <= lane) ? a[c] : 0.0;
                        sDTp[c * 32 + lane] = (c <= lane) ? a[c] : 0.0;
                    }
                }
                if (stamp && sp < 2) g_potf2_clk[sp == 0 ? 4 : 9] = clock64();     // diagonal block of sub-panel sp factored
                if (sp == 0) __syncthreads();              // block staged by warps 1..15 AND D_0 final
                else {
                    __threadfence_block();
                    asm volatile("bar.arrive 1, 256;\n" ::: "memory");                          // D_sp final for warps 1-7 (not waited for)
                    asm volatile("bar.arrive %0, 512;\n" ::"r"(4 + sp) : "memory");             // ... and for the inverse group
                }
                if (s_fail) break;
                if (c1 >= 128) {                           // last diagonal block: its rows are final, write them back
#pragma unroll
                    for (int c = 0; c < 32; ++c) A[(int64_t)(c0 + lane) * ld + c0 + c] = (c <= lane) ? a[c] : 0.0;
                    break;
                }
                // column block sp is written back by the other warps; this arrival only completes the count
                asm volatile("bar.arrive %0, 512;\n" ::"r"(8 + sp) : "memory");
                continue;
            }
            // ------------------------------- warps 1..7 -------------------------------
            if (sp == 0) __syncthreads();
            else {
                bar_named(1, 256);
                asm volatile("bar.arrive %0, 512;\n" ::"r"(4 + sp) : "memory");
            }
            if (tid == 32 && blockIdx.x == 0 && sp == 0) g_potf2_clk[15] = clock64();
            if (s_fail) break;
            if (c1 >= 128) break;                          // nothing below the last diagonal block
            {
                // rows c1 .. 127 over the 224 threads: warp 1 owns the rows of the next diagonal block
                const int r = c1 + (warp - 1) * 32 + lane;
                if (r < 128) {
                    double x[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) x[c] = sL[r * POTF2_LD + c0 + c];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        x[j] *= sRinvp[j];
#pragma unroll
                        for (int c2 = 0; c2 < 16; ++c2) {
                            if (2 * c2 + 1 > j) {
                                const double2 lc = *reinterpret_cast<const double2*>(sDTp + j * 32 + 2 * c2);
                                if (2 * c2 > j) x[2 * c2] = fma(-x[j], lc.x, x[2 * c2]);
                                x[2 * c2 + 1] = fma(-x[j], lc.y, x[2 * c2 + 1]);
                            }
                        }
                    }
#pragma unroll
                    for (int c = 0; c < 32; ++c) { sL[r * POTF2_LD + c0 + c] = x[c]; sP[c * POTF2_PLD + r] = x[c]; }
                }
            }
            if (tid == 32 && blockIdx.x == 0 && sp == 0) g_potf2_clk[7] = clock64();
            bar_named(3, 224);                             // panel (and its transpose sP) complete
            if (tid == 32 && blockIdx.x == 0 && sp == 0) g_potf2_clk[8] = clock64();
            const int nt = (128 - c1) / 16;
            const int ntile = nt * (nt + 1) / 2;           // >= 3; tiles 0, 1, 2 = the next diagonal block (c1 .. c1+32)^2
            auto update_tile = [&](int t) {
                int ti = 0, acc_t = t;
                while (acc_t > ti) { acc_t -= ti + 1; ++ti; }
                const int tj = acc_t;
                const int r0 = c1 + 16 * ti, q0 = c1 + 16 * tj;
                double cacc[2][2][2] = {{{0.0, 0.0}, {0.0, 0.0}}, {{0.0, 0.0}, {0.0, 0.0}}};
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    double a[2], bq[2];
#pragma unroll
                    for (int mi = 0; mi < 2; ++mi) a[mi] = sP[(4 * kk + fk) * POTF2_PLD + r0 + 8 * mi + fr];
#pragma unroll
                    for (int ni = 0; ni < 2; ++ni) bq[ni] = sP[(4 * kk + fk) * POTF2_PLD + q0 + 8 * ni + fr];
#pragma unroll
                    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 2; ++ni) dmma8x8x4(cacc[mi][ni][0], cacc[mi][ni][1], a[mi], bq[ni]);
                }
#pragma unroll
                for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 2; ++ni) {
                        double* dst = sL + (r0 + 8 * mi + fr) * POTF2_LD + q0 + 8 * ni + 2 * fk;
                        dst[0] -= cacc[mi][ni][0];
                        dst[1] -= cacc[mi][ni][1];
                    }
            };
            if (warp <= 3) {                               // the critical tiles first, then warp 0 is released
                update_tile(warp - 1);
                if (tid == 32 && blockIdx.x == 0 && sp == 0) g_potf2_clk[10] = clock64();
                __threadfence_block();
                asm volatile("bar.arrive 12, 128;\n" ::: "memory");
            }
            // column block sp of L is final: write it back (rows c0 .. 127; the diagonal block's upper part as zeros)
            for (int e = tid - 32; e < 128 * 32; e += 224) {
                const int r = e >> 5, cc = c0 + (e & 31);
                A[(int64_t)r * ld + cc] = (cc <= r) ? sL[r * POTF2_LD + cc] : 0.0;
            }
            // rows below column block sp are final AND D_sp has been written back: the inverse group may read the former and
            // overwrite the latter (it parks X_sp,sp there)
            asm volatile("bar.arrive %0, 512;\n" ::"r"(8 + sp) : "memory");
            for (int t = (warp <= 3 ? warp - 1 + 7 : warp - 1); t < ntile; t += 7)
                if (t >= 3) update_tile(t);
            bar_named(13, 224);                            // whole trailing update done: the next substitution may read it / reuse sP
            if (stamp && false) g_potf2_clk[7] = clock64();
        }
        if (stamp) { g_potf2_clk[2] = clock64(); g_potf2_clk[3] = g_potf2_clk[2]; }
    } else {
        // =============================== INVERSE GROUP ===============================
        const int it = tid - 256, iw = warp - 8;
        for (int e = it; e < 128 * 128; e += 256) {          // strictly-upper 32-blocks of the result are zero
            int r = e >> 7, c = e & 127;
            if ((c >> 5) > (r >> 5)) Di[e] = 0.0;
        }
        for (int s = 0; s < 4; ++s) {
            const int c0 = s * 32;
            if (s > 0) {
                // ---- (ahead of the hand-off) S_st = sum_{u=t}^{s-1} L_su X_ut : strips (t, ti) of four
                //      8x8 tiles; needs X rows < s (this group) and L_s,u<s (factor group: barrier 3)
                bar_named(8 + s - 1, 512);
                // X_{s-1,s-1} (still in sXs) takes the place of D_{s-1} in sL; the strictly-upper 32-blocks of
                // sL are free and hold the off-diagonal X_ut at block position (t, u): everything the S
                // products need is then in shared memory
                for (int e = it; e < 32 * 32; e += 256) {
                    const int r = e >> 5, cc = e & 31;
                    sL[(c0 - 32 + r) * POTF2_LD + c0 - 32 + cc] = sXs[r * PW_XLD + cc];
                }
                bar_named(2, 256);
                for (int g = iw; g < 4 * s; g += 8) {
                    const int t = g >> 2, ti = g & 3;
                    double cc[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
                    const double* arow = sL + (c0 + ti * 8 + fr) * POTF2_LD + fk;
                    for (int kq = 32 * t; kq < c0; kq += 4) {
                        const double a = arow[kq];
                        // X_ut[k][n], u = kq / 32: block (t, t) on the diagonal for u == t, else upper block (t, u)
                        const int u = kq >> 5;
                        const double* brow = (u == t) ? sL + (kq + fk) * POTF2_LD + 32 * t + fr
                                                      : sL + (32 * t + (kq & 31) + fk) * POTF2_LD + 32 * u + fr;
#pragma unroll
                        for (int q = 0; q < 4; ++q) dmma8x8x4(cc[q][0], cc[q][1], a, brow[q * 8]);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        double* dst = sS + t * 32 * PW_XLD + (ti * 8 + fr) * PW_XLD + q * 8 + 2 * fk;
                        dst[0] = cc[q][0]; dst[1] = cc[q][1];
                    }
                }
            }
            const bool istamp = (it == 0 && blockIdx.x == 0 && s == 3);
            if (istamp) g_potf2_clk[11] = clock64();
            if (s == 0) __syncthreads();                   // block staged and D_0 final
            else bar_named(4 + s, 512);                    // hand-off: D_s is final (factor group only arrives)
            if (istamp) g_potf2_clk[12] = clock64();
            if (s_fail) break;
            // ---- X_ss = inv(D_s) by ONE warp, no barriers: lane = column c of the inverse, right-looking
            //      substitution  x_j = acc_j / L_jj ; acc_i -= L_ij x_j (i > j)  with L broadcast from sL.
            //      Columns left of c come out as exact zeros (acc_j = 0 for j < c).
            if (iw == 0) {
                sTi[lane] = 1.0 / sL[(c0 + lane) * POTF2_LD + c0 + lane];
                __syncwarp();
                double acc[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[i] = (i == lane) ? 1.0 : 0.0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const double xj = acc[j] * sTi[j];
                    acc[j] = xj;
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (i > j) acc[i] = fma(-sL[(c0 + i) * POTF2_LD + c0 + j], xj, acc[i]);
                }
#pragma unroll
                for (int i = 0; i < 32; ++i) sXs[i * PW_XLD + lane] = acc[i];
            }
            bar_named(2, 256);
            if (istamp) g_potf2_clk[13] = clock64();
            for (int e = it; e < 32 * 32; e += 256) {          // X_ss -> global (upper part is zero)
                int r = e >> 5, c = e & 31;
                Di[(c0 + r) * 128 + c0 + c] = sXs[r * PW_XLD + c];
            }
            if (s > 0) {
                // ---- X_st = - X_ss S_st  -> global
                for (int g = iw; g < 4 * s; g += 8) {
                    const int t = g >> 2, ti = g & 3;
                    double cc[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
                    const double* arow = sXs + (ti * 8 + fr) * PW_XLD + fk;
                    const double* bcol = sS + t * 32 * PW_XLD + fk * PW_XLD + fr;
                    for (int k = 0; k < (ti + 1) * 8; k += 4) {
                        const double a = arow[k];
#pragma unroll
                        for (int q = 0; q < 4; ++q) dmma8x8x4(cc[q][0], cc[q][1], a, bcol[k * PW_XLD + q * 8]);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        double* dst = Di + (c0 + ti * 8 + fr) * 128 + 32 * t + q * 8 + 2 * fk;
                        dst[0] = -cc[q][0]; dst[1] = -cc[q][1];
                        double* dsm = sL + (32 * t + ti * 8 + fr) * POTF2_LD + c0 + q * 8 + 2 * fk;   // upper block (t, s)
                        dsm[0] = -cc[q][0]; dsm[1] = -cc[q][1];
                    }
                }
            }
            bar_named(2, 256);                               // sXs / sS free for the next round
            if (istamp) g_potf2_clk[14] = clock64();
        }
    }
    __syncthreads();
    if (s_fail) {                                            // harmless identity as the inverse; A stays as it is
        for (int e = tid; e < 128 * 128; e += 512) Di[e] = ((e >> 7) == (e & 127)) ? 1.0 : 0.0;
    }
    if (stamp) g_potf2_clk[6] = clock64();
}

// ------------------------------------------------------------------------------------------
// O(n^2) vector kernels on row-major lower-triangular matrices
// ------------------------------------------------------------------------------------------
// out[r] = sum_{k <= r} T[r][k] * v[k]        one warp per row, fixed-order reduction
__global__ void trmv_lower_kernel(const double* __restrict__ T, int64_t ld, int64_t N,
                                  const double* __restrict__ v, double* __restrict__ out, int64_t strideT,
                                  int64_t strideV) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (r >= N) return;
    const double* row = T + (int64_t)blockIdx.y * strideT + r * ld;
    const double* vv = v + (int64_t)blockIdx.y * strideV;
    double s = 0.0;
#pragma unroll 8
    for (int64_t k = lane; k <= r; k += 32) s = fma(row[k], vv[k], s);      // 8 loads in flight per lane
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[(int64_t)blockIdx.y * strideV + r] = s;
}

// part[chunk][j] = sum_{i in chunk, i >= j} T[i][j] * v[i]     (T^T v, two-stage, deterministic)
constexpr int TRMVT_ROWS = 256;
__global__ void trmvT_lower_partial_kernel(const double* __restrict__ T, int64_t ld, int64_t N,
                                           const double* __restrict__ v, double* __restrict__ part,
                                           int64_t strideT, int64_t strideV, int64_t strideP) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * TRMVT_ROWS;
    if (j >= N) return;
    const double* Tb = T + (int64_t)blockIdx.z * strideT;
    const double* vv = v + (int64_t)blockIdx.z * strideV;
    int64_t i1 = i0 + TRMVT_ROWS; if (i1 > N) i1 = N;
    double s = 0.0;
#pragma unroll 8
    for (int64_t i = (i0 > j ? i0 : j); i < i1; ++i) s = fma(Tb[i * ld + j], vv[i], s);
    part[(int64_t)blockIdx.z * strideP + (int64_t)blockIdx.y * N + j] = s;
}
__global__ void reduce_rows_kernel(const double* __restrict__ part, int nchunks, int64_t N,
                                   double* __restrict__ out, int64_t strideP, int64_t strideO) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= N) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += part[(int64_t)blockIdx.y * strideP + (int64_t)c * N + j];
    out[(int64_t)blockIdx.y * strideO + j] = s;
}

// ------------------------------------------------------------------------------------------
// cross-kernel tile builder:  Ks[c][idx] = gradKernel((x_i, a), (x*_c, bo))  for a chunk of
// candidates, K-contiguous (row per candidate, ld = Npad), zeros in the padding columns, plus
// the posterior-mean partials  pmean[point-block][c] = sum_{idx in block} Ks[c][idx]*alpha[idx]
// (StandardGP.jl:361-363: mean = m(x*) + K*^T alpha).
// Thread = training point (coordinates in registers), CTA loops over KS_CB candidates held in
// shared memory.  grid (point blocks of 128, candidate blocks).
// bo = candidate output (0 = value: posterior_mean/var; b >= 1: posterior_grad_*).
// ------------------------------------------------------------------------------------------
constexpr int KS_CB = 32;

template <int DT, bool GRAD>
__global__ void __launch_bounds__(128) ks_build_kernel(KSpec spec, const double* __restrict__ XsT, int64_t ldx,
                                                       int64_t npts, int64_t N, int64_t Npad,
                                                       const double* __restrict__ alpha,
                                                       const double* __restrict__ Xc, int64_t c_begin,
                                                       int64_t m_total, int bo, double* __restrict__ Ks,
                                                       double* __restrict__ pmean, int64_t mc) {
    __shared__ double sc[KS_CB][DT];
    __shared__ double swsum[4][KS_CB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t i = blockIdx.x * 128LL + tid;            // training point
    const int64_t cb0 = (int64_t)blockIdx.y * KS_CB;       // first candidate of this CTA (chunk-local)
    for (int e = tid; e < KS_CB * DT; e += 128) {
        int c = e / DT, k = e - c * DT;
        int64_t gc = c_begin + cb0 + c;
        sc[c][k] = (k < spec.d && gc < m_total) ? spec.sk(k) * Xc[gc * spec.d + k] : 0.0;
    }
    double x[DT];
#pragma unroll
    for (int k = 0; k < DT; ++k) x[k] = (k < spec.d && i < npts) ? XsT[k * ldx + i] : 0.0;
    const int p = spec.p;
    const int64_t idx0 = i * p;
    const double al0 = (!GRAD && i < npts) ? alpha[idx0] : 0.0;
    __syncthreads();
    for (int c = 0; c < KS_CB; ++c) {
        double u = 0.0, Db = 0.0;
#pragma unroll
        for (int k = 0; k < DT; ++k) {
            double df = x[k] - sc[c][k];
            u = fma(df, df, u);
            if (k == bo - 1) Db = df;
        }
        double contrib = 0.0;
        double* row = Ks + (cb0 + c) * Npad;
        if (i < npts) {
            double ph, dph, ddph;
            phi_eval(spec.kind, u, ph, dph, ddph);
            if (!GRAD) {
                double v = gk_entry(spec, ph, dph, ddph, 0, bo, 0.0, Db);
                row[idx0] = v;
                contrib = v * al0;
            } else {
                for (int a = 0; a < p; ++a) {
                    // D_a re-read through L1 (keeps x[] in registers: no dynamic indexing)
                    double Da = (a == 0) ? 0.0 : XsT[(a - 1) * ldx + i] - sc[c][a - 1];
                    double v = gk_entry(spec, ph, dph, ddph, a, bo, Da, Db);
                    row[idx0 + a] = v;
                    contrib = fma(v, alpha[idx0 + a], contrib);
                }
            }
        } else {
            for (int a = 0; a < p; ++a)
                if (idx0 + a < Npad) row[idx0 + a] = 0.0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        if (lane == 0) swsum[warp][c] = contrib;
    }
    __syncthreads();
    if (tid < KS_CB)
        pmean[(int64_t)blockIdx.x * mc + cb0 + tid] = ((swsum[0][tid] + swsum[1][tid]) + swsum[2][tid]) + swsum[3][tid];
}

// generic-d fallback (d > 32): coordinates re-read from global memory
__global__ void __launch_bounds__(128) ks_build_generic_kernel(KSpec spec, const double* __restrict__ XsT,
                                                               int64_t ldx, int64_t npts, int64_t N, int64_t Npad,
                                                               const double* __restrict__ alpha,
                                                               const double* __restrict__ Xc, int64_t c_begin,
                                                               int64_t m_total, int bo, double* __restrict__ Ks,
                                                               double* __restrict__ pmean, int64_t mc) {
    __shared__ double swsum[4][KS_CB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t i = blockIdx.x * 128LL + tid;
    const int64_t cb0 = (int64_t)blockIdx.y * KS_CB;
    const int p = spec.p;
    const int64_t idx0 = i * p;
    for (int c = 0; c < KS_CB; ++c) {
        const int64_t gc = c_begin + cb0 + c;
        double contrib = 0.0;
        double* row = Ks + (cb0 + c) * Npad;
        if (i < npts) {
            double u = 0.0, Db = 0.0;
            for (int k = 0; k < spec.d; ++k) {
                double ck = (gc < m_total) ? spec.s * Xc[gc * spec.d + k] : 0.0;
                double df = XsT[k * ldx + i] - ck;
                u = fma(df, df, u);
                if (k == bo - 1) Db = df;
            }
            double ph, dph, ddph;
            phi_eval(spec.kind, u, ph, dph, ddph);
            for (int a = 0; a < p; ++a) {
                double Da = 0.0;
                if (a > 0) {
                    double ck = (gc < m_total) ? spec.s * Xc[gc * spec.d + a - 1] : 0.0;
                    Da = XsT[(a - 1) * ldx + i] - ck;
                }
                double v = gk_entry(spec, ph, dph, ddph, a, bo, Da, Db);
                row[idx0 + a] = v;
                contrib = fma(v, alpha[idx0 + a], contrib);
            }
        } else {
            for (int a = 0; a < p; ++a)
                if (idx0 + a < Npad) row[idx0 + a] = 0.0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        if (lane == 0) swsum[warp][c] = contrib;
    }
    __syncthreads();
    if (tid < KS_CB)
        pmean[(int64_t)blockIdx.x * mc + cb0 + tid] = ((swsum[0][tid] + swsum[1][tid]) + swsum[2][tid]) + swsum[3][tid];
}

// ------------------------------------------------------------------------------------------
// acquisition epilogue: mean, variance, EI / PI / UCB  for one chunk of candidates
//   mean = m + sum_blocks pmean ; var = (k** - sum_tiles sumsq) + 1e-18
//   EI  (ExpectedImprovement.jl:40-66), PI (ProbabilityImprovement.jl:38-63),
//   UCB (UpperConfidenceBound.jl:38-45) — same operation order as the reference.
// ------------------------------------------------------------------------------------------
struct AcqSpec {
    int acq;            // -1: posterior only
    double p0, p1;      // EI/PI: xi, best_y ; UCB: beta
    double mean_c;      // prior mean of the queried output
    double kss;         // prior variance of the queried output
};

__device__ __forceinline__ double normcdf_ref(double z) { return erfc(-z * 0.70710678118654752440) / 2; }
__device__ __forceinline__ double normpdf_ref(double z) { return exp(-(z * z) / 2) * 0.39894228040143267794; }

__device__ __forceinline__ double acq_value(const AcqSpec& a, double mu, double var) {
    if (a.acq == ACQ_UCB) return -mu + a.p0 * sqrt(fmax(var, 0.0));
    const double delta = (a.p1 - a.p0) - mu;
    if (var <= 1e-12) return fmax(delta, 0.0);
    const double sig = sqrt(var);
    const double z = delta / sig;
    if (a.acq == ACQ_EI) return delta * normcdf_ref(z) + sig * normpdf_ref(z);
    return normcdf_ref(z);
}

__global__ void acq_epilogue_kernel(AcqSpec a, const double* __restrict__ pmean, int npb,
                                    const double* __restrict__ sumsq, int ntile, int64_t mc, int64_t mvalid,
                                    double* __restrict__ mean_out, double* __restrict__ var_out,
                                    double* __restrict__ score_out) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= mvalid) return;
    double mu = 0.0;
    for (int b = 0; b < npb; ++b) mu += pmean[(int64_t)b * mc + c];
    mu += a.mean_c;
    double q = 0.0;
    for (int t = 0; t < ntile; ++t) q += sumsq[(int64_t)t * mc + c];
    const double var = (a.kss - q) + JITTER;
    if (mean_out) mean_out[c] = mu;
    if (var_out) var_out[c] = var;
    if (score_out && a.acq >= 0) score_out[c] = acq_value(a, mu, var);
}

// ------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------
// delta (point-major) from y (out-major at the ABI):  delta[i*p + a] = y[a*n + i] - mean_c[a]
__global__ void delta_kernel(const double* __restrict__ y, const double* __restrict__ mean_c, int64_t n, int p,
                             double* __restrict__ delta) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * p) return;
    const int64_t i = t / p;
    const int a = (int)(t % p);
    delta[t] = y[(int64_t)a * n + i] - mean_c[a];
}
// batched: the same delta replicated for every restart of the batch (blockIdx.y)
__global__ void delta_batched_kernel(const double* __restrict__ y, const double* __restrict__ mean_c, int64_t n, int p,
                                     double* __restrict__ delta, int64_t stride) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * p) return;
    const int64_t i = t / p;
    const int a = (int)(t % p);
    delta[(int64_t)blockIdx.y * stride + t] = y[(int64_t)a * n + i] - mean_c[a];
}
// out-major <- point-major permutation of a length n*p vector
__global__ void to_out_major_kernel(const double* __restrict__ v, int64_t n, int p, double* __restrict__ out) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * p) return;
    out[(t % p) * n + t / p] = v[t];
}
__global__ void fill_kernel(double* __restrict__ p, int64_t n, double v) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < n) p[t] = v;
}

// ------------------------------------------------------------------------------------------
// O(n^2) row append (StandardGP, p = 1): kernels around the two TRMVs
// ------------------------------------------------------------------------------------------
// kv[i] = sig2 * phi(|| xs_i - s*x_new ||^2), zero in the padding
__global__ void kvec_kernel(KSpec spec, const double* __restrict__ XsT, int64_t ldx, int64_t n, int64_t Npad,
                            const double* __restrict__ xnew, double* __restrict__ kv) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= Npad) return;
    if (i >= n) { kv[i] = 0.0; return; }
    double u = 0.0;
    for (int k = 0; k < spec.d; ++k) {
        double df = XsT[k * ldx + i] - spec.sk(k) * xnew[k];
        u = fma(df, df, u);
    }
    double p, dp, ddp;
    phi_eval(spec.kind, u, p, dp, ddp);
    kv[i] = spec.scale * p;
}
// out[0] = sum v[i]^2 (single block, fixed-order tree)
__global__ void __launch_bounds__(1024) sumsq_vec_kernel(const double* __restrict__ v, int64_t n, double* __restrict__ out) {
    __shared__ double sh[1024];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s = fma(v[i], v[i], s);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}
// commit the new row n:  L[n][:n] = w, L[n][n] = l ; Linv[n][:n] = -r/l, Linv[n][n] = 1/l ;
// delta[n], beta[n] = Linv[n][:n].delta + delta_n/l ; alpha[:n] += Linv[n][:n]*beta_n ; alpha[n] = beta_n/l ;
// XsT[:, n] = s*x_new.      Single block.
__global__ void __launch_bounds__(1024) append_commit_kernel(double* __restrict__ L, double* __restrict__ Linv, int64_t ld,
                                                             int64_t n, const double* __restrict__ w,
                                                             const double* __restrict__ r, double l, double delta_n,
                                                             double* __restrict__ delta, double* __restrict__ beta,
                                                             double* __restrict__ alpha, double* __restrict__ XsT,
                                                             int64_t ldx, const double* __restrict__ xnew, int d, KSpec spec) {
    __shared__ double sh[1024];
    __shared__ double s_beta;
    const double linv = 1.0 / l;
    double acc = 0.0;
    for (int64_t j = threadIdx.x; j < n; j += 1024) {
        const double li = -r[j] * linv;
        L[n * ld + j] = w[j];
        Linv[n * ld + j] = li;
        acc = fma(li, delta[j], acc);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double bn = sh[0] + delta_n * linv;
        s_beta = bn;
        L[n * ld + n] = l;
        Linv[n * ld + n] = linv;
        delta[n] = delta_n;
        beta[n] = bn;
        alpha[n] = bn * linv;
    }
    __syncthreads();
    const double bn = s_beta;
    for (int64_t j = threadIdx.x; j < n; j += 1024) alpha[j] = fma(Linv[n * ld + j], bn, alpha[j]);
    for (int k = threadIdx.x; k < d; k += 1024) XsT[k * ldx + n] = spec.sk(k) * xnew[k];
}
// ---- skinny triangular products for a handful of right-hand sides (block append): bandwidth-bound passes over
//      the triangle instead of 128-wide padded GEMM tiles.  RHS columns are processed 8 at a time (blockIdx.y).
// W[r][b] = sum_{k <= r} T[r][k] * Bt[b][k]        (Bt: one K-contiguous row per right-hand side), warp per row
__global__ void trmm_skinny_lower_kernel(const double* __restrict__ T, int64_t ld, int64_t N, const double* __restrict__ Bt,
                                         int64_t ldb, int nrhs, double* __restrict__ W, int64_t ldw) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (r >= N) return;
    const int b0 = blockIdx.y * 8;
    const double* row = T + r * ld;
    double acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.0;
#pragma unroll 4
    for (int64_t k = lane; k <= r; k += 32) {
        const double a = row[k];
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (b0 + q < nrhs) acc[q] = fma(a, Bt[(int64_t)(b0 + q) * ldb + k], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        if (lane == 0 && b0 + q < nrhs) W[r * ldw + b0 + q] = acc[q];
    }
}
// part[chunk][b][j] = sum_{i in chunk, i >= j} T[i][j] * V[i][b]     (T^T V, two-stage, deterministic)
__global__ void trmmT_skinny_partial_kernel(const double* __restrict__ T, int64_t ld, int64_t N, const double* __restrict__ V,
                                            int64_t ldv, int nrhs, double* __restrict__ part) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * TRMVT_ROWS;
    const int b0 = blockIdx.z * 8;
    if (j >= N) return;
    int64_t i1 = i0 + TRMVT_ROWS; if (i1 > N) i1 = N;
    double acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.0;
#pragma unroll 4
    for (int64_t i = (i0 > j ? i0 : j); i < i1; ++i) {
        const double a = T[i * ld + j];
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (b0 + q < nrhs) acc[q] = fma(a, V[i * ldv + b0 + q], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < 8; ++q)
        if (b0 + q < nrhs) part[((int64_t)blockIdx.y * nrhs + b0 + q) * N + j] = acc[q];
}
// Z[j][b] = sum_chunks part[chunk][b][j]
__global__ void trmmT_skinny_reduce_kernel(const double* __restrict__ part, int nchunks, int64_t N, int nrhs,
                                           double* __restrict__ Z, int64_t ldz) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (j >= N) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += part[((int64_t)c * nrhs + b) * N + j];
    Z[j * ldz + b] = s;
}
// G[a][b] = sum_k W[k][a] * W[k][b]     one block per (a, b)
__global__ void __launch_bounds__(256) gram_skinny_kernel(const double* __restrict__ W, int64_t ldw, int64_t N, double* __restrict__ G,
                                                          int64_t ldg) {
    __shared__ double sh[256];
    const int a = blockIdx.y, b = blockIdx.x;
    double acc = 0.0;
    for (int64_t k = threadIdx.x; k < N; k += 256) acc = fma(W[k * ldw + a], W[k * ldw + b], acc);
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) G[(int64_t)a * ldg + b] = sh[0];
}

// ---- block append of the p outputs of one new point (GradientGP) ------------------------------------
// W = L^-1 Kn  [Npad][ldw], G = W^T W [..][ldg].  out = S (p x p, row-major) | wb (p):
//   S = Knn + noise I - W^T W   (Knn: gradKernel of the point with itself, closed form at u = 0)
//   wb = W^T beta
__global__ void __launch_bounds__(256) append_block_stats_kernel(KSpec spec, const double* __restrict__ G, int64_t ldg,
                                                                 const double* __restrict__ W, int64_t ldw,
                                                                 const double* __restrict__ beta, int64_t N,
                                                                 double* __restrict__ out) {
    __shared__ double sh[256];
    const int p = spec.p, tid = threadIdx.x;
    double ph, dph, ddph;
    phi_eval(spec.kind, 0.0, ph, dph, ddph);
    for (int e = tid; e < p * p; e += 256) {
        const int a = e / p, b = e % p;
        double knn = gk_entry(spec, ph, dph, ddph, a, b, 0.0, 0.0);
        if (a == b) knn += spec.noise;
        out[e] = knn - G[(int64_t)a * ldg + b];
    }
    for (int a = 0; a < p; ++a) {
        double acc = 0.0;
        for (int64_t k = tid; k < N; k += 256) acc = fma(W[k * ldw + a], beta[k], acc);
        sh[tid] = acc;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (tid < o) sh[tid] += sh[tid + o];
            __syncthreads();
        }
        if (tid == 0) out[p * p + a] = sh[0];
        __syncthreads();
    }
}
// small: LS (p x p) | LSinv (p x p) | beta_new (p) | gamma (p) | delta_new (p) | x (d)   — from the host
//   L[N+a, :]    = [ W[:, a]^T , LS[a, :a+1] ]
//   Linv[N+a, :] = [ -(LSinv Z^T)[a, :] , LSinv[a, :a+1] ]
//   alpha[:N]   -= Z gamma ; alpha[N+a] = gamma[a] ; beta[N+a] = beta_new[a] ; delta[N+a] = delta_new[a]
__global__ void __launch_bounds__(256) append_block_commit_kernel(double* __restrict__ L, double* __restrict__ Linv, int64_t ld,
                                                                  int64_t N, int p, const double* __restrict__ W,
                                                                  const double* __restrict__ Z, int64_t ldw,
                                                                  const double* __restrict__ small, double* __restrict__ delta,
                                                                  double* __restrict__ beta, double* __restrict__ alpha,
                                                                  double* __restrict__ XsT, int64_t ldx, int64_t npts, int d,
                                                                  KSpec spec) {
    const double* LS = small;
    const double* LSinv = small + p * p;
    const double* bnew = LSinv + p * p;
    const double* gamma = bnew + p;
    const double* dnew = gamma + p;
    const double* x = dnew + p;
    const int64_t k = blockIdx.x * 256LL + threadIdx.x;
    if (k < N) {
        double da = 0.0;
        for (int a = 0; a < p; ++a) {
            L[(N + a) * ld + k] = W[k * ldw + a];
            double li = 0.0;
            for (int b = 0; b <= a; ++b) li = fma(LSinv[a * p + b], Z[k * ldw + b], li);
            Linv[(N + a) * ld + k] = -li;
            da = fma(Z[k * ldw + a], gamma[a], da);
        }
        alpha[k] -= da;
    }
    if (blockIdx.x == 0) {
        for (int e = threadIdx.x; e < p * p; e += 256) {
            const int a = e / p, b = e % p;
            if (b <= a) { L[(N + a) * ld + N + b] = LS[e]; Linv[(N + a) * ld + N + b] = LSinv[e]; }
        }
        for (int a = threadIdx.x; a < p; a += 256) { alpha[N + a] = gamma[a]; beta[N + a] = bnew[a]; delta[N + a] = dnew[a]; }
        for (int q = threadIdx.x; q < d; q += 256) XsT[q * ldx + npts] = spec.sk(q) * x[q];
    }
}
// grow a padded lower-triangular matrix: copy the old Npad x Npad block, identity in the new part
__global__ void grow_matrix_kernel(const double* __restrict__ src, int64_t old_pad, int64_t old_ld,
                                   double* __restrict__ dst, int64_t new_pad) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= new_pad * new_pad) return;
    const int64_t r = t / new_pad, c = t % new_pad;
    dst[t] = (r < old_pad && c < old_pad) ? src[r * old_ld + c] : (r == c ? 1.0 : 0.0);
}

// ------------------------------------------------------------------------------------------
// batched NLML (value + analytic gradient)
// ------------------------------------------------------------------------------------------
// per-batch scaled coordinates: XsT[b][k*ldx + i] = s_b * X[i*d + k]
__global__ void scale_transpose_batched_kernel(const double* __restrict__ X, double* __restrict__ XsT, int64_t n, int d,
                                               int64_t ldx, const double* __restrict__ sb, int ard) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ldx * d) return;
    int k = (int)(t / ldx);
    int64_t i = t % ldx;
    const double s = ard ? sb[(int64_t)blockIdx.y * d + k] : sb[blockIdx.y];
    XsT[(int64_t)blockIdx.y * ldx * d + t] = (i < n) ? s * X[i * d + k] : 0.0;
}
// d/dlog(l) of a gradKernel entry.  s = 1/l, u = s^2 r^2, D = s * Delta:
//   ds = -s, du = -2u, dD = -D.  uphi3 = u * (third derivative of phi at u).
__device__ __forceinline__ double gk_dlogl_entry(const KSpec& ks, double u, double dp, double ddp, double uphi3, int a,
                                                 int b, double Da, double Db) {
    if (a == 0 && b == 0) return -2.0 * ks.scale * dp * u;
    if (b == 0) return -4.0 * ks.scale * ks.s * Da * (dp + u * ddp);
    if (a == 0) return 4.0 * ks.scale * ks.s * Db * (dp + u * ddp);
    const double s2 = ks.s * ks.s;
    return ks.scale * (16.0 * s2 * ddp * Da * Db + 8.0 * s2 * uphi3 * Da * Db + (a == b ? 4.0 * s2 * (dp + u * ddp) : 0.0));
}
// u times the third derivative of phi, from the second derivative ddp (no second exponential):
//   SE: phi3 = -ddp/2;  Matern-5/2: ddp = (25/12) e^{-sqrt5 r}, phi3 = -(25 sqrt5/24) e^{-sqrt5 r} / r;
//   Matern-7/2: ddp = (49/60)(1 + sqrt7 r) e^{-sqrt7 r}, phi3 = -(343/120) e^{-sqrt7 r}
__device__ __forceinline__ double u_phi3(int kind, double u, double ddp) {
    if (kind == K_SE) return -u * ddp / 2;
    const double r = sqrt(u);
    if (kind == K_M52 || kind == K_AM52 || kind == K_ADM52) {
        if (kind == K_AM52 && u < 1e-10) return 0.0;
        return -(2.23606797749978969641 / 2.0) * r * ddp;
    }
    if (kind == K_AM72 && u < 1e-10) return 0.0;
    return -(343.0 / 120.0) * (60.0 / 49.0) * u * ddp / (1 + 2.64575131106459059050 * r);
}
// per lower tile:  part[b][tile][0] = sum_ij M_ij dK_ij/dlog l ,  part[..][1] = sum_ij M_ij K_ij
// with M = Cinv - alpha alpha^T, counted over the FULL symmetric matrix (strict-lower entries x2).
// grid (T, T, batch), 256 threads, tiles above the diagonal write zeros.
__global__ void __launch_bounds__(256) nlml_grad_tile_kernel(KSpec spec, KmatBatch bt, const double* __restrict__ XsT,
                                                             int64_t ldx, int64_t N, const double* __restrict__ Cinv,
                                                             int64_t ld, int64_t strideC, const double* __restrict__ alpha,
                                                             int64_t strideV, double* __restrict__ part) {
    __shared__ double sh[2][256];
    const int bi = blockIdx.y, bj = blockIdx.x;
    const int T = gridDim.x;
    double g0 = 0.0, g1 = 0.0;
    if (bj <= bi) {
        apply_batch(spec, bt, blockIdx.z);
        const double* X = XsT + (int64_t)blockIdx.z * bt.strideX;
        const double* Cb = Cinv + (int64_t)blockIdx.z * strideC;
        const double* al = alpha + (int64_t)blockIdx.z * strideV;
        const int c = threadIdx.x & 127;
        const int64_t gc = (int64_t)bj * NB + c;
        const bool p1 = spec.p == 1;
        const int64_t j = p1 ? gc : gc / spec.p;
        const int b = p1 ? 0 : (int)(gc % spec.p);
        for (int r = threadIdx.x >> 7; r < NB; r += 2) {
            const int64_t gr = (int64_t)bi * NB + r;
            if (gr >= N || gc >= N || gc > gr) continue;
            const int64_t i = p1 ? gr : gr / spec.p;
            const int a = p1 ? 0 : (int)(gr % spec.p);
            double u = 0.0, Da = 0.0, Db = 0.0;
            for (int k = 0; k < spec.d; ++k) {
                double df = X[k * ldx + i] - X[k * ldx + j];
                u = fma(df, df, u);
                if (k == a - 1) Da = df;
                if (k == b - 1) Db = df;
            }
            double p, dp, ddp;
            phi_eval(spec.kind, u, p, dp, ddp);
            const double kv = gk_entry(spec, p, dp, ddp, a, b, Da, Db);
            const double dk = gk_dlogl_entry(spec, u, dp, ddp, p1 ? 0.0 : u_phi3(spec.kind, u, ddp), a, b, Da, Db);
            const double m = (Cb[gr * ld + gc] - al[gr] * al[gc]) * (gr == gc ? 1.0 : 2.0);
            g0 = fma(m, dk, g0);
            g1 = fma(m, kv, g1);
        }
    }
    sh[0][threadIdx.x] = g0; sh[1][threadIdx.x] = g1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double* o = part + ((int64_t)blockIdx.z * T * T + (int64_t)bi * T + bj) * 2;
        o[0] = sh[0][0]; o[1] = sh[1][0];
    }
}
// scalar GP (p = 1), d <= DT: register/shared-memory tiling as kmat_p1_kernel
template <int DT, int CPT>
__global__ void __launch_bounds__(256, 2) nlml_grad_p1_kernel(KSpec spec, KmatBatch bt, const double* __restrict__ XsT,
                                                           int64_t ldx, int64_t N, const double* __restrict__ Cinv,
                                                           int64_t ld, int64_t strideC, const double* __restrict__ alpha,
                                                           int64_t strideV, double* __restrict__ part) {
    __shared__ double sxi[DT][NB];
    __shared__ double sal[NB];
    __shared__ double sh[2][256];
    const int bi = blockIdx.y, bj = blockIdx.x;
    const int T = gridDim.x;
    const int tid = threadIdx.x;
    double g0 = 0.0, g1 = 0.0;
    if (bj <= bi) {
        apply_batch(spec, bt, blockIdx.z);
        const double* X = XsT + (int64_t)blockIdx.z * bt.strideX;
        const double* Cb = Cinv + (int64_t)blockIdx.z * strideC;
        const double* al = alpha + (int64_t)blockIdx.z * strideV;
        for (int e = tid; e < DT * NB; e += 256) {
            const int k = e >> 7, r = e & 127;
            const int64_t gr = (int64_t)bi * NB + r;
            sxi[k][r] = (k < spec.d && gr < N) ? X[k * ldx + gr] : 0.0;
        }
        if (tid < NB) { const int64_t gr = (int64_t)bi * NB + tid; sal[tid] = gr < N ? al[gr] : 0.0; }
        constexpr int TPG = NB / CPT, NG = 256 / TPG, RPG = NB / NG;
        const int tg = tid % TPG, grp = tid / TPG;
        double xj[CPT][DT], alc[CPT];
#pragma unroll
        for (int q = 0; q < CPT; ++q) {
            const int64_t gc = (int64_t)bj * NB + tg + q * TPG;
            alc[q] = gc < N ? al[gc] : 0.0;
#pragma unroll
            for (int k = 0; k < DT; ++k) xj[q][k] = (k < spec.d && gc < N) ? X[k * ldx + gc] : 0.0;
        }
        __syncthreads();
        constexpr int RB = 4;                              // rows per batch: their Cinv loads are issued together
        for (int rr0 = 0; rr0 < RPG; rr0 += RB) {
            double cv[RB][CPT];
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const int64_t gr = (int64_t)bi * NB + grp * RPG + rr0 + i;
#pragma unroll
                for (int q = 0; q < CPT; ++q) {
                    const int64_t gc = (int64_t)bj * NB + tg + q * TPG;
                    cv[i][q] = (gr < N && gc <= gr) ? __ldg(Cb + gr * ld + gc) : 0.0;
                }
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const int r = grp * RPG + rr0 + i;
                const int64_t gr = (int64_t)bi * NB + r;
                double u[CPT];
#pragma unroll
                for (int q = 0; q < CPT; ++q) u[q] = 0.0;
#pragma unroll
                for (int k = 0; k < DT; ++k) {
                    const double xi = sxi[k][r];
#pragma unroll
                    for (int q = 0; q < CPT; ++q) { const double df = xi - xj[q][k]; u[q] = fma(df, df, u[q]); }
                }
                const double alr = sal[r];
#pragma unroll
                for (int q = 0; q < CPT; ++q) {
                    const int64_t gc = (int64_t)bj * NB + tg + q * TPG;
                    const bool valid = gr < N && gc <= gr;
                    double p, dp, ddp;
                    phi_eval(spec.kind, u[q], p, dp, ddp);
                    const double kv = spec.scale * p;
                    const double dk = -2.0 * spec.scale * dp * u[q];
                    const double m = valid ? (cv[i][q] - alr * alc[q]) * (gr == gc ? 1.0 : 2.0) : 0.0;
                    g0 = fma(m, dk, g0);
                    g1 = fma(m, kv, g1);
                }
            }
        }
    }
    sh[0][tid] = g0; sh[1][tid] = g1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) { sh[0][tid] += sh[0][tid + o]; sh[1][tid] += sh[1][tid + o]; }
        __syncthreads();
    }
    if (tid == 0) {
        double* o = part + ((int64_t)blockIdx.z * T * T + (int64_t)bi * T + bj) * 2;
        o[0] = sh[0][0]; o[1] = sh[1][0];
    }
}

// ARD (per-dimension length scales), scalar GP: per lower tile the d + 1 partial sums
//   part[b][tile][k]  = sum_ij M_ij dK_ij/dlog l_k = sum_ij M_ij (-2 sig2 phi'(u_ij) D_ij,k^2)      k < d
//   part[b][tile][d]  = sum_ij M_ij K_ij                                                           (d/dlog sig2)
// (u = sum_k D_k^2, D_k = s_k (x_ik - x_jk): du/dlog l_k = -2 D_k^2), M = Cinv - alpha alpha^T over the full symmetric matrix.
template <int DT>
__global__ void __launch_bounds__(256) nlml_grad_ard_kernel(KSpec spec, KmatBatch bt, const double* __restrict__ XsT, int64_t ldx,
                                                            int64_t N, const double* __restrict__ Cinv, int64_t ld, int64_t strideC,
                                                            const double* __restrict__ alpha, int64_t strideV,
                                                            double* __restrict__ part) {
    __shared__ double sh[8][DT + 1];
    const int bi = blockIdx.y, bj = blockIdx.x, T = gridDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d = spec.d;
    double g[DT + 1];
#pragma unroll
    for (int k = 0; k <= DT; ++k) g[k] = 0.0;
    if (bj <= bi) {
        apply_batch(spec, bt, blockIdx.z);
        const double* X = XsT + (int64_t)blockIdx.z * bt.strideX;
        const double* Cb = Cinv + (int64_t)blockIdx.z * strideC;
        const double* al = alpha + (int64_t)blockIdx.z * strideV;
        const int64_t gc = (int64_t)bj * NB + (tid & 127);
        double xj[DT];
#pragma unroll
        for (int k = 0; k < DT; ++k) xj[k] = (k < d && gc < N) ? X[k * ldx + gc] : 0.0;
        const double alc = gc < N ? al[gc] : 0.0;
        for (int r = tid >> 7; r < NB; r += 2) {
            const int64_t gr = (int64_t)bi * NB + r;
            if (gr >= N || gc >= N || gc > gr) continue;
            double df2[DT], u = 0.0;
#pragma unroll
            for (int k = 0; k < DT; ++k) { const double df = (k < d ? X[k * ldx + gr] : 0.0) - xj[k]; df2[k] = df * df; u += df2[k]; }
            double ph, dph, ddph;
            phi_eval(spec.kind, u, ph, dph, ddph);
            const double m = (Cb[gr * ld + gc] - al[gr] * alc) * (gr == gc ? 1.0 : 2.0);
            const double w = -2.0 * spec.scale * dph * m;
#pragma unroll
            for (int k = 0; k < DT; ++k) g[k] = fma(w, df2[k], g[k]);
            g[DT] = fma(m, spec.scale * ph, g[DT]);
        }
    }
#pragma unroll
    for (int k = 0; k <= DT; ++k) {
        double v = g[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) sh[warp][k] = v;
    }
    __syncthreads();
    if (tid <= d) {
        const int k = (tid == d) ? DT : tid;
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += sh[w][k];
        part[((int64_t)blockIdx.z * T * T + (int64_t)bi * T + bj) * (d + 1) + tid] = v;
    }
}
// one block per batch entry: out[b] = { nlml, g_1 .. g_ng }
__global__ void __launch_bounds__(256) nlml_finish_ard_kernel(const double* __restrict__ L, int64_t ld, int64_t strideM, int64_t N,
                                                              const double* __restrict__ beta, int64_t strideV,
                                                              const double* __restrict__ part, int ntile, int ng,
                                                              const int* __restrict__ info, double* __restrict__ out) {
    __shared__ double sh[2][256];
    const double* Lb = L + (int64_t)blockIdx.x * strideM;
    const double* bb = beta + (int64_t)blockIdx.x * strideV;
    double* o = out + (int64_t)blockIdx.x * (1 + ng);
    const int tid = threadIdx.x;
    double ld_ = 0.0, qq = 0.0;
    for (int64_t i = tid; i < N; i += 256) { ld_ += log(Lb[i * ld + i]); qq = fma(bb[i], bb[i], qq); }
    sh[0][tid] = ld_; sh[1][tid] = qq;
    __syncthreads();
    for (int s_ = 128; s_ > 0; s_ >>= 1) {
        if (tid < s_) { sh[0][tid] += sh[0][tid + s_]; sh[1][tid] += sh[1][tid + s_]; }
        __syncthreads();
    }
    const bool bad = info[blockIdx.x] != 0;
    if (tid == 0) o[0] = bad ? CUDART_INF : 0.5 * ((double)N * 1.8378770664093454836 + 2.0 * sh[0][0] + sh[1][0]);
    if (tid < ng) {
        double v = 0.0;
        for (int t = 0; t < ntile; ++t) v += part[((int64_t)blockIdx.x * ntile + t) * ng + tid];
        o[1 + tid] = bad ? CUDART_NAN : 0.5 * v;
    }
}

// dispatch on d: scalar GPs with d <= 32 take the tiled kernels, everything else the generic ones
inline void launch_kmat(const KSpec& spec, const double* XsT, int64_t ldx, int64_t N, double* K, int64_t ld, const KmatBatch& bt,
                        int T, int batch, cudaStream_t st) {
    const dim3 grid(T, T, batch);
    if (spec.p == 1 && spec.d <= 4) kmat_p1_kernel<4, 4><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else if (spec.p == 1 && spec.d <= 8) kmat_p1_kernel<8, 4><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else if (spec.p == 1 && spec.d <= 12) kmat_p1_kernel<12, 2><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else if (spec.p == 1 && spec.d <= 16) kmat_p1_kernel<16, 2><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else if (spec.p == 1 && spec.d <= 20) kmat_p1_kernel<20, 2><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else if (spec.p == 1 && spec.d <= 32) kmat_p1_kernel<32, 1><<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
    else kmat_kernel<<<grid, 256, 0, st>>>(spec, XsT, ldx, N, K, ld, bt);
}
inline void launch_nlml_grad(const KSpec& spec, const KmatBatch& bt, const double* XsT, int64_t ldx, int64_t N, const double* Cinv,
                             int64_t ld, int64_t strideC, const double* alpha, int64_t strideV, double* part, int T, int batch,
                             cudaStream_t st) {
    const dim3 grid(T, T, batch);
#define ABO_NG(DT, CPT) nlml_grad_p1_kernel<DT, CPT><<<grid, 256, 0, st>>>(spec, bt, XsT, ldx, N, Cinv, ld, strideC, alpha, strideV, part)
    if (spec.p == 1 && spec.d <= 4) ABO_NG(4, 4);
    else if (spec.p == 1 && spec.d <= 8) ABO_NG(8, 4);
    else if (spec.p == 1 && spec.d <= 12) ABO_NG(12, 2);
    else if (spec.p == 1 && spec.d <= 16) ABO_NG(16, 2);
    else if (spec.p == 1 && spec.d <= 20) ABO_NG(20, 2);
    else if (spec.p == 1 && spec.d <= 32) ABO_NG(32, 1);
    else nlml_grad_tile_kernel<<<grid, 256, 0, st>>>(spec, bt, XsT, ldx, N, Cinv, ld, strideC, alpha, strideV, part);
#undef ABO_NG
}

// one block per batch: nlml = (N log 2pi + 2 sum log L_ii + ||beta||^2) / 2, grad = (sum of tile partials) / 2
__global__ void __launch_bounds__(256) nlml_finish_kernel(const double* __restrict__ L, int64_t ld, int64_t strideM, int64_t N,
                                                          const double* __restrict__ beta, int64_t strideV,
                                                          const double* __restrict__ part, int ntile,
                                                          const int* __restrict__ info, double* __restrict__ out) {
    __shared__ double sh[4][256];
    const double* Lb = L + (int64_t)blockIdx.x * strideM;
    const double* bb = beta + (int64_t)blockIdx.x * strideV;
    double ld_ = 0.0, qq = 0.0, g0 = 0.0, g1 = 0.0;
    for (int64_t i = threadIdx.x; i < N; i += 256) { ld_ += log(Lb[i * ld + i]); qq = fma(bb[i], bb[i], qq); }
    for (int t = threadIdx.x; t < ntile; t += 256) {
        g0 += part[((int64_t)blockIdx.x * ntile + t) * 2];
        g1 += part[((int64_t)blockIdx.x * ntile + t) * 2 + 1];
    }
    sh[0][threadIdx.x] = ld_; sh[1][threadIdx.x] = qq; sh[2][threadIdx.x] = g0; sh[3][threadIdx.x] = g1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o)
            for (int q = 0; q < 4; ++q) sh[q][threadIdx.x] += sh[q][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double* o = out + (int64_t)blockIdx.x * 3;
        if (info[blockIdx.x] != 0) {
            o[0] = CUDART_INF; o[1] = CUDART_NAN; o[2] = CUDART_NAN;
        } else {
            o[0] = 0.5 * ((double)N * 1.8378770664093454836 + 2.0 * sh[0][0] + sh[1][0]);
            o[1] = 0.5 * sh[2][0];
            o[2] = 0.5 * sh[3][0];
        }
    }
}

}  // namespace abo

// ------------------------------------------------------------------------------------------
// Device-side stable top-k of the scores: sortperm(scores; rev = true)[1:k] (acq_utils.jl:51-52) as an exact radix
// select on the 64-bit order keys (Julia isless: NaN largest, -0.0 < 0.0), ties resolved by the smaller index.
//   8 x (digit histogram over the elements matching the prefix found so far, pick the digit that contains the
//   k-th largest)  ->  threshold key T and r = how many elements equal to T are still needed
//   tie ranks in index order (per-chunk counts, exclusive scan)  ->  gather {key > T} and the first r of {key == T}
// The K selected (index, value) pairs come back unordered; the caller sorts K items.
// ------------------------------------------------------------------------------------------
namespace abo {
struct SelState {
    unsigned long long prefix;        // high digits of the threshold key found so far
    long long remaining;              // how many of the elements matching the prefix are still needed
    unsigned long long hist[256];
    unsigned int out_count;
    unsigned int pad;
};
constexpr int SEL_CHUNK = 4096;       // elements per block in the tie / gather passes (256 threads x 16 consecutive)

__device__ __forceinline__ unsigned long long ordkey_dev(double v) {
    if (v != v) return ~0ull;
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__global__ void sel_init_kernel(SelState* st, long long k) {
    const int t = threadIdx.x;
    if (t < 256) st->hist[t] = 0;
    if (t == 0) { st->prefix = 0; st->remaining = k; st->out_count = 0; }
}
__global__ void __launch_bounds__(256) sel_hist_kernel(const double* __restrict__ s, int64_t m, int pass, SelState* st) {
    __shared__ unsigned int sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const int shift = 56 - 8 * pass;
    const unsigned long long prefix = st->prefix;
    for (int64_t i = blockIdx.x * 256LL + threadIdx.x; i < m; i += (int64_t)gridDim.x * 256) {
        const unsigned long long key = ordkey_dev(s[i]);
        if (pass == 0 || (key >> (shift + 8)) == prefix) atomicAdd(&sh[(unsigned)(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}
__global__ void sel_pick_kernel(SelState* st) {
    if (threadIdx.x == 0) {
        long long rem = st->remaining, cum = 0;
        int dgt = 255;
        for (; dgt > 0; --dgt) {
            const long long cnt = (long long)st->hist[dgt];
            if (cum + cnt >= rem) break;
            cum += cnt;
        }
        st->prefix = (st->prefix << 8) | (unsigned long long)dgt;
        st->remaining = rem - cum;
    }
    __syncthreads();
    if (threadIdx.x < 256) st->hist[threadIdx.x] = 0;
}
// ties[b] = number of elements equal to the threshold key in chunk b
__global__ void __launch_bounds__(256) sel_tiecount_kernel(const double* __restrict__ s, int64_t m, const SelState* st,
                                                           unsigned int* __restrict__ ties) {
    __shared__ unsigned int sh[256];
    const unsigned long long T = st->prefix;
    const int64_t base = (int64_t)blockIdx.x * SEL_CHUNK + threadIdx.x * 16;
    unsigned int cnt = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int64_t i = base + q;
        if (i < m && ordkey_dev(s[i]) == T) ++cnt;
    }
    sh[threadIdx.x] = cnt;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) ties[blockIdx.x] = sh[0];
}
// in-place exclusive scan of the chunk counts (64-bit running sum kept in registers; one thread: <= a few thousand chunks)
__global__ void sel_tiescan_kernel(unsigned int* ties, int nblk, unsigned long long* excl) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        unsigned long long run = 0;
        for (int b = 0; b < nblk; ++b) { excl[b] = run; run += ties[b]; }
    }
}
__global__ void __launch_bounds__(256) sel_gather_kernel(const double* __restrict__ s, int64_t m, SelState* st,
                                                         const unsigned long long* __restrict__ excl,
                                                         long long* __restrict__ out_idx, double* __restrict__ out_val) {
    __shared__ unsigned int sh[256];
    const unsigned long long T = st->prefix;
    const unsigned long long need = (unsigned long long)st->remaining;      // ties to take, in index order
    const int64_t base = (int64_t)blockIdx.x * SEL_CHUNK + threadIdx.x * 16;
    double v[16];
    unsigned int cnt = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int64_t i = base + q;
        v[q] = (i < m) ? s[i] : 0.0;
        if (i < m && ordkey_dev(v[q]) == T) ++cnt;
    }
    sh[threadIdx.x] = cnt;
    __syncthreads();
    // exclusive scan over the 256 threads (Hillis-Steele on the shared array)
    for (int o = 1; o < 256; o <<= 1) {
        unsigned int add = ((int)threadIdx.x >= o) ? sh[threadIdx.x - o] : 0u;
        __syncthreads();
        sh[threadIdx.x] += add;
        __syncthreads();
    }
    unsigned long long rank = excl[blockIdx.x] + (unsigned long long)(sh[threadIdx.x] - cnt);
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int64_t i = base + q;
        if (i >= m) break;
        const unsigned long long key = ordkey_dev(v[q]);
        bool take = key > T;
        if (key == T) { take = rank < need; ++rank; }
        if (take) {
            const unsigned int pos = atomicAdd(&st->out_count, 1u);
            out_idx[pos] = (long long)i;
            out_val[pos] = v[q];
        }
    }
}
}  // namespace abo

// ------------------------------------------------------------------------------------------
// acquisition value AND gradient for a small batch of points (batched local refinement of
// optimize_acquisition, src/acquisition_functions/acq_utils.jl:55-71, which the reference drives
// with finite differences of single-point evaluations):
//     mu   = m + k*^T alpha                  grad mu   =  sum_idx alpha_idx * dk*_idx/dx*
//     var  = k** - |w|^2,  w = L^-1 k*       grad var  = -2 sum_idx z_idx * dk*_idx/dx*,  z = L^-T w
// dk*_idx/dx*_b is the (a, b) block of gradKernel with a = output of training row idx.
// ------------------------------------------------------------------------------------------
namespace abo {

// colsq[c] = sum_i W[i][c]^2        (W: Npad x mpad row-major), one thread per column, fixed order
__global__ void colsumsq_kernel(const double* __restrict__ W, int64_t Npad, int64_t mpad, double* __restrict__ out) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= mpad) return;
    double s = 0.0;
    for (int64_t i = 0; i < Npad; ++i) { const double v = W[i * mpad + c]; s = fma(v, v, s); }
    out[c] = s;
}

// part[pb][c][b] = sum over the 128 training points of block pb of
//                  sum_a ( alpha[idx] , z[idx][c] ) * d gk((x_i,a),(x*_c,0)) / d x*_b
// grid (point blocks, candidates), 128 threads; output two planes: gmu and gvar partials.
constexpr int AG_MAXD = 32;
__global__ void __launch_bounds__(128) acq_grad_partial_kernel(KSpec spec, const double* __restrict__ XsT, int64_t ldx,
                                                               int64_t npts, const double* __restrict__ alpha,
                                                               const double* __restrict__ Z, int64_t mpad,
                                                               const double* __restrict__ Xc, int64_t m,
                                                               double* __restrict__ part) {
    __shared__ double sh[4][2 * AG_MAXD];
    const int c = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t i = blockIdx.x * 128LL + tid;
    const int d = spec.d, p = spec.p;
    double gmu[AG_MAXD], gva[AG_MAXD];
#pragma unroll
    for (int b = 0; b < AG_MAXD; ++b) { gmu[b] = 0.0; gva[b] = 0.0; }
    if (i < npts && c < m) {
        double u = 0.0;
        for (int k = 0; k < d; ++k) {
            const double df = XsT[k * ldx + i] - spec.sk(k) * Xc[(int64_t)c * d + k];
            u = fma(df, df, u);
        }
        double ph, dph, ddph;
        phi_eval(spec.kind, u, ph, dph, ddph);
        for (int a = 0; a < p; ++a) {
            const int64_t idx = i * p + a;
            const double al = alpha[idx], zz = Z[idx * mpad + c];
            const double Da = (a == 0) ? 0.0 : XsT[(a - 1) * ldx + i] - spec.sk(a - 1) * Xc[(int64_t)c * d + a - 1];
#pragma unroll
            for (int b = 0; b < AG_MAXD; ++b) {
                if (b < d) {
                    const double Db = XsT[b * ldx + i] - spec.sk(b) * Xc[(int64_t)c * d + b];
                    const double dk = gk_entry(spec, ph, dph, ddph, a, b + 1, Da, Db);
                    gmu[b] = fma(al, dk, gmu[b]);
                    gva[b] = fma(zz, dk, gva[b]);
                }
            }
        }
    }
#pragma unroll
    for (int b = 0; b < AG_MAXD; ++b) {
        if (b < d) {
            double x = gmu[b], y = gva[b];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { x += __shfl_xor_sync(0xffffffffu, x, o); y += __shfl_xor_sync(0xffffffffu, y, o); }
            if (lane == 0) { sh[warp][b] = x; sh[warp][AG_MAXD + b] = y; }
        }
    }
    __syncthreads();
    if (tid < 2 * AG_MAXD) {
        const int b = tid % AG_MAXD;
        if (b < d) {
            const double v = ((sh[0][tid] + sh[1][tid]) + sh[2][tid]) + sh[3][tid];
            part[(((int64_t)blockIdx.x * gridDim.y + c) * 2 + tid / AG_MAXD) * AG_MAXD + b] = v;
        }
    }
}

// one thread per candidate: value and gradient of EI / PI / UCB from (mu, var, grad mu, grad var)
__global__ void acq_grad_finish_kernel(AcqSpec a, int d, const double* __restrict__ pmean, int npb_mean,
                                       const double* __restrict__ colsq, const double* __restrict__ part, int npb,
                                       int64_t mc, int64_t mpad, int64_t m, double* __restrict__ score,
                                       double* __restrict__ grad, double* __restrict__ mean_out,
                                       double* __restrict__ var_out) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= m) return;
    double mu = 0.0;
    for (int b = 0; b < npb_mean; ++b) mu += pmean[(int64_t)b * mc + c];
    mu += a.mean_c;
    const double var = (a.kss - colsq[c]) + JITTER;
    if (mean_out) mean_out[c] = mu;
    if (var_out) var_out[c] = var;
    score[c] = acq_value(a, mu, var);
    // d acq / d mu, d acq / d var
    double dmu, dvar;
    if (a.acq == ACQ_UCB) {
        dmu = -1.0;
        dvar = (var > 0.0) ? a.p0 * 0.5 / sqrt(var) : 0.0;
    } else {
        const double delta = (a.p1 - a.p0) - mu;
        if (var <= 1e-12) {
            dmu = (delta > 0.0) ? -1.0 : 0.0;
            dvar = 0.0;
        } else {
            const double sig = sqrt(var), z = delta / sig;
            if (a.acq == ACQ_EI) { dmu = -normcdf_ref(z); dvar = normpdf_ref(z) * 0.5 / sig; }
            else { dmu = -normpdf_ref(z) / sig; dvar = -normpdf_ref(z) * z * 0.5 / var; }
        }
    }
    for (int b = 0; b < d; ++b) {
        double gm = 0.0, gv = 0.0;
        for (int pb = 0; pb < npb; ++pb) {
            gm += part[(((int64_t)pb * mpad + c) * 2 + 0) * AG_MAXD + b];
            gv += part[(((int64_t)pb * mpad + c) * 2 + 1) * AG_MAXD + b];
        }
        grad[c * d + b] = dmu * gm + dvar * (-2.0 * gv);
    }
}

}  // namespace abo

// posterior covariance over all (point, output) pairs of a small query set, out-major
// (posterior_grad_cov, src/surrogates/GradientGP.jl:968-971):
//   cov[(b,c),(b',c')] = gk((x_c,b),(x_c',b')) - G[b*mp + c][b'*mp + c'] + 1e-18 * delta
// with G = W^T W, W = L^-1 K*; one thread per output entry.
//   Dense form (pad = 0): the M x M matrix, M = m nout, leading dimension ldc.
//   Factor form (pad = the padded size, a multiple of 128): the pad x pad input of potrf_lookahead — lower 128-tiles only
//   (tiles above the diagonal are not written), the strict upper part of the diagonal tiles zero, identity in the padding,
//   and tau added to the diagonal on top of the 1e-18 (G is only read in its lower tiles).
namespace abo {
__global__ void cov_finish_kernel(KSpec spec, const double* __restrict__ Xc, int64_t m, int nout, int64_t mp,
                                  const double* __restrict__ G, int64_t ldg, double* __restrict__ cov, int64_t ldc,
                                  int64_t pad, double tau) {
    const int64_t M = m * nout, R = pad > 0 ? pad : M;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= R * R) return;
    const int64_t r = t / R, q = t % R;
    if (pad > 0) {
        if (q / 128 > r / 128) return;
        if (r >= M || q >= M || q > r) { cov[r * ldc + q] = (r == q) ? 1.0 : 0.0; return; }
    }
    const int b = (int)(r / m), b2 = (int)(q / m);
    const int64_t c = r % m, c2 = q % m;
    double u = 0.0, Da = 0.0, Db = 0.0;
    for (int k = 0; k < spec.d; ++k) {
        const double df = spec.sk(k) * Xc[c * spec.d + k] - spec.sk(k) * Xc[c2 * spec.d + k];
        u = fma(df, df, u);
        if (k == b - 1) Da = df;
        if (k == b2 - 1) Db = df;
    }
    double p, dp, ddp;
    phi_eval(spec.kind, u, p, dp, ddp);
    const double prior = gk_entry(spec, p, dp, ddp, b, b2, Da, Db);
    const double v = (prior - G[((int64_t)b * mp + c) * ldg + (int64_t)b2 * mp + c2]) + (r == q ? JITTER : 0.0);
    cov[r * ldc + q] = (r == q) ? v + tau : v;
}
}  // namespace abo

// fill distance  max_s min_j || x_s - X_j ||  (monte_carlo_fill_distance, src/BO_utils.jl:140-159):
// one thread per sample, training points streamed through shared memory; block maxima out.
namespace abo {
__global__ void __launch_bounds__(256) fill_distance_kernel(const double* __restrict__ X, int64_t n, int d,
                                                            const double* __restrict__ S, int64_t m,
                                                            double* __restrict__ blockmax) {
    extern __shared__ double sx[];                      // [tile][d]
    __shared__ double red[8];
    const int tile = 256;
    const int64_t sidx = blockIdx.x * 256LL + threadIdx.x;
    double best = CUDART_INF;
    for (int64_t j0 = 0; j0 < n; j0 += tile) {
        const int cnt = (int)((n - j0 < tile) ? (n - j0) : tile);
        __syncthreads();
        for (int e = threadIdx.x; e < cnt * d; e += 256) sx[e] = X[j0 * d + e];
        __syncthreads();
        if (sidx < m) {
            for (int j = 0; j < cnt; ++j) {
                double u = 0.0;
                for (int k = 0; k < d; ++k) { const double df = sx[j * d + k] - S[sidx * d + k]; u = fma(df, df, u); }
                best = fmin(best, u);
            }
        }
    }
    double v = (sidx < m) ? sqrt(best) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = red[0];
        for (int w = 1; w < 8; ++w) r = fmax(r, red[w]);
        blockmax[blockIdx.x] = r;
    }
}
}  // namespace abo
