// qei.cuh — device kernels of Monte-Carlo batch expected improvement (abo_acq_qei) over B batches of q points:
//     qEI = (1/S) sum_s max((best_y - xi) - min_j f_{s,j}, 0),   f_s = mu + chol(Sigma + tau I) z_s,
// with the same normals z_s for every batch.  Per chunk of whole batches the driver in abo_api.cu builds K* and
// W = L^-1 K*^T on the TMA GEMM; then
//   qei_gram_kernel         the q x q diagonal blocks of W^T W and the posterior means of every batch,
//   qei_batch_kernel        Sigma + tau I, its Cholesky on the tau ladder, the S-sample estimate and, for the gradient,
//                           d qEI / d mu and the Cholesky backward pass to C = d qEI / d Sigma (symmetric),
//   qei_combine_kernel      R_c = sum_j 2 C_cj Z_j, Z = L^-T W (the DMMA GEMM), the input of acq_grad_partial_kernel,
//   qei_grad_finish_kernel  grad_c = (d qEI / d mu_c) dk^T alpha - dk^T R_c + sum_{j != c} 2 C_cj d1 k(x_c, x_j).
// Every reduction runs in a fixed order over quantities of its own batch, so a batch's results do not depend on the
// other batches of the call or on where chunks start.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "kernels.cuh"
#include "sample.cuh"

namespace abo {

constexpr int QEI_MAXQ = 32;
constexpr int QEI_JITTER_STEPS = 7;         // tau_k = jitter * sigma^2 * 10^k, k = 0 .. 6 (abo_gp_posterior_sample's ladder)
constexpr int QEI_KT = 64;                  // rows of W staged per step of the Gram kernel
constexpr int QEI_PAIRS_PT = 5;             // (i >= j) pairs per thread: 128 * 5 >= 32 * 33 / 2

// One CTA (128 threads) per batch b of the chunk: Gm[b][i][j] = sum_k W[k][b q + i] W[k][b q + j] for j <= i (k ascending),
// and mu[b][i] = mean_c + sum_pb pmean[pb][b q + i] (the order of posterior_mean_var).
__global__ void __launch_bounds__(128) qei_gram_kernel(const double* __restrict__ W, int64_t Npad, int64_t ldw, int q,
                                                       const double* __restrict__ pmean, int npb, int64_t ldp, double mean_c,
                                                       double* __restrict__ Gm, double* __restrict__ mu) {
    __shared__ double t[QEI_KT][QEI_MAXQ + 1];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t col0 = (int64_t)b * q;
    const int npair = q * (q + 1) / 2;
    int pi[QEI_PAIRS_PT], pj[QEI_PAIRS_PT];
    double acc[QEI_PAIRS_PT];
#pragma unroll
    for (int r = 0; r < QEI_PAIRS_PT; ++r) {
        const int e = tid + 128 * r;
        int i = 0;
        while ((i + 1) * (i + 2) / 2 <= e) ++i;           // e = i (i + 1) / 2 + j
        pi[r] = i; pj[r] = e - i * (i + 1) / 2;
        acc[r] = 0.0;
    }
    for (int64_t k0 = 0; k0 < Npad; k0 += QEI_KT) {
        __syncthreads();
        for (int e = tid; e < QEI_KT * q; e += 128) {
            const int r = e / q, c = e - r * q;
            t[r][c] = W[(k0 + r) * ldw + col0 + c];
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < QEI_PAIRS_PT; ++r) {
            if (tid + 128 * r < npair) {
                const int i = pi[r], j = pj[r];
                double a = acc[r];
                for (int k = 0; k < QEI_KT; ++k) a = fma(t[k][i], t[k][j], a);
                acc[r] = a;
            }
        }
    }
#pragma unroll
    for (int r = 0; r < QEI_PAIRS_PT; ++r)
        if (tid + 128 * r < npair) Gm[((int64_t)b * q + pi[r]) * q + pj[r]] = acc[r];
    if (tid < q) {
        double m = 0.0;
        for (int pb = 0; pb < npb; ++pb) m += pmean[(int64_t)pb * ldp + col0 + tid];
        mu[(int64_t)b * q + tid] = m + mean_c;
    }
}

// warp-wide minimum of (key, lane) in the total order of findmin_key, ties to the smaller lane; every lane gets the result
__device__ __forceinline__ void qei_warp_argmin(uint64_t& key, int& idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint64_t k2 = __shfl_xor_sync(0xffffffffu, key, o);
        const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        if (k2 < key || (k2 == key && i2 < idx)) { key = k2; idx = i2; }
    }
}

// One warp per batch b.  Lane i < q owns row i of Sigma, L and L-bar.  Shared memory: four q x (q + 1) matrices.
//   Sigma[i][j] = (sigma^2 phi(|s (x_i - x_j)|^2) - Gm[i][j]) + 1e-18 delta_ij    (abo_gp_posterior_cov's form)
//   L = chol(Sigma + tau I), tau the first rung of the ladder that factors; a batch with none gets NaN value and tau.
//   Forward, s ascending: f = mu + L z_s, j* its first minimiser, I_s = max(delta - f_j*, 0), acc += I_s; value = acc / S.
//   With want_grad: mu-bar_j = -#{s : I_s > 0, j* = j} / S, L-bar[j][k] = -sum_{s : I_s > 0, j* = j} z_s[k] / S (k <= j), and
//   (Murray 2016) A-bar = L^-T Phi(L^T L-bar) L^-1, Phi = the lower triangle with the diagonal halved; C = (A-bar + A-bar^T) / 2.
//   C and mu-bar are 0 for a failed batch (its gradient is written as NaN by qei_grad_finish_kernel, which reads tau).
__global__ void __launch_bounds__(32) qei_batch_kernel(KSpec spec, const double* __restrict__ Xb, int q,
                                                       const double* __restrict__ Gm, const double* __restrict__ mu,
                                                       const double* __restrict__ Z, int64_t S, int ldz, double delta,
                                                       double jitter, int want_grad, double* __restrict__ value,
                                                       double* __restrict__ tau_out, double* __restrict__ dmu,
                                                       double* __restrict__ Cout) {
    extern __shared__ double qsm[];
    const int ld = q + 1;
    double* Sg = qsm;                  // Sigma, later Phi(L^T L-bar)
    double* L = Sg + q * ld;
    double* Lb = L + q * ld;           // sum of z over the samples won by each row, later A-bar
    double* Y = Lb + q * ld;
    const int b = blockIdx.x, lane = threadIdx.x, d = spec.d;
    const bool row = lane < q;
    const double* xb = Xb + (int64_t)b * q * d;
    if (row) {
        for (int j = 0; j <= lane; ++j) {
            double u = 0.0;
            for (int k = 0; k < d; ++k) {
                const double df = spec.sk(k) * xb[lane * d + k] - spec.sk(k) * xb[j * d + k];
                u = fma(df, df, u);
            }
            double p, dp, ddp;
            phi_eval(spec.kind, u, p, dp, ddp);
            const double prior = gk_entry(spec, p, dp, ddp, 0, 0, 0.0, 0.0);
            Sg[lane * ld + j] = (prior - Gm[((int64_t)b * q + lane) * q + j]) + (j == lane ? JITTER : 0.0);
        }
        for (int j = 0; j < q; ++j) Lb[lane * ld + j] = 0.0;
    }
    // Cholesky on the ladder, left-looking by column: lane i forms L[i][c] from its own row and row c
    double tau = 0.0;
    bool ok = false;
    for (int k = 0; k < QEI_JITTER_STEPS && !ok; ++k) {
        double p10 = 1.0;
        for (int e = 0; e < k; ++e) p10 *= 10.0;
        tau = jitter * spec.scale * p10;
        if (row)
            for (int j = 0; j <= lane; ++j) L[lane * ld + j] = (j == lane) ? Sg[lane * ld + j] + tau : Sg[lane * ld + j];
        __syncwarp();
        ok = true;
        for (int c = 0; c < q; ++c) {
            double dg = 0.0;
            if (lane == c) {
                dg = L[c * ld + c];
                for (int j = 0; j < c; ++j) dg -= L[c * ld + j] * L[c * ld + j];
            }
            dg = __shfl_sync(0xffffffffu, dg, c);
            if (!(dg > 0.0)) { ok = false; break; }       // warp-uniform
            const double ljj = sqrt(dg);
            if (lane > c && row) {
                double v = L[lane * ld + c];
                for (int j = 0; j < c; ++j) v -= L[lane * ld + j] * L[c * ld + j];
                L[lane * ld + c] = v / ljj;
            }
            if (lane == c) L[c * ld + c] = ljj;
            __syncwarp();
        }
        __syncwarp();
    }
    if (!ok) {
        if (lane == 0) { value[b] = CUDART_NAN; tau_out[b] = CUDART_NAN; }
        if (want_grad) {
            if (row) {
                dmu[(int64_t)b * q + lane] = 0.0;
                for (int j = 0; j < q; ++j) Cout[((int64_t)b * q + lane) * q + j] = 0.0;
            }
        }
        return;
    }
    // forward: f_lane = mu_lane + sum_{k <= lane} L[lane][k] z_k
    const double mul = row ? mu[(int64_t)b * q + lane] : 0.0;
    double acc = 0.0, wins = 0.0;
    for (int64_t s = 0; s < S; ++s) {
        const double z = row ? Z[s * ldz + lane] : 0.0;
        double f = mul;
        for (int k = 0; k < q; ++k) {
            const double zk = __shfl_sync(0xffffffffu, z, k);
            if (row && k <= lane) f = fma(L[lane * ld + k], zk, f);      // lanes >= q own no row of L
        }
        uint64_t key = row ? findmin_key(f) : ~0ull;
        int js = row ? lane : QEI_MAXQ;
        qei_warp_argmin(key, js);
        const double fmin = __shfl_sync(0xffffffffu, f, js & 31);
        const double imp = delta - fmin;
        if (imp > 0.0) {
            acc += imp;
            if (want_grad) {
                if (lane == js) wins += 1.0;
                if (lane <= js) Lb[js * ld + lane] += z;
            }
        }
        __syncwarp();
    }
    if (lane == 0) { value[b] = acc / (double)S; tau_out[b] = tau; }
    if (!want_grad) return;
    const double Sd = (double)S;
    if (row) {
        dmu[(int64_t)b * q + lane] = -wins / Sd;
        for (int j = 0; j <= lane; ++j) Lb[lane * ld + j] = -Lb[lane * ld + j] / Sd;
    }
    __syncwarp();
    // Phi(L^T L-bar) into Sg: lane k forms column k, B[i][k] = sum_{j >= i} L[j][i] L-bar[j][k] for i >= k
    if (row) {
        for (int i = 0; i < q; ++i) {
            double v = 0.0;
            if (i >= lane) {
                for (int j = i; j < q; ++j) v = fma(L[j * ld + i], Lb[j * ld + lane], v);
                if (i == lane) v *= 0.5;
            }
            Sg[i * ld + lane] = v;
        }
    }
    __syncwarp();
    // Y = Phi L^-1 (Y L = Phi, row by row; Y is lower triangular): lane r, k descending
    if (row) {
        for (int j = lane + 1; j < q; ++j) Y[lane * ld + j] = 0.0;
        for (int k = lane; k >= 0; --k) {
            double v = Sg[lane * ld + k];
            for (int i = k + 1; i <= lane; ++i) v -= Y[lane * ld + i] * L[i * ld + k];
            Y[lane * ld + k] = v / L[k * ld + k];
        }
    }
    __syncwarp();
    // A-bar = L^-T Y (L^T A-bar = Y, column by column): lane c, k descending; A-bar into Lb
    if (row) {
        for (int k = q - 1; k >= 0; --k) {
            double v = Y[k * ld + lane];
            for (int i = k + 1; i < q; ++i) v -= L[i * ld + k] * Lb[i * ld + lane];
            Lb[k * ld + lane] = v / L[k * ld + k];
        }
    }
    __syncwarp();
    if (row)
        for (int j = 0; j < q; ++j)
            Cout[((int64_t)b * q + lane) * q + j] = 0.5 * (Lb[lane * ld + j] + Lb[j * ld + lane]);
}

// R[r][b q + c] = sum_j 2 C_b[c][j] Z[r][b q + j] (j ascending) for the ncols = nb q columns of the chunk.  grid (ceil(ncols /
// 128), Npad), 128 threads.
__global__ void __launch_bounds__(128) qei_combine_kernel(const double* __restrict__ Z, int64_t ld, int q, int64_t ncols,
                                                          const double* __restrict__ C, double* __restrict__ R) {
    const int64_t col = blockIdx.x * 128LL + threadIdx.x, r = blockIdx.y;
    if (col >= ncols) return;
    const int64_t b = col / q;
    const int c = (int)(col - b * q);
    const double* z = Z + r * ld + b * q;
    const double* cr = C + (b * q + c) * q;
    double v = 0.0;
    for (int j = 0; j < q; ++j) v = fma(2.0 * cr[j], z[j], v);
    R[r * ld + col] = v;
}

// One thread per point c = b q + i of the chunk:
//   grad[c][t] = dmu[c] sum_pb part_mu - sum_pb part_R + sum_{j != i} 2 C_b[i][j] d k(x_c, x_{b q + j}) / d x_c[t],
// d k / d x_c[t] = 2 s_t sigma^2 phi'(u) s_t (x_c[t] - x_j[t]); NaN for a batch whose Cholesky failed (tau NaN).
__global__ void qei_grad_finish_kernel(KSpec spec, const double* __restrict__ Xb, int q, int64_t ncols,
                                       const double* __restrict__ part, int npb, int64_t mpad, const double* __restrict__ dmu,
                                       const double* __restrict__ C, const double* __restrict__ tau, double* __restrict__ grad) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= ncols) return;
    const int d = spec.d;
    const int64_t b = c / q;
    const int i = (int)(c - b * q);
    double* gout = grad + c * d;
    if (tau[b] != tau[b]) {
        for (int t = 0; t < d; ++t) gout[t] = CUDART_NAN;
        return;
    }
    const double dm = dmu[c];
    const double* xc = Xb + c * d;
    // coordinate by coordinate (the prior pairs are re-evaluated per coordinate: no per-point arrays, no local memory)
    for (int t = 0; t < d; ++t) {
        double gm = 0.0, gv = 0.0;
        for (int pb = 0; pb < npb; ++pb) {
            gm += part[(((int64_t)pb * mpad + c) * 2 + 0) * AG_MAXD + t];
            gv += part[(((int64_t)pb * mpad + c) * 2 + 1) * AG_MAXD + t];
        }
        double g = dm * gm - gv;
        for (int j = 0; j < q; ++j) {
            if (j == i) continue;
            const double* xj = Xb + (b * q + j) * d;
            double u = 0.0;
            for (int k = 0; k < d; ++k) {
                const double df = spec.sk(k) * xc[k] - spec.sk(k) * xj[k];
                u = fma(df, df, u);
            }
            double p, dp, ddp;
            phi_eval(spec.kind, u, p, dp, ddp);
            const double Dt = spec.sk(t) * xc[t] - spec.sk(t) * xj[t];
            g = fma(2.0 * C[(b * q + i) * q + j], gk_entry(spec, p, dp, ddp, t + 1, 0, Dt, 0.0), g);
        }
        gout[t] = g;
    }
}

}  // namespace abo
