// acq_multi.cuh — GradientNormUCB (src/acquisition_functions/gradNormUCB.jl:43-51) and EnsembleAcquisition
// (EnsembleAcq.jl:53-55) on the device, ONE posterior pass shared by all members.
// Per candidate x*:   K*_b = gradKernel((X, all outputs), (x*, b)),  b = 0..d        (ks_build_kernel, one output at a time)
//                     W_b  = L^-1 K*_b                                              (DMMA triangular GEMM, all b and candidates at once)
//                     mean_b = c_b + K*_b^T alpha ;   Sigma_bb' = prior_bb' - W_b^T W_b' + 1e-18 delta_bb'
//                     GradientNormUCB: m = mean[1:], S = Sigma[1:,1:]:  -(m.m + tr S) + beta sqrt(max(4 m^T S m + 2 |S|_F^2, 1e-12))
//                     EI / PI / UCB members: acq_value(mean_0, Sigma_00)
// Only the p x p diagonal blocks of the (m p)^2 posterior covariance are ever formed (the host version built all of it).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels.cuh"

namespace abo {

constexpr int AM_MAXMEM = 8;      // ensemble members
constexpr int AM_ROWS = 512;      // rows of W per partial block
struct MultiSpec {
    int nmem;
    double w[AM_MAXMEM];
    AcqSpec acq[AM_MAXMEM];       // EI, PI, UCB or GradientNormUCB (p0 = beta)
};

// part[chunk][pair][c] = sum_{i in chunk} W[i][b*mp + c] * W[i][b2*mp + c],  pair = b(b+1)/2 + b2, b2 <= b < nout
// thread = (pair, candidate) with the candidate fastest: coalesced along c
__global__ void __launch_bounds__(256) gram_blocks_partial_kernel(const double* __restrict__ W, int64_t ldw, int64_t N, int64_t mp, int64_t mc,
                                                                  int nout, double* __restrict__ part) {
    const int npair = nout * (nout + 1) / 2;
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    if (t >= (int64_t)npair * mc) return;
    const int pair = (int)(t / mc);
    const int64_t c = t % mc;
    int b = 0;
    while ((b + 1) * (b + 2) / 2 <= pair) ++b;
    const int b2 = pair - b * (b + 1) / 2;
    const int64_t i0 = (int64_t)blockIdx.y * AM_ROWS;
    const int64_t i1 = (i0 + AM_ROWS < N) ? i0 + AM_ROWS : N;
    const double* w1 = W + (int64_t)b * mp + c;
    const double* w2 = W + (int64_t)b2 * mp + c;
    double acc = 0.0;
#pragma unroll 4
    for (int64_t i = i0; i < i1; ++i) acc = fma(w1[i * ldw], w2[i * ldw], acc);
    part[((int64_t)blockIdx.y * npair + pair) * mc + c] = acc;
}

// one thread per candidate: posterior means and p x p covariance block -> weighted sum of the members
constexpr int AM_MAXP = 33;
__global__ void __launch_bounds__(128) acq_multi_finish_kernel(KSpec spec, MultiSpec ms, const double* __restrict__ mean_c,
                                                               const double* __restrict__ pmean, int npb, int64_t Mpad,
                                                               const double* __restrict__ part, int nchunks, int64_t mp, int64_t mc,
                                                               int nout, double* __restrict__ score) {
    const int64_t c = blockIdx.x * 128LL + threadIdx.x;
    if (c >= mc) return;
    const int npair = nout * (nout + 1) / 2;
    double mu[AM_MAXP];
    for (int b = 0; b < nout; ++b) {
        double s = 0.0;
        for (int pb = 0; pb < npb; ++pb) s += pmean[(int64_t)pb * Mpad + (int64_t)b * mp + c];
        mu[b] = s + mean_c[b];
    }
    double ph, dph, ddph;
    phi_eval(spec.kind, 0.0, ph, dph, ddph);
    const double kvv = spec.scale * ph;                   // prior variances (off-diagonals vanish at D = 0); gradient output b: -2 s_b^2 sig2 phi'(0)
    auto sigma = [&](int b, int b2) {                     // posterior covariance of outputs b >= b2 at this point
        double g = 0.0;
        const int pair = b * (b + 1) / 2 + b2;
        for (int ch = 0; ch < nchunks; ++ch) g += part[((int64_t)ch * npair + pair) * mc + c];
        const double kgg = (b > 0) ? -2.0 * spec.sk(b - 1) * spec.sk(b - 1) * spec.scale * dph : 0.0;
        return ((b == b2) ? (b == 0 ? kvv : kgg) : 0.0) - g + ((b == b2) ? JITTER : 0.0);
    };
    double total = 0.0;
    bool need_grad = false;
    for (int q = 0; q < ms.nmem; ++q) need_grad |= ms.acq[q].acq == ACQ_GRADNORM_UCB;
    double gn_mu = 0.0, gn_var = 0.0;
    if (need_grad) {
        // mu_sq = m.m + tr S ;  var_sq = 4 m^T S m + 2 sum S_ij^2      (S symmetric: off-diagonals counted twice)
        double mm = 0.0, tr = 0.0, msm = 0.0, fro = 0.0;
        for (int b = 1; b < nout; ++b) {
            mm = fma(mu[b], mu[b], mm);
            for (int b2 = 1; b2 <= b; ++b2) {
                const double sg = sigma(b, b2);
                if (b == b2) { tr += sg; msm = fma(mu[b] * mu[b], sg, msm); fro = fma(sg, sg, fro); }
                else { msm = fma(2.0 * mu[b] * mu[b2], sg, msm); fro = fma(2.0 * sg, sg, fro); }
            }
        }
        gn_mu = mm + tr;
        gn_var = 4.0 * msm + 2.0 * fro;
    }
    const double var0 = sigma(0, 0);
    for (int q = 0; q < ms.nmem; ++q) {
        double v;
        if (ms.acq[q].acq == ACQ_GRADNORM_UCB) v = -gn_mu + ms.acq[q].p0 * sqrt(fmax(gn_var, 1e-12));
        else v = acq_value(ms.acq[q], mu[0], var0);
        total = fma(ms.w[q], v, total);
    }
    score[c] = total;
}

// members that only need the value output: combine from (mean, var)
__global__ void acq_multi_combine_kernel(MultiSpec ms, const double* __restrict__ mean, const double* __restrict__ var, int64_t m,
                                         double* __restrict__ score) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= m) return;
    double total = 0.0;
    for (int q = 0; q < ms.nmem; ++q) total = fma(ms.w[q], acq_value(ms.acq[q], mean[c], var[c]), total);
    score[c] = total;
}

}  // namespace abo
