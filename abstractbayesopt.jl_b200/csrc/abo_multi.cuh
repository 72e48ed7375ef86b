// abo_multi.cuh — abo_acq_eval_multi: EnsembleAcquisition / GradientNormUCB with one shared posterior pass.
// Included at the end of abo_api.cu (one translation unit owns every __global__ definition).
#include "acq_multi.cuh"

extern "C" int32_t abo_acq_eval_multi(abo_gp* g, int32_t nmem, const int32_t* acq_ids, const double* weights, const double* params,
                                      const double* Xc, int64_t m, double* scores, int64_t k, int64_t* top_idx, double* top_val) {
    if (!acq_ids || !weights) return abo_fail(ABO_ERR_INVALID, "null argument");
    int rc = acq_check(g, params, Xc, m, k, top_idx, top_val);
    if (rc) return rc;
    if (nmem < 1 || nmem > AM_MAXMEM) return abo_fail(ABO_ERR_INVALID, "1 <= members <= %d", AM_MAXMEM);
    MultiSpec ms;
    ms.nmem = nmem;
    bool need_grad = false;
    for (int q = 0; q < nmem; ++q) {            // ABO_ACQ_MES is not a member
        if (acq_ids[q] < ACQ_EI || acq_ids[q] > ACQ_GRADNORM_UCB) return abo_fail(ABO_ERR_INVALID, "unknown acquisition id %d", acq_ids[q]);
        ms.acq[q] = with_acq(AcqSpec{}, acq_ids[q], params + 2 * q);
        ms.w[q] = weights[q];
        need_grad |= acq_ids[q] == ACQ_GRADNORM_UCB;
    }
    if (need_grad && g->p < 2) return abo_fail(ABO_ERR_INVALID, "GradientNormUCB needs a GradientGP surrogate (p = d + 1)");
    if (g->p > AM_MAXP) return abo_fail(ABO_ERR_INVALID, "abo_acq_eval_multi supports p <= %d", AM_MAXP);
    if (m == 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int d = g->d;
    double *dXc, *dS;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * d, (void**)&dXc))) return rc;
    if ((rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)m, (void**)&dS))) return rc;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * d, cudaMemcpyHostToDevice, st));
    if (!need_grad) {
        // value output only: the (fused) sweep gives mean and variance once, every member is a formula on them
        double *dM, *dV;
        if ((rc = ws_get(c, WS_OUT_B, sizeof(double) * (size_t)m * 2, (void**)&dM))) return rc;
        dV = dM + m;
        if ((rc = sweep_device(g, dXc, m, 0, AcqSweep{prior_spec(g, 0)}, dM, dV, nullptr))) return rc;
        acq_multi_combine_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(ms, dM, dV, m, dS);
        KL(c);
        return scores_select_readback(c, dS, m, scores, k, top_idx, top_val);
    }
    const int p = g->p;
    const int64_t Npad = g->Npad;
    const int64_t mp_max = std::max<int64_t>(KS_CB, (4096 / p) / KS_CB * KS_CB);      // candidates per pass: p * mp <= 4096 columns
    const int64_t Mcap = (mp_max * p + NB - 1) / NB * NB;
    const int64_t vpts = (Npad + p - 1) / p;
    const int npb = (int)((vpts + 127) / 128);
    const int nchunks = (int)((g->N + AM_ROWS - 1) / AM_ROWS);
    const int npair = p * (p + 1) / 2;
    double *Ks, *pmean, *W, *part;
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)Mcap * Npad, (void**)&Ks))) return rc;
    if ((rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * Mcap, (void**)&pmean))) return rc;
    if ((rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)Mcap * Npad, (void**)&W))) return rc;
    if ((rc = ws_get(c, WS_GRAD_PART, sizeof(double) * (size_t)nchunks * npair * mp_max, (void**)&part))) return rc;
    for (int64_t c0 = 0; c0 < m; c0 += mp_max) {
        const int64_t mc = std::min(mp_max, m - c0);
        const int64_t mp = (mc + KS_CB - 1) / KS_CB * KS_CB;
        const int64_t Mpad = (mp * p + NB - 1) / NB * NB;
        CU(cudaMemsetAsync(Ks + (size_t)mp * p * Npad, 0, sizeof(double) * (size_t)(Mpad - mp * p) * Npad, st));   // padding rows
        for (int bo = 0; bo < p; ++bo)
            if ((rc = launch_ks_d(c, g, dXc, c0, m, bo, Ks + (size_t)bo * mp * Npad, pmean + (size_t)bo * mp, mp, Mpad, npb, st))) return rc;
        if ((rc = linv_times_ks(c, g, Ks, Mpad, W, st))) return rc;      // W = L^-1 K*^T  [Npad][Mpad] on the TMA pipeline
        gram_blocks_partial_kernel<<<dim3((unsigned)(((int64_t)npair * mc + 255) / 256), nchunks), 256, 0, st>>>(W, Mpad, g->N, mp, mc, p, part);
        KL(c);
        acq_multi_finish_kernel<<<(unsigned)((mc + 127) / 128), 128, 0, st>>>(gp_spec(g), ms, g->dMeanC, pmean, npb, Mpad, part, nchunks, mp,
                                                                             mc, p, dS + c0);
        KL(c);
    }
    return scores_select_readback(c, dS, m, scores, k, top_idx, top_val);
}

// ------------------------------------------------------------------------------------------
// abo_standardize — get_mean_std + std_y of standardize_problem (src/BO_utils.jl:44-64, StandardGP.jl:164-204,
// GradientGP.jl:756-783) on the device: mean (pairwise tree), corrected sample standard deviation (two-pass), the
// standardised observations and the incumbent min of the standardised value output, one launch.
//   StandardGP (p = 1): y_std = (y - mu) / sd.   GradientGP: mu = (mean of the VALUE output, 0, ...), sd = std of the value
//   output for every output; y_std[a] = (y[a] - mu[a]) / sd[0].   choice: 0 mean_scale, 1 scale_only (mu = 0), 2 mean_only (sd = 1).
// ------------------------------------------------------------------------------------------
namespace abo {
__global__ void __launch_bounds__(1024) standardize_kernel(const double* __restrict__ y, int64_t n, int p, int choice,
                                                           double* __restrict__ y_std, double* __restrict__ out /* mu, sd, best */) {
    __shared__ double sh[1024];
    __shared__ double s_mu, s_sd;
    const int t = threadIdx.x;
    auto reduce = [&](double v, bool take_min) {
        sh[t] = v;
        __syncthreads();
        for (int o = 512; o > 0; o >>= 1) {
            if (t < o) sh[t] = take_min ? fmin(sh[t], sh[t + o]) : sh[t] + sh[t + o];
            __syncthreads();
        }
        const double r = sh[0];
        __syncthreads();
        return r;
    };
    double acc = 0.0;
    for (int64_t i = t; i < n; i += 1024) acc += y[i];                  // value output = the first n entries (out-major)
    const double mean = reduce(acc, false) / (double)n;
    acc = 0.0;
    for (int64_t i = t; i < n; i += 1024) { const double dv = y[i] - mean; acc = fma(dv, dv, acc); }
    const double sd_raw = sqrt(reduce(acc, false) / (double)(n - 1));
    if (t == 0) { s_mu = (choice == 1) ? 0.0 : mean; s_sd = (choice == 2) ? 1.0 : sd_raw; }
    __syncthreads();
    const double mu = s_mu, sd = s_sd;
    double best = CUDART_INF;
    for (int64_t i = t; i < n * p; i += 1024) {
        const double v = (y[i] - (i < n ? mu : 0.0)) / sd;
        y_std[i] = v;
        if (i < n) best = fmin(best, v);
    }
    best = reduce(best, true);
    if (t == 0) { out[0] = mu; out[1] = sd; out[2] = best; }
}
}  // namespace abo

extern "C" int32_t abo_standardize(abo_ctx* c, const double* y, int64_t n, int32_t p, int32_t choice, double* mu, double* sd,
                                   double* y_std, double* best) {
    if (!c || !y || !mu || !sd || !y_std) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (n < 2 || p < 1) return abo_fail(ABO_ERR_DIM, "standardisation needs at least two observations");
    if (choice < 0 || choice > 2) return abo_fail(ABO_ERR_INVALID, "choice must be 0 (mean_scale), 1 (scale_only) or 2 (mean_only)");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    double *dy, *dout;
    int rc;
    if ((rc = ws_get(c, WS_STAGE_Y, sizeof(double) * (size_t)(2 * n * p + 8), (void**)&dy))) return rc;
    dout = dy + 2 * n * p;
    CU(cudaMemcpyAsync(dy, y, sizeof(double) * n * p, cudaMemcpyHostToDevice, st));
    standardize_kernel<<<1, 1024, 0, st>>>(dy, n, p, choice, dy + n * p, dout);
    KL(c);
    double h[3];
    CU(cudaMemcpyAsync(y_std, dy + n * p, sizeof(double) * n * p, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h, dout, sizeof(h), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int a = 0; a < p; ++a) { mu[a] = a == 0 ? h[0] : 0.0; sd[a] = h[1]; }
    if (best) *best = h[2];
    return ABO_OK;
}
