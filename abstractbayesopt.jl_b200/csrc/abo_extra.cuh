// abo_extra.cuh — O(n^2) row append and the batched NLML (+ analytic gradient) entry points.
// Included at the end of abo_api.cu (one translation unit owns every __global__ definition).
#include <algorithm>
#include <cmath>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/abo.h"
#include "gemm_dmma.cuh"
#include "kernels.cuh"
#include "abo_internal.h"

using namespace abo;

static KSpec spec_of(const abo_gp* g) {
    KSpec k;
    k.kind = g->kind; k.d = g->d; k.p = g->p; k.s = g->s; k.scale = g->scale; k.noise = g->noise;
    for (int q = 0; q < ARD_MAXD; ++q) k.sv[q] = (q < g->d && q < (int)g->sv.size()) ? g->sv[q] : g->s;
    return k;
}

// ------------------------------------------------------------------------------------------
// abo_gp_append — one new observation, O(n^2):
//   w = L^-1 k(X, x)           (TRMV, reads L^-1 once)
//   pivot = k(x,x) + noise - |w|^2   -> not positive: ABO_ERR_NOT_POSDEF, state untouched
//   L[n,:] = [w, sqrt(pivot)] ;  L^-1[n,:] = [-(L^-T w)/l, 1/l]   (second pass over L^-1)
//   beta_n, alpha += L^-1[n,:]^T beta_n
// The reference has no such path (it re-fits, src/bayesian_opt.jl:125); the result equals a
// re-fit up to rounding (the GPU tests compare it with a full re-fit).
// ------------------------------------------------------------------------------------------
static int grow_capacity(abo_gp* g) {
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    const int64_t old_pad = g->cap_pad, new_pad = old_pad + NB;
    double *nL = nullptr, *nLinv = nullptr, *nA = nullptr, *nB = nullptr, *nD = nullptr;
    size_t mat = sizeof(double) * (size_t)new_pad * new_pad;
    cudaError_t e;
    if ((e = cudaMalloc(&nL, mat)) != cudaSuccess || (e = cudaMalloc(&nLinv, mat)) != cudaSuccess ||
        (e = cudaMalloc(&nA, sizeof(double) * new_pad)) != cudaSuccess ||
        (e = cudaMalloc(&nB, sizeof(double) * new_pad)) != cudaSuccess ||
        (e = cudaMalloc(&nD, sizeof(double) * new_pad)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(nL); cudaFree(nLinv); cudaFree(nA); cudaFree(nB); cudaFree(nD);
        return abo_fail(ABO_ERR_ALLOC, "growing the posterior to %lld rows failed: %s", (long long)new_pad, cudaGetErrorString(e));
    }
    const int64_t tot = new_pad * new_pad;
    grow_matrix_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(g->dL, old_pad, g->ld, nL, new_pad);
    KL(c);
    grow_matrix_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(g->dLinv, old_pad, g->ld, nLinv, new_pad);
    KL(c);
    CU(cudaMemsetAsync(nA, 0, sizeof(double) * new_pad, st));
    CU(cudaMemsetAsync(nB, 0, sizeof(double) * new_pad, st));
    CU(cudaMemsetAsync(nD, 0, sizeof(double) * new_pad, st));
    CU(cudaMemcpyAsync(nA, g->dAlpha, sizeof(double) * old_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(nB, g->dBeta, sizeof(double) * old_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(nD, g->dDelta, sizeof(double) * old_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaStreamSynchronize(st));
    cudaFree(g->dL); cudaFree(g->dLinv); cudaFree(g->dAlpha); cudaFree(g->dBeta); cudaFree(g->dDelta);
    g->dL = nL; g->dLinv = nLinv; g->dAlpha = nA; g->dBeta = nB; g->dDelta = nD;
    g->cap_pad = new_pad; g->ld = new_pad; g->Npad = new_pad;
    return ABO_OK;
}

static int grow_points(abo_gp* g) {
    abo_ctx* c = g->ctx;
    const int64_t new_ldx = g->ldx + 4 * NB;
    double* nX = nullptr;
    cudaError_t e = cudaMalloc(&nX, sizeof(double) * (size_t)new_ldx * g->d);
    if (e != cudaSuccess) { cudaGetLastError(); return abo_fail(ABO_ERR_ALLOC, "growing the coordinate store failed"); }
    CU(cudaMemsetAsync(nX, 0, sizeof(double) * new_ldx * g->d, c->stream));
    CU(cudaMemcpy2DAsync(nX, sizeof(double) * new_ldx, g->dXsT, sizeof(double) * g->ldx, sizeof(double) * g->ldx, g->d,
                         cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    cudaFree(g->dXsT);
    g->dXsT = nX; g->ldx = new_ldx;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// block append for a GradientGP: the p = d + 1 outputs of ONE new point become the last p rows of
// the (point-major) system.
//   Kn = K((X, all outputs), (x, b)), b < p       (K* builder, one output at a time)
//   W  = L^-1 Kn ,  S = Knn + noise I - W^T W  ->  host Cholesky S = LS LS^T (p x p; failure leaves the
//   posterior untouched),  Z = L^-T W
//   L_new = [[L, 0], [W^T, LS]] ,  Linv_new = [[Linv, 0], [-LS^-1 Z^T, LS^-1]]
//   beta_new = LS^-1 (delta_new - W^T beta) ,  alpha = [alpha - Z gamma ; gamma],  gamma = LS^-T beta_new
// O(N^2 p) instead of the O(N^3) re-fit of GradientGP.jl:659-668.
// ------------------------------------------------------------------------------------------
static int append_block(abo_gp* g, const double* x, const double* y, int64_t* info_out) {
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int p = g->p, d = g->d;
    if (p > 96) return abo_fail(ABO_ERR_INVALID, "block append supports p <= 96");
    const int64_t N = g->N, Npad = g->Npad;
    const int64_t vpts = (Npad + p - 1) / p;
    const int npb = (int)((vpts + 127) / 128);
    const int64_t WB = NB;                                    // padded width of the p-column operands
    int rc;
    double *dx, *Ks, *pmean, *W, *Z, *G, *dsmall;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)d, (void**)&dx))) return rc;
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)WB * Npad, (void**)&Ks))) return rc;
    if ((rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * WB, (void**)&pmean))) return rc;
    if ((rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)WB * Npad, (void**)&W))) return rc;
    if ((rc = ws_get(c, WS_GRAD_Z, sizeof(double) * (size_t)WB * Npad, (void**)&Z))) return rc;
    if ((rc = ws_get(c, WS_GRAD_OUT, sizeof(double) * (size_t)WB * WB, (void**)&G))) return rc;
    const int nsmall = 2 * p * p + 3 * p + d;
    if ((rc = ws_get(c, WS_APPEND, sizeof(double) * (size_t)(nsmall + p * p + p + 8), (void**)&dsmall))) return rc;
    double* dstats = dsmall + nsmall;                          // S | wb
    CU(cudaMemcpyAsync(dx, x, sizeof(double) * d, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(Ks, 0, sizeof(double) * (size_t)WB * Npad, st));
    // row b of Ks = column b of Kn; every launch also zeroes the 31 rows after its own, later launches overwrite them
    for (int b = 0; b < p; ++b)
        if ((rc = launch_ks_d(c, g, dx, 0, 1, b, Ks + (size_t)b * Npad, pmean, KS_CB, WB, npb, st))) return rc;
    // W = L^-1 Kn [N][WB], G = W^T W: p right-hand sides only -> bandwidth-bound passes over the triangle
    // (128-wide padded GEMM tiles would run on 44 CTAs with k-loops of up to N)
    const int ngrp = (p + 7) / 8;
    trmm_skinny_lower_kernel<<<dim3((unsigned)((N * 32 + 255) / 256), ngrp), 256, 0, st>>>(g->dLinv, g->ld, N, Ks, Npad, p, W, WB);
    KL(c);
    gram_skinny_kernel<<<dim3(p, p), 256, 0, st>>>(W, WB, N, G, WB);
    KL(c);
    append_block_stats_kernel<<<1, 256, 0, st>>>(spec_of(g), G, WB, W, WB, g->dBeta, N, dstats);
    KL(c);
    std::vector<double> hs((size_t)p * p + p);
    CU(cudaMemcpyAsync(hs.data(), dstats, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(c->ev_a, st));
    {   // Z = L^-T W, launched now so that it overlaps the host Cholesky
        const int nchunks = (int)((N + TRMVT_ROWS - 1) / TRMVT_ROWS);
        double* part;
        if ((rc = ws_get(c, WS_VEC_PART, sizeof(double) * (size_t)nchunks * p * N, (void**)&part))) return rc;
        trmmT_skinny_partial_kernel<<<dim3((unsigned)((N + 127) / 128), nchunks, ngrp), 128, 0, st>>>(g->dLinv, g->ld, N, W, WB, p, part);
        KL(c);
        trmmT_skinny_reduce_kernel<<<dim3((unsigned)((N + 127) / 128), p), 128, 0, st>>>(part, nchunks, N, p, Z, WB);
        KL(c);
    }
    CU(cudaEventSynchronize(c->ev_a));                         // S and wb are on the host; Z is still being computed
    // host: Cholesky of S, its inverse, beta_new, gamma
    std::vector<double> small((size_t)nsmall, 0.0);
    double* LS = small.data(); double* LSi = LS + p * p; double* bnew = LSi + p * p; double* gamma = bnew + p;
    double* dnew = gamma + p; double* hx = dnew + p;
    const double* S = hs.data(); const double* wb = S + p * p;
    for (int a = 0; a < p; ++a) {
        for (int b = 0; b <= a; ++b) {
            double v = S[a * p + b];
            for (int k = 0; k < b; ++k) v -= LS[a * p + k] * LS[b * p + k];
            if (a == b) {
                if (!(v > 0.0)) {
                    if (info_out) *info_out = N + a + 1;
                    return abo_fail(ABO_ERR_NOT_POSDEF, "matrix is not positive definite; Cholesky factorization failed at pivot %lld",
                                    (long long)(N + a + 1));
                }
                LS[a * p + a] = std::sqrt(v);
            } else {
                LS[a * p + b] = v / LS[b * p + b];
            }
        }
    }
    if (info_out) *info_out = 0;
    for (int j = 0; j < p; ++j) {                              // LSi = LS^-1 (lower), column by column
        LSi[j * p + j] = 1.0 / LS[j * p + j];
        for (int a = j + 1; a < p; ++a) {
            double v = 0.0;
            for (int k = j; k < a; ++k) v -= LS[a * p + k] * LSi[k * p + j];
            LSi[a * p + j] = v / LS[a * p + a];
        }
    }
    for (int a = 0; a < p; ++a) dnew[a] = y[a] - g->mean_c[a];
    for (int a = 0; a < p; ++a) {
        double v = 0.0;
        for (int b = 0; b <= a; ++b) v += LSi[a * p + b] * (dnew[b] - wb[b]);
        bnew[a] = v;
    }
    for (int a = 0; a < p; ++a) {
        double v = 0.0;
        for (int b = a; b < p; ++b) v += LSi[b * p + a] * bnew[b];
        gamma[a] = v;
    }
    for (int k = 0; k < d; ++k) hx[k] = x[k];
    if ((rc = gp_unshare(g))) return rc;                       // copy-on-write: clones keep the un-appended posterior
    while (N + p > g->cap_pad) { if ((rc = grow_capacity(g))) return rc; }
    if (g->n + 1 > g->ldx) { if ((rc = grow_points(g))) return rc; }
    CU(cudaMemcpyAsync(dsmall, small.data(), sizeof(double) * nsmall, cudaMemcpyHostToDevice, st));
    append_block_commit_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(g->dL, g->dLinv, g->ld, N, p, W, Z, WB, dsmall, g->dDelta,
                                                                           g->dBeta, g->dAlpha, g->dXsT, g->ldx, g->n, d, spec_of(g));
    KL(c);
    CU(cudaStreamSynchronize(st));
    g->n += 1; g->N += p;
    return ABO_OK;
}

extern "C" int32_t abo_gp_append(abo_gp* g, const double* x, const double* y, int64_t* info_out) {
    if (!g || !x || !y) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "append needs a fitted surrogate (call abo_gp_fit first)");
    if (g->p != 1) return append_block(g, x, y, info_out);
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t n = g->n;
    int rc;
    // scratch: xnew[d] | kv[Npad] | w[Npad] | r[Npad] | ss[1]
    const int64_t Np = g->Npad;
    double* buf;
    if ((rc = ws_get(c, WS_APPEND, sizeof(double) * (size_t)(g->d + 3 * Np + 8), (void**)&buf))) return rc;
    double *dx = buf, *kv = buf + g->d, *w = kv + Np, *r = w + Np, *ss = r + Np;
    CU(cudaMemcpyAsync(dx, x, sizeof(double) * g->d, cudaMemcpyHostToDevice, st));
    kvec_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, st>>>(spec_of(g), g->dXsT, g->ldx, n, Np, dx, kv);
    KL(c);
    {
        dim3 grid((unsigned)((n * 32 + 255) / 256), 1);
        trmv_lower_kernel<<<grid, 256, 0, st>>>(g->dLinv, g->ld, n, kv, w, 0, 0);
        KL(c);
    }
    sumsq_vec_kernel<<<1, 1024, 0, st>>>(w, n, ss);
    KL(c);
    double hss = 0.0;
    CU(cudaMemcpyAsync(&hss, ss, sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const double piv = (g->scale + g->noise) - hss;          // k(x,x) = sig2 * phi(0) = sig2
    if (!(piv > 0.0)) {
        if (info_out) *info_out = n + 1;
        return abo_fail(ABO_ERR_NOT_POSDEF, "matrix is not positive definite; Cholesky factorization failed at pivot %lld",
                        (long long)(n + 1));
    }
    if (info_out) *info_out = 0;
    const double l = std::sqrt(piv);
    // r = Linv^T w over rows 0..n-1
    const int nchunks = (int)((n + TRMVT_ROWS - 1) / TRMVT_ROWS);
    double* part;                              // sized by the padded dimension: no re-allocation as n grows
    if ((rc = ws_get(c, WS_VEC_PART, sizeof(double) * (size_t)(Np / TRMVT_ROWS + 2) * (Np + NB), (void**)&part))) return rc;
    {
        dim3 grid((unsigned)((n + 127) / 128), nchunks, 1);
        trmvT_lower_partial_kernel<<<grid, 128, 0, st>>>(g->dLinv, g->ld, n, w, part, 0, 0, 0);
        KL(c);
        reduce_rows_kernel<<<dim3((unsigned)((n + 127) / 128), 1), 128, 0, st>>>(part, nchunks, n, r, 0, 0);
        KL(c);
    }
    if ((rc = gp_unshare(g))) return rc;      // copy-on-write: clones keep the un-appended posterior
    if (n + 1 > g->cap_pad) {                 // no padding row left: one more tile
        if ((rc = grow_capacity(g))) return rc;
    }
    if (n + 1 > g->ldx) { if ((rc = grow_points(g))) return rc; }
    append_commit_kernel<<<1, 1024, 0, st>>>(g->dL, g->dLinv, g->ld, n, w, r, l, y[0] - g->mean_c[0], g->dDelta, g->dBeta,
                                             g->dAlpha, g->dXsT, g->ldx, dx, g->d, spec_of(g));
    KL(c);
    CU(cudaStreamSynchronize(st));
    g->n = n + 1; g->N = n + 1;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// abo_nlml_batch — R hyper-parameter vectors in lock-step:
//   K_b + noise I (batched kmat) -> batched blocked Cholesky -> batched triangular inverse ->
//   beta_b, alpha_b -> Cinv_b = Linv_b^T Linv_b (DMMA, structurally-zero k skipped) ->
//   fused reduction  sum (Cinv - alpha alpha^T) .* dK/dtheta  with dK recomputed from X.
// ------------------------------------------------------------------------------------------
static int nlml_batch_impl(abo_gp* g, const double* X, const double* y, int64_t n, const double* logparams,
                           int64_t R, double* nlml, double* grad, int32_t* info, bool ard) {
    if (!g || !X || !y || !logparams || !nlml) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (ard && (g->p != 1 || g->d > ARD_MAXD))
        return abo_fail(ABO_ERR_INVALID, "the ARD marginal likelihood is implemented for StandardGP (p = 1) with d <= %d", ARD_MAXD);
    if (n < 1) return abo_fail(ABO_ERR_DIM, "need at least one observation");
    if (R <= 0) return ABO_OK;
    if (!g->ctx) return abo_fail(ABO_ERR_INVALID, "the context of this handle has been destroyed");
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int d = g->d, p = g->p;
    const int np_ = ard ? d + 1 : 2;                      // parameters (and gradient components) per restart
    const int ns_ = ard ? d : 1;                          // inverse length scales per restart
    const int64_t N = n * p, Npad = (N + NB - 1) / NB * NB, ldx = (n + NB - 1) / NB * NB;
    const int T = (int)(Npad / NB);
    const size_t mat = sizeof(double) * (size_t)Npad * Npad;
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    size_t budget = std::min<size_t>((size_t)24 << 30, free_b / 2);
    int64_t Rc = std::max<int64_t>(1, std::min<int64_t>(R, (int64_t)(budget / (4 * mat))));
    int rc;
    double *Kb, *Linv, *W, *Ub, *Xb, *vec, *par, *Dinv, *dXraw, *dYraw;
    int* dinfo;
    if ((rc = ws_get(c, WS_NLML_K, mat * Rc, (void**)&Kb))) return rc;
    if ((rc = ws_get(c, WS_NLML_LINV, mat * Rc, (void**)&Linv))) return rc;
    if ((rc = ws_get(c, WS_NLML_W, mat * Rc, (void**)&W))) return rc;
    // U = (L^-1)^T of every matrix: keeps all GEMM operands k-contiguous (gemm_tma.cuh)
    if ((rc = ws_get(c, WS_NLML_U, mat * Rc, (void**)&Ub))) return rc;
    if ((rc = ws_get(c, WS_NLML_X, sizeof(double) * (size_t)Rc * ldx * d, (void**)&Xb))) return rc;
    // vec: delta[Rc][Npad] | beta | alpha | out[Rc][1 + np]
    if ((rc = ws_get(c, WS_NLML_VEC, sizeof(double) * (size_t)Rc * (3 * Npad + 2 + np_), (void**)&vec))) return rc;
    // par: s[Rc][ns] | scale[Rc] | tile partials [Rc][T*T][np]
    if ((rc = ws_get(c, WS_NLML_PAR, sizeof(double) * (size_t)Rc * (ns_ + 1 + np_ * (size_t)T * T), (void**)&par))) return rc;
    if ((rc = ws_get(c, WS_DINV, sizeof(double) * (size_t)Rc * T * NB * NB, (void**)&Dinv))) return rc;
    if ((rc = ws_get(c, WS_INFO, sizeof(int) * std::max<int64_t>(16, Rc), (void**)&dinfo))) return rc;
    if ((rc = ws_get(c, WS_STAGE_X, sizeof(double) * (size_t)n * d, (void**)&dXraw))) return rc;
    if ((rc = ws_get(c, WS_STAGE_Y, sizeof(double) * (size_t)(N + p), (void**)&dYraw))) return rc;
    double *delta = vec, *beta = vec + Rc * Npad, *alpha = beta + Rc * Npad, *out = alpha + Rc * Npad;
    double *sb = par, *scb = par + Rc * ns_, *tpart = par + Rc * (ns_ + 1);
    CU(cudaMemcpyAsync(dXraw, X, sizeof(double) * n * d, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dYraw, y, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dYraw + N, g->mean_c.data(), sizeof(double) * p, cudaMemcpyHostToDevice, st));
    std::vector<double> hs(Rc * ns_), hsc(Rc), hout((1 + np_) * Rc);
    std::vector<int> hinfo(Rc);
    KSpec spec = spec_of(g);
    for (int64_t r0 = 0; r0 < R; r0 += Rc) {
        const int nb = (int)std::min<int64_t>(Rc, R - r0);
        for (int b = 0; b < nb; ++b) {
            for (int k = 0; k < ns_; ++k) hs[b * ns_ + k] = std::exp(-logparams[np_ * (r0 + b) + k]);   // s = 1 / l
            hsc[b] = std::exp(logparams[np_ * (r0 + b) + np_ - 1]);
        }
        CU(cudaMemcpyAsync(sb, hs.data(), sizeof(double) * nb * ns_, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(scb, hsc.data(), sizeof(double) * nb, cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(dinfo, 0, sizeof(int) * nb, st));
        CU(cudaMemsetAsync(delta, 0, sizeof(double) * (size_t)nb * Npad, st));
        {
            int64_t tot = ldx * d;
            scale_transpose_batched_kernel<<<dim3((unsigned)((tot + 255) / 256), nb), 256, 0, st>>>(dXraw, Xb, n, d, ldx, sb, ard ? 1 : 0);
            KL(c);
            delta_batched_kernel<<<dim3((unsigned)((N + 255) / 256), nb), 256, 0, st>>>(dYraw, dYraw + N, n, p, delta, Npad);
            KL(c);
        }
        KmatBatch bt{sb, scb, ldx * d, Npad * Npad, ard ? 1 : 0};
        launch_kmat(spec, Xb, ldx, N, Kb, Npad, bt, T, nb, st);
        KL(c);
        if ((rc = potrf_blocked(c, Kb, Npad, Npad, Dinv, dinfo, nb))) return rc;
        if ((rc = trtri_tma(c, Kb, Linv, Ub, W, Npad, Npad, Npad * Npad, Dinv, (int64_t)T * NB * NB, nb))) return rc;
        if ((rc = solve_alpha(c, Linv, Npad, Npad, delta, beta, alpha, Npad * Npad, Npad, nb))) return rc;
        if (grad) {
            // Cinv = Linv^T Linv, lower tiles:  Cinv[m][n] = sum_k X[k][m] X[k][n] = sum_{k >= m} U[m][k] U[n][k]: both operands
            // rows of U, k-contiguous
            CUtensorMap tmU;
            if ((rc = make_tmap_k4(&tmU, Ub, Npad, (int64_t)nb * Npad, Npad))) return rc;
            TmaGemmParams t{};
            t.Mt = T; t.Nt = T; t.batch = nb; t.K = (int)Npad; t.flags = KLO_M | LOWER_ONLY; t.alpha = 1.0; t.beta = 0.0;
            t.a_row0 = 0; t.a_rstep = (int)Npad; t.a_col0 = 0; t.a_cstep = 0;
            t.b_row0 = 0; t.b_rstep = (int)Npad; t.b_col0 = 0; t.b_cstep = 0;
            t.C = W; t.ldc = Npad; t.c_off0 = 0; t.c_zstep = Npad * Npad;
            if ((rc = launch_gemm_tma(c, tmU, tmU, t, st))) return rc;
            if (ard) {
                const dim3 grid(T, T, nb);
                if (d <= 8) nlml_grad_ard_kernel<8><<<grid, 256, 0, st>>>(spec, bt, Xb, ldx, N, W, Npad, Npad * Npad, alpha, Npad, tpart);
                else if (d <= 20) nlml_grad_ard_kernel<20><<<grid, 256, 0, st>>>(spec, bt, Xb, ldx, N, W, Npad, Npad * Npad, alpha, Npad, tpart);
                else nlml_grad_ard_kernel<32><<<grid, 256, 0, st>>>(spec, bt, Xb, ldx, N, W, Npad, Npad * Npad, alpha, Npad, tpart);
            } else {
                launch_nlml_grad(spec, bt, Xb, ldx, N, W, Npad, Npad * Npad, alpha, Npad, tpart, T, nb, st);
            }
            KL(c);
        } else {
            CU(cudaMemsetAsync(tpart, 0, sizeof(double) * (size_t)nb * T * T * np_, st));
        }
        if (ard) nlml_finish_ard_kernel<<<nb, 256, 0, st>>>(Kb, Npad, Npad * Npad, N, beta, Npad, tpart, T * T, np_, dinfo, out);
        else nlml_finish_kernel<<<nb, 256, 0, st>>>(Kb, Npad, Npad * Npad, N, beta, Npad, tpart, T * T, dinfo, out);
        KL(c);
        CU(cudaMemcpyAsync(hout.data(), out, sizeof(double) * (1 + np_) * nb, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(hinfo.data(), dinfo, sizeof(int) * nb, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int b = 0; b < nb; ++b) {
            nlml[r0 + b] = hout[(1 + np_) * b];
            if (grad) for (int k = 0; k < np_; ++k) grad[np_ * (r0 + b) + k] = hout[(1 + np_) * b + 1 + k];
            if (info) info[r0 + b] = hinfo[b];
        }
    }
    if (4 * mat * Rc > ((size_t)16 << 30)) {       // an optimiser calls this in a loop: keep up to 16 GB of scratch resident
        ws_release(c, WS_NLML_K); ws_release(c, WS_NLML_LINV); ws_release(c, WS_NLML_W); ws_release(c, WS_NLML_U);
    }
    return ABO_OK;
}

extern "C" int32_t abo_nlml_batch(abo_gp* g, const double* X, const double* y, int64_t n, const double* logparams,
                                  int64_t R, double* nlml, double* grad, int32_t* info) {
    return nlml_batch_impl(g, X, y, n, logparams, R, nlml, grad, info, false);
}
extern "C" int32_t abo_nlml_batch_ard(abo_gp* g, const double* X, const double* y, int64_t n, const double* logparams,
                                      int64_t R, double* nlml, double* grad, int32_t* info) {
    return nlml_batch_impl(g, X, y, n, logparams, R, nlml, grad, info, true);
}
