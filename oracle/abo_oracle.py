"""CPU oracle for the GP-surrogate + acquisition hot path of AbstractBayesOpt.jl.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package imports this file; the only
callers are tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs, and there only as the checker or as the timed CPU baseline.

It is a NumPy/SciPy (OpenBLAS LAPACK) restatement of the reference's Float64 path.  The
reference is pure Julia and delegates the arithmetic to AbstractGPs 0.5 / KernelFunctions 0.10
/ Distributions 0.25 / ForwardDiff 1.2, none of which are vendored under /root/reference and
none of which can run in this image (no Julia).  Every function below cites the reference
call site it follows (paths relative to /root/reference) and, where the arithmetic lives in a
third-party package, restates that package's published algorithm.

Parity pinning: the oracle is pinned against the closed-form known-answer tests the
reference's own test-suite holds for this path (tests/test_oracle_golden.py reproduces
test/test_surrogates.jl:59-105,145-170,235-352, test/test_kernels.jl:40-88,205-254,
test/test_bayesian_opt.jl:552-558) and against a 50-digit mpmath arbiter.  EI / PI numeric
values and n > 8 behaviour are NOT pinned by any reference test ("parity unpinned" for those:
the source lines ExpectedImprovement.jl:59-66 and ProbabilityImprovement.jl:57-63 are the
only specification).

Conventions: X is (n, d) row-per-point; GradientGP outputs are "out-major"
idx = out * n + i (src/surrogates/GradientGP.jl:919-922, 937).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import scipy.linalg as sla
from scipy.special import erfc

# kernel ids shared with include/abo.h
SE, MATERN52, MATERN72, APPROX_MATERN52, APPROX_MATERN72, AD_MATERN52, AD_MATERN72 = range(7)
KERNEL_NAMES = ["se", "matern52", "matern72", "approx_matern52", "approx_matern72",
                "ad_matern52", "ad_matern72"]
EI, PI, UCB = 0, 1, 2

SQRT5 = math.sqrt(5.0)
SQRT7 = math.sqrt(7.0)
JITTER = 1e-18  # AbstractGPs default_σ² added by FiniteGP(posterior, x) (StandardGP.jl:361-379)


# --------------------------------------------------------------------------------------
# radial profiles  phi(u), phi'(u), phi''(u)   with u = || s (x - y) ||^2
# --------------------------------------------------------------------------------------
def phi_all(kind: int, u: np.ndarray, dtype=np.float64):
    """Kernel profile and its first two derivatives with respect to u = d^2.

    SE: KernelFunctions SqExponentialKernel kappa(d2) = exp(-d2/2) (metric SqEuclidean).
    MATERN52 / MATERN72: KernelFunctions Matern52Kernel/Matern72Kernel on d = sqrt(u).
    APPROX_*: src/surrogates/GradientGP.jl:94-101, 320-327 (Taylor branch for u < 1e-10;
      its ForwardDiff derivatives are those of the branch taken, so phi'' = 0 there).
    AD_*: src/surrogates/GradientGP.jl:176-209, 400-437 (closed forms, no threshold).
    """
    u = np.asarray(u, dtype=dtype)
    SQRT5, SQRT7 = np.sqrt(dtype(5.0)), np.sqrt(dtype(7.0))       # math.sqrt values for float64; 80-bit for the arbiter
    if kind == SE:
        p = np.exp(-u / 2)
        return p, -p / 2, p / 4
    r = np.sqrt(u)
    if kind in (MATERN52, APPROX_MATERN52, AD_MATERN52):
        z = np.exp(-SQRT5 * r)
        p = (1 + SQRT5 * r + 5 * u / 3) * z
        dp = (-5.0 / 6.0) * (1 + SQRT5 * r) * z
        ddp = (25.0 / 12.0) * z
        if kind == APPROX_MATERN52:
            small = u < 1e-10
            p = np.where(small, 1.0 - (5.0 / 6.0) * u, p)
            dp = np.where(small, -5.0 / 6.0, dp)
            ddp = np.where(small, 0.0, ddp)
        return p, dp, ddp
    if kind in (MATERN72, APPROX_MATERN72, AD_MATERN72):
        z = np.exp(-SQRT7 * r)
        p = (1 + SQRT7 * r + 14 * u / 5 + 7 * SQRT7 * r * u / 15) * z
        dp = (-7.0 / 10.0) * (1 + SQRT7 * r + 7 * u / 3) * z
        ddp = (49.0 / 60.0) * (1 + SQRT7 * r) * z
        if kind == APPROX_MATERN72:
            small = u < 1e-10
            p = np.where(small, 1.0 - (7.0 / 10.0) * u, p)
            dp = np.where(small, -7.0 / 10.0, dp)
            ddp = np.where(small, 0.0, ddp)
        return p, dp, ddp
    raise ValueError(f"unknown kernel id {kind}")


def sqdist(Xs: np.ndarray, Ys: np.ndarray, dtype=np.float64) -> np.ndarray:
    """Pairwise squared distances by DIRECT differences, sum_k (a_k - b_k)^2 — what
    KernelFunctions does for Vector{Vector{Float64}} inputs (SURVEY §3.2).  Inputs are the
    already scaled coordinates s*x (ScaleTransform is applied to coordinates first)."""
    n, d = Xs.shape
    m = Ys.shape[0]
    out = np.zeros((n, m), dtype=dtype)
    for k in range(d):  # sequential accumulation over coordinates, like the reference loop
        diff = Xs[:, k][:, None] - Ys[:, k][None, :]
        out += diff * diff
    return out


def kernelmatrix(kind: int, inv_ls: float, scale: float, X: np.ndarray, Y: np.ndarray | None = None, dtype=np.float64):
    """sigma^2 * kappa(metric(s x, s y))  — ScaledKernel(TransformedKernel(base, ScaleTransform(s)))
    as assembled at src/surrogates/StandardGP.jl:41-64 (s = 1/l is what is stored)."""
    sv = np.asarray(inv_ls, dtype=dtype)               # scalar (ScaleTransform) or one per dimension (ARDTransform)
    Xs = np.asarray(X, dtype=dtype) * sv
    Ys = Xs if Y is None else np.asarray(Y, dtype=dtype) * sv
    p, _, _ = phi_all(kind, sqdist(Xs, Ys, dtype), dtype)
    return dtype(scale) * p


def grad_kernelmatrix(kind, inv_ls, scale, X, Y=None, out_x=None, out_y=None, dtype=np.float64):
    """Multi-output matrix of gradKernel (src/surrogates/GradientGP.jl:573-606), out-major on
    both sides.  out_x / out_y: list of output indices (0 = value, a = d/dx_a) to include
    (default: all d+1).  Closed forms of the ForwardDiff derivatives (SURVEY §8a row a6):
        k          = sig2 * phi(u)
        dk/dx_a    =  2 s^2 sig2 phi'(u) D_a            D = x - y
        dk/dy_b    = -2 s^2 sig2 phi'(u) D_b
        d2k/dx_a dy_b = -sig2 [ 4 s^4 phi''(u) D_a D_b + 2 s^2 phi'(u) delta_ab ]
    """
    X = np.asarray(X, dtype=dtype)
    Y = X if Y is None else np.asarray(Y, dtype=dtype)
    n, d = X.shape
    m = Y.shape[0]
    out_x = list(range(d + 1)) if out_x is None else list(out_x)
    out_y = list(range(d + 1)) if out_y is None else list(out_y)
    sv = np.broadcast_to(np.asarray(inv_ls, dtype=dtype), (d,))      # s_k = 1/l_k (all equal for an isotropic kernel)
    scale = dtype(scale)
    Xs, Ys = X * sv, Y * sv
    u = sqdist(Xs, Ys, dtype)
    p, dp, ddp = phi_all(kind, u, dtype)
    K = np.empty((len(out_x) * n, len(out_y) * m), dtype=dtype)
    for ia, a in enumerate(out_x):
        Da = None if a == 0 else (Xs[:, a - 1][:, None] - Ys[:, a - 1][None, :])  # s * D_a
        for ib, b in enumerate(out_y):
            Db = None if b == 0 else (Xs[:, b - 1][:, None] - Ys[:, b - 1][None, :])
            if a == 0 and b == 0:
                blk = scale * p
            elif a > 0 and b == 0:
                blk = 2 * sv[a - 1] * scale * dp * Da
            elif a == 0 and b > 0:
                blk = -2 * sv[b - 1] * scale * dp * Db
            else:
                blk = -scale * (4 * sv[a - 1] * sv[b - 1] * ddp * Da * Db + (2 * sv[a - 1] ** 2 * dp if a == b else 0.0))
            K[ia * n:(ia + 1) * n, ib * m:(ib + 1) * m] = blk
    return K


# --------------------------------------------------------------------------------------
# surrogate state (what AbstractGPs' PosteriorGP holds: alpha, C = chol, x, delta)
# --------------------------------------------------------------------------------------
@dataclass
class Posterior:
    kind: int
    inv_ls: float
    scale: float
    noise: float
    mean_c: np.ndarray          # prior mean constant per output (length p)
    p: int                      # 1 (StandardGP) or d + 1 (GradientGP)
    X: np.ndarray               # (n, d)
    U: np.ndarray               # upper Cholesky factor of K + noise I  (N x N)
    alpha: np.ndarray           # (N,)
    delta: np.ndarray           # (N,)  y - m
    extras: dict = field(default_factory=dict)

    @property
    def n(self):
        return self.X.shape[0]


class PosDefException(Exception):
    """Mirrors LinearAlgebra.PosDefException(info) thrown by cholesky() inside
    AbstractGPs.posterior (src/bayesian_opt.jl:126-141 catches it)."""

    def __init__(self, info):
        super().__init__(f"matrix is not positive definite; Cholesky failed at pivot {info}")
        self.info = info


def _chol_upper(C):
    try:
        return sla.cholesky(C, lower=False, check_finite=False)
    except sla.LinAlgError as e:  # recover LAPACK info like Julia does
        _, info = sla.lapack.dpotrf(C, lower=0)
        raise PosDefException(int(info)) from e


def fit_standard(X, y, kind, inv_ls, scale, noise, mean_c=0.0) -> Posterior:
    """update(::StandardGP, xs, ys)  (src/surrogates/StandardGP.jl:79-83) →
    AbstractGPs.posterior(FiniteGP(GP(mean, kernel), xs, noise), ys):
    C = K + noise I; chol = cholesky(Symmetric(C)) (upper); delta = y - m; alpha = chol \\ delta."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    y = np.asarray(y, dtype=np.float64).ravel()
    if X.shape[0] != y.shape[0]:
        raise ValueError("DimensionMismatch: xs and ys lengths differ")
    C = kernelmatrix(kind, inv_ls, scale, X)
    C[np.diag_indices_from(C)] += noise
    U = _chol_upper(C)
    delta = y - mean_c
    alpha = sla.cho_solve((U, False), delta, check_finite=False)
    return Posterior(kind, inv_ls, scale, noise, np.array([mean_c], dtype=np.float64), 1, X, U, alpha, delta)


def prep_output(ys) -> np.ndarray:
    """vec(permutedims(hcat(ys...))) — out-major flattening (GradientGP.jl:919-922).
    ys: (n, p) rows [f, df/dx_1 ... df/dx_d]."""
    return np.asarray(ys, dtype=np.float64).T.reshape(-1)


def fit_gradient(X, Y, kind, inv_ls, scale, noise, mean_c=None) -> Posterior:
    """update(::GradientGP, xs, ys) (src/surrogates/GradientGP.jl:659-668): N = n(d+1) system,
    same noise on value and gradient rows (:664)."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    n, d = X.shape
    p = d + 1
    Y = np.asarray(Y, dtype=np.float64)
    if Y.shape != (n, p):
        raise ValueError("DimensionMismatch: ys must be n x (d+1)")
    mean_c = np.zeros(p) if mean_c is None else np.asarray(mean_c, dtype=np.float64)
    C = grad_kernelmatrix(kind, inv_ls, scale, X)
    C[np.diag_indices_from(C)] += noise
    U = _chol_upper(C)
    delta = prep_output(Y) - np.repeat(mean_c, n)
    alpha = sla.cho_solve((U, False), delta, check_finite=False)
    return Posterior(kind, inv_ls, scale, noise, mean_c, p, X, U, alpha, delta)


def _kstar(post: Posterior, Xc, outputs):
    """cov(prior, data.x, x*): rows = training outputs (all p, out-major), columns = candidate
    outputs `outputs` (out-major)."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    if post.p == 1:
        return kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, Xc)
    return grad_kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, Xc, out_y=outputs)


def _prior_var(post: Posterior, m, outputs):
    """kernelmatrix_diag of the prior at x* for each requested output: value rows sig2*phi(0);
    gradient rows -2 s^2 sig2 phi'(0) (the a == b, D = 0 case of grad_kernelmatrix)."""
    p0, dp0, _ = phi_all(post.kind, np.zeros(1))
    v = []
    sv = np.broadcast_to(np.asarray(post.inv_ls, dtype=np.float64), (post.X.shape[1],))
    for o in outputs:
        v.append(np.full(m, post.scale * p0[0] if o == 0 else -2 * sv[o - 1] ** 2 * post.scale * dp0[0]))
    return np.concatenate(v)


def posterior_mean_var(post: Posterior, Xc, outputs=(0,), chunk=8192):
    """posterior_mean / posterior_var (StandardGP.jl:361-379, GradientGP.jl:936-1003):
      mean = m(x*) + K*^T alpha
      var  = k** - sum(abs2, U' \\ K*, dims=1) + 1e-18      (AbstractGPs diag_Xt_invA_X)
    Returned out-major over `outputs` when more than one output is requested."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    m = Xc.shape[0]
    outputs = list(outputs)
    mean = np.empty(len(outputs) * m)
    var = np.empty(len(outputs) * m)
    for c0 in range(0, m, chunk):
        c1 = min(m, c0 + chunk)
        mc = c1 - c0
        Ks = _kstar(post, Xc[c0:c1], outputs)                      # N x (nout*mc)
        mu = Ks.T @ post.alpha
        V = sla.solve_triangular(post.U, Ks, trans="T", lower=False, check_finite=False)
        q = np.sum(V * V, axis=0)
        kss = _prior_var(post, mc, outputs)
        for io, o in enumerate(outputs):
            mean[io * m + c0: io * m + c1] = post.mean_c[o] + mu[io * mc:(io + 1) * mc]
            var[io * m + c0: io * m + c1] = (kss[io * mc:(io + 1) * mc] - q[io * mc:(io + 1) * mc]) + JITTER
    return mean, var


def posterior_cov(post: Posterior, Xc, outputs=None):
    """posterior_grad_cov (GradientGP.jl:968-971): cov(prior,x*) - K*^T C^-1 K* + 1e-18 I."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    outputs = list(range(post.p)) if outputs is None else list(outputs)
    Ks = _kstar(post, Xc, outputs)
    if post.p == 1:
        Kss = kernelmatrix(post.kind, post.inv_ls, post.scale, Xc)
    else:
        Kss = grad_kernelmatrix(post.kind, post.inv_ls, post.scale, Xc, out_x=outputs, out_y=outputs)
    V = sla.solve_triangular(post.U, Ks, trans="T", lower=False, check_finite=False)
    return Kss - V.T @ V + JITTER * np.eye(Kss.shape[0])


# --------------------------------------------------------------------------------------
# negative log marginal likelihood  (+ analytic gradient)
# --------------------------------------------------------------------------------------
def nlml(X, y_flat, kind, log_ls, log_scale, noise, mean_c=None, gradient_gp=False, want_grad=False):
    """nlml(model, (log l, log sig2), xs, ys)  (StandardGP.jl:99-114, GradientGP.jl:684-698):
    -logpdf(FiniteGP) = 1/2 [ N log 2pi + logdet C + || U^-T (y - m) ||^2 ].
    The reference differentiates this with ForwardDiff (bayesian_opt.jl:284); the analytic
    gradient returned here is the same quantity:
        d/dtheta = 1/2 tr(C^-1 dC) - 1/2 alpha^T dC alpha,
        dC/dlog(sig2) = K,   dC/dlog(l) = -2 sig2 phi'(u) u  (value block; derivative blocks
        by the product rule on the closed forms).
    Raises PosDefException like the reference's cholesky."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    n, d = X.shape
    ell = math.exp(log_ls)
    s = 1.0 / ell
    sc = math.exp(log_scale)
    y_flat = np.asarray(y_flat, dtype=np.float64).ravel()
    if gradient_gp:
        p = d + 1
        mean_c = np.zeros(p) if mean_c is None else np.asarray(mean_c, dtype=np.float64)
        K = grad_kernelmatrix(kind, s, sc, X)
        mvec = np.repeat(mean_c, n)
    else:
        K = kernelmatrix(kind, s, sc, X)
        mvec = 0.0 if mean_c is None else float(np.ravel(mean_c)[0])
    N = K.shape[0]
    C = K.copy()
    C[np.diag_indices_from(C)] += noise
    U = _chol_upper(C)
    delta = y_flat - mvec
    w = sla.solve_triangular(U, delta, trans="T", lower=False, check_finite=False)
    val = 0.5 * (N * math.log(2 * math.pi) + 2.0 * np.sum(np.log(np.diag(U))) + float(w @ w))
    if not want_grad:
        return val
    alpha = sla.solve_triangular(U, w, lower=False, check_finite=False)
    Cinv = sla.cho_solve((U, False), np.eye(N), check_finite=False)
    dK_ls = dK_dlogls(kind, s, sc, X, gradient_gp)
    M = Cinv - np.outer(alpha, alpha)
    g_ls = 0.5 * np.sum(M * dK_ls)
    g_sc = 0.5 * np.sum(M * K)
    return val, np.array([g_ls, g_sc])


def nlml_ard(X, y, kind, log_ls, log_scale, noise, mean_c=0.0, want_grad=False):
    """NLML of a StandardGP with one length scale per dimension (ARDTransform; the extension of the nlml parameter vector
    planned at src/bayesian_opt.jl:193-194) and its analytic gradient with respect to (log l_1 .. log l_d, log sig2):
    dK/dlog l_k = -2 sig2 phi'(u) D_k^2 with D_k = (x_k - y_k) / l_k,  dK/dlog sig2 = K."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    n, d = X.shape
    sv = np.exp(-np.asarray(log_ls, dtype=np.float64)); sc = math.exp(log_scale)
    K = kernelmatrix(kind, sv, sc, X)
    C = K.copy(); C[np.diag_indices_from(C)] += noise
    U = _chol_upper(C)
    delta = np.asarray(y, dtype=np.float64).ravel() - mean_c
    w = sla.solve_triangular(U, delta, trans="T", lower=False, check_finite=False)
    val = 0.5 * (n * math.log(2 * math.pi) + 2.0 * np.sum(np.log(np.diag(U))) + float(w @ w))
    if not want_grad:
        return val
    alpha = sla.solve_triangular(U, w, lower=False, check_finite=False)
    M = sla.cho_solve((U, False), np.eye(n), check_finite=False) - np.outer(alpha, alpha)
    Xs = X * sv
    _, dp, _ = phi_all(kind, sqdist(Xs, Xs))
    g = [0.5 * np.sum(M * (-2.0 * sc * dp * (Xs[:, k][:, None] - Xs[:, k][None, :]) ** 2)) for k in range(d)]
    return val, np.array(g + [0.5 * np.sum(M * K)])


def dK_dlogls(kind, s, sc, X, gradient_gp=False, eps=None):
    """dK/dlog(l).  Value block: K = sc*phi(u), u = s^2 r^2, du/dlog l = -2u  =>  -2 sc phi' u.
    Derivative blocks (needs phi'''): obtained by a 5-point Richardson-free complex-step-like
    central difference in log l on the closed forms — the oracle only needs ~1e-10 here and
    the GPU path is checked against it with that tolerance."""
    Xs = X * s
    if not gradient_gp:
        u = sqdist(Xs, Xs)
        _, dp, _ = phi_all(kind, u)
        return -2.0 * sc * dp * u
    h = 1e-3 if eps is None else eps
    # 4th-order central difference in theta = log l  (s = exp(-theta))
    def Kat(t):
        return grad_kernelmatrix(kind, s * math.exp(-t), sc, X)
    return (-Kat(2 * h) + 8 * Kat(h) - 8 * Kat(-h) + Kat(-2 * h)) / (12 * h)


# --------------------------------------------------------------------------------------
# acquisition functions
# --------------------------------------------------------------------------------------
def normcdf(z):
    """Distributions.cdf(Normal(0,1), z) = StatsFuns.normcdf(z) = erfc(-z/sqrt2)/2."""
    return erfc(-np.asarray(z) / math.sqrt(2.0)) / 2


def normpdf(z):
    """Distributions.pdf(Normal(0,1), z) = exp(-z^2/2) / sqrt(2 pi)."""
    z = np.asarray(z)
    return np.exp(-(z * z) / 2) / math.sqrt(2 * math.pi)


def expected_improvement(mu, var, xi, best_y):
    """src/acquisition_functions/ExpectedImprovement.jl:40-66, same operation order."""
    delta = (best_y - xi) - np.asarray(mu)
    var = np.asarray(var)
    small = var <= 1e-12
    sig = np.sqrt(np.where(small, 1.0, var))
    z = delta / sig
    val = delta * normcdf(z) + sig * normpdf(z)
    return np.where(small, np.maximum(delta, 0.0), val)


def probability_improvement(mu, var, xi, best_y):
    """src/acquisition_functions/ProbabilityImprovement.jl:38-63 (incl. the max(delta,0) quirk)."""
    delta = (best_y - xi) - np.asarray(mu)
    var = np.asarray(var)
    small = var <= 1e-12
    sig = np.sqrt(np.where(small, 1.0, var))
    return np.where(small, np.maximum(delta, 0.0), normcdf(delta / sig))


def upper_confidence_bound(mu, var, beta):
    """src/acquisition_functions/UpperConfidenceBound.jl:38-45."""
    return -np.asarray(mu) + beta * np.sqrt(np.maximum(np.asarray(var), 0.0))


def grad_norm_ucb(post: Posterior, Xc, beta):
    """src/acquisition_functions/gradNormUCB.jl:43-51, point by point."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    out = np.empty(len(Xc))
    for c, x in enumerate(Xc):
        mean, _ = posterior_mean_var(post, x[None, :], outputs=range(post.p))
        S = posterior_cov(post, x[None, :])[1:, 1:]
        m = mean[1:]
        mu_sq = m @ m + np.trace(S)
        var_sq = 4 * m @ (S @ m) + 2 * np.sum(S ** 2)
        out[c] = -mu_sq + beta * math.sqrt(max(var_sq, 1e-12))
    return out


def acquisition(acq_id, params, mu, var):
    if acq_id == EI:
        return expected_improvement(mu, var, params[0], params[1])
    if acq_id == PI:
        return probability_improvement(mu, var, params[0], params[1])
    if acq_id == UCB:
        return upper_confidence_bound(mu, var, params[0])
    raise ValueError("unknown acquisition id")


def sortperm_rev(scores, k=None):
    """sortperm(scores; rev=true)[1:k]  (src/acquisition_functions/acq_utils.jl:51-52):
    stable, descending by isless (NaN sorts as the largest, so NaNs come first), ties keep
    ascending index order.  Returns 0-based indices."""
    s = np.asarray(scores, dtype=np.float64)
    key = np.where(np.isnan(s), np.inf, s)
    nanfirst = np.isnan(s)
    # lexsort: last key is primary.  primary: NaN first, then value descending, then index.
    order = np.lexsort((np.arange(s.size), -key, ~nanfirst))
    return order if k is None else order[:min(k, s.size)]


# --------------------------------------------------------------------------------------
# O(n^2) row append (absent in the reference, which re-fits: bayesian_opt.jl:125); the oracle
# for it is simply a full re-fit on the extended data.
# --------------------------------------------------------------------------------------
def refit_after_append(post: Posterior, x_new, y_new):
    X = np.vstack([post.X, np.atleast_2d(x_new)])
    if post.p == 1:
        y = np.concatenate([post.delta + post.mean_c[0], np.ravel(y_new)])
        return fit_standard(X, y, post.kind, post.inv_ls, post.scale, post.noise, post.mean_c[0])
    n = post.n
    Yold = (post.delta + np.repeat(post.mean_c, n)).reshape(post.p, n).T
    Y = np.vstack([Yold, np.atleast_2d(y_new)])
    return fit_gradient(X, Y, post.kind, post.inv_ls, post.scale, post.noise, post.mean_c)


# --------------------------------------------------------------------------------------
# high-precision arbiter (small n)
# --------------------------------------------------------------------------------------
def mp_posterior_standard(X, y, kind, inv_ls, scale, noise, mean_c, Xc, dps=50):
    """50-digit evaluation of mean/var for StandardGP (SE / Matern) used to arbitrate when two
    FP64 evaluations legitimately differ (SURVEY H3)."""
    import mpmath as mp
    mp.mp.dps = dps
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    n, d = X.shape

    def kfun(a, b):
        u = mp.mpf(0)
        for k in range(d):
            t = mp.mpf(float(a[k])) * mp.mpf(inv_ls) - mp.mpf(float(b[k])) * mp.mpf(inv_ls)
            u += t * t
        if kind == SE:
            return mp.mpf(scale) * mp.e ** (-u / 2)
        r = mp.sqrt(u)
        if kind in (MATERN52, APPROX_MATERN52, AD_MATERN52):
            return mp.mpf(scale) * (1 + mp.sqrt(5) * r + 5 * u / 3) * mp.e ** (-mp.sqrt(5) * r)
        return mp.mpf(scale) * (1 + mp.sqrt(7) * r + 14 * u / 5 + 7 * mp.sqrt(7) * r ** 3 / 15) * mp.e ** (-mp.sqrt(7) * r)

    K = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            K[i, j] = kfun(X[i], X[j]) + (mp.mpf(noise) if i == j else 0)
    dl = mp.matrix([mp.mpf(float(v)) - mp.mpf(mean_c) for v in y])
    alpha = mp.lu_solve(K, dl)
    means, vars_ = [], []
    for c in range(Xc.shape[0]):
        ks = mp.matrix([kfun(X[i], Xc[c]) for i in range(n)])
        sol = mp.lu_solve(K, ks)
        means.append(mp.mpf(mean_c) + sum(ks[i] * alpha[i] for i in range(n)))
        vars_.append(mp.mpf(scale) - sum(ks[i] * sol[i] for i in range(n)) + mp.mpf(JITTER))
    return means, vars_


def ld_posterior_truth(post: Posterior, Xc, iters=5, outputs=(0,)):
    """80-bit arbiter at FULL problem size (SURVEY H3, §8c "arbiter"): posterior mean / variance of the outputs
    `outputs` (0 = value, a = d/dx_a; out-major like posterior_mean_var) at a handful of query points, accurate to
    ~1e-18 relative to the problem scale.
    The kernel matrix is evaluated in long double from the same FP64 inputs; K z = b is solved by iterative
    refinement: FP64 LAPACK Cholesky as the preconditioner, residuals b - K z accumulated in long double
    (converges geometrically while cond(K) * 2^-53 < 1).  Returns (mean, var) as long double arrays."""
    LD = np.longdouble
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    mc = Xc.shape[0]
    outputs = list(outputs)
    if post.p == 1:
        assert outputs == [0]
        K = kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, dtype=LD)
        Ks = kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, Xc, dtype=LD)
    else:
        K = grad_kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, dtype=LD)
        Ks = grad_kernelmatrix(post.kind, post.inv_ls, post.scale, post.X, Xc, out_y=outputs, dtype=LD)
    K[np.diag_indices_from(K)] += LD(post.noise)
    B = np.concatenate([post.delta.astype(LD)[:, None], Ks], axis=1)          # delta is exact in FP64 (y - m)
    Z = np.zeros_like(B)
    scale_b = np.maximum(np.max(np.abs(B), axis=0), LD(1e-300))
    for it in range(iters):
        R = B - K @ Z
        Z = Z + sla.cho_solve((post.U, False), R.astype(np.float64), check_finite=False).astype(LD)
        if np.all(np.max(np.abs(R), axis=0) <= LD(1e-19) * scale_b) and it >= 1:
            break
    resid = np.max(np.abs(B - K @ Z), axis=0) / scale_b
    alpha = Z[:, 0]
    mean = np.repeat(np.asarray([post.mean_c[o] for o in outputs], dtype=LD), mc) + Ks.T @ alpha
    q = np.einsum("ij,ij->j", Ks, Z[:, 1:])
    var = (_prior_var(post, mc, outputs).astype(LD) - q) + LD(JITTER)
    assert mean.shape == (mc * len(outputs),)
    return mean, var, float(np.max(resid))


def cond_estimate(U, iters=40, seed=0):
    """2-norm condition number of K = U^T U from power iteration (largest eigenvalue) and inverse power
    iteration (smallest) with triangular products / solves only: O(iters N^2) — np.linalg.cond of an
    8192 x 8192 factor would be an SVD."""
    rng = np.random.default_rng(seed)
    N = U.shape[0]
    v = rng.standard_normal(N); v /= np.linalg.norm(v)
    w = v.copy()
    lmax = lmin_inv = 1.0
    for _ in range(iters):
        t = U.T @ (U @ v); lmax = np.linalg.norm(t); v = t / lmax
        # two triangular solves, not cho_solve: LAPACK potrs with one right-hand side is ~15x slower at N = 8400
        t = sla.solve_triangular(U, sla.solve_triangular(U, w, trans="T", check_finite=False), check_finite=False)
        lmin_inv = np.linalg.norm(t); w = t / lmin_inv
    return float(lmax * lmin_inv)


def ld_nlml(X, y_flat, kind, log_ls, log_scale, noise, mean_c=0.0):
    """80-bit NLML of a StandardGP (arbiter for nlml(model, theta, xs, ys), StandardGP.jl:99-114): kernel matrix,
    column-by-column Cholesky and forward substitution all in long double."""
    LD = np.longdouble
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    N = X.shape[0]
    s = np.exp(-LD(log_ls)); sc = np.exp(LD(log_scale))
    A = kernelmatrix(kind, s, sc, X, dtype=LD)
    A[np.diag_indices_from(A)] += LD(noise)
    L = np.zeros_like(A)
    for j in range(N):
        v = A[j:, j] - L[j:, :j] @ L[j, :j]
        if not v[0] > 0:
            raise PosDefException(j + 1)
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    delta = np.asarray(y_flat, dtype=np.float64).astype(LD) - LD(mean_c)
    w = np.zeros(N, dtype=LD)
    for j in range(N):
        w[j] = (delta[j] - L[j, :j] @ w[:j]) / L[j, j]
    two_pi = LD(2) * np.arctan(LD(1)) * LD(4)
    return (LD(N) * np.log(two_pi) + LD(2) * np.sum(np.log(np.diag(L))) + w @ w) / LD(2)


def mp_acquisition(acq_id, params, mean_ld, var_ld, dps=40):
    """Acquisition values from long-double mean / variance in 40-digit arithmetic (erfc has no long-double
    implementation in SciPy), same formulas and branches as ExpectedImprovement.jl:59-66,
    ProbabilityImprovement.jl:57-63, UpperConfidenceBound.jl:38-45.  Returns long double."""
    import mpmath as mp
    mp.mp.dps = dps

    def to_mp(x):
        hi = float(x)
        return mp.mpf(hi) + mp.mpf(float(x - np.longdouble(hi)))
    out = []
    for mu_, var_ in zip(mean_ld, var_ld):
        mu, var = to_mp(mu_), to_mp(var_)
        if acq_id == UCB:
            v = -mu + mp.mpf(params[0]) * mp.sqrt(max(var, mp.mpf(0)))
        else:
            delta = (mp.mpf(params[1]) - mp.mpf(params[0])) - mu
            if var <= mp.mpf("1e-12"):
                v = max(delta, mp.mpf(0))
            else:
                sig = mp.sqrt(var)
                z = delta / sig
                cdf = mp.erfc(-z / mp.sqrt(2)) / 2
                v = delta * cdf + sig * mp.exp(-z * z / 2) / mp.sqrt(2 * mp.pi) if acq_id == EI else cdf
        hi = float(v)
        out.append(np.longdouble(hi) + np.longdouble(float(v - mp.mpf(hi))))
    return np.array(out, dtype=np.longdouble)


# --------------------------------------------------------------------------------------
# deterministic synthetic workloads for the BASELINE.json configs (SURVEY §8d)
# --------------------------------------------------------------------------------------
def branin(X):
    x1, x2 = X[:, 0], X[:, 1]
    return (x2 - 5.1 * x1 ** 2 / (4 * math.pi ** 2) + 5 * x1 / math.pi - 6) ** 2 \
        + 10 * (1 - 1 / (8 * math.pi)) * np.cos(x1) + 10


_H6_A = np.array([[10, 3, 17, 3.5, 1.7, 8], [0.05, 10, 17, 0.1, 8, 14],
                  [3, 3.5, 1.7, 10, 17, 8], [17, 8, 0.05, 10, 0.1, 14]], dtype=np.float64)
_H6_P = 1e-4 * np.array([[1312, 1696, 5569, 124, 8283, 5886], [2329, 4135, 8307, 3736, 1004, 9991],
                         [2348, 1451, 3522, 2883, 3047, 6650], [4047, 8828, 8732, 5743, 1091, 381]],
                        dtype=np.float64)
_H6_ALPHA = np.array([1.0, 1.2, 3.0, 3.2])


def hartmann6(X):
    inner = np.einsum("ij,nij->ni", _H6_A, (X[:, None, :] - _H6_P[None, :, :]) ** 2)
    return -np.sum(_H6_ALPHA[None, :] * np.exp(-inner), axis=1)


def rosenbrock_with_grad(X):
    x = X
    f = np.sum(100 * (x[:, 1:] - x[:, :-1] ** 2) ** 2 + (1 - x[:, :-1]) ** 2, axis=1)
    g = np.zeros_like(x)
    g[:, :-1] += -400 * x[:, :-1] * (x[:, 1:] - x[:, :-1] ** 2) - 2 * (1 - x[:, :-1])
    g[:, 1:] += 200 * (x[:, 1:] - x[:, :-1] ** 2)
    return np.column_stack([f, g])


def standardize(y):
    """standardize_problem(..., "mean_scale") (src/BO_utils.jl:44-64; get_mean_std
    StandardGP.jl:164-176 uses Statistics.std = corrected sample std)."""
    mu = float(np.mean(y))
    sd = float(np.std(y, ddof=1))
    return (y - mu) / sd, mu, sd


def make_config(name: str, seed: int = 42, n=None, m=None, d=None):
    """Seeded synthetic data for configs C1..C5 (SURVEY §8d).  Returns a dict with X, y (or Y),
    candidates Xc and the hyper-parameters; sizes can be scaled down with n / m / d."""
    rng = np.random.default_rng(seed)
    rc = np.random.default_rng(seed + 1)
    if name == "C1":   # StandardGP SE + EI, 2-D Branin
        n = 10 if n is None else n
        m = 10_000 if m is None else m
        lo, hi = np.array([-5.0, 0.0]), np.array([10.0, 15.0])
        X = lo + (hi - lo) * rng.random((n, 2))
        y, mu, sd = standardize(branin(X))
        Xc = lo + (hi - lo) * rc.random((m, 2))
        return dict(X=X, y=y, Xc=Xc, kind=SE, inv_ls=1.0 / 3.0, scale=1.0, noise=1e-6, mean_c=0.0,
                    acq=EI, acq_params=(0.01, float(y.min())), lower=lo, upper=hi)
    if name == "C2":   # Matern-5/2, 6-D Hartmann, n = 2048, EI over 1M
        n = 2048 if n is None else n
        m = 1 << 20 if m is None else m
        X = rng.random((n, 6))
        y, mu, sd = standardize(hartmann6(X))
        Xc = rc.random((m, 6))
        return dict(X=X, y=y, Xc=Xc, kind=MATERN52, inv_ls=1.0 / 0.5, scale=1.0, noise=1e-4, mean_c=0.0,
                    acq=EI, acq_params=(0.01, float(y.min())), lower=np.zeros(6), upper=np.ones(6))
    if name == "C3":   # GradientGP 10-D Rosenbrock, n = 512 -> N = 5632
        n = 512 if n is None else n
        m = 65_536 if m is None else m
        d = 10 if d is None else d
        X = -2 + 4 * rng.random((n, d))
        Y = rosenbrock_with_grad(X)
        mu = float(np.mean(Y[:, 0])); sd = float(np.std(Y[:, 0], ddof=1))
        Y = Y.copy(); Y[:, 0] -= mu; Y /= sd            # std_y(::GradientGP) GradientGP.jl:780-783
        Xc = -2 + 4 * rc.random((m, d))
        return dict(X=X, Y=Y, Xc=Xc, kind=APPROX_MATERN52, inv_ls=1.0 / 1.5, scale=1.0, noise=1e-6,
                    mean_c=np.zeros(d + 1), acq=EI, acq_params=(0.01, float(Y[:, 0].min())),
                    lower=-2 * np.ones(d), upper=2 * np.ones(d))
    if name == "C4":   # UCB, n = 8192, d = 20
        n = 8192 if n is None else n
        m = 1 << 21 if m is None else m
        d = 20 if d is None else d
        X = rng.random((n, d))
        y = np.sum(np.sin(3 * X), axis=1) / d + 0.1 * rng.standard_normal(n)
        y, mu, sd = standardize(y)
        Xc = rc.random((m, d))
        return dict(X=X, y=y, Xc=Xc, kind=SE, inv_ls=1.0, scale=1.0, noise=1e-2, mean_c=0.0,
                    acq=UCB, acq_params=(2.0,), lower=np.zeros(d), upper=np.ones(d))
    if name == "C5":   # NLML multi-start, n = 1024, d = 8, R = 256
        n = 1024 if n is None else n
        R = 256 if m is None else m
        d = 8 if d is None else d
        X = rng.random((n, d))
        y = np.sum(np.sin(3 * X), axis=1) / d + 0.03 * rng.standard_normal(n)
        y, mu, sd = standardize(y)
        lo = np.log(np.array([5e-2, 1e-3])); hi = np.log(np.array([1e1, 1e3]))
        theta = lo + (hi - lo) * rc.random((R, 2))
        return dict(X=X, y=y, theta=theta, kind=SE, noise=1e-3, mean_c=0.0)
    raise ValueError(name)
