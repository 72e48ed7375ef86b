"""Host-side callers of the hot path, mirroring src/bayesian_opt.jl and
src/acquisition_functions/acq_utils.jl: BOStruct, update(BO, x, y, i) with the
PosDef/Singular rollback protocol, the multi-start acquisition optimiser and the multi-start
hyper-parameter MLE.  These are thin: the arithmetic is in libabo_cuda.so."""
from __future__ import annotations

import logging
import math

import numpy as np
from scipy.optimize import minimize

from ._lib import PosDefException
from .kernels import with_lengthscale
from .surrogates import (GradientGP, _update_model_parameters, get_kernel_constructor, get_lengthscale,
                         get_mean_std, get_scale, nlml_batch, rescale_model, std_y, update_surrogate)

log = logging.getLogger("abo_b200")


def latin_hypercube(n, lower, upper, rng):
    """QuasiMonteCarlo.sample(n, lb, ub, LatinHypercubeSample()) (acq_utils.jl:44-46): one point
    per stratum and dimension, independently permuted."""
    d = len(lower)
    u = (np.argsort(rng.random((d, n)), axis=1).T + rng.random((n, d))) / n
    return lower + (upper - lower) * u


def monte_carlo_fill_distance(x_train, domain, n_samples=10_000, rng=None, ctx=None):
    """monte_carlo_fill_distance (BO_utils.jl:140-159): the n_samples x n nearest-neighbour scan runs
    on the device (abo_fill_distance); the uniform samples are drawn on the host."""
    from ._lib import default_context
    rng = np.random.default_rng() if rng is None else rng
    X = np.asarray(x_train, dtype=np.float64).reshape(len(x_train), -1)
    S = domain.lower + rng.random((n_samples, len(domain.lower))) * (domain.upper - domain.lower)
    return (ctx or default_context()).fill_distance(X, S)


def lengthscale_bounds(x_train, domain, min_frac=0.1, max_frac=1.0, n_samples=10_000, rng=None, ctx=None):
    """lengthscale_bounds (BO_utils.jl:87-128): upper = max_frac * box side; lower = min_frac * fill
    distance (Monte-Carlo for d > 1, exact largest gap incl. the domain edges for d = 1), floored at 1e-12."""
    d = len(domain.lower)
    X = np.asarray(x_train, dtype=np.float64).reshape(len(x_train), -1)
    if X.shape[1] != d:
        raise ValueError(f"All points in X_train must have dimension {d}")
    upper = max_frac * (domain.upper - domain.lower)
    if d > 1:
        h = monte_carlo_fill_distance(X, domain, n_samples=n_samples, rng=rng, ctx=ctx)
    else:
        h = float(np.max(np.diff(np.concatenate([[domain.lower[0]], np.sort(X[:, 0]), [domain.upper[0]]]))))
    return np.full(d, max(min_frac * h, 1e-12)), upper


def optimize_acquisition(acqf, surrogate, domain, n_grid=10_000, n_local=100, rng=None, refine=True):
    """optimize_acquisition (acq_utils.jl:33-73): LHS grid → ONE batched, fused sweep that also
    returns the stable top-n_local (replaces acqf(...) + sortperm, :50-52) → box-constrained L-BFGS
    refinement from those starts.  The reference refines the starts one after the other with
    finite-difference gradients of single-point evaluations (:55-63); here all starts advance in
    lock-step and every step is ONE batched call returning the acquisition and its gradient for all of
    them (refine=True): analytic for EI / PI / UCB (abo_acq_eval_grad), batched central differences —
    all starts x (2 d + 1) points in one device call — for GradientNormUCB and ensembles.  refine="scipy" keeps the reference's sequential,
    finite-difference scheme (SciPy L-BFGS-B); refine=False returns the best grid point, and so does an acquisition
    without a gradient (ThompsonSampling), whatever `refine` says."""
    rng = np.random.default_rng() if rng is None else rng
    grid = latin_hypercube(n_grid, domain.lower, domain.upper, rng)
    _, top_idx, top_val = acqf.topk(surrogate, grid, n_local, want_scores=False)
    starts = grid[top_idx]
    if refine is False or len(starts) == 0 or not getattr(acqf, "has_gradient", True):
        return np.array(starts[0])
    if refine == "scipy":
        best_acq, best_x = -math.inf, None
        bounds = list(zip(domain.lower, domain.upper))
        for x0 in starts:
            res = minimize(lambda x: -float(acqf(surrogate, x[None, :])[0]), x0, method="L-BFGS-B", bounds=bounds,
                           options=dict(gtol=1e-5, ftol=2.2e-9, maxls=20))
            if -float(res.fun) > best_acq:
                best_acq, best_x = -float(res.fun), np.array(res.x)
        return best_x

    def fg(X, idx):
        val, grad = acqf.value_and_grad(surrogate, X[idx])
        return -val, -grad

    X, f, _, failed = lockstep_lbfgsb(fg, starts, domain.lower, domain.upper, g_tol=1e-5, f_abstol=2.2e-9, max_iter=50)
    f = np.where(failed | ~np.isfinite(f), np.inf, f)
    return np.array(X[int(np.argmin(f))])                 # first best on ties, like the `>` update of :67-70


def lockstep_lbfgsb(fg, x0, lower, upper, g_tol=1e-6, f_abstol=2.2e-9, max_iter=100, history=6, max_ls=20):
    """Box-constrained L-BFGS for R independent problems advanced in LOCK-STEP: `fg(X, idx)` evaluates
    the objective and gradient for the rows `idx` of the R x p array X in ONE batched call (here:
    abo_nlml_batch).  Projected quasi-Newton direction per problem, Armijo back-tracking where every
    trial step evaluates all still-searching problems together.  Stopping rule as the reference's
    Optim options (projected-gradient inf-norm <= g_tol or |df| <= f_abstol, bayesian_opt.jl:262).
    Returns (X, f, converged, failed)."""
    X = np.clip(np.array(x0, dtype=np.float64), lower, upper)
    R, p = X.shape
    H = history
    f = np.full(R, np.inf); G = np.zeros((R, p))
    f[:], G[:] = fg(X, np.arange(R))
    failed = ~np.isfinite(f)                              # restart whose start already fails (bayesian_opt.jl:296-299)
    converged = np.zeros(R, dtype=bool)
    # curvature pairs of all problems, oldest first in slots 0 .. cnt-1; every step below is one
    # vectorised NumPy operation over the problems (no per-problem Python loop)
    S = np.zeros((R, H, p)); Y = np.zeros((R, H, p)); SY = np.ones((R, H)); cnt = np.zeros(R, dtype=np.int64)
    rows = np.arange(R)

    for it in range(max_iter):
        active = ~converged & ~failed
        if not active.any():
            break
        PG = G.copy()
        PG[((X <= lower) & (G > 0)) | ((X >= upper) & (G < 0))] = 0.0
        converged |= active & (np.max(np.abs(PG), axis=1) <= g_tol)
        active &= ~converged
        live = np.flatnonzero(active)
        if live.size == 0:
            break
        Q = PG.copy()
        AL = np.zeros((R, H))
        for h in range(H - 1, -1, -1):                     # newest to oldest
            v = h < cnt
            a_ = np.where(v, np.einsum("ij,ij->i", S[:, h], Q) / SY[:, h], 0.0)
            AL[:, h] = a_
            Q -= a_[:, None] * Y[:, h]
        last = np.maximum(cnt - 1, 0)
        yl = Y[rows, last]
        gamma = np.where(cnt > 0, SY[rows, last] / np.maximum(np.einsum("ij,ij->i", yl, yl), 1e-300),
                         1.0 / np.maximum(1.0, np.linalg.norm(PG, axis=1)))
        Q *= gamma[:, None]
        for h in range(H):                                 # oldest to newest
            v = h < cnt
            b_ = np.where(v, np.einsum("ij,ij->i", Y[:, h], Q) / SY[:, h], 0.0)
            Q += np.where(v, AL[:, h] - b_, 0.0)[:, None] * S[:, h]
        D = -Q
        D[PG == 0.0] = 0.0
        up = np.einsum("ij,ij->i", D, G) >= 0              # not a descent direction: steepest descent
        D[up] = -PG[up]
        D[~active] = 0.0
        t = np.ones(R)
        pending = live.copy()
        Xn = X.copy(); fn = f.copy(); Gn = G.copy()
        for _ in range(max_ls):
            Xt = np.clip(X[pending] + t[pending, None] * D[pending], lower, upper)
            Xfull = X.copy(); Xfull[pending] = Xt
            ft, gt = fg(Xfull, pending)
            dec = np.einsum("ij,ij->i", G[pending], Xt - X[pending])
            ok = np.isfinite(ft) & (ft <= f[pending] + 1e-4 * dec)
            acc = pending[ok]
            Xn[acc] = Xt[ok]; fn[acc] = ft[ok]; Gn[acc] = gt[ok]
            pending = pending[~ok]
            if pending.size == 0:
                break
            t[pending] *= 0.5
        converged[pending] = True                          # no further progress along a descent direction
        moved = active.copy(); moved[pending] = False
        Sn = Xn - X; Yn = Gn - G
        sy = np.einsum("ij,ij->i", Sn, Yn)
        keep = moved & (sy > 1e-12 * np.linalg.norm(Sn, axis=1) * np.linalg.norm(Yn, axis=1))
        full = keep & (cnt == H)                           # drop the oldest pair where the history is full
        if full.any():
            S[full, :-1] = S[full, 1:]; Y[full, :-1] = Y[full, 1:]; SY[full, :-1] = SY[full, 1:]
            cnt[full] -= 1
        kr = np.flatnonzero(keep)
        S[kr, cnt[kr]] = Sn[kr]; Y[kr, cnt[kr]] = Yn[kr]; SY[kr, cnt[kr]] = sy[kr]
        cnt[kr] += 1
        converged |= moved & (np.abs(f - fn) <= f_abstol)
        X, f, G = Xn, fn, Gn
    return X, f, converged, failed


def optimize_hyperparameters(model, x_train, y_train, old_params, scale_std=1.0, length_scale_only=False,
                             num_restarts=1, domain=None, rng=None, max_iter=100, ard=False):
    """optimize_hyperparameters (bayesian_opt.jl:196-328).  Same log-space box, clamped start and
    uniform random restarts; all restarts advance in LOCK-STEP so that every objective/gradient
    evaluation is ONE batched abo_nlml_batch call (value + analytic gradient for all restarts) instead
    of one ForwardDiff evaluation per restart and step.
    ard=True optimises one length scale per input dimension, params = (log l_1 .. log l_d, log sig2) — the extension
    of the nlml parameter vector the reference lists as a TODO (bayesian_opt.jl:193-194); `old_params` may be the
    isotropic pair (replicated) or the full vector."""
    rng = np.random.default_rng() if rng is None else rng
    ls_lo, ls_hi = 1e-3, 1e3
    if domain is not None:                               # data-informed bounds (bayesian_opt.jl:216-228)
        lL, lU = lengthscale_bounds(x_train, domain, rng=rng, ctx=model.ctx)
        ls_lo, ls_hi = max(float(np.min(lL)), 1e-6), float(np.max(lU))
        assert ls_lo < ls_hi
    sc_lo, sc_hi = 1e-3 / scale_std ** 2, 1e6 / scale_std ** 2
    nd = np.asarray(x_train, dtype=np.float64).reshape(len(x_train), -1).shape[1] if ard else 1
    lo = np.log([ls_lo] * nd + [sc_lo]); hi = np.log([ls_hi] * nd + [sc_hi])
    old = np.asarray(old_params, dtype=np.float64).reshape(-1)
    if ard and old.size == 2:
        old = np.concatenate([np.full(nd, old[0]), old[1:]])
    eps2 = 2 * np.finfo(float).eps
    start = np.clip(old, lo + eps2, hi - eps2)                                             # bayesian_opt.jl:248
    inits = np.array([start] + [lo + (hi - lo) * rng.random(nd + 1) for _ in range(num_restarts - 1)])
    lower, upper = lo.copy(), hi.copy()
    if length_scale_only:                                  # nlml_ls: log scale frozen at the start value
        inits[:, -1] = start[-1]; lower[-1] = upper[-1] = start[-1]

    def fg(X, idx):
        val, grad, info = nlml_batch(model, X[idx], x_train, y_train, ard=ard)
        val = np.where(info != 0, np.inf, val)
        grad = np.where(np.isfinite(grad), grad, 0.0)
        if length_scale_only:
            grad[:, -1] = 0.0
        return val, grad

    X, f, converged, failed = lockstep_lbfgsb(fg, inits, lower, upper, max_iter=max_iter)
    good = converged & ~failed & np.isfinite(f)
    if not good.any():
        log.info("All restarts failed to converge.")
        return model
    best = X[np.flatnonzero(good)[np.argmin(f[good])]]
    ell = np.exp(best[:nd]) if ard else math.exp(best[0])
    scale = get_scale(model)[0] if length_scale_only else math.exp(best[-1])
    k_opt = scale * with_lengthscale(get_kernel_constructor(model), ell)
    return _update_model_parameters(model, k_opt)


class BOStruct:
    """BOStruct(f, acq, model, domain, xs, ys, max_iter, noise) (bayesian_opt.jl:38-92)."""

    def __init__(self, func, acq, model, domain, x_train, y_train, max_iter, noise):
        self.func, self.acq, self.model, self.domain = func, acq.copy(), model.copy(), domain
        self.xs = [np.asarray(x, dtype=np.float64).reshape(-1) for x in x_train]
        self.ys = [np.asarray(y, dtype=np.float64) for y in y_train]
        self.ys_non_std = [np.array(y, dtype=np.float64) for y in y_train]
        self.max_iter, self.iter, self.noise, self.flag = max_iter, 0, noise, False

    def __repr__(self):
        return _make_info(self)


def _make_info(BO):
    """_make_info / print_info / Base.show(::BOStruct) (BO_utils.jl:5-24)."""
    return ("== BOStruct Information ==\n"
            f"Target function: {getattr(BO.func, '__name__', BO.func)}\n"
            f"Domain: {BO.domain.bounds}\n"
            f"Number of data points: {len(BO.xs)}\n"
            f"Acquisition function: {BO.acq}\n"
            f"Max iterations: {BO.max_iter}\n"
            f"Noise level: {BO.noise}\n"
            "=========================")


def print_info(BO):
    print(_make_info(BO))


def update_bo(BO: BOStruct, x, y, i):
    """update(BO, x, y, i) (bayesian_opt.jl:113-150): snapshot → push → update → on
    PosDefException roll back xs/ys/ys_non_std, restore the snapshot, set `flag`."""
    prev = BO.model.copy()
    BO.xs.append(np.asarray(x, dtype=np.float64).reshape(-1))
    BO.ys.append(np.asarray(y, dtype=np.float64))
    try:
        # the lists go down as they are: a new point of the wrong dimension must surface as DimensionMismatch
        # (test/test_bayesian_opt.jl:788-817), which — like any error but PosDef/Singular — propagates (:127-131)
        BO.model = update_surrogate(BO.model, BO.xs, BO.ys)
    except PosDefException:
        log.info("We reached ill-conditioning, returning NON-UPDATED GP. Killing BO loop.")
        BO.model = prev
        BO.xs.pop(); BO.ys.pop()
        if len(BO.ys_non_std) > len(BO.ys):
            BO.ys_non_std.pop()
        BO.flag = True
        return BO
    BO.acq = BO.acq.update(np.array(BO.ys), BO.model)
    BO.iter = i + 1
    return BO


def stop_criteria(BO):
    return BO.iter > BO.max_iter


def standardize_problem(BO, choice):
    """standardize_problem (BO_utils.jl:44-64).  The empirical mean / standard deviation, the standardised observations
    and the new incumbent come from ONE device call (abo_standardize); rescale_model stays a host-side parameter update."""
    if choice not in ("mean_scale", "scale_only", "mean_only"):
        raise ValueError("choice must be one of: 'mean_scale', 'scale_only', 'mean_only'")
    from ._lib import default_context
    is_grad = isinstance(BO.model, GradientGP)
    Y = np.asarray(BO.ys_non_std, dtype=np.float64)
    n = len(BO.ys_non_std)
    p = BO.model.p
    flat = Y.T.reshape(-1) if is_grad else Y.reshape(-1)              # out-major (prep_output)
    mu_v, sd_v, y_std, _best = (BO.model.ctx or default_context()).standardize(flat, n, p, choice)
    if is_grad:
        mu, sd = mu_v, sd_v
        BO.ys = list(y_std.reshape(p, n).T)
    else:
        mu, sd = float(mu_v[0]), float(sd_v[0])
        BO.ys = list(y_std)
    if choice in ("scale_only", "mean_scale"):
        BO.model = rescale_model(BO.model, sd)
    BO.model = update_surrogate(BO.model, np.array(BO.xs), np.array(BO.ys))
    BO.acq = BO.acq.update(np.array(BO.ys), BO.model)
    return BO, (mu, sd)


def rescale_output(ys, params):
    """rescale_output (BO_utils.jl:162-182): standardised observations back on the original scale; (None, None) is the
    identity."""
    mu, sd = params
    if mu is None or sd is None:
        return [y for y in ys]
    return [np.asarray(y, dtype=np.float64) * sd + mu if np.ndim(y) else float(y) * float(np.ravel(sd)[0]) + float(np.ravel(mu)[0])
            for y in ys]


def optimize(BO: BOStruct, standardize="mean_scale", hyper_params="all", num_restarts_HP=1, n_grid=10_000,
             n_local=100, rng=None, refine=True, ard=False):
    """optimize(BO; standardize, hyper_params, num_restarts_HP) (bayesian_opt.jl:364-449)."""
    if standardize not in ("mean_scale", "scale_only", "mean_only", None):
        raise ValueError("standardize must be one of mean_scale, scale_only, mean_only, None")
    if hyper_params not in ("all", "length_scale_only", None):
        raise ValueError("hyper_params must be one of all, length_scale_only, None")
    rng = np.random.default_rng() if rng is None else rng
    if standardize is not None:
        BO, (mu, sd) = standardize_problem(BO, standardize)
    else:
        is_grad = isinstance(BO.model, GradientGP)
        mu, sd = (np.zeros(BO.model.p), np.ones(BO.model.p)) if is_grad else (0.0, 1.0)
        BO.model = update_surrogate(BO.model, np.array(BO.xs), np.array(BO.ys))
        BO.acq = BO.acq.update(np.array(BO.ys), BO.model)
    acq_list = []
    i = 0
    while not stop_criteria(BO) and not BO.flag:
        if hyper_params is not None and i % 10 == 0:
            ls = get_lengthscale(BO.model)
            old = [math.log(v) for v in (ls if ard and len(ls) > 1 else ls[:1])] + [math.log(get_scale(BO.model)[0])]
            m2 = optimize_hyperparameters(BO.model, np.array(BO.xs), np.array(BO.ys), old,
                                          scale_std=float(np.ravel(sd)[0]),
                                          length_scale_only=(hyper_params == "length_scale_only"),
                                          num_restarts=num_restarts_HP, domain=BO.domain, rng=rng, ard=ard)
            BO.model = update_surrogate(m2, np.array(BO.xs), np.array(BO.ys))
        x_cand = optimize_acquisition(BO.acq, BO.model, BO.domain, n_grid=n_grid, n_local=n_local, rng=rng,
                                      refine=refine)
        acq_list.append(float(BO.acq(BO.model, x_cand[None, :])[0]))
        y = np.asarray(BO.func(x_cand), dtype=np.float64)
        s0 = float(np.ravel(sd)[0])
        y = y + math.sqrt(BO.noise) / s0 * rng.standard_normal(y.shape) if BO.noise > 0 else y
        BO.ys_non_std.append(y)
        y_std = (y - mu) / s0 if isinstance(BO.model, GradientGP) else (y - mu) / sd
        i += 1                                           # incremented BEFORE update(BO, ...) (bayesian_opt.jl:441-445):
        BO = update_bo(BO, x_cand, y_std, i)             # BO.iter = i + 1, so exactly max_iter passes run
    return BO, acq_list, (mu, sd)
