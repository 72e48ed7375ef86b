"""GPU surrogate subtypes behind the reference's AbstractSurrogate API (src/abstract.jl:33):
`StandardGP` (src/surrogates/StandardGP.jl) and `GradientGP` (src/surrogates/GradientGP.jl).
Same names, argument meaning and error behaviour; the arithmetic runs in libabo_cuda.so."""
from __future__ import annotations

import math

import numpy as np

from . import _lib
from ._lib import DimensionMismatch, GpHandle, PosDefException, default_context
from .kernels import Kernel, normalized, with_lengthscale


class AbstractSurrogate:
    pass


def _as_points(x, d=None):
    """Vector of points -> (m, d) array.  A vector of reals is a set of 1-D points
    (src/abstract.jl:67-69, StandardGP.jl:329-347)."""
    try:
        a = np.asarray(x, dtype=np.float64)
    except ValueError as e:                       # ragged input: points of different dimensions
        raise DimensionMismatch(f"points do not all have the same dimension ({e})") from None
    if a.ndim == 0:
        a = a.reshape(1, 1)
    elif a.ndim == 1:
        a = a.reshape(-1, 1)
    if d is not None and a.shape[1] != d:
        raise DimensionMismatch(f"points have dimension {a.shape[1]}, the surrogate was conditioned on dimension {d}")
    return np.ascontiguousarray(a)


class _GpBase(AbstractSurrogate):
    p_of_d = staticmethod(lambda d: 1)

    def __init__(self, kernel: Kernel, noise_var: float, mean_c, ctx=None, _handle=None, _data=None):
        self.kernel = normalized(kernel)
        self.noise_var = float(noise_var)
        self.mean_c = mean_c
        self.ctx = ctx
        self.gpx = _handle                 # posterior handle (None before update, like `gpx === nothing`)
        self._data = _data                 # (X, Yflat) host copies of the conditioning set



# -- accessors (StandardGP.jl:261-287, GradientGP.jl:842-870)
def get_lengthscale(model):
    s = model.kernel.inv_lengthscale
    return [1.0 / v for v in s] if isinstance(s, tuple) else [1.0 / s]


def is_ard(model): return isinstance(model.kernel.inv_lengthscale, tuple)


def get_scale(model): return [model.kernel.scale]
def get_kernel_constructor(model): return model.kernel.constructor()


class StandardGP(_GpBase):
    """StandardGP(kernel, noise_var; mean=nothing) (StandardGP.jl:41-64).  `mean` is None
    (ZeroMean) or a float (ConstMean(c))."""

    def __init__(self, kernel: Kernel, noise_var: float, mean=None, ctx=None, _handle=None, _data=None):
        super().__init__(kernel, noise_var, 0.0 if mean is None else float(mean), ctx, _handle, _data)

    @property
    def p(self): return 1

    def copy(self):
        """Base.copy(::StandardGP) (StandardGP.jl:26): shares the prior, deep-copies the posterior."""
        h = None if self.gpx is None else self.gpx.clone()
        return StandardGP(self.kernel, self.noise_var, self.mean_c, self.ctx, h, self._data)

    def _new(self, kernel, noise_var, mean):
        return StandardGP(kernel, noise_var, mean, self.ctx)


class GradientGP(_GpBase):
    """GradientGP(kernel, p, noise_var; mean=gradConstMean(zeros(p))) (GradientGP.jl:622-644)."""

    def __init__(self, kernel: Kernel, p: int, noise_var: float, mean=None, ctx=None, _handle=None, _data=None):
        mc = np.zeros(p) if mean is None else np.asarray(mean, dtype=np.float64)
        if mc.size != p:
            raise DimensionMismatch("mean must have p entries")
        super().__init__(kernel, noise_var, mc, ctx, _handle, _data)
        self._p = int(p)

    @property
    def p(self): return self._p

    def copy(self):
        h = None if self.gpx is None else self.gpx.clone()
        return GradientGP(self.kernel, self._p, self.noise_var, self.mean_c, self.ctx, h, self._data)

    def _new(self, kernel, noise_var, mean):
        return GradientGP(kernel, self._p, noise_var, mean, self.ctx)


def prep_input(model, xs):
    return xs


def prep_output(model, ys):
    """StandardGP.jl:305 (identity) / GradientGP.jl:919-922 (out-major flattening)."""
    if isinstance(model, GradientGP):
        return np.asarray(ys, dtype=np.float64).T.reshape(-1)
    return np.asarray(ys, dtype=np.float64).reshape(-1)


def _flat_y(model, ys, n):
    try:
        y = np.asarray(ys, dtype=np.float64)
    except ValueError as e:
        raise DimensionMismatch(f"observations do not all have the same length ({e})") from None
    if isinstance(model, GradientGP):
        if y.ndim == 1 and y.size == n * model.p:
            return np.ascontiguousarray(y)            # already prepped (out-major)
        if y.shape != (n, model.p):
            raise DimensionMismatch(f"ys must be {n} x {model.p}")
        return prep_output(model, y)
    y = y.reshape(-1)
    if y.size != n:
        raise DimensionMismatch("xs and ys have different lengths")
    return np.ascontiguousarray(y)


def update_surrogate(model, xs, ys, allow_append=True):
    """update(model, xs, ys) (StandardGP.jl:79-83, GradientGP.jl:659-668): returns a NEW model
    conditioned on (xs, ys); raises PosDefException when the Cholesky fails (the BO loop catches
    it, src/bayesian_opt.jl:126-141) and DimensionMismatch on inconsistent inputs.
    When (xs, ys) extends the data the model already holds by exactly one observation the
    O(n²) row append (abo_gp_append; p rows at once for a GradientGP) is used on a copy-on-write
    clone instead of the O(n³) re-fit."""
    X = _as_points(xs)
    n, d = X.shape
    if isinstance(model, GradientGP) and model.p != d + 1:
        raise DimensionMismatch("GradientGP: p must equal d + 1")
    y = _flat_y(model, ys, n)
    ctx = model.ctx or default_context()
    old = model.gpx
    pp = model.p
    if (allow_append and old is not None and model._data is not None and old.d == d
            and model._data[0].shape[0] == n - 1 and np.array_equal(model._data[0], X[:-1])
            and np.array_equal(model._data[1].reshape(pp, n - 1), y.reshape(pp, n)[:, :-1])):
        h = old.clone()                                  # O(1): copy-on-write handle
        try:
            h.append(X[-1], y.reshape(pp, n)[:, -1])     # out-major y: the new point's p outputs
        except Exception:
            h.close()
            raise
    else:
        h = GpHandle(ctx, model.kernel.kernel_id, d, model.p)
        try:
            h.set_params(model.kernel.inv_lengthscale, model.kernel.scale, model.noise_var,
                         np.atleast_1d(model.mean_c))
            h.fit(X, y)
        except Exception:
            h.close()
            raise
    new = model._new(model.kernel, model.noise_var, model.mean_c if isinstance(model, GradientGP) else
                     (None if model.mean_c == 0.0 else model.mean_c))
    new.mean_c = model.mean_c
    new.ctx = ctx
    new.gpx = h
    new._data = (X.copy(), y.copy())
    return new


def empty_posterior_like(model, d):
    """A copy of `model` holding an un-fitted device handle of the right (kernel, d, p): the receive
    side of `sync_posterior` on non-root ranks."""
    new = model.copy()
    new.ctx = model.ctx or default_context()
    new.gpx = GpHandle(new.ctx, model.kernel.kernel_id, int(d), model.p)
    new.gpx.set_params(model.kernel.inv_lengthscale, model.kernel.scale, model.noise_var, np.atleast_1d(model.mean_c))
    return new


def _need_posterior(model):
    if model.gpx is None:
        raise _lib.AboCudaError("surrogate has no posterior: call update(model, xs, ys) first")
    return model.gpx


def posterior_mean(model, x):
    """StandardGP.jl:361-363 / GradientGP.jl:985-987 (value output only)."""
    h = _need_posterior(model)
    return h.posterior(_as_points(x, h.d), 1, True, False)[0]


def posterior_var(model, x):
    """StandardGP.jl:377-379 / GradientGP.jl:1001-1003."""
    h = _need_posterior(model)
    return h.posterior(_as_points(x, h.d), 1, False, True)[1]


def posterior_grad_mean(model, x):
    """GradientGP.jl:936-939 — out-major (f(x1..xm), ∂1 f(x1..xm), ...)."""
    h = _need_posterior(model)
    return h.posterior(_as_points(x, h.d), model.p, True, False)[0]


def posterior_grad_var(model, x):
    h = _need_posterior(model)
    return h.posterior(_as_points(x, h.d), model.p, False, True)[1]


def posterior_grad_cov(model, x):
    """GradientGP.jl:968-971 — full covariance over (point, output) pairs, out-major."""
    h = _need_posterior(model)
    return h.posterior_cov(_as_points(x, h.d), model.p)


def posterior_cov(model, x):
    """cov(model.gpx(x)) for the value output."""
    h = _need_posterior(model)
    return h.posterior_cov(_as_points(x, h.d), 1)


def posterior_sample(model, x, num_samples, *, seed, jitter=1e-10):
    """Joint draws of the latent value f over the points x: an (S, m) array, row s = draw s (AbstractGPs
    rand(rng, posterior(fx)(x), S), transposed).  Draw s depends only on (seed, s): the first S' rows of S > S' draws are
    the S' draws.  jitter is relative to the kernel scale and raised tenfold, up to six times, until the covariance
    factors."""
    h = _need_posterior(model)
    return h.posterior_sample(_as_points(x, h.d), num_samples, seed, jitter)[0]


def thompson_batch(model, x, q, *, seed, jitter=1e-10):
    """q candidate indices (0-based) into x: the minimiser of each of q joint posterior draws, a Thompson-sampling batch
    drawn with replacement.  Only the q indices leave the device."""
    h = _need_posterior(model)
    return h.posterior_sample(_as_points(x, h.d), q, seed, jitter, want_samples=False)[1]


def unstandardized_mean_and_var(model, xs, params):
    """StandardGP.jl:395-404 / GradientGP.jl:1019-1030."""
    h = _need_posterior(model)
    X = _as_points(xs, h.d)
    if isinstance(model, GradientGP):
        mu, sig = np.asarray(params[0], dtype=np.float64), float(np.ravel(params[1])[0])
        m, v = h.posterior(X, model.p, True, True)
        m = m.reshape(model.p, -1).T
        v = v.reshape(model.p, -1).T
        return m * sig + mu[None, :], v * sig ** 2
    mu, sig = float(params[0]), float(params[1])
    m, v = h.posterior(X, 1, True, True)
    return m * sig + mu, v * sig ** 2


def nlml(model, params, xs, ys):
    """nlml(model, [log ℓ, log σ²], xs, ys) (StandardGP.jl:99-114, GradientGP.jl:684-698)."""
    return nlml_batch(model, np.asarray(params, dtype=np.float64)[None, :], xs, ys, want_grad=False)[0][0]


def nlml_ls(model, log_ls, log_scale, xs, ys):
    """StandardGP.jl:133-149 / GradientGP.jl:719-738."""
    return nlml(model, [log_ls, log_scale], xs, ys)


def nlml_batch(model, logparams, xs, ys, want_grad=True, ard=False):
    """Value and analytic gradient of the NLML for R hyper-parameter vectors in one call
    (replaces the ForwardDiff.Dual evaluation of bayesian_opt.jl:284).  ard=True: rows are
    {log l_1 .. log l_d, log sig2} (per-dimension length scales, the extension planned at bayesian_opt.jl:193-194)."""
    X = _as_points(xs)
    n, d = X.shape
    y = _flat_y(model, ys, n)
    ctx = model.ctx or default_context()
    h = GpHandle(ctx, model.kernel.kernel_id, d, model.p)
    try:
        isl = model.kernel.inv_lengthscale
        h.set_params(isl[0] if isinstance(isl, tuple) else isl, model.kernel.scale, model.noise_var, np.atleast_1d(model.mean_c))
        return h.nlml_batch(X, y, logparams, want_grad, ard=ard)
    finally:
        h.close()


# ---- standardisation helpers (StandardGP.jl:164-232, GradientGP.jl:756-822)
def get_mean_std(model, y_train, choice):
    if isinstance(model, GradientGP):
        Y = np.asarray(y_train, dtype=np.float64)
        mu = Y.mean(axis=0); mu[1:] = 0.0
        sd = Y.std(axis=0, ddof=1); sd[1:] = sd[0]
        if choice == "scale_only": mu[:] = 0.0
        elif choice == "mean_only": sd[:] = 1.0
        return mu, sd
    y = np.asarray(y_train, dtype=np.float64).reshape(-1)
    mu, sd = float(y.mean()), float(y.std(ddof=1))
    if choice == "scale_only": mu = 0.0
    elif choice == "mean_only": sd = 1.0
    return mu, sd


def std_y(model, ys, mu, sd):
    if isinstance(model, GradientGP):
        return (np.asarray(ys, dtype=np.float64) - np.asarray(mu)[None, :]) / np.ravel(sd)[0]
    return (np.asarray(ys, dtype=np.float64) - mu) / sd


def rescale_model(model, sd):
    s = float(np.ravel(sd)[0])
    ell = get_lengthscale(model) if is_ard(model) else get_lengthscale(model)[0]
    new_kernel = (get_scale(model)[0] / s ** 2) * with_lengthscale(get_kernel_constructor(model), ell)
    if isinstance(model, GradientGP):
        # quirk mirrored: gradConstMean's inner constructor returns a CustomMean, so the
        # `isa(mean, gradConstMean)` branch never fires and the prior mean is NOT rescaled
        # (GradientGP.jl:505-515, 811-819; SURVEY appendix A)
        return GradientGP(new_kernel, model.p, model.noise_var / s ** 2, model.mean_c, model.ctx)
    mean = None if model.mean_c == 0.0 else model.mean_c / s
    return StandardGP(new_kernel, model.noise_var / s ** 2, mean, model.ctx)


def _update_model_parameters(model, kernel):
    if isinstance(model, GradientGP):
        return GradientGP(kernel, model.p, model.noise_var, model.mean_c, model.ctx)
    return StandardGP(kernel, model.noise_var, None if model.mean_c == 0.0 else model.mean_c, model.ctx)


def _get_minimum(model, ys):
    """StandardGP.jl:418 / GradientGP.jl:1044."""
    y = np.asarray(ys, dtype=np.float64)
    return float(y[:, 0].min()) if isinstance(model, GradientGP) else float(y.min())
