"""Acquisition functions behind the reference's AbstractAcquisition API (src/abstract.jl:49):
functor `acq(surrogate, x)` over a SET of points, `update(acq, ys, surrogate)`, `copy`.
For the GPU surrogates the posterior mean, variance and the formula are evaluated in ONE fused
sweep (abo_acq_eval) instead of two posterior passes (ExpectedImprovement.jl:41-42)."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from .surrogates import _as_points, _get_minimum, _max_value_samples, _need_posterior, pathwise_sample, posterior_sample
from .parallel import merge_topk

ACQ_EI, ACQ_PI, ACQ_UCB, ACQ_GRADNORM_UCB, ACQ_MES = 0, 1, 2, 3, 4


class AbstractAcquisition:
    acq_id = -1
    has_gradient = True          # False: optimize_acquisition returns the best grid point without refinement

    def params(self):
        raise NotImplementedError

    def __call__(self, surrogate, x):
        h = _need_posterior(surrogate)
        scores, _, _ = h.acq_eval(self.acq_id, self.params(), _as_points(x, h.d), k=0)
        return scores

    def value_and_grad(self, surrogate, x):
        """acq(surrogate, x) and its analytic gradient w.r.t. each point, one batched call."""
        h = _need_posterior(surrogate)
        return h.acq_eval_grad(self.acq_id, self.params(), _as_points(x, h.d))

    def topk(self, surrogate, x, k, want_scores=True):
        """scores and sortperm(scores; rev=true)[1:k] (acq_utils.jl:50-52) in one call; 0-based.
        want_scores=False returns None for the scores: only the k selected (index, value) pairs
        leave the device."""
        h = _need_posterior(surrogate)
        return h.acq_eval(self.acq_id, self.params(), _as_points(x, h.d), k=k, want_scores=want_scores)


@dataclass(frozen=True)
class ExpectedImprovement(AbstractAcquisition):
    """ExpectedImprovement(ξ, best_y) (ExpectedImprovement.jl:13-16)."""
    xi: float
    best_y: float
    acq_id = ACQ_EI

    def params(self): return [self.xi, self.best_y]
    def copy(self): return ExpectedImprovement(self.xi, self.best_y)
    def update(self, ys, surrogate): return ExpectedImprovement(self.xi, _get_minimum(surrogate, ys))


@dataclass(frozen=True)
class ProbabilityImprovement(AbstractAcquisition):
    """ProbabilityImprovement(ξ, best_y) (ProbabilityImprovement.jl:11-14)."""
    xi: float
    best_y: float
    acq_id = ACQ_PI

    def params(self): return [self.xi, self.best_y]
    def copy(self): return ProbabilityImprovement(self.xi, self.best_y)
    def update(self, ys, surrogate): return ProbabilityImprovement(self.xi, _get_minimum(surrogate, ys))


@dataclass(frozen=True)
class UpperConfidenceBound(AbstractAcquisition):
    """UpperConfidenceBound(β) (UpperConfidenceBound.jl:12-14)."""
    beta: float
    acq_id = ACQ_UCB

    def params(self): return [self.beta]
    def copy(self): return UpperConfidenceBound(self.beta)
    def update(self, ys, surrogate): return self


@dataclass(frozen=True)
class ThompsonSampling(AbstractAcquisition):
    """Thompson sampling: the acquisition is minus ONE joint posterior draw of f over the evaluated point set
    (abo_gp_posterior_sample), so its maximiser is the minimiser of that draw.  The draw is a function of (seed, point
    set); `update` advances the seed, so every BO iteration draws afresh.  A draw has no gradient: optimize_acquisition
    returns the best grid point."""
    seed: int
    has_gradient = False

    def __call__(self, surrogate, x):
        return -posterior_sample(surrogate, x, 1, seed=self.seed)[0]

    def topk(self, surrogate, x, k, want_scores=True):
        s = self(surrogate, x)
        ti, tv = merge_topk([np.arange(len(s))], [s], k)
        return (s if want_scores else None), ti, tv

    def value_and_grad(self, surrogate, x):
        raise TypeError("ThompsonSampling has no gradient: a posterior draw is not differentiable in x")

    def copy(self): return ThompsonSampling(self.seed)
    def update(self, ys, surrogate): return ThompsonSampling(self.seed + 1)


@dataclass(frozen=True)
class PathwiseThompsonSampling(AbstractAcquisition):
    """Thompson sampling on any grid: the acquisition is minus ONE pathwise posterior draw of f (abo_gp_pathwise_sample,
    num_features random Fourier features conditioned by Matheron's rule), so its maximiser is the minimiser of that draw.
    The draw is a function of (seed, x), whatever else the grid holds; `update` advances the seed.  There is no cap on
    the grid size, unlike ThompsonSampling.  A draw has no gradient here: optimize_acquisition returns the best grid point."""
    seed: int
    num_features: int = 4096
    has_gradient = False

    def __call__(self, surrogate, x):
        return -pathwise_sample(surrogate, x, 1, seed=self.seed, num_features=self.num_features)[0]

    def topk(self, surrogate, x, k, want_scores=True):
        s = self(surrogate, x)
        ti, tv = merge_topk([np.arange(len(s))], [s], k)
        return (s if want_scores else None), ti, tv

    def value_and_grad(self, surrogate, x):
        raise TypeError("PathwiseThompsonSampling has no gradient: draws are evaluated at the grid points only")

    def copy(self): return PathwiseThompsonSampling(self.seed, self.num_features)
    def update(self, ys, surrogate): return PathwiseThompsonSampling(self.seed + 1, self.num_features)


@dataclass(frozen=True)
class MaxValueEntropySearch(AbstractAcquisition):
    """Max-value entropy search (Wang & Jegelka, ICML 2017; BoTorch qMaxValueEntropy), minimising: the expected reduction
    of the entropy of the minimum value f* from observing x, averaged over num_max_values sampled values y*_k
    (ABO_ACQ_MES in include/abo.h: (1/K) sum_k h((mu - y*_k) / sigma), evaluated in the fused sweep, with an analytic
    gradient).  y*_k = min(argmin_val_k, best_y), the minimum of pathwise posterior draw k over the grid clamped at the
    incumbent (max_value_samples); the draws depend on seed, which `update` advances with the incumbent.
    topk(surrogate, grid, k) draws y* over the grid, the standard discretisation.  __call__ and value_and_grad reuse the
    y* of the last topk on the same posterior (the refinement and the reported acquisition value then optimise the
    function the grid was ranked by); without such a draw they draw over the points they evaluate."""
    seed: int
    best_y: float
    num_max_values: int = 16
    num_features: int = 4096
    _cache: dict = field(default_factory=dict, init=False, compare=False, repr=False)
    acq_id = ACQ_MES

    @staticmethod
    def _params(ys):
        return np.concatenate([[float(len(ys))], ys])

    def _draw(self, h, X, best_y):
        return _max_value_samples(h, X, self.num_max_values, self.seed, self.num_features, best_y)

    def _keep(self, h, ys):
        self._cache.clear()
        self._cache.update(token=h.token, ystar=ys)

    def _ystar(self, h, X):
        if self._cache.get("token") == h.token:
            return self._cache["ystar"]
        return self._draw(h, X, self.best_y)

    def __call__(self, surrogate, x):
        h = _need_posterior(surrogate)
        X = _as_points(x, h.d)
        return h.acq_eval(ACQ_MES, self._params(self._ystar(h, X)), X, k=0)[0]

    def value_and_grad(self, surrogate, x):
        h = _need_posterior(surrogate)
        X = _as_points(x, h.d)
        return h.acq_eval_grad(ACQ_MES, self._params(self._ystar(h, X)), X)

    def topk(self, surrogate, x, k, want_scores=True):
        h = _need_posterior(surrogate)
        X = _as_points(x, h.d)
        ys = self._draw(h, X, self.best_y)
        self._keep(h, ys)
        return h.acq_eval(ACQ_MES, self._params(ys), X, k=k, want_scores=want_scores)

    def shard_topk(self, surrogate, shard, k, gather):
        """topk of one rank's shard of a candidate set split over ranks, with the y* of the WHOLE set: each rank draws the
        per-draw minima over its shard, `gather(values)` returns every rank's values in rank order, and their
        NaN-propagating elementwise minimum is what one GPU draws over the whole set (a draw's value at a point does not
        depend on the rest of the set, and min is exact).  Sharded top-k lists then merge to the single-GPU top-k."""
        h = _need_posterior(surrogate)
        X = _as_points(shard, h.d)
        ys = np.minimum(nan_min_reduce(gather(self._draw(h, X, None))), float(self.best_y))
        self._keep(h, ys)
        return h.acq_eval(ACQ_MES, self._params(ys), X, k=k)

    def copy(self):
        return MaxValueEntropySearch(self.seed, self.best_y, self.num_max_values, self.num_features)

    def update(self, ys, surrogate):
        return MaxValueEntropySearch(self.seed + 1, _get_minimum(surrogate, ys), self.num_max_values, self.num_features)


@dataclass(frozen=True)
class qExpectedImprovement(AbstractAcquisition):
    """Monte-Carlo batch expected improvement, qEI (Ginsbourger et al. 2010; BoTorch qExpectedImprovement), minimising:
    the expected improvement of the best of q points evaluated together, (1/S) sum_s max((best_y - xi) - min_j f_{s,j}, 0)
    over S joint posterior draws f_s of the batch (abo_acq_qei).  Batches of near-duplicates score no better than one of
    their points, so a maximiser spreads its q points where each adds something.  The draws use the same num_samples base
    normals for every batch (from `seed`), so the value is a smooth, deterministic function of the points with an exact
    gradient.  optimize_acquisition proposes (q, d) batches for it and `optimize` evaluates q points per iteration;
    `update` takes the new incumbent and advances the seed."""
    xi: float
    best_y: float
    q: int
    num_samples: int = 512
    seed: int = 0

    @staticmethod
    def _batches(h, batches):
        b = np.asarray(batches, dtype=np.float64)
        return b[None] if b.ndim == 2 else b

    def __call__(self, surrogate, batches):
        """qEI of each batch of `batches`, shape (B, q, d) (or one (q, d) batch): B values."""
        h = _need_posterior(surrogate)
        return h.acq_qei([self.xi, self.best_y], self.q, self._batches(h, batches), self.num_samples, self.seed)[0]

    def value_and_grad(self, surrogate, batches):
        """qEI of each batch and its gradient with respect to every coordinate of its points: (B,), (B, q, d)."""
        h = _need_posterior(surrogate)
        v, g, _ = h.acq_qei([self.xi, self.best_y], self.q, self._batches(h, batches), self.num_samples, self.seed,
                            want_grad=True)
        return v, g

    def topk(self, surrogate, x, k, want_scores=True):
        raise TypeError("qExpectedImprovement scores batches of q points, not single points (see optimize_acquisition)")

    def copy(self): return qExpectedImprovement(self.xi, self.best_y, self.q, self.num_samples, self.seed)

    def update(self, ys, surrogate):
        return qExpectedImprovement(self.xi, _get_minimum(surrogate, ys), self.q, self.num_samples, self.seed + 1)


def nan_min_reduce(arrays):
    """Elementwise minimum of equally long arrays; a NaN in any of them gives NaN there (np.minimum)."""
    out = np.asarray(arrays[0], dtype=np.float64)
    for a in arrays[1:]:
        out = np.minimum(out, np.asarray(a, dtype=np.float64))
    return out


def _fd_value_and_grad(acq, surrogate, x, rel_step=6.0554544523933395e-06):
    """Value and central-difference gradient for a batch of points in ONE batched evaluation of m (2 d + 1) points
    (what Optim's finite-difference default does one point and one coordinate at a time, acq_utils.jl:55-63);
    step = cbrt(eps) * max(1, |x_k|)."""
    X = np.asarray(x, dtype=np.float64)
    m, d = X.shape
    h = rel_step * np.maximum(1.0, np.abs(X))
    P = np.repeat(X[:, None, :], 2 * d + 1, axis=1)
    for k in range(d):
        P[:, 1 + 2 * k, k] += h[:, k]; P[:, 2 + 2 * k, k] -= h[:, k]
    v = np.asarray(acq(surrogate, P.reshape(-1, d))).reshape(m, 2 * d + 1)
    grad = (v[:, 1::2] - v[:, 2::2]) / (2 * h)
    return v[:, 0].copy(), grad


@dataclass(frozen=True)
class GradientNormUCB(AbstractAcquisition):
    """GradientNormUCB(β) (gradNormUCB.jl:12-51): UCB on the squared 2-norm of the gradient of a GradientGP.  Per point:
    m = posterior gradient mean, Σ = posterior gradient covariance (d x d), -(m·m + tr Σ) + β sqrt(max(4 mᵀΣm + 2‖Σ‖_F², 1e-12)).
    Evaluated on the device for the whole candidate set (abo_acq_eval_multi: K* with all p output columns, one DMMA
    triangular product, the p x p covariance blocks and the formula in the epilogue kernels)."""
    beta: float
    acq_id = ACQ_GRADNORM_UCB

    def params(self): return [self.beta]
    def copy(self): return GradientNormUCB(self.beta)
    def update(self, ys, surrogate): return self

    def _eval(self, surrogate, x, k=0, want_scores=True):
        h = _need_posterior(surrogate)
        if h.p < 2:
            raise TypeError("GradientNormUCB needs a GradientGP surrogate")
        return h.acq_eval_multi([ACQ_GRADNORM_UCB], [1.0], [[self.beta, 0.0]], _as_points(x, h.d), k=k, want_scores=want_scores)

    def __call__(self, surrogate, x):
        return self._eval(surrogate, x)[0]

    def topk(self, surrogate, x, k, want_scores=True):
        return self._eval(surrogate, x, k=k, want_scores=want_scores)

    def value_and_grad(self, surrogate, x):
        return _fd_value_and_grad(self, surrogate, _as_points(x, _need_posterior(surrogate).d))


class EnsembleAcquisition(AbstractAcquisition):
    """EnsembleAcquisition(weights, acquisitions) (EnsembleAcq.jl:12-55): non-negative weights, normalised to sum 1;
    value = Σ w_i acq_i(surrogate, x).  When every member is EI / PI / UCB / GradientNormUCB the members share ONE
    posterior pass on the device (abo_acq_eval_multi); other members are evaluated one after the other."""

    def __init__(self, weights, acquisitions):
        w = np.asarray(weights, dtype=np.float64)
        if len(w) != len(acquisitions):
            raise ValueError("weights and acquisitions must align")
        if np.any(w < 0):
            raise ValueError("weights must be non-negative")
        if not w.sum() > 0:
            raise ValueError("sum of weights must be positive")
        self.weights = w / w.sum()
        self.acquisitions = list(acquisitions)

    def copy(self): return EnsembleAcquisition(self.weights.copy(), [a.copy() for a in self.acquisitions])
    def update(self, ys, surrogate): return EnsembleAcquisition(self.weights, [a.update(ys, surrogate) for a in self.acquisitions])

    def _fusable(self):
        return len(self.acquisitions) <= 8 and all(getattr(a, "acq_id", -1) in (ACQ_EI, ACQ_PI, ACQ_UCB, ACQ_GRADNORM_UCB)
                                                   and not isinstance(a, EnsembleAcquisition)
                                                   for a in self.acquisitions)

    def _eval(self, surrogate, x, k=0, want_scores=True, grid=False):
        h = _need_posterior(surrogate)
        if self._fusable():
            return h.acq_eval_multi([a.acq_id for a in self.acquisitions], self.weights, [a.params() for a in self.acquisitions],
                                    _as_points(x, h.d), k=k, want_scores=want_scores)
        # the grid sweep of the sequential path is every member's own grid sweep (topk, same scores as the functor), so
        # that a member which draws per grid (MaxValueEntropySearch) keeps that draw for the refinement
        s = sum(w * (a.topk(surrogate, x, 0)[0] if grid else a(surrogate, x)) for w, a in zip(self.weights, self.acquisitions))
        ti, tv = merge_topk([np.arange(len(s))], [s], k)
        return s, ti, tv

    def __call__(self, surrogate, x):
        return self._eval(surrogate, x)[0]

    def topk(self, surrogate, x, k, want_scores=True):
        return self._eval(surrogate, x, k=k, want_scores=want_scores, grid=True)

    def value_and_grad(self, surrogate, x):
        return _fd_value_and_grad(self, surrogate, _as_points(x, _need_posterior(surrogate).d))
