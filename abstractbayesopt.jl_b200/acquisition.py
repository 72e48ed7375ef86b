"""Acquisition functions behind the reference's AbstractAcquisition API (src/abstract.jl:49):
functor `acq(surrogate, x)` over a SET of points, `update(acq, ys, surrogate)`, `copy`.
For the GPU surrogates the posterior mean, variance and the formula are evaluated in ONE fused
sweep (abo_acq_eval) instead of two posterior passes (ExpectedImprovement.jl:41-42)."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .surrogates import _as_points, _get_minimum, _need_posterior, posterior_sample
from .parallel import merge_topk

ACQ_EI, ACQ_PI, ACQ_UCB = 0, 1, 2


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


ACQ_GRADNORM_UCB = 3


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
        return len(self.acquisitions) <= 8 and all(getattr(a, "acq_id", -1) in (0, 1, 2, 3) and not isinstance(a, EnsembleAcquisition)
                                                   for a in self.acquisitions)

    def _eval(self, surrogate, x, k=0, want_scores=True):
        h = _need_posterior(surrogate)
        if self._fusable():
            return h.acq_eval_multi([a.acq_id for a in self.acquisitions], self.weights, [a.params() for a in self.acquisitions],
                                    _as_points(x, h.d), k=k, want_scores=want_scores)
        s = sum(w * a(surrogate, x) for w, a in zip(self.weights, self.acquisitions))
        ti, tv = merge_topk([np.arange(len(s))], [s], k)
        return s, ti, tv

    def __call__(self, surrogate, x):
        return self._eval(surrogate, x)[0]

    def topk(self, surrogate, x, k, want_scores=True):
        return self._eval(surrogate, x, k=k, want_scores=want_scores)

    def value_and_grad(self, surrogate, x):
        return _fd_value_and_grad(self, surrogate, _as_points(x, _need_posterior(surrogate).d))
