"""Joint posterior draws on the device (abo_gp_posterior_sample): parity with the NumPy reference fed the same normals
and the same jitter, sample statistics, shapes up to the caps, the determinism contract of the header, the posterior left
untouched, the jitter ladder, argument errors, and Thompson sampling inside the BO loop."""
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sla

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sample_reference as ref  # noqa: E402

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
KNAME = {0: "SqExponentialKernel", 1: "Matern52Kernel"}


@pytest.fixture(scope="module")
def abo():
    import abo_b200
    return abo_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import abo_oracle
    return abo_oracle


def data(rng, n, d, gradient=False):
    X = rng.random((n, d))
    f = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, -1]) + 0.5 * X.sum(1)
    if not gradient:
        return X, f
    g = np.zeros((n, d)); g[:, 0] = 3 * np.cos(3 * X[:, 0]); g[:, -1] += -2 * np.sin(2 * X[:, -1]); g += 0.5
    return X, np.column_stack([f, g])


def check_parity(F, post, Xc, S, seed, tau, scale, cond=None):
    Fo, sig, Z = ref.posterior_sample(post, Xc, S, seed, tau)
    if cond is None:
        w = np.linalg.eigvalsh(sig)
        cond = w[-1] / w[0]
    tol = max(1e-9, 16 * EPS * cond) * np.sqrt(scale) * np.max(np.abs(Z))
    err = np.max(np.abs(F - Fo))
    assert err <= tol, (err, tol, cond)
    return Fo


@pytest.mark.parametrize("case", ["se", "matern52", "ard"])
def test_standard_gp_parity(abo, orc, case):
    rng = np.random.default_rng({"se": 1, "matern52": 2, "ard": 3}[case])
    n, d, m, S, seed = 500, 6, 1000, 64, 2024
    kind = 1 if case == "matern52" else 0
    ell = np.array([0.4, 0.9, 1.5, 0.6, 2.0, 0.8]) if case == "ard" else 0.7
    X, y = data(rng, n, d)
    Xc = rng.random((m, d))
    gp = abo.update(abo.StandardGP(1.7 * abo.with_lengthscale(abo.Kernel(KNAME[kind]), ell), 1e-4, mean=0.2), X, y)
    F, ai, av, tau = gp.gpx.posterior_sample(Xc, S, seed)
    assert tau in [1e-10 * 1.7 * 10.0 ** k for k in range(7)]
    post = orc.fit_standard(X, y, kind, 1.0 / np.asarray(ell), 1.7, 1e-4, 0.2)
    check_parity(F, post, Xc, S, seed, tau, 1.7)
    mu_o, _ = orc.posterior_mean_var(post, Xc)
    assert np.max(np.abs(abo.posterior_mean(gp, Xc) - mu_o)) <= 1e-9 * max(np.max(np.abs(mu_o)), np.sqrt(1.7))
    assert np.array_equal(ai, np.argmin(F, axis=1)) and np.array_equal(av, F[np.arange(S), ai])


def test_gradient_gp_value_parity(abo, orc):
    rng = np.random.default_rng(4)
    n, d, m, S, seed = 300, 3, 1000, 64, 5
    X, Y = data(rng, n, d, gradient=True)
    Xc = rng.random((m, d))
    gp = abo.update(abo.GradientGP(1.3 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.8), d + 1, 1e-4), X, Y)
    F, _, _, tau = gp.gpx.posterior_sample(Xc, S, seed)
    post = orc.fit_gradient(X, Y, 0, 1.0 / 0.8, 1.3, 1e-4)
    # cond2(K) of the N = 1200 gradient system is 4e6, so the two FP64 evaluations of Sigma already differ by about
    # cond2(K) eps sigma^2, which the factorisation amplifies by up to cond2(Sigma) = 2.6e6: the draws then differ by
    # ~1e-7, beyond the factorisation-only bound.  Sigma is compared on its own (the device's abo_gp_posterior_cov against
    # the oracle, which test_gpu_parity covers for the gradient blocks); the draws are checked against the reference
    # factorisation of the device's Sigma, with the oracle's mean and the same normals.
    sig_dev = gp.gpx.posterior_cov(Xc, 1)
    sig_o = orc.posterior_cov(post, Xc, outputs=[0])
    assert np.max(np.abs(sig_dev - sig_o)) <= 1e-9 * 1.3
    sig = sig_dev + tau * np.eye(m)
    w = np.linalg.eigvalsh(sig)
    L = sla.cholesky(sig, lower=True)
    Z = ref.normals(seed, S, m)
    mean_o, _ = orc.posterior_mean_var(post, Xc)
    tol = max(1e-9, 16 * EPS * w[-1] / w[0]) * np.sqrt(1.3) * np.max(np.abs(Z))
    assert np.max(np.abs(F - (mean_o[None, :] + Z @ L.T))) <= tol
    assert np.max(np.abs(F - ref.posterior_sample(post, Xc, S, seed, tau)[0])) <= 1e-6 * np.sqrt(1.3)


def test_sample_statistics(abo, orc):
    rng = np.random.default_rng(6)
    X, y = data(rng, 40, 2)
    Xc = rng.random((48, 2)) * 1.5
    gp = abo.update(abo.StandardGP(2.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.5), 1e-3), X, y)
    S = 4096
    F = abo.posterior_sample(gp, Xc, S, seed=99)
    post = orc.fit_standard(X, y, 0, 2.0, 2.0, 1e-3)
    mu, _ = orc.posterior_mean_var(post, Xc)
    sig = orc.posterior_cov(post, Xc, outputs=[0])
    dg = np.diag(sig)
    assert np.all(np.abs(F.mean(0) - mu) <= 5 * np.sqrt(dg / S))
    C_ = np.cov(F, rowvar=False, bias=True)
    assert np.all(np.abs(C_ - sig) <= 6 * np.sqrt((np.outer(dg, dg) + sig ** 2) / S))


@pytest.mark.parametrize("m", [1, 127, 128, 129, 4224])
def test_shapes_against_reference(abo, orc, m):
    rng = np.random.default_rng(m)
    X, y = data(rng, 200, 4)
    Xc = rng.random((m, 4))
    gp = abo.update(abo.StandardGP(1.1 * abo.with_lengthscale(abo.Matern52Kernel(), 0.6), 1e-4), X, y)
    S = 8
    F, ai, _, tau = gp.gpx.posterior_sample(Xc, S, 31)
    assert F.shape == (S, m) and ai.shape == (S,)
    post = orc.fit_standard(X, y, 1, 1.0 / 0.6, 1.1, 1e-4)
    cond = None
    if m > 2000:
        L = sla.cholesky(orc.posterior_cov(post, Xc, outputs=[0]) + tau * np.eye(m), lower=True)
        cond = orc.cond_estimate(L.T)
    check_parity(F, post, Xc, S, 31, tau, 1.1, cond)


def test_m8192_n4096_against_reference(abo, orc):
    rng = np.random.default_rng(8)
    X, y = data(rng, 4096, 8)
    Xc = rng.random((8192, 8))
    gp = abo.update(abo.StandardGP(1.0 * abo.with_lengthscale(abo.Matern52Kernel(), 0.5), 1e-3), X, y)
    S = 4
    F, ai, _, tau = gp.gpx.posterior_sample(Xc, S, 77)
    post = orc.fit_standard(X, y, 1, 2.0, 1.0, 1e-3)
    mean, _ = orc.posterior_mean_var(post, Xc)
    sig = orc.posterior_cov(post, Xc, outputs=[0]) + tau * np.eye(len(Xc))
    L = sla.cholesky(sig, lower=True, check_finite=False)
    Z = ref.normals(77, S, len(Xc))
    Fo = mean[None, :] + Z @ L.T
    tol = max(1e-9, 16 * EPS * orc.cond_estimate(L.T)) * np.max(np.abs(Z))
    assert np.max(np.abs(F - Fo)) <= tol
    assert np.array_equal(ai, np.argmin(F, axis=1))


def test_caps_m16384_n8192_d20(abo):
    rng = np.random.default_rng(9)
    X, y = data(rng, 8192, 20)
    Xc = rng.random((16384, 20))
    gp = abo.update(abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 1.5), 1e-3), X, y)
    S = 32
    F, ai, av, tau = gp.gpx.posterior_sample(Xc, S, 3)
    assert np.all(np.isfinite(F)) and np.array_equal(ai, np.argmin(F, axis=1)) and np.array_equal(av, F.min(1))
    mu, var = gp.gpx.posterior(Xc, 1, True, True)
    assert np.all(np.abs(F - mu[None, :]) <= 8 * np.sqrt(var + tau)[None, :])
    F16, ai16, _, _ = gp.gpx.posterior_sample(Xc, 16, 3)
    assert np.array_equal(F16, F[:16]) and np.array_equal(ai16, ai[:16])
    gp.ctx.trim()


def test_determinism_and_argmin(abo):
    rng = np.random.default_rng(10)
    X, y = data(rng, 300, 3)
    Xc = rng.random((3000, 3))
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 0.4), 1e-4), X, y)
    h = gp.gpx
    F64, ai64, av64, tau = h.posterior_sample(Xc, 64, 123)
    again = h.posterior_sample(Xc, 64, 123)
    assert np.array_equal(F64, again[0]) and np.array_equal(ai64, again[1]) and again[3] == tau
    F16, ai16, _, _ = h.posterior_sample(Xc, 16, 123)
    assert np.array_equal(F16, F64[:16]) and np.array_equal(ai16, ai64[:16])
    none, ai_only, av_only, _ = h.posterior_sample(Xc, 64, 123, want_samples=False)
    assert none is None and np.array_equal(ai_only, np.argmin(F64, axis=1)) and np.array_equal(av_only, F64.min(1))
    assert np.array_equal(abo.thompson_batch(gp, Xc, 64, seed=123), ai_only)
    other = h.posterior_sample(Xc, 64, 124)[0]
    assert np.mean(other == F64) < 1e-3
    # ties go to the first index: duplicated candidates draw (nearly) equal values, the argmin is checked exactly
    Xd = np.repeat(Xc[:50], 2, axis=0)
    Fd, aid, _, _ = h.posterior_sample(Xd, 32, 5)
    assert np.array_equal(aid, np.argmin(Fd, axis=1))


def test_posterior_untouched_and_clone(abo):
    rng = np.random.default_rng(11)
    X, y = data(rng, 400, 3)
    Xc = rng.random((2000, 3))
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.Matern52Kernel(), 0.5), 1e-4), X, y)
    clone = gp.copy()
    a0, L0, Li0 = gp.gpx.alpha(), gp.gpx.factor(0), gp.gpx.factor(1)
    mu0 = abo.posterior_mean(gp, Xc)
    abo.posterior_sample(gp, Xc, 256, seed=1)
    assert np.array_equal(gp.gpx.alpha(), a0) and np.array_equal(gp.gpx.factor(0), L0) and np.array_equal(gp.gpx.factor(1), Li0)
    assert np.array_equal(clone.gpx.alpha(), a0) and np.array_equal(clone.gpx.factor(0), L0)
    assert np.array_equal(abo.posterior_mean(clone, Xc), mu0) and np.array_equal(abo.posterior_mean(gp, Xc), mu0)
    assert np.array_equal(abo.posterior_sample(clone, Xc, 8, seed=2), abo.posterior_sample(gp, Xc, 8, seed=2))


def test_jitter_ladder(abo):
    rng = np.random.default_rng(12)
    X, y = data(rng, 100, 2)
    gp = abo.update(abo.StandardGP(3.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.7), 1e-6), X, y)
    x0 = rng.random(2)
    Xc = np.vstack([np.repeat(x0[None, :], 32, axis=0), rng.random((32, 2))])
    F, _, _, tau = gp.gpx.posterior_sample(Xc, 8, 4, jitter=1e-14)
    ladder = [1e-14 * 3.0 * 10.0 ** k for k in range(7)]
    assert any(abs(tau - t) <= 1e-12 * t for t in ladder), tau
    assert np.all(np.isfinite(F))
    assert np.max(np.abs(F[:, :32] - F[:, :1])) <= 10 * np.sqrt(tau)


def test_errors(abo):
    from abo_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(13)
    X, y = data(rng, 50, 2)
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 1e-4), X, y)
    h = gp.gpx

    def call(handle, Xc, m, S, jitter=1e-10, xc_null=False):
        out = np.empty(max(S, 1) * max(m, 1))
        return L.abo_gp_posterior_sample(handle, None if xc_null else _lib.ptr(Xc), m, S, 1, jitter, _lib.ptr(out),
                                         None, None, None)

    Xc = rng.random((16385, 2))
    unfit = _lib.GpHandle(gp.ctx, 0, 2, 1)
    assert call(unfit._h, Xc, 10, 4) == _lib.ABO_ERR_NOT_FITTED
    assert call(h._h, Xc, 16385, 4) == _lib.ABO_ERR_INVALID
    assert call(h._h, Xc, 10, 4097) == _lib.ABO_ERR_INVALID
    for bad in (0.0, -1e-10, float("nan"), float("inf")):
        assert call(h._h, Xc, 10, 4, jitter=bad) == _lib.ABO_ERR_INVALID
    assert call(h._h, Xc, 10, 4, xc_null=True) == _lib.ABO_ERR_INVALID
    assert call(h._h, Xc, 0, 4) == _lib.ABO_OK and call(h._h, Xc, 10, 0) == _lib.ABO_OK
    with pytest.raises(ValueError):
        h.posterior_sample(Xc[:10], 4, -1)
    # the handle still samples after the failed calls
    assert np.all(np.isfinite(h.posterior_sample(Xc[:10], 4, 1)[0]))


def _himmelblau_run(abo, seed):
    f = lambda x: (x[0] ** 2 + x[1] - 11) ** 2 + (x[0] + x[1] ** 2 - 7) ** 2
    domain = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    rng = np.random.default_rng(0)
    xs = [domain.lower + (domain.upper - domain.lower) * rng.random(2) for _ in range(5)]
    ys = [f(x) for x in xs]
    model = abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0), 1e-9)
    bo = abo.BOStruct(f, abo.ThompsonSampling(seed), model, domain, xs, ys, 15, 0.0)
    bo, acq_values, _ = abo.optimize(bo, standardize="mean_only", hyper_params="all", num_restarts_HP=4, rng=rng)
    return bo, acq_values, min(ys)


def test_thompson_sampling_bo_loop(abo):
    bo, acq_values, best0 = _himmelblau_run(abo, 2024)
    assert len(acq_values) == 15 or bo.flag
    assert bo.acq.seed > 2024 + len(acq_values) - 1                          # every iteration drew with a fresh seed
    assert min(np.ravel(bo.ys_non_std)) < best0
    bo2, acq2, _ = _himmelblau_run(abo, 2024)
    assert all(np.array_equal(a, b) for a, b in zip(bo.xs, bo2.xs)) and acq2 == acq_values
