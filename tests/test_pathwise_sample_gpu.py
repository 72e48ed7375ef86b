"""Pathwise posterior draws on the device (abo_gp_pathwise_sample): parity with the NumPy reference on the same streams,
the bitwise guarantees of the header across sets, pieces, entry points and draw counts, sample statistics against the
exact posterior, the posterior left untouched, argument errors, and Thompson sampling on a grid above the exact
sampler's cap inside the BO loop."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import pathwise_reference as pref  # noqa: E402

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
KNAME = {0: "SqExponentialKernel", 1: "Matern52Kernel", 2: "Matern72Kernel"}


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


def check_parity(F, post, Xc, S, seed, L, scale):
    """The device and the reference differ by the rounding of v = (K + noise I)^-1 R, which cond(K + noise I) amplifies:
    |dF| <= c eps cond sqrt(sigma^2) max|theta, eps normals|, with c = 64 covering the O(1) norms of k* and of the
    feature rows.  Every other term is evaluated elementwise to a few ulps."""
    Fo, Theta = pref.pathwise_sample(post, Xc, S, seed, L)
    U = post.U
    cond = np.linalg.cond(U.T @ U)
    tol = max(1e-9, 64 * EPS * cond) * np.sqrt(scale) * np.max(np.abs(Theta))
    err = np.max(np.abs(F - Fo))
    assert err <= tol, (err, tol, cond)


@pytest.mark.parametrize("case", ["se", "matern52", "matern72", "ard"])
def test_standard_gp_parity(abo, orc, case):
    rng = np.random.default_rng({"se": 1, "matern52": 2, "matern72": 3, "ard": 4}[case])
    n, d, m, S, L, seed = 500, 6, 3000, 64, 1024, 2024
    kind = {"se": 0, "matern52": 1, "matern72": 2, "ard": 1}[case]
    ell = np.array([0.4, 0.9, 1.5, 0.6, 2.0, 0.8]) if case == "ard" else 0.7
    X, y = data(rng, n, d)
    Xc = rng.random((m, d)) * 1.2 - 0.1
    gp = abo.update(abo.StandardGP(1.7 * abo.with_lengthscale(abo.Kernel(KNAME[kind]), ell), 1e-4, mean=0.2), X, y)
    F, ai, av = gp.gpx.pathwise_sample(Xc, S, seed, L)
    post = orc.fit_standard(X, y, kind, 1.0 / np.asarray(ell), 1.7, 1e-4, 0.2)
    check_parity(F, post, Xc, S, seed, L, 1.7)
    assert np.array_equal(ai, np.argmin(F, axis=1)) and np.array_equal(av, F[np.arange(S), ai])


def test_gradient_gp_value_parity(abo, orc):
    rng = np.random.default_rng(5)
    n, d, m, S, L, seed = 300, 3, 3000, 64, 1024, 5
    X, Y = data(rng, n, d, gradient=True)
    Xc = rng.random((m, d))
    gp = abo.update(abo.GradientGP(1.3 * abo.with_lengthscale(abo.ApproxMatern52Kernel(), 0.8), d + 1, 1e-4), X, Y)
    F, ai, _ = gp.gpx.pathwise_sample(Xc, S, seed, L)
    post = orc.fit_gradient(X, Y, 3, 1.0 / 0.8, 1.3, 1e-4)
    check_parity(F, post, Xc, S, seed, L, 1.3)
    assert np.array_equal(ai, np.argmin(F, axis=1))


def test_bitwise_guarantees(abo):
    import torch
    rng = np.random.default_rng(6)
    X, y = data(rng, 2048, 4)
    gp = abo.update(abo.StandardGP(1.2 * abo.with_lengthscale(abo.Matern52Kernel(), 0.5), 1e-4), X, y)
    h = gp.gpx
    m, S, L, seed = 1_000_000, 64, 2048, 99
    Xc = rng.random((m, 4))
    F, ai, av = h.pathwise_sample(Xc, S, seed, L)                   # host set above the piece size: staged in pieces
    assert np.array_equal(ai, np.argmin(F, axis=1)) and np.array_equal(av, F[np.arange(S), ai])
    dX = torch.from_numpy(Xc).cuda()
    dF = torch.empty((S, m), dtype=torch.float64, device="cuda")
    ai_d, av_d = h.pathwise_sample_dev(dX.data_ptr(), m, S, seed, L, dF.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(dF.cpu().numpy(), F) and np.array_equal(ai_d, ai) and np.array_equal(av_d, av)
    del dX, dF
    idx = rng.choice(m, 5000, replace=False)
    Fs, ais, avs = h.pathwise_sample(Xc[idx], S, seed, L)
    assert np.array_equal(Fs, F[:, idx])
    assert np.array_equal(ais, np.argmin(F[:, idx], axis=1)) and np.array_equal(avs, Fs[np.arange(S), ais])
    F16, ai16, _ = h.pathwise_sample(Xc[:300_000], 16, seed, L)
    assert np.array_equal(F16, F[:16, :300_000]) and np.array_equal(ai16, np.argmin(F[:16, :300_000], axis=1))
    none, ai_only, av_only = h.pathwise_sample(Xc, S, seed, L, want_samples=False)
    assert none is None and np.array_equal(ai_only, ai) and np.array_equal(av_only, av)
    assert np.array_equal(abo.pathwise_thompson_batch(gp, Xc[idx], S, seed=seed, num_features=L), ais)
    again = h.pathwise_sample(Xc[idx], S, seed, L)
    assert np.array_equal(again[0], Fs) and np.array_equal(again[1], ais)
    assert np.mean(h.pathwise_sample(Xc[idx], S, seed + 1, L)[0] == Fs) < 1e-3
    gp.ctx.trim()


def test_statistics_against_the_exact_posterior(abo, orc):
    """The draws are unbiased for any fixed features, so the sample mean is checked at 5 Monte-Carlo standard errors.  The
    covariance differs from the exact one by the Monte-Carlo error (6 standard errors of a covariance estimate) plus the
    feature approximation of the prior: with per-entry error at most sigma^2 / sqrt(L) (each feature term 2 cos cos has
    variance <= 1), propagated through the conditioning x -> [1, -K^-1 k*] as 6 a_i a_j sigma^2 / sqrt(L), a_i the
    1-norm of that row."""
    rng = np.random.default_rng(7)
    X, y = data(rng, 40, 2)
    Xc = np.vstack([X[:16] + 0.02 * rng.standard_normal((16, 2)), rng.random((24, 2)) * 1.5, 1.5 + rng.random((24, 2))])
    sc, ell, noise = 2.0, 0.5, 1e-3
    gp = abo.update(abo.StandardGP(sc * abo.with_lengthscale(abo.SqExponentialKernel(), ell), noise), X, y)
    S, L = 4096, 16384
    F = abo.pathwise_sample(gp, Xc, S, seed=12, num_features=L)
    post = orc.fit_standard(X, y, 0, 1.0 / ell, sc, noise)
    mu, _ = orc.posterior_mean_var(post, Xc)
    mu_dev, _ = gp.gpx.posterior(Xc, 1, True, True)
    sig = orc.posterior_cov(post, Xc, outputs=[0])
    dg = np.diag(sig)
    assert np.all(np.abs(F.mean(0) - mu_dev) <= 5 * np.sqrt(dg / S))
    w = np.linalg.solve(post.U.T @ post.U, orc._kstar(post, Xc, [0]))
    a = 1.0 + np.abs(w).sum(0)
    C_ = np.cov(F, rowvar=False, bias=True)
    bound = 6 * np.sqrt((np.outer(dg, dg) + sig ** 2) / S) + 6 * np.outer(a, a) * sc / np.sqrt(L)
    assert np.all(np.abs(C_ - sig) <= bound)
    assert np.abs(np.diag(C_) - dg).max() <= 0.2 * sc             # the draws do carry the posterior spread


def test_posterior_untouched_and_clone(abo):
    rng = np.random.default_rng(8)
    X, y = data(rng, 400, 3)
    Xc = rng.random((2000, 3))
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.Matern52Kernel(), 0.5), 1e-4), X, y)
    clone = gp.copy()
    a0, L0, Li0 = gp.gpx.alpha(), gp.gpx.factor(0), gp.gpx.factor(1)
    mu0 = abo.posterior_mean(gp, Xc)
    abo.pathwise_sample(gp, Xc, 256, seed=1)
    assert np.array_equal(gp.gpx.alpha(), a0) and np.array_equal(gp.gpx.factor(0), L0) and np.array_equal(gp.gpx.factor(1), Li0)
    assert np.array_equal(clone.gpx.alpha(), a0) and np.array_equal(clone.gpx.factor(0), L0)
    assert np.array_equal(abo.posterior_mean(clone, Xc), mu0) and np.array_equal(abo.posterior_mean(gp, Xc), mu0)
    assert np.array_equal(abo.pathwise_sample(clone, Xc, 8, seed=2), abo.pathwise_sample(gp, Xc, 8, seed=2))


def test_errors(abo):
    from abo_b200 import _lib
    Lb = _lib.lib()
    rng = np.random.default_rng(9)
    X, y = data(rng, 50, 2)
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 1e-4), X, y)
    h = gp.gpx
    Xc = rng.random((100, 2))

    def call(handle, m, S, L, xc_null=False):
        out = np.empty(max(S, 1) * max(m, 1))
        return Lb.abo_gp_pathwise_sample(handle, None if xc_null else _lib.ptr(Xc), m, S, L, 1, _lib.ptr(out), None, None)

    unfit = _lib.GpHandle(gp.ctx, 0, 2, 1)
    assert call(unfit._h, 10, 4, 64) == _lib.ABO_ERR_NOT_FITTED
    assert call(h._h, 10, 4097, 64) == _lib.ABO_ERR_INVALID
    assert call(h._h, 10, 4, 0) == _lib.ABO_ERR_INVALID and call(h._h, 10, 4, 16385) == _lib.ABO_ERR_INVALID
    assert call(h._h, 10, 4, 64, xc_null=True) == _lib.ABO_ERR_INVALID
    assert Lb.abo_gp_pathwise_sample_dev(h._h, None, 10, 4, 64, 1, None, None, None) == _lib.ABO_ERR_INVALID
    assert call(h._h, 0, 4, 64) == _lib.ABO_OK and call(h._h, 10, 0, 64) == _lib.ABO_OK
    with pytest.raises(ValueError):
        h.pathwise_sample(Xc, 4, -1)
    assert np.all(np.isfinite(h.pathwise_sample(Xc, 4, 1, 64)[0]))


def test_pathwise_thompson_bo_loop_on_a_large_grid(abo):
    f = lambda x: (x[0] ** 2 + x[1] - 11) ** 2 + (x[0] + x[1] ** 2 - 7) ** 2
    domain = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    rng = np.random.default_rng(0)
    xs = [domain.lower + (domain.upper - domain.lower) * rng.random(2) for _ in range(5)]
    ys = [f(x) for x in xs]
    best0 = min(ys)
    model = abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0), 1e-9)
    bo = abo.BOStruct(f, abo.PathwiseThompsonSampling(2024), model, domain, xs, ys, 15, 0.0)
    bo, acq_values, _ = abo.optimize(bo, standardize="mean_only", hyper_params="all", num_restarts_HP=4, n_grid=200_000, rng=rng)
    assert len(acq_values) == 15 or bo.flag
    assert bo.acq.seed > 2024 + len(acq_values) - 1
    assert min(np.ravel(bo.ys_non_std)) < best0
