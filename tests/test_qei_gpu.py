"""Monte-Carlo batch expected improvement on the device (abo_acq_qei): parity of values and gradients with the torch
reference, the determinism contract of the header (chunk boundaries, other batches, a NULL gradient, repeated calls), q = 1
against analytic EI, the jitter ladder and the zero-improvement case, the posterior left untouched, argument errors, and
qExpectedImprovement inside optimize_acquisition and the BO loop."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import qei_reference as qref  # noqa: E402

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


def model(abo, orc, case, n=500, d=6, seed=0):
    """(surrogate, oracle posterior, kernel scale) for case se / matern52 / ard / gradient."""
    rng = np.random.default_rng(seed)
    scale = 1.7
    if case == "gradient":
        X, Y = data(rng, n, d, gradient=True)
        gp = abo.update(abo.GradientGP(scale * abo.with_lengthscale(abo.SqExponentialKernel(), 0.8), d + 1, 1e-4), X, Y)
        return gp, orc.fit_gradient(X, Y, 0, 1.0 / 0.8, scale, 1e-4), scale, rng
    kind = 1 if case == "matern52" else 0
    ell = np.array([0.4, 0.9, 1.5, 0.6, 2.0, 0.8])[:d] if case == "ard" else 0.7
    X, y = data(rng, n, d)
    gp = abo.update(abo.StandardGP(scale * abo.with_lengthscale(abo.Kernel(KNAME[kind]), ell), 1e-4, mean=0.2), X, y)
    return gp, orc.fit_standard(X, y, kind, 1.0 / np.asarray(ell), scale, 1e-4, 0.2), scale, rng


@pytest.mark.parametrize("q", [1, 3, 8, 32])
@pytest.mark.parametrize("case", ["se", "matern52", "ard", "gradient"])
def test_parity_with_reference(abo, orc, case, q):
    gp, post, scale, rng = model(abo, orc, case)
    B, S, seed, xi = 50, 256, 11, 0.01
    Xb = rng.random((B, q, 6))
    mu, _ = orc.posterior_mean_var(post, Xb.reshape(-1, 6))
    best = float(np.quantile(mu, 0.3))
    v, g, tau = gp.gpx.acq_qei([xi, best], q, Xb, S, seed, want_grad=True)
    vr, gr, taur, _ = qref.qei(post, Xb, xi, best, S, seed)
    assert np.array_equal(tau, taur) and np.all(tau == 1e-10 * scale)
    # Sigma enters through W = L^-1 K*: the two FP64 evaluations of Sigma differ by about cond(K + noise I) eps sigma^2, and
    # its Cholesky (and, for the gradient, the Cholesky backward, which applies L_Sigma^-1 twice) amplifies that by up to
    # cond(Sigma + tau I) per application.  The draws scale with sigma max|z|.
    condK = np.linalg.cond(post.U) ** 2
    sig, _ = qref._sigma_mu(post, torch.as_tensor(Xb))
    w = np.linalg.eigvalsh(sig.numpy() + tau[:, None, None] * np.eye(q))
    condS = float(np.max(w[:, -1] / w[:, 0]))
    zmax = float(np.max(np.abs(qref.normals(seed, S, q))))
    tol_v = max(1e-9, 16 * EPS * condK * condS) * np.sqrt(scale) * zmax
    tol_g = max(1e-9, 16 * EPS * condK * condS * condS) * np.sqrt(scale) * zmax * max(1.0, float(np.max(np.abs(gr))))
    assert np.max(np.abs(v - vr)) <= tol_v, (np.max(np.abs(v - vr)), tol_v, condK, condS)
    assert np.max(np.abs(g - gr)) <= tol_g, (np.max(np.abs(g - gr)), tol_g, condK, condS)


def test_bitwise_contract(abo, orc):
    gp, _, _, rng = model(abo, orc, "se", n=300, d=4, seed=3)
    h = gp.gpx
    q, B, S, seed = 3, 5000, 64, 5
    Xb = rng.random((B, q, 4))
    pr = [0.0, float(np.quantile(abo.posterior_mean(gp, Xb.reshape(-1, 4)), 0.2))]
    v, g, tau = h.acq_qei(pr, q, Xb, S, seed, want_grad=True)
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(g)) and np.mean(v > 0) > 0.3
    # 682 batches (2046 points) per chunk: these straddle chunk boundaries of the full call
    for b in (0, 681, 682, 683, 1364, 2500, 4999):
        vb, gb, tb = h.acq_qei(pr, q, Xb[b:b + 1], S, seed, want_grad=True)
        assert vb[0] == v[b] and np.array_equal(gb[0], g[b]) and tb[0] == tau[b], b
    sub = rng.permutation(B)[:900]
    vs, gs, ts = h.acq_qei(pr, q, Xb[sub], S, seed, want_grad=True)
    assert np.array_equal(vs, v[sub]) and np.array_equal(gs, g[sub]) and np.array_equal(ts, tau[sub])
    vn, gn, tn = h.acq_qei(pr, q, Xb, S, seed)
    assert gn is None and np.array_equal(vn, v) and np.array_equal(tn, tau)
    again = h.acq_qei(pr, q, Xb, S, seed, want_grad=True)
    assert np.array_equal(again[0], v) and np.array_equal(again[1], g) and np.array_equal(again[2], tau)
    assert not np.array_equal(h.acq_qei(pr, q, Xb[:50], S, seed + 1)[0], v[:50])


def test_q1_against_analytic_ei(abo, orc):
    gp, post, scale, rng = model(abo, orc, "matern52", n=200, d=3, seed=4)
    Xc = rng.random((20, 3))
    mu, var = orc.posterior_mean_var(post, Xc)
    best, xi, S = float(np.max(mu)) + 0.1, 0.01, 4096
    v, _, tau = gp.gpx.acq_qei([xi, best], 1, Xc[:, None, :], S, 9)
    ei, _, _ = gp.gpx.acq_eval(0, [xi, best], Xc)
    _, _, _, imp = qref.qei(post, Xc[:, None, :], xi, best, S, 9, want_grad=False, tau=tau)
    se = imp.std(axis=1) / np.sqrt(S)
    assert np.all(np.abs(v - ei) <= 5 * se), (v, ei, se)


def test_jitter_ladder_and_neighbours(abo):
    rng = np.random.default_rng(6)
    X, y = data(rng, 20, 2)
    gp = abo.update(abo.StandardGP(2.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.3), 1e-6), X, y)
    q, jitter = 8, 1e-20
    Xb = rng.random((5, q, 2))
    Xb[2] = np.array([3.0, -2.0])                                      # one point, eight times, far from the data
    v, g, tau = gp.gpx.acq_qei([0.0, float(y.min())], q, Xb, 128, 1, jitter=jitter, want_grad=True)
    ladder = [jitter * 2.0 * 10.0 ** k for k in range(7)]
    assert tau[2] in ladder[1:], tau
    assert np.isfinite(v[2]) and np.all(np.isfinite(g[2]))
    assert all(tau[b] == ladder[0] for b in (0, 1, 3, 4)), tau


def test_no_improvement_is_exactly_zero(abo, orc):
    gp, post, scale, rng = model(abo, orc, "se", n=100, d=3, seed=7)
    Xb = rng.random((6, 4, 3))
    mu, var = orc.posterior_mean_var(post, Xb.reshape(-1, 3))
    best = float(np.min(mu)) - 200 * np.sqrt(scale)
    v, g, _ = gp.gpx.acq_qei([0.0, best], 4, Xb, 512, 2, want_grad=True)
    assert np.all(v == 0.0) and np.all(g == 0.0)


def test_posterior_untouched(abo, orc):
    gp, _, _, rng = model(abo, orc, "matern52", n=400, d=3, seed=8)
    h = gp.gpx
    a0, L0, Li0 = h.alpha(), h.factor(0), h.factor(1)
    Xb = rng.random((300, 5, 3))
    h.acq_qei([0.0, 0.0], 5, Xb, 256, 1, want_grad=True)
    h.acq_qei([0.0, 0.0], 5, Xb, 256, 1)
    assert np.array_equal(h.alpha(), a0) and np.array_equal(h.factor(0), L0) and np.array_equal(h.factor(1), Li0)


def test_errors(abo):
    from abo_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(13)
    X, y = data(rng, 50, 2)
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 1e-4), X, y)
    h = gp.gpx
    Xb = rng.random((40 * 33 * 2,))
    pr = _lib.f64([0.0, 0.5])
    out = np.empty(64); gr = np.empty(40 * 33 * 2); tau = np.empty(64)

    def call(handle, q=2, B=4, S=16, jitter=1e-10, params=True, xb=True, values=True):
        return L.abo_acq_qei(handle, _lib.ptr(pr) if params else None, q, _lib.ptr(Xb) if xb else None, B, S, 1, jitter,
                             _lib.ptr(out) if values else None, _lib.ptr(gr), _lib.ptr(tau))

    assert call(h._h) == _lib.ABO_OK
    for kw in (dict(q=0), dict(q=33), dict(S=0), dict(S=4097), dict(jitter=0.0), dict(jitter=-1.0),
               dict(jitter=float("nan")), dict(jitter=float("inf")), dict(params=False), dict(xb=False), dict(values=False)):
        assert call(h._h, **kw) == _lib.ABO_ERR_INVALID, kw
    assert L.abo_acq_qei(None, _lib.ptr(pr), 2, _lib.ptr(Xb), 4, 16, 1, 1e-10, _lib.ptr(out), None, None) == _lib.ABO_ERR_INVALID
    unfit = _lib.GpHandle(gp.ctx, 0, 2, 1)
    assert call(unfit._h) == _lib.ABO_ERR_NOT_FITTED
    wide = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 1e-4), rng.random((10, 33)), rng.random(10))
    assert call(wide.gpx._h) == _lib.ABO_ERR_INVALID
    out[:] = -7.0
    assert call(h._h, B=0) == _lib.ABO_OK and call(h._h, B=-3) == _lib.ABO_OK and np.all(out == -7.0)
    assert np.all(np.isfinite(h.acq_qei([0.0, 0.5], 2, Xb[:8].reshape(2, 2, 2), 16, 1)[0]))


def test_refined_batch_scores_at_least_the_best_raw(abo):
    rng = np.random.default_rng(2)
    X = rng.random((60, 2)) * 12 - 6
    f = lambda x: (x[:, 0] ** 2 + x[:, 1] - 11) ** 2 + (x[:, 0] + x[:, 1] ** 2 - 7) ** 2
    y = f(X); y = (y - y.mean()) / y.std()
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 2.0), 1e-6), X, y)
    dom = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    acq = abo.qExpectedImprovement(0.0, float(y.min()), 4, num_samples=256, seed=3)
    raw = abo.optimize_acquisition(acq, gp, dom, n_grid=2000, n_local=20, rng=np.random.default_rng(0), refine=False)
    ref = abo.optimize_acquisition(acq, gp, dom, n_grid=2000, n_local=20, rng=np.random.default_rng(0))
    assert raw.shape == ref.shape == (4, 2)
    assert np.all(ref >= dom.lower) and np.all(ref <= dom.upper)
    vr, vf = acq(gp, raw[None])[0], acq(gp, ref[None])[0]
    assert vf >= vr > 0, (vr, vf)
    v, g = acq.value_and_grad(gp, ref)
    assert v.shape == (1,) and g.shape == (1, 4, 2) and v[0] == vf


def test_bo_loop_with_batches(abo):
    f = lambda x: (x[0] ** 2 + x[1] - 11) ** 2 + (x[0] + x[1] ** 2 - 7) ** 2
    domain = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    rng = np.random.default_rng(0)
    xs = [domain.lower + (domain.upper - domain.lower) * rng.random(2) for _ in range(5)]
    ys = [f(x) for x in xs]
    model = abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0), 1e-9)
    bo = abo.BOStruct(f, abo.qExpectedImprovement(0.0, min(ys), 4), model, domain, xs, ys, 5, 0.0)
    bo, acq_values, _ = abo.optimize(bo, standardize="mean_only", hyper_params="all", num_restarts_HP=4, rng=rng)
    assert not bo.flag
    assert len(acq_values) == 5 and all(np.isfinite(acq_values))
    assert len(bo.xs) == 5 + 20 and len(bo.ys_non_std) == 5 + 20
    new = np.array(bo.xs[5:])
    assert np.all(new >= domain.lower) and np.all(new <= domain.upper)
    assert min(np.ravel(bo.ys_non_std)) < min(ys)
