"""Max-value entropy search on the device (ABO_ACQ_MES): the scores against the NumPy reference at the GPU's own
posterior on the fused, three-kernel and host-piece paths, end to end against the oracle posterior, the analytic
gradient, the top-k orders, the y* draws, no side effects on the handle, argument errors, the BO loop, and the sharded
top-k."""
import os
import subprocess
import socket
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mes_reference as mref  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
KNAME = {0: "SqExponentialKernel", 1: "Matern52Kernel", 2: "Matern72Kernel", 3: "ApproxMatern52Kernel"}


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


def standard(abo, rng, kind, n, d, ell=0.7, noise=1e-4, mean=0.2, scale=1.3):
    X, y = data(rng, n, d)
    return abo.update(abo.StandardGP(scale * abo.with_lengthscale(abo.Kernel(KNAME[kind]), ell), noise, mean=mean), X, y), X, y


def ystar(rng, mu, K=16, var=None):
    """y* spread from well below the smallest mean to its middle: gamma from O(1) to the left tail.  Given the variances,
    within a few typical standard deviations of the smallest mean instead, so that most gamma stay inside [-40, 40]."""
    lo, mid = float(np.min(mu)), float(np.median(mu))
    if var is None:
        return rng.uniform(lo - 1.0, mid, K)
    s = float(np.median(np.sqrt(np.maximum(var, 0.0))))
    return lo + s * rng.uniform(-4.0, 2.0, K)


def params(ys):
    return np.concatenate([[float(len(ys))], ys])


def assert_formula(scores, mu, var, ys):
    """1e-12 relative where every |gamma_k| <= 40 (the accuracy range of the header); finite and non-negative beyond,
    where the error of h grows like eps gamma^2 (points close to the data, where sigma is small)."""
    ref = mref.mes(mu, var, ys)
    g = (mu[:, None] - np.asarray(ys)[None, :]) / np.sqrt(np.maximum(var, 1e-300))[:, None]
    inside = (var <= 1e-12) | np.all(np.abs(g) <= 40.0, axis=1)
    assert inside.sum() >= min(20, inside.size // 10), inside.sum()
    err = np.abs(scores - ref)
    assert np.all(err[inside] <= 1e-12 * np.abs(ref[inside]) + 1e-300), np.max(err[inside] / (np.abs(ref[inside]) + 1e-300))
    assert np.all(np.isfinite(scores)) and np.all(scores >= 0.0)


# ---- 1. the formula at the GPU's own posterior --------------------------------------------------------------------
@pytest.mark.parametrize("case", ["se", "matern52", "matern72", "ard"])
def test_fused_path_formula(abo, case):
    rng = np.random.default_rng({"se": 1, "matern52": 2, "matern72": 3, "ard": 4}[case])
    kind = {"se": 0, "matern52": 1, "matern72": 2, "ard": 1}[case]
    ell = np.array([0.4, 0.9, 1.5, 0.6, 2.0, 0.8]) if case == "ard" else 0.7
    gp, _, _ = standard(abo, rng, kind, 500, 6, ell=ell)
    Xc = rng.random((20_000, 6)) * 1.2 - 0.1
    h = gp.gpx
    mu, var = h.posterior(Xc)
    ys = ystar(rng, mu, var=var)
    scores = h.acq_eval(4, params(ys), Xc)[0]
    assert_formula(scores, mu, var, ys)
    # one y* (K = 1) and the most (K = 256) are accepted
    for K in (1, 256):
        ysk = ystar(rng, mu, K, var=var)
        assert_formula(h.acq_eval(4, params(ysk), Xc[:3000])[0], mu[:3000], var[:3000], ysk)


def test_three_kernel_path_formula_standard_d40(abo):
    rng = np.random.default_rng(5)
    gp, _, _ = standard(abo, rng, 0, 300, 40, ell=3.0)
    Xc = rng.random((5000, 40))
    h = gp.gpx
    mu, var = h.posterior(Xc)
    ys = ystar(rng, mu, var=var)
    assert_formula(h.acq_eval(4, params(ys), Xc)[0], mu, var, ys)


def test_three_kernel_path_formula_gradient_gp(abo):
    rng = np.random.default_rng(6)
    X, Y = data(rng, 80, 3, gradient=True)
    gp = abo.update(abo.GradientGP(1.1 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.6), 4, 1e-5), X, Y)
    Xc = 0.5 + 2.0 * rng.random((6000, 3))            # half outside the data's box: sigma from small to the prior's
    h = gp.gpx
    mu, var = h.posterior(Xc, 1)
    ys = ystar(rng, mu, var=var)
    assert_formula(h.acq_eval(4, params(ys), Xc)[0], mu, var, ys)


def test_host_piece_path_formula(abo):
    rng = np.random.default_rng(7)
    gp, _, _ = standard(abo, rng, 1, 200, 4)
    Xc = rng.random((300_000, 4))                        # above the 262 144-candidate host piece
    h = gp.gpx
    mu, var = h.posterior(Xc)
    ys = ystar(rng, mu, var=var)
    s, ti, tv = h.acq_eval(4, params(ys), Xc, k=20)
    assert_formula(s, mu, var, ys)
    order = np.lexsort((np.arange(len(s)), -s))[:20]
    assert np.array_equal(ti, order) and np.array_equal(tv, s[order])


def test_no_uncertainty_gives_zero(abo):
    rng = np.random.default_rng(8)
    X = rng.random((40, 2))
    y = np.sin(4 * X[:, 0]) + X[:, 1]
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 0.5), 1e-14), X, y)
    h = gp.gpx
    Xc = np.concatenate([X, rng.random((200, 2))])
    mu, var = h.posterior(Xc)
    tiny = var <= 1e-12
    assert tiny.any(), "no candidate with var <= 1e-12"
    ys = ystar(rng, mu, var=var)
    s = h.acq_eval(4, params(ys), Xc)[0]
    assert np.all(s[tiny] == 0.0)
    assert_formula(s, mu, var, ys)


# ---- 2. end to end against the oracle posterior --------------------------------------------------------------------
@pytest.mark.parametrize("kind", [0, 1])
def test_against_oracle_posterior(abo, orc, kind):
    rng = np.random.default_rng(10 + kind)
    n, d, ell, scale, noise, mean = 500, 6, 0.7, 1.3, 1e-4, 0.2
    gp, X, y = standard(abo, rng, kind, n, d, ell=ell, noise=noise, mean=mean, scale=scale)
    post = orc.fit_standard(X, y, kind, 1.0 / ell, scale, noise, mean)
    Xc = rng.random((4000, d)) * 1.2 - 0.1
    mu, var = gp.gpx.posterior(Xc)
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    ys = ystar(rng, mu)
    s = gp.gpx.acq_eval(4, params(ys), Xc)[0]
    ref_o = mref.mes(mu_o, var_o, ys)
    dmu1, dvar1 = mref.mes_dmu_dvar(mu, var, ys)
    dmu2, dvar2 = mref.mes_dmu_dvar(mu_o, var_o, ys)
    bound = (np.maximum(np.abs(dmu1), np.abs(dmu2)) * np.abs(mu - mu_o) + np.maximum(np.abs(dvar1), np.abs(dvar2)) * np.abs(var - var_o)
             + 1e-12 * np.abs(ref_o) + 1e-300)
    assert np.all(np.abs(s - ref_o) <= bound), np.max(np.abs(s - ref_o) / bound)


# ---- 3. gradient ---------------------------------------------------------------------------------------------------
def fd_check(orc, post, ys, Xq, grad):
    hstep = 1e-6
    for b in range(Xq.shape[1]):
        Xp = Xq.copy(); Xp[:, b] += hstep; Xm = Xq.copy(); Xm[:, b] -= hstep
        fd = (mref.mes(*orc.posterior_mean_var(post, Xp), ys) - mref.mes(*orc.posterior_mean_var(post, Xm), ys)) / (2 * hstep)
        sc = max(np.max(np.abs(fd)), 1e-12)
        assert np.all(np.abs(grad[:, b] - fd) <= 2e-5 * sc + 1e-7 * np.abs(fd)), (b, np.max(np.abs(grad[:, b] - fd)), sc)


@pytest.mark.parametrize("kind", [0, 2])
def test_gradient_standard_gp(abo, orc, kind):
    rng = np.random.default_rng(20 + kind)
    n, d, ell, scale, noise = 120, 4, 0.6, 1.2, 1e-3
    X = rng.random((n, d)); y = np.sin(3 * X).sum(1) / d + 0.05 * rng.standard_normal(n); y = (y - y.mean()) / y.std(ddof=1)
    gp = abo.update(abo.StandardGP(scale * abo.with_lengthscale(abo.Kernel(KNAME[kind]), ell), noise), X, y)
    post = orc.fit_standard(X, y, kind, 1.0 / ell, scale, noise)
    Xq = rng.random((37, d))
    mu, _ = gp.gpx.posterior(Xq)
    ys = ystar(rng, mu)
    val, grad = gp.gpx.acq_eval_grad(4, params(ys), Xq)
    s = gp.gpx.acq_eval(4, params(ys), Xq)[0]
    # the gradient pass accumulates mu and var in another order than the sweep: the same to 1e-12 of the largest score
    assert np.all(np.abs(val - s) <= 1e-12 * np.max(np.abs(s))), np.max(np.abs(val - s)) / np.max(np.abs(s))
    fd_check(orc, post, ys, Xq, grad)


def test_gradient_gradient_gp(abo, orc):
    rng = np.random.default_rng(3)
    n, d = 30, 3
    X = -2 + 4 * rng.random((n, d)); Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    gp = abo.update(abo.GradientGP(abo.with_lengthscale(abo.Kernel(KNAME[3]), 1.5), d + 1, 1e-4), X, Y)
    post = orc.fit_gradient(X, Y, 3, 1 / 1.5, 1.0, 1e-4)
    Xq = -2 + 4 * rng.random((20, d))
    mu, _ = gp.gpx.posterior(Xq, 1)
    ys = ystar(rng, mu)
    val, grad = gp.gpx.acq_eval_grad(4, params(ys), Xq)
    s = gp.gpx.acq_eval(4, params(ys), Xq)[0]
    # the gradient pass accumulates mu and var in another order than the sweep: the same to 1e-12 of the largest score
    assert np.all(np.abs(val - s) <= 1e-12 * np.max(np.abs(s))), np.max(np.abs(val - s)) / np.max(np.abs(s))
    fd_check(orc, post, ys, Xq, grad)


# ---- 4. top-k ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [20_000, 100_000])
def test_topk_orders_and_device_entry(abo, m):
    import torch
    rng = np.random.default_rng(30)
    gp, _, _ = standard(abo, rng, 0, 300, 5)
    h = gp.gpx
    Xc = rng.random((m, 5))
    ys = ystar(rng, h.posterior(Xc[:2000])[0])
    s, ti, tv = h.acq_eval(4, params(ys), Xc, k=64)
    order = np.lexsort((np.arange(m), -s))[:64]
    assert np.array_equal(ti, order) and np.array_equal(tv, s[order])
    d_x = torch.from_numpy(Xc).cuda(); d_s = torch.empty(m, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ti2, tv2 = h.acq_eval_dev(4, params(ys), d_x.data_ptr(), m, d_s.data_ptr(), k=64)
    torch.cuda.synchronize()
    assert np.array_equal(d_s.cpu().numpy(), s)
    assert np.array_equal(ti2, ti) and np.array_equal(tv2, tv)


# ---- 5. y* sampling ------------------------------------------------------------------------------------------------
def test_max_value_samples(abo):
    rng = np.random.default_rng(40)
    gp, _, y = standard(abo, rng, 0, 200, 3)
    Xc = rng.random((50_000, 3))
    best = float(np.min(y)) + 0.3
    ys = abo.max_value_samples(gp, Xc, 16, seed=5, num_features=1024, best_y=best)
    _, _, av = gp.gpx.pathwise_sample(Xc, 16, 5, 1024, want_samples=False)
    assert np.array_equal(ys, np.minimum(av, best))
    assert np.array_equal(abo.max_value_samples(gp, Xc, 16, seed=5, num_features=1024), av)
    assert np.array_equal(abo.max_value_samples(gp, Xc, 5, seed=5, num_features=1024, best_y=best), ys[:5])
    from abo_b200.acquisition import nan_min_reduce
    halves = [abo.max_value_samples(gp, Xc[:20_000], 16, seed=5, num_features=1024),
              abo.max_value_samples(gp, Xc[20_000:], 16, seed=5, num_features=1024)]
    assert np.array_equal(np.minimum(nan_min_reduce(halves), best), ys)
    a = abo.MaxValueEntropySearch(5, best, 16, 1024)
    s, ti, _ = a.topk(gp, Xc, 10)
    assert np.array_equal(s, gp.gpx.acq_eval(4, params(ys), Xc)[0])
    assert np.array_equal(a(gp, Xc[ti]), s[ti])                                 # the grid's y* are reused
    b = abo.MaxValueEntropySearch(5, best, 16, 1024)                              # without a topk: y* over the points given
    assert np.array_equal(b(gp, Xc[:100]), gp.gpx.acq_eval(4, params(abo.max_value_samples(
        gp, Xc[:100], 16, seed=5, num_features=1024, best_y=best)), Xc[:100])[0])
    gp2 = abo.update(gp, np.vstack([gp._data[0], [[0.5, 0.5, 0.5]]]), np.append(gp._data[1], 0.0))
    assert a._cache["token"] != gp2.gpx.token                                   # a new posterior draws afresh


# ---- 6. no side effects --------------------------------------------------------------------------------------------
def test_no_side_effects(abo):
    rng = np.random.default_rng(50)
    gp, _, y = standard(abo, rng, 1, 300, 4)
    h = gp.gpx
    Xc = rng.random((30_000, 4))

    def snapshot():
        return ([h.acq_eval(a, p, Xc)[0] for a, p in ((0, [0.01, float(y.min())]), (1, [0.01, float(y.min())]), (2, [2.0]))],
                h.alpha(), h.factor(0), h.factor(1))
    before = snapshot()
    ys = abo.max_value_samples(gp, Xc, 16, seed=1, best_y=float(y.min()))
    h.acq_eval(4, params(ys), Xc, k=10)
    h.acq_eval_grad(4, params(ys), Xc[:500])
    abo.MaxValueEntropySearch(1, float(y.min())).topk(gp, Xc, 5)
    after = snapshot()
    for a, b in zip(before[0], after[0]):
        assert np.array_equal(a, b)
    for a, b in zip(before[1:], after[1:]):
        assert np.array_equal(a, b)


# ---- 7. argument errors --------------------------------------------------------------------------------------------
def test_argument_errors(abo):
    import ctypes as C
    from abo_b200._lib import lib, ptr
    rng = np.random.default_rng(60)
    gp, _, _ = standard(abo, rng, 0, 50, 2)
    h = gp.gpx
    Xc = np.ascontiguousarray(rng.random((10, 2)))
    scores = np.empty(10); grad = np.empty((10, 2))
    bad = [np.array([0.0, 0.1]), np.concatenate([[257.0], np.zeros(257)]), np.array([2.5, 0.1, 0.2, 0.3]),
           np.array([2.0, 0.1, np.nan]), np.array([1.0, np.inf])]
    for p in bad:
        p = np.ascontiguousarray(p)
        assert lib().abo_acq_eval(h._h, 4, ptr(p), ptr(Xc), 10, ptr(scores), 0, None, None) == 1
        assert lib().abo_acq_eval_grad(h._h, 4, ptr(p), ptr(Xc), 10, ptr(scores), ptr(grad), None, None) == 1
    ok = np.ascontiguousarray(np.array([2.0, 0.1, 0.2]))
    assert lib().abo_acq_eval(h._h, 4, ptr(ok), ptr(Xc), 10, ptr(scores), 0, None, None) == 0
    ids = np.array([4], dtype=np.int32); w = np.array([1.0]); pr = np.array([1.0, 0.0])
    assert lib().abo_acq_eval_multi(h._h, 1, ptr(ids), ptr(w), ptr(pr), ptr(Xc), 10, ptr(scores), 0, None, None) == 1
    with pytest.raises(ValueError):
        h.acq_eval(4, [0.0, 1.0], Xc)


# ---- 8. the BO loop ------------------------------------------------------------------------------------------------
def himmelblau(x):
    return (x[0] ** 2 + x[1] - 11) ** 2 + (x[0] + x[1] ** 2 - 7) ** 2


def himmelblau_grad(x):
    a, b = x[0] ** 2 + x[1] - 11, x[0] + x[1] ** 2 - 7
    return np.array([himmelblau(x), 4 * a * x[0] + 2 * b, 2 * a + 4 * b * x[1]])


@pytest.mark.parametrize("case", ["standard", "gradient", "ensemble"])
def test_bo_loop(abo, case):
    domain = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    rng = np.random.default_rng(0)
    xs = [domain.lower + (domain.upper - domain.lower) * rng.random(2) for _ in range(5)]
    if case == "gradient":
        f = himmelblau_grad
        ys = [f(x) for x in xs]
        model = abo.GradientGP(abo.with_lengthscale(abo.SqExponentialKernel(), 1.0), 3, 1e-6)
        best0 = min(float(v[0]) for v in ys)
        acq = abo.MaxValueEntropySearch(0, best0)
    else:
        f = himmelblau
        ys = [f(x) for x in xs]
        model = abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 1.0), 1e-9)
        best0 = min(ys)
        acq = abo.MaxValueEntropySearch(0, best0)
        if case == "ensemble":
            acq = abo.EnsembleAcquisition([0.5, 0.5], [acq, abo.ExpectedImprovement(0.0, best0)])
    bo = abo.BOStruct(f, acq, model, domain, xs, ys, 15, 0.0)
    bo, acq_values, _ = abo.optimize(bo, standardize="mean_only", hyper_params="all", num_restarts_HP=4, n_grid=200_000,
                                     rng=rng, refine=True)
    assert not bo.flag
    assert len(acq_values) == 15
    assert all(np.isfinite(v) and v >= 0.0 for v in acq_values), acq_values
    X = np.array(bo.xs[5:])
    assert np.all(X >= domain.lower) and np.all(X <= domain.upper)
    final = min(float(np.ravel(v)[0]) for v in bo.ys_non_std)
    assert final < best0, (final, best0)


# ---- 9. sharded top-k ----------------------------------------------------------------------------------------------
def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.skipif(_ngpu() < 2, reason="needs >= 2 GPUs")
def test_sharded_topk_two_ranks():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0)); port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tools", "mes_sharded_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=420)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "mes_sharded_check ok" in r.stdout
