"""GPU parity tests: the CUDA path (through the C ABI, via the host mirror of the reference
API) against the CPU oracle on the same seeded inputs.  Tolerance (BASELINE.json north_star):
posterior mean / variance within 1e-9 relative, applied as |a - b| <= 1e-9 * max(|b|, sigma_f); where two valid
FP64 evaluations legitimately differ by more (cond(K) * eps, SURVEY H3) the 80-bit arbiter decides:
err_gpu <= max(1e-9 * scale, 4 * err_oracle) against oracle.ld_posterior_truth at full problem size (h3_parity).
Acquisition values: the formula is exact on the GPU's own posterior and the arg-max / top-k are identical on the
same candidate set; tests/test_parity_report.py records the achieved errors of C1-C5."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-9


@pytest.fixture(scope="module")
def abo():
    import abo_b200
    return abo_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import abo_oracle
    return abo_oracle


KNAME = {0: "SqExponentialKernel", 1: "Matern52Kernel", 2: "Matern72Kernel", 3: "ApproxMatern52Kernel",
         4: "ApproxMatern72Kernel", 5: "ADMatern52Kernel", 6: "ADMatern72Kernel"}


def make_kernel(abo, kind, inv_ls, scale):
    return scale * abo.with_lengthscale(abo.Kernel(KNAME[kind]), 1.0 / inv_ls)


def close(a, b, scale, tol=RTOL):
    a = np.asarray(a); b = np.asarray(b)
    return np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), scale))


def h3_parity(orc, post, Xc, outputs, gpu_mean, gpu_var, ora_mean, ora_var, scale_mean, scale_var, nsample=24, seed=0):
    """The contract's tolerance (north_star: 1e-9) with SURVEY H3's arbiter where FP64 legitimately diverges:
    pass if |gpu - oracle| <= 1e-9 * max(|oracle|, scale) everywhere; otherwise the points where the two differ most
    (plus a random sample) are judged against the 80-bit truth at full problem size (oracle.ld_posterior_truth) and the
    GPU's largest error may not exceed max(1e-9 * scale, 4 x the oracle's largest error).  Returns a short record of
    what decided, for the assertion message."""
    rec = {}
    outputs = list(outputs)
    m = len(np.atleast_2d(Xc))
    for name, g, o, sc in (("mean", gpu_mean, ora_mean, scale_mean), ("var", gpu_var, ora_var, scale_var)):
        g = np.asarray(g, dtype=np.float64).ravel(); o = np.asarray(o, dtype=np.float64).ravel()
        assert g.shape == o.shape == (m * len(outputs),)
        dev = np.abs(g - o) / np.maximum(np.abs(o), sc)
        if np.all(dev <= RTOL):
            rec[name] = ("strict", float(dev.max()))
            continue
        # candidates (columns of the out-major layout) holding the largest deviations + a random sample
        worst = np.unique(np.argsort(dev)[-nsample:] % m)
        rnd = np.random.default_rng(seed).integers(0, m, nsample)
        pick = np.unique(np.concatenate([worst, rnd]))
        mt, vt, resid = orc.ld_posterior_truth(post, np.atleast_2d(Xc)[pick], outputs=outputs)
        assert resid < 1e-15, resid
        truth = (mt if name == "mean" else vt)
        idx = (np.arange(len(outputs))[:, None] * m + pick[None, :]).ravel()          # out-major positions of the picked points
        e_g = float(np.max(np.abs(g[idx] - truth) / np.maximum(np.abs(truth), sc)))
        e_o = float(np.max(np.abs(o[idx] - truth) / np.maximum(np.abs(truth), sc)))
        rec[name] = ("arbiter", e_g, e_o)
        assert e_g <= max(RTOL, 4 * e_o), (name, "gpu", e_g, "oracle", e_o, "max dev", float(dev.max()))
    return rec


# ---- reference known-answer tests through the GPU path (G1, G2-less, G3) ---------------
def test_known_answers_g1_g3(abo):
    gp = abo.StandardGP(abo.SqExponentialKernel(), 0.1)
    gp1 = abo.update(gp, [0.0, 0.5, 1.0], [0.0, 0.25, 1.0])          # test_surrogates.jl:59-105
    assert abs(abo.posterior_mean(gp1, [0.25])[0] - 0.1771247751991296) < 1e-10
    assert abs(abo.posterior_var(gp1, [0.25])[0] - 0.050320225208722924) < 1e-10
    gp3 = abo.update(gp, [0.0, 0.5, 1.0], [2.0, 1.0, 0.5])           # test_acquisition.jl:20-43
    ei = abo.ExpectedImprovement(0.01, 0.5)(gp3, [0.25])[0]
    pi = abo.ProbabilityImprovement(0.01, 0.5)(gp3, [0.25])[0]
    ucb = abo.UpperConfidenceBound(2.0)(gp3, [0.25])[0]
    assert abs(ei - 3.11345832411526e-07) < 1e-9 * 3.2e-7 and ei >= 0
    assert abs(pi - 6.608138679027337e-06) < 1e-9 * 6.7e-6 and 0 <= pi <= 1
    assert abs(ucb - (-1.0186125700256665)) < 1e-10
    mu = abo.posterior_mean(gp3, [0.25])[0]; var = abo.posterior_var(gp3, [0.25])[0]
    assert abs(ucb - (-mu + 2.0 * math.sqrt(var))) < 1e-10            # test_bayesian_opt.jl:552-558


@pytest.mark.parametrize("kind", [0, 1, 2, 3, 5])
@pytest.mark.parametrize("n,d,m", [(3, 1, 7), (50, 2, 1000), (130, 6, 1500), (300, 20, 999), (1000, 6, 4096),
                                   (257, 40, 300)])
def test_posterior_parity(abo, orc, kind, n, d, m):
    rng = np.random.default_rng(100 * n + d)
    X = rng.random((n, d)); y = np.sin(3 * X).sum(1) + 0.1 * rng.standard_normal(n)
    Xc = rng.random((m, d))
    inv_ls, scale, noise, mean_c = 1.0 / (0.4 * math.sqrt(d)), 1.7, 1e-3, 0.3
    gp = abo.update(abo.StandardGP(make_kernel(abo, kind, inv_ls, scale), noise, mean=mean_c), X, y)
    post = orc.fit_standard(X, y, kind, inv_ls, scale, noise, mean_c)
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    mu = abo.posterior_mean(gp, Xc); var = abo.posterior_var(gp, Xc)
    # 1e-9 of the contract, or the 80-bit arbiter where two valid FP64 evaluations differ by more (SURVEY H3)
    h3_parity(orc, post, Xc, (0,), mu, var, mu_o, var_o, scale, scale)
    # alpha = K^-1 delta is not an output of the reference's API (the mean above is); its own FP64 floor is cond(K) * eps
    cond = np.linalg.cond(post.U) ** 2
    a = gp.gpx.alpha()
    assert close(a, post.alpha, np.max(np.abs(post.alpha)), max(1e-8, 100 * cond * 2.2e-16))


@pytest.mark.parametrize("n", [1, 2, 7, 15, 16, 17, 31, 33, 127, 128, 129, 255, 256, 257, 383, 385])
def test_fused_sweep_ragged_shapes(abo, orc, n):
    """Edge shapes of the fused sweep: n around the k16 / fragment / 128-tile boundaries, candidate counts around the
    128-candidate tile and the one-tile-per-SM boundary, every acquisition; mean, variance and scores against the oracle
    at 1e-9, the device result independent of how the candidate set is cut."""
    rng = np.random.default_rng(1000 + n)
    d = 1 + n % 5
    X = rng.random((n, d)); y = np.cos(2 * X).sum(1) + 0.05 * rng.standard_normal(n)
    kind = [0, 1, 2, 3, 4][n % 5]
    inv_ls, scale, noise = 1.0 / 0.6, 1.3, 1e-3
    gp = abo.update(abo.StandardGP(make_kernel(abo, kind, inv_ls, scale), noise), X, y)
    post = orc.fit_standard(X, y, kind, inv_ls, scale, noise)
    for m in (1, 127, 128, 129, 148 * 128 + 1):
        Xc = rng.random((m, d))
        mu_o, var_o = orc.posterior_mean_var(post, Xc)
        mu = abo.posterior_mean(gp, Xc); var = abo.posterior_var(gp, Xc)
        h3_parity(orc, post, Xc, (0,), mu, var, mu_o, var_o, scale, scale)
        for acq_id, acq in ((0, abo.ExpectedImprovement(0.01, float(y.min()))), (1, abo.ProbabilityImprovement(0.01, float(y.min()))),
                            (2, abo.UpperConfidenceBound(2.0))):
            s_all = acq(gp, Xc)
            assert s_all.shape == (m,) and np.all(np.isfinite(s_all))
            assert close(s_all, orc.acquisition(acq_id, acq.params(), mu, var), 1.0, 1e-12)
            if m > 1:
                cut = m // 3 + 1
                assert np.array_equal(np.concatenate([acq(gp, Xc[:cut]), acq(gp, Xc[cut:])]), s_all)


def test_factor_matches_lapack(abo, orc):
    rng = np.random.default_rng(5)
    X = rng.random((300, 4)); y = rng.standard_normal(300)
    gp = abo.update(abo.StandardGP(make_kernel(abo, 0, 2.0, 1.0), 1e-2), X, y)
    post = orc.fit_standard(X, y, 0, 2.0, 1.0, 1e-2)
    L = gp.gpx.factor(0); Linv = gp.gpx.factor(1)
    assert np.max(np.abs(L - post.U.T)) < 1e-11
    assert np.max(np.abs(Linv @ post.U.T - np.eye(300))) < 1e-9


@pytest.mark.parametrize("acq_name,params", [("EI", (0.01, None)), ("PI", (0.01, None)), ("UCB", (2.0,))])
@pytest.mark.parametrize("cfg,kw", [("C1", dict(n=10, m=10_000)), ("C1", dict(n=61, m=10_000)),
                                    ("C2", dict(n=512, m=20_000)), ("C4", dict(n=700, m=5_000, d=20))])
def test_acquisition_parity_and_topk(abo, orc, acq_name, params, cfg, kw):
    c = orc.make_config(cfg, **kw)
    gp = abo.update(abo.StandardGP(make_kernel(abo, c["kind"], c["inv_ls"], c["scale"]), c["noise"]), c["X"], c["y"])
    post = orc.fit_standard(c["X"], c["y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    mu_o, var_o = orc.posterior_mean_var(post, c["Xc"])
    best = float(c["y"].min())
    if acq_name == "EI":
        acq = abo.ExpectedImprovement(params[0], best); ref = orc.expected_improvement(mu_o, var_o, params[0], best)
    elif acq_name == "PI":
        acq = abo.ProbabilityImprovement(params[0], best); ref = orc.probability_improvement(mu_o, var_o, params[0], best)
    else:
        acq = abo.UpperConfidenceBound(params[0]); ref = orc.upper_confidence_bound(mu_o, var_o, params[0])
    k = 100
    scores, top_idx, top_val = acq.topk(gp, c["Xc"], k)
    # EI/PI amplify posterior differences by ~ |z|/sigma in the far tail; compare on the
    # posterior-consistent scale: the acquisition evaluated by the ORACLE formula on the GPU's
    # mean/var must match the GPU scores to 1e-12, and scores vs oracle within 1e-9 of the range.
    mu = abo.posterior_mean(gp, c["Xc"]); var = abo.posterior_var(gp, c["Xc"])
    mine = orc.acquisition({"EI": 0, "PI": 1, "UCB": 2}[acq_name], acq.params(), mu, var)
    assert close(scores, mine, np.max(np.abs(mine)), 1e-12)
    assert close(scores, ref, np.max(np.abs(ref)), 1e-9 * 10)
    # top-k: exactly sortperm(scores; rev=true)[1:k] of the GPU's own scores ...
    assert list(top_idx) == list(orc.sortperm_rev(scores, k))
    assert np.array_equal(top_val, scores[top_idx])
    # ... and the same arg-max candidate as the oracle on the same candidate set
    assert int(top_idx[0]) == int(orc.sortperm_rev(ref, 1)[0])


def test_topk_ties_and_nan_order(abo, orc):
    # exact ties: EI is exactly 0 where sigma^2 <= 1e-12 and delta < 0 -> duplicates of candidates
    c = orc.make_config("C1", n=20, m=300)
    Xc = np.vstack([c["Xc"][:50], c["Xc"][:50], c["Xc"][50:]])      # duplicated candidates -> tied scores
    gp = abo.update(abo.StandardGP(make_kernel(abo, 0, c["inv_ls"], 1.0), 1e-6), c["X"], c["y"])
    acq = abo.UpperConfidenceBound(2.0)
    scores, ti, tv = acq.topk(gp, Xc, 40)
    assert list(ti) == list(orc.sortperm_rev(scores, 40))
    assert np.array_equal(scores[:50], scores[50:100])


@pytest.mark.parametrize("m_big,k", [(70_000, 64), (600_000, 100), (300_001, 5000), (66_001, 66_001), (65_537, 1)])
def test_device_selection_ties_nan_and_piece_merge(abo, orc, m_big, k):
    """Above 65 536 candidates the K best are selected on the device (radix select on the order keys) and, above
    262 144, per piece with a merge: same list as sortperm(scores; rev = true)[1:k] with heavy ties (a block of
    300 candidates repeated all over the set, so the threshold key itself is tied across pieces) and NaN scores
    (NaN sorts first, Julia isless)."""
    c = orc.make_config("C1", n=20, m=300)
    gp = abo.update(abo.StandardGP(make_kernel(abo, 0, c["inv_ls"], 1.0), 1e-6), c["X"], c["y"])
    reps = -(-m_big // 300)
    Xc = np.tile(c["Xc"], (reps, 1))[:m_big].copy()
    Xc[[7, 123_45 % m_big, m_big - 3]] = np.nan                   # NaN coordinates -> NaN scores
    for acq in (abo.UpperConfidenceBound(2.0), abo.ExpectedImprovement(0.01, float(np.min(c["y"])))):
        scores, ti, tv = acq.topk(gp, Xc, k)
        assert np.isnan(scores[[7, 123_45 % m_big, m_big - 3]]).all()
        ref = orc.sortperm_rev(scores, k)
        assert list(ti) == list(ref)
        assert np.array_equal(tv, scores[ti], equal_nan=True)
    none, ti3, tv3 = abo.UpperConfidenceBound(2.0).topk(gp, Xc, k, want_scores=False)     # only K pairs cross PCIe
    s_full, ti4, _ = abo.UpperConfidenceBound(2.0).topk(gp, Xc, k)
    assert none is None and list(ti3) == list(ti4) and np.array_equal(tv3, s_full[ti4], equal_nan=True)
    # device-resident candidates through abo_acq_eval_dev (no pieces): same selection
    import torch
    dX = torch.from_numpy(Xc).cuda()
    dS = torch.empty(m_big, dtype=torch.float64, device="cuda")
    acq = abo.UpperConfidenceBound(2.0)
    ti2, tv2 = gp.gpx.acq_eval_dev(acq.acq_id, acq.params(), dX.data_ptr(), m_big, dS.data_ptr(), k)
    torch.cuda.synchronize()
    sc = dS.cpu().numpy()
    assert list(ti2) == list(orc.sortperm_rev(sc, k))


def test_edge_sizes(abo, orc):
    c = orc.make_config("C2", n=200, m=300)
    gp = abo.update(abo.StandardGP(make_kernel(abo, 1, c["inv_ls"], 1.0), c["noise"]), c["X"], c["y"])
    post = orc.fit_standard(c["X"], c["y"], 1, c["inv_ls"], 1.0, c["noise"])
    for m in (1, 2, 127, 128, 129):
        mu_o, var_o = orc.posterior_mean_var(post, c["Xc"][:m])
        assert close(abo.posterior_mean(gp, c["Xc"][:m]), mu_o, 1.0)
        assert close(abo.posterior_var(gp, c["Xc"][:m]), var_o, 1.0)
    acq = abo.ExpectedImprovement(0.0, 0.0)
    s, ti, tv = acq.topk(gp, c["Xc"][:5], 100)          # k > m
    assert len(ti) == 5
    assert acq(gp, np.empty((0, 6))).size == 0


def test_failure_protocol(abo, orc):
    # test/test_bayesian_opt.jl:749-817
    gp = abo.StandardGP(abo.SqExponentialKernel(), 0.0)
    xs = [[-1.0, -1.0], [5.0, -5.0]]; ys = [2.0, 50.0]
    g2 = abo.update(gp, xs, ys)
    with pytest.raises(abo.PosDefException) as ei:
        abo.update(g2, xs + [[-1.0 + 1e-12, -1.0 + 1e-12]], ys + [2.0])
    assert ei.value.info == 3
    assert abs(abo.posterior_mean(g2, [[-1.0, -1.0]])[0] - 2.0) < 1e-8      # previous model untouched
    with pytest.raises(abo.DimensionMismatch):
        abo.posterior_mean(g2, [[0.0, 0.0, 0.0]])                             # query of the wrong dimension
    with pytest.raises(abo.DimensionMismatch):
        abo.update(g2, xs + [[0.0, 0.0, 0.0]], ys + [1.0])                    # ragged xs: a 3-D point among 2-D ones
    g3d = abo.update(g2, [[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]], [1.0, 2.0])  # update() conditions the PRIOR: new data of another
    assert g3d.gpx.d == 3 and g2.gpx.d == 2                               # dimension is a fresh posterior (StandardGP.jl:79-83)
    with pytest.raises(abo.DimensionMismatch):
        abo.update(gp, xs, ys[:1])
    # BOStruct rollback
    f = lambda x: float(np.sum(np.asarray(x) ** 2))
    dom = abo.ContinuousDomain([-2.0, -2.0], [2.0, 2.0])
    bo = abo.BOStruct(f, abo.ExpectedImprovement(0.01, 2.0), g2, dom, xs, ys, 10, 0.0)
    bo = abo.update(bo, [-1.0 + 1e-12, -1.0 + 1e-12], 2.0, 0)
    assert len(bo.xs) == 2 and len(bo.ys) == 2 and bo.iter == 0 and bo.flag
    # test/test_bayesian_opt.jl:788-817: a new point of the wrong dimension -> DimensionMismatch propagates out of update(BO, ...)
    g3 = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 0.1), xs, ys)
    bo2 = abo.BOStruct(f, abo.ExpectedImprovement(0.01, 2.0), g3, dom, xs, ys, 10, 0.0)
    with pytest.raises(abo.DimensionMismatch):
        abo.update(bo2, [0.0], 0.0, 0)


@pytest.mark.parametrize("kind", [0, 3, 5, 4])
@pytest.mark.parametrize("n,d", [(3, 2), (20, 3), (40, 10)])
def test_gradient_gp_parity(abo, orc, kind, n, d):
    rng = np.random.default_rng(n * 10 + d)
    X = -2 + 4 * rng.random((n, d))
    Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    Xc = -2 + 4 * rng.random((500, d))
    inv_ls, scale, noise = 1.0 / 1.5, 1.3, 1e-4
    gp = abo.update(abo.GradientGP(make_kernel(abo, kind, inv_ls, scale), d + 1, noise), X, Y)
    post = orc.fit_gradient(X, Y, kind, inv_ls, scale, noise)
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    sc = max(scale, np.max(np.abs(mu_o)))
    h3_parity(orc, post, Xc, (0,), abo.posterior_mean(gp, Xc), abo.posterior_var(gp, Xc), mu_o, var_o, sc, scale)
    gm_o, gv_o = orc.posterior_mean_var(post, Xc[:50], outputs=range(d + 1))
    h3_parity(orc, post, Xc[:50], range(d + 1), abo.posterior_grad_mean(gp, Xc[:50]), abo.posterior_grad_var(gp, Xc[:50]),
              gm_o, gv_o, max(sc, np.max(np.abs(gm_o))), max(scale, np.max(np.abs(gv_o))))


def test_gradient_gp_known_answer(abo, orc):
    # test/test_surrogates.jl:293-352 through the GPU path
    xs = np.array([[0.0, 0.0], [0.5, 0.5], [1.0, 1.0]])
    ys = np.array([[1.0, 0.1, 0.1], [0.5, 0.0, 0.0], [0.0, -0.1, -0.1]])
    gp = abo.update(abo.GradientGP(abo.SqExponentialKernel(), 3, 0.1), xs, ys)
    post = orc.fit_gradient(xs, ys, 0, 1.0, 1.0, 0.1)
    gm_o, gv_o = orc.posterior_mean_var(post, [[0.25, 0.25]], outputs=(0, 1, 2))
    assert np.max(np.abs(abo.posterior_grad_mean(gp, [[0.25, 0.25]]) - gm_o)) < 1e-10
    assert np.max(np.abs(abo.posterior_grad_var(gp, [[0.25, 0.25]]) - gv_o)) < 1e-10


def test_potrf_dev(abo):
    """The look-ahead Cholesky at tile counts T = n / 128 on every branch of its schedule: T <= 3 (inside the first
    outer blocks of the ramp), the outer-block ramp 1, 2, 3 (T = 4, 5, 7, 8, 17), around the overlapped inverse's b_top = 32 (31-33), the PDL
    threshold of 40 trailing tiles (40, 41) and the 64-row panel GEMMs of panels with 4096 rows or more (33 on; 44, 64-66).
    Against LAPACK, by the backward error |L L^T - A| <= N eps max|A| (gamma_{N+1}), and bit-identical when repeated."""
    import torch
    ctx = abo.default_context()
    eps = np.finfo(np.float64).eps
    for T in (1, 2, 3, 4, 5, 7, 8, 17, 31, 32, 33, 40, 41, 44, 64, 65, 66):
        n = 128 * T
        g = torch.Generator(device="cpu").manual_seed(n)
        B = torch.randn(n, n, dtype=torch.float64, generator=g).cuda()
        A = B @ B.T / n + torch.eye(n, dtype=torch.float64, device="cuda")     # O(n^3) products on the device: n = 8448
        dA = A.clone(); dB = A.clone()
        torch.cuda.synchronize()
        assert ctx.potrf_dev(dA.data_ptr(), n, n) == 0
        assert ctx.potrf_dev(dB.data_ptr(), n, n) == 0
        L = torch.tril(dA)
        assert torch.equal(L, torch.tril(dB)), T
        resid = float((L @ L.T - A).abs().max())
        assert resid <= n * eps * float(A.abs().max()), (T, resid)
        ref = np.linalg.cholesky(A.cpu().numpy())
        assert np.max(np.abs(L.cpu().numpy() - ref)) < 1e-11, T


def test_standardgp_copy_semantics(abo):
    # test/test_surrogates.jl:139-142: copy shares the prior, owns its posterior
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 0.1), [0.0, 0.5, 1.0], [0.0, 0.25, 1.0])
    cp = abo.copy(gp)
    assert cp.kernel is gp.kernel and cp.gpx is not gp.gpx
    assert abo.posterior_mean(cp, [0.25])[0] == abo.posterior_mean(gp, [0.25])[0]


# ---- O(n^2) row append vs a full re-fit (the reference re-fits: bayesian_opt.jl:125) --------
def test_append_matches_refit(abo, orc):
    c = orc.make_config("C2", n=330, m=500)
    kern = make_kernel(abo, 1, c["inv_ls"], 1.0)
    gp = abo.update(abo.StandardGP(kern, c["noise"]), c["X"][:190], c["y"][:190])
    for i in range(190, 330):                       # crosses two padding tiles (256, 384 -> grows)
        gp = abo.update(gp, c["X"][:i + 1], c["y"][:i + 1])
    assert gp.gpx.n() == 330
    post = orc.fit_standard(c["X"], c["y"], 1, c["inv_ls"], 1.0, c["noise"])
    mu_o, var_o = orc.posterior_mean_var(post, c["Xc"])
    assert close(abo.posterior_mean(gp, c["Xc"]), mu_o, 1.0)
    assert close(abo.posterior_var(gp, c["Xc"]), var_o, 1.0)
    assert np.max(np.abs(gp.gpx.factor(0) - post.U.T)) < 1e-10
    full = abo.update(abo.StandardGP(kern, c["noise"]), c["X"], c["y"])
    assert close(abo.posterior_var(gp, c["Xc"]), abo.posterior_var(full, c["Xc"]), 1.0, 1e-11)


def test_append_is_transactional(abo, orc):
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 0.0), [[-1.0, -1.0], [5.0, -5.0]], [2.0, 50.0])
    h = gp.gpx.clone()
    with pytest.raises(abo.PosDefException) as ei:
        h.append([-1.0 + 1e-12, -1.0 + 1e-12], [2.0])
    assert ei.value.info == 3 and h.n() == 2
    m1, v1 = h.posterior(np.array([[0.3, 0.2]]))
    m0, v0 = gp.gpx.posterior(np.array([[0.3, 0.2]]))
    assert m1[0] == m0[0] and v1[0] == v0[0]


@pytest.mark.parametrize("kind,n0,n1,d", [(0, 5, 30, 2), (3, 20, 40, 10), (4, 11, 26, 4)])
def test_gradient_gp_block_append_matches_refit(abo, orc, kind, n0, n1, d):
    """GradientGP: appending the p = d + 1 outputs of one point at a time (O(N^2 p)) equals the re-fit the
    reference does (GradientGP.jl:659-668), across tile boundaries (N crosses 128 / 256 / 384)."""
    rng = np.random.default_rng(17 * n1 + d)
    X = -2 + 4 * rng.random((n1, d))
    Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    Xc = -2 + 4 * rng.random((200, d))
    inv_ls, scale, noise = 1.0 / 1.5, 1.3, 1e-4
    gp = abo.update(abo.GradientGP(make_kernel(abo, kind, inv_ls, scale), d + 1, noise), X[:n0], Y[:n0])
    snapshots = []
    for i in range(n0, n1):
        prev = gp
        gp = abo.update(gp, X[:i + 1], Y[:i + 1])
        assert gp.gpx.n() == i + 1 and prev.gpx.n() == i            # functional update: the old model is untouched
        if i == n0 + 2:
            snapshots.append((prev, abo.posterior_mean(prev, Xc[:20]).copy()))
    post = orc.fit_gradient(X, Y, kind, inv_ls, scale, noise)
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    sc = max(scale, np.max(np.abs(mu_o)))
    h3_parity(orc, post, Xc, (0,), abo.posterior_mean(gp, Xc), abo.posterior_var(gp, Xc), mu_o, var_o, sc, scale)
    gm_o, gv_o = orc.posterior_mean_var(post, Xc[:40], outputs=range(d + 1))
    h3_parity(orc, post, Xc[:40], range(d + 1), abo.posterior_grad_mean(gp, Xc[:40]), abo.posterior_grad_var(gp, Xc[:40]),
              gm_o, gv_o, max(sc, np.max(np.abs(gm_o))), max(scale, np.max(np.abs(gv_o))))
    full = abo.update(abo.GradientGP(make_kernel(abo, kind, inv_ls, scale), d + 1, noise), X, Y, allow_append=False)
    # alpha is internal state (not a reference output): appended vs re-fitted factorisations agree to the FP64 floor cond(K) * eps
    cond = np.linalg.cond(post.U) ** 2
    assert close(gp.gpx.alpha(), full.gpx.alpha(), np.max(np.abs(full.gpx.alpha())), max(RTOL, 200 * cond * 2.2e-16))
    for m_old, mu_then in snapshots:                                  # copy-on-write kept the snapshot intact
        assert np.array_equal(abo.posterior_mean(m_old, Xc[:20]), mu_then)
    # transactional failure: a duplicate point with zero noise is not positive definite
    g0 = abo.update(abo.GradientGP(abo.SqExponentialKernel(), d + 1, 0.0), X[:3], Y[:3])
    h = g0.gpx.clone()
    with pytest.raises(abo.PosDefException):
        h.append(X[0], Y[0])
    assert h.n() == 3
    assert np.array_equal(h.posterior(Xc[:5])[0], g0.gpx.posterior(Xc[:5])[0])


def test_context_destroyed_before_its_handles(abo, orc):
    """Finalizers of garbage-collected bindings run in arbitrary order: destroying a context orphans its live
    handles (device memory released, calls fail cleanly, abo_gp_destroy stays valid)."""
    c = orc.make_config("C4", n=150, m=50, d=3)
    ctx2 = abo.Context(abo.default_context().device)
    h = abo.GpHandle(ctx2, c["kind"], 3, 1); h.set_params(c["inv_ls"], c["scale"], c["noise"]); h.fit(c["X"], c["y"])
    h2 = h.clone()
    m0, _ = h.posterior(c["Xc"])
    ctx2.close()                                                   # context first
    for hh in (h, h2):
        with pytest.raises(abo.AboCudaError):
            hh.posterior(c["Xc"])
        with pytest.raises(ValueError):
            hh.fit(c["X"], c["y"])
    h3 = h.clone()                                                 # a clone of an orphan is an orphan
    for hh in (h, h2, h3):
        hh.close()
    # the default context is unaffected
    g = abo.GpHandle(abo.default_context(), c["kind"], 3, 1); g.set_params(c["inv_ls"], c["scale"], c["noise"]); g.fit(c["X"], c["y"])
    assert np.array_equal(g.posterior(c["Xc"])[0], m0)


def test_clone_is_copy_on_write(abo, orc):
    """abo_gp_clone shares the device buffers; every writer (append, re-fit, destroy) must leave the
    other holders' posterior bit-identical (value semantics of Base.copy, StandardGP.jl:26)."""
    c = orc.make_config("C4", n=250, m=400, d=5)
    k = make_kernel(abo, c["kind"], c["inv_ls"], c["scale"])
    gp = abo.update(abo.StandardGP(k, c["noise"]), c["X"], c["y"])
    h0 = gp.gpx
    m0, v0 = h0.posterior(c["Xc"])
    L0 = h0.factor(0)
    h1 = h0.clone(); h2 = h0.clone()
    h1.append(c["Xc"][0], [0.1])                                  # writer 1: append on a clone (crosses 256 -> grows later)
    for i in range(1, 8):
        h1.append(c["Xc"][i], [0.1 * i])
    assert h1.n() == 258 and h0.n() == 250 and h2.n() == 250
    for h in (h0, h2):
        m, v = h.posterior(c["Xc"])
        assert np.array_equal(m, m0) and np.array_equal(v, v0) and np.array_equal(h.factor(0), L0)
    Xa = np.vstack([c["X"], c["Xc"][:8]]); ya = np.concatenate([c["y"], 0.1 * np.arange(8)]); ya[250] = 0.1
    ref = abo.GpHandle(abo.default_context(), c["kind"], 5, 1); ref.set_params(c["inv_ls"], c["scale"], c["noise"]); ref.fit(Xa, ya)
    ma, va = h1.posterior(c["Xc"][20:]); mr, vr = ref.posterior(c["Xc"][20:])
    assert close(ma, mr, 1.0, 1e-10) and close(va, vr, 1.0, 1e-10)
    h2.set_params(2 * c["inv_ls"], c["scale"], c["noise"]); h2.fit(c["X"][:100], c["y"][:100])     # writer 2: re-fit of a sharer
    assert h2.n() == 100
    m, v = h0.posterior(c["Xc"])
    assert np.array_equal(m, m0) and np.array_equal(v, v0)
    h3 = h0.clone()
    h0.close()                                                     # writer 3: the original goes away
    m, v = h3.posterior(c["Xc"])
    assert np.array_equal(m, m0) and np.array_equal(v, v0)
    h3.append(c["Xc"][0], [0.1])                                  # sole owner now: in place, still correct
    assert h3.n() == 251


# ---- batched NLML + analytic gradient (StandardGP.jl:99-114, bayesian_opt.jl:259-300) ------
def test_nlml_known_answer(abo):
    gp = abo.StandardGP(abo.SqExponentialKernel(), 0.1)
    val = abo.nlml(gp, [math.log(1.0), math.log(1.0)], [0.0, 0.5, 1.0], [0.0, 0.25, 1.0])   # test_surrogates.jl:145-170
    assert abs(val - 2.6769327097262567) < 1e-10


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_nlml_batch_standard(abo, orc, kind):
    rng = np.random.default_rng(11 + kind)
    n, d = 300, 4
    X = rng.random((n, d)); y = np.sin(3 * X).sum(1) + 0.05 * rng.standard_normal(n)
    theta = np.column_stack([np.log(rng.uniform(0.2, 2.0, 7)), np.log(rng.uniform(0.3, 5.0, 7))])
    gp = abo.StandardGP(make_kernel(abo, kind, 1.0, 1.0), 1e-3, mean=0.1)
    val, grad, info = abo.nlml_batch(gp, theta, X, y)
    assert np.all(info == 0)
    for r in range(theta.shape[0]):
        v_o, g_o = orc.nlml(X, y, kind, theta[r, 0], theta[r, 1], 1e-3, mean_c=0.1, want_grad=True)
        assert abs(val[r] - v_o) <= 1e-9 * abs(v_o), (val[r], v_o)
        assert np.all(np.abs(grad[r] - g_o) <= 1e-7 * np.maximum(np.abs(g_o), 1.0)), (grad[r], g_o)


def test_nlml_batch_gradient_gp(abo, orc):
    rng = np.random.default_rng(5)
    n, d = 25, 3
    X = -2 + 4 * rng.random((n, d)); Y = orc.rosenbrock_with_grad(X) / 100.0
    theta = np.array([[math.log(1.2), math.log(2.0)], [math.log(0.8), math.log(0.7)], [math.log(2.5), math.log(4.0)]])
    for kind in (0, 3, 5, 6):
        gp = abo.GradientGP(make_kernel(abo, kind, 1.0, 1.0), d + 1, 1e-4)
        val, grad, info = abo.nlml_batch(gp, theta, X, Y)
        assert np.all(info == 0)
        for r in range(3):
            v_o, g_o = orc.nlml(X, orc.prep_output(Y), kind, theta[r, 0], theta[r, 1], 1e-4, gradient_gp=True, want_grad=True)
            assert abs(val[r] - v_o) <= 1e-9 * abs(v_o)
            assert np.all(np.abs(grad[r] - g_o) <= 2e-6 * np.maximum(np.abs(g_o), 1.0)), (kind, grad[r], g_o)


def test_nlml_batch_reports_failed_restarts(abo):
    # the reference's own ill-conditioned set-up (test/test_bayesian_opt.jl:749-786): noise 0 and a
    # point 1e-12 away from an existing one -> pivot 3 is exactly <= 0 whatever the rounding
    X = np.array([[-1.0, -1.0], [5.0, -5.0], [-1.0 + 1e-12, -1.0 + 1e-12]]); y = np.array([2.0, 50.0, 2.0])
    gp = abo.StandardGP(abo.SqExponentialKernel(), 0.0)
    val, grad, info = abo.nlml_batch(gp, np.array([[0.0, 0.0], [0.5, 0.0]]), X, y)   # sigma^2 = 1: l31 = 1 exactly
    assert np.all(info == 3) and np.all(np.isinf(val))
    val2, _, info2 = abo.nlml_batch(gp, np.array([[0.0, 0.0]]), X[:2], y[:2])      # the first two points are fine
    assert info2[0] == 0 and np.isfinite(val2[0])


def test_hyperparameter_optimisation_improves_nlml(abo, orc):
    # test/test_bayesian_opt.jl:108-137, 597-653: returns a model, NLML does not get worse
    rng = np.random.default_rng(0)
    X = rng.random((60, 2)) * 4 - 2; y = np.sum(X ** 2, axis=1)
    y = (y - y.mean()) / y.std(ddof=1)
    gp = abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 0.3), 1e-6)
    old = [math.log(0.3), math.log(1.0)]
    new = abo.optimize_hyperparameters(gp, X, y, old, num_restarts=3, rng=rng)
    assert isinstance(new, abo.StandardGP)
    th = [math.log(abo.get_lengthscale(new)[0]), math.log(abo.get_scale(new)[0])]
    assert abo.nlml(new, th, X, y) <= abo.nlml(gp, old, X, y) + 1e-6


def test_bo_loop_branin(abo, orc):
    # config C1 shape at reduced size: StandardGP-SE + EI on 2-D Branin
    rng = np.random.default_rng(42)
    dom = abo.ContinuousDomain([-5.0, 0.0], [10.0, 15.0])
    f = lambda x: float(orc.branin(np.asarray(x)[None, :])[0])
    X0 = dom.lower + (dom.upper - dom.lower) * rng.random((10, 2))
    y0 = [f(x) for x in X0]
    gp = abo.StandardGP(1.0 * abo.with_lengthscale(abo.SqExponentialKernel(), 3.0), 1e-6)
    bo = abo.BOStruct(f, abo.ExpectedImprovement(0.01, min(y0)), gp, dom, list(X0), y0, 8, 0.0)
    bo, acq_list, _ = abo.optimize(bo, standardize="mean_scale", hyper_params=None, n_grid=4000, n_local=4, rng=rng)
    assert len(bo.xs) == 10 + 8 and len(acq_list) == 8          # exactly max_iter passes: i += 1 precedes update(BO, ..., i) (bayesian_opt.jl:441-445, 163-165)
    assert min(float(v) for v in bo.ys_non_std) <= min(y0) + 1e-12
    assert all(a >= 0 for a in acq_list)


def test_bo_loop_gradient_gp(abo, orc):
    # GradientGP + EI on Himmelblau with analytic gradients (the 2-D tutorial's objective, docs 2D_BO.jl:19-22),
    # hyper-parameters re-optimised in the loop, standardisation "scale_only" as the gradient tutorials use
    rng = np.random.default_rng(3)
    dom = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])

    def f(x):
        x1, x2 = float(x[0]), float(x[1])
        a, b = x1 * x1 + x2 - 11.0, x1 + x2 * x2 - 7.0
        return np.array([a * a + b * b, 4 * x1 * a + 2 * b, 2 * a + 4 * x2 * b])

    X0 = dom.lower + (dom.upper - dom.lower) * rng.random((6, 2))
    y0 = [f(x) for x in X0]
    gp = abo.GradientGP(1.0 * abo.with_lengthscale(abo.ApproxMatern52Kernel(), 2.0), 3, 1e-8)
    best0 = min(float(v[0]) for v in y0)
    bo = abo.BOStruct(f, abo.ExpectedImprovement(0.0, best0), gp, dom, list(X0), y0, 11, 0.0)
    bo, acq_list, (mu, sd) = abo.optimize(bo, standardize="scale_only", hyper_params="all", num_restarts_HP=2,
                                         n_grid=3000, n_local=8, rng=rng)
    assert bo.flag or len(bo.xs) == 6 + 11
    assert len(bo.ys_non_std) == len(bo.xs) and all(np.asarray(v).shape == (3,) for v in bo.ys_non_std)
    assert min(float(v[0]) for v in bo.ys_non_std) <= best0
    assert isinstance(bo.model, abo.GradientGP) and bo.model.gpx.n() == len(bo.xs)
    # the surrogate interpolates value AND gradient at the data (noise 1e-8) in standardised units
    Xd = np.array(bo.xs); Yd = np.array(bo.ys)
    gm = abo.posterior_grad_mean(bo.model, Xd).reshape(3, -1).T
    assert np.max(np.abs(gm - Yd)) <= 1e-3 * max(1.0, np.max(np.abs(Yd)))


# ---- BASELINE.json configurations at FULL size: a seeded sample of the sweep against the oracle
#      plus size-independent properties (top-k consistency, determinism, shard independence) ----
def _sample_check(abo, orc, gp, post, Xc, acq, acq_id, scale, nsample=3000, seed=0):
    rng = np.random.default_rng(seed)
    scores, ti, tv = acq.topk(gp, Xc, 100)
    sel = np.unique(np.concatenate([rng.integers(0, len(Xc), nsample), ti]))
    mu_o, var_o = orc.posterior_mean_var(post, Xc[sel])
    ref = orc.acquisition(acq_id, acq.params(), mu_o, var_o)
    mu = abo.posterior_mean(gp, Xc[sel]); var = abo.posterior_var(gp, Xc[sel])
    rec = h3_parity(orc, post, Xc[sel], (0,), mu, var, mu_o, var_o, max(scale, np.max(np.abs(mu_o))), scale, nsample=12)
    # acquisition: the formula is exact on the GPU's own posterior (1e-12), and against the oracle it is within 1e-9 of the
    # range wherever the posterior passed the strict bound; where the arbiter decided, tests/test_parity_report.py carries
    # the propagated-error analysis for this configuration (profiles/parity_r02.json)
    mine = orc.acquisition(acq_id, acq.params(), mu, var)
    assert close(scores[sel], mine, np.max(np.abs(mine)), 1e-12)
    if rec["mean"][0] == "strict" and rec["var"][0] == "strict":
        assert close(scores[sel], ref, np.max(np.abs(ref)), 10 * RTOL)
    # properties on the full set
    assert np.all(np.isfinite(scores))
    assert list(ti) == list(orc.sortperm_rev(scores, 100))                  # stable descending top-k
    assert np.array_equal(tv, scores[ti])
    # the oracle, evaluated on the GPU's top-100 plus the sample, picks the same arg-max
    assert sel[int(orc.sortperm_rev(ref, 1)[0])] == ti[0]
    # the same sweep in two shards gives the same scores (chunking / sharding independence)
    half = len(Xc) // 2 + 77
    s1 = acq(gp, Xc[:half]); s2 = acq(gp, Xc[half:])
    assert np.array_equal(np.concatenate([s1, s2]), scores)
    return scores


def test_config_c2_full_size(abo, orc):
    c = orc.make_config("C2")                                              # n = 2048, d = 6, m = 1,048,576, Matern-5/2, EI
    gp = abo.update(abo.StandardGP(make_kernel(abo, c["kind"], c["inv_ls"], c["scale"]), c["noise"]), c["X"], c["y"])
    post = orc.fit_standard(c["X"], c["y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    acq = abo.ExpectedImprovement(*c["acq_params"])
    s = _sample_check(abo, orc, gp, post, c["Xc"], acq, 0, c["scale"])
    # EI >= 0 (test/test_acquisition.jl:36-42) up to the cancellation of delta*Phi(z) + sigma*phi(z) once
    # Phi(z) is a subnormal (z < -37): the same formula gives the same few-ulp-of-subnormal noise in Julia
    assert np.all(s >= -1e-280), s.min()


def test_config_c3_full_size(abo, orc):
    c = orc.make_config("C3")                                              # GradientGP n = 512, d = 10 -> N = 5632
    gp = abo.update(abo.GradientGP(make_kernel(abo, c["kind"], c["inv_ls"], c["scale"]), 11, c["noise"]), c["X"], c["Y"])
    post = orc.fit_gradient(c["X"], c["Y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    acq = abo.ExpectedImprovement(*c["acq_params"])
    _sample_check(abo, orc, gp, post, c["Xc"], acq, 0, c["scale"], nsample=1500)


def test_config_c4_full_n(abo, orc):
    c = orc.make_config("C4", m=200_000)                                   # n = 8192, d = 20, UCB; one shard-sized slice
    gp = abo.update(abo.StandardGP(make_kernel(abo, c["kind"], c["inv_ls"], c["scale"]), c["noise"]), c["X"], c["y"])
    post = orc.fit_standard(c["X"], c["y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    acq = abo.UpperConfidenceBound(2.0)
    _sample_check(abo, orc, gp, post, c["Xc"], acq, 2, c["scale"], nsample=1500)
    L = gp.gpx.factor(0)
    assert np.max(np.abs(L - post.U.T)) < 1e-9


def test_config_c5_full_size(abo, orc):
    c = orc.make_config("C5")                                              # 256 restarts, n = 1024, d = 8
    gp = abo.StandardGP(abo.SqExponentialKernel(), c["noise"])
    val, grad, info = abo.nlml_batch(gp, c["theta"], c["X"], c["y"])
    ok = info == 0
    assert ok.sum() >= 200 and np.all(np.isfinite(val[ok])) and np.all(np.isinf(val[~ok]))
    for r in np.flatnonzero(ok)[::37]:
        v_o, g_o = orc.nlml(c["X"], c["y"], 0, c["theta"][r, 0], c["theta"][r, 1], c["noise"], want_grad=True)
        assert abs(val[r] - v_o) <= 1e-8 * abs(v_o), (r, val[r], v_o)
        assert np.all(np.abs(grad[r] - g_o) <= 1e-6 * np.maximum(np.abs(g_o), 1.0)), (r, grad[r], g_o)
    # batching independence: a restart evaluated alone gives the same bits
    r = int(np.flatnonzero(ok)[5])
    v1, g1, _ = abo.nlml_batch(gp, c["theta"][r:r + 1], c["X"], c["y"])
    assert v1[0] == val[r] and np.array_equal(g1[0], grad[r])


# ---- acquisition value + analytic gradient (batched local refinement, acq_utils.jl:55-71) ------
@pytest.mark.parametrize("acq_name", ["EI", "PI", "UCB"])
@pytest.mark.parametrize("kind,n,d", [(0, 200, 2), (1, 400, 6), (0, 700, 20)])
def test_acquisition_gradient(abo, orc, acq_name, kind, n, d):
    rng = np.random.default_rng(7 * n + d)
    X = rng.random((n, d)); y = np.sin(3 * X).sum(1) / d + 0.05 * rng.standard_normal(n)
    y = (y - y.mean()) / y.std(ddof=1)
    inv_ls, scale, noise = 1.0 / (0.5 * math.sqrt(d)), 1.2, 1e-3
    gp = abo.update(abo.StandardGP(make_kernel(abo, kind, inv_ls, scale), noise), X, y)
    post = orc.fit_standard(X, y, kind, inv_ls, scale, noise)
    best = float(np.median(y))          # a threshold in the bulk of the data: EI / PI are O(0.1), not 1e-30 tails
    acq = {"EI": abo.ExpectedImprovement(0.01, best), "PI": abo.ProbabilityImprovement(0.01, best),
           "UCB": abo.UpperConfidenceBound(2.0)}[acq_name]
    aid = {"EI": 0, "PI": 1, "UCB": 2}[acq_name]
    Xq = rng.random((37, d))
    val, grad = acq.value_and_grad(gp, Xq)
    assert close(val, acq(gp, Xq), np.max(np.abs(val)), 1e-10)      # same value as the sweep path
    # oracle: central differences of the oracle acquisition (what the reference's optimiser sees)
    h = 1e-6
    for b in range(d):
        Xp = Xq.copy(); Xp[:, b] += h; Xm = Xq.copy(); Xm[:, b] -= h
        fp = orc.acquisition(aid, acq.params(), *orc.posterior_mean_var(post, Xp))
        fm = orc.acquisition(aid, acq.params(), *orc.posterior_mean_var(post, Xm))
        fd = (fp - fm) / (2 * h)
        sc = max(np.max(np.abs(fd)), 1e-12)
        assert np.all(np.abs(grad[:, b] - fd) <= 2e-5 * sc + 1e-7 * np.abs(fd)), (b, np.max(np.abs(grad[:, b] - fd)), sc)


def test_acquisition_gradient_gradient_gp(abo, orc):
    rng = np.random.default_rng(3)
    n, d = 30, 3
    X = -2 + 4 * rng.random((n, d)); Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    gp = abo.update(abo.GradientGP(make_kernel(abo, 3, 1 / 1.5, 1.0), d + 1, 1e-4), X, Y)
    post = orc.fit_gradient(X, Y, 3, 1 / 1.5, 1.0, 1e-4)
    acq = abo.UpperConfidenceBound(2.0)
    Xq = -2 + 4 * rng.random((20, d))
    val, grad = acq.value_and_grad(gp, Xq)
    h = 1e-6
    for b in range(d):
        Xp = Xq.copy(); Xp[:, b] += h; Xm = Xq.copy(); Xm[:, b] -= h
        fd = (orc.upper_confidence_bound(*orc.posterior_mean_var(post, Xp), 2.0)
              - orc.upper_confidence_bound(*orc.posterior_mean_var(post, Xm), 2.0)) / (2 * h)
        assert np.all(np.abs(grad[:, b] - fd) <= 2e-5 * max(np.max(np.abs(fd)), 1e-12))


def test_batched_refinement_beats_grid(abo, orc):
    c = orc.make_config("C1", n=25, m=10)
    gp = abo.update(abo.StandardGP(make_kernel(abo, 0, c["inv_ls"], 1.0), 1e-6), c["X"], c["y"])
    acq = abo.ExpectedImprovement(0.01, float(c["y"].min()))
    dom = abo.ContinuousDomain(c["lower"], c["upper"])
    x_grid = abo.optimize_acquisition(acq, gp, dom, n_grid=3000, n_local=20, rng=np.random.default_rng(1), refine=False)
    x_ref = abo.optimize_acquisition(acq, gp, dom, n_grid=3000, n_local=20, rng=np.random.default_rng(1), refine=True)
    x_sci = abo.optimize_acquisition(acq, gp, dom, n_grid=3000, n_local=20, rng=np.random.default_rng(1), refine="scipy")
    a_grid, a_ref, a_sci = (float(acq(gp, x[None, :])[0]) for x in (x_grid, x_ref, x_sci))
    assert a_ref >= a_grid - 1e-15 and np.all(x_ref >= dom.lower) and np.all(x_ref <= dom.upper)
    assert a_ref >= 0.98 * a_sci                                  # as good as the sequential finite-difference scheme


# ---- posterior_grad_cov (GradientGP.jl:968-971; reference test test_surrogates.jl:331-351) ----
def test_posterior_grad_cov(abo, orc):
    xs = np.array([[0.0, 0.0], [0.5, 0.5], [1.0, 1.0]])
    ys = np.array([[1.0, 0.1, 0.1], [0.5, 0.0, 0.0], [0.0, -0.1, -0.1]])
    gp = abo.update(abo.GradientGP(abo.SqExponentialKernel(), 3, 0.1), xs, ys)
    post = orc.fit_gradient(xs, ys, 0, 1.0, 1.0, 0.1)
    cov = abo.posterior_grad_cov(gp, [[0.25, 0.25]])
    assert cov.shape == (3, 3) and np.max(np.abs(cov - orc.posterior_cov(post, [[0.25, 0.25]]))) < 1e-10
    rng = np.random.default_rng(2)
    X = -2 + 4 * rng.random((40, 4)); Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    gp = abo.update(abo.GradientGP(make_kernel(abo, 5, 0.6, 1.5), 5, 1e-4), X, Y)
    post = orc.fit_gradient(X, Y, 5, 0.6, 1.5, 1e-4)
    Xq = -2 + 4 * rng.random((7, 4))
    ref = orc.posterior_cov(post, Xq)
    cov = abo.posterior_grad_cov(gp, Xq)
    assert cov.shape == (35, 35) and np.max(np.abs(cov - ref)) < 1e-9 * max(1.0, np.max(np.abs(ref)))
    assert np.allclose(np.diag(cov), abo.posterior_grad_var(gp, Xq), rtol=0, atol=1e-11)
    sgp = abo.update(abo.StandardGP(make_kernel(abo, 1, 0.6, 1.5), 1e-4), X, Y[:, 0])
    spost = orc.fit_standard(X, Y[:, 0], 1, 0.6, 1.5, 1e-4)
    assert np.max(np.abs(abo.posterior_cov(sgp, Xq) - orc.posterior_cov(spost, Xq))) < 1e-10


# ---- GradientNormUCB and EnsembleAcquisition (gradNormUCB.jl:43-51, EnsembleAcq.jl:53-55) -----
def test_grad_norm_ucb_and_ensemble(abo, orc):
    rng = np.random.default_rng(9)
    X = -2 + 4 * rng.random((30, 3)); Y = orc.rosenbrock_with_grad(X); Y = Y / np.std(Y[:, 0])
    gp = abo.update(abo.GradientGP(make_kernel(abo, 3, 0.7, 1.2), 4, 1e-4), X, Y)
    post = orc.fit_gradient(X, Y, 3, 0.7, 1.2, 1e-4)
    Xq = -2 + 4 * rng.random((1500, 3))                      # spans two chunks of 1024 points
    g = abo.GradientNormUCB(1.5)
    val = g(gp, Xq)
    ref = orc.grad_norm_ucb(post, Xq[:60], 1.5)
    assert np.all(np.isfinite(val)) and close(val[:60], ref, np.max(np.abs(ref)), 1e-9)
    ei = abo.ExpectedImprovement(0.01, float(Y[:, 0].min()))
    ens = abo.EnsembleAcquisition([2.0, 6.0], [ei, g])          # test_acquisition.jl:223-253: weighted sum
    assert np.allclose(ens.weights, [0.25, 0.75])
    assert np.allclose(ens(gp, Xq[:100]), 0.25 * ei(gp, Xq[:100]) + 0.75 * val[:100], rtol=0, atol=1e-13)
    s, ti, tv = ens.topk(gp, Xq[:200], 10)
    assert list(ti) == list(orc.sortperm_rev(s, 10))
    e2 = ens.update(Y, gp)
    assert isinstance(e2.acquisitions[0], abo.ExpectedImprovement) and e2.acquisitions[0].best_y == float(Y[:, 0].min())
    with pytest.raises(ValueError):
        abo.EnsembleAcquisition([-1.0, 1.0], [ei, g])
    dom = abo.ContinuousDomain([-2.0] * 3, [2.0] * 3)
    x = abo.optimize_acquisition(ens, gp, dom, n_grid=500, n_local=2, rng=np.random.default_rng(0))
    assert x.shape == (3,) and np.all(x >= dom.lower) and np.all(x <= dom.upper)
    # the device top-k of the fused members is sortperm(scores; rev = true)[1:k] of the scores it returns
    sg, tg, vg = g.topk(gp, Xq, 25)
    assert list(tg) == list(orc.sortperm_rev(sg, 25)) and np.array_equal(vg, sg[tg]) and np.array_equal(sg, val)
    # batched refinement (central differences of ONE batched call per step) does not lose to the best grid point
    xg = abo.optimize_acquisition(g, gp, dom, n_grid=800, n_local=6, rng=np.random.default_rng(3), refine=False)
    xr = abo.optimize_acquisition(g, gp, dom, n_grid=800, n_local=6, rng=np.random.default_rng(3), refine=True)
    assert float(g(gp, xr[None, :])[0]) >= float(g(gp, xg[None, :])[0]) - 1e-12
    # three members incl. PI and UCB share the pass; equals the member-by-member sum
    pi = abo.ProbabilityImprovement(0.01, float(Y[:, 0].min())); ucb = abo.UpperConfidenceBound(2.0)
    e3 = abo.EnsembleAcquisition([1.0, 1.0, 2.0, 4.0], [ei, pi, ucb, g])
    ref3 = 0.125 * ei(gp, Xq[:300]) + 0.125 * pi(gp, Xq[:300]) + 0.25 * ucb(gp, Xq[:300]) + 0.5 * val[:300]
    assert np.allclose(e3(gp, Xq[:300]), ref3, rtol=1e-12, atol=1e-13)
    # value-only members on a StandardGP go through the fused sweep once
    sgp = abo.update(abo.StandardGP(make_kernel(abo, 1, 0.7, 1.2), 1e-4), X, Y[:, 0])
    e2s = abo.EnsembleAcquisition([1.0, 3.0], [ei, ucb])
    assert np.allclose(e2s(sgp, Xq[:400]), 0.25 * ei(sgp, Xq[:400]) + 0.75 * ucb(sgp, Xq[:400]), rtol=1e-13, atol=1e-14)
    with pytest.raises(TypeError):
        g(sgp, Xq[:4])                                          # GradientNormUCB needs a GradientGP


def test_grad_norm_ucb_c3_shape(abo, orc):
    """d = 10 (p = 11), the C3 kernel family: per-candidate 10 x 10 posterior gradient covariance on the device."""
    c = orc.make_config("C3", n=60, m=700)
    gp = abo.update(abo.GradientGP(make_kernel(abo, c["kind"], c["inv_ls"], c["scale"]), 11, c["noise"]), c["X"], c["Y"])
    post = orc.fit_gradient(c["X"], c["Y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    g = abo.GradientNormUCB(2.0)
    val = g(gp, c["Xc"])                                        # 700 candidates: two passes of 352
    ref = orc.grad_norm_ucb(post, c["Xc"][340:370], 2.0)
    assert np.all(np.isfinite(val)) and close(val[340:370], ref, np.max(np.abs(ref)), 1e-9)


# ---- lengthscale_bounds / monte_carlo_fill_distance (BO_utils.jl:87-159; test_bayesian_opt.jl:419-456)
def test_fill_distance_and_lengthscale_bounds(abo):
    rng = np.random.default_rng(0)
    dom = abo.ContinuousDomain([0.0, -1.0, 2.0], [1.0, 1.0, 5.0])
    X = dom.lower + rng.random((700, 3)) * (dom.upper - dom.lower)
    S = dom.lower + rng.random((5000, 3)) * (dom.upper - dom.lower)
    ref = max(np.sqrt(np.min(np.sum((X - s) ** 2, axis=1))) for s in S)
    assert abs(abo.default_context().fill_distance(X, S) - ref) <= 1e-15 * ref * 4
    lo, up = abo.lengthscale_bounds(X, dom, rng=np.random.default_rng(1))
    assert np.array_equal(up, dom.upper - dom.lower) and np.all(lo == lo[0]) and 0 < lo[0] < 0.1 * np.max(up)
    # 1-D: exact largest gap including the domain edges (test_bayesian_opt.jl:419-440)
    d1 = abo.ContinuousDomain([0.0], [1.0])
    lo1, up1 = abo.lengthscale_bounds([0.1, 0.5, 0.6], d1)
    assert abs(lo1[0] - 0.1 * 0.4) < 1e-15 and up1[0] == 1.0
    # 2-D Monte-Carlo estimate close to the analytic fill distance of a regular grid (atol 1e-2)
    g = np.array([[i, j] for i in (0.25, 0.75) for j in (0.25, 0.75)])
    d2 = abo.ContinuousDomain([0.0, 0.0], [1.0, 1.0])
    h = abo.monte_carlo_fill_distance(g, d2, n_samples=20000, rng=np.random.default_rng(2))
    assert abs(h - math.sqrt(2) * 0.25) < 1e-2


# ---- the CUDA path against the committed golden fixture and a 50-digit arbiter ----------------
def test_gpu_against_golden_fixture(abo):
    import json, os
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "known_answers.json")))
    gp = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 0.1), [0.0, 0.5, 1.0], [0.0, 0.25, 1.0])
    assert abs(abo.posterior_mean(gp, [0.25])[0] - g["G1"]["mean"]) < 1e-10
    assert abs(abo.posterior_var(gp, [0.25])[0] - g["G1"]["var"]) < 1e-10
    assert abs(abo.nlml(abo.StandardGP(abo.SqExponentialKernel(), 0.1), [0.0, 0.0], [0.0, 0.5, 1.0], [0.0, 0.25, 1.0])
               - g["G2"]["nlml"]) < 1e-10
    gp3 = abo.update(abo.StandardGP(abo.SqExponentialKernel(), 0.1), [0.0, 0.5, 1.0], [2.0, 1.0, 0.5])
    assert abs(abo.ExpectedImprovement(0.01, 0.5)(gp3, [0.25])[0] - g["G3"]["EI"]) < 1e-9 * g["G3"]["EI"]
    assert abs(abo.ProbabilityImprovement(0.01, 0.5)(gp3, [0.25])[0] - g["G3"]["PI"]) < 1e-9 * g["G3"]["PI"]
    assert abs(abo.UpperConfidenceBound(2.0)(gp3, [0.25])[0] - g["G3"]["UCB_beta2"]) < 1e-10


@pytest.mark.parametrize("noise", [1e-4, 1e-8, 1e-10])
def test_ill_conditioned_against_mpmath_arbiter(abo, orc, noise):
    """SURVEY H3: with cond(K) up to ~1e9 two valid FP64 evaluations differ by more than 1e-9, so the
    GPU is judged against 50-digit truth: its error may not exceed max(1e-9*scale, 4 x the oracle's)."""
    rng = np.random.default_rng(12)
    X = rng.random((40, 2)); y = np.sin(4 * X[:, 0]) * np.cos(3 * X[:, 1])
    Xc = rng.random((25, 2))
    gp = abo.update(abo.StandardGP(make_kernel(abo, 0, 1.0 / 0.6, 1.0), noise), X, y)
    post = orc.fit_standard(X, y, 0, 1.0 / 0.6, 1.0, noise)
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    mu_t, var_t = orc.mp_posterior_standard(X, y, 0, 1.0 / 0.6, 1.0, noise, 0.0, Xc)
    mu_t = np.array([float(v) for v in mu_t]); var_t = np.array([float(v) for v in var_t])
    mu = abo.posterior_mean(gp, Xc); var = abo.posterior_var(gp, Xc)
    e_gpu_m, e_orc_m = np.max(np.abs(mu - mu_t)), np.max(np.abs(mu_o - mu_t))
    e_gpu_v, e_orc_v = np.max(np.abs(var - var_t)), np.max(np.abs(var_o - var_t))
    assert e_gpu_m <= max(1e-9, 4 * e_orc_m), (e_gpu_m, e_orc_m)
    assert e_gpu_v <= max(1e-9, 4 * e_orc_v), (e_gpu_v, e_orc_v)


def test_determinism_and_instrumentation(abo, orc):
    """Replicas must be bit-identical (SURVEY §8e: redundant per-rank fits instead of a broadcast are only
    valid if the kernels are deterministic): two independent fits and sweeps give the same bits."""
    c = orc.make_config("C4", n=900, m=6000, d=20)
    k = make_kernel(abo, c["kind"], c["inv_ls"], c["scale"])
    g1 = abo.update(abo.StandardGP(k, c["noise"]), c["X"], c["y"])
    g2 = abo.update(abo.StandardGP(k, c["noise"]), c["X"], c["y"])
    assert np.array_equal(g1.gpx.factor(0), g2.gpx.factor(0)) and np.array_equal(g1.gpx.factor(1), g2.gpx.factor(1))
    acq = abo.UpperConfidenceBound(2.0)
    ctx = abo.default_context()
    n0 = ctx.launch_count()
    s1, t1, _ = acq.topk(g1, c["Xc"], 50)
    assert ctx.launch_count() > n0                                   # our kernels ran (no fallback exists)
    s2, t2, _ = acq.topk(g2, c["Xc"], 50)
    assert np.array_equal(s1, s2) and np.array_equal(t1, t2)
    ctx.profile(True); acq(g1, c["Xc"]); ms, cnt = ctx.profile_read(); ctx.profile(False)
    assert cnt[0] == cnt[1] == cnt[2] >= 1 and ms[1] > 0
    # clone is a deep copy: appending to the clone leaves the original untouched
    g3 = abo.copy(g1)
    g4 = abo.update(g3, np.vstack([c["X"], c["Xc"][:1]]), np.concatenate([c["y"], [0.3]]))
    assert g4.gpx.n() == 901 and g1.gpx.n() == 900 and g3.gpx.n() == 900
    assert np.array_equal(acq(g1, c["Xc"][:500]), s1[:500])
