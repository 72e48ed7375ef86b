"""abo_gp_fit at the tile counts T = ceil(N / 128), N = n p, where its conditioning schedule changes.  From T = 32 on
(FIT_OVERLAP_MIN_TILES) the triangular inverse of the leading b_top tile columns (b_top: the largest power of two below T)
runs on a second stream while the Cholesky factorisation finishes.  That stream is ordered after the factorisation at
the first outer-block boundary in [b_top, T) or, where the ramped boundaries 1, 3, 6, 9, ... leave none there
(T = 33, 65, 66, 129, ...), after the whole factor.  Each fit is checked against the CPU oracle on the same data: the
factor L, L^-1 by O(N^2) probes, alpha and the posterior; a second fit of the same data gives the same bits.  The O(N^2)
append (one more point, no re-fit) crosses the same tile boundaries on a path of its own and must agree with both.
The hyper-parameters keep cond(K + noise I) <= 1e5, so the strict 1e-9 bound of h3_parity decides, not its arbiter."""
import numpy as np
import pytest
import scipy.linalg as sla

from test_gpu_parity import close, h3_parity, make_kernel

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
COND_MAX = 1e5
STANDARD = dict(kind=1, inv_ls=1 / 0.15, scale=1.0, noise=1e-2, mean=0.3)      # Matern-5/2, d = 6
GRADIENT = dict(kind=3, inv_ls=1 / 0.12, scale=1.0, noise=1e-1)                # ApproxMatern-5/2 (differentiable at 0)


@pytest.fixture(scope="module")
def abo():
    import abo_b200
    return abo_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import abo_oracle
    return abo_oracle


def _tiles(n, p):
    return -(-n * p // 128)


def _data(d, n, p):
    """n seeded points in [0, 1]^d with values (p = 1) or values and gradients (p = d + 1) of sum(sin(6 x)); the data
    for n are a prefix of the data for any larger n, so an append and a re-fit see the same points."""
    X = np.random.default_rng(2024 + d).random((n, d))
    f = np.sin(6 * X).sum(1)
    return (X, f) if p == 1 else (X, np.column_stack([f, 6 * np.cos(6 * X)]))


def _model(abo, d, p):
    if p == 1:
        s = STANDARD
        return abo.StandardGP(make_kernel(abo, s["kind"], s["inv_ls"], s["scale"]), s["noise"], mean=s["mean"])
    g = GRADIENT
    return abo.GradientGP(make_kernel(abo, g["kind"], g["inv_ls"], g["scale"]), d + 1, g["noise"])


@pytest.fixture(scope="module")
def oracle_fit(orc):
    """The oracle posterior of _data(d, n, p), its condition-number estimate and its factor in the library's order,
    computed once per module: the re-fit and the append tests at the same size share them."""
    cache = {}

    def get(d, n, p):
        if (d, n, p) not in cache:
            X, Y = _data(d, n, p)
            if p == 1:
                s = STANDARD
                post = orc.fit_standard(X, Y, s["kind"], s["inv_ls"], s["scale"], s["noise"], s["mean"])
            else:
                g = GRADIENT
                post = orc.fit_gradient(X, Y, g["kind"], g["inv_ls"], g["scale"], g["noise"])
            cond = orc.cond_estimate(post.U, iters=10)
            assert cond <= COND_MAX, cond                  # keeps the strict 1e-9 comparison in charge
            cache[(d, n, p)] = (post, cond, _reference_factor(orc, post))
        return cache[(d, n, p)]
    return get


def _reference_factor(orc, post):
    """The oracle's lower Cholesky factor in the library's point-major system order (index i p + a, include/abo.h).
    For a GradientGP that is the factor of the permuted matrix, which is not a permutation of the out-major factor."""
    if post.p == 1:
        return post.U.T
    n, p = post.n, post.p
    perm = np.arange(n * p).reshape(p, n).T.ravel()               # point-major index i p + a -> out-major a n + i
    C = orc.grad_kernelmatrix(post.kind, post.inv_ls, post.scale, post.X)[np.ix_(perm, perm)]
    C[np.diag_indices_from(C)] += post.noise
    return sla.cholesky(C, lower=True, check_finite=False)


def _check_factor_and_alpha(gp, post, L_ref, cond, seed):
    """L against the oracle's factor; L^-1 by probes L^-1 (L v) = v (O(N^2), no N^3 product); alpha = K^-1 (y - m) to
    its FP64 floor cond(K) eps."""
    N = post.U.shape[0]
    L = gp.gpx.factor(0)
    err = float(np.max(np.abs(L - L_ref)))
    assert err <= 1e-10, ("factor", err)
    V = np.random.default_rng(seed).standard_normal((N, 4))
    LV = L @ V
    del L
    R = gp.gpx.factor(1) @ LV - V
    err = float(np.max(np.max(np.abs(R), axis=0) / np.max(np.abs(V), axis=0)))
    assert err <= 1e-10, ("L^-1 L v - v", err)
    a = gp.gpx.alpha()
    tol = max(1e-10, 100 * cond * EPS)
    assert close(a, post.alpha, np.max(np.abs(post.alpha)), tol), ("alpha", float(np.max(np.abs(a - post.alpha))), tol)


def _check_posterior(abo, orc, gp, post, Xc, p, m_grad=300):
    """Value-output mean and variance at Xc; for a GradientGP also every output's mean and variance at Xc[:m_grad]."""
    scale = post.scale
    mu_o, var_o = orc.posterior_mean_var(post, Xc)
    sc = max(scale, np.max(np.abs(mu_o)))
    h3_parity(orc, post, Xc, (0,), abo.posterior_mean(gp, Xc), abo.posterior_var(gp, Xc), mu_o, var_o, sc, scale)
    if p > 1:
        Xg = Xc[:m_grad]
        gm_o, gv_o = orc.posterior_mean_var(post, Xg, outputs=range(p))
        h3_parity(orc, post, Xg, range(p), abo.posterior_grad_mean(gp, Xg), abo.posterior_grad_var(gp, Xg), gm_o, gv_o,
                  max(sc, np.max(np.abs(gm_o))), max(scale, np.max(np.abs(gv_o))))


def _check_same_bits(abo, gp, d, p, X, Y, Xc):
    """A second fit of the same data on a fresh handle: the fit has no atomics, so any difference is a race."""
    gp2 = abo.update(_model(abo, d, p), X, Y)
    assert np.array_equal(gp.gpx.alpha(), gp2.gpx.alpha())
    assert np.array_equal(abo.posterior_mean(gp, Xc), abo.posterior_mean(gp2, Xc))
    assert np.array_equal(abo.posterior_var(gp, Xc), abo.posterior_var(gp2, Xc))


# T = 31: no overlap; T = 32: the first overlapped size; T = 33, 65, 66, 129: no outer-block boundary in [b_top, T).
# N = 16400 is also above FS_MAX_NPAD, so its posterior takes the three-kernel sweep (gemm_tma_kernel<EPI_COLSUMSQ>), not sweep_fused.
@pytest.mark.parametrize("n", [pytest.param(n, id=f"T{_tiles(n, 1)}-n{n}") for n in (3900, 4096, 4097, 4224, 8193, 8400, 16400)])
def test_standard_fit_across_overlap_schedule(abo, orc, oracle_fit, n):
    post, cond, L_ref = oracle_fit(6, n, 1)
    X, y = _data(6, n, 1)
    Xc = np.random.default_rng(n).random((2000, 6))
    gp = abo.update(_model(abo, 6, 1), X, y)
    _check_factor_and_alpha(gp, post, L_ref, cond, seed=n)
    _check_posterior(abo, orc, gp, post, Xc, 1)
    _check_same_bits(abo, gp, 6, 1, X, y, Xc)


@pytest.mark.parametrize("d,n", [pytest.param(d, n, id=f"T{_tiles(n, d + 1)}-d{d}-n{n}") for d, n in ((3, 1025), (3, 2100), (10, 373))])
def test_gradient_fit_across_overlap_schedule(abo, orc, oracle_fit, d, n):
    p = d + 1
    post, cond, L_ref = oracle_fit(d, n, p)
    X, Y = _data(d, n, p)
    Xc = np.random.default_rng(n).random((1000, d))
    gp = abo.update(_model(abo, d, p), X, Y)
    _check_factor_and_alpha(gp, post, L_ref, cond, seed=n)
    _check_posterior(abo, orc, gp, post, Xc, p)
    _check_same_bits(abo, gp, d, p, X, Y, Xc)


# N = 4096 -> 4097, 8192 -> 8193 (StandardGP) and 4096 -> 4100 (GradientGP, d = 3): the append grows the factor by one tile
@pytest.mark.parametrize("d,n0,p", [pytest.param(6, 4096, 1, id="standard-n4096"), pytest.param(6, 8192, 1, id="standard-n8192"),
                                    pytest.param(3, 1024, 4, id="gradient-d3-n1024")])
def test_append_across_tile_boundary_matches_refit(abo, orc, oracle_fit, d, n0, p):
    n = n0 + 1
    post, cond, L_ref = oracle_fit(d, n, p)
    X, Y = _data(d, n, p)
    Xc = np.random.default_rng(n).random((2000, d))
    gp0 = abo.update(_model(abo, d, p), X[:n0], Y[:n0])
    ctx = abo.default_context()
    launches = ctx.launch_count()
    gp = abo.update(gp0, X, Y)                              # copy-on-write clone + O(N^2) append
    assert gp.gpx.n() == n and gp0.gpx.n() == n0
    assert ctx.launch_count() - launches < _tiles(n, p)     # not a re-fit: a fit enqueues more than one launch per tile
    _check_factor_and_alpha(gp, post, L_ref, cond, seed=n)
    _check_posterior(abo, orc, gp, post, Xc, p)
    full = abo.update(_model(abo, d, p), X, Y)               # a fresh fit at the new size, on the GPU
    assert np.max(np.abs(gp.gpx.factor(0) - full.gpx.factor(0))) <= 1e-10
    for f in ((abo.posterior_mean, abo.posterior_var) if p == 1 else (abo.posterior_grad_mean, abo.posterior_grad_var)):
        ref = f(full, Xc)
        assert close(f(gp, Xc), ref, max(post.scale, np.max(np.abs(ref))))
