"""Max-value entropy search without a GPU: the NumPy reference of h and h' (tests/mes_reference.py) against 50-digit
mpmath over gamma in [-40, 40], h >= 0, and the value semantics of MaxValueEntropySearch."""
import dataclasses
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mes_reference as mref  # noqa: E402

mp = pytest.importorskip("mpmath")


def _grid():
    g = np.linspace(-40.0, 40.0, 8001)
    extra = [0.0, 1e-8, -1e-8, 1e-300, -1e-300, mref.MES_TAIL, np.nextafter(mref.MES_TAIL, 0), np.nextafter(mref.MES_TAIL, -1),
             -40.0, 40.0, -3.999, -4.001, 0.5, -0.5, 7.25, -7.25, 37.5, -37.5]
    return np.unique(np.concatenate([g, extra]))


def _exact(g):
    with mp.workdps(50):
        x = mp.mpf(float(g))
        Phi = mp.ncdf(x)
        logPhi = mp.log(Phi) if x < 0 else mp.log1p(-mp.ncdf(-x))      # 1 - Phi without cancellation in the right tail
        r = mp.npdf(x) / Phi
        return float(x * r / 2 - logPhi), float(-(r / 2) * (1 + x * (x + r)))


@pytest.fixture(scope="module")
def exact():
    g = _grid()
    e = np.array([_exact(v) for v in g])
    return g, e[:, 0], e[:, 1]


def test_h_matches_mpmath(exact):
    g, h, _ = exact
    err = np.abs(mref.h(g) - h)
    assert np.all(err <= 1e-12 * np.abs(h) + 1e-300), (g[np.argmax(err / (np.abs(h) + 1e-300))], np.max(err / (np.abs(h) + 1e-300)))


def test_hprime_matches_mpmath(exact):
    g, _, hp = exact
    err = np.abs(mref.hprime(g) - hp)
    assert np.all(err <= 1e-12 * np.abs(hp) + 1e-300), (g[np.argmax(err / (np.abs(hp) + 1e-300))], np.max(err / (np.abs(hp) + 1e-300)))


def test_h_non_negative(exact):
    g, _, _ = exact
    assert np.all(mref.h(g) >= 0.0)
    assert np.all(np.isfinite(mref.h(np.array([-1e3, -1e5, 1e3, 1e5]))))
    assert np.all(mref.h(np.array([-1e3, -1e5, 1e3, 1e5])) >= 0.0)


def test_mes_reference_semantics():
    mu = np.array([0.0, 1.0, -2.0, 0.3]); var = np.array([1.0, 1e-12, 0.25, 4.0]); ys = np.array([-1.0, -0.5, 0.2])
    v = mref.mes(mu, var, ys)
    assert v[1] == 0.0                                                   # var <= 1e-12: no information
    manual = (mref.h((mu - ys[0]) / np.sqrt(var)) + mref.h((mu - ys[1]) / np.sqrt(var)) + mref.h((mu - ys[2]) / np.sqrt(var))) / 3
    assert np.array_equal(v[[0, 2, 3]], manual[[0, 2, 3]])
    dmu, dvar = mref.mes_dmu_dvar(mu, var, ys)
    assert dmu[1] == 0.0 and dvar[1] == 0.0
    eps = 1e-6
    fd_mu = (mref.mes(mu + eps, var, ys) - mref.mes(mu - eps, var, ys)) / (2 * eps)
    fd_var = (mref.mes(mu, var + eps, ys) - mref.mes(mu, var - eps, ys)) / (2 * eps)
    live = var > 1e-6
    assert np.allclose(dmu[live], fd_mu[live], rtol=1e-6, atol=1e-9)
    assert np.allclose(dvar[live], fd_var[live], rtol=1e-6, atol=1e-9)


def test_max_value_entropy_search_value_semantics():
    import abo_b200 as abo
    a = abo.MaxValueEntropySearch(7, 0.25)
    assert a.acq_id == 4 and a.has_gradient is True
    assert (a.num_max_values, a.num_features) == (16, 4096)
    with pytest.raises(dataclasses.FrozenInstanceError):
        a.seed = 8
    a._cache.update(token=1, ystar=np.zeros(16))
    b = a.copy()
    assert b == a and b is not a and b._cache == {} and hash(a) == hash(b)
    c = abo.MaxValueEntropySearch(7, 0.25, 32)
    assert c != a
    model = abo.StandardGP(abo.SqExponentialKernel(), 1e-6)
    u = a.update(np.array([1.0, -0.5, 2.0]), model)
    assert u == abo.MaxValueEntropySearch(8, -0.5) and u._cache == {}
    g = abo.GradientGP(abo.SqExponentialKernel(), 3, 1e-6)
    ug = abo.update(abo.MaxValueEntropySearch(0, 1.0, 4, 256), np.array([[2.0, 0, 0], [-3.0, 9, 9]]), g)
    assert ug == abo.MaxValueEntropySearch(1, -3.0, 4, 256)
    e = abo.EnsembleAcquisition([1.0, 1.0], [a, abo.ExpectedImprovement(0.0, 0.25)])
    assert not e._fusable()                                             # MES members take the sequential path
