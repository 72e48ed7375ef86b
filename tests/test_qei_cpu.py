"""Host-side checks of Monte-Carlo batch expected improvement (abo_acq_qei): the torch reference against analytic EI and
against central differences, qExpectedImprovement's value semantics, the FFI bindings of the entry point and the batch
branch of optimize_acquisition.  The device path is in test_qei_gpu.py."""
import importlib.util
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import qei_reference as qref  # noqa: E402
import sample_reference as sref  # noqa: E402

from oracle import abo_oracle as orc  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fit(case, n=40, d=3, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    f = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, -1]) + 0.5 * X.sum(1)
    if case == "gradient":
        g = np.zeros((n, d)); g[:, 0] = 3 * np.cos(3 * X[:, 0]); g[:, -1] += -2 * np.sin(2 * X[:, -1]); g += 0.5
        return orc.fit_gradient(X, np.column_stack([f, g]), 1, 1.0 / 0.7, 1.3, 1e-4), rng
    kind = 1 if case == "matern52" else 0
    inv_ls = np.array([2.0, 0.9, 1.4])[:d] if case == "ard" else 1.0 / 0.6
    return orc.fit_standard(X, f, kind, inv_ls, 1.5, 1e-4, 0.3), rng


def test_stream_key_range():
    z = qref.normals(9, 3, 5)
    for s in range(3):
        assert np.array_equal(z[s], sref.philox_normals(9, 2 ** 62 + s, 5))
    assert not np.array_equal(z[0], sref.philox_normals(9, 0, 5))


@pytest.mark.parametrize("case", ["se", "matern52"])
def test_q1_matches_analytic_ei(case):
    post, rng = fit(case)
    Xb = rng.random((6, 1, 3))
    mu, var = orc.posterior_mean_var(post, Xb[:, 0])
    best = float(np.max(mu)) + 0.1                                     # every point improves with fair probability
    S = 4096
    v, _, tau, imp = qref.qei(post, Xb, 0.01, best, S, seed=3, want_grad=False)
    ei = orc.expected_improvement(mu, var + tau, 0.01, best)
    se = imp.std(axis=1) / np.sqrt(S)
    assert np.all(np.abs(v - ei) <= 5 * se + 1e-12), (v, ei, se)


@pytest.mark.parametrize("case", ["se", "matern52", "ard", "gradient"])
def test_reference_gradient_against_central_differences(case):
    post, rng = fit(case, seed=1)
    q, d, S = 3, 3, 64
    Xb = rng.random((4, q, d))
    mu, _ = orc.posterior_mean_var(post, Xb.reshape(-1, d))
    best = float(np.max(mu))
    v, g, tau, _ = qref.qei(post, Xb, 0.0, best, S, seed=5)
    assert np.all(v > 0)
    h = 1e-6
    fd = np.zeros_like(g)
    for j in range(q):
        for k in range(d):
            P = Xb.copy(); P[:, j, k] += h
            M = Xb.copy(); M[:, j, k] -= h
            fd[:, j, k] = (qref.qei(post, P, 0.0, best, S, 5, want_grad=False, tau=tau)[0] -
                           qref.qei(post, M, 0.0, best, S, 5, want_grad=False, tau=tau)[0]) / (2 * h)
    assert np.max(np.abs(g - fd)) <= 1e-6 * max(1.0, np.max(np.abs(g))), np.max(np.abs(g - fd))


def test_qei_value_semantics():
    import abo_b200 as abo
    a = abo.qExpectedImprovement(0.01, 1.5, 4)
    assert a.num_samples == 512 and a.seed == 0 and a.q == 4 and a.has_gradient
    assert a.copy() == a and a.copy() is not a
    b = a.update(np.array([3.0, 0.25, 2.0]), None)
    assert b == abo.qExpectedImprovement(0.01, 0.25, 4, 512, 1) and a.seed == 0 and a.best_y == 1.5
    c = abo.qExpectedImprovement(0.0, 0.0, 2, num_samples=128, seed=7)
    assert c.update(np.array([[1.0], [-2.0]]), None) == abo.qExpectedImprovement(0.0, -2.0, 2, 128, 8)
    with pytest.raises(TypeError):
        a.topk(None, np.zeros((3, 2)), 1)


def test_ffi_bindings_of_the_qei_entry_point():
    spec = importlib.util.spec_from_file_location("check_ffi", os.path.join(ROOT, "tools", "check_ffi_signatures.py"))
    chk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(chk)
    protos = chk.c_prototypes()
    sig = ["ptr:void", "ptr:double", "int32", "ptr:double", "int64", "int64", "uint64", "double", "ptr:double", "ptr:double",
           "ptr:double"]
    assert protos["abo_acq_qei"] == ("int32", sig)
    assert not chk.check_julia(protos)[1] and not chk.check_ctypes(protos)[1]
    assert "abo_acq_qei" in {c[0] for c in chk.julia_ccalls()}


class _FakeBatchAcq:
    """A smooth batch acquisition with a known maximiser: -sum_j |x_j - c_j|^2 over the q points of a batch."""
    has_gradient = True

    def __init__(self, centres):
        self.c = np.asarray(centres, dtype=np.float64)
        self.q = len(self.c)
        self.calls = []

    def __call__(self, surrogate, batches):
        b = np.asarray(batches)
        self.calls.append(("value", b.shape))
        return -np.sum((b - self.c[None]) ** 2, axis=(1, 2))

    def value_and_grad(self, surrogate, batches):
        b = np.asarray(batches)
        self.calls.append(("grad", b.shape))
        return -np.sum((b - self.c[None]) ** 2, axis=(1, 2)), -2 * (b - self.c[None])


def test_batch_branch_of_optimize_acquisition():
    import abo_b200 as abo
    domain = abo.ContinuousDomain([-1.0, 0.0], [1.0, 2.0])
    acq = _FakeBatchAcq([[0.5, 1.0], [-0.25, 0.5], [1.5, 1.9]])         # the last centre lies outside the box
    x = abo.optimize_acquisition(acq, None, domain, n_grid=300, n_local=7, rng=np.random.default_rng(0))
    assert x.shape == (3, 2)
    assert np.all(x >= domain.lower) and np.all(x <= domain.upper)
    assert np.allclose(x, [[0.5, 1.0], [-0.25, 0.5], [1.0, 1.9]], atol=1e-4)
    assert acq.calls[0] == ("value", (100, 3, 2)) and all(c[0] == "grad" and c[1][1:] == (3, 2) for c in acq.calls[1:])
    raw = abo.optimize_acquisition(acq, None, domain, n_grid=300, n_local=7, rng=np.random.default_rng(0), refine=False)
    assert raw.shape == (3, 2) and acq(None, raw[None])[0] <= acq(None, x[None])[0]
