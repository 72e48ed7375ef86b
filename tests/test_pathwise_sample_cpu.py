"""Host-side checks of the pathwise sampler (abo_gp_pathwise_sample): the feature and draw streams of the header against
raw NumPy Philox words, the random features against the kernels they approximate, PathwiseThompsonSampling's value
semantics and the FFI bindings of the new entry points.  The device path is in test_pathwise_sample_gpu.py."""
import importlib.util
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import pathwise_reference as pref  # noqa: E402
import sample_reference as sref  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def raw(seed, key, nblk):
    return np.random.Philox(key=np.array([seed, key], dtype=np.uint64)).random_raw(4 * nblk).reshape(nblk, 4)


def box_muller(w):
    u = pref.u01(w)
    r0, r2 = np.sqrt(-2.0 * np.log(u[0])), np.sqrt(-2.0 * np.log(u[2]))
    return [r0 * np.cos(2 * np.pi * u[1]), r0 * np.sin(2 * np.pi * u[1]), r2 * np.cos(2 * np.pi * u[3]), r2 * np.sin(2 * np.pi * u[3])]


@pytest.mark.parametrize("kind,d", [(0, 3), (1, 6), (2, 5), (3, 1)])
def test_feature_stream_from_raw_words(kind, d):
    seed, L = 2024, 5
    Om, b = pref.features(seed, L, d, kind)
    kdf = pref.KDF[kind]
    nblk = (d + kdf + 3) // 4
    for l in range(L):
        key = 2 ** 64 - 1 - l
        w = raw(seed, key, nblk + 1)
        assert [int(v) for v in w[0]] == sref.philox4x64_10((1, 0, 0, 0), (seed, key))
        z = np.concatenate([box_muller(w[j]) for j in range(nblk)])
        t = np.sqrt(kdf / np.sum(z[d:d + kdf] ** 2)) if kdf else 1.0
        assert np.array_equal(Om[l], z[:d] * t)
        assert b[l] == 2.0 * np.pi * ((int(w[nblk, 0]) >> 11) + 0.5) * 2.0 ** -53


def test_draw_stream_from_raw_words():
    seed, S, L, N = 7, 3, 6, 9                          # eps starts inside a Philox block (L = 6 is not a multiple of 4)
    Th = pref.draw_normals(seed, S, L + N)
    for s in range(S):
        w = raw(seed, 2 ** 63 + s, (L + N + 3) // 4)
        z = np.concatenate([box_muller(w[j]) for j in range(len(w))])
        assert np.array_equal(Th[s], z[:L + N])
        assert np.array_equal(sref.philox_normals(seed, s, 8), raw_normals(seed, s, 8))   # the joint sampler's key space is separate


def raw_normals(seed, key, m):
    w = raw(seed, key, (m + 3) // 4)
    return np.concatenate([box_muller(w[j]) for j in range(len(w))])[:m]


@pytest.mark.parametrize("case", ["se", "matern52", "matern72", "ard"])
def test_features_approximate_the_kernel(case):
    """E_l[2 cos(omega_l x + b_l) cos(omega_l x' + b_l)] = k(x, x') / sigma^2.  Each pair is checked against 5 Monte-Carlo
    standard errors of that mean at L = 65536: a Gaussian frequency in place of the Student-t one, a wrong degree of
    freedom, or the ARD scales applied to the wrong dimensions move k by many standard errors."""
    from oracle import abo_oracle as orc
    kind = {"se": 0, "matern52": 1, "matern72": 2, "ard": 1}[case]
    d = 3
    sv = np.array([2.5, 0.7, 1.3]) if case == "ard" else np.full(d, 1.0 / 0.8)
    L = 65536
    Om, b = pref.features(11, L, d, kind)
    rng = np.random.default_rng(5)
    X = rng.random((6, d))
    Y = np.vstack([X[:3] + np.array([0.3, 0.0, 0.0]), X[3:] + np.array([0.0, 0.0, 0.6])])   # pairs along one axis each
    Y = np.vstack([Y, X[:1]])
    X = np.vstack([X, X[:1] + np.array([0.2, 0.5, -0.3])])
    for x, y in zip(X, Y):
        terms = 2.0 * pref.phi_value(x, sv, Om, b)[0] * pref.phi_value(y, sv, Om, b)[0]
        k = orc.kernelmatrix(kind, sv, 1.0, x[None, :], y[None, :])[0, 0]
        se = terms.std() / np.sqrt(L)
        assert abs(terms.mean() - k) <= 5 * se, (case, terms.mean(), k, se)


def test_pathwise_thompson_value_semantics():
    import abo_b200 as abo
    a = abo.PathwiseThompsonSampling(7)
    assert a.num_features == 4096 and a.has_gradient is False
    b = a.update(None, None)
    assert isinstance(b, abo.PathwiseThompsonSampling) and b.seed == 8 and a.seed == 7
    c = abo.PathwiseThompsonSampling(3, num_features=1024)
    assert c.copy() == c and c.copy() is not c and c.update(None, None) == abo.PathwiseThompsonSampling(4, 1024)
    with pytest.raises(TypeError):
        a.value_and_grad(None, np.zeros((1, 2)))


def test_ffi_bindings_of_the_pathwise_entry_points():
    spec = importlib.util.spec_from_file_location("check_ffi", os.path.join(ROOT, "tools", "check_ffi_signatures.py"))
    chk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(chk)
    protos = chk.c_prototypes()
    sig = ["ptr:void", "ptr:double", "int64", "int64", "int64", "uint64", "ptr:double", "ptr:int64", "ptr:double"]
    assert protos["abo_gp_pathwise_sample"] == ("int32", sig)
    assert protos["abo_gp_pathwise_sample_dev"] == ("int32", sig)
    assert not chk.check_julia(protos)[1] and not chk.check_ctypes(protos)[1]
    assert "abo_gp_pathwise_sample" in {c[0] for c in chk.julia_ccalls()}
